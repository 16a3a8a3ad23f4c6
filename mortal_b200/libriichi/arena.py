"""libriichi.arena — OneVsThree / TwoVsTwo on the CUDA environment.

Call-compatible with arena/one_vs_three.rs:17-113 and arena/two_vs_two.rs:17-110 for the `py_vs_py` entry
(the one mortal/player.py:64-69,142-147 and mortal/one_vs_three.py:88-93 use). Seat / seed layout:
one_vs_three.rs:140-191 (game g = 4*s + r uses seed (seed_start[0] + s, seed_start[1]); the challenger
sits at absolute seat r). The step loop is BatchGame::run (game.rs:286-304) executed by mjx kernels;
engines are called once per cycle per agent like MortalBatchAgent::evaluate (mortal.rs:114-159).

With `adopt_reference_engines` (libriichi.install(adopt_reference_engines=True)), MortalEngine objects of versions 2-4 on the
arena's device are played through mortal_b200.engine.ReferenceEngine: the observations never leave the GPU, the rows are split per
agent on the device and each engine's forward + action selection replays as one CUDA graph, greedy or sampled, with or without logs.

Tables are independent, so for reference-protocol engines (react_batch over host arrays) the batch is played as TWO half-batches
stepped alternately (`pipeline`): while an engine works on the rows of one half on the host, the environment kernels and the
D2H copies of the other half run. Results are those of one batch. Device engines run the batch as one.
"""
from __future__ import annotations

import time

import numpy as np

from ..engine import HostProtocolEngine, ReferenceEngine
from ..env import BatchEnv
from ..model import OBS_ROWS


class _MetaRecorder:
    """Collects what agent/mortal.rs:161-186 gen_meta puts into a logged reaction: per step the rows' (table, seat, kan-select,
    action, legal mask, Q-values, shanten / furiten read back from the v4 observation) and the per-table log length right after
    every environment step; `finish()` groups them per game for mortal_b200.mjai_log.attach_meta."""

    def __init__(self, n_games: int, version: int):
        self.n, self.version = n_games, version
        self.bounds, self.rows, self.q = [], [], {}
        self.error = None  # the metadata is optional: a failure while recording must never take the game loop down

    def _guard(fn):
        def wrapped(self, *a, **k):
            if self.error is not None:
                return None
            try:
                return fn(self, *a, **k)
            except Exception as exc:
                self.error = exc
                return None
        return wrapped

    @_guard
    def add_bounds(self, log_len_dev):
        self.bounds.append(log_len_dev.cpu().numpy().copy())

    @_guard
    def add_agent(self, cycle, idx, q, eval_ns, greedy=None):
        """eval_ns: nanoseconds, or a (start, end) pair of CUDA events around the engine's work on the recording stream"""
        g = None if greedy is None else np.asarray(greedy.cpu() if hasattr(greedy, "cpu") else greedy, dtype=bool)
        entry = (idx.cpu().numpy(), q.float().cpu().numpy())  # synchronises the stream, so both events have completed
        if isinstance(eval_ns, tuple):
            eval_ns = max(1, int(eval_ns[0].elapsed_time(eval_ns[1]) * 1e6))
        self.q.setdefault(cycle, []).append((*entry, int(eval_ns), g))

    @_guard
    def add_rows(self, cycle, tbl, row_seat, actions, masks, obs):
        sh = fu = None
        if self.version == 4:  # v4 rows 861 (furiten) and 862-868 (shanten one-hot), obs_repr.rs
            sh = obs[:, 862:869, 0].argmax(1).cpu().numpy()
            fu = (obs[:, 861, 0] > 0).cpu().numpy()
        self.rows.append((cycle, tbl.cpu().numpy(), row_seat.cpu().numpy(), actions.cpu().numpy(), masks.cpu().numpy().astype(bool), sh, fu))

    def finish(self):
        from ..mjai_log import make_meta

        if self.error is not None:
            raise self.error
        decisions = [dict() for _ in range(self.n)]
        for cycle, tbl, rs, act, masks, sh, fu in self.rows:
            nr = len(tbl)
            q_rows = np.zeros((nr, 46), dtype=np.float32)
            batch, ns = np.zeros(nr, dtype=np.int64), np.zeros(nr, dtype=np.int64)
            greedy = np.ones(nr, dtype=bool)
            for idx, q, eval_ns, g in self.q.get(cycle, []):
                q_rows[idx] = q
                batch[idx] = len(idx)
                ns[idx] = eval_ns
                if g is not None:
                    greedy[idx] = g
            pos = {(int(tbl[r]), int(rs[r] & 3), bool(rs[r] & 4)): r for r in range(nr)}
            for (t, seat, kan), r in pos.items():
                if kan:
                    continue
                common = dict(batch_size=int(batch[r]), eval_time_ns=int(ns[r]), shanten=None if sh is None else int(sh[r]),
                              at_furiten=None if fu is None else bool(fu[r]))
                kan_meta = None
                kr = pos.get((t, seat, True))
                if kr is not None and int(act[r]) == 42:
                    km = make_meta(int(act[kr]), masks[kr], q_rows[kr], is_greedy=bool(greedy[kr]), **common)
                    kan_meta = {k: v for k, v in km.items() if not k.startswith("_") and v is not None}
                decisions[t].setdefault(cycle, {})[seat] = make_meta(int(act[r]), masks[r], q_rows[r], is_greedy=bool(greedy[r]),
                                                                     kan_select=kan_meta, **common)
        return np.array(self.bounds), decisions


class _Part:
    """One independently stepped slice of the batch: a BatchGame (game.rs:222-316) over tables [offset, offset + n)."""

    def __init__(self, arena, agents, nonces, keys, offset, per, challenger_seats, versions, quick_evals, use_stream):
        import torch

        self.arena, self.agents, self.offset, self.per = arena, agents, offset, per
        self.nonces, self.keys, self.n = nonces, keys, len(nonces)
        version, quick_eval = versions[0], quick_evals[0]
        self.versions = list(versions)
        self.mixed = versions[0] != versions[1]  # agent/mortal.rs:54-74: every agent encodes with its own obs version
        self.env = env = arena.env_factory(nonces, keys, obs_version=version, shuffle_kind=arena.shuffle_kind,
                                           enable_quick_eval=quick_eval, device=arena.device)
        self.dev = dev = env.device
        self.stream = torch.cuda.Stream(dev) if (use_stream and dev.type == "cuda") else None
        self.is_challenger = torch.zeros((per, 4), dtype=torch.bool, device=dev)
        for g in range(per):
            for s in challenger_seats(g):
                self.is_challenger[g, s] = True
        self.ic_host = self.is_challenger.cpu().numpy()
        if quick_evals[0] != quick_evals[1]:  # enable_quick_eval is the agent's, so the seat's (mortal.rs:210-250)
            qf = np.zeros((self.n, 4), dtype=np.uint8)
            for g in range(self.n):
                for seat in range(4):
                    qf[g, seat] = quick_evals[0] if self.ic_host[g % per, seat] else quick_evals[1]
            env.set_quick_eval(qf)
        if arena.record_grp and hasattr(env, "enable_grp"):
            env.enable_grp()
        self.meta_rec = None
        if arena.log_dir is not None:
            env.enable_log()
            self.meta_rec = _MetaRecorder(self.n, 0 if self.mixed else version) if arena.log_meta else None
        self.actions = torch.zeros(env.row_cap, dtype=torch.int64, device=dev)
        guards = [bool(getattr(a, "enable_rule_based_agari_guard", False)) for a in agents]
        self.q_all = None
        if any(guards):  # mortal.rs:319-336 needs the Q-values of the previous decision
            flags = np.zeros((self.n, 4), dtype=np.uint8)
            for g in range(self.n):
                for seat in range(4):
                    flags[g, seat] = guards[0] if self.ic_host[g % per, seat] else guards[1]
            env.set_agari_guard(flags)
            self.q_all = torch.zeros((env.row_cap, 46), dtype=torch.float32, device=dev)
        # engines that only speak the reference protocol (react_batch over host arrays) get the observations through
        # mjx_env_encode_obs_host: pinned host buffers, D2H overlapped with the single-player kernels
        self.host_mode = all(isinstance(a, HostProtocolEngine) for a in agents)
        rows_of = {1: 938, 2: 942, 3: 934, 4: 1012}
        if self.host_mode:
            pin = (lambda t: t.pin_memory()) if dev.type == "cuda" else (lambda t: t)
            self.h_obs = pin(torch.empty((env.row_cap, env.obs_rows, 34), dtype=torch.float32))
            # a second host buffer when the champion encodes another obs version
            self.h_obs2 = pin(torch.empty((env.row_cap, rows_of[versions[1]], 34), dtype=torch.float32)) if self.mixed else None
            self.h_masks = pin(torch.empty((env.row_cap, 46), dtype=torch.bool))
            self.h_actions = pin(torch.zeros(env.row_cap, dtype=torch.int64))
            self.h_q = pin(torch.zeros((env.row_cap, 46), dtype=torch.float32)) if self.q_all is not None else None
            self.obs_np, self.masks_np = self.h_obs.numpy(), self.h_masks.numpy()
        # agent/mortal.rs:253-255: engines with is_oracle also get the invisible observation (board.rs:680-782) of their rows
        self.oracle = [bool(getattr(a, "is_oracle", False)) for a in agents]
        self.version = version
        self.h_inv = None
        if any(self.oracle) and self.host_mode:
            inv_rows = 211 if version == 1 else 217
            self.h_inv = pin(torch.empty((env.row_cap, inv_rows, 34), dtype=torch.float32))
        # MortalEngines adopted onto the device path (ReferenceEngine): persistent per-version observation buffers (stable graph
        # keys), the Q / greedy outputs of the select kernel, and for two engines the device-side split of the rows
        self.adopted = all(isinstance(a, ReferenceEngine) for a in agents)
        if self.adopted:
            self.obs_bufs = {v: torch.empty((env.row_cap, OBS_ROWS[v], 34), dtype=torch.float32, device=dev) for v in set(versions)}
            self.q_dev = self.q_all if self.q_all is not None else torch.zeros((env.row_cap, 46), dtype=torch.float32, device=dev)
            self.greedy = torch.ones(env.row_cap, dtype=torch.uint8, device=dev)
            if agents[0] is not agents[1]:  # agent 0 = challenger, 1 = champion
                self.agent_of = torch.from_numpy((~self.ic_host[np.arange(self.n) % per]).astype(np.uint8)).to(dev)
                self.split = [torch.zeros(env.row_cap, dtype=torch.int32, device=dev) for _ in range(2)]
                self.counts = torch.zeros(2, dtype=torch.int32, device=dev)
        self.first, self.cycles, self.nr = True, 0, 0
        self.recorded, self.recorded_masks = [], []
        self.mask_weights = (1 << torch.arange(46, dtype=torch.int64))

    # every device call of the part goes to its own stream, so the two parts overlap on the GPU
    def _ctx(self):
        import contextlib

        import torch

        return torch.cuda.stream(self.stream) if self.stream is not None else contextlib.nullcontext()

    def start(self, fast_forward):
        with self._ctx():
            if fast_forward:
                self.env.step(None)
                for _ in range(int(fast_forward)):
                    self.env.policy_test(2, self.actions)
                    self.env.step(self.actions)
                self.first = False
                self._after_step()
            else:
                self.begin()

    def begin(self):
        """One BatchGame::run iteration for this part: commit the decisions, poll to the next decision point (game.rs:286-296);
        in host mode the encode and the D2H copies are enqueued right away."""
        with self._ctx():
            self.env.step(None if self.first else self.actions, None if self.first else self.q_all)
            self.first = False
            self._after_step()

    def _after_step(self):
        if self.meta_rec is not None:
            self.meta_rec.add_bounds(self.env.log_len)
        if self.host_mode and not self.mixed:
            self.nr = self.env.encode_obs_host_begin(self.h_obs, self.h_masks)

    def finish(self):
        """Wait for the part's step; game.rs:288,292: an error from any table aborts the whole batch at that cycle (`?`);
        so does a single-player arena overflow, which would otherwise hand zeroed rows 889-1011 to the engines."""
        with self._ctx():
            if self.host_mode and not self.mixed:
                self.env.encode_obs_host_finish()
            nr, n_live, n_err, sp_ovf = self.env.poll()
        if n_err:
            res = self.env.results()
            bad = int(np.nonzero(res["err"])[0][0])
            raise RuntimeError(f"table {self.offset + bad} (seed {int(self.nonces[bad])},{int(self.keys[bad])}) failed at cycle "
                               f"{self.cycles} with mjx error code {int(res['err'][bad])} (invalid action or inconsistent state; "
                               "board.rs:527-532)")
        if sp_ovf:
            raise RuntimeError(f"single-player state arena overflowed at cycle {self.cycles}: observation rows 889-1011 would be "
                               "zero; run fewer tables per environment")
        self.nr = nr
        return nr, n_live

    def decide(self):
        import torch

        env, nr, agents, cycles, meta_rec = self.env, self.nr, self.agents, self.cycles, self.meta_rec
        if nr == 0:
            return
        with self._ctx():
            if self.host_mode:
                h_actions, h_q = self.h_actions, self.h_q
                tbl_h = env.row_table[:nr].cpu().numpy()
                rs_h = env.row_seat[:nr].cpu().numpy()
                chal_h = self.ic_host[tbl_h % self.per, rs_h & 3]
                same = agents[0] is agents[1]
                groups = ((np.arange(nr), agents[0], self.oracle[0]),) if same else (
                    (np.nonzero(chal_h)[0], agents[0], self.oracle[0]), (np.nonzero(~chal_h)[0], agents[1], self.oracle[1]))
                inv_np = None
                if self.h_inv is not None:
                    self.h_inv[:nr].copy_(env.encode_invisible(self.version)[:nr])
                    inv_np = self.h_inv.numpy()
                for k, (idx, agent, is_oracle) in enumerate(groups):
                    if idx.size == 0:
                        continue
                    obs_np = self.obs_np
                    if self.mixed:  # each agent's rows in its own layout (mortal.rs:256-287): one encode per version
                        env.set_obs_version(self.versions[k])
                        buf = self.h_obs if k == 0 else self.h_obs2
                        assert env.encode_obs_host(buf, self.h_masks) == nr
                        obs_np = buf.numpy()
                    t_eval = time.perf_counter_ns()
                    a, q, greedy = agent.react_host(obs_np, self.masks_np, idx, inv_np if is_oracle else None)
                    if meta_rec is not None:
                        meta_rec.add_agent(cycles, torch.from_numpy(idx), torch.from_numpy(q).reshape(-1, 46), time.perf_counter_ns() - t_eval, greedy)
                    h_actions[torch.from_numpy(idx)] = torch.from_numpy(a)
                    if h_q is not None:
                        h_q[torch.from_numpy(idx)] = torch.from_numpy(q).reshape(-1, 46)
                if meta_rec is not None:
                    meta_rec.add_rows(cycles, torch.from_numpy(tbl_h).long(), torch.from_numpy(rs_h), h_actions[:nr], self.h_masks[:nr], self.h_obs[:nr])
                self.actions[:nr].copy_(h_actions[:nr], non_blocking=True)
                if h_q is not None:
                    self.q_all[:nr].copy_(h_q[:nr], non_blocking=True)
                if self.arena.record_decisions:
                    self.recorded.append(torch.stack([torch.from_numpy(tbl_h).long() + self.offset, env.row_step[:nr].cpu().long(),
                                                      torch.from_numpy(rs_h & 3).long(), torch.from_numpy((rs_h >> 2) & 1).long(),
                                                      h_actions[:nr].clone()], dim=1))
                    self.recorded_masks.append((self.h_masks[:nr].long() * self.mask_weights).sum(1))
                return
            if self.adopted:
                obs = self._decide_adopted(nr, cycles, meta_rec)
                if meta_rec is not None or self.arena.record_decisions:
                    self._record(cycles, nr, env.row_table[:nr].long(), (env.row_seat[:nr] & 3).long(), env.masks[:nr], obs[:nr])
                return
            obs_buf = env.encode_obs()
            obs, masks = obs_buf[:nr], env.masks[:nr]
            tbl = env.row_table[:nr].long()
            seat = (env.row_seat[:nr] & 3).long()
            inv = env.encode_invisible(self.version)[:nr] if any(self.oracle) else None
            if agents[0] is agents[1]:  # one engine for every seat: no gather of the rows, CUDA-graph replay when the engine has one
                agent = agents[0]
                t_eval = time.perf_counter_ns()
                greedy = None
                if hasattr(agent, "react_static") and not meta_rec and not self.oracle[0]:
                    a, q = agent.react_static(obs_buf, env.masks, nr)
                else:
                    out = agent.react_device(obs, masks, invisible_obs=inv) if self.oracle[0] else agent.react_device(obs, masks)
                    a, q = out[0], out[1]
                self.actions[:nr] = a.to(torch.int64)
                if self.q_all is not None:
                    self.q_all[:nr] = q.float()
                if meta_rec is not None:
                    meta_rec.add_agent(cycles, torch.arange(nr), q, time.perf_counter_ns() - t_eval, greedy)
            else:
                chal = self.is_challenger[tbl % self.per, seat]
                for k, (idx, agent, is_oracle) in enumerate(((chal.nonzero().squeeze(1), agents[0], self.oracle[0]),
                                                             ((~chal).nonzero().squeeze(1), agents[1], self.oracle[1]))):
                    if idx.numel() == 0:
                        continue
                    if self.mixed and k == 1:  # the champion's rows in its own layout (mortal.rs:256-287)
                        env.set_obs_version(self.versions[1])
                        obs = env.encode_obs()[:nr]
                        env.set_obs_version(self.versions[0])
                    t_eval = time.perf_counter_ns()
                    out = agent.react_device(obs[idx], masks[idx], invisible_obs=inv[idx]) if is_oracle else agent.react_device(obs[idx], masks[idx])
                    a, q = out[0], out[1]
                    self.actions[idx] = a.to(torch.int64)
                    if self.q_all is not None:
                        self.q_all[idx] = q.float()
                    if meta_rec is not None:
                        meta_rec.add_agent(cycles, idx, q, time.perf_counter_ns() - t_eval)
            self._record(cycles, nr, tbl, seat, masks, obs)

    def _decide_adopted(self, nr, cycles, meta_rec):
        """ReferenceEngine agents: encode each obs version into its persistent buffer, split the rows per agent on the device (one
        small read-back of the two counts), replay each engine's graph; the select kernel writes actions / Q / greedy in place."""
        import torch

        env, agents = self.env, self.agents
        for v in (self.versions if self.mixed else self.versions[:1]):
            if self.mixed:
                env.set_obs_version(v)
            env.encode_obs(out=self.obs_bufs[v])
        if self.mixed:
            env.set_obs_version(self.versions[0])
        if agents[0] is agents[1]:
            jobs = [(agents[0], None, env.n_rows_dev, nr, self.versions[0])]
        else:
            from .. import nn_ops

            nn_ops.split_rows(env.row_table, env.row_seat, env.n_rows_dev, self.agent_of, self.split[0], self.split[1], self.counts)
            counts = self.counts.tolist()
            jobs = [(agents[k], self.split[k], self.counts[k:k + 1], counts[k], self.versions[k]) for k in range(2) if counts[k]]
        for agent, rows, count, n, version in jobs:
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) if meta_rec is not None else None
            if ev:
                ev[0].record()
            agent.decide(self.obs_bufs[version], env, rows, count, n, table_offset=self.offset, actions=self.actions, q_out=self.q_dev,
                         greedy=self.greedy)
            if ev:
                ev[1].record()
                idx = torch.arange(n, device=self.dev) if rows is None else rows[:n].long()
                meta_rec.add_agent(cycles, idx, self.q_dev[idx], ev, self.greedy[idx])
        return self.obs_bufs[self.versions[0]]

    def _record(self, cycles, nr, tbl, seat, masks, obs):
        import torch

        env, meta_rec = self.env, self.meta_rec
        if meta_rec is not None:
            meta_rec.add_rows(cycles, tbl, env.row_seat[:nr], self.actions[:nr], masks, obs)
        if self.arena.record_decisions:
            self.recorded.append(torch.stack([tbl + self.offset, env.row_step[:nr].long(), seat, (env.row_seat[:nr] >> 2).long() & 1,
                                              self.actions[:nr]], dim=1).cpu())
            self.recorded_masks.append((masks.long() * self.mask_weights.to(self.dev)).sum(1).cpu())


class _RunState:
    """What a cycle_hook sees."""

    def __init__(self, parts):
        self.parts = parts

    def total_steps(self):
        return sum(p.env.total_steps() for p in self.parts)

    def synchronize(self):
        for p in self.parts:
            if p.stream is not None:
                p.stream.synchronize()


class _Arena:
    SEATS_PER_SEED = 4
    adopt_reference_engines = False  # play eligible MortalEngines on the device path (ReferenceEngine); libriichi.install() sets it

    def __init__(self, *, disable_progress_bar: bool = False, log_dir=None, shuffle_kind: int = 0, device: int = 0):
        self.disable_progress_bar = disable_progress_bar
        self.shuffle_kind = shuffle_kind
        self.device = device
        self.last_stats = None
        self.record_decisions = False  # test hook: keep (table, step, seat, kan_select, action) of every row
        self.last_decisions = None
        self.log_dir = log_dir  # arena/one_vs_three.rs:26-34: gz mjai logs are written here when set
        self.log_meta = True    # attach the per-decision meta (q-values, mask bits, ...) to the agent events (mortal.rs:161-186)
        self.last_meta_error = None
        self.record_grp = False  # keep the per-kyoku GRP features of every game (read on device, no logs): last_grp
        self.last_grp = None
        self.pipeline = True    # play the batch as two half-batches stepped alternately (see the module docstring)
        self.pipeline_device_engines = False  # the same for device engines (env kernels of one half under the other half's forward)
        self.max_cycles = 0     # test hook: stop after this many BatchGame::run cycles (0 = play every table to the end)
        self.fast_forward_steps = 0  # bench hook: play this many batch steps with the counter-free test policy (kind 2) first
        self.cycle_hook = None       # bench hook: callable(cycle_index, run_state) when the first part starts a cycle
        self.env_factory = BatchEnv  # test hook: tests/emul_batch_env.py injects the host-emulated environment; the product has no CPU path
        self.last_decision_masks = None  # with record_decisions: the legal mask (46 bits) each recorded row was decided under

    def _challenger_seats(self, game_in_seed: int):
        raise NotImplementedError

    def _adapt(self, engine):
        if hasattr(engine, "react_device"):
            return engine
        if self.adopt_reference_engines and ReferenceEngine.eligible(engine, self.device):
            return ReferenceEngine(engine)
        return HostProtocolEngine(engine)

    def _run(self, challenger, champion, seed_start, seed_count):
        import torch

        if challenger is champion:
            agents = [self._adapt(challenger)] * 2
        else:
            agents = [self._adapt(challenger), self._adapt(champion)]
        if not all(isinstance(a, ReferenceEngine) for a in agents):  # adoption covers both agents or neither
            agents = [HostProtocolEngine(a.engine) if isinstance(a, ReferenceEngine) else a for a in agents]
        for a in {id(a): a for a in agents}.values():
            if isinstance(a, ReferenceEngine):
                a.refresh()
        self.last_agents = agents
        for a in agents:
            if getattr(a, "version", 4) not in (1, 2, 3, 4):
                raise ValueError(f"unsupported obs version {a.version} (consts.rs:18 MAX_VERSION = 4)")
        versions = [int(getattr(a, "version", 4)) for a in agents]
        qe = [bool(getattr(a, "enable_quick_eval", True)) for a in agents]
        per = self.GAMES_PER_SEED
        seed_count = int(seed_count)
        n = seed_count * per
        nonces = np.repeat(np.arange(seed_start[0], seed_start[0] + seed_count, dtype=np.uint64), per)
        keys = np.full(n, seed_start[1], dtype=np.uint64)
        # the seat rotations of a seed stay together; two parts when there is something to overlap: host-side engines (their
        # numpy / list work and the D2H copies of the other half). Device engines already keep the GPU busy back to back — two
        # half-size forward passes on two streams measured slower than one full-size pass (profiles/r02_summary.md).
        cuts = [0, n]
        host_engines = all(isinstance(a, HostProtocolEngine) for a in agents)
        if self.pipeline and (host_engines or self.pipeline_device_engines) and seed_count >= 2:
            cuts = [0, (seed_count // 2) * per, n]
        parts = []
        try:
            for lo, hi in zip(cuts[:-1], cuts[1:]):
                parts.append(_Part(self, agents, nonces[lo:hi], keys[lo:hi], lo, per, self._challenger_seats, versions, qe,
                                   use_stream=len(cuts) > 2))
            state = _RunState(parts)
            for p in parts:
                p.start(self.fast_forward_steps)
            live = list(parts)
            while live:
                for p in list(live):
                    if p is parts[0] and self.cycle_hook is not None:
                        self.cycle_hook(p.cycles, state)
                    if self.max_cycles and p.cycles >= self.max_cycles:
                        live.remove(p)
                        continue
                    nr, n_live = p.finish()
                    if nr == 0 and n_live == 0:
                        live.remove(p)
                        continue
                    p.decide()
                    p.cycles += 1
                    if self.max_cycles and p.cycles >= self.max_cycles:
                        continue  # the decisions of the last cycle are computed but not applied (oracle replay cuts there too)
                    p.begin()
            state.synchronize()
            results = [p.env.results() for p in parts]
            res = {k: np.concatenate([r[k] for r in results]) for k in results[0]}
            if self.log_dir is not None:  # one_vs_three.rs:195-225: one {seed}_{key}_{split}.json.gz per game
                from .. import mjai_log

                agent_names = [str(getattr(a, "name", "NoName")) for a in agents]
                self.last_log_paths = []
                for p in parts:
                    words, lens = p.env.read_log()
                    names = [[agent_names[0] if p.ic_host[g % per, seat] else agent_names[1] for seat in range(4)] for g in range(p.n)]
                    seeds = [(int(p.nonces[g]), int(p.keys[g])) for g in range(p.n)]
                    bounds = decisions = None
                    if p.meta_rec is not None:
                        try:
                            bounds, decisions = p.meta_rec.finish()
                        except Exception as exc:  # the logs themselves must not depend on the optional metadata
                            self.last_meta_error = exc
                            bounds = decisions = None
                    self.last_log_paths += mjai_log.write_logs(self.log_dir, words, lens, seeds, names, "abcd"[:per], bounds, decisions)
            if self.record_grp:  # dataset/grp.rs:90-164 straight from the table records: what reward_calculator.py:13-38 consumes
                from ..dataset import Grp

                feats = [f for p in parts for f in p.env.read_grp()]
                self.last_grp = [Grp(feats[g], [int(x) for x in res["ranks"][g]], [int(x) for x in res["scores"][g]]) for g in range(n)]
            sp_overflows = sum(p.env.sp_overflows() for p in parts)
            self.last_stats = dict(cycles=max(p.cycles for p in parts), table_steps=int(res["steps"].sum()), sp_overflows=sp_overflows,
                                   parts=len(parts), launches=sum(p.env.launch_count() for p in parts if hasattr(p.env, "launch_count")))
            self.last_results = res
            if self.record_decisions:
                rec = [x for p in parts for x in p.recorded]
                recm = [x for p in parts for x in p.recorded_masks]
                self.last_decisions = torch.cat(rec).numpy() if rec else np.zeros((0, 5), dtype=np.int64)
                self.last_decision_masks = torch.cat(recm).numpy() if recm else np.zeros(0, dtype=np.int64)
        finally:
            for p in parts:
                p.env.close()
        if sp_overflows:
            raise RuntimeError("single-player state arena overflowed during the run: observation rows 889-1011 were zero in "
                               f"{sp_overflows} step(s)")
        if (res["err"] != 0).any():
            bad = int(np.nonzero(res["err"])[0][0])
            raise RuntimeError(f"table {bad} failed with mjx error code {int(res['err'][bad])}")
        return res

    def ako_vs_py(self, *a, **k):
        raise NotImplementedError("akochan subprocess agents are out of scope (SURVEY.md §2.1 row 5)")

    py_vs_ako = ako_vs_py


class OneVsThree(_Arena):
    GAMES_PER_SEED = 4

    def _challenger_seats(self, g):
        return [g % 4]

    def py_vs_py(self, challenger, champion, seed_start, seed_count):
        res = self._run(challenger, champion, seed_start, seed_count)
        rankings = [0, 0, 0, 0]
        for i in range(res["ranks"].shape[0]):  # one_vs_three.rs:55-60
            rankings[int(res["ranks"][i, i % 4])] += 1
        return rankings


class TwoVsTwo(_Arena):
    GAMES_PER_SEED = 2

    def _challenger_seats(self, g):
        return [0, 2] if g % 2 == 0 else [1, 3]  # two_vs_two.rs:137-191

    def py_vs_py(self, challenger, champion, seed_start, seed_count):
        self._run(challenger, champion, seed_start, seed_count)
        return None
