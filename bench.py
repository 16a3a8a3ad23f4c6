#!/usr/bin/env python
"""Benchmark: table-steps/sec of batched riichi self-play (BASELINE.json metric).

A "step" = one iteration of libriichi's BatchGame::run loop (arena/game.rs:286-304) over the whole batch:
commit the previous decisions, poll every live table to its next decision point, encode one v4
observation per decision row, run the policy. One table-step = that iteration for one live table.

Default arm (this repo): 4096 tables per GPU (BASELINE configs[1]), random-init Mortal brain
(192 channels x 40 blocks, bf16 autocast, greedy), everything resident in HBM. JSON also carries
  env_only      the same loop with the device test policy (kind 2: a function of the legal mask and the obs planes only)
  roofline      the full v4 encode_obs (feature + store + single-player kernels): algorithmic bytes / CUDA-event time;
                .kernels holds k_encode_store alone and the encoder pair
  e2e           libriichi.arena.OneVsThree.py_vs_py with a react_batch engine over lists of HOST numpy arrays (the plugin call)
  e2e_with_net  the same through DeviceEngine.react_batch (np.stack -> H2D -> 192x40 net -> lists), i.e. the `value` workload
  shanten_1m / agari_1m / encode_65536   BASELINE configs[2] and [3]
  cpu_baseline  the CPU oracle on this box's host cores, bounded sample (rank 0, N=1 only)
`--impl reference` times libriichi's own CPU path restated by the oracle (oracle/, all host threads): the same 4096 tables, the
same policy (kind 2) and therefore the same games as `env_only` and `e2e`.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (it may be read-only)

N_TABLES = 4096
DUMP_OBS_ROWS = 256  # --dump-outputs: observation rows kept (256 x 137,632 B = 35 MB)
SEED_START = (10000, 0x2000)  # mortal/player.py:67
OBS_BYTES = 1012 * 34 * 4
MASK_BYTES = 46
STATE_BYTES = 1952  # sizeof(TableState) read per encoded row


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.samples = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def seeds_for_rank(rank: int, n_tables: int):
    import numpy as np

    count = n_tables // 4
    start = SEED_START[0] + count * rank  # SURVEY.md §8(d) config 5: rank r takes seed_start + 1024 r
    nonces = np.repeat(np.arange(start, start + count, dtype=np.uint64), 4)
    keys = np.full(n_tables, SEED_START[1], dtype=np.uint64)
    return nonces, keys


# ---------------------------------------------------------------------------------------------- reference arm
def cpu_arm(args, n_warm, n_timed):
    """libriichi's CPU path (oracle restatement; the Rust crate cannot be built here): poll/commit loop + one v4 obs encode
    (incl. the single-player tables) per decision row, all host threads, the full 4096-table batch kept alive across steps.
    One step = every live table advances one table-step (BatchGame::run's loop body). The fast-forward is outside the clock."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O

    cores = host_cores()
    nonces, keys = seeds_for_rank(0, N_TABLES)
    batch = O.Batch(nonces, keys, shuffle_kind=0, policy_kind=2, quick_eval=True, encode_obs=4, sp_mode=1, n_threads=cores)
    batch.run(args.skip, encode_from=args.skip)  # untimed, nothing encoded
    at = args.skip
    for _ in range(n_warm):
        at += 1
        batch.run(at, encode_from=args.skip)
    per_step = []
    for _ in range(n_timed):
        at += 1
        ts, rows, sec = batch.run(at, encode_from=args.skip)
        per_step.append((ts, rows, sec))
    batch.close()
    tot_steps = sum(p[0] for p in per_step)
    tot_sec = sum(p[2] for p in per_step)
    thirds = [per_step[i * len(per_step) // 3:(i + 1) * len(per_step) // 3] for i in range(3)]
    rates = sorted(sum(p[0] for p in t) / max(sum(p[2] for p in t), 1e-9) for t in thirds if t)
    sample = (f"{N_TABLES} tables (seeds {SEED_START[0]}.., the GPU arm's), table-steps {at - n_timed}..{at} of every table "
              f"({tot_steps} table-steps, {sum(p[1] for p in per_step)} rows), policy kind 2, v4 obs + SP encode per decision, "
              f"{tot_sec:.1f} s timed after an untimed {args.skip}-step fast-forward")
    return {"value": tot_steps / tot_sec, "unit": "table-steps/s", "cores": cores, "kind": "port", "sample": sample,
            "thirds_min_median_max": rates, "seconds": tot_sec, "table_steps": tot_steps}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = cpu_arm(args, args.warmup, args.steps)
    value = cb["value"]
    line = {
        "impl": "reference", "metric": "table-steps/sec batched self-play", "value": value, "unit": "table-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * cb["seconds"] / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/i32 (+f32 SP)", "data": "synthetic",
        "config": workload_config(1, args),
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "thirds_min_median_max")},
        "e2e": {"value": value, "unit": "table-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(world, args):
    return {"workload": "BatchGame 4096 tables/GPU, random-init Mortal brain (192ch x 40 blocks, v4 obs), self-play step loop (BASELINE configs[1])",
            "tables_per_gpu": N_TABLES, "global_tables": N_TABLES * world, "obs_version": 4,
            "seed_start": list(SEED_START), "fast_forward_steps": args.skip, "parallelism": f"tables sharded dp{world}, no data-path collective",
            "l2": "per-step obs output (~0.56 GB) exceeds the 126 MB L2, no explicit flush",
            "sp_block": "rows 889-1011 (single-player tables) computed on device by the k_sp_* kernels"}


# ---------------------------------------------------------------------------------------------- this repo's arm
def pin_to_gpu_numa(local_rank):
    """Multi-rank runs: keep this rank's threads (and therefore its first-touched pinned buffers) on the NUMA node its GPU
    hangs off, so that 8 ranks draining ~0.55 GB of observations per step do not all cross the socket link."""
    try:
        import torch

        p = torch.cuda.get_device_properties(local_rank)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        return None
    return None


def splitmix64_np(x):
    import numpy as np

    with np.errstate(over="ignore"):
        x = x + np.uint64(0x9E3779B97F4A7C15)
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return x ^ (x >> np.uint64(31))


class MaskHashEngine:
    """A reference-protocol engine (agent/mortal.rs:54-74, 126-152: react_batch over LISTS of numpy arrays, lists out) that
    plays the test policy kind 2 (oracle/board.cc test_policy, csrc/mjx_policy.cuh) from what it is handed: the legal mask and
    the v4 observation planes 870 (kan-select), 875 / 876 (keep / next-shanten discards). Same decisions as the CPU arm."""

    engine_type = "mortal"
    name = "maskhash"
    version = 4
    is_oracle = False
    enable_quick_eval = True
    enable_rule_based_agari_guard = False

    def __init__(self):
        self.rows = 0
        self.calls = 0

    @staticmethod
    def _kth(cand, k):
        import numpy as np

        cs = np.cumsum(cand, axis=1)
        return np.argmax((cs == (k[:, None] + 1)) & cand, axis=1)

    def react_batch(self, obs, masks, invisible_obs):
        import numpy as np

        n = len(obs)
        self.rows += n
        self.calls += 1
        m = np.stack(masks).astype(bool)
        bits = (m.astype(np.uint64) << np.arange(46, dtype=np.uint64)).sum(axis=1)
        sel = np.stack([o[870:877] for o in obs])  # one pass over the list: planes 870 (kan-select) .. 876
        kan = sel[:, 0, 0] > 0
        keep = sel[:, 5] > 0
        nxt = sel[:, 6] > 0
        h = splitmix64_np(bits)
        h2 = splitmix64_np(h)
        h3 = splitmix64_np(h2)
        act = np.full(n, -1, dtype=np.int64)
        one = np.uint64(1)
        # kan-select rows: uniform over the mask by the hash
        popc = m.sum(axis=1).astype(np.uint64)
        if kan.any():
            act[kan] = self._kth(m[kan], (h[kan] % popc[kan]).astype(np.int64))
        todo = act < 0
        sel = todo & m[:, 43]
        act[sel] = 43
        todo &= ~sel
        sel = todo & m[:, 37] & ((h2 & np.uint64(3)) != 0)
        act[sel] = 37
        todo &= ~sel
        disc = m[:, :37]
        other = m.copy()
        other[:, :38] = False
        n_disc = disc.sum(axis=1)
        n_other = other.sum(axis=1).astype(np.uint64)
        sel = todo & (n_other > 0) & ((n_disc == 0) | ((h3 & one) != 0))
        if sel.any():
            act[sel] = self._kth(other[sel], ((h3[sel] >> one) % n_other[sel]).astype(np.int64))
        todo &= ~sel
        if todo.any():
            aka = np.array([4, 13, 22])
            d = disc[todo]
            pref = d & np.concatenate([nxt[todo], nxt[todo][:, aka]], axis=1)
            none = ~pref.any(axis=1)
            pk = d & np.concatenate([keep[todo], keep[todo][:, aka]], axis=1)
            pref[none] = pk[none]
            none = ~pref.any(axis=1)
            pref[none] = d[none]
            cnt = pref.sum(axis=1).astype(np.uint64)
            act[todo] = self._kth(pref, ((h3[todo] >> one) % cnt).astype(np.int64))
        q = np.where(m, np.float32(0.0), np.float32(-np.inf))
        # sequences of the protocol's shapes (B, Bx46, Bx46, B); numpy arrays spare both sides the list round trip
        return act, q, m, np.ones(n, dtype=bool)


class HostNetEngine:
    """The `value` workload behind the reference protocol: lists of host arrays in, np.stack -> H2D -> 192x40 net -> lists out
    (what mortal/engine.py:43-81 does with the observations libriichi hands it)."""

    engine_type = "mortal"
    name = "hostnet"
    version = 4
    is_oracle = False
    enable_quick_eval = True
    enable_rule_based_agari_guard = False

    def __init__(self, device_engine):
        self.e = device_engine
        self.rows = 0

    def react_batch(self, obs, masks, invisible_obs):
        self.rows += len(obs)
        return self.e.react_batch(obs, masks, invisible_obs)


class LastStepRecorder:
    """The DeviceEngine as the arena drives it, plus a device copy of one cycle's exchange: the rows the engine is handed
    (observations, legal masks, and the rows' table / seat from the environment) and the actions and Q-values it returns.
    Armed for the last timed cycle by the bench's cycle hook (--dump-outputs)."""

    def __init__(self, engine):
        self.e = engine
        for attr in ("engine_type", "name", "version", "is_oracle", "enable_quick_eval", "enable_rule_based_agari_guard"):
            setattr(self, attr, getattr(engine, attr))
        self.env = None
        self.last = None

    def react_device(self, obs, masks, invisible_obs=None):
        return self.e.react_device(obs, masks)

    def react_static(self, obs_buf, masks_buf, nr):
        a, q = self.e.react_static(obs_buf, masks_buf, nr)
        if self.env is not None:
            self.last = dict(obs=obs_buf[:nr].clone(), masks=masks_buf[:nr].clone(), actions=a.clone(), q_values=q.clone(),
                             row_table=self.env.row_table[:nr].clone(), row_seat=self.env.row_seat[:nr].clone())
            self.env = None
        return a, q


def dump_outputs(out_dir, last):
    """Write one recorded cycle as DIR/<name>.npy (float32 / float64). Rows are sorted by (table, seat byte): the environment
    appends decision rows through an atomic counter, so their order differs from run to run while their content does not.
    The observations are a fixed seeded sample of DUMP_OBS_ROWS of the sorted rows (obs_sample_rows: their positions).
    The engine returns -inf as the Q-value of an illegal action; q_values holds 0 there (masks says which entries are legal),
    so every written value is finite and a non-finite one is an error."""
    import numpy as np
    import torch

    if last is None:
        raise SystemExit("bench.py --dump-outputs: the last timed step had no decision rows to record")
    order = torch.argsort(last["row_table"].long() * 8 + last["row_seat"].long())
    n = int(order.numel())
    pick = np.sort(np.random.default_rng(0).choice(n, min(n, DUMP_OBS_ROWS), replace=False))
    arrays = {
        "row_table": last["row_table"][order].double(),
        "row_seat": last["row_seat"][order].double(),  # seat | 4 on kan-select rows
        "masks": last["masks"][order].float(),
        "actions": last["actions"][order].double(),
        "q_values": last["q_values"][order].float().masked_fill(~last["masks"][order], 0.0),
        "obs_sample": last["obs"][order[torch.from_numpy(pick).to(order.device)]].float(),
        "obs_sample_rows": torch.from_numpy(pick).double(),
    }
    for name, t in arrays.items():
        if not bool(torch.isfinite(t).all()):
            raise SystemExit(f"bench.py --dump-outputs: {name} of the last timed step holds a non-finite value")
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; mortal_b200 has no CPU path")
    numa_node = pin_to_gpu_numa(local_rank) if world > 1 else None
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import mortal_b200
    from mortal_b200.engine import DeviceEngine
    from mortal_b200.libriichi.arena import OneVsThree
    from mortal_b200.model import DQN, Brain

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    nonces, keys = seeds_for_rank(rank, N_TABLES)
    torch.manual_seed(0)
    engine = DeviceEngine(Brain(conv_channels=192, num_blocks=40, version=4), DQN(version=4), device=dev,
                          enable_amp=True, enable_quick_eval=True)

    def fresh_env():
        """A new batch, fast-forwarded (untimed, test policy kind 2, no encode) by --skip batch steps so that the timed
        steps see the steady-state mix of early/late kyoku positions instead of 4096 freshly dealt hands."""
        env = mortal_b200.BatchEnv(nonces, keys, obs_version=4, shuffle_kind=0, enable_quick_eval=True, device=local_rank)
        actions = torch.zeros(env.row_cap, dtype=torch.int64, device=dev)
        env.step(None)
        env.policy_test(2, actions)
        for _ in range(args.skip):
            env.step(actions)
            env.policy_test(2, actions)
        return env, actions

    W, K = args.warmup, args.steps

    def loop(env_actions, policy, n_warm, n_timed, time_encode=False, split_events=None):
        env, actions = env_actions
        obs = env.obs_buffer()
        enc_events = []

        def cycle(timed):
            if timed and split_events is not None:  # where the step goes: env kernels vs policy (events only, no sync)
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                ev[0].record()
                env.step(actions)
                env.encode_obs(obs)
                ev[1].record()
                r = policy(env, obs, actions)
                ev[2].record()
                split_events.append(ev)
                return r
            env.step(actions)
            if timed and time_encode:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                env.encode_obs(obs)
                e1.record()
                enc_events.append((e0, e1))
            else:
                env.encode_obs(obs)
            return policy(env, obs, actions)

        for _ in range(n_warm):
            cycle(False)
        barrier()
        steps0, rows, l0 = env.total_steps(), 0, env.launch_count()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(n_timed):
            rows += cycle(True)
        t1.record()
        barrier()
        ms = t0.elapsed_time(t1)
        steps = env.total_steps() - steps0
        enc_ms = sum(a.elapsed_time(b) for a, b in enc_events)
        return dict(ms=ms, table_steps=steps, rows=rows, enc_ms=enc_ms, n=n_timed, launches=env.launch_count() - l0)

    def nn_policy(env, obs, actions):
        nr = env.num_rows()  # the only host sync of the cycle: the batch size the network runs at
        if nr:
            a, _ = engine.react_static(obs, env.masks, nr)  # CUDA-graph replay over the env's persistent buffers
            actions[:nr] = a
        return nr

    def test_policy(env, obs, actions):
        env.policy_test(2, actions)
        return 0

    # -------- the product path: libriichi.arena.OneVsThree.py_vs_py (for host-protocol engines two half-batches stepped alternately:
    # kernels + D2H of one half overlap the engine's host work on the other), timed between two cycle hooks
    def run_arena(agent, n_warm, n_timed, pipeline=True):
        arena = OneVsThree(disable_progress_bar=True, device=local_rank)
        arena.pipeline = pipeline
        arena.fast_forward_steps = args.skip
        arena.max_cycles = n_warm + n_timed + 1  # the hook of cycle n_warm + n_timed must fire
        marks = {}
        rows = lambda: getattr(agent, "rows", 0)

        def hook(c, state):
            if c in (n_warm, n_warm + n_timed):
                torch.cuda.synchronize()
                marks[c] = (time.perf_counter(), state.total_steps(), rows())
            if c == n_warm + n_timed - 1 and isinstance(agent, LastStepRecorder):
                agent.env = state.parts[0].env

        arena.cycle_hook = hook
        # same tables as the other loops: rank r starts at seed_start + 1024 r
        arena.py_vs_py(agent, agent, (int(nonces[0]), int(keys[0])), N_TABLES // 4)
        (t0, s0, r0), (t1, s1, r1) = marks[n_warm], marks[n_warm + n_timed]
        return dict(ms=(t1 - t0) * 1000.0, table_steps=s1 - s0, rows=r1 - r0, n=n_timed, launches=arena.last_stats["launches"],
                    cycles=arena.last_stats["cycles"])

    run_e2e = run_arena

    # -------- loop A: with the network (the BASELINE config), HBM resident
    sampler = ClockSampler(local_rank)
    sampler.start()
    ea = fresh_env()
    a_split = []
    a = loop(ea, nn_policy, W, K, split_events=a_split)
    a_env_ms = sum(e[0].elapsed_time(e[1]) for e in a_split) / K
    a_nn_ms = sum(e[1].elapsed_time(e[2]) for e in a_split) / K
    ea[0].close()
    barrier()
    recorder = LastStepRecorder(engine) if args.dump_outputs else None
    av = run_arena(recorder or engine, W, K)  # the headline `value`: the same workload through the arena (pipelined half-batches)
    barrier()
    clocks = sampler.stop()
    if recorder is not None and rank == 0:
        dump_outputs(args.dump_outputs, recorder.last)
        recorder.last = None

    # -------- loop B: env only (test policy on device, no host sync); B2 = the same with the single-player block off
    ea = fresh_env()
    b = loop(ea, test_policy, W, K)
    sp_overflows = ea[0].sp_overflows()
    sp_states, sp_edges, sp_levels = ea[0].sp_stats()  # size of the last step's single-player DP
    ea[0].close()
    ea = fresh_env()
    ea[0].set_sp(False)
    b2 = loop(ea, test_policy, W, K)
    ea[0].close()
    # -------- the encode alone, the same deterministic K cycles again: whole encode_obs (feature + store + single-player kernels)
    # bracketed by CUDA events on the launch stream, the two encoder kernels by events inside libmjx; row count read each step
    # (a sync per step, so this pass is not the one `env_only` is quoted from)
    env, actions = fresh_env()
    env.set_encode_timing(True)
    obs_t = env.obs_buffer()
    b_rows, feat_ms, store_ms, full_ms = 0, 0.0, 0.0, 0.0
    for i in range(W + K):
        env.step(actions)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        env.encode_obs(obs_t)
        e1.record()
        env.policy_test(2, actions)
        nr_i = env.num_rows()
        if i >= W:
            b_rows += nr_i
            f_ms, s_ms = env.last_encode_ms()
            feat_ms += f_ms
            store_ms += s_ms
            full_ms += e0.elapsed_time(e1)
    env.close()

    extras = {}
    if world == 1 and rank == 0:
        if not args.no_encode_64k:
            extras["encode_65536"] = bench_encode_64k(mortal_b200, torch, np, dev, local_rank)
        if not args.no_algo_1m:
            extras.update(bench_algo_1m(torch, np, dev, args))

    barrier()
    c = run_e2e(MaskHashEngine(), W, K)
    barrier()
    cn = None
    if not args.no_e2e_net:
        kn = max(3, min(K, args.e2e_net_steps))
        cn = run_e2e(HostNetEngine(engine), max(W, 4), kn)
        barrier()
    # what the link gives for the same bytes: one plain pinned D2H copy (context for e2e, not a claim)
    nprobe = max(1, c["rows"] // K)
    dsrc = torch.empty((nprobe, 1012, 34), dtype=torch.float32, device=dev)
    hdst = torch.empty((nprobe, 1012, 34), dtype=torch.float32, pin_memory=True)
    hdst.copy_(dsrc, non_blocking=True)
    torch.cuda.synchronize()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    hdst.copy_(dsrc, non_blocking=True)
    p1.record()
    torch.cuda.synchronize()
    pcie_gbs = nprobe * OBS_BYTES / (p0.elapsed_time(p1) * 1e-3) / 1e9
    del dsrc, hdst

    # -------- reduce over ranks: max time, sum of units
    def reduce(ms, units):
        if world == 1:
            return ms, units
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        u = torch.tensor([units], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(u, op=dist.ReduceOp.SUM)
        return float(t.item()), float(u.item())

    a_ms, a_units = reduce(a["ms"], a["table_steps"])
    av_ms, av_units = reduce(av["ms"], av["table_steps"])
    b_ms, b_units = reduce(b["ms"], b["table_steps"])
    c_ms, c_units = reduce(c["ms"], c["table_steps"])
    cn_ms, cn_units = reduce(cn["ms"], cn["table_steps"]) if cn else (None, None)

    # -------- the one collective of the path: all-gather of end-of-hanchan returns (SURVEY.md §8e), on REAL returns:
    # every rank plays a small shard of hanchans to the end, the returns are gathered and rank 0 checks them all against the oracle
    collective = {"bytes_per_table": 20}
    if world > 1:
        from mortal_b200 import dist as mdist

        n_small = 256
        sn, sk = mdist.shard_seeds((SEED_START[0] + 100000, SEED_START[1]), n_small // 4, rank)
        env = mortal_b200.BatchEnv(sn, sk, device=local_rank)
        res = env.run_test_policy(kind=2)
        env.close()
        mdist.gather_returns(res["scores"], res["ranks"], device=dev)  # warm-up (NCCL channel setup)
        torch.cuda.synchronize()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        g_scores, g_ranks = mdist.gather_returns(res["scores"], res["ranks"], device=dev)
        g1.record()
        torch.cuda.synchronize()
        collective.update(all_gather_us=g0.elapsed_time(g1) * 1000.0, tables_gathered=int(g_scores.shape[0]))
        if rank == 0:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle_lib as O

            all_n = np.concatenate([mdist.shard_seeds((SEED_START[0] + 100000, SEED_START[1]), n_small // 4, r)[0] for r in range(world)])
            ref = O.run_batch(all_n, np.full(len(all_n), SEED_START[1], dtype=np.uint64), policy_kind=2, n_threads=min(32, host_cores()))
            collective["returns_equal_oracle"] = bool((ref["scores"] == g_scores).all() and (ref["ranks"] == g_ranks).all())

    if rank == 0:
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except Exception:
            pass
        peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
        traffic = {}
        try:  # dram__bytes_read + dram__bytes_write per launch, from the committed ncu --set full summaries
            with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
                traffic = json.load(f)
        except Exception:
            pass
        rows_per_launch = b_rows / K
        bytes_per_launch = rows_per_launch * (OBS_BYTES + MASK_BYTES + STATE_BYTES)
        gbs = lambda ms: bytes_per_launch / (ms / K * 1e-3) / 1e9 if ms > 0 else 0.0
        line = {
            "metric": "table-steps/sec batched self-play", "value": av_units / (av_ms * 1e-3), "unit": "table-steps/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": av_ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8/i32 env + bf16 policy net", "data": "synthetic",
            "config": dict(workload_config(world, args), sp_arena_overflows=sp_overflows, numa_node=numa_node),
            # the timed step split with CUDA events (rank 0): env kernels (k_step + encode + single-player block, whose cost
            # depends on the positions the policy steers the tables into) and the policy network incl. the row-count sync
            "step_breakdown_ms": {"env": a_env_ms, "policy_net": a_nn_ms, "sequential_total": a_ms / K, "pipelined_total": av_ms / K,
                                  "note": "`value` runs OneVsThree.py_vs_py with the DeviceEngine for all seats (one batch, one stream, CUDA-graph "
                                          "forward); env / policy_net split the same workload driven by bench.py's own loop (CUDA events), whose "
                                          "throughput is value_sequential. Two half-batches on two streams were measured SLOWER for device engines "
                                          "(208 K vs 252 K table-steps/s): the arena pipelines half-batches for host-protocol engines only (e2e)"},
            "value_sequential": a_units / (a_ms * 1e-3),
            "env_only": {"value": b_units / (b_ms * 1e-3), "unit": "table-steps/s", "ms_per_step": b_ms / K,
                         "policy": "device test policy kind 2 (mask-hash; the CPU arm's and the e2e engine's policy), no host sync",
                         "without_sp_block": {"value": b2["table_steps"] / (b2["ms"] * 1e-3), "ms_per_step": b2["ms"] / K}},
            # The unit SURVEY.md §8(d) defines is one acting seat's v4 observation: 137,632 B obs + 46 B mask written, 1952 B record
            # read = 139,630 B. libriichi's encode_obs includes the single-player tables (agent_helper.rs:509-593, rows 889-1011),
            # so the roofline of the path is rows x 139,630 B over the time of ALL encode kernels of the step (feature + store +
            # single-player DP), measured with CUDA events around mjx_env_encode_obs. `kernels` holds the HBM-bound store kernel
            # alone and the encoder pair without the single-player DP.
            "roofline": {"kernel": "v4 encode_obs: k_encode_features + k_encode_store + k_sp_* (single-player tables)", "bound": "hbm",
                         "achieved": gbs(full_ms), "peak": peak_gbs, "unit": "GB/s", "frac": gbs(full_ms) / peak_gbs,
                         "traffic": traffic.get("encode_full"), "peak_source": peak_src, "bytes_per_launch": bytes_per_launch,
                         "ms_per_launch": full_ms / K, "rows_per_launch": rows_per_launch,
                         "kernels": {
                             "k_encode_store": {"ms_per_launch": store_ms / K, "achieved": gbs(store_ms), "frac": gbs(store_ms) / peak_gbs,
                                                "traffic": traffic.get("k_encode_store")},
                             "k_encode_features": {"ms_per_launch": feat_ms / K},
                             "encoder_pair": {"ms_per_launch": (feat_ms + store_ms) / K, "achieved": gbs(feat_ms + store_ms),
                                              "frac": gbs(feat_ms + store_ms) / peak_gbs},
                             "single_player": {"ms_per_launch": (full_ms - feat_ms - store_ms) / K}}},
            # the single-player block: a graph DP (state interning + value propagation), reported as states/s beside its time.
            # ms = env_only minus the same loop with the block switched off.
            "sp_block": {"ms_per_step": (b["ms"] - b2["ms"]) / K, "states_last_step": sp_states, "edges_last_step": sp_edges,
                         "states_per_level_D3_W3_D2_W2_D1_W1_D0_W0": sp_levels,
                         "states_per_s": sp_states / max((b["ms"] - b2["ms"]) / K * 1e-3, 1e-9), "share_of_env_step": 1.0 - b2["ms"] / b["ms"]},
            "e2e": {"value": c_units / (c_ms * 1e-3), "unit": "table-steps/s", "ms_per_step": c_ms / K,
                    "h2d_bytes_per_step": 8 * int(c["rows"] / K),
                    "d2h_bytes_per_step": int(c["rows"] / K * (OBS_BYTES + MASK_BYTES)),
                    "path": "libriichi.arena.OneVsThree.py_vs_py (mortal_b200 mirror) -> engine.react_batch(list[np.ndarray (1012,34)], "
                            "list[np.ndarray (46,)], None) -> lists; observations reach the host through mjx_env_encode_obs_host "
                            "(pinned buffers; the single-player block runs in 4 row groups whose finished observations drain through "
                            "the copy engine meanwhile); engine = the CPU arm's policy (kind 2) in numpy",
                    "plain_d2h_copy_gbs": pcie_gbs},
            "e2e_with_net": (None if cn is None else {
                "value": cn_units / (cn_ms * 1e-3), "unit": "table-steps/s", "ms_per_step": cn_ms / cn["n"], "steps": cn["n"],
                "path": "the same arena call with DeviceEngine.react_batch: np.stack(obs) -> H2D -> 192x40 bf16 net -> lists "
                        "(mortal/engine.py:43-81's protocol), i.e. the `value` workload end to end through host buffers"}),
            # this library's kernels in the timed region: env kernels counted by libmjx, plus the fused policy-net kernels
            # (4 per residual block + 1, csrc/mjx_nn.cuh) that each CUDA-graph replay of the forward contains
            "gpu_launches": int(av["launches"] * K / max(av["cycles"], 1)) + 2 * K * (4 * 40 + 1), "gpu_launches_env": a["launches"], "clocks": clocks,
            "collective": collective,
        }
        line.update(extras)
        if world == 1 and not args.no_cpu_baseline:
            cb = cpu_arm(args, 2, args.cpu_baseline_steps)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "thirds_min_median_max")}
            line["cpu_baseline"]["same_games_as_env_only"] = "policy kind 2 on both arms: identical trajectories"
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def bench_encode_64k(mortal_b200, torch, np, dev, local_rank):
    """BASELINE configs[3]: encode_obs throughput at ~65536 decision rows per launch, full v4 (single-player block ON) and
    with the block off (the two encoder kernels alone)."""
    n64 = 65536
    n_nonce = np.repeat(np.arange(SEED_START[0], SEED_START[0] + n64 // 4, dtype=np.uint64), 4)
    env = mortal_b200.BatchEnv(n_nonce, np.full(n64, SEED_START[1], dtype=np.uint64), obs_version=4, device=local_rank)
    acts = torch.zeros(env.row_cap, dtype=torch.int64, device=dev)
    env.step(None)
    env.policy_test(2, acts)
    for _ in range(60):
        env.step(acts)
        env.policy_test(2, acts)
    obs64 = env.obs_buffer()
    out = {}
    for name, sp_on, reps in (("sp_off", False, 5), ("full_v4", True, 3)):
        env.set_sp(sp_on)
        rows64, ms64 = 0, 0.0
        for i in range(2 + reps):
            env.step(acts)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            env.encode_obs(obs64)
            e1.record()
            env.policy_test(2, acts)
            nr64 = env.num_rows()
            if i >= 2:
                rows64 += nr64
                ms64 += e0.elapsed_time(e1)
        gbs64 = rows64 * (OBS_BYTES + MASK_BYTES + STATE_BYTES) / (ms64 * 1e-3) / 1e9
        out[name] = {"rows_per_launch": rows64 / reps, "ms_per_launch": ms64 / reps, "achieved": gbs64, "unit": "GB/s",
                     "states_per_s": rows64 / (ms64 * 1e-3)}
    out["sp_arena_overflows"] = env.sp_overflows()
    env.close()
    del obs64
    torch.cuda.empty_cache()
    peak = 6650.0
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak = float(json.load(f).get("hbm_gbs", peak))
    except Exception:
        pass
    for k in ("sp_off", "full_v4"):
        out[k]["frac"] = out[k]["achieved"] / peak
    return out


def bench_algo_1m(torch, np, dev, args):
    """BASELINE configs[2]: shanten and agari at 1M hands (inputs resident in HBM, CUDA events), with the oracle beside them."""
    import ctypes as C

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import gen_hands as G
    import oracle_lib as O
    from mortal_b200 import _lib

    L = _lib.load()
    n = 1_000_000
    tiles, lens = G.random_hands(n)
    d_t, d_l = torch.from_numpy(tiles).to(dev), torch.from_numpy(lens).to(dev)
    d_o = torch.empty(n, dtype=torch.int8, device=dev)
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    # the 34 MB of hands would stay in the 126 MB L2 between repetitions: rotate through 8 copies (272 MB) so every launch reads HBM
    d_ts = [d_t] + [d_t.clone() for _ in range(7)]
    rot = [0]

    def next_tiles():
        rot[0] = (rot[0] + 1) % len(d_ts)
        return d_ts[rot[0]].data_ptr()

    def time_it(fn, reps=20):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    ms = time_it(lambda: _lib.check(L.mjx_shanten(next_tiles(), d_l.data_ptr(), d_o.data_ptr(), n, st), "mjx_shanten"))
    t0 = time.perf_counter()
    ref = O.shanten(tiles, lens)
    cpu_s = time.perf_counter() - t0
    assert (d_o.cpu().numpy() == ref).all()
    tmp = np.zeros(n, dtype=np.int8)
    host_s = float("inf")
    for _ in range(4):  # first call sizes the library's device scratch; best of the rest
        t0 = time.perf_counter()
        _lib.check(L.mjx_shanten_host(tiles.ctypes.data, lens.ctypes.data, tmp.ctypes.data, n), "mjx_shanten_host")
        if _:
            host_s = min(host_s, time.perf_counter() - t0)
    assert (tmp == ref).all()
    out = {"shanten_1m": {"hands": n, "ms_per_launch": ms, "hands_per_s": n / (ms * 1e-3), "table_lookups_per_s": 4 * n / (ms * 1e-3),
                          "achieved": n * 36 / (ms * 1e-3) / 1e9, "unit": "GB/s", "bytes_per_hand": 36,
                          "note": "L2-latency bound (4 gathers into the 16 MB table per hand), not HBM bound; inputs resident in HBM, "
                                  "8 rotating input copies (272 MB) so that no launch finds its hands in L2",
                          "e2e_host_buffers_hands_per_s": n / host_s,
                          "cpu_oracle_1_thread_hands_per_s": n / cpu_s, "bit_exact_vs_oracle": True}}
    q = G.winning_hands(n)
    d_q = torch.from_numpy(q.view(np.uint8).reshape(n, -1)).to(dev)
    d_r = torch.empty((n, 16), dtype=torch.uint8, device=dev)
    d_qs = [d_q] + [d_q.clone() for _ in range(3)]  # 4 x 62 MB: L2 rotation as above

    def next_q():
        rot[0] = (rot[0] + 1) % len(d_qs)
        return d_qs[rot[0]].data_ptr()

    ms = time_it(lambda: _lib.check(L.mjx_agari(next_q(), d_r.data_ptr(), n, 1, st), "mjx_agari"))
    t0 = time.perf_counter()
    ref = O.agari(q, 1)
    cpu_s = time.perf_counter() - t0
    got = d_r.cpu().numpy().view(G.AGARI_OUT_DTYPE).reshape(n)
    assert all((got[f] == ref[f]).all() for f in ("kind", "fu", "han", "yakuman", "ron", "tsumo_ko", "tsumo_oya"))
    out["agari_1m"] = {"hands": n, "mode": "agari() incl. points", "ms_per_launch": ms, "hands_per_s": n / (ms * 1e-3),
                       "achieved": n * (62 + 16) / (ms * 1e-3) / 1e9, "unit": "GB/s", "bytes_per_hand": 78,
                       "cpu_oracle_1_thread_hands_per_s": n / cpu_s, "bit_exact_vs_oracle": True}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--skip", type=int, default=300, help="untimed fast-forward batch steps before warm-up (both arms)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-baseline-steps", type=int, default=12, help="timed batch steps of the cpu_baseline leg of the default arm")
    ap.add_argument("--e2e-net-steps", type=int, default=12)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e-net", action="store_true")
    ap.add_argument("--no-algo-1m", action="store_true", help="skip BASELINE configs[2] (shanten / agari at 1M hands)")
    ap.add_argument("--no-encode-64k", action="store_true", help="skip the BASELINE configs[3] encode measurement (27 GB obs buffer)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed `value` path computed in its last timed step (observation sample, masks, "
                         "actions, Q-values, row ids) as DIR/<name>.npy; inputs are seeded, so runs with the same arguments compare")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
