#!/usr/bin/env python
"""Self-play throughput at mortal/player.py TrainPlayer.train_play's call site, in one invocation, as one JSON line.

Arms (4096 tables, 192 x 40 version-4 networks held in Mortal's state_dict layout, timed after the usual fast-forward):
  adopted  OneVsThree.py_vs_py(trainee, champion) with adopt_reference_engines: trainee epsilon 0.005 / temp 0.05 / top_p 1.0,
           champion with the rule-based agari guard, log_dir set (logs with per-decision meta)
  host     the same engines and configuration through their react_batch (the reference protocol: observations to the host
           and back, the stock eager module under fp16 autocast, as MortalEngine runs it)
  value    one greedy DeviceEngine for every seat, no logs: the single-engine device path, for reference
Also reported: the card's name and power limit, and the time of k_select_actions per step at the adopted arm's rows per step
(CUDA events over repeated launches on the same shapes).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True


class MortalShaped:
    """The attributes mortal/engine.py MortalEngine sets, and its react_batch (autocast, stock forward, sampling)"""

    def __init__(self, brain_mod, dqn_mod, fwd, *, device, name, eps=0.0, temp=1.0, top_p=1.0, guard=False):
        self.engine_type, self.device, self.name = "mortal", device, name
        self.brain, self.dqn = brain_mod, dqn_mod
        self._fwd = fwd  # (Brain, DQN) with the same weights in this repo's module layout, for react_batch
        self.is_oracle, self.version, self.stochastic_latent = False, 4, False
        self.enable_amp, self.enable_quick_eval, self.enable_rule_based_agari_guard = True, True, guard
        self.boltzmann_epsilon, self.boltzmann_temp, self.top_p = eps, temp, top_p

    def react_batch(self, obs, masks, invisible_obs):
        import numpy as np
        import torch

        from mortal_b200.engine import sample_top_p

        with torch.autocast(self.device.type, enabled=self.enable_amp), torch.inference_mode():
            obs = torch.as_tensor(np.stack(obs, axis=0), device=self.device)
            masks = torch.as_tensor(np.stack(masks, axis=0), device=self.device)
            q = self._fwd[1](self._fwd[0](obs), masks)
            if self.boltzmann_epsilon > 0:
                greedy = torch.full((obs.shape[0],), 1 - self.boltzmann_epsilon, device=self.device).bernoulli().to(torch.bool)
                logits = (q / self.boltzmann_temp).masked_fill(~masks, -torch.inf)
                actions = torch.where(greedy, q.argmax(-1), sample_top_p(logits, self.top_p))
            else:
                greedy = torch.ones(obs.shape[0], dtype=torch.bool, device=self.device)
                actions = q.argmax(-1)
        return actions.tolist(), q.tolist(), masks.tolist(), greedy.tolist()


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as exc:  # the numbers stay valid without it, but say so
        return {"error": str(exc)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tables", type=int, default=4096)
    ap.add_argument("--skip", type=int, default=200, help="fast-forward batch steps before the first engine call")
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--steps", type=int, default=48)
    ap.add_argument("--host-steps", type=int, default=12)
    args = ap.parse_args()

    import numpy as np
    import torch

    import ref_checkpoint_fixture as F
    from mortal_b200.checkpoint import load_reference_state_dicts, reference_schema
    from mortal_b200.engine import DeviceEngine
    from mortal_b200.libriichi.arena import OneVsThree

    if not torch.cuda.is_available():
        raise SystemExit("bench_call_site.py: no CUDA device")
    dev = torch.device("cuda", 0)
    schema = reference_schema(4, 192, 40)

    def engine(seed, **kw):
        bsd, dsd = F.make_state_dicts(schema, seed)
        fwd = load_reference_state_dicts(bsd, dsd, 4)
        return MortalShaped(F.as_module(bsd).to(dev).eval(), F.as_module(dsd).to(dev).eval(), (fwd[0].to(dev), fwd[1].to(dev)),
                            device=dev, **kw)

    torch.manual_seed(0)
    trainee = engine(11, name="trainee", eps=0.005, temp=0.05, top_p=1.0)
    champion = engine(12, name="champion", guard=True)
    greedy = DeviceEngine(*load_reference_state_dicts(*F.make_state_dicts(schema, 12), 4), device=dev, enable_amp=True, name="value")

    def run(a, b, n_timed, adopt, log):
        arena = OneVsThree(disable_progress_bar=True, log_dir=tempfile.mkdtemp(prefix="callsite_") if log else None)
        arena.adopt_reference_engines = adopt
        arena.fast_forward_steps = args.skip
        arena.max_cycles = args.warmup + n_timed + 1
        marks = {}

        def hook(c, state):
            if c in (args.warmup, args.warmup + n_timed):
                torch.cuda.synchronize()
                marks[c] = (time.perf_counter(), state.total_steps())

        arena.cycle_hook = hook
        arena.py_vs_py(a, b, (10000, 0x2000), args.tables // 4)
        (t0, s0), (t1, s1) = marks[args.warmup], marks[args.warmup + n_timed]
        return arena, {"value": (s1 - s0) / (t1 - t0), "unit": "table-steps/s", "ms_per_step": (t1 - t0) * 1e3 / n_timed, "steps": n_timed,
                       "meta_error": None if arena.last_meta_error is None else str(arena.last_meta_error)}

    out = {"tool": "bench_call_site", "tables": args.tables, "net": "192x40 v4", "card": card()}
    arena, out["adopted"] = run(trainee, champion, args.steps, True, True)
    out["adopted"]["graph_replays"] = sum(a.graph_replays for a in arena.last_agents)
    out["adopted"]["graph_captures"] = sum(a.graph_captures for a in arena.last_agents)
    _, out["host"] = run(trainee, champion, args.host_steps, False, True)
    _, out["value"] = run(greedy, greedy, args.steps, False, False)
    out["adopted_over_host"] = out["adopted"]["value"] / out["host"]["value"]
    out["adopted_over_value"] = out["adopted"]["value"] / out["value"]["value"]

    # k_select_actions alone at the rows of one adopted step (~1 decision row per table), trainee settings, 200 launches
    from mortal_b200 import nn_ops

    n = args.tables
    g = torch.Generator(device=dev).manual_seed(0)
    v, a = torch.randn(n, 1, device=dev, generator=g), torch.randn(n, 46, device=dev, generator=g)
    masks = torch.rand(n, 46, device=dev, generator=g) < 0.3
    masks[:, 0] = True
    rows = torch.randperm(n, device=dev, generator=g).int()
    tbl, step, seat = torch.arange(n, dtype=torch.int32, device=dev), torch.zeros(n, dtype=torch.int32, device=dev), torch.zeros(n, dtype=torch.uint8, device=dev)
    count = torch.tensor([n], dtype=torch.int32, device=dev)
    act, q, gr = torch.zeros(n, dtype=torch.int64, device=dev), torch.zeros(n, 46, device=dev), torch.zeros(n, dtype=torch.uint8, device=dev)
    call = lambda: nn_ops.select_actions(v, a, rows, count, masks, tbl, step, seat, seed=1, table_offset=0, epsilon=0.005, temp=0.05, top_p=1.0,
                                         actions=act, q_out=q, greedy=gr)
    for _ in range(10):
        call()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(200):
        call()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / 200
    bytes_per = n * (4 + 46 * 4 + 4 + 46 + 12 + 8 + 46 * 4 + 1)
    out["select_kernel"] = {"rows": n, "us_per_launch": us, "bytes_per_launch": bytes_per, "GB_per_s": bytes_per / (us * 1e-6) / 1e9,
                            "note": "includes the ctypes launch; rows in a random order"}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
