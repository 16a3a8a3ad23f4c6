"""GPU parity at the sizes bench.py measures, and against reference-held vectors directly (not only via the oracle).

* BASELINE configs[1] size: 4096 tables, steady-state positions (300 fast-forward steps), full v4 observations incl. the
  single-player block (rows 889-1011, exact) of >= 2000 sampled decision rows vs the oracle.
* BASELINE configs[2] size: 1M shanten hands, 1M agari hands, bit-exact vs the oracle.
* The reference's own KATs (algo/shanten.rs:157-202, algo/agari.rs:919-1380) straight through mjx_shanten_host / mjx_agari_host,
  and its seeded golden log (log-viewer/index.example.html) through the device log replay with the reference-written mask_bits.
* BASELINE configs[1] workload: random-init 192x40 Mortal brain driving 4096 tables, decisions + legal masks replayed in the oracle.
* BASELINE configs[4] shape: 2 NCCL ranks, real end-of-hanchan returns all-gathered and checked against the oracle (needs 2 GPUs).
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import gen_hands as G
import oracle_lib as O
from obs_check import EXP_ROWS
from test_oracle_algo import AGARI_KATS
from test_oracle_golden import AGENT_EVENTS, load_golden, strip_meta

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
NCPU = max(1, min(64, os.cpu_count() or 1))


@pytest.fixture(scope="module")
def mjx():
    import torch

    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import mortal_b200
    from mortal_b200 import _lib

    _lib.init(0)
    return mortal_b200


def test_obs_parity_4096_tables_steady_state(mjx):
    """bench.py's env-only loop, checked: 4096 tables fast-forwarded 300 steps, then 20 encoded steps; 2560 sampled decision rows
    (all 1012 x 34 cells incl. the single-player block, the legal mask) equal the oracle's; no arena overflow."""
    import torch

    n, ff, steps, per_step = 4096, 300, 20, 128
    nonces = np.repeat(np.arange(10000, 10000 + n // 4, dtype=np.uint64), 4)
    keys = np.full(n, 0x2000, dtype=np.uint64)
    env = mjx.BatchEnv(nonces, keys)
    actions = torch.zeros(env.row_cap, dtype=torch.int64, device=env.device)
    gen = torch.Generator(device="cpu").manual_seed(0)
    env.step(None)
    for _ in range(ff):
        env.policy_test(1, actions)
        env.step(actions)
    samples, got_obs, got_masks, got_inv = [], [], [], []
    states = []
    for _ in range(steps):
        obs = env.encode_obs()
        inv = env.encode_invisible()
        nr = env.num_rows()
        states.append(env.sp_stats()[0])
        pick = torch.randperm(nr, generator=gen)[:per_step].to(env.device)
        got_obs.append(obs[pick].cpu().numpy())
        got_inv.append(inv[pick].cpu().numpy())
        got_masks.append(env.masks[pick].cpu().numpy())
        rs = env.row_seat[pick].long()
        samples.append(torch.stack([env.row_table[pick].long(), env.row_step[:nr].long()[pick], rs & 3, (rs >> 2) & 1], dim=1).cpu().numpy())
        env.policy_test(1, actions)
        env.step(actions)
    assert env.sp_overflows() == 0
    env.close()
    samples = np.concatenate(samples); got_obs = np.concatenate(got_obs); got_masks = np.concatenate(got_masks)
    assert len(samples) >= 2000 and min(states) > 100_000, (len(samples), states)  # the contended regime of the state arena
    ref_obs, ref_masks, found, ref_inv = O.run_sample_obs(nonces, keys, samples, n_threads=NCPU, max_steps=ff + steps + 2, invisible=True)
    assert found.all(), "the oracle never reached some sampled decisions: the trajectories differ"
    got_inv = np.concatenate(got_inv)
    assert got_inv.shape == ref_inv.shape == (len(samples), 217, 34) and (got_inv == ref_inv).all()  # board.rs:680-782, exact
    assert (ref_masks == got_masks).all()
    exact = np.ones(1012, dtype=bool)
    exact[EXP_ROWS] = False
    d = np.abs(got_obs - ref_obs)
    bad = np.argwhere(d[:, exact] != 0)
    assert len(bad) == 0, (len(bad), samples[bad[0, 0]], np.nonzero(exact)[0][bad[0, 1]], bad[0, 2])
    assert d[:, ~exact].max() <= 1e-6
    assert (got_obs[:, 889:] != 0).any(axis=(1, 2)).mean() > 0.9  # the single-player block is populated


def test_shanten_1m_hands_bit_exact(mjx):
    from mortal_b200 import _lib

    L = _lib.load()
    tiles, lens = G.random_hands(1_000_000)
    out = np.zeros(len(lens), dtype=np.int8)
    _lib.check(L.mjx_shanten_host(tiles.ctypes.data, lens.ctypes.data, out.ctypes.data, len(lens)), "mjx_shanten_host")
    ref = O.shanten(tiles, lens)
    assert (out == ref).all(), np.nonzero(out != ref)[0][:5]
    assert len(np.unique(ref)) >= 7


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_agari_1m_hands_bit_exact(mjx, mode):
    from mortal_b200 import _lib

    L = _lib.load()
    q = G.winning_hands(1_000_000)
    out = np.zeros(len(q), dtype=G.AGARI_OUT_DTYPE)
    _lib.check(L.mjx_agari_host(q.ctypes.data, out.ctypes.data, len(q), mode), "mjx_agari_host")
    ref = O.agari(q, mode)
    for f in ("kind", "fu", "han", "yakuman", "ron", "tsumo_ko", "tsumo_oya"):
        bad = np.nonzero(out[f] != ref[f])[0]
        assert len(bad) == 0, (f, bad[:5], out[bad[:5]], ref[bad[:5]])
    assert (ref["kind"] != 0).mean() > 0.4 and (mode == 2 or (ref["kind"] == 2).sum() > 1000)


def test_reference_kats_straight_through_the_cuda_path(mjx):
    """The reference's own known answers, asked of the CUDA kernels directly (no oracle in between)."""
    from mortal_b200 import _lib
    from oracle_lib import hand, tid

    L = _lib.load()
    sh = [("1111m 333p 222s 444z", 4, 1), ("147m 258p 369s 1234z", 4, 6), ("468m 33346p 7s", 3, 2), ("147m 258p 3s", 2, 4),
          ("4455s", 1, 0), ("7z", 0, 0), ("15559m 19p 19s 1234z", 4, 3), ("9999m 6677p 88s 355z", 4, 2),
          ("19m 19p 159s 123456z", 4, 1),                                                     # shanten.rs:157-177
          ("2344456m 14p 127s 2z 7p", 4, 3), ("2344456m 14p 127s 2z 5p", 4, 2), ("344455667p 1139s 9m", 4, 2),
          ("344455667p 1139s 9p", 4, 1), ("122334m 678p 37s 22z 5s", 4, 0), ("122334m 678p 12s 22z 4s", 4, 0),
          ("12223456m 78889p 2m", 4, -1), ("34778p", 1, 0), ("34s", 0, 0), ("55m", 0, -1)]   # shanten.rs:179-201
    tiles = np.stack([hand(s) for s, _, _ in sh]).astype(np.uint8)
    lens = np.array([n for _, n, _ in sh], dtype=np.uint8)
    out = np.zeros(len(sh), dtype=np.int8)
    _lib.check(L.mjx_shanten_host(tiles.ctypes.data, lens.ctypes.data, out.ctypes.data, len(sh)), "mjx_shanten_host")
    assert out.tolist() == [e for _, _, e in sh]

    q = np.concatenate([O.agari_query(t, **kw) for t, kw, _ in AGARI_KATS])             # agari.rs:959-1380
    res = np.zeros(len(q), dtype=G.AGARI_OUT_DTYPE)
    _lib.check(L.mjx_agari_host(q.ctypes.data, res.ctypes.data, len(q), 0), "mjx_agari_host")
    for r, (t, kw, exp) in zip(res, AGARI_KATS):
        got = None if r["kind"] == 0 else (("yakuman", int(r["yakuman"])) if r["kind"] == 2 else (int(r["fu"]), int(r["han"])))
        if isinstance(exp, tuple) and exp[0] == "han":
            assert got is not None and got[0] != "yakuman" and got[1] == exp[1], (t, got, exp)
        else:
            assert got == exp, (t, got, exp)
    # agari.rs:977-1000 / 1014-1016: points
    qq = np.concatenate([O.agari_query("12334m 345p 22s 777z 2m", bakaze="E", jikaze="E", winning_tile="3m", is_ron=False,
                                       additional_hans=2, doras=0, is_oya=True),
                         O.agari_query("2255m 445p 667788s 5p", bakaze="E", jikaze="S", winning_tile="5p", is_ron=True)])
    rr = np.zeros(2, dtype=G.AGARI_OUT_DTYPE)
    _lib.check(L.mjx_agari_host(qq[:1].ctypes.data, rr[:1].ctypes.data, 1, 1), "mjx_agari_host")
    assert (rr[0]["ron"], rr[0]["tsumo_ko"], rr[0]["tsumo_oya"]) == (7700, 2600, 0)
    _lib.check(L.mjx_agari_host(qq[1:].ctypes.data, rr[1:].ctypes.data, 1, 0), "mjx_agari_host")
    assert rr[1]["ron"] == 3200

    # agari.rs:919-957 check_ankan_after_riichi: the Tenhou rule (strict = false) is what PlayerState asks (update.rs:278).
    # `None` = the reference only lists the strict answer for that hand; strict-true implies non-strict-true.
    ankan = [("12345m 567s 11222z", "S", 4, True), ("12345m 444567s 11z", "4s", 4, True), ("22m 11112356p 444s", "4s", 4, True),
             ("123456m 4445s 111z", "4s", 4, False), ("1113444p 222z", "1p", 3, True), ("1113444p 222z", "S", 3, True),
             ("23m 999p 33345666s", "6s", 4, True), ("23m 999p 33345666s", "9p", 4, True), ("1113445678999m", "1m", 4, True),
             ("23m 999p 33345666s", "3s", 4, None), ("1113445678999m", "9m", 4, None), ("1113444p 222z", "4p", 3, None)]
    qa = np.zeros(len(ankan), dtype=G.AGARI_IN_DTYPE)
    for i, (t, tile, ld, _) in enumerate(ankan):
        h = hand(t)
        h[tid(tile)] += 1
        qa["tehai"][i] = h
        qa["winning_tile"][i] = tid(tile)
        qa["additional_hans"][i] = ld
    ra = np.zeros(len(ankan), dtype=G.AGARI_OUT_DTYPE)
    _lib.check(L.mjx_agari_host(qa.ctypes.data, ra.ctypes.data, len(ankan), 3), "mjx_agari_host mode 3")
    for i, (t, tile, ld, exp) in enumerate(ankan):
        if exp is None:
            exp = bool(O.lib().orc_check_ankan_after_riichi(qa["tehai"][i].ctypes.data, ld, tid(tile), 0))
        assert bool(ra["kind"][i]) == exp, (t, tile)


def test_golden_log_through_the_device_replay(mjx):
    """The reference's seeded example game through GameplayLoader.load_log on device (rand-0.8 era log, full information):
    every extracted non-pass move is the agent event the log holds, agari labels equal the log's hora events, and the legal
    mask of each decision equals the `meta.mask_bits` the REFERENCE wrote (105 decisions)."""
    from mortal_b200.libriichi.dataset import GameplayLoader

    golden = load_golden()
    text = "\n".join(json.dumps(strip_meta(e)) for e in golden)
    per_player = GameplayLoader(4, oracle=False).load_log(text)
    assert len(per_player) == 4
    tile_id = {name: i for i, name in enumerate(O.TILE_NAMES)}
    checked = 0
    for gp in per_player:
        p = gp.take_player_id()
        actions = np.array(gp.take_actions())
        masks = gp.take_masks(host=True)
        obs = gp.take_obs(host=True)
        assert obs.shape == (len(actions), 1012, 34) and obs.min() >= 0.0 and obs.max() <= 1.0
        moves = [(int(a), masks[i]) for i, a in enumerate(actions) if a not in (43, 45)]
        assert int((actions == 43).sum()) == sum(e["type"] == "hora" and e["actor"] == p for e in golden)
        logged = [e for e in golden if e.get("actor") == p and e["type"] in AGENT_EVENTS]
        assert len(moves) == len(logged) > 20
        for (label, mask), e in zip(moves, logged):
            if e["type"] == "dahai":
                assert label == tile_id[e["pai"]], (p, e, label)
            elif e["type"] == "reach":
                assert label == 37
            elif e["type"] == "pon":
                assert label == 41
            elif e["type"] == "chi":
                assert label in (38, 39, 40)
            if "meta" in e and "mask_bits" in e["meta"]:
                assert sum(1 << i for i in range(46) if mask[i]) == e["meta"]["mask_bits"], (p, e)
                checked += 1
        ak = np.array(gp.take_at_kyoku())
        assert ak[0] == 0 and ak[-1] == 2 and (np.diff(ak.astype(int)) >= 0).all()
    assert checked >= 100


def test_network_policy_action_replay_at_config2_size(mjx):
    """BASELINE configs[1] as bench.py runs it: 4096 tables, random-init 192ch x 40-block brain (bf16 fast path, greedy),
    60 BatchGame cycles through OneVsThree.py_vs_py. Every recorded decision must be requested by the oracle at the same
    (table, step, seat, kan-select), under a bit-identical legal mask, and be legal there; running scores agree."""
    import torch

    import mortal_b200.libriichi as lr
    from mortal_b200.engine import DeviceEngine
    from mortal_b200.model import DQN, Brain

    lr.install()
    from libriichi.arena import OneVsThree

    torch.manual_seed(0)
    dev = torch.device("cuda", 0)
    brain, dqn = Brain(conv_channels=192, num_blocks=40, version=4), DQN(version=4)
    eng = DeviceEngine(brain, dqn, device=dev, enable_amp=True, enable_quick_eval=True, name="m")
    assert brain.stem.weight.dtype == torch.float32 and brain.bn.running_var.dtype == torch.float32  # caller's module untouched
    arena = OneVsThree(disable_progress_bar=True)
    arena.record_decisions = True
    arena.max_cycles = 60
    seed_start, seed_count = (10000, 0x2000), 1024
    arena.py_vs_py(challenger=eng, champion=eng, seed_start=seed_start, seed_count=seed_count)
    n = 4 * seed_count
    dec, bits = arena.last_decisions, arena.last_decision_masks
    assert len(dec) == len(bits) > 60 * n * 0.8
    nonces = np.repeat(np.arange(seed_start[0], seed_start[0] + seed_count, dtype=np.uint64), 4)
    keys = np.full(n, seed_start[1], dtype=np.uint64)
    ref = O.run_replay(nonces, keys, dec, quick_eval=True, mask_bits=bits, max_steps=60, n_threads=NCPU)
    assert (ref["steps"] == 60).all() and (arena.last_results["steps"] == 60).all()


def test_two_rank_nccl_real_returns_match_oracle(mjx):
    """Tables sharded over 2 NCCL ranks, short hanchans played to the end, the REAL returns all-gathered
    (mortal_b200.dist.gather_returns) and every rank's slice compared with the oracle."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29517", os.path.join(HERE, "dist_returns_check.py"), "--seeds-per-rank", "64"]
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "RETURNS_OK world=2" in out.stdout
