"""CPU-only checks of the host layer: the C ABI library loads and exports every declared symbol, fails loudly
without a GPU (no CPU fallback), the libriichi mirror has the reference's surface, and the N>1 plumbing
(seed sharding + the all-gather of returns) works over gloo with world_size 2."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_c_abi_exports_every_declared_symbol():
    import mortal_b200
    from mortal_b200 import _lib

    L = mortal_b200.load()
    header = open(os.path.join(ROOT, "include", "mjx.h")).read()
    declared = set(re.findall(r"\b(mjx_[a-z0-9_]+)\s*\(", header))
    declared -= {"mjx_status"}
    assert declared, "no declarations parsed"
    for name in declared:
        assert hasattr(L, name), f"libmjx.so does not export {name}"
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    assert C.sizeof(_lib.AgariIn) == 62 and C.sizeof(_lib.AgariOut) == 16


def test_product_fails_loudly_without_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import mortal_b200
    from mortal_b200 import _lib

    L = mortal_b200.load()
    rc = L.mjx_init(_lib.DATA_DIR.encode(), 0)
    assert rc != 0 and b"no CUDA device" in L.mjx_last_error()
    with pytest.raises(mortal_b200.MjxError):
        mortal_b200.BatchEnv(np.array([1], dtype=np.uint64), np.array([2], dtype=np.uint64))
    out = np.zeros(1, dtype=np.int8)
    assert L.mjx_shanten_host(np.zeros(34, dtype=np.uint8).ctypes.data, np.zeros(1, dtype=np.uint8).ctypes.data,
                              out.ctypes.data, 1) != 0


def test_product_never_touches_the_oracle():
    """oracle/ and tests/host_emul are test infrastructure: nothing under mortal_b200/ may reference them."""
    for dirpath, _, files in os.walk(os.path.join(ROOT, "mortal_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "liboracle" not in src and "oracle_lib" not in src and "libmjx_emul" not in src, f
                if f.endswith(".py"):
                    assert "emul_lib" not in src, f


def test_libriichi_mirror_surface():
    import mortal_b200.libriichi as lr

    lr.install()
    from libriichi.arena import OneVsThree, TwoVsTwo
    from libriichi.consts import ACTION_SPACE, GRP_SIZE, MAX_VERSION, obs_shape, oracle_obs_shape

    assert (ACTION_SPACE, GRP_SIZE, MAX_VERSION) == (46, 7, 4)
    assert [obs_shape(v) for v in (1, 2, 3, 4)] == [(938, 34), (942, 34), (934, 34), (1012, 34)]
    assert oracle_obs_shape(1) == (211, 34) and oracle_obs_shape(4) == (217, 34)
    env = OneVsThree(disable_progress_bar=True, log_dir=None)
    assert hasattr(env, "py_vs_py") and hasattr(TwoVsTwo(), "py_vs_py")
    assert env._challenger_seats(6) == [2] and TwoVsTwo()._challenger_seats(1) == [1, 3]


WORKER = r'''
import os, sys
import numpy as np
import torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from mortal_b200.dist import shard_seeds, gather_returns
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
nonces, keys = shard_seeds((10000, 0x2000), 8, rank)
assert nonces[0] == 10000 + 8 * rank and len(nonces) == 32 and (keys == 0x2000).all()
scores = (np.arange(32 * 4, dtype=np.int32).reshape(32, 4) + 1000 * rank) - 500
ranks = np.tile(np.array([[(0 + rank) % 4, 1, 2, 3]], dtype=np.uint8), (32, 1))
s_all, r_all = gather_returns(scores, ranks)
assert s_all.shape == (32 * world, 4) and r_all.shape == (32 * world, 4)
for r in range(world):
    assert (s_all[32 * r: 32 * r + 32] == np.arange(128, dtype=np.int32).reshape(32, 4) + 1000 * r - 500).all()
    assert (r_all[32 * r: 32 * r + 32, 0] == r % 4).all()
dist.destroy_process_group()
print("ok", rank)
'''


def test_world_size_2_gloo_gather(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29731", str(script), ROOT],
                         capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert out.stdout.count("ok") == 2


def test_grp_on_the_reference_golden_log():
    """dataset/grp.rs:90-164 on the seeded example log (log-viewer/index.example.html): features per kyoku, final scores with
    the busted player's sticks handling, stable ranking."""
    import json

    from mortal_b200.dataset import Grp

    with open(os.path.join(ROOT, "tests", "golden", "golden_game.jsonl")) as f:
        events = [json.loads(ln) for ln in f if ln.strip()]
    g = Grp.load_events(events)
    assert g.feature.shape == (3, 7) and len(g) == 3
    assert g.feature[0].tolist() == [0.0, 0.0, 0.0, 2.5, 2.5, 2.5, 2.5]
    assert g.feature[1].tolist() == [0.0, 1.0, 0.0, 3.27, 2.5, 1.73, 2.5]
    assert g.feature[2].tolist() == [1.0, 0.0, 0.0, 3.27, 3.02, 1.31, 2.4]
    # last kyoku: 32700/30200/13100/24000 + hora [0, 20000, -18000, 0] - one riichi stick of the winner, returned to the top
    assert sum(g.take_final_scores()) == 100_000
    assert g.take_rank_by_player() == [1, 0, 3, 2]


def test_stat_on_the_reference_golden_log_and_invariants():
    """stat.rs:263-442 on the seeded example log (hand-checked) and field-wise invariants over emulated self-play logs."""
    import json
    import math

    from mortal_b200.stat import Stat

    with open(os.path.join(ROOT, "tests", "golden", "golden_game.jsonl")) as f:
        events = [json.loads(ln) for ln in f if ln.strip()]
    st = [Stat.from_game(events, p) for p in range(4)]
    # 3 kyoku; hora by 0 (ron on 2, riichi), by 1 (ron on 2, no riichi stick of its own counted), by 1 (ron on 2): see the log
    assert [s.round for s in st] == [3, 3, 3, 3] and [s.agari for s in st] == [1, 2, 0, 0] and [s.houjuu for s in st] == [0, 0, 3, 0]
    assert st[2].tobi == 1 and [s.rank_1 + s.rank_2 + s.rank_3 + s.rank_4 for s in st] == [1, 1, 1, 1]
    assert st[1].rank_1 == 1 and st[0].rank_2 == 1 and st[3].rank_3 == 1 and st[2].rank_4 == 1
    assert sum(s.point for s in st) == 0
    assert st[0].agari_point_oya == 8700 - 1000 and st[0].riichi_agari == 1  # own stick not counted (stat.rs:336)
    assert math.isnan(st[3].avg_point_per_agari) and st[2].houjuu_rate == 1.0
    total = sum(st[1:], st[0])
    assert total.game == 4 and total.agari == 3 and abs(total.avg_rank - 2.5) < 1e-12
    assert st[1].avg_pt([90, 45, 0, -135]) == 90.0


def test_stat_from_dir_and_field_invariants(tmp_path):
    import gzip
    import json

    from mortal_b200 import mjai_log
    from mortal_b200.stat import COUNTERS, Stat
    from test_emul_vs_oracle import _selfplay_logs

    games = _selfplay_logs(8, 1, 4321)
    for g, ev in enumerate(games):
        ev[0]["names"] = ["hero" if s == g % 4 else "villain" for s in range(4)]
        with gzip.open(tmp_path / f"{g}.json.gz", "wt") as f:
            f.write("\n".join(json.dumps(e, separators=(",", ":")) for e in ev) + "\n")
    hero = Stat.from_dir(str(tmp_path), "hero")
    villain = Stat.from_dir(str(tmp_path), "villain")
    assert hero.game == 8 and villain.game == 24
    n_hora = sum(e["type"] == "hora" for ev in games for e in ev)
    assert hero.agari + villain.agari == n_hora
    assert hero.rank_1 + hero.rank_2 + hero.rank_3 + hero.rank_4 == 8
    assert hero.point + villain.point == 0 and hero.round * 3 == villain.round
    assert hero.dama_agari + hero.fuuro_agari + hero.riichi_agari == hero.agari
    assert 1.0 <= hero.avg_rank <= 4.0 and all(getattr(hero, c) >= 0 for c in COUNTERS if "point" not in c)
    assert str(hero).startswith("Games 8") and "agari_rate" in str(hero)


def test_event_codec_round_trip_on_golden_and_selfplay_logs():
    """mortal_b200.dataset_codec.encode_events is the inverse of mortal_b200.mjai_log.decode_events for everything the replay
    needs: every event survives a round trip except the payloads the replay does not use (hora / ryukyoku deltas, ura markers)."""
    import json

    from mortal_b200 import dataset_codec as DC
    from mortal_b200 import mjai_log
    from test_emul_vs_oracle import _selfplay_logs

    with open(os.path.join(ROOT, "tests", "golden", "golden_game.jsonl")) as f:
        golden = [{k: v for k, v in json.loads(ln).items() if k != "meta"} for ln in f if ln.strip()]
    for events in [golden] + _selfplay_logs(3, 0, 77):
        hdr, pay = DC.encode_events(events)
        assert len(hdr) == len(events) and pay.shape == (sum(e["type"] == "start_kyoku" for e in events), DC.KYOKU_WORDS)
        # re-expand into the multi-word stream decode_events reads (payload after each start_kyoku, zero deltas after hora/ryukyoku)
        words, k = [], 0
        for w in hdr:
            ty = int(w) & 0xFF
            if ty in (DC.START_GAME, DC.END_GAME):
                continue
            words.append(int(w))
            if ty == mjai_log.START_KYOKU:
                words += [int(x) for x in pay[k][:9]]  # the device log carries scores + the 52 dealt tiles only
                k += 1
            elif ty in (mjai_log.HORA, mjai_log.RYUKYOKU):
                words += [0, 0]
        back = mjai_log.decode_events(words)
        inner = [e for e in events if e["type"] not in ("start_game", "end_game")]
        assert len(back) == len(inner)
        for a, b in zip(back, inner):
            if b["type"] in ("hora", "ryukyoku"):
                assert a["type"] == b["type"] and a.get("actor") == b.get("actor") and a.get("target") == b.get("target")
            else:
                assert a == b, (a, b)


def test_arena_meta_recorder_writes_meta_into_logs(tmp_path):
    """The arena's _MetaRecorder + mjai_log.write_logs on CPU tensors (driven by the emulated env with the call pattern of
    _Arena._run): the written .json.gz files carry a `meta` with the reference's fields on the agent events, the events
    themselves are unchanged, and a recorder failure degrades to logs without meta instead of an exception."""
    import gzip
    import json

    import torch

    import emul_lib as E
    from mortal_b200 import mjai_log
    from mortal_b200.libriichi.arena import _MetaRecorder

    n = 4
    nonces = np.arange(3300, 3300 + n, dtype=np.uint64)
    keys = np.full(n, 2, dtype=np.uint64)
    env = E.EmulEnv(nonces, keys, enable_quick_eval=True)
    env.enable_log()
    rec = _MetaRecorder(n, 4)
    acts, cycles = None, 0
    while True:
        env.step(acts)
        rec.add_bounds(torch.from_numpy(env.log_lens()))
        rt, rs, masks = env.rows()
        nr = len(rt)
        if nr == 0 and env.num_live() == 0:
            break
        acts = env.policy_test(1)
        if nr:
            obs = torch.from_numpy(env.encode_obs(sp=False, version=4))
            idx = torch.arange(nr)
            q = torch.where(torch.from_numpy(masks), torch.rand(nr, 46), torch.full((nr, 46), -float("inf")))
            rec.add_agent(cycles, idx, q, 12345)
            rec.add_rows(cycles, torch.from_numpy(rt).long(), torch.from_numpy(rs), torch.from_numpy(acts[:nr]), torch.from_numpy(masks), obs)
        cycles += 1
    words, lens = env.read_log()
    env.close()
    bounds, decisions = rec.finish()
    seeds = [(int(nonces[g]), 2) for g in range(n)]
    names = [["a", "b", "c", "d"]] * n
    paths = mjai_log.write_logs(str(tmp_path / "m"), words, lens, seeds, names, "abcd", bounds, decisions)
    plain = mjai_log.write_logs(str(tmp_path / "p"), words, lens, seeds, names, "abcd")
    n_meta = 0
    for pm, pp in zip(paths, plain):
        with_meta = [json.loads(ln) for ln in gzip.open(pm, "rt")]
        without = [json.loads(ln) for ln in gzip.open(pp, "rt")]
        assert [{k: v for k, v in e.items() if k != "meta"} for e in with_meta] == without
        for e in with_meta:
            if "meta" in e:
                m = e["meta"]
                assert list(m)[:5] == ["q_values", "mask_bits", "is_greedy", "batch_size", "eval_time_ns"] and "shanten" in m and "at_furiten" in m
                assert 0 <= m["shanten"] <= 6 and m["eval_time_ns"] == 12345 and all(np.isfinite(m["q_values"]))
                n_meta += 1
    assert n_meta > 800
    broken = _MetaRecorder(n, 4)
    broken.add_rows(0, None, None, None, None, None)  # bad input: recorded as an error, not raised
    assert broken.error is not None
    with pytest.raises(Exception):
        broken.finish()


def test_policy_net_fast_path_equals_stock_forward_on_cpu():
    """mortal_b200/model.py: the BN-folded, channels-last (1x3 conv2d) inference path is the same function as the stock module
    (mortal/model.py architecture) in fp32; the DQN head's masked dueling combination (mortal/model.py DQN) and the nucleus
    sampler behave as specified."""
    import torch

    from mortal_b200.engine import sample_top_p
    from mortal_b200.model import DQN, Brain

    torch.manual_seed(0)
    brain = Brain(conv_channels=32, num_blocks=3).eval()
    for m in brain.modules():
        if isinstance(m, torch.nn.BatchNorm1d):
            m.running_mean.normal_(); m.running_var.uniform_(0.5, 2); m.weight.data.normal_(1, 0.2); m.bias.data.normal_()
    obs = (torch.rand(7, 1012, 34) < 0.05).float()
    with torch.no_grad():
        ref = brain(obs)
        brain.prepare_fast(None)
        fast = brain.forward_fast(obs)
    assert ref.shape == (7, 1024) and (ref - fast).abs().max() < 1e-5
    dqn = DQN().eval()
    mask = torch.rand(7, 46) > 0.5
    mask[:, 45] = True
    with torch.no_grad():
        q = dqn(ref, mask)
        v, a = dqn.net(ref).split((1, 46), dim=-1)
    assert torch.isneginf(q[~mask]).all()
    want = v + a - (a * mask).sum(-1, keepdim=True) / mask.sum(-1, keepdim=True)
    assert torch.allclose(q[mask], want[mask], atol=1e-6)
    logits = torch.tensor([[2.0, 1.0, 0.5, -1.0, -float("inf")]]).repeat(4000, 1)
    s = sample_top_p(logits, 0.7)
    assert set(s.tolist()) <= {0, 1} and 0.68 < (s == 0).float().mean() < 0.78  # nucleus {0, 1}: 0.61 / (0.61 + 0.224)
    assert sample_top_p(logits[:3], 0.0).tolist() == [0, 0, 0]


import oracle_lib as O  # noqa: E402 (test infrastructure)


def _emul_arena(cls):
    from emul_batch_env import EmulBatchEnv

    arena = cls(disable_progress_bar=True)
    arena.env_factory = EmulBatchEnv
    return arena


def test_arena_host_protocol_loop_on_emulated_env_fail_fast():
    """The arena's host-protocol loop on the host-emulated environment: (1) an engine that answers an illegal action makes
    py_vs_py raise at that very cycle (game.rs:288,292 aborts the batch), not after the games were played out; (2) a legal
    engine's recorded decisions replay in the oracle to the same scores."""
    import pytest

    from mortal_b200.libriichi.arena import OneVsThree

    class Eng:
        engine_type = "mortal"; name = "e"; version = 4; is_oracle = False
        enable_quick_eval = True; enable_rule_based_agari_guard = False

        def __init__(self, bad_at=None):
            self.calls, self.bad_at = 0, bad_at

        def react_batch(self, obs, masks, invisible_obs):
            self.calls += 1
            m = np.stack(masks)
            a = [int(np.nonzero(r)[0][-1]) for r in m]            # the highest legal action id
            if self.bad_at is not None and self.calls >= self.bad_at:
                a[0] = int(np.nonzero(~m[0])[0][0])               # an illegal one
            return a, np.where(m, 0.0, -np.inf).tolist(), m.tolist(), [True] * len(a)

    bad = Eng(bad_at=7)
    arena = _emul_arena(OneVsThree)
    with pytest.raises(RuntimeError, match="failed at cycle"):
        arena.py_vs_py(bad, bad, (5000, 3), 1)
    assert bad.calls <= 9, "the batch must abort at the offending cycle"

    good = Eng()
    arena = _emul_arena(OneVsThree)
    arena.record_decisions = True
    rankings = arena.py_vs_py(good, good, (5000, 3), 3)  # 12 games: two half-batches (4 + 8 tables) stepped alternately
    assert sum(rankings) == 12 and arena.last_stats["parts"] == 2
    nonces = np.repeat(np.arange(5000, 5003, dtype=np.uint64), 4)
    keys = np.full(12, 3, dtype=np.uint64)
    ref = O.run_replay(nonces, keys, arena.last_decisions, quick_eval=True, mask_bits=arena.last_decision_masks)
    assert (ref["scores"] == arena.last_results["scores"]).all() and (ref["ranks"] == arena.last_results["ranks"]).all()


def test_arena_feeds_oracle_engines_the_invisible_observation():
    """agent/mortal.rs:253-255, 137-146: an engine with is_oracle=True receives invisible_obs (list of (217, 34) arrays, one per row)
    next to obs and masks; an ordinary engine receives None. Checked on the host-emulated environment: the other seats' hand
    planes of the invisible observation hold 13/14-tile hands and the wall planes are populated."""
    from mortal_b200.libriichi.arena import OneVsThree

    seen = dict(oracle_rows=0, plain_calls=0)

    class Eng:
        engine_type = "mortal"; version = 4; enable_quick_eval = True; enable_rule_based_agari_guard = False

        def __init__(self, name, is_oracle):
            self.name, self.is_oracle = name, is_oracle

        def react_batch(self, obs, masks, invisible_obs):
            m = np.stack(masks)
            if self.is_oracle:
                assert invisible_obs is not None and len(invisible_obs) == len(obs)
                for iv in invisible_obs:
                    assert iv.shape == (217, 34) and iv.dtype == np.float32
                    for k in range(3):  # 4 count planes per opponent: a 13- or 14-tile hand minus its melds
                        assert iv[17 * k:17 * k + 4].sum() in (1, 2, 4, 5, 7, 8, 10, 11, 13, 14)
                    assert iv[51:51 + 138].sum() > 0
                seen["oracle_rows"] += len(obs)
            else:
                assert invisible_obs is None
                seen["plain_calls"] += 1
            a = [int(np.nonzero(r)[0][0]) for r in m]
            return a, np.where(m, 0.0, -np.inf).tolist(), m.tolist(), [True] * len(a)

    arena = _emul_arena(OneVsThree)
    arena.max_cycles = 40
    arena.py_vs_py(Eng("o", True), Eng("p", False), (7100, 2), 2)
    assert seen["oracle_rows"] > 20 and seen["plain_calls"] > 20


def test_arena_agents_with_different_obs_version_and_quick_eval():
    """agent/mortal.rs:54-74, 256-287: `version` and `enable_quick_eval` belong to the agent. A version-4 quick-eval challenger
    against a version-2 champion without quick-eval: each engine sees observations of its own layout, the champion's seats emit
    rows for forced discards too, and the recorded decisions replay in the oracle with the same per-seat settings."""
    from mortal_b200.libriichi.arena import OneVsThree

    class Eng:
        engine_type = "mortal"; is_oracle = False; enable_rule_based_agari_guard = False

        def __init__(self, name, version, qe):
            self.name, self.version, self.enable_quick_eval, self.rows = name, version, qe, 0

        def react_batch(self, obs, masks, invisible_obs):
            assert all(o.shape == ({2: 942, 4: 1012}[self.version], 34) for o in obs)
            m = np.stack(masks)
            self.rows += len(obs)
            a = [int(np.nonzero(r)[0][0]) for r in m]  # the lowest legal action id
            return a, np.where(m, 0.0, -np.inf).tolist(), m.tolist(), [True] * len(a)

    chal, champ = Eng("c4", 4, True), Eng("c2", 2, False)
    arena = _emul_arena(OneVsThree)
    arena.record_decisions = True
    arena.max_cycles = 70
    arena.py_vs_py(chal, champ, (8100, 4), 2)
    assert chal.rows > 50 and champ.rows > 3 * chal.rows * 0.8
    n = 8
    nonces = np.repeat(np.arange(8100, 8102, dtype=np.uint64), 4)
    keys = np.full(n, 4, dtype=np.uint64)
    qf = np.array([[1 if seat == g % 4 else 0 for seat in range(4)] for g in range(n)], dtype=np.uint8)
    ref = O.run_replay(nonces, keys, arena.last_decisions, mask_bits=arena.last_decision_masks, max_steps=70, quick_eval_seats=qf)
    assert (ref["steps"] == arena.last_results["steps"]).all()
