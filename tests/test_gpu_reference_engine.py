"""MortalEngine-shaped engines on the device path (mortal_b200.engine.ReferenceEngine): the select kernel against torch and the
exact sampling distribution, the loaded networks against Mortal's own Q-values (tests/golden/ref_model_outputs.json), and the
mortal/player.py train_play configuration end to end through the arena, replayed in the oracle."""
import gzip
import json
import types

import numpy as np
import pytest
import scipy.stats

import oracle_lib as O
import ref_checkpoint_fixture as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    import torch

    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    from mortal_b200 import _lib

    _lib.init(0)
    return torch.device("cuda", 0)


def _env_rows(n, dev, masks):
    """the per-row buffers of an environment step with n rows: row i = table i // 4 at step i, seat i % 4"""
    import torch

    return types.SimpleNamespace(masks=masks.to(dev, torch.bool).contiguous(), row_table=torch.arange(n, dtype=torch.int32, device=dev) // 4,
                                 row_step=torch.arange(n, dtype=torch.int32, device=dev), row_seat=(torch.arange(n, device=dev) % 4).to(torch.uint8))


def _select(env, v, a, *, rows=None, eps=0.0, temp=1.0, top_p=1.0, seed=1234):
    import torch

    from mortal_b200 import nn_ops

    n, dev = a.shape[0], a.device
    actions = torch.full((n,), -1, dtype=torch.int64, device=dev)
    q = torch.zeros((n, 46), dtype=torch.float32, device=dev)
    greedy = torch.zeros(n, dtype=torch.uint8, device=dev)
    count = torch.tensor([n], dtype=torch.int32, device=dev)
    nn_ops.select_actions(v, a, rows, count, env.masks, env.row_table, env.row_step, env.row_seat, seed=seed, table_offset=0,
                          epsilon=eps, temp=temp, top_p=top_p, actions=actions, q_out=q, greedy=greedy)
    return actions, q, greedy


def test_select_kernel_greedy_equals_torch(dev):
    import torch

    g = torch.Generator().manual_seed(0)
    n = 4096
    a = torch.randn(n, 46, generator=g)
    v = torch.randn(n, 1, generator=g)
    masks = torch.rand(n, 46, generator=g) < 0.4
    masks[:, 7] |= torch.arange(n) % 5 == 0
    a[::3, 7] = a[::3, 11] = 10.0  # tied maxima (equal advantages give bit-equal Q): the lower index wins
    masks[::3, 7] = masks[::3, 11] = True
    masks[1::7] = False
    masks[1::7, 40] = True  # single legal action
    masks[2::11] = True      # everything legal
    env = _env_rows(n, dev, masks)
    v, a = v.to(dev), a.to(dev)
    m = env.masks
    want_q = (v + a - a.masked_fill(~m, 0).sum(-1, keepdim=True) / m.sum(-1, keepdim=True)).masked_fill(~m, -torch.inf)
    actions, q, greedy = _select(env, v, a)
    assert torch.equal(actions, want_q.argmax(-1))
    assert (actions[::3] != 11).all()
    assert torch.equal(torch.isneginf(q), ~m)
    assert ((q - want_q)[m].abs().max() <= 1e-6 * want_q[m].abs().max()).item()
    assert (greedy == 1).all()
    perm = torch.randperm(n, generator=g).to(dev)
    a2, q2, _ = _select(env, v[perm], a[perm], rows=perm.int())  # batch row i is environment row perm[i]
    assert torch.equal(a2, actions) and torch.equal(q2, q)


def _nucleus(q, temp, top_p):
    logits = np.asarray(q, dtype=np.float64) / temp
    p = np.exp(logits - logits.max())
    p /= p.sum()
    if top_p >= 1:
        return p
    if top_p <= 0:
        out = np.zeros_like(p)
        out[np.argmax(q)] = 1
        return out
    order = np.lexsort((np.arange(len(p)), -p))
    before = np.cumsum(p[order]) - p[order]
    keep = np.zeros(len(p), dtype=bool)
    keep[order[before <= top_p]] = True
    out = np.where(keep, p, 0)
    return out / out.sum()


@pytest.mark.parametrize("temp", [1.0, 0.05])
@pytest.mark.parametrize("top_p", [1.0, 0.9, 0.5, 0.0])
def test_select_kernel_sampling_distribution(dev, temp, top_p):
    import torch

    n = 1 << 18
    legal = [0, 3, 5, 9, 17, 30, 37, 41, 45]
    qv = np.array([0.10, 0.083, 0.061, 0.034, 0.0, -0.022, -0.047, -0.09, -0.13])
    a_row = torch.full((46,), 5.0)  # illegal advantages: must not matter
    a_row[legal] = torch.tensor(qv, dtype=torch.float32)
    mask_row = torch.zeros(46, dtype=torch.bool)
    mask_row[legal] = True
    env = _env_rows(n, dev, mask_row.expand(n, 46))
    a = a_row.to(dev).expand(n, 46).contiguous()
    v = torch.zeros(n, 1, device=dev)
    actions, q, greedy = _select(env, v, a, eps=1.0, temp=temp, top_p=top_p)
    assert (greedy == 0).all()
    q_legal = q[0, legal].double().cpu().numpy()
    want = _nucleus(q_legal, temp, top_p)
    counts = np.bincount(actions.cpu().numpy(), minlength=46)
    assert counts[~mask_row.numpy()].sum() == 0, "illegal action drawn"
    got = counts[legal]
    assert got[want == 0].sum() == 0, "action outside the nucleus drawn"
    kept = want > 0
    if kept.sum() > 1:
        assert scipy.stats.chisquare(got[kept], want[kept] * n).pvalue > 1e-4
    else:
        assert got[kept].sum() == n


def test_select_kernel_epsilon_rate_and_row_order(dev):
    import torch

    n, eps = 1 << 18, 0.005
    g = torch.Generator().manual_seed(1)
    masks = torch.rand(n, 46, generator=g) < 0.5
    masks[:, 0] = True
    env = _env_rows(n, dev, masks)
    a, v = torch.randn(n, 46, generator=g).to(dev), torch.zeros(n, 1, device=dev)
    actions, _, greedy = _select(env, v, a, eps=eps, temp=0.05, top_p=1.0)
    rate = 1 - greedy.float().mean().item()
    assert abs(rate - eps) <= 5 * np.sqrt(eps * (1 - eps) / n)
    perm = torch.randperm(n, generator=g).to(dev)
    a2, _, g2 = _select(env, v[perm], a[perm], rows=perm.int(), eps=eps, temp=0.05, top_p=1.0)
    assert torch.equal(a2, actions) and torch.equal(g2, greedy)  # a decision's draw is keyed by (table, step, seat), not its position
    a3, _, _ = _select(env, v, a, eps=eps, temp=0.05, top_p=1.0, seed=99)
    assert not torch.equal(a3, actions)


class StandIn:
    """The attributes mortal/engine.py MortalEngine.__init__ sets, nothing else"""

    def __init__(self, version, device, *, weight_seed=None, name="standin", enable_amp=True, eps=0.0, temp=1.0, top_p=1.0, guard=False):
        from mortal_b200.checkpoint import reference_schema

        schema = reference_schema(version, F.CHANNELS, F.BLOCKS)
        bsd, dsd = F.make_state_dicts(schema, 7000 + version if weight_seed is None else weight_seed)
        self.engine_type = "mortal"
        self.device = device
        self.brain, self.dqn = F.as_module(bsd).to(device).eval(), F.as_module(dsd).to(device).eval()
        self.is_oracle, self.version, self.stochastic_latent = False, version, False
        self.enable_amp, self.enable_quick_eval, self.enable_rule_based_agari_guard = enable_amp, True, guard
        self.name = name
        self.boltzmann_epsilon, self.boltzmann_temp, self.top_p = eps, temp, top_p

    def react_batch(self, obs, masks, invisible_obs):
        raise AssertionError("an adopted engine is never called through react_batch")


@pytest.mark.parametrize("version", F.VERSIONS)
def test_adopted_network_matches_mortal_q_values(dev, version):
    import torch

    from mortal_b200.engine import ReferenceEngine

    fix = F.load_fixture()["versions"][str(version)]
    obs, masks = F.make_inputs(version, F.ROWS, fix["input_seed"])
    want = fix["q"]
    n = F.ROWS
    env = _env_rows(n, dev, torch.from_numpy(masks))
    obs_buf = torch.from_numpy(obs).to(dev)
    legal = masks
    scale = np.abs(want[legal]).max()
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(3)).int().to(dev)
    tf32 = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        for amp, tol in ((False, 1e-4), (True, 0.05)):
            eng = ReferenceEngine(StandIn(version, dev, enable_amp=amp))
            eng.refresh()
            for rows in (None, perm):
                actions = torch.zeros(n, dtype=torch.int64, device=dev)
                q = torch.zeros((n, 46), dtype=torch.float32, device=dev)
                greedy = torch.zeros(n, dtype=torch.uint8, device=dev)
                count = torch.tensor([n], dtype=torch.int32, device=dev)
                eng.decide(obs_buf, env, rows, count, n, table_offset=0, actions=actions, q_out=q, greedy=greedy, bucket=64)
                got = q.double().cpu().numpy()
                assert (np.isneginf(got) == ~legal).all()
                err = np.abs(got[legal] - want[legal]).max()
                assert err <= tol * scale, (amp, rows is None, err, scale)
                assert (greedy.cpu().numpy() == 1).all()
            assert eng.graph_captures == 2 and eng.graph_replays == 2
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32


def _meta_events(paths):
    out = []
    for p in paths:
        with gzip.open(p, "rt") as f:
            out += [json.loads(ln)["meta"] for ln in f if '"meta"' in ln]
    return out


def _play(arena_cls, challenger, champion, seed_start, seed_count, tmp_path=None):
    arena = arena_cls(disable_progress_bar=True, log_dir=None if tmp_path is None else str(tmp_path))
    arena.adopt_reference_engines = True
    arena.record_decisions = True
    out = arena.py_vs_py(challenger=challenger, champion=champion, seed_start=seed_start, seed_count=seed_count)
    return arena, out


def _replay(arena, seed_start, seed_count, per):
    n = per * seed_count
    nonces = np.repeat(np.arange(seed_start[0], seed_start[0] + seed_count, dtype=np.uint64), per)
    keys = np.full(n, seed_start[1], dtype=np.uint64)
    ref = O.run_replay(nonces, keys, arena.last_decisions, quick_eval=True, mask_bits=arena.last_decision_masks)
    got = arena.last_results
    assert (got["scores"] == ref["scores"]).all() and (got["ranks"] == ref["ranks"]).all() and (got["steps"] == ref["steps"]).all()


def test_train_play_configuration_end_to_end(dev, tmp_path):
    """mortal/player.py TrainPlayer.train_play: a sampling trainee against a greedy champion with the agari guard, logs on."""
    import torch

    from mortal_b200.engine import ReferenceEngine
    from mortal_b200.libriichi.arena import OneVsThree, TwoVsTwo

    torch.manual_seed(0)
    trainee = StandIn(4, dev, name="trainee", eps=0.5, temp=0.05, top_p=0.9)
    champion = StandIn(4, dev, weight_seed=17, name="champion", guard=True)
    seed_start, seed_count = (20000, 0x3000), 6
    arena, rankings = _play(OneVsThree, trainee, champion, seed_start, seed_count, tmp_path / "logs")
    assert sum(rankings) == 4 * seed_count
    assert arena.last_meta_error is None
    assert all(isinstance(a, ReferenceEngine) for a in arena.last_agents)
    assert all(a.graph_captures > 0 and a.graph_replays > a.graph_captures for a in arena.last_agents)
    meta = _meta_events(arena.last_log_paths)
    assert len(meta) > 1000 and any(m["is_greedy"] is False for m in meta) and all(m["eval_time_ns"] > 0 for m in meta)

    # without the guard the recorded decisions are exactly what the environment played: replay them in the oracle
    champion.enable_rule_based_agari_guard = False
    arena, _ = _play(OneVsThree, trainee, champion, seed_start, seed_count)
    _replay(arena, seed_start, seed_count, 4)

    # a version-3 challenger against a version-4 champion: each encodes its own observation version
    v3 = StandIn(3, dev, name="v3", eps=0.5, temp=0.05, top_p=0.9)
    arena, rankings = _play(OneVsThree, v3, champion, seed_start, 4)
    assert sum(rankings) == 16 and all(a.graph_replays > 0 for a in arena.last_agents)
    _replay(arena, seed_start, 4, 4)

    arena, _ = _play(TwoVsTwo, trainee, champion, seed_start, 6)
    _replay(arena, seed_start, 6, 2)


def test_sampled_self_play_is_reproducible(dev):
    import torch

    from mortal_b200.libriichi.arena import OneVsThree

    det = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        runs = []
        for seed in (5, 5, 6):
            torch.manual_seed(seed)
            trainee = StandIn(4, dev, name="trainee", eps=0.5, temp=0.05, top_p=0.9)
            champion = StandIn(4, dev, weight_seed=17, name="champion")
            arena, rankings = _play(OneVsThree, trainee, champion, (30000, 0x10), 4)
            order = np.lexsort(arena.last_decisions[:, ::-1].T)
            runs.append((arena.last_decisions[order], arena.last_results["scores"].copy(), rankings))
    finally:
        torch.backends.cudnn.deterministic = det
    assert np.array_equal(runs[0][0], runs[1][0]) and np.array_equal(runs[0][1], runs[1][1]) and runs[0][2] == runs[1][2]
    assert runs[0][0].shape != runs[2][0].shape or not np.array_equal(runs[0][0], runs[2][0])
