"""mortal_b200.checkpoint: Mortal's own Brain / DQN state_dicts (versions 2-4) load into mortal_b200.model and compute what
Mortal's modules compute (tests/golden/ref_model_outputs.json); and which engines the arena adopts onto the device path."""
import numpy as np
import pytest
import torch

import ref_checkpoint_fixture as F
from mortal_b200.checkpoint import load_reference_checkpoint, load_reference_state_dicts, reference_schema

FIX = F.load_fixture()


def _schema(v):
    d = FIX["versions"][str(v)]
    return {k: tuple(s) for k, s in d["brain_schema"]}, {k: tuple(s) for k, s in d["dqn_schema"]}


def _state_dicts(v, prefix=""):
    bsd, dsd = F.make_state_dicts(_schema(v), FIX["versions"][str(v)]["weight_seed"])
    t = lambda sd: {prefix + k: torch.from_numpy(x) for k, x in sd.items()}
    return t(bsd), t(dsd)


@pytest.mark.parametrize("version", F.VERSIONS)
def test_schema_matches_mortal_modules(version):
    brain, dqn = reference_schema(version, FIX["channels"], FIX["blocks"])
    want_brain, want_dqn = _schema(version)
    assert list(brain.items()) == list(want_brain.items())
    assert list(dqn.items()) == list(want_dqn.items())


@pytest.mark.parametrize("version", F.VERSIONS)
def test_loaded_modules_reproduce_mortal_q_values(version):
    d = FIX["versions"][str(version)]
    brain, dqn = load_reference_state_dicts(*_state_dicts(version), version)
    assert brain.version == dqn.version == version
    assert all(bn.eps == (1e-5 if version == 2 else 1e-3) for bn in brain.modules() if isinstance(bn, torch.nn.BatchNorm1d))
    obs, masks = F.make_inputs(version, FIX["rows"], d["input_seed"])
    with torch.no_grad():
        q = dqn(brain(torch.from_numpy(obs)), torch.from_numpy(masks)).double().numpy()
    want = d["q"]
    assert (np.isneginf(q) == np.isneginf(want)).all() and (np.isneginf(q) == ~masks).all()
    legal = masks
    scale = np.abs(want[legal]).max()
    assert np.abs(q[legal] - want[legal]).max() <= 1e-5 * scale


def test_engine_modules_in_mortal_layout_load():
    bsd, dsd = _state_dicts(2)
    brain, dqn = load_reference_state_dicts(F.as_module(bsd).state_dict(), F.as_module(dsd).state_dict(), 2)
    plain_b, plain_d = load_reference_state_dicts(bsd, dsd, 2)
    assert all(torch.equal(a, b) for a, b in zip(brain.state_dict().values(), plain_b.state_dict().values()))
    assert all(torch.equal(a, b) for a, b in zip(dqn.state_dict().values(), plain_d.state_dict().values()))


def test_compiled_prefix_and_checkpoint_layout():
    bsd, dsd = _state_dicts(3, prefix="_orig_mod.")
    bsd["_orig_mod.encoder.net.1.res_unit.0.num_batches_tracked"] = torch.tensor(5)
    brain, dqn = load_reference_state_dicts(bsd, dsd, 3)
    plain_b, _ = load_reference_state_dicts(*_state_dicts(3), 3)
    for (k, a), (_, b) in zip(brain.state_dict().items(), plain_b.state_dict().items()):
        if not k.endswith("num_batches_tracked"):
            assert torch.equal(a, b), k
    ckpt = {"mortal": _state_dicts(4)[0], "current_dqn": _state_dicts(4)[1],
            "config": {"control": {"version": 4}, "resnet": {"conv_channels": 32, "num_blocks": 2}}}
    brain, dqn, version = load_reference_checkpoint(ckpt)
    assert version == 4 and brain.stem.weight.shape == (32, 1012, 3) and len(brain.blocks) == 2
    ckpt["config"]["resnet"]["num_blocks"] = 3
    with pytest.raises(ValueError, match="num_blocks"):
        load_reference_checkpoint(ckpt)


def test_missing_or_misshaped_keys_are_named():
    bsd, dsd = _state_dicts(2)
    del bsd["encoder.net.2.ca.shared_mlp.2.bias"]
    with pytest.raises(ValueError, match=r"encoder\.net\.2\.ca\.shared_mlp\.2\.bias"):
        load_reference_state_dicts(bsd, dsd, 2)
    bsd, dsd = _state_dicts(2)
    dsd["a_head.0.weight"] = torch.zeros(256, 1024)  # the v3 hidden size in a v2 head
    with pytest.raises(ValueError, match=r"a_head\.0\.weight"):
        load_reference_state_dicts(bsd, dsd, 2)
    with pytest.raises(ValueError, match="version"):
        load_reference_state_dicts(*_state_dicts(4), 1)


class StandIn:
    """The attributes mortal/engine.py MortalEngine.__init__ sets, nothing else"""

    def __init__(self, version=4, is_oracle=False, device=torch.device("cpu")):
        self.engine_type = "mortal"
        self.device = device
        bsd, dsd = _state_dicts(version)
        self.brain, self.dqn = F.as_module(bsd), F.as_module(dsd)
        self.is_oracle, self.version = is_oracle, version
        self.stochastic_latent = False
        self.enable_amp, self.enable_quick_eval, self.enable_rule_based_agari_guard = False, True, False
        self.name = "standin"
        self.boltzmann_epsilon, self.boltzmann_temp, self.top_p = 0, 1, 1

    def react_batch(self, obs, masks, invisible_obs):
        raise AssertionError("not called here")


def test_adoption_is_opt_in_and_limited_to_eligible_engines():
    from mortal_b200.engine import HostProtocolEngine, ReferenceEngine
    from mortal_b200.libriichi.arena import OneVsThree

    arena = OneVsThree(disable_progress_bar=True)
    assert arena.adopt_reference_engines is False
    cuda = torch.device("cuda", 0)
    eligible = StandIn(4, device=cuda)
    assert isinstance(arena._adapt(eligible), HostProtocolEngine)
    arena.adopt_reference_engines = True
    assert isinstance(arena._adapt(eligible), ReferenceEngine)
    v1 = StandIn(4, device=cuda)
    v1.version = 1
    for e in (v1, StandIn(4, is_oracle=True, device=cuda), StandIn(4), StandIn(2, device=torch.device("cuda", 1))):
        assert isinstance(arena._adapt(e), HostProtocolEngine)

    class Device:
        version = 4

        def react_device(self, obs, masks):
            pass

    dev = Device()
    assert arena._adapt(dev) is dev
