"""Load Mortal's own Brain / DQN weights (mortal/model.py, versions 2-4) into mortal_b200.model.

Mortal's Brain keeps its trunk in one `nn.Sequential` (`encoder.net`): the stem conv at index 0, the residual blocks at
1..n (each a `res_unit` Sequential of BN, Mish, conv, BN, Mish, conv plus the channel attention's `ca.shared_mlp`), then
BN at n+1, the 32-channel conv at n+3 and the Linear at n+6. mortal_b200.model names the same modules `stem`, `blocks`,
`bn`, `neck` and `fc`; this module translates between the two. The BatchNorm eps is not part of a state_dict: it
follows from the version (model.BN_EPS).
"""
from __future__ import annotations

import re

import torch

from .model import ACTION_SPACE, DQN, DQN_HIDDEN, OBS_ROWS, Brain, _check_version

_BN = ("weight", "bias", "running_mean", "running_var")
_STRIP = "_orig_mod."  # torch.compile wraps a module and prefixes every key with this


def _bn(prefix, c):
    return {f"{prefix}.{k}": (c,) for k in _BN}


def reference_schema(version: int, conv_channels: int, num_blocks: int):
    """Ordered ({key: shape} of Mortal's Brain.state_dict(), {key: shape} of its DQN.state_dict()), without the
    BatchNorms' num_batches_tracked."""
    _check_version(version)
    c, n, h = conv_channels, num_blocks, conv_channels // 16
    brain = {"encoder.net.0.weight": (c, OBS_ROWS[version], 3)}
    for i in range(n):
        p = f"encoder.net.{1 + i}"
        brain.update(_bn(f"{p}.res_unit.0", c))
        brain[f"{p}.res_unit.2.weight"] = (c, c, 3)
        brain.update(_bn(f"{p}.res_unit.3", c))
        brain[f"{p}.res_unit.5.weight"] = (c, c, 3)
        brain.update({f"{p}.ca.shared_mlp.0.weight": (h, c), f"{p}.ca.shared_mlp.0.bias": (h,),
                      f"{p}.ca.shared_mlp.2.weight": (c, h), f"{p}.ca.shared_mlp.2.bias": (c,)})
    brain.update(_bn(f"encoder.net.{n + 1}", c))
    brain.update({f"encoder.net.{n + 3}.weight": (32, c, 3), f"encoder.net.{n + 3}.bias": (32,),
                  f"encoder.net.{n + 6}.weight": (1024, 32 * 34), f"encoder.net.{n + 6}.bias": (1024,)})
    if version == 4:
        dqn = {"net.weight": (1 + ACTION_SPACE, 1024), "net.bias": (1 + ACTION_SPACE,)}
    else:
        hd = DQN_HIDDEN[version]
        dqn = {}
        for head, out in (("v_head", 1), ("a_head", ACTION_SPACE)):
            dqn.update({f"{head}.0.weight": (hd, 1024), f"{head}.0.bias": (hd,), f"{head}.2.weight": (out, hd), f"{head}.2.bias": (out,)})
    return brain, dqn


def _clean(sd):
    out = {}
    for k, v in sd.items():
        if k.startswith(_STRIP):
            k = k[len(_STRIP):]
        if k.endswith("num_batches_tracked"):
            continue
        out[k] = v
    return out


def _check(sd, schema, what):
    for k, shape in schema.items():
        if k not in sd:
            raise ValueError(f"{what} state_dict: missing key {k!r}")
        if tuple(sd[k].shape) != shape:
            raise ValueError(f"{what} state_dict: key {k!r} has shape {tuple(sd[k].shape)}, expected {shape}")
    extra = sorted(set(sd) - set(schema))
    if extra:
        raise ValueError(f"{what} state_dict: unexpected key {extra[0]!r}")


def _infer_shape(brain_sd):
    """(conv_channels, num_blocks) from the keys of a cleaned Brain state_dict"""
    if "encoder.net.0.weight" not in brain_sd:
        raise ValueError("Brain state_dict: missing key 'encoder.net.0.weight'")
    blocks = {int(m.group(1)) for k in brain_sd if (m := re.match(r"encoder\.net\.(\d+)\.res_unit\.", k))}
    return int(brain_sd["encoder.net.0.weight"].shape[0]), len(blocks)


def _brain_key_map(num_blocks: int):
    """Mortal's Brain key -> mortal_b200.model.Brain key"""
    n = num_blocks
    m = {"encoder.net.0.weight": "stem.weight"}
    for i in range(n):
        p, q = f"encoder.net.{1 + i}", f"blocks.{i}"
        for src, dst in (("res_unit.0", "bn1"), ("res_unit.3", "bn2")):
            m.update({f"{p}.{src}.{k}": f"{q}.{dst}.{k}" for k in _BN})
        m[f"{p}.res_unit.2.weight"] = f"{q}.conv1.weight"
        m[f"{p}.res_unit.5.weight"] = f"{q}.conv2.weight"
        for src, dst in (("ca.shared_mlp.0", "gate.fc1"), ("ca.shared_mlp.2", "gate.fc2")):
            m.update({f"{p}.{src}.{k}": f"{q}.{dst}.{k}" for k in ("weight", "bias")})
    m.update({f"encoder.net.{n + 1}.{k}": f"bn.{k}" for k in _BN})
    m.update({f"encoder.net.{n + 3}.{k}": f"neck.{k}" for k in ("weight", "bias")})
    m.update({f"encoder.net.{n + 6}.{k}": f"fc.{k}" for k in ("weight", "bias")})
    return m


def load_reference_state_dicts(brain_sd, dqn_sd, version: int):
    """Mortal Brain / DQN state_dicts (version 2, 3 or 4; `_orig_mod.` prefixes allowed) -> (mortal_b200.model.Brain,
    mortal_b200.model.DQN) in eval mode on the CPU, fp32. Raises ValueError naming the first missing, unexpected or
    wrongly shaped key."""
    version = int(version)
    _check_version(version)
    brain_sd, dqn_sd = _clean(brain_sd), _clean(dqn_sd)
    c, n = _infer_shape(brain_sd)
    want_brain, want_dqn = reference_schema(version, c, n)
    _check(brain_sd, want_brain, "Brain")
    _check(dqn_sd, want_dqn, "DQN")
    brain = Brain(conv_channels=c, num_blocks=n, version=version)
    keys = _brain_key_map(n)
    f32 = lambda t: torch.as_tensor(t).detach().to("cpu", torch.float32)
    brain.load_state_dict({keys[k]: f32(v) for k, v in brain_sd.items()}, strict=False)
    dqn = DQN(version=version)
    dqn.load_state_dict({k: f32(v) for k, v in dqn_sd.items()})
    return brain.eval(), dqn.eval()


def load_reference_checkpoint(path_or_dict):
    """A Mortal `.pth` (or the dict torch.load returns for one) as mortal/player.py reads it: `mortal` (Brain) and
    `current_dqn` state_dicts, `config.control.version` and `config.resnet.{conv_channels, num_blocks}` ->
    (Brain, DQN, version)."""
    state = path_or_dict
    if not isinstance(state, dict):
        state = torch.load(path_or_dict, map_location="cpu", weights_only=True)
    cfg = state["config"]
    version = int(cfg["control"]["version"])
    brain, dqn = load_reference_state_dicts(state["mortal"], state["current_dqn"], version)
    res = cfg.get("resnet", {})
    for k, got in (("conv_channels", brain.stem.weight.shape[0]), ("num_blocks", len(brain.blocks))):
        if k in res and int(res[k]) != got:
            raise ValueError(f"checkpoint config resnet.{k} = {res[k]} but the weights have {got}")
    return brain, dqn, version
