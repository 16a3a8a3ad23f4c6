"""Seeded stand-ins for Mortal checkpoints (shared by tools/extract_ref_fixtures.py and the tests).

`make_state_dicts(schema, seed)` fills a Brain / DQN key schema (mortal_b200.checkpoint.reference_schema) with weights drawn
from numpy's PCG64: normal weights scaled by 1/sqrt(fan_in), BatchNorm affines near identity, running_mean normal and
running_var uniform in [0.5, 1.5]. `make_inputs(version, n, seed)` draws observation rows (sparse 0/1 features plus a few
fractional rows) and legal masks with at least one legal action. tests/golden/ref_model_outputs.json holds, per version, the
schema, the seeds and the Q-values Mortal's own modules compute from these weights and inputs.
"""
from __future__ import annotations

import json
import os

import numpy as np

FIXTURE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_model_outputs.json")
VERSIONS = (2, 3, 4)
CHANNELS, BLOCKS, ROWS = 32, 2, 64
OBS_ROWS = {2: 942, 3: 934, 4: 1012}


def make_state_dicts(schema, seed: int):
    """{key: shape} dicts (brain, dqn) -> {key: float32 numpy array} dicts"""
    rng = np.random.Generator(np.random.PCG64(seed))
    out = []
    for part in schema:
        sd = {}
        for k, shape in part.items():
            shape = tuple(shape)
            if k.endswith("running_var"):
                v = rng.uniform(0.5, 1.5, shape)
            elif k.endswith("running_mean"):
                v = rng.normal(0.0, 0.2, shape)
            elif len(shape) == 1 and _is_bn(k, part):
                v = (1.0 if k.endswith("weight") else 0.0) + rng.normal(0.0, 0.1, shape)
            elif len(shape) == 1:  # Linear / conv bias
                v = rng.normal(0.0, 0.05, shape)
            else:
                fan_in = int(np.prod(shape[1:]))
                v = rng.normal(0.0, 1.0 / np.sqrt(fan_in), shape)
            sd[k] = v.astype(np.float32)
        out.append(sd)
    return tuple(out)


def _is_bn(key, part):
    return key.rsplit(".", 1)[0] + ".running_var" in part


def make_inputs(version: int, n: int, seed: int):
    """-> obs float32 [n, rows, 34], masks bool [n, 46]"""
    rng = np.random.Generator(np.random.PCG64(seed))
    obs = (rng.random((n, OBS_ROWS[version], 34)) < 0.08).astype(np.float32)
    obs[:, -40:] = rng.random((n, 40, 34)).astype(np.float32)  # fractional features, like the single-player tail of v4
    masks = rng.random((n, 46)) < 0.3
    masks[np.arange(n), rng.integers(0, 46, n)] = True
    return obs, masks


def load_fixture():
    with open(FIXTURE) as f:
        data = json.load(f)
    for v in data["versions"].values():
        v["q"] = np.array([[-np.inf if x is None else x for x in row] for row in v["q"]], dtype=np.float64)
    return data


def as_module(sd):
    """A torch module whose state_dict() is `sd` under the same keys (numpy or torch values): Mortal's key layout without its
    module code, which is all a MortalEngine's brain / dqn expose to ReferenceEngine."""
    import torch

    root = torch.nn.Module()
    for key, value in sd.items():
        *path, leaf = key.split(".")
        mod = root
        for name in path:
            if not hasattr(mod, name):
                mod.add_module(name, torch.nn.Module())
            mod = getattr(mod, name)
        t = torch.as_tensor(value)
        if leaf.startswith("running_") or leaf == "num_batches_tracked":
            mod.register_buffer(leaf, t.clone())
        else:
            mod.register_parameter(leaf, torch.nn.Parameter(t.clone(), requires_grad=False))
    return root
