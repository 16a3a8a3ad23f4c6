"""Python surface of libriichi for the self-play hot path, backed by the CUDA environment.

Mirrors the submodule layout of libriichi's PyO3 module (lib.rs:152-157, py_helper.rs:5-18): `consts`,
`arena`, `dataset` (GameplayLoader, Grp), `stat` (Stat), `state` (PlayerState, ActionCandidate), `mjai` (Bot). `install()` registers
this package as `libriichi` (and `libriichi.<sub>`) in sys.modules the way the reference's `add_submodule` does, so
`from libriichi.arena import OneVsThree` / `from libriichi.mjai import Bot` in mortal/*.py resolve here.
"""
import sys

from .. import dataset, stat  # GameplayLoader / Grp (dataset/gameplay.rs, dataset/grp.rs) and Stat (stat.rs): the modules themselves
from . import arena, consts, mjai, state  # noqa: F401

# `mortal_b200.libriichi.dataset` / `.stat` are the implementation modules under their libriichi names (no re-export shims)
sys.modules.setdefault(__name__ + ".dataset", dataset)
sys.modules.setdefault(__name__ + ".stat", stat)

__profile__ = "release"
__version__ = "0.1.0-mortal_b200"


def install(adopt_reference_engines: bool = False) -> None:
    """With adopt_reference_engines, the arenas play MortalEngine objects (versions 2-4, not oracle, on the arena's CUDA device)
    through mortal_b200.engine.ReferenceEngine on the device path instead of their react_batch; mortal/*.py stay unchanged."""
    arena._Arena.adopt_reference_engines = bool(adopt_reference_engines)
    mod = sys.modules[__name__]
    sys.modules.setdefault("libriichi", mod)
    for sub in ("arena", "consts", "dataset", "stat", "state", "mjai"):
        sys.modules.setdefault(f"libriichi.{sub}", getattr(mod, sub))
