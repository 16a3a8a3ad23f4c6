"""ctypes loader for mortal_b200/libmjx.so (the C ABI declared in include/mjx.h)."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
DATA_DIR = os.path.join(HERE, "data")
_LIB = None
_INIT_DEVICE = None


class MjxError(RuntimeError):
    pass


def lib_path() -> str:
    return os.path.join(HERE, "libmjx.so")


class AgariIn(C.Structure):
    _fields_ = [
        ("tehai", C.c_uint8 * 34),
        ("chis", C.c_uint8 * 4), ("pons", C.c_uint8 * 4), ("minkans", C.c_uint8 * 4), ("ankans", C.c_uint8 * 4),
        ("n_chis", C.c_uint8), ("n_pons", C.c_uint8), ("n_minkans", C.c_uint8), ("n_ankans", C.c_uint8),
        ("bakaze", C.c_uint8), ("jikaze", C.c_uint8), ("winning_tile", C.c_uint8), ("is_ron", C.c_uint8),
        ("additional_hans", C.c_uint8), ("doras", C.c_uint8), ("is_oya", C.c_uint8), ("pad", C.c_uint8),
    ]


class AgariOut(C.Structure):
    _fields_ = [("kind", C.c_uint8), ("fu", C.c_uint8), ("han", C.c_uint8), ("yakuman", C.c_uint8),
                ("ron", C.c_int32), ("tsumo_ko", C.c_int32), ("tsumo_oya", C.c_int32)]


# every symbol include/mjx.h declares: (restype, argtypes)
SYMBOLS = {
    "mjx_last_error": (C.c_char_p, []),
    "mjx_init": (C.c_int, [C.c_char_p, C.c_int]),
    "mjx_obs_rows": (C.c_int, [C.c_int]),
    "mjx_env_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "mjx_env_destroy": (None, [C.c_void_p]),
    "mjx_env_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mjx_env_set_quick_eval": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mjx_env_set_agari_guard": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mjx_env_encode_obs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "mjx_oracle_obs_rows": (C.c_int, [C.c_int]),
    "mjx_env_encode_invisible": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "mjx_env_set_obs_version": (C.c_int, [C.c_void_p, C.c_int]),
    "mjx_state_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_int]),
    "mjx_state_update": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mjx_state_view": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "mjx_state_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "mjx_state_query": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "mjx_state_copy": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "mjx_env_set_sp": (C.c_int, [C.c_void_p, C.c_int]),
    "mjx_env_encode_obs_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int), C.c_void_p]),
    "mjx_env_encode_obs_host_begin": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int), C.c_void_p]),
    "mjx_env_encode_obs_host_finish": (C.c_int, [C.c_void_p]),
    "mjx_env_sp_overflows": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]),
    "mjx_env_sp_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]),
    "mjx_env_enable_grp": (C.c_int, [C.c_void_p, C.c_int]),
    "mjx_env_read_grp": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mjx_env_enable_log": (C.c_int, [C.c_void_p, C.c_int]),
    "mjx_env_log_len_dev": (C.c_void_p, [C.c_void_p]),
    "mjx_env_read_log": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mjx_nn_affine_mish_bf16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p]),
    "mjx_nn_pool_bf16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "mjx_nn_gate_residual_bf16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "mjx_nn_obs_to_nhwc_bf16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "mjx_nn_block_tail_bf16": (C.c_int, [C.c_void_p] * 11 + [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "mjx_nn_obs_rows_to_nhwc_bf16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "mjx_select_actions": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_ulonglong, C.c_int, C.c_float, C.c_float, C.c_float,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mjx_split_rows": (C.c_int, [C.c_void_p] * 8),
    "mjx_env_create_replay": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p,
                                        C.c_void_p, C.c_longlong, C.c_void_p, C.c_int, C.c_int]),
    "mjx_env_replay_trust_seeds": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "mjx_env_replay_step": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mjx_env_row_label": (C.c_void_p, [C.c_void_p]),
    "mjx_env_row_meta": (C.c_void_p, [C.c_void_p]),
    "mjx_env_set_encode_timing": (C.c_int, [C.c_void_p, C.c_int]),
    "mjx_env_last_encode_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "mjx_env_launch_count": (C.c_longlong, [C.c_void_p]),
    "mjx_env_num_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]),
    "mjx_env_poll": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]),
    "mjx_env_num_live": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]),
    "mjx_env_total_steps": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]),
    "mjx_env_row_cap": (C.c_int, [C.c_void_p]),
    "mjx_env_masks": (C.c_void_p, [C.c_void_p]),
    "mjx_env_row_table": (C.c_void_p, [C.c_void_p]),
    "mjx_env_row_seat": (C.c_void_p, [C.c_void_p]),
    "mjx_env_row_step": (C.c_void_p, [C.c_void_p]),
    "mjx_env_num_rows_dev": (C.c_void_p, [C.c_void_p]),
    "mjx_env_results": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mjx_env_policy_test": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mjx_shanten": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "mjx_agari": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "mjx_shanten_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "mjx_agari_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "mjx_make_wall_host": (C.c_int, [C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_void_p]),
}


def load():
    """Load libmjx.so and bind every symbol. Fails loudly if the library was not built."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise MjxError(f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(nvcc, sm_100a). mortal_b200 has no CPU fallback.")
    L = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _LIB = L
    return L


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().mjx_last_error()
        raise MjxError(f"{what}: {msg.decode() if msg else rc}")


def init(device: int = 0) -> None:
    """mjx_init: upload the lookup tables to `device` (idempotent)."""
    global _INIT_DEVICE
    L = load()
    if _INIT_DEVICE == device:
        return
    check(L.mjx_init(DATA_DIR.encode(), device), "mjx_init")
    _INIT_DEVICE = device
