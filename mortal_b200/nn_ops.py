"""ctypes wrappers of the fused policy-net kernels in libmjx (csrc/mjx_nn.cuh). Tensors are CUDA bf16, logically
[B, C, 1, L] in channels_last memory format, i.e. [B, L, C] in memory."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib


def _stream(t: torch.Tensor):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _check_nhwc(x: torch.Tensor):
    assert x.is_cuda and x.dtype == torch.bfloat16 and x.dim() == 4 and x.shape[2] == 1
    b, c, _, l = x.shape
    assert c % 8 == 0 and x.stride(1) == 1 and x.stride(3) == c and x.stride(0) == c * l, "expected channels_last [B, C, 1, L]"
    return b, c, l


def affine_mish(x: torch.Tensor, scale: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """mish(x * scale[c] + bias[c]); scale / bias float32 [C]"""
    b, c, l = _check_nhwc(x)
    assert scale.dtype == torch.float32 and bias.dtype == torch.float32 and scale.numel() == c == bias.numel()
    out = torch.empty_like(x)
    _lib.check(_lib.load().mjx_nn_affine_mish_bf16(C.c_void_p(x.data_ptr()), C.c_void_p(scale.data_ptr()), C.c_void_p(bias.data_ptr()),
                                                   C.c_void_p(out.data_ptr()), x.numel(), c, _stream(x)), "mjx_nn_affine_mish_bf16")
    return out


def pool_mean_max(x: torch.Tensor):
    """(mean over L, max over L) -> two bf16 [B, C] tensors"""
    b, c, l = _check_nhwc(x)
    avg = torch.empty((b, c), dtype=torch.bfloat16, device=x.device)
    mx = torch.empty((b, c), dtype=torch.bfloat16, device=x.device)
    _lib.check(_lib.load().mjx_nn_pool_bf16(C.c_void_p(x.data_ptr()), C.c_void_p(avg.data_ptr()), C.c_void_p(mx.data_ptr()), b, l, c,
                                            _stream(x)), "mjx_nn_pool_bf16")
    return avg, mx


def gate_residual(y: torch.Tensor, gate: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """y * gate[b, c] + x; gate bf16 [B, C] contiguous"""
    b, c, l = _check_nhwc(y)
    assert _check_nhwc(x) == (b, c, l) and gate.dtype == torch.bfloat16 and gate.shape == (b, c) and gate.is_contiguous()
    out = torch.empty_like(y)
    _lib.check(_lib.load().mjx_nn_gate_residual_bf16(C.c_void_p(y.data_ptr()), C.c_void_p(gate.data_ptr()), C.c_void_p(x.data_ptr()),
                                                     C.c_void_p(out.data_ptr()), b, l, c, _stream(y)), "mjx_nn_gate_residual_bf16")
    return out


def block_tail(y: torch.Tensor, x: torch.Tensor, w1: torch.Tensor, b1: torch.Tensor, w2t: torch.Tensor, b2: torch.Tensor,
               scale: torch.Tensor, bias: torch.Tensor):
    """Channel gate + residual + the next pre-activation: gate = sigmoid(mlp(mean_L y) + mlp(max_L y)) with
    mlp(v) = w2 @ mish(w1 @ v + b1) + b2 (float32: w1 [H, C], w2t = w2.T [H, C]); returns (y * gate + x, mish((y * gate + x) * scale + bias))."""
    b, c, l = _check_nhwc(y)
    assert _check_nhwc(x) == (b, c, l)
    h = w1.shape[0]
    for t, shape in ((w1, (h, c)), (b1, (h,)), (w2t, (h, c)), (b2, (c,)), (scale, (c,)), (bias, (c,))):
        assert t.dtype == torch.float32 and tuple(t.shape) == shape and t.is_contiguous() and t.is_cuda
    assert c <= 256, "block_tail: at most 256 channels"
    x_out, a_out = torch.empty_like(y), torch.empty_like(y)
    gate = torch.empty((b, c), dtype=torch.bfloat16, device=y.device)
    p = lambda t: C.c_void_p(t.data_ptr())
    _lib.check(_lib.load().mjx_nn_block_tail_bf16(p(y), p(x), p(w1), p(b1), p(w2t), p(b2), p(scale), p(bias), p(gate), p(x_out), p(a_out),
                                                  b, l, c, h, _stream(y)), "mjx_nn_block_tail_bf16")
    return x_out, a_out


def obs_to_nhwc(obs: torch.Tensor, channels_padded: int) -> torch.Tensor:
    """f32 [B, C, L] (contiguous) -> bf16 [B, channels_padded, 1, L] in channels_last memory format, extra channels zero."""
    assert obs.is_cuda and obs.dtype == torch.float32 and obs.dim() == 3 and obs.is_contiguous()
    b, c, l = obs.shape
    assert channels_padded >= c and channels_padded % 64 == 0
    out = torch.empty((b, channels_padded, 1, l), dtype=torch.bfloat16, device=obs.device, memory_format=torch.channels_last)
    _lib.check(_lib.load().mjx_nn_obs_to_nhwc_bf16(C.c_void_p(obs.data_ptr()), C.c_void_p(out.data_ptr()), b, c, l, channels_padded,
                                                   _stream(obs)), "mjx_nn_obs_to_nhwc_bf16")
    return out


def obs_rows_to_nhwc(obs: torch.Tensor, rows: torch.Tensor, count: torch.Tensor, batch: int, channels_padded: int) -> torch.Tensor:
    """obs_to_nhwc of obs[rows[i]] for i < count (int32 device scalar), zero rows up to `batch`: an engine's share of the
    environment's observation buffer, converted without an intermediate f32 gather."""
    assert obs.is_cuda and obs.dtype == torch.float32 and obs.dim() == 3 and obs.is_contiguous()
    assert rows.dtype == torch.int32 and rows.is_contiguous() and rows.numel() >= batch and count.dtype == torch.int32
    _, c, l = obs.shape
    out = torch.empty((batch, channels_padded, 1, l), dtype=torch.bfloat16, device=obs.device, memory_format=torch.channels_last)
    _lib.check(_lib.load().mjx_nn_obs_rows_to_nhwc_bf16(C.c_void_p(obs.data_ptr()), C.c_void_p(rows.data_ptr()), C.c_void_p(count.data_ptr()),
                                                        C.c_void_p(out.data_ptr()), batch, c, l, channels_padded, _stream(obs)),
               "mjx_nn_obs_rows_to_nhwc_bf16")
    return out


def select_actions(v: torch.Tensor, a: torch.Tensor, rows, count: torch.Tensor, masks: torch.Tensor, row_table: torch.Tensor,
                   row_step: torch.Tensor, row_seat: torch.Tensor, *, seed: int, table_offset: int, epsilon: float, temp: float,
                   top_p: float, actions: torch.Tensor, q_out: torch.Tensor, greedy=None) -> None:
    """Masked dueling Q + greedy / epsilon-Boltzmann top-p selection (csrc/mjx_select.cuh k_select_actions) for batch rows
    i < count (int32 device scalar) of v f32 [n, 1] and a f32 [n, 46], written at the environment rows rows[i] (rows None: i) of
    actions int64, q_out f32 [., 46] and greedy uint8/bool."""
    n = a.shape[0]
    assert v.dtype == a.dtype == torch.float32 and a.shape[1] == 46 and a.stride(1) == 1 and v.shape[0] == n
    assert count.dtype == torch.int32 and masks.element_size() == 1 and masks.is_contiguous()
    assert row_table.dtype == torch.int32 and row_step.element_size() == 4 and row_seat.element_size() == 1
    assert actions.dtype == torch.int64 and q_out.dtype == torch.float32 and q_out.is_contiguous()
    if rows is not None:
        assert rows.dtype == torch.int32 and rows.is_contiguous() and rows.numel() >= n
    assert greedy is None or (greedy.element_size() == 1 and greedy.is_contiguous())
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    _lib.check(_lib.load().mjx_select_actions(p(v), v.stride(0), p(a), a.stride(0), p(rows), p(count), n, p(masks), p(row_table),
                                              p(row_step), p(row_seat), int(seed) & (2 ** 64 - 1), int(table_offset), float(epsilon),
                                              float(temp), float(top_p), p(actions), p(q_out), p(greedy), _stream(a)),
               "mjx_select_actions")


def split_rows(row_table: torch.Tensor, row_seat: torch.Tensor, count: torch.Tensor, agent_of: torch.Tensor, rows0: torch.Tensor,
               rows1: torch.Tensor, counts: torch.Tensor) -> None:
    """Stable split of the step's `count` rows by agent_of[table, seat & 3] (uint8 [n_tables, 4], 0 or 1) into rows0 / rows1
    (int32) and counts (int32 [2]), on the device."""
    assert row_table.dtype == torch.int32 and row_seat.element_size() == 1 and count.dtype == torch.int32
    assert agent_of.dtype == torch.uint8 and agent_of.is_contiguous() and agent_of.shape[1] == 4
    assert rows0.dtype == rows1.dtype == counts.dtype == torch.int32 and counts.numel() >= 2
    p = lambda t: C.c_void_p(t.data_ptr())
    _lib.check(_lib.load().mjx_split_rows(p(row_table), p(row_seat), p(count), p(agent_of), p(rows0), p(rows1), p(counts),
                                          _stream(row_table)), "mjx_split_rows")
