"""Policy/value network used by the benchmark and examples (stays ordinary PyTorch, as north_star asks).

Architecture restated from mortal/model.py:10-231 (versions 2-4): Conv1d stem -> `num_blocks` pre-activation
residual blocks (BN -> Mish -> Conv1d k3, twice) each gated by a squeeze/excite style channel attention
-> BN -> Mish -> Conv1d(C, 32, k3) -> Mish -> Linear(32*34, 1024) -> Mish ; dueling head Linear(1024, 1+46) (v4) or
two Linear -> Mish -> Linear MLPs (v2: hidden 512, v3: 256) with the advantage mean taken over legal actions only and illegal
actions at -inf. Versions differ in the stem's input rows and the BatchNorm eps (v2 1e-5, v3/v4 1e-3). Mortal checkpoints load
through mortal_b200.checkpoint.
"""
from __future__ import annotations

import torch
from torch import nn

OBS_ROWS = {1: 938, 2: 942, 3: 934, 4: 1012}  # consts.rs:20-28
ACTION_SPACE = 46
BN_EPS = {2: 1e-5, 3: 1e-3, 4: 1e-3}  # not stored in a state_dict: the versions' BatchNorm1d constructors differ
DQN_HIDDEN = {2: 512, 3: 256}


def _check_version(version: int):
    if version not in BN_EPS:
        raise ValueError(f"network version {version} is not supported (2, 3 or 4)")


class ChannelGate(nn.Module):
    def __init__(self, channels: int, ratio: int = 16):
        super().__init__()
        self.fc1 = nn.Linear(channels, channels // ratio)
        self.fc2 = nn.Linear(channels // ratio, channels)
        nn.init.zeros_(self.fc1.bias)
        nn.init.zeros_(self.fc2.bias)
        self.act = nn.Mish(inplace=True)

    def _mlp(self, v):
        return self.fc2(self.act(self.fc1(v)))

    def forward(self, x):
        gate = torch.sigmoid(self._mlp(x.mean(-1)) + self._mlp(x.amax(-1)))
        return x * gate.unsqueeze(-1)

    def forward_fast(self, x):
        # x: [B, C, 1, L] channels_last; same maths as forward()
        gate = torch.sigmoid(self._mlp(x.mean((2, 3))) + self._mlp(x.amax((2, 3))))
        return x * gate.view(gate.shape[0], gate.shape[1], 1, 1)


class PreActBlock(nn.Module):
    def __init__(self, channels: int, eps: float = 1e-3):
        super().__init__()
        self.bn1 = nn.BatchNorm1d(channels, momentum=0.01, eps=eps)
        self.conv1 = nn.Conv1d(channels, channels, 3, padding=1, bias=False)
        self.bn2 = nn.BatchNorm1d(channels, momentum=0.01, eps=eps)
        self.conv2 = nn.Conv1d(channels, channels, 3, padding=1, bias=False)
        self.act = nn.Mish(inplace=True)
        self.gate = ChannelGate(channels)

    def forward(self, x):
        y = self.conv1(self.act(self.bn1(x)))
        y = self.conv2(self.act(self.bn2(y)))
        return self.gate(y) + x

    @staticmethod
    def _affine(bn):
        # eval-mode BatchNorm is a per-channel affine map: y = x * scale + shift
        scale = bn.weight / torch.sqrt(bn.running_var + bn.eps)
        shift = bn.bias - bn.running_mean * scale
        return scale.view(1, -1, 1, 1).contiguous(), shift.view(1, -1, 1, 1).contiguous()

    def forward_fast(self, x, aff, w1, w2, aff32=None):
        (s1, b1), (s2, b2) = aff
        F = torch.nn.functional
        if aff32 is not None and x.is_cuda and x.dtype == torch.bfloat16:
            # fused bandwidth-bound passes (libmjx, csrc/mjx_nn.cuh) around the two cuDNN convolutions
            from . import nn_ops

            (f1, g1), (f2, g2) = aff32
            y = F.conv2d(nn_ops.affine_mish(x, f1, g1), w1, padding=(0, 1))
            y = F.conv2d(nn_ops.affine_mish(y, f2, g2), w2, padding=(0, 1))
            avg, mx = nn_ops.pool_mean_max(y)
            h = self.gate._mlp(torch.cat((avg, mx), 0))  # both pooled vectors through the gate MLP in one call
            gate = torch.sigmoid(h[: avg.shape[0]] + h[avg.shape[0]:])
            return nn_ops.gate_residual(y, gate.contiguous(), x)
        y = F.conv2d(F.mish(torch.addcmul(b1, x, s1)), w1, padding=(0, 1))
        y = F.conv2d(F.mish(torch.addcmul(b2, y, s2)), w2, padding=(0, 1))
        return self.gate.forward_fast(y) + x


class Brain(nn.Module):
    def __init__(self, *, conv_channels: int = 192, num_blocks: int = 40, version: int = 4):
        super().__init__()
        _check_version(version)
        self.version = version
        c, eps = conv_channels, BN_EPS[version]
        self.stem = nn.Conv1d(OBS_ROWS[version], c, 3, padding=1, bias=False)
        self.blocks = nn.Sequential(*[PreActBlock(c, eps) for _ in range(num_blocks)])
        self.bn = nn.BatchNorm1d(c, momentum=0.01, eps=eps)
        self.act = nn.Mish(inplace=True)
        self.neck = nn.Conv1d(c, 32, 3, padding=1)
        self.fc = nn.Linear(32 * 34, 1024)

    def forward(self, obs):
        x = self.blocks(self.stem(obs))
        x = self.act(self.neck(self.act(self.bn(x))))
        return self.act(self.fc(x.flatten(1)))

    @torch.no_grad()
    def prepare_fast(self, dtype=None):
        """Inference-only fast path: eval-mode BatchNorms pre-folded into per-channel affines (two elementwise
        kernels instead of cuDNN's NCHW batch-norm kernel) and optional reduced-precision weights so that no
        autocast casts are needed. Mathematically the same network; call after loading weights / .eval()."""
        assert not self.training, "prepare_fast() is for eval mode"
        # fp32 copies of the folded affines for the fused kernels, taken before any down-cast of the parameters
        flat = lambda a: (a[0].float().flatten().contiguous(), a[1].float().flatten().contiguous())
        self._aff32 = [(flat(PreActBlock._affine(b.bn1)), flat(PreActBlock._affine(b.bn2))) for b in self.blocks]
        self._aff32_out = flat(PreActBlock._affine(self.bn))
        if dtype is not None:
            self.to(dtype)
        self._aff = [(PreActBlock._affine(b.bn1), PreActBlock._affine(b.bn2)) for b in self.blocks]
        self._aff_out = PreActBlock._affine(self.bn)
        # the channel-gate MLPs as fp32 copies of the (possibly down-cast) parameters, for the fused block tail
        f32 = lambda t: t.detach().float().contiguous()
        self._gate32 = [(f32(b.gate.fc1.weight), f32(b.gate.fc1.bias), f32(b.gate.fc2.weight.t()), f32(b.gate.fc2.bias)) for b in self.blocks]
        # the Conv1d kernels as (1 x 3) Conv2d kernels in channels_last, so cuDNN runs NHWC without layout round trips
        cl = lambda conv: conv.weight.unsqueeze(2).contiguous(memory_format=torch.channels_last)
        self._w = [(cl(b.conv1), cl(b.conv2)) for b in self.blocks]
        self._w_stem, self._w_neck = cl(self.stem), cl(self.neck)
        # the stem with its input channels zero-padded to a multiple of 64 (1012 -> 1024): nn_ops.obs_to_nhwc emits that layout
        cin = self.stem.weight.shape[1]
        self._cpad = (cin + 63) // 64 * 64
        wp = torch.zeros((self.stem.weight.shape[0], self._cpad, 3), dtype=self.stem.weight.dtype, device=self.stem.weight.device)
        wp[:, :cin] = self.stem.weight.detach()
        self._w_stem_pad = wp.unsqueeze(2).contiguous(memory_format=torch.channels_last)
        self._fast_dtype = dtype
        return self

    def forward_fast(self, obs):
        F = torch.nn.functional
        fused = obs.is_cuda and self._fast_dtype == torch.bfloat16
        if fused and obs.dtype == torch.float32 and obs.is_contiguous():
            from . import nn_ops

            return self.forward_fast_nhwc(nn_ops.obs_to_nhwc(obs, self._cpad))
        if self._fast_dtype is not None:
            obs = obs.to(self._fast_dtype)
        x = obs.unsqueeze(2).contiguous(memory_format=torch.channels_last)  # [B, C, 1, 34]
        return self._trunk_fast(F.conv2d(x, self._w_stem, padding=(0, 1)))

    def forward_fast_nhwc(self, x):
        """forward_fast from the stem input already in the padded bf16 channels-last layout nn_ops.obs_to_nhwc emits"""
        return self._trunk_fast(torch.nn.functional.conv2d(x, self._w_stem_pad, padding=(0, 1)))

    def _trunk_fast(self, x):
        F = torch.nn.functional
        fused = x.is_cuda and self._fast_dtype == torch.bfloat16
        if fused:
            # libmjx kernels (csrc/mjx_nn.cuh) around the cuDNN convolutions: per block one BN-affine+Mish pass and one pass for
            # everything between conv2 and the next block's conv1 (pooling, gate MLP, sigmoid, gate * y + x, next BN-affine+Mish)
            from . import nn_ops

            n = len(self.blocks)
            a = nn_ops.affine_mish(x, *self._aff32[0][0]) if n else nn_ops.affine_mish(x, *self._aff32_out)
            for i in range(n):
                (w1, w2), (_, (f2, g2)) = self._w[i], self._aff32[i]
                y = F.conv2d(a, w1, padding=(0, 1))
                y = F.conv2d(nn_ops.affine_mish(y, f2, g2), w2, padding=(0, 1))
                nxt = self._aff32[i + 1][0] if i + 1 < n else self._aff32_out
                x, a = nn_ops.block_tail(y, x, *self._gate32[i], *nxt)
            x = a
        else:
            for blk, aff, (w1, w2) in zip(self.blocks, self._aff, self._w):
                x = blk.forward_fast(x, aff, w1, w2, None)
            s, b = self._aff_out
            x = F.mish(torch.addcmul(b, x, s))
        x = F.mish(F.conv2d(x, self._w_neck, self.neck.bias, padding=(0, 1)))
        return F.mish(self.fc(x.flatten(1)))


class DQN(nn.Module):
    def __init__(self, *, version: int = 4):
        super().__init__()
        _check_version(version)
        self.version = version
        if version == 4:
            self.net = nn.Linear(1024, 1 + ACTION_SPACE)
            nn.init.zeros_(self.net.bias)
        else:
            h = DQN_HIDDEN[version]
            self.v_head = nn.Sequential(nn.Linear(1024, h), nn.Mish(inplace=True), nn.Linear(h, 1))
            self.a_head = nn.Sequential(nn.Linear(1024, h), nn.Mish(inplace=True), nn.Linear(h, ACTION_SPACE))

    def heads(self, phi):
        """(value [B, 1], advantage [B, 46]) before the masked dueling combination"""
        if self.version == 4:
            return self.net(phi).split((1, ACTION_SPACE), dim=-1)
        return self.v_head(phi), self.a_head(phi)

    def forward(self, phi, mask):
        v, a = self.heads(phi)
        a_mean = a.masked_fill(~mask, 0.0).sum(-1, keepdim=True) / mask.sum(-1, keepdim=True)
        return (v + a - a_mean).masked_fill(~mask, -torch.inf)
