"""Engines: the decision makers the environment calls back into.

`DeviceEngine` is the zero-copy fast path: it consumes the on-device observation / mask tensors and returns
on-device actions, with the selection semantics of mortal/engine.py:43-94 (masked dueling Q, greedy argmax or
epsilon-Boltzmann with top-p). Any object following the reference's duck-typed protocol
(agent/mortal.rs:54-74, 126-152: `engine_type == 'mortal'`, `react_batch(list[np], list[np], None)`)
still works through `HostProtocolEngine`, which pays the device->host->device round trip the reference pays.
`ReferenceEngine` puts Mortal's own MortalEngine (versions 2-4) on the device path when the arena is told to adopt it.
"""
from __future__ import annotations

import copy

import numpy as np
import torch


class DeviceEngine:
    engine_type = "mortal"

    def __init__(self, brain, dqn, *, version=4, device=None, enable_amp=True, enable_quick_eval=True,
                 enable_rule_based_agari_guard=False, name="NoName", boltzmann_epsilon=0.0, boltzmann_temp=1.0,
                 top_p=1.0, is_oracle=False, fast_inference=True):
        self.device = device or torch.device("cuda")
        self.brain = brain.to(self.device).eval()
        self.dqn = dqn.to(self.device).eval()
        # BN-folded bf16 inference path when the brain offers one (mortal_b200.model.Brain); plain autocast otherwise
        self.fast = bool(fast_inference and enable_amp and hasattr(self.brain, "prepare_fast") and self.device.type == "cuda")
        self._fast_brain = None
        if self.fast:
            from . import _lib

            _lib.init(self.device.index or 0)  # the fused elementwise kernels live in libmjx
            self.refresh()
        self.version = version
        self.is_oracle = is_oracle
        self.enable_amp = enable_amp
        self.enable_quick_eval = enable_quick_eval
        self.enable_rule_based_agari_guard = enable_rule_based_agari_guard
        self.name = name
        self.boltzmann_epsilon = boltzmann_epsilon
        self.boltzmann_temp = boltzmann_temp
        self.top_p = top_p
        self._graphs = {}

    @torch.no_grad()
    def refresh(self):
        """(Re)build the bf16 BN-folded inference copy from the caller's module. The caller's `brain` is never touched:
        mortal/train.py:317 and player.py:120 hand the live training model to the engine and keep training it afterwards, so its
        fp32 parameters and BatchNorm statistics must survive. Call again after the weights changed."""
        if self.fast:
            self._fast_brain = copy.deepcopy(self.brain).eval()
            self._fast_brain.prepare_fast(torch.bfloat16)
            self._graphs = {}

    @torch.inference_mode()
    def react_device(self, obs: torch.Tensor, masks: torch.Tensor, return_greedy: bool = False):
        """obs [B, C, 34] f32 cuda, masks [B, 46] bool cuda -> (actions int64 [B], q [B, 46][, is_greedy bool [B]])"""
        if self.fast:
            q = self.dqn(self._fast_brain.forward_fast(obs).float(), masks)
        else:
            with torch.autocast(self.device.type, dtype=torch.bfloat16, enabled=self.enable_amp):
                q = self.dqn(self.brain(obs), masks)
        if self.boltzmann_epsilon > 0:
            b = obs.shape[0]
            greedy = torch.full((b,), 1 - self.boltzmann_epsilon, device=self.device).bernoulli().to(torch.bool)
            logits = (q / self.boltzmann_temp).masked_fill(~masks, -torch.inf)
            sampled = sample_top_p(logits, self.top_p)
            actions = torch.where(greedy, q.argmax(-1), sampled)
        else:
            actions = q.argmax(-1)
            greedy = None
        if return_greedy:
            if greedy is None:
                greedy = torch.ones(obs.shape[0], dtype=torch.bool, device=self.device)
            return actions, q, greedy
        return actions, q

    @torch.inference_mode()
    def react_static(self, obs_buf: torch.Tensor, masks_buf: torch.Tensor, nr: int, bucket: int = 256):
        """react_device(obs_buf[:nr], masks_buf[:nr]) for PERSISTENT buffers (BatchEnv.obs_buffer() / .masks): the forward
        over the first ceil(nr / bucket) * bucket rows is captured once per bucket as a CUDA graph and replayed, which
        removes the ~600 kernel-launch calls per step from the host. Greedy engines only; rows past nr are stale and ignored."""
        if self.boltzmann_epsilon > 0 or not self.fast:
            return self.react_device(obs_buf[:nr], masks_buf[:nr])
        nb = min(((nr + bucket - 1) // bucket) * bucket, obs_buf.shape[0])
        key = (obs_buf.data_ptr(), masks_buf.data_ptr(), nb)
        entry = self._graphs.get(key)
        if entry is None:
            cur = torch.cuda.current_stream(self.device)
            side = torch.cuda.Stream(self.device)
            side.wait_stream(cur)
            with torch.cuda.stream(side):  # warm-up outside the capture (cuDNN algorithm selection, lazy init)
                for _ in range(2):
                    self.react_device(obs_buf[:nb], masks_buf[:nb])
            cur.wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                a, q = self.react_device(obs_buf[:nb], masks_buf[:nb])
            entry = (graph, a, q)
            self._graphs[key] = entry
        entry[0].replay()
        return entry[1][:nr], entry[2][:nr]

    # the reference protocol, for callers that only know libriichi's calling convention
    def react_batch(self, obs, masks, invisible_obs):
        o = torch.as_tensor(_stack_rows(obs), device=self.device)
        m = torch.as_tensor(_stack_rows(masks), device=self.device)
        actions, q, greedy = self.react_device(o, m, return_greedy=True)
        return actions.tolist(), q.float().tolist(), m.tolist(), greedy.tolist()


def _stack_rows(rows):
    """np.stack(rows) without the copy when the rows already are consecutive slices of one buffer — which is how the arena hands
    them out (views over the pinned buffer mjx_env_encode_obs_host filled), so the H2D copy then reads pinned memory directly."""
    first = rows[0]
    n, step = len(rows), first.nbytes
    if n > 1 and first.flags.c_contiguous and step:
        p0 = first.__array_interface__["data"][0]
        if all(r.__array_interface__["data"][0] == p0 + i * step and r.shape == first.shape and r.dtype == first.dtype
               for i, r in enumerate(rows)):
            return np.lib.stride_tricks.as_strided(first, shape=(n, *first.shape), strides=(step, *first.strides), writeable=bool(first.flags.writeable))
    return np.stack(rows, axis=0)


def sample_top_p(logits, p):
    """Nucleus sampling over the last axis: draw from the smallest set of highest-probability actions whose mass reaches
    `p` (engine.py:83-94 semantics: p >= 1 is plain categorical sampling, p <= 0 the argmax)."""
    if p >= 1:
        return torch.distributions.Categorical(logits=logits).sample()
    if p <= 0:
        return logits.argmax(-1)
    order = logits.argsort(-1, descending=True)
    mass = logits.gather(-1, order).softmax(-1)
    before = mass.cumsum(-1) - mass               # probability mass ranked strictly above each action
    nucleus = torch.where(before <= p, mass, torch.zeros_like(mass))
    pick = nucleus.multinomial(1)                 # multinomial renormalises the kept mass itself
    return order.gather(-1, pick).squeeze(-1)


class HostProtocolEngine:
    """Adapter: drives a reference-style engine (react_batch over lists of numpy arrays) from device rows."""

    def __init__(self, engine):
        assert getattr(engine, "engine_type", None) == "mortal", "only engine_type='mortal' is supported"
        self.engine = engine
        for attr in ("name", "version", "is_oracle", "enable_quick_eval", "enable_rule_based_agari_guard"):
            setattr(self, attr, getattr(engine, attr))

    def react_host(self, obs_np: np.ndarray, masks_np: np.ndarray, idx: np.ndarray, inv_np=None):
        """rows `idx` of host arrays (views over pinned buffers filled by mjx_env_encode_obs_host) -> (actions, q, is_greedy) numpy,
        through the reference protocol: lists of per-row arrays in, lists out (agent/mortal.rs:126-152)."""
        invisible = None if inv_np is None else [inv_np[i] for i in idx]  # mortal.rs:137-146: Some(list) for oracle engines only
        actions, q, _, greedy = self.engine.react_batch([obs_np[i] for i in idx], [masks_np[i] for i in idx], invisible)
        return np.asarray(actions, dtype=np.int64), np.asarray(q, dtype=np.float32), np.asarray(greedy, dtype=bool)

    def react_device(self, obs: torch.Tensor, masks: torch.Tensor, invisible_obs=None):
        obs_h = obs.cpu().numpy()
        masks_h = masks.cpu().numpy()
        inv = None if invisible_obs is None else list(invisible_obs.cpu().numpy())
        actions, q, _, _ = self.engine.react_batch(list(obs_h), list(masks_h), inv)
        dev = obs.device
        return torch.as_tensor(actions, dtype=torch.int64, device=dev), torch.as_tensor(q, dtype=torch.float32, device=dev)


class ReferenceEngine:
    """The device path for an unmodified mortal/engine.py MortalEngine holding a version 2, 3 or 4 Brain / DQN.

    Reads only the attributes MortalEngine.__init__ sets and never touches the caller's modules: `refresh()` builds an inference
    copy through their state_dict() and mortal_b200.checkpoint (mortal/train.py keeps training the same modules between plays, so
    the arena calls it at every py_vs_py). `enable_amp=True` runs the BN-folded bf16 fused path (MortalEngine autocasts to fp16
    instead), `enable_amp=False` fp32 channels-last convolutions. Per (observation buffer, batch bucket) one CUDA graph covers the
    stem conversion of the engine's rows, the network, the Q head and k_select_actions (csrc/mjx_select.cuh), greedy or
    epsilon-Boltzmann / top-p alike. The sampling seed is drawn from torch's default generator at construction, so
    torch.manual_seed makes sampled self-play repeat exactly."""

    engine_type = "mortal"
    ATTRS = ("version", "is_oracle", "enable_amp", "enable_quick_eval", "enable_rule_based_agari_guard", "name",
             "boltzmann_epsilon", "boltzmann_temp", "top_p")

    @staticmethod
    def eligible(engine, device: int) -> bool:
        """MortalEngine-shaped (engine_type 'mortal', brain, dqn), version 2-4, not an oracle, on CUDA device `device`"""
        if hasattr(engine, "react_device") or getattr(engine, "engine_type", None) != "mortal":
            return False
        if not (hasattr(engine, "brain") and hasattr(engine, "dqn")):
            return False
        dev = getattr(engine, "device", None)
        return (getattr(engine, "version", None) in (2, 3, 4) and not getattr(engine, "is_oracle", False)
                and isinstance(dev, torch.device) and dev.type == "cuda" and (dev.index or 0) == int(device))

    def __init__(self, engine):
        self.engine = engine
        for attr in self.ATTRS:
            setattr(self, attr, getattr(engine, attr))
        self.device = torch.device("cuda", engine.device.index or 0)
        self.seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        self.brain = self.dqn = None
        self._graphs = {}
        self.graph_captures = 0
        self.graph_replays = 0

    @torch.no_grad()
    def refresh(self):
        from . import _lib
        from .checkpoint import load_reference_state_dicts

        _lib.init(self.device.index)
        brain, dqn = load_reference_state_dicts(self.engine.brain.state_dict(), self.engine.dqn.state_dict(), self.version)
        self.brain = brain.to(self.device).eval().prepare_fast(torch.bfloat16 if self.enable_amp else None)
        self.dqn = dqn.to(self.device).eval()
        self._graphs = {}

    def _forward_select(self, obs_buf, env, rows, count, nb, table_offset, actions, q_out, greedy):
        from . import nn_ops

        if self.enable_amp:
            if rows is None:
                x = nn_ops.obs_to_nhwc(obs_buf[:nb], self.brain._cpad)
            else:
                x = nn_ops.obs_rows_to_nhwc(obs_buf, rows, count, nb, self.brain._cpad)
            phi = self.brain.forward_fast_nhwc(x).float()
        else:
            phi = self.brain.forward_fast(obs_buf[:nb] if rows is None else obs_buf.index_select(0, rows[:nb]))
        v, a = self.dqn.heads(phi)
        nn_ops.select_actions(v, a, rows, count, env.masks, env.row_table, env.row_step, env.row_seat, seed=self.seed,
                              table_offset=table_offset, epsilon=self.boltzmann_epsilon, temp=self.boltzmann_temp, top_p=self.top_p,
                              actions=actions, q_out=q_out, greedy=greedy)

    @torch.inference_mode()
    def decide(self, obs_buf, env, rows, count, n: int, *, table_offset: int, actions, q_out, greedy, bucket: int = 256):
        """Decide batch rows i < n of the environment `env`: row rows[i] (rows None: i) of the persistent buffer obs_buf; `count` is
        the same number as an int32 device tensor, which the captured graph reads at every replay. Writes actions, q_out and greedy
        at the environment rows."""
        nb = min((n + bucket - 1) // bucket * bucket, obs_buf.shape[0])
        key = (obs_buf.data_ptr(), None if rows is None else rows.data_ptr(), count.data_ptr(), actions.data_ptr(), nb)
        graph = self._graphs.get(key)
        if graph is None:
            args = (obs_buf, env, rows, count, nb, table_offset, actions, q_out, greedy)
            cur = torch.cuda.current_stream(self.device)
            side = torch.cuda.Stream(self.device)
            side.wait_stream(cur)
            with torch.cuda.stream(side):  # warm-up outside the capture (cuDNN algorithm selection, lazy init)
                for _ in range(2):
                    self._forward_select(*args)
            cur.wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                self._forward_select(*args)
            self._graphs[key] = graph
            self.graph_captures += 1
        graph.replay()
        self.graph_replays += 1
