"""Fused GRU actor-critic inference for the collection and evaluation loops (rs_policy_act / rs_policy_value).

`FusedGruPolicy` runs the recurrent actor-critic of the RAD-A2C core -- torch.nn.GRUCell(d_in, H) followed by a policy head
over the 8 moves and a value head (algos/test_environment/core.py) -- as one kernel launch per call instead of a dozen
cuBLAS / elementwise launches.  The torch modules stay the source of truth: the PPO update trains them, and `sync()` repacks
their weights into the buffer the kernels read.  It satisfies rollout.RolloutPolicy (RolloutCollector) and
evaluate.Policy (MonteCarloEvaluator.run).

Supported modules (anything else raises ValueError):
  trunk        torch.nn.GRUCell(d_in, H) with biases, d_in = 11 (the observation) or 13 (observation + a two-column source
               prediction the caller passes as `pred`), H in 1..64
  policy head  Linear(H, 8), or Sequential(Linear(H, P), Tanh() | ReLU(), Linear(P, 8)) with P in 1..64
  value head   Linear(H, 1), or Sequential(Linear(H, V), activation, Linear(V, 1)); both heads use the same activation
All parameters float32.  The arithmetic is float32 FMAs (no TF32), so the log-probabilities the collector stores match the
ones the torch modules recompute in the PPO ratio to float32 rounding.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Tuple

import torch

from . import _lib as L

N_ACTIONS = 8
_ACTS = {torch.nn.Tanh: 0, torch.nn.ReLU: 1}


def _ptr(t: Optional[torch.Tensor]) -> Optional[C.c_void_p]:
    return None if t is None else C.c_void_p(t.data_ptr())


def _check_linear(m: torch.nn.Module, n_in: int, n_out: int, what: str) -> List[torch.Tensor]:
    if type(m) is not torch.nn.Linear:
        raise ValueError(f"{what}: unsupported layer {type(m).__name__} (expected torch.nn.Linear)")
    if m.bias is None:
        raise ValueError(f"{what}: Linear without bias is unsupported")
    if m.in_features != n_in or m.out_features != n_out:
        raise ValueError(f"{what}: Linear({m.in_features}, {m.out_features}) where Linear({n_in}, {n_out}) is needed")
    return [m.weight, m.bias]


def _parse_head(m: torch.nn.Module, H: int, n_out: int, what: str) -> Tuple[int, Optional[int], List[torch.Tensor]]:
    """-> (hidden width, 0 for a linear head; activation code or None; parameters in packing order)"""
    if type(m) is torch.nn.Linear:
        return 0, None, _check_linear(m, H, n_out, what)
    if type(m) is not torch.nn.Sequential:
        raise ValueError(f"{what}: unsupported module {type(m).__name__} (Linear or Sequential(Linear, Tanh|ReLU, Linear))")
    if len(m) != 3:
        raise ValueError(f"{what}: Sequential of {len(m)} modules is unsupported (one hidden layer: Linear, Tanh|ReLU, Linear)")
    if type(m[0]) is not torch.nn.Linear:
        raise ValueError(f"{what}: unsupported layer {type(m[0]).__name__} (expected torch.nn.Linear)")
    width = m[0].out_features
    if not 1 <= width <= 64:
        raise ValueError(f"{what}: hidden width {width} is unsupported (1..64)")
    if type(m[1]) not in _ACTS:
        raise ValueError(f"{what}: activation {type(m[1]).__name__} is unsupported (Tanh or ReLU)")
    return width, _ACTS[type(m[1])], _check_linear(m[0], H, width, what) + _check_linear(m[2], width, n_out, what)


class FusedGruPolicy:
    """gru / pi / v: the torch modules (see the module docstring).  num_rows: rows of every call (N envs x A agents,
    env-major n * A + a).  seed, row_id_offset: the action noise of row m is keyed by (seed, row_id_offset + m, call
    counter), so shards of one batch with row_id_offset = the shard's first row sample what one policy over the whole
    batch would.  obs_in: the observation tensor act() reads when called without one (e.g. env.obs in graph mode);
    action_out: an int32 tensor of num_rows elements the actions are written to (e.g. env.action_buffer), so that nothing
    is copied.

    act(obs, pred=None) -> (action int32, value f32, logp f32), persistent [num_rows] tensors; advances hidden_state.
    value(obs, pred=None) -> f32 [num_rows], the value under the current hidden state (hidden_state untouched).
    hidden_state: float32 [num_rows, H], contiguous, restarted in place by rs_rollout_post.
    policy(obs, t) -> actions: MonteCarloEvaluator.run's policy; t == 0 restarts every row.
    sync(): repack the weights from the modules (after an optimiser step), on the current stream.
    Everything is queued on the current stream without a host synchronisation; the call counter lives on the device, so
    a captured act() draws fresh noise on every replay."""

    def __init__(self, gru: torch.nn.GRUCell, pi: torch.nn.Module, v: torch.nn.Module, num_rows: int, seed: int = 0,
                 row_id_offset: int = 0, device=None, obs_in: Optional[torch.Tensor] = None,
                 action_out: Optional[torch.Tensor] = None):
        if type(gru) is not torch.nn.GRUCell:
            raise ValueError(f"trunk: unsupported module {type(gru).__name__} (expected torch.nn.GRUCell)")
        if not gru.bias:
            raise ValueError("trunk: GRUCell without bias is unsupported")
        d_in, H = gru.input_size, gru.hidden_size
        if d_in not in (11, 13):
            raise ValueError(f"trunk: GRUCell input size {d_in} is unsupported (11, or 13 with a source prediction)")
        if not 1 <= H <= 64:
            raise ValueError(f"trunk: GRUCell hidden size {H} is unsupported (1..64)")
        P, act_p, pi_params = _parse_head(pi, H, N_ACTIONS, "policy head")
        V, act_v, v_params = _parse_head(v, H, 1, "value head")
        if act_p is not None and act_v is not None and act_p != act_v:
            raise ValueError("the policy and value heads use different activations (both Tanh or both ReLU)")
        self._params = [gru.weight_ih, gru.weight_hh, gru.bias_ih, gru.bias_hh] + pi_params + v_params
        for prm in self._params:
            if prm.dtype != torch.float32:
                raise ValueError(f"parameters must be float32, found {prm.dtype}")
        num_rows, row_id_offset = int(num_rows), int(row_id_offset)
        if num_rows < 1 or row_id_offset < 0 or row_id_offset + num_rows > 2 ** 32:
            raise ValueError("need num_rows >= 1 and 0 <= row_id_offset, row_id_offset + num_rows <= 2^32")
        self.device = torch.device(device) if device is not None else gru.weight_ih.device
        if self.device.type != "cuda":
            raise ValueError("FusedGruPolicy runs on a CUDA device")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.d_in, self.H, self.rows, self.seed, self.row_id_offset = d_in, H, num_rows, int(seed), row_id_offset
        self.cfg = L.RsPolicyConfig(d_in, H, P, V, act_p if act_p is not None else (act_v or 0))
        lib = L.load()
        count = lib.rs_policy_param_count(C.byref(self.cfg))
        assert count == sum(prm.numel() for prm in self._params), "packed size differs from the modules' parameter count"
        dev = self.device
        self.params = torch.empty(count, dtype=torch.float32, device=dev)
        self.h = torch.zeros(num_rows, H, dtype=torch.float32, device=dev)
        self.hidden_state = self.h
        self.obs_in = obs_in
        if action_out is not None and (action_out.dtype != torch.int32 or not action_out.is_contiguous() or
                                       action_out.numel() != num_rows or action_out.device != dev):
            raise ValueError("action_out must be a contiguous int32 tensor of num_rows elements on the policy's device")
        self.action = torch.zeros(num_rows, dtype=torch.int32, device=dev) if action_out is None else action_out
        self.val = torch.zeros(num_rows, dtype=torch.float32, device=dev)
        self.logp = torch.zeros(num_rows, dtype=torch.float32, device=dev)
        self.v_next = torch.zeros(num_rows, dtype=torch.float32, device=dev)
        self.ctr = torch.zeros(1, dtype=torch.int64, device=dev)        # call counter of the action noise (uint64 on the device)
        self.ticket = torch.zeros(1, dtype=torch.int32, device=dev)     # CTA completion counter, zero between launches
        self._lib = lib
        self._fixed = [C.c_void_p(t.data_ptr()) for t in (self.params, self.h, self.action, self.val, self.logp, self.v_next,
                                                           self.ctr, self.ticket)]
        self.sync()

    def sync(self) -> None:
        """Repack the weights from the modules (torch copies on the current stream, no host synchronisation)."""
        with torch.no_grad():
            torch.cat([prm.detach().reshape(-1).to(self.device) for prm in self._params], out=self.params)

    def _input(self, x: torch.Tensor, width: int, what: str) -> torch.Tensor:
        if x.dtype != torch.float32 or not x.is_contiguous() or x.device != self.device:
            x = x.to(device=self.device, dtype=torch.float32).contiguous()
        if x.numel() != self.rows * width:
            raise ValueError(f"{what} must hold {self.rows} rows of {width} floats, got shape {tuple(x.shape)}")
        return x

    def _inputs(self, obs: Optional[torch.Tensor], pred: Optional[torch.Tensor]):
        """-> (obs, pred) as contiguous float32 device tensors; pred None for an 11-wide trunk"""
        if obs is None:
            if self.obs_in is None:
                raise ValueError("no observation given and no obs_in")
            obs = self.obs_in
        if (pred is None) != (self.d_in == 11):
            raise ValueError("a 13-wide policy needs pred [rows, 2]; an 11-wide one takes none")
        return self._input(obs, L.OBS_DIM, "obs"), None if pred is None else self._input(pred, 2, "pred")

    def _stream(self) -> C.c_void_p:
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def act(self, obs: Optional[torch.Tensor] = None, pred: Optional[torch.Tensor] = None
            ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        obs, pred = self._inputs(obs, pred)
        prm, h, a, val, lp, _, ctr, ticket = self._fixed
        L.check(self._lib.rs_policy_act(C.byref(self.cfg), prm, _ptr(obs), _ptr(pred), h, a, val, lp, self.rows,
                                        self.row_id_offset, self.seed & 0xFFFFFFFFFFFFFFFF, ctr, ticket, self._stream()),
                "rs_policy_act")
        return self.action, self.val, self.logp

    def value(self, obs: torch.Tensor, pred: Optional[torch.Tensor] = None) -> torch.Tensor:
        obs, pred = self._inputs(obs, pred)
        prm, h, _, _, _, vn, _, _ = self._fixed
        L.check(self._lib.rs_policy_value(C.byref(self.cfg), prm, _ptr(obs), _ptr(pred), h, vn, self.rows, self._stream()),
                "rs_policy_value")
        return self.v_next

    def reset_state(self, mask: Optional[torch.Tensor]) -> None:
        if mask is None:
            self.h.zero_()
        else:
            self.h.masked_fill_(mask.reshape(-1, 1).to(device=self.device, dtype=torch.bool), 0.0)

    def __call__(self, obs: torch.Tensor, t: int) -> torch.Tensor:
        if t == 0:
            self.reset_state(None)
        return self.act(obs)[0]
