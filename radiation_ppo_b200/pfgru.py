"""Fused PFGRU source localiser inference for the collection and evaluation loops (rs_pfgru_predict / peek / restart).

`FusedPFGRU` runs the particle-filter GRU of RAD-A2C (RADA2C_core.py:215-307, the PF-GRU cell of PF-RNN with K = 40
particles, soft resampling alpha = 0.7, tanh) and its prediction head `hid_obs` as one kernel launch per call.  Its
prediction, the source location in scaled coordinates, is the two extra input columns of a 13-wide FusedGruPolicy.  The
torch modules stay the source of truth: torch trains them, and `sync()` repacks their weights into the buffer the kernels
read.

Supported modules (anything else raises ValueError), H = fc_z.out_features, d_in = fc_z.in_features - H:
  fc_z, fc_r  Linear(H + d_in, H) with bias, d_in in 1..11 (the reference feeds obs[:, :3]), H in 1..64
  fc_n        Linear(H + d_in, 2 H)
  fc_obs      Linear(H + d_in, 1)
  hid_obs     Sequential(Linear(H, W), ReLU(), Linear(W, 2)), W in 1..64, optionally with a trailing Identity (SpinningUp's
              `mlp` adds one)
  activation  "tanh" only: the reference's ReLU branch normalises over the particles with BatchNorm, which is not fused
All parameters float32.  The arithmetic is float32 FMAs (no TF32); the rules are in include/radsearch_b200.h.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional

import torch

from . import _lib as L


def _ptr(t: Optional[torch.Tensor]) -> Optional[C.c_void_p]:
    return None if t is None else C.c_void_p(t.data_ptr())


def _linear(m: torch.nn.Module, n_in: int, n_out: int, what: str) -> List[torch.Tensor]:
    if type(m) is not torch.nn.Linear:
        raise ValueError(f"{what}: unsupported layer {type(m).__name__} (expected torch.nn.Linear)")
    if m.bias is None:
        raise ValueError(f"{what}: Linear without bias is unsupported")
    if m.in_features != n_in or m.out_features != n_out:
        raise ValueError(f"{what}: Linear({m.in_features}, {m.out_features}) where Linear({n_in}, {n_out}) is needed")
    return [m.weight, m.bias]


class FusedPFGRU:
    """fc_z / fc_r / fc_n / fc_obs / hid_obs: the torch modules (see the module docstring).  num_rows: rows of every call
    (N envs x A agents, env-major n * A + a, as the policy).  num_particles K in 1..64, resamp_alpha in (0, 1], resample:
    soft resampling after every step.  seed, row_id_offset: the noise of row m is keyed by (seed, row_id_offset + m, call
    counter), so shards of one batch with row_id_offset = the shard's first row compute what one localiser over the whole
    batch would.  obs_in: the observation tensor predict() reads when called without one (e.g. env.obs in graph mode).

    predict(obs=None, out=None) -> f32 [num_rows, 2]: one step on the state (written in place), the prediction into `out`
        (e.g. a rollout buffer's pred row) or a persistent tensor; advances the call counter.
    peek(obs, mask=None, mask_bits=0) -> f32 [num_rows, 2], persistent: the same step on the current state, for the
        selected rows only (mask uint8 [num_rows]; row m is selected when mask[m] & mask_bits != 0, mask_bits 0 = any
        non-zero byte; None = all rows); the state, the counter and the other rows' output are left as they were.
    reset_state(mask=None, mask_bits=0): fresh particles (U[0, 1) per element) and uniform log-weights for the selected
        rows (init_hidden).
    particles f32 [num_rows, K, H], log_weights f32 [num_rows, K]: the state, contiguous.
    localizer(obs, t) -> prediction: restarts every row at t == 0, then predict(obs) (MonteCarloEvaluator.run).
    sync(): repack the weights from the modules (after an optimiser step), on the current stream.
    Everything is queued on the current stream without a host synchronisation; the call counter lives on the device, so
    a captured predict() draws fresh noise on every replay."""

    def __init__(self, fc_z: torch.nn.Module, fc_r: torch.nn.Module, fc_n: torch.nn.Module, fc_obs: torch.nn.Module,
                 hid_obs: torch.nn.Module, num_rows: int, num_particles: int = 40, resamp_alpha: float = 0.7,
                 resample: bool = True, seed: int = 0, row_id_offset: int = 0, device=None,
                 obs_in: Optional[torch.Tensor] = None, activation: str = "tanh"):
        if activation != "tanh":
            raise ValueError(f"activation {activation!r} is unsupported (tanh only: the reference's ReLU branch normalises "
                             "over the particles with BatchNorm)")
        if type(fc_z) is not torch.nn.Linear:
            raise ValueError(f"fc_z: unsupported layer {type(fc_z).__name__} (expected torch.nn.Linear)")
        H = fc_z.out_features
        d_in = fc_z.in_features - H
        if not 1 <= H <= 64:
            raise ValueError(f"fc_z: hidden size {H} is unsupported (1..64)")
        if not 1 <= d_in <= 11:
            raise ValueError(f"fc_z: input size {d_in} is unsupported (1..11 observation columns)")
        I = H + d_in
        params = _linear(fc_z, I, H, "fc_z") + _linear(fc_r, I, H, "fc_r") + _linear(fc_n, I, 2 * H, "fc_n") + \
            _linear(fc_obs, I, 1, "fc_obs")
        if type(hid_obs) is not torch.nn.Sequential:
            raise ValueError(f"hid_obs: unsupported module {type(hid_obs).__name__} "
                             "(Sequential(Linear(H, W), ReLU(), Linear(W, 2)))")
        layers = list(hid_obs)
        if len(layers) == 4 and type(layers[3]) is torch.nn.Identity:
            layers = layers[:3]
        if len(layers) != 3:
            raise ValueError(f"hid_obs: Sequential of {len(hid_obs)} modules is unsupported "
                             "(Linear(H, W), ReLU(), Linear(W, 2), optionally Identity())")
        if type(layers[0]) is not torch.nn.Linear:
            raise ValueError(f"hid_obs: unsupported layer {type(layers[0]).__name__} (expected torch.nn.Linear)")
        W = layers[0].out_features
        if not 1 <= W <= 64:
            raise ValueError(f"hid_obs: hidden width {W} is unsupported (1..64)")
        if type(layers[1]) is not torch.nn.ReLU:
            raise ValueError(f"hid_obs: activation {type(layers[1]).__name__} is unsupported (ReLU)")
        params += _linear(layers[0], H, W, "hid_obs") + _linear(layers[2], W, 2, "hid_obs")
        for prm in params:
            if prm.dtype != torch.float32:
                raise ValueError(f"parameters must be float32, found {prm.dtype}")
        K = int(num_particles)
        if not 1 <= K <= 64:
            raise ValueError(f"num_particles {K} is unsupported (1..64)")
        alpha = float(resamp_alpha)
        if not 0.0 < alpha <= 1.0:
            raise ValueError(f"resamp_alpha {alpha} is unsupported (0 < alpha <= 1)")
        num_rows, row_id_offset = int(num_rows), int(row_id_offset)
        if num_rows < 1 or row_id_offset < 0 or row_id_offset + num_rows > 2 ** 32:
            raise ValueError("need num_rows >= 1 and 0 <= row_id_offset, row_id_offset + num_rows <= 2^32")
        self.device = torch.device(device) if device is not None else fc_z.weight.device
        if self.device.type != "cuda":
            raise ValueError("FusedPFGRU runs on a CUDA device")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._params = params
        self.d_in, self.H, self.K, self.W = d_in, H, K, W
        self.rows, self.seed, self.row_id_offset = num_rows, int(seed), row_id_offset
        self.cfg = L.RsPfgruConfig(d_in, H, K, W, int(bool(resample)), alpha)
        lib = L.load()
        count = lib.rs_pfgru_param_count(C.byref(self.cfg))
        assert count == sum(prm.numel() for prm in params), "packed size differs from the modules' parameter count"
        dev = self.device
        self.params = torch.empty(count, dtype=torch.float32, device=dev)
        self.particles = torch.zeros(num_rows, K, H, dtype=torch.float32, device=dev)
        self.log_weights = torch.zeros(num_rows, K, dtype=torch.float32, device=dev)
        self.pred = torch.zeros(num_rows, 2, dtype=torch.float32, device=dev)
        self.pred_peek = torch.zeros(num_rows, 2, dtype=torch.float32, device=dev)
        self.ctr = torch.zeros(1, dtype=torch.int64, device=dev)        # call counter of the noise (uint64 on the device)
        self.ticket = torch.zeros(1, dtype=torch.int32, device=dev)     # CTA completion counter, zero between launches
        self.obs_in = obs_in
        self._lib = lib
        self._fixed = [_ptr(t) for t in (self.params, self.particles, self.log_weights, self.ctr, self.ticket)]
        self.sync()
        self.reset_state(None)

    def sync(self) -> None:
        """Repack the weights from the modules (torch copies on the current stream, no host synchronisation)."""
        with torch.no_grad():
            torch.cat([prm.detach().reshape(-1).to(self.device) for prm in self._params], out=self.params)

    def _obs(self, obs: Optional[torch.Tensor]) -> torch.Tensor:
        if obs is None:
            if self.obs_in is None:
                raise ValueError("no observation given and no obs_in")
            obs = self.obs_in
        if obs.dtype != torch.float32 or not obs.is_contiguous() or obs.device != self.device:
            obs = obs.to(device=self.device, dtype=torch.float32).contiguous()
        if obs.numel() != self.rows * L.OBS_DIM:
            raise ValueError(f"obs must hold {self.rows} rows of {L.OBS_DIM} floats, got shape {tuple(obs.shape)}")
        return obs

    def _mask(self, mask: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
        if mask is None:
            return None
        if mask.dtype != torch.uint8 or not mask.is_contiguous() or mask.device != self.device:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        if mask.numel() != self.rows:
            raise ValueError(f"mask must hold {self.rows} bytes, got shape {tuple(mask.shape)}")
        return mask

    def _stream(self) -> C.c_void_p:
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def predict(self, obs: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        obs = self._obs(obs)
        if out is None:
            out = self.pred
        elif out.dtype != torch.float32 or not out.is_contiguous() or out.numel() != 2 * self.rows or out.device != self.device:
            raise ValueError("out must be a contiguous float32 tensor of num_rows x 2 elements on the localiser's device")
        prm, part, lw, ctr, ticket = self._fixed
        L.check(self._lib.rs_pfgru_predict(C.byref(self.cfg), prm, _ptr(obs), part, lw, _ptr(out), self.rows,
                                           self.row_id_offset, self.seed & 0xFFFFFFFFFFFFFFFF, ctr, ticket, self._stream()),
                "rs_pfgru_predict")
        return out

    def peek(self, obs: torch.Tensor, mask: Optional[torch.Tensor] = None, mask_bits: int = 0) -> torch.Tensor:
        obs, mask = self._obs(obs), self._mask(mask)
        prm, part, lw, ctr, _ = self._fixed
        L.check(self._lib.rs_pfgru_peek(C.byref(self.cfg), prm, _ptr(obs), part, lw, _ptr(self.pred_peek), _ptr(mask),
                                        int(mask_bits), self.rows, self.row_id_offset, self.seed & 0xFFFFFFFFFFFFFFFF, ctr,
                                        self._stream()), "rs_pfgru_peek")
        return self.pred_peek

    def reset_state(self, mask: Optional[torch.Tensor] = None, mask_bits: int = 0) -> None:
        mask = self._mask(mask)
        _, part, lw, ctr, _ = self._fixed
        L.check(self._lib.rs_pfgru_restart(C.byref(self.cfg), part, lw, _ptr(mask), int(mask_bits), self.rows,
                                           self.row_id_offset, self.seed & 0xFFFFFFFFFFFFFFFF, ctr, self._stream()),
                "rs_pfgru_restart")

    def __call__(self, obs: torch.Tensor, t: int) -> torch.Tensor:
        if t == 0:
            self.reset_state(None)
        return self.predict(obs)
