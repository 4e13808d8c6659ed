"""RAD-TEAM map observation on the GPU (SURVEY.md 8f-1).

Mirrors /root/reference/algos/multiagent/NeuralNetworkCores/RADTEAM_core.py::MapsBuffer (M:394-932): `observation_to_map`
(M:532-616) turns the agents' 11-element observations into the map stacks the actor / critic CNNs read -- source
prediction, own location, others' locations, readings (median of the samples of a grid cell -> per-episode running
z-score), visit counts (log-scale normalised), obstacle detections, and the combined locations for the critic
(`get_map_stack`, M:1799-1836) -- and `reset` (M:513-523) clears them for a new episode.

`BatchedMapsBuffer` holds the stacks of all N environments x A agents persistently in HBM and updates them sparsely in
place with one kernel launch per call (rs_maps_update / rs_maps_reset, include/radsearch_b200.h); the tensors it returns
are those persistent stacks.  `replay` rebuilds the stacks the policy saw at any (env, step) of a rollout buffer for the
PPO update (rs_maps_replay): storing them is out of reach at batch scale (4*(6A+4)*X*Y bytes per env and step, 81.6 KB at
A = 4), their inputs are already in the buffer.  `MapsBuffer` is the single-buffer form with the reference's method names.
There is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from . import _lib as L

# readings an episode's sample table can hold: the map kernels keep 4 warps' tables in one block's shared memory,
# 40 * log_cap + 16 bytes, and sm_100 allows 227 KB (rs_maps.cu)
MAX_LOG_CAP = 5810
ACTOR_MAPS = ("prediction", "location", "others_locations", "readings", "visit_counts", "obstacles")   # M:1811-1820
CRITIC_MAPS = ("combined_location", "readings", "visit_counts", "obstacles")                            # M:1825-1832


def calculate_resolution_accuracy(resolution_multiplier: float, scale: float) -> float:               # M:69-70
    return resolution_multiplier * 1 / scale


def calculate_map_dimensions(grid_bounds: Tuple, resolution_accuracy: float, offset: float) -> Tuple[int, int]:   # M:60-66
    return (int(grid_bounds[0] * resolution_accuracy) + int(offset * resolution_accuracy),
            int(grid_bounds[1] * resolution_accuracy) + int(offset * resolution_accuracy))


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


class BatchedMapsBuffer:
    """Map stacks of N environments x A agents.

    Reference parameters (same meaning): ``steps_per_episode``, ``number_of_agents``, ``grid_bounds``,
    ``resolution_accuracy``, ``offset``; ``environment_scale`` is the env's ``scale`` (1 / 2200).  ``use_prediction``
    is the module switch PFGRU (M:39)."""

    def __init__(self, num_envs: int, number_of_agents: int, steps_per_episode: int = 120,
                 grid_bounds: Tuple = (1, 1), resolution_accuracy: float = 22.0, offset: float = 0.22727272727272727,
                 environment_scale: float = 1 / 2200.0, use_prediction: bool = True, device=None) -> None:
        if not torch.cuda.is_available():
            raise L.RadSearchLibraryError("BatchedMapsBuffer needs a CUDA device: the map kernels have no CPU fallback")
        self._lib = L.load()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if self.device.type != "cuda":
            raise L.RadSearchLibraryError("BatchedMapsBuffer needs a CUDA device: the map kernels have no CPU fallback")
        self.num_envs, self.number_of_agents, self.steps_per_episode = int(num_envs), int(number_of_agents), int(steps_per_episode)
        self.resolution_accuracy = float(resolution_accuracy)
        self.map_dimensions = calculate_map_dimensions(grid_bounds, resolution_accuracy, offset)       # M:503-509
        self.x_limit_scaled, self.y_limit_scaled = self.map_dimensions
        self.base = (self.steps_per_episode + 1) * self.number_of_agents                               # M:500
        N, A, (X, Y) = self.num_envs, self.number_of_agents, self.map_dimensions
        cap = self.base + 2 * A              # one call per step, the reset observation and the bootstrap call
        if cap > MAX_LOG_CAP:
            raise ValueError(f"steps_per_episode={self.steps_per_episode} with number_of_agents={A}: the sample table "
                             f"holds (steps_per_episode + 3) * number_of_agents = {cap} readings, at most {MAX_LOG_CAP} "
                             f"fit the 227 KB of shared memory a block of the map kernels gets on sm_100 "
                             f"(steps_per_episode <= {MAX_LOG_CAP // A - 3} at {A} agents)")
        cfg = L.RsMapsConfig()
        cfg.n_agents, cfg.dim_x, cfg.dim_y, cfg.base, cfg.log_cap = A, X, Y, self.base, cap
        cfg.use_prediction = int(bool(use_prediction))
        cfg.resolution_accuracy, cfg.scale = self.resolution_accuracy, float(environment_scale)
        self._cfg = cfg
        dev = self.device
        z = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt, device=dev)     # noqa: E731
        # stored channel-innermost (rs_maps.cu): the public tensors are channels-first VIEWS of that storage, i.e. torch's
        # channels_last memory format -- what cuDNN convolutions take natively; .contiguous() gives the planar copy
        self._actor_store = z(N, A, X, Y, 6)
        self._critic_store = z(N, X, Y, 4)
        self.actor_maps = self._actor_store.permute(0, 1, 4, 2, 3)       # [N, A, 6, X, Y]
        self.critic_maps = self._critic_store.permute(0, 3, 1, 2)        # [N, 4, X, Y]
        self._log_cell, self._log_val, self._log_len = z(N, cap, dt=torch.int16), z(N, cap), z(N, dt=torch.int32)
        self._last_cell = torch.full((N, A), -1, dtype=torch.int32, device=dev)
        self._last_pred = torch.full((N, A), -1, dtype=torch.int32, device=dev)
        self._std, self._std_count = z(N, 2, dt=torch.float64), z(N, dt=torch.int32)
        # normalize_incremental_logscale(current = 2 i, base, increment 2) M:356-360, evaluated with the host's math.log
        # exactly as the reference writes it, stored as the float32 the map holds
        lut = [(math.log(2 + 2 * i, self.base)) * 1 / math.log(2 * self.base, self.base) for i in range(cap + 1)]
        self._visit_lut = torch.tensor(np.asarray(lut, dtype=np.float64).astype(np.float32), device=dev)
        self.status = z(N, dt=torch.int32)
        self._st = L.RsMapsState(*[t.data_ptr() for t in (
            self._actor_store, self._critic_store, self._log_cell, self._log_val, self._log_len,
            self._last_cell, self._last_pred, self._std, self._std_count, self._visit_lut, self.status)])

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _mask(self, mask: Optional[torch.Tensor]):
        if mask is None:
            return None
        if mask.dtype == torch.uint8 and mask.device == self.device and mask.is_contiguous():
            return mask                                   # e.g. the env's `ended` tensor itself, with mask_bits
        return mask.to(device=self.device, dtype=torch.uint8).contiguous()

    def update(self, obs: torch.Tensor, loc_prediction: Optional[torch.Tensor] = None,
               mask: Optional[torch.Tensor] = None, mask_bits: int = 0) -> Tuple[torch.Tensor, torch.Tensor]:
        """observation_to_map for every agent's buffer of the selected envs.  obs: float32 CUDA [N, A, 11] (the env's
        observation tensor, raw counts); loc_prediction: float32 [N, A, 2] scaled source predictions of each agent's
        PFGRU (None / NaN rows = none); mask: uint8 / bool [N] selects envs (mask[n] & mask_bits, 0 = any non-zero), e.g.
        ``mask=env.ended, mask_bits=4`` for the envs the step just reset.  Returns (actor stacks [N, A, 6, X, Y], critic
        stacks [N, 4, X, Y])."""
        o = obs.to(device=self.device, dtype=torch.float32).reshape(self.num_envs, self.number_of_agents, L.OBS_DIM).contiguous()
        p = None if loc_prediction is None else loc_prediction.to(device=self.device, dtype=torch.float32).reshape(
            self.num_envs, self.number_of_agents, 2).contiguous()
        m = self._mask(mask)
        with torch.cuda.device(self.device):
            L.check(self._lib.rs_maps_update(C.byref(self._cfg), C.byref(self._st), _ptr(o), _ptr(p), _ptr(m),
                                             int(mask_bits), self.num_envs, self._stream()), "rs_maps_update")
        return self.actor_maps, self.critic_maps

    def reset(self, mask: Optional[torch.Tensor] = None, mask_bits: int = 0) -> None:
        """MapsBuffer.reset (M:513-523) for the selected envs (all when mask is None; see update for mask_bits)."""
        m = self._mask(mask)
        with torch.cuda.device(self.device):
            L.check(self._lib.rs_maps_reset(C.byref(self._cfg), C.byref(self._st), _ptr(m), int(mask_bits),
                                            self.num_envs, self._stream()), "rs_maps_reset")


    def replay(self, buf, ranges: torch.Tensor, out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None):
        """The stacks the policy read during the collection of `buf` (a BatchedPPOBuffer made with agents=A, filled by
        TeamRolloutCollector), for the requested ranges: int32 [M, 3] rows (env n, first step t0, last step t1), e.g.
        episode_ranges(...) of pack_episodes().  Range i fills rows sum(len[:i]) .. + len[i] - 1, len = t1 - t0 + 1 (0 for
        an inverted range).  Returns (actor [R, A, 6, X, Y], critic [R, 4, X, Y]) -- channels_last views like the live
        stacks -- and status int32 [M]: the RS_MS_* bits of the replayed calls, | MR_BAD_RANGE (8) for a range outside the
        buffer (zero stacks) or inverted.  `out`: (actor store [R, A, X, Y, 6], critic store [R, X, Y, 4]) float32 to fill
        (no host synchronisation then; otherwise R is read back once).  The live state is neither read nor written."""
        if buf.A != self.number_of_agents or buf.num_envs != self.num_envs or buf.D != L.OBS_DIM:
            raise ValueError("replay needs a BatchedPPOBuffer(11, T, num_envs, agents=number_of_agents) of this batch")
        A, (X, Y) = self.number_of_agents, self.map_dimensions
        rg = ranges.to(device=self.device, dtype=torch.int32).reshape(-1, 3).contiguous()
        m = rg.shape[0]
        lens = (rg[:, 2].long() - rg[:, 1].long() + 1).clamp(min=0)
        row0 = (torch.cumsum(lens, 0) - lens).contiguous()
        if out is None:
            R = int(lens.sum().item()) if m else 0
            a_store = torch.empty(R, A, X, Y, 6, dtype=torch.float32, device=self.device)
            c_store = torch.empty(R, X, Y, 4, dtype=torch.float32, device=self.device)
        else:
            a_store, c_store = out
            R = a_store.shape[0]
            if a_store.shape != (R, A, X, Y, 6) or c_store.shape != (R, X, Y, 4) or not a_store.is_contiguous() or \
                    not c_store.is_contiguous() or a_store.dtype != torch.float32 or c_store.dtype != torch.float32:
                raise ValueError("out must be contiguous float32 stores [R, A, X, Y, 6] and [R, X, Y, 4]")
        status = torch.zeros(m, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            L.check(self._lib.rs_maps_replay(C.byref(self._cfg), C.byref(self._st), _ptr(buf._obs_store), _ptr(buf.pred_buf),
                                             _ptr(buf.end_buf), buf.T, self.num_envs, _ptr(rg), m, _ptr(row0),
                                             _ptr(a_store), _ptr(c_store), _ptr(status), self._stream()), "rs_maps_replay")
        return a_store.permute(0, 1, 4, 2, 3), c_store.permute(0, 3, 1, 2), status


def episode_ranges(ep_start: torch.Tensor, ep_len: torch.Tensor, steps_per_epoch: int, agents: int = 1) -> torch.Tensor:
    """Replay ranges int32 [E', 3] = (env, t0, t1) of the episodes of a BatchedPPOBuffer.pack_episodes() table.  With
    agents=A the table lists every episode once per agent column (n*A + a) and the A columns of an env end together: the
    episodes of agent 0's columns are kept, once per env, in (env, time) order."""
    T = int(steps_per_epoch)
    col = ep_start.long() // T
    t0 = ep_start.long() - col * T
    keep = (col % agents) == 0
    col, t0, n_steps = col[keep], t0[keep], ep_len.long()[keep]
    return torch.stack((col // agents, t0, t0 + n_steps - 1), dim=1).to(torch.int32).contiguous()


class MapsBuffer:
    """One agent's buffer with the reference's interface (M:394-616): `observation_to_map(observation, id,
    loc_prediction)` returns the seven maps (prediction, location, others, readings, visit counts, obstacles, combined)
    as numpy arrays; `reset()` clears them."""

    def __init__(self, observation_dimension: int, steps_per_episode: int, number_of_agents: int,
                 grid_bounds: Tuple = (1, 1), resolution_accuracy: float = 22.0, resolution_multiplier: float = 0.01,
                 offset: float = 0.22727272727272727, obstacle_state_offset: int = 3,
                 environment_scale: float = 1 / 2200.0, device=None) -> None:
        assert observation_dimension == L.OBS_DIM and obstacle_state_offset == 3
        self.observation_dimension, self.steps_per_episode, self.number_of_agents = observation_dimension, steps_per_episode, number_of_agents
        self.grid_bounds, self.resolution_accuracy, self.resolution_multiplier, self.offset = grid_bounds, resolution_accuracy, resolution_multiplier, offset
        self._b = BatchedMapsBuffer(1, number_of_agents, steps_per_episode, grid_bounds, resolution_accuracy, offset,
                                    environment_scale=environment_scale, device=device)
        self.map_dimensions = self._b.map_dimensions
        self.x_limit_scaled, self.y_limit_scaled = self.map_dimensions
        self.base = self._b.base
        self.map_count = 6
        self.reset_flag = 1

    def reset(self) -> None:
        self._b.reset()
        self.reset_flag += 1 if self.reset_flag < 100 else 1

    def observation_to_map(self, observation: Dict[int, np.ndarray], id: int, loc_prediciton: Tuple[float, float]):
        A = self.number_of_agents
        obs = torch.as_tensor(np.stack([np.asarray(observation[i], dtype=np.float64) for i in range(A)]).astype(np.float32))
        pred = torch.full((1, A, 2), float("nan"))
        pred[0, id, 0], pred[0, id, 1] = float(loc_prediciton[0]), float(loc_prediciton[1])
        actor, critic = self._b.update(obs.reshape(1, A, L.OBS_DIM), pred)
        a = actor[0, id].cpu().numpy()
        return (a[0], a[1], a[2], a[3], a[4], a[5], critic[0, 0].cpu().numpy())
