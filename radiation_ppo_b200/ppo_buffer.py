"""PPO rollout buffers whose GAE / returns / normalisation run in the CUDA kernels of include/radsearch_b200.h.

`PPOBuffer` keeps the interface of /root/reference/algos/multiagent/ppo.py::PPOBuffer (P:220-502: constructor fields,
`store`, `store_episode_length`, `GAE_advantage_and_rewardsToGO`, `get`, `quick_reset`, and the `*_buf` / `ptr` /
`path_start_idx` fields the reference's unit tests poke).  `BatchedPPOBuffer` is the [T, N] form the batched env feeds:
one `store_batch` per step and one `finish_paths` launch per epoch (SURVEY.md Appendix C).
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Union

import numpy as np
import torch

from . import _lib as L


def combined_shape(length: int, shape=None):
    """P:35-59."""
    if shape is None:
        return (length,)
    return (length, shape) if np.isscalar(shape) else (length, *shape)


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _need_cuda(device) -> torch.device:
    if not torch.cuda.is_available():
        raise L.RadSearchLibraryError("the PPO buffers need a CUDA device: the GAE kernels have no CPU fallback")
    dev = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
    if dev.type != "cuda":
        raise L.RadSearchLibraryError("the PPO buffers need a CUDA device: the GAE kernels have no CPU fallback")
    return dev


def gae_advantages(rew: torch.Tensor, val: torch.Tensor, path_end: torch.Tensor, boot: torch.Tensor,
                   gamma: float = 0.99, lam: float = 0.90, adv: Optional[torch.Tensor] = None,
                   ret: Optional[torch.Tensor] = None, stats: Optional[torch.Tensor] = None, variant: int = 0):
    """rs_gae over [T, N] float32 CUDA tensors (path_end uint8/bool).  Returns (adv, ret)."""
    lib = L.load()
    T, N = rew.shape
    rew, val, boot = (x.contiguous() for x in (rew, val, boot))
    pe = path_end.to(torch.uint8).contiguous()
    adv = torch.empty_like(rew) if adv is None else adv
    ret = torch.empty_like(rew) if ret is None else ret
    for x in (rew, val, boot, adv, ret):
        if x.dtype != torch.float32 or not x.is_cuda:
            raise TypeError("gae_advantages needs float32 CUDA tensors")
    with torch.cuda.device(rew.device):
        L.check(lib.rs_gae(_ptr(rew), _ptr(val), _ptr(pe), _ptr(boot), _ptr(adv), _ptr(ret), T, N, float(gamma),
                           float(lam), _ptr(stats), int(variant), _stream(rew.device)), "rs_gae")
    return adv, ret


def advantage_statistics(adv: torch.Tensor, group=None):
    """Global mean and population std of `adv` over all ranks, the two-pass way mpi_statistics_scalar does it
    (mpi_tools.py:71-95): all-reduce {sum, n}, then all-reduce sum((x-mean)^2).  Returns device doubles (mean, std)."""
    lib = L.load()
    x = adv.contiguous().view(-1)
    dev = x.device
    s = torch.zeros(2, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        L.check(lib.rs_adv_stats(_ptr(x), x.numel(), None, _ptr(s), _stream(dev)), "rs_adv_stats")
    sn = torch.stack([s[0], torch.tensor(float(x.numel()), dtype=torch.float64, device=dev)])
    dist_on = torch.distributed.is_available() and torch.distributed.is_initialized()
    if dist_on:
        torch.distributed.all_reduce(sn, group=group)
    mean = (sn[0] / sn[1]).reshape(1)
    s2 = torch.zeros(2, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        L.check(lib.rs_adv_stats(_ptr(x), x.numel(), _ptr(mean), _ptr(s2), _stream(dev)), "rs_adv_stats")
    ss = s2[1:2].clone()
    if dist_on:
        torch.distributed.all_reduce(ss, group=group)
    std = torch.sqrt(ss / sn[1])
    return mean, std


def normalize_advantages_(adv: torch.Tensor, mean: torch.Tensor, std: torch.Tensor) -> torch.Tensor:
    """In place (adv - mean) / std (P:446)."""
    lib = L.load()
    x = adv.view(-1)
    with torch.cuda.device(x.device):
        L.check(lib.rs_adv_normalize(_ptr(x), x.numel(), _ptr(mean), _ptr(std), _stream(x.device)), "rs_adv_normalize")
    return adv


class PPOBuffer:
    """Reference-compatible single-trajectory buffer (P:220-502).

    Like the reference's, the `*_buf` fields are float32 numpy arrays of length `max_size` on the host (its unit tests read
    and assign them directly, unit_tests/test_PPO.py:315-660), `store` is a handful of array writes, and `get()` returns
    CPU float32 torch tensors.  What runs on the GPU is the arithmetic: `GAE_advantage_and_rewardsToGO` sends the finished
    trajectory through rs_gae (thread-per-column form, the reference's float64 operation order) and `get()` takes the
    advantage statistics and the normalisation from rs_adv_stats / rs_adv_normalize.  One env stepping at a time is the
    reference's own regime (BASELINE configs[0]); batches belong in BatchedPPOBuffer."""

    def __init__(self, observation_dimension: int, max_size: int, max_episode_length: int, number_agents: int,
                 gamma: float = 0.99, lam: float = 0.90, device=None) -> None:
        self.observation_dimension = observation_dimension
        self.max_size = max_size
        self.max_episode_length = max_episode_length
        self.number_agents = number_agents
        self.gamma, self.lam = gamma, lam
        self.device = _need_cuda(device)
        L.load()
        self.ptr = 0
        self.path_start_idx = 0
        self.episode_lengths_buffer: List[int] = []
        z = lambda *s: np.zeros(s, dtype=np.float32)   # noqa: E731
        self.obs_buf = z(*combined_shape(max_size, observation_dimension))
        self.act_buf = z(max_size)
        self.adv_buf = z(max_size)
        self.rew_buf = z(max_size)
        self.ret_buf = z(max_size)
        self.val_buf = z(max_size)
        self.source_tar = z(max_size, 2)
        self.logp_buf = z(max_size)
        self.heatmap_buffer = {"actor": [None] * max_size, "critic": [None] * max_size}
        self.full_observation_buffer = None
        self.obs_win = z(observation_dimension)
        self.obs_win_std = z(observation_dimension)

    def quick_reset(self) -> None:                                   # P:333-337
        self.ptr = 0
        self.path_start_idx = 0
        self.episode_lengths_buffer = []

    def store(self, obs, act, rew, val, logp, src, full_observation=None, heatmap_stacks=None, terminal=False) -> None:
        """P:339-381."""
        assert self.ptr < self.max_size
        p = self.ptr
        self.obs_buf[p, :] = obs
        self.act_buf[p] = act
        self.rew_buf[p] = rew
        self.val_buf[p] = val
        self.source_tar[p] = np.asarray(src, dtype=np.float32).reshape(2)
        self.logp_buf[p] = logp
        if heatmap_stacks:
            self.heatmap_buffer["actor"][p] = heatmap_stacks.actor
            self.heatmap_buffer["critic"][p] = heatmap_stacks.critic
        self.ptr += 1

    def store_episode_length(self, episode_length: int) -> None:      # P:383-389
        self.episode_lengths_buffer.append(episode_length)

    def _dev(self, x) -> torch.Tensor:
        return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32)).to(self.device)

    def GAE_advantage_and_rewardsToGO(self, last_state_value: float = 0.0) -> None:
        """P:391-423: finish the trajectory [path_start_idx, ptr) with bootstrap `last_state_value` (carried to the device
        as float32, like the buffer's own values; the reference appends it to float32 slices as a Python float)."""
        s, e = self.path_start_idx, self.ptr
        n = e - s
        if n > 0:
            for name in ("rew_buf", "val_buf", "adv_buf", "ret_buf"):     # the reference's tests assign lists / float64 arrays
                v = getattr(self, name)
                if not (isinstance(v, np.ndarray) and v.dtype == np.float32):
                    setattr(self, name, np.array(v, dtype=np.float32))
            pe = torch.zeros(n, 1, dtype=torch.uint8, device=self.device)
            boot = torch.zeros(n, 1, dtype=torch.float32, device=self.device)
            boot[n - 1, 0] = float(last_state_value)
            adv, ret = gae_advantages(self._dev(self.rew_buf[s:e]).reshape(n, 1), self._dev(self.val_buf[s:e]).reshape(n, 1),
                                      pe, boot, self.gamma, self.lam, variant=1)
            both = torch.stack((adv.view(-1), ret.view(-1))).cpu().numpy()      # one device -> host copy
            self.adv_buf[s:e] = both[0]
            self.ret_buf[s:e] = both[1]
        self.path_start_idx = self.ptr

    def get(self) -> Dict[str, object]:
        """P:425-502."""
        assert self.ptr == self.max_size
        episode_lengths = self.episode_lengths_buffer
        number_episodes = len(episode_lengths)
        total_episode_length = sum(episode_lengths)
        assert number_episodes > 0, "0 completed episodes. Usually caused by having epochs shorter than an episode"
        adv = self._dev(self.adv_buf)
        mean, std = advantage_statistics(adv)                         # mpi_statistics_scalar P:445
        normalize_advantages_(adv, mean.float().double(), std.float().double())
        self.adv_buf = adv.cpu().numpy()
        self.quick_reset()
        # ep_form (P:456-486): one [len, D + 6] tensor of [obs | adv | ret | logp | act | source_tar] rows per recorded
        # episode, plus the unfinished tail of the buffer when the recorded lengths do not cover it
        rows = torch.as_tensor(np.hstack((self.obs_buf, self.adv_buf[:, None], self.ret_buf[:, None], self.logp_buf[:, None],
                                          self.act_buf[:, None], self.source_tar)), dtype=torch.float32)
        sizes = list(episode_lengths)
        tail = rows.shape[0] - total_episode_length
        if tail:
            sizes.append(tail)
        episode_form: List[List[torch.Tensor]] = [[piece.clone()] for piece in torch.split(rows, sizes, dim=0)]
        t = lambda x: torch.as_tensor(np.copy(x), dtype=torch.float32)          # noqa: E731
        return dict(obs=t(self.obs_buf), act=t(self.act_buf), ret=t(self.ret_buf), adv=t(self.adv_buf), logp=t(self.logp_buf),
                    loc_pred=t(self.obs_win_std), ep_len=t(total_episode_length), ep_form=episode_form)


class BatchedPPOBuffer:
    """[T, N] rollout storage for N environments (x A agents flattened into the column axis by the caller).

    store_batch() appends one step for every column; `end`/`boot` carry the caller rules of train.py:446-491
    (end[t, n] != 0 where the reference would call GAE_advantage_and_rewardsToGO after step t, boot[t, n] the bootstrap
    value passed there).  finish_paths() is one rs_gae launch; get() normalises the advantages with the global
    (all-rank) statistics.

    ``agents=A`` (RAD-TEAM, TeamRolloutCollector): `num_columns` counts environments and the buffer has N*A env-major
    columns (column n*A + a, the memory order of the env's [N, A] outputs), plus `pred_buf` [T, N*A, 2], the PFGRU's
    source predictions the map observation was updated with (what BatchedMapsBuffer.replay needs besides the
    observations and path ends).  GAE runs per column; agent_view() gives the [T, N] per-agent slices.

    ``predictions=True`` gives a single-agent buffer `pred_buf` [T, N, 2] as well: the source predictions of a localiser
    (pfgru.FusedPFGRU) that a 13-wide policy read, which its PPO ratio needs again (RolloutCollector(localizer=...))."""

    def __init__(self, observation_dimension: int, steps_per_epoch: int, num_columns: int, gamma: float = 0.99,
                 lam: float = 0.90, device=None, agents: Optional[int] = None, predictions: bool = False) -> None:
        self.device = _need_cuda(device)
        L.load()
        if agents is not None and not 1 <= int(agents) <= L.MAX_A:
            raise ValueError("agents must be in 1..8")
        self.A = None if agents is None else int(agents)
        self.num_envs = num_columns
        T, N, D = steps_per_epoch, num_columns * (self.A or 1), observation_dimension
        self.T, self.N, self.D = T, N, D
        self.gamma, self.lam = gamma, lam
        z = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt, device=self.device)   # noqa: E731
        # T + 1 observation rows: row t is what the policy saw at step t, row T the observation that follows the epoch's
        # last step (it opens the next epoch).  A step kernel that is handed step_outputs(t) stores row t + 1 itself.
        self._obs_store = z(T + 1, N, D)
        self.obs_buf = self._obs_store[:T]
        self.act_buf = z(T, N)
        self.rew_buf, self.val_buf, self.logp_buf = z(T, N), z(T, N), z(T, N)
        self.adv_buf, self.ret_buf = z(T, N), z(T, N)
        self.boot_buf = z(T, N)
        self.end_buf = z(T, N, dt=torch.uint8)
        self.source_tar = z(T, N, 2)
        self.pred_buf = None if self.A is None and not predictions else torch.full((T, N, 2), float("nan"), dtype=torch.float32, device=self.device)
        self.stats = z(2, dt=torch.float64)
        self.ptr = 0

    def quick_reset(self) -> None:
        self.ptr = 0

    # ---- zero-copy rollout (P:339-381 without the per-step copies): the env step and the policy write the rows ---------
    def start_epoch(self, first_obs: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Row 0 of the epoch: `first_obs` (the env's reset observation) or, when omitted, the observation that followed
        the previous epoch's last step.  Returns the row (the policy's first input)."""
        self.ptr = 0
        self._obs_store[0].copy_(self._obs_store[self.T] if first_obs is None else first_obs.reshape(self.N, self.D))
        return self._obs_store[0]

    def step_outputs(self, t: Optional[int] = None) -> Dict[str, torch.Tensor]:
        """What RadSearch.step_batch(..., out=) should fill for step t (default: the current one): the observation the
        policy sees next -> obs row t + 1, the step's reward -> rew_buf[t], its path-end flags (rs_step's `ended` byte is
        non-zero exactly where train.py:446-491 finishes a trajectory) -> end_buf[t]."""
        t = self.ptr if t is None else t
        assert 0 <= t < self.T
        if self.A is not None:
            # the env's reward [N, A] / ended [N] are not the rows' layout (team reward rule, A path-end bytes per env):
            # rs_rollout_post_team writes those rows
            return {"obs": self._obs_store[t + 1]}
        return {"obs": self._obs_store[t + 1], "reward": self.rew_buf[t], "ended": self.end_buf[t]}

    def policy_rows(self, t: Optional[int] = None) -> Dict[str, torch.Tensor]:
        """Rows of step t the policy side fills: obs (read), act / val / logp / boot / src (write), and pred (write) in a
        buffer with predictions."""
        t = self.ptr if t is None else t
        rows = {"obs": self._obs_store[t], "act": self.act_buf[t], "val": self.val_buf[t], "logp": self.logp_buf[t],
                "boot": self.boot_buf[t], "src": self.source_tar[t]}
        if self.A is not None:
            rows.update(pred=self.pred_buf[t], rew=self.rew_buf[t], end=self.end_buf[t])
        elif self.pred_buf is not None:
            rows.update(pred=self.pred_buf[t])
        return rows

    def agent_view(self, a: int) -> Dict[str, torch.Tensor]:
        """Agent a's columns of a buffer made with ``agents=A``: [T, N] (obs [T, N, D], src / pred [T, N, 2]) strided views
        of obs / act / rew / val / logp / adv / ret / boot / end / src / pred, for a per-agent update."""
        if self.A is None:
            raise ValueError("agent_view needs a buffer made with agents=A")
        if not 0 <= a < self.A:
            raise ValueError("agent index out of range")
        T, N, A = self.T, self.num_envs, self.A
        v = lambda x: x.reshape(T, N, A, *x.shape[2:])[:, :, a]                  # noqa: E731
        return dict(obs=v(self.obs_buf), act=v(self.act_buf), rew=v(self.rew_buf), val=v(self.val_buf),
                    logp=v(self.logp_buf), adv=v(self.adv_buf), ret=v(self.ret_buf), boot=v(self.boot_buf),
                    end=v(self.end_buf), src=v(self.source_tar), pred=v(self.pred_buf))

    def advance(self) -> None:
        assert self.ptr < self.T
        self.ptr += 1

    def store_batch(self, obs, act, rew, val, logp, src=None, end=None, boot=None) -> None:
        assert self.ptr < self.T
        t = self.ptr
        self.obs_buf[t].copy_(obs.reshape(self.N, self.D))
        self.act_buf[t].copy_(act.reshape(self.N))
        self.rew_buf[t].copy_(rew.reshape(self.N))
        self.val_buf[t].copy_(val.reshape(self.N))
        self.logp_buf[t].copy_(logp.reshape(self.N))
        # rows that are not supplied are cleared: rs_gae reads boot[t] wherever end[t] is set and at t = T-1, so a value
        # left over from the previous epoch must never survive (the reference passes last_state_value on every call)
        if src is not None:
            self.source_tar[t].copy_(src.reshape(self.N, 2))
        else:
            self.source_tar[t].zero_()
        if end is not None:
            self.end_buf[t].copy_(end.reshape(self.N))
        else:
            self.end_buf[t].zero_()
        if boot is not None:
            self.boot_buf[t].copy_(boot.reshape(self.N))
        else:
            self.boot_buf[t].zero_()
        self.ptr += 1

    def finish_paths(self, variant: int = 0) -> None:
        """GAE-lambda + rewards-to-go for the whole [T, N] buffer (every column ends at T-1, train.py:403-405)."""
        assert self.ptr == self.T
        self.stats.zero_()
        gae_advantages(self.rew_buf, self.val_buf, self.end_buf, self.boot_buf, self.gamma, self.lam, self.adv_buf,
                       self.ret_buf, self.stats, variant)

    def pack_episodes(self):
        """The reference's `ep_form` (P:456-486) for the whole buffer: `packed` [N*T, D+6] float32 holds the rows
        [obs | adv | ret | logp | act | source_tar] episode-major (column n's steps at rows n*T .. n*T+T-1), and
        (`ep_start`, `ep_len`) int32 [E] describe every trajectory as the slice packed[ep_start[e] : ep_start[e] +
        ep_len[e]], in (column, time) order.  Two kernel launches + one prefix sum; no per-episode host loop."""
        lib = L.load()
        T, N, D = self.T, self.N, self.D
        packed = torch.empty(N * T, D + 6, dtype=torch.float32, device=self.device)
        ep_count = torch.empty(N, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            L.check(lib.rs_pack_rollout(_ptr(self.obs_buf), _ptr(self.adv_buf), _ptr(self.ret_buf), _ptr(self.logp_buf),
                                        _ptr(self.act_buf), _ptr(self.source_tar), _ptr(packed), T, N, D,
                                        _stream(self.device)), "rs_pack_rollout")
            L.check(lib.rs_episode_table(_ptr(self.end_buf), T, N, _ptr(ep_count), None, None, None,
                                         _stream(self.device)), "rs_episode_table")
            incl = torch.cumsum(ep_count, 0, dtype=torch.int32)
            offset = (incl - ep_count).contiguous()
            n_ep = int(incl[-1].item())
            ep_start = torch.empty(n_ep, dtype=torch.int32, device=self.device)
            ep_len = torch.empty(n_ep, dtype=torch.int32, device=self.device)
            L.check(lib.rs_episode_table(_ptr(self.end_buf), T, N, _ptr(ep_count), _ptr(offset), _ptr(ep_start),
                                         _ptr(ep_len), _stream(self.device)), "rs_episode_table")
        return packed, ep_start, ep_len

    def get(self, group=None, episodes: bool = False) -> Dict[str, torch.Tensor]:
        """P:425-502 for the batched buffer: global (all-rank) advantage normalisation, flat views of the step data, and
        with ``episodes=True`` the episode-major `packed` rows with their (`ep_start`, `ep_len`) table (pack_episodes)."""
        assert self.ptr == self.T
        mean, std = advantage_statistics(self.adv_buf, group=group)
        normalize_advantages_(self.adv_buf, mean.float().double(), std.float().double())
        self.quick_reset()
        f = lambda x: x.reshape(self.T * self.N, *x.shape[2:])                 # noqa: E731
        out = dict(obs=f(self.obs_buf), act=f(self.act_buf), ret=f(self.ret_buf), adv=f(self.adv_buf),
                   logp=f(self.logp_buf), src=f(self.source_tar), end=self.end_buf, adv_mean=mean, adv_std=std)
        if episodes:
            out["packed"], out["ep_start"], out["ep_len"] = self.pack_episodes()
        return out
