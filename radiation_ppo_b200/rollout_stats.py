"""Episode bookkeeping of the rollout loop on the device (the caller side of the env step).

Mirrors what /root/reference/algos/multiagent/train.py keeps per MPI rank around `env.step` (T:359-527): the running
`episode_return` (T:361-375, float32 rewards summed in float64), `steps_in_episode`, the per-agent `terminal_counter`
and `out_of_bounds_count` (T:378-391), `EpRet` / `EpLen` logged when an episode is over by a terminal state or the
timeout (T:493-500; an episode cut by the epoch end is not logged) and `DoneCount` / `OutOfBound` logged at the epoch end
(T:520-527).  `epoch_summary` is the logger's `log_tabular(..., with_min_and_max=True)` view of them, with the statistics
taken over all envs of all ranks the way `mpi_statistics_scalar` (rl_tools/mpi_tools.py:71-95) does.

One instance covers N envs x A agents; `update` is a handful of tensor ops on the step outputs, no host round trip.
"""
from __future__ import annotations

from typing import Dict

import torch

from . import _lib as L
from .dist import _on


class EpisodeStats:
    def __init__(self, num_envs: int, number_agents: int, device, team_mode: str = "cooperative") -> None:
        self.N, self.A, self.device, self.team_mode = int(num_envs), int(number_agents), torch.device(device), team_mode
        z = lambda *s, dt=torch.float64: torch.zeros(*s, dtype=dt, device=self.device)     # noqa: E731
        self.episode_return = z(self.N, self.A)                       # T:288-289
        self.steps_in_episode = z(self.N, dt=torch.int32)             # T:290
        self._acc = z(6, self.A)             # per agent: count, sum EpRet, sum EpRet^2, sum EpLen, DoneCount, OutOfBound
        self._min = torch.full((self.A,), float("inf"), dtype=torch.float64, device=self.device)
        self._max = torch.full((self.A,), float("-inf"), dtype=torch.float64, device=self.device)

    def update(self, reward: torch.Tensor, team_reward: torch.Tensor, done: torch.Tensor, info: torch.Tensor,
               ended: torch.Tensor) -> None:
        """After one batched step: reward [N, A] / team_reward [N] float32, done / info [N, A] uint8 (RS_I_* bits),
        ended [N] uint8 (RS_E_* bits) as rs_step writes them."""
        r = reward if self.team_mode == "individual" else team_reward[:, None].expand(self.N, self.A)   # T:361-375
        self.episode_return += r.double()
        self.steps_in_episode += 1
        over = (ended & (L.E_TERMINAL | L.E_TIMEOUT)) != 0                                        # episode_over T:394-400
        self._acc[4] += (done != 0).sum(dim=0)                                                    # T:388-391
        self._acc[5] += ((info & L.I_OOB) != 0).sum(dim=0)                                        # T:378-384
        w = over[:, None].double()
        ret = self.episode_return
        self._acc[0] += w.sum(dim=0)
        self._acc[1] += (ret * w).sum(dim=0)
        self._acc[2] += (ret * ret * w).sum(dim=0)
        self._acc[3] += (self.steps_in_episode[:, None].double() * w).sum(dim=0)
        inf = torch.tensor(float("inf"), dtype=torch.float64, device=self.device)
        self._min = torch.minimum(self._min, torch.where(over[:, None], ret, inf).amin(dim=0))
        self._max = torch.maximum(self._max, torch.where(over[:, None], ret, -inf).amax(dim=0))
        reset = (ended & L.E_RESET) != 0                                                          # env.reset() follows T:530-535
        self.episode_return.masked_fill_(reset[:, None], 0.0)
        self.steps_in_episode.masked_fill_(reset, 0)

    def fused_args(self):
        """The accumulators for rs_rollout_post / rs_rollout_post_team (which do what `update` does, in the same launch as
        the bootstrap rule): ep_return [N, A] f64, ep_steps [N] i32, acc [6, A] f64, min [A], max [A].  The fused kernels
        implement the 'individual' rule (each agent's own reward) and the team reward of the other modes except
        'competitive'."""
        if self.team_mode == "competitive":
            raise ValueError("the fused bookkeeping covers one agent per environment or the individual / cooperative "
                             "reward rules")
        return (self.episode_return, self.steps_in_episode, self._acc, self._min, self._max)

    def epoch_summary(self, group=None, clear: bool = True) -> Dict[str, torch.Tensor]:
        """Per agent [A]: Episodes, AverageEpRet, StdEpRet (population), MinEpRet, MaxEpRet, EpLen (mean), DoneCount,
        OutOfBound -- over all envs of all ranks (sums all-reduced once, min / max once each)."""
        acc, mn, mx = self._acc.clone(), self._min.clone(), self._max.clone()
        if _on():
            torch.distributed.all_reduce(acc, group=group)
            torch.distributed.all_reduce(mn, op=torch.distributed.ReduceOp.MIN, group=group)
            torch.distributed.all_reduce(mx, op=torch.distributed.ReduceOp.MAX, group=group)
        n = acc[0].clamp(min=1.0)
        mean = acc[1] / n
        var = (acc[2] / n - mean * mean).clamp(min=0.0)
        out = {"Episodes": acc[0], "AverageEpRet": mean, "StdEpRet": var.sqrt(), "MinEpRet": mn, "MaxEpRet": mx,
               "EpLen": acc[3] / n, "DoneCount": acc[4], "OutOfBound": acc[5]}
        if clear:                                                                                  # T:526-527
            self._acc.zero_()
            self._min.fill_(float("inf"))
            self._max.fill_(float("-inf"))
        return out
