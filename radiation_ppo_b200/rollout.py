"""One epoch of experience collection for a batched RadSearch env: the loop of
/root/reference/algos/multiagent/train.py:321-571 (single-agent RAD-A2C branch) with every environment of the batch
stepping at once and NO per-step copies -- the policy reads its observations from the rollout buffer's row t, writes
action / value / log-probability into the same row, and the env step kernel stores the next observation, the reward and
the path-end flags straight into the buffer (RadSearch.step_batch(out=BatchedPPOBuffer.step_outputs(t))).

Caller rules reproduced (T: = train.py):
  * T:394-405  timeout / episode_over / epoch_ended: applied on the device by rs_step (auto_reset, `ended` bits);
  * T:446-487  a trajectory that ends by timeout or at the epoch's last step is bootstrapped with the critic's value of the
               observation that follows (with the recurrent state of that moment); one that only reached the source gets 0;
  * T:484      the epoch's last step asks for new obstructions (epoch_end=True);
  * T:509-511  the recurrent state of an env restarts with its episode (not at the epoch's last step: T:326 resets all);
  * T:359-527  EpRet / EpLen / DoneCount / OutOfBound bookkeeping -> rollout_stats.EpisodeStats.
The policy is the caller's (any torch module); this module only fixes the order of operations around the kernels.

`TeamRolloutCollector` is the multi-agent (RAD-TEAM) branch of the same loop: the policy reads the map stacks of
maps_buffer.BatchedMapsBuffer, which are updated before the policy acts, on the last observation of every episode that
ended (bootstrap) and reset with the env (INTEGRATION.md section 3).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Protocol, Tuple

import torch

from . import _lib as L
from .envs.rad_search_env import RadSearch
from .maps_buffer import BatchedMapsBuffer
from .ppo_buffer import BatchedPPOBuffer
from .rollout_stats import EpisodeStats


class RolloutPolicy(Protocol):
    def act(self, obs: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """obs [N, D] f32 -> (action int32 [N], state value f32 [N], log-probability f32 [N]); advances the policy's own
        recurrent state (T:345-353).  With a localizer the collector calls act(obs, pred), pred f32 [N, 2]."""

    def value(self, obs: torch.Tensor) -> torch.Tensor:
        """State value f32 [N] of `obs` under the current recurrent state, without advancing it (T:470-477).  With a
        localizer: value(obs, pred)."""

    def reset_state(self, mask: Optional[torch.Tensor]) -> None:
        """Restart the recurrent state of the envs in `mask` (bool [N]; None = all) (T:326, 509-511).  A policy that
        exposes its state as `hidden_state` (float32 [N, H], contiguous) has it restarted in place by rs_rollout_post and
        is only called with mask=None."""


class RolloutCollector:
    """Collects `buf.T` steps of every env into `buf` and finishes the trajectories (GAE) -- one epoch of T:321-571.

    mode "rows" (default): the env step stores observation t+1 / reward / path-end flags straight into the buffer rows
    (step_batch(out=...)): no copies at all, plain stream launches.
    mode "graph" (needs an env with prefetch=True, use_cuda_graph=True): the env replays its captured step graph, whose
    outputs are the env's own fixed tensors, and the two bookkeeping launches that exist anyway carry them into the rows
    (49 bytes per env and step): fewer, cheaper launches per step when the host is the bottleneck.  A policy may read
    `env.obs` and write `env.action_buffer` in place, so nothing else moves.  Both modes fill the buffer identically.

    localizer (optional, e.g. pfgru.FusedPFGRU over the N rows; needs BatchedPPOBuffer(..., predictions=True)): the source
    predictions of a 13-wide policy.  Per step t, in this order:
      1. pred = localizer.predict(obs, out=buf.pred_buf[t])
      2. action, value, logp = policy.act(obs, pred)
      3. rs_rollout_pre, 4. the env step
      5. v_next = policy.value(final_obs, localizer.peek(final_obs, mask=<the rows rs_rollout_post bootstraps>))
      6. rs_rollout_post
      7. localizer.reset_state(<ended rows>), the rows whose policy state rs_rollout_post restarts (not at the last step)
    and localizer.reset_state(None) opens every epoch (T:326)."""

    def __init__(self, env: RadSearch, buf: BatchedPPOBuffer, policy: RolloutPolicy, stats: Optional[EpisodeStats] = None,
                 mode: str = "rows", localizer=None):
        if env.number_agents != 1:
            raise ValueError("RolloutCollector drives single-agent envs (the RAD-A2C branch of train.py)")
        if not env.auto_reset:
            raise ValueError("RolloutCollector needs auto_reset=True (the caller rules run on the device)")
        if buf.N != env.num_envs or buf.D != L.OBS_DIM:
            raise ValueError("buffer shape does not match the env batch")
        if mode not in ("rows", "graph"):
            raise ValueError("mode must be 'rows' or 'graph'")
        if mode == "graph" and not env.use_cuda_graph:
            raise ValueError("mode='graph' needs an env created with prefetch=True, use_cuda_graph=True")
        if localizer is not None and buf.pred_buf is None:
            raise ValueError("a localizer needs a buffer with pred_buf (BatchedPPOBuffer(..., predictions=True))")
        self.env, self.buf, self.policy, self.stats, self.mode = env, buf, policy, stats, mode
        self.localizer = localizer
        self._first = True
        # the rows of the (persistent) buffer every step writes: resolved once, not at every step
        self._rows = [buf.policy_rows(t) for t in range(buf.T)]
        self._outs = [buf.step_outputs(t) for t in range(buf.T)]
        self._outs_resolved = [env.resolve_outputs(o) for o in self._outs] if mode == "rows" else None

    def collect(self, gae_variant: int = 0) -> None:
        env, buf, pol, loc = self.env, self.buf, self.policy, self.localizer
        T, N, D = buf.T, buf.N, buf.D
        lib = L.load()
        stream = C.c_void_p(torch.cuda.current_stream(env.device).cuda_stream)
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())             # noqa: E731
        rows_mode = self.mode == "rows"
        # the observation that opens the epoch: the env's reset observation the first time, afterwards the one that
        # followed the previous epoch's last step (rows mode: already in the buffer's row T; graph mode: in env.obs)
        if rows_mode:
            buf.start_epoch(env.obs if self._first else None)
        else:
            buf.ptr = 0
        self._first = False
        pol.reset_state(None)                                                        # T:326
        if loc is not None:
            loc.reset_state(None)
        hidden = getattr(pol, "hidden_state", None)                                  # [N, H] float32, restarted in place
        hdim = 0 if hidden is None else hidden.shape[1]
        st = [p(x) for x in (self.stats.fused_args() if self.stats is not None else (None,) * 5)]
        final_obs = env.final_obs.reshape(N, D)
        env_obs = env.obs.reshape(N, D)
        p_src, p_done, p_info, p_hidden = p(env._src), p(env.done_flags), p(env.info_flags), p(hidden)
        p_obs, p_rew, p_end = p(env.obs), p(env.reward), p(env.ended)
        for t in range(T):
            rows, outs = self._rows[t], self._outs[t]
            last = t == T - 1
            obs = rows["obs"] if rows_mode else env_obs
            if loc is None:
                action, value, logp = pol.act(obs)
            else:
                action, value, logp = pol.act(obs, loc.predict(obs, out=rows["pred"]))
            # row t of the buffer <- action, value, log-probability, source coordinates (T:416-428), one launch
            L.check(lib.rs_rollout_pre(p(action), p(value), p(logp), p_src, p(rows["act"]), p(rows["val"]), p(rows["logp"]),
                                       p(rows["src"]), None if rows_mode else p_obs, None if rows_mode else p(rows["obs"]), D, N,
                                       stream), "rs_rollout_pre")
            if rows_mode:
                env.step_batch(action, epoch_end=last, out=self._outs_resolved[t])   # obs -> row t+1, reward / ended -> row t
                p_r, p_e, rr, er = p(outs["reward"]), p(outs["ended"]), None, None
            else:
                env.step_batch(action, epoch_end=last)                               # captured graph, the env's own outputs
                p_r, p_e, rr, er = p_rew, p_end, p(outs["reward"]), p(outs["ended"])
            # T:462-487 bootstrap where the trajectory was cut, T:509-511 recurrent state, T:361-391 episode statistics
            if loc is None:
                v_next = pol.value(final_obs)
            else:                           # the prediction for exactly the rows rs_rollout_post bootstraps below
                ended = outs["ended"] if rows_mode else env.ended
                v_next = pol.value(final_obs, loc.peek(final_obs, mask=None if last else ended, mask_bits=L.E_TIMEOUT))
            L.check(lib.rs_rollout_post(p_r, p_e, p_done, p_info, p(v_next), p(rows["boot"]), p_hidden, hdim, st[0], st[1],
                                        st[2], st[3], st[4], rr, er, N, int(last), stream), "rs_rollout_post")
            if hidden is None and not last:
                pol.reset_state(outs["ended"] != 0)                                  # T:509-511
            if loc is not None and not last:
                loc.reset_state(outs["ended"])                                       # T:509-511 (ended byte != 0)
            buf.advance()
        buf.finish_paths(variant=gae_variant)


class TeamRolloutPolicy(Protocol):
    def predict(self, obs: torch.Tensor) -> Optional[torch.Tensor]:
        """obs [N, A, 11] f32 -> the PFGRU's source prediction float32 [N, A, 2] in scaled coordinates (NaN = none for
        that agent), or None when the policy has no predictor.  Called before every map update: on the observation the
        policy is about to act on, and on the last observation of the episodes that just ended (RADTEAM_core.py:1854-1858,
        T:476-480)."""

    def act(self, obs: torch.Tensor, actor_stacks: torch.Tensor, critic_stacks: torch.Tensor
            ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """obs [N, A, 11], actor_stacks [N, A, 6, X, Y], critic_stacks [N, 4, X, Y] (channels_last views of the live map
        stacks) -> (action int32 [N, A], state value f32 [N, A], log-probability f32 [N, A]); advances the policy's own
        recurrent state."""

    def value(self, critic_stacks: torch.Tensor) -> torch.Tensor:
        """State value f32 [N, A] of every agent from critic_stacks [N, 4, X, Y], without advancing any state: the
        bootstrap of the trajectories that were cut (T:462-487)."""

    def reset_state(self, mask: Optional[torch.Tensor]) -> None:
        """Restart the recurrent state of the envs in `mask` (bool [N]; None = all) (T:326, 509-511).  A policy that
        exposes its state as `hidden_state` (float32 [N*A, H], contiguous, env-major rows) has it restarted in place by
        rs_rollout_post_team and is only called with mask=None."""


class TeamRolloutCollector:
    """Collects `buf.T` steps of a RAD-TEAM env batch (A = number_agents in 1..8 agents per env) into `buf` and finishes
    the trajectories (GAE per agent column) -- one epoch of the multi-agent branch of T:321-571.

    env: RadSearch(auto_reset=True, standardize=0) -- the maps standardise the raw counts themselves; buf:
    BatchedPPOBuffer(11, T, N, agents=A); maps: BatchedMapsBuffer(N, A, ...); team_mode: "individual" (each agent's own
    reward goes into its column and its returns) or "cooperative" (the team reward); stats: EpisodeStats with the same
    team_mode.  Per step t, in this order:
      1. pred = policy.predict(obs)                                  (PFGRU, [N, A, 2] or None)
      2. maps.update(obs, pred)                                      (observation_to_map, RADTEAM_core.py:1854-1858)
      3. action, value, logp = policy.act(obs, actor_stacks, critic_stacks)
      4. rs_rollout_pre_team: row t <- action / value / logp / pred / source (graph mode: and the observation)
      5. env.step_batch(...)                                         (rows mode: the observation goes into row t + 1)
      6. maps.update(final_obs, policy.predict(final_obs), mask=ended & RS_E_RESET); v_next = policy.value(critic_stacks)
      7. rs_rollout_post_team: reward / path-end rows, bootstrap, recurrent-state restart, episode statistics
      8. maps.reset(mask=ended & RS_E_RESET)                         (reset_agent, T:536-538)
    The first collect() resets every env's maps; afterwards every epoch opens on fresh maps, because the epoch's last step
    resets every env (RS_F_EPOCH_END).  So every episode of the buffer starts inside it, and BatchedMapsBuffer.replay can
    rebuild the stacks of any of its rows.  Modes as RolloutCollector's."""

    def __init__(self, env: RadSearch, buf: BatchedPPOBuffer, maps: BatchedMapsBuffer, policy: TeamRolloutPolicy,
                 stats: Optional[EpisodeStats] = None, mode: str = "rows", team_mode: str = "cooperative"):
        A, N = env.number_agents, env.num_envs
        if not 1 <= A <= L.MAX_A:
            raise ValueError("TeamRolloutCollector drives 1..8 agents per env")
        if not env.auto_reset:
            raise ValueError("TeamRolloutCollector needs auto_reset=True (the caller rules run on the device)")
        if env.standardize != 0:
            raise ValueError("TeamRolloutCollector needs standardize=0: the maps standardise the raw counts themselves")
        if buf.A != A or buf.num_envs != N or buf.D != L.OBS_DIM:
            raise ValueError("buffer shape does not match the env batch (BatchedPPOBuffer(11, T, num_envs, agents=A))")
        if maps.num_envs != N or maps.number_of_agents != A:
            raise ValueError("maps shape does not match the env batch")
        if mode not in ("rows", "graph"):
            raise ValueError("mode must be 'rows' or 'graph'")
        if mode == "graph" and not env.use_cuda_graph:
            raise ValueError("mode='graph' needs an env created with prefetch=True, use_cuda_graph=True")
        if team_mode not in ("individual", "cooperative"):
            raise ValueError("team_mode must be 'individual' or 'cooperative'")
        if stats is not None and (stats.team_mode != team_mode or stats.N != N or stats.A != A):
            raise ValueError("stats must be an EpisodeStats(num_envs, number_agents, team_mode=team_mode) of this batch")
        self.env, self.buf, self.maps, self.policy, self.stats = env, buf, maps, policy, stats
        self.mode, self.team_mode = mode, team_mode
        self._first = True
        self._rows = [buf.policy_rows(t) for t in range(buf.T)]
        self._outs_resolved = [env.resolve_outputs(buf.step_outputs(t)) for t in range(buf.T)] if mode == "rows" else None

    def collect(self, gae_variant: int = 0) -> None:
        env, buf, maps, pol = self.env, self.buf, self.maps, self.policy
        T, N, A, D = buf.T, env.num_envs, env.number_agents, buf.D
        lib = L.load()
        stream = C.c_void_p(torch.cuda.current_stream(env.device).cuda_stream)
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())             # noqa: E731
        rows_mode = self.mode == "rows"
        if self._first:
            maps.reset()
        if rows_mode:
            buf.start_epoch(env.obs if self._first else None)
        else:
            buf.ptr = 0
        self._first = False
        pol.reset_state(None)                                                        # T:326
        hidden = getattr(pol, "hidden_state", None)                                  # [N*A, H] float32, restarted in place
        hdim = 0 if hidden is None else hidden.shape[1]
        st = [p(x) for x in (self.stats.fused_args() if self.stats is not None else (None,) * 5)]
        individual = int(self.team_mode == "individual")
        final_obs = env.final_obs
        p_src, p_done, p_info, p_hidden = p(env._src), p(env.done_flags), p(env.info_flags), p(hidden)
        p_rew, p_team, p_end = p(env.reward), p(env.team_reward), p(env.ended)
        for t in range(T):
            rows = self._rows[t]
            last = t == T - 1
            obs = rows["obs"].view(N, A, D) if rows_mode else env.obs
            pred = _f32(pol.predict(obs))
            actor, critic = maps.update(obs, pred)
            action, value, logp = pol.act(obs, actor, critic)
            action = action if action.dtype == torch.int32 and action.is_contiguous() else action.to(torch.int32).contiguous()
            value, logp = _f32(value), _f32(logp)
            # row t <- action, value, log-probability, prediction, source coordinates (T:416-428), one launch
            L.check(lib.rs_rollout_pre_team(p(action), p(value), p(logp), p(pred), p_src, p(rows["act"]), p(rows["val"]),
                                            p(rows["logp"]), p(rows["pred"]), p(rows["src"]),
                                            None if rows_mode else p(env.obs), None if rows_mode else p(rows["obs"]), D, N, A,
                                            stream), "rs_rollout_pre_team")
            if rows_mode:
                env.step_batch(action, epoch_end=last, out=self._outs_resolved[t])   # obs -> row t+1
            else:
                env.step_batch(action, epoch_end=last)                               # captured graph, the env's own outputs
            # T:476-480: the bootstrap value is read from maps updated with the last observation of the ended episodes
            maps.update(final_obs, _f32(pol.predict(final_obs)), mask=env.ended, mask_bits=L.E_RESET)
            v_next = _f32(pol.value(critic))
            # T:462-487 bootstrap, T:509-511 recurrent state, T:361-391 rewards per team mode and episode statistics
            L.check(lib.rs_rollout_post_team(p_rew, p_team, p_end, p_done, p_info, p(v_next), p(rows["boot"]), p_hidden, hdim,
                                             st[0], st[1], st[2], st[3], st[4], p(rows["rew"]), p(rows["end"]), N, A,
                                             individual, int(last), stream), "rs_rollout_post_team")
            if hidden is None and not last:
                pol.reset_state(env.ended != 0)                                      # T:509-511
            maps.reset(mask=env.ended, mask_bits=L.E_RESET)                          # reset_agent T:536-538
            buf.advance()
        buf.finish_paths(variant=gae_variant)


def _f32(x: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    if x is None or (x.dtype == torch.float32 and x.is_contiguous()):
        return x
    return x.to(torch.float32).contiguous()
