"""Batched Monte-Carlo evaluation over saved test scenarios (SURVEY.md 8f-3).

Mirrors the measurement of /root/reference/algos/multiagent/evaluate.py::EpisodeRunner.run (E:333-475): every test
scenario (`env_<i>` of a `test_env_dict_*_v4` file, E:203, loaded by `refresh_environment`, rad_search_env.py:799-874) is
played `montecarlo_runs` times by a policy until an agent reaches the source or `steps_per_episode` steps have passed;
per scenario it reports the success count, the episode lengths and the episode returns of the successful and the
unsuccessful runs, and the source / background intensities (E:428-450, `MonteCarloResults` E:88-103).

The reference runs the scenarios one after the other, one environment, one Monte-Carlo run at a time.  Here all
scenarios x runs are ONE batched environment (100 runs x 1000 scenarios = 100,000 envs in a launch): `rs_load_scenarios`
builds them, `rs_step` advances them, and the bookkeeping is a handful of tensor ops per step.  The Monte-Carlo runs
of a scenario differ in their Poisson draws (Philox keyed by the env id) and in whatever the policy samples.

`run_team` plays a RAD-TEAM policy, whose agents read the map stacks of their buffers (select_action,
RADTEAM_core.py:1854-1858), with maps_buffer.BatchedMapsBuffer in the loop; its per-step bookkeeping is one launch
(rs_eval_step) and its early stop reads the count of runs still playing with a fixed lag instead of draining the device.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Callable, Dict, Iterable, Optional, Protocol

import numpy as np
import torch

from . import _lib as L
from .envs.rad_search_env import RadSearch
from .maps_buffer import BatchedMapsBuffer
from .rollout import _f32
from .scenario_io import scenario_arrays


@dataclass
class MonteCarloResults:
    """Per-scenario results, arrays of shape [scenarios, runs] unless noted (cf. E:88-103)."""

    success: torch.Tensor                  # bool: a terminal state was reached before the timeout
    episode_length: torch.Tensor           # int32 (`total_episode_length`)
    episode_return: torch.Tensor           # float64 sum of the float32 (team) rewards, agent 0's tally (E:402-409, 441)
    success_counter: torch.Tensor          # int32 [scenarios]
    intensity: torch.Tensor                # int32 [scenarios]
    background_intensity: torch.Tensor     # int32 [scenarios]
    completed_runs: int = 0
    extra: Dict = field(default_factory=dict)

    def summary(self) -> Dict[str, float]:
        s = self.success
        f = lambda x, m: float(x[m].float().median()) if bool(m.any()) else float("nan")     # noqa: E731
        return {"success_rate": float(s.float().mean()), "median_len_success": f(self.episode_length, s),
                "median_len_fail": f(self.episode_length, ~s), "median_ret_success": f(self.episode_return, s),
                "median_ret_fail": f(self.episode_return, ~s)}


@dataclass
class TeamMonteCarloResults(MonteCarloResults):
    """MonteCarloResults of MonteCarloEvaluator.run_team: the inherited fields keep their meaning (episode_return is agent
    0's tally in the configured team mode), plus per-agent detail.  Arrays [scenarios, runs, agents] unless noted."""

    agent_return: Optional[torch.Tensor] = None     # float64: every agent's return under the team mode
    out_of_bounds: Optional[torch.Tensor] = None    # int32: steps that ended out of bounds
    finders: Optional[torch.Tensor] = None          # uint8 [scenarios, runs]: bit mask of the agents that reached the source
    steps_played: int = 0                           # env steps executed (< steps_per_episode after an early stop)
    # Localisation error of the source predictions (an addition: not a field of the reference's MonteCarloResults), in
    # cm, over the steps the run was playing and the agent gave a prediction; NaN where it never did.  None when the
    # policy made no predictions.
    loc_err_mean: Optional[torch.Tensor] = None     # float64
    loc_err_final: Optional[torch.Tensor] = None    # float32: the error of the agent's last prediction

    def summary(self) -> Dict[str, float]:
        s = super().summary()
        if self.loc_err_final is not None:
            # median over the agents that made a prediction, the mean of the two middle values for an even count (as
            # numpy / statistics.median; torch's median would return the lower one)
            e = self.loc_err_final.double().flatten()
            e = e[~e.isnan()].cpu().numpy()
            s["median_loc_err_final"] = float(np.median(e)) if e.size else float("nan")
        return s


Policy = Callable[[torch.Tensor, int], torch.Tensor]     # (obs [N, A, 11] on the device, step index) -> actions [N, A]


def uniform_policy(seed: int = 0) -> Policy:
    """The reference's `uniform_search` baseline: actions drawn uniformly from the 8 directions."""
    gen: Dict[str, torch.Generator] = {}

    def act(obs: torch.Tensor, t: int) -> torch.Tensor:
        g = gen.setdefault("g", torch.Generator(device=obs.device).manual_seed(seed))
        return torch.randint(0, 8, obs.shape[:2], generator=g, device=obs.device, dtype=torch.int32)

    return act


class TeamEvalPolicy(Protocol):
    """A RAD-TEAM policy as run_team drives it; rollout.TeamRolloutPolicy satisfies it."""

    def predict(self, obs: torch.Tensor) -> Optional[torch.Tensor]:
        """obs [N, A, 11] f32 -> the source prediction float32 [N, A, 2] in scaled coordinates (NaN = none for that agent),
        or None when the policy has no predictor."""

    def act(self, obs: torch.Tensor, actor_stacks: torch.Tensor, critic_stacks: torch.Tensor):
        """obs [N, A, 11], actor_stacks [N, A, 6, X, Y], critic_stacks [N, 4, X, Y] -> actions [N, A], or a tuple whose
        first element is the actions (e.g. (action, value, log-probability))."""

    # optional: reset_state(mask) -- called once with None before the first step


class MonteCarloEvaluator:
    """All scenarios x Monte-Carlo runs as one batched RadSearch.

    env_dict: the joblib dict of a `test_env_dict_*` file (or None with `scenarios` = the arrays of
    scenario_io.scenario_arrays); ids: which scenarios; env_kwargs: the reference's env kwargs
    (`obstruction_count`, `enforce_grid_boundaries`, `number_agents`, ...).  Env n = scenario n // runs, run n % runs."""

    def __init__(self, env_dict: Optional[Dict] = None, ids: Optional[Iterable[int]] = None, montecarlo_runs: int = 100,
                 steps_per_episode: int = 120, obstruction_count: int = 0, scenarios: Optional[Dict[str, np.ndarray]] = None,
                 seed: int = 0, device=None, team_mode: str = "cooperative", standardize: int = 0, **env_kwargs) -> None:
        k_max = max(int(obstruction_count), 0)
        if scenarios is None:
            if env_dict is None:
                raise ValueError("give env_dict or scenarios")
            scenarios = scenario_arrays(env_dict, ids, k_max=max(k_max, 1), with_obstacles=obstruction_count > 0)
        self.n_scenarios = int(len(scenarios["intensity"]))
        self.runs, self.steps_per_episode, self.team_mode = int(montecarlo_runs), int(steps_per_episode), team_mode
        N = self.n_scenarios * self.runs
        self.env = RadSearch(obstruction_count=obstruction_count, num_envs=N, seed=seed, device=device,
                             steps_per_episode=steps_per_episode, k_max=k_max, standardize=standardize, **env_kwargs)
        rep = lambda a: np.repeat(np.asarray(a), self.runs, axis=0)          # noqa: E731
        self._arrays = {k: rep(v) for k, v in scenarios.items()}
        if k_max > 0:
            if int(np.max(scenarios["num_obs"])) > k_max:
                raise ValueError("a scenario has more obstructions than obstruction_count")
            self._arrays["rects"] = np.ascontiguousarray(self._arrays["rects"][:, :k_max])
        self.intensity = torch.as_tensor(np.asarray(scenarios["intensity"]), dtype=torch.int32, device=self.env.device)
        self.background = torch.as_tensor(np.asarray(scenarios["bkg"]), dtype=torch.int32, device=self.env.device)

    def run(self, policy: Policy, on_step: Optional[Callable[[int, torch.Tensor, torch.Tensor], None]] = None,
            localizer: Optional[Callable[[torch.Tensor, int], torch.Tensor]] = None) -> MonteCarloResults:
        """Plays every scenario x run: actions = policy(obs, t), or with a localizer (e.g. pfgru.FusedPFGRU over the N*A
        rows) policy(obs, t, localizer(obs, t)), the source prediction [N*A, 2] of a 13-wide policy."""
        env, S, R, A = self.env, self.n_scenarios, self.runs, self.env.number_agents
        N = S * R
        dev = env.device
        a = self._arrays
        obs = env.load_scenarios(a["src"], a["det"], a["intensity"], a["bkg"],
                                 rects=a["rects"] if env._cfg.k_max > 0 else None, num_obs=a["num_obs"])
        active = torch.ones(N, dtype=torch.bool, device=dev)
        success = torch.zeros(N, dtype=torch.bool, device=dev)
        length = torch.zeros(N, dtype=torch.int32, device=dev)
        ret = torch.zeros(N, dtype=torch.float64, device=dev)
        for t in range(self.steps_per_episode):
            acts = policy(obs, t) if localizer is None else policy(obs, t, localizer(obs, t))
            acts = acts.to(device=dev, dtype=torch.int32).reshape(N, A)
            obs, reward, team, done, _, _ = env.step_batch(acts, auto_reset=False)
            r = team if self.team_mode != "individual" else reward[:, 0]      # E:402-409 (agent 0's tally is reported)
            ret += torch.where(active, r, torch.zeros_like(r)).double()
            length += active.to(torch.int32)
            terminal = (done != 0).any(dim=1) & active                          # E:415-419
            success |= terminal
            active &= ~terminal
            if on_step is not None:
                on_step(t, obs, active)
            if t % 8 == 7 and not bool(active.any()):                           # every run has finished early
                break
        return MonteCarloResults(
            success=success.view(S, R), episode_length=length.view(S, R), episode_return=ret.view(S, R),
            success_counter=success.view(S, R).sum(dim=1).to(torch.int32), intensity=self.intensity,
            background_intensity=self.background, completed_runs=R)

    def run_team(self, policy: TeamEvalPolicy, maps: Optional[BatchedMapsBuffer] = None, early_stop: bool = True,
                 on_step: Optional[Callable[[int, torch.Tensor, torch.Tensor], None]] = None) -> TeamMonteCarloResults:
        """EpisodeRunner.run (E:333-475) for a RAD-TEAM policy: per step t, pred = policy.predict(obs); the map stacks of
        the runs still playing are updated with (obs, pred) (RADTEAM_core.py:1854-1858; a run that finished keeps its
        stacks as they were at its last step, and costs no update); actions = policy.act(obs, actor, critic); env step;
        one rs_eval_step launch for the bookkeeping; on_step(t, obs, active) if given.

        maps: a BatchedMapsBuffer of num_envs = scenarios x runs and number_agents = A (e.g. the 147 x 147 grid of
        unenforced boundaries, or use_prediction=False); None builds the default 27 x 27 one once and keeps it.  The env
        must have standardize=0: the maps standardise the raw counts themselves.  early_stop: the count of runs still
        playing after step t - 4 is read at every t with t % 8 == 7 and the loop stops when it is 0; the count travels to
        the host by an asynchronous copy queued four steps earlier, so the check never drains the device, and the number
        of steps played depends on the results only.  False plays all steps_per_episode steps."""
        env, S, R, A = self.env, self.n_scenarios, self.runs, self.env.number_agents
        N = S * R
        dev = env.device
        if env.standardize != 0:
            raise ValueError("run_team needs standardize=0: the maps standardise the raw counts themselves")
        if self.team_mode not in ("individual", "cooperative"):
            raise ValueError("run_team supports team_mode 'individual' or 'cooperative'")
        if maps is None:
            maps = getattr(self, "_maps", None)
            if maps is None:
                maps = self._maps = BatchedMapsBuffer(N, A, self.steps_per_episode, environment_scale=env.scale, device=dev)
        elif maps.num_envs != N or maps.number_of_agents != A:
            raise ValueError(f"maps must be a BatchedMapsBuffer of {N} envs x {A} agents (scenarios x runs, number_agents)")
        a = self._arrays
        obs = env.load_scenarios(a["src"], a["det"], a["intensity"], a["bkg"],
                                 rects=a["rects"] if env._cfg.k_max > 0 else None, num_obs=a["num_obs"])
        maps.reset()
        if hasattr(policy, "reset_state"):
            policy.reset_state(None)
        z = lambda *s, dt: torch.zeros(*s, dtype=dt, device=dev)      # noqa: E731
        active, success, finders = torch.ones(N, dtype=torch.uint8, device=dev), z(N, dt=torch.uint8), z(N, dt=torch.uint8)
        length, ret, oob = z(N, dt=torch.int32), z(N, A, dt=torch.float64), z(N, A, dt=torch.int32)
        n_active = torch.full((1,), N, dtype=torch.int32, device=dev)
        loc = None                                                      # (sum, count, last), allocated at the first prediction
        host_count = torch.empty(1, dtype=torch.int32, pin_memory=True)
        copied = torch.cuda.Event()
        lib = L.load()
        p = lambda x: None if x is None else C.c_void_p(x.data_ptr())   # noqa: E731
        individual = int(self.team_mode == "individual")
        fixed = [p(x) for x in (env.reward, env.team_reward, env.done_flags, env.info_flags, active, success, length, ret,
                                oob, finders, n_active)]
        steps = 0
        for t in range(self.steps_per_episode):
            pred = policy.predict(obs)
            pred = None if pred is None else _f32(pred.to(device=dev).reshape(N, A, 2))
            actor, critic = maps.update(obs, pred, mask=active)
            out = policy.act(obs, actor, critic)
            acts = (out[0] if isinstance(out, tuple) else out).to(device=dev, dtype=torch.int32).reshape(N, A)
            env.step_batch(acts, auto_reset=False)
            if pred is not None and loc is None:
                loc = (z(N, A, dt=torch.float64), z(N, A, dt=torch.int32),
                       torch.full((N, A), float("nan"), dtype=torch.float32, device=dev))
            lg = (None,) * 3 if pred is None else loc
            with torch.cuda.device(dev):
                L.check(lib.rs_eval_step(*fixed, p(pred), p(env._src), env.scale, p(lg[0]), p(lg[1]), p(lg[2]), N, A,
                                         individual, C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "rs_eval_step")
            steps = t + 1
            if on_step is not None:
                on_step(t, obs, active.view(torch.bool))
            if early_stop:
                if t % 8 == 3:                                          # read back at t + 4
                    host_count.copy_(n_active, non_blocking=True)
                    copied.record(torch.cuda.current_stream(dev))
                elif t % 8 == 7:
                    copied.synchronize()
                    if int(host_count[0]) == 0:                         # every run had finished by step t - 4
                        break
        v = lambda x: x.view(S, R, *x.shape[1:])                        # noqa: E731
        res = TeamMonteCarloResults(
            success=v(success.bool()), episode_length=v(length), episode_return=v(ret[:, 0]),
            success_counter=v(success).sum(dim=1, dtype=torch.int32), intensity=self.intensity,
            background_intensity=self.background, completed_runs=R, agent_return=v(ret), out_of_bounds=v(oob),
            finders=v(finders), steps_played=steps)
        if loc is not None:
            res.loc_err_mean = v(loc[0] / loc[1])
            res.loc_err_final = v(loc[2])
        return res
