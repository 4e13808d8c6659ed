"""GPU tests (pytest -m gpu) of the RAD-TEAM Monte-Carlo evaluation: MonteCarloEvaluator.run_team (EpisodeRunner.run,
evaluate.py:333-475, with the map observation in the loop, RADTEAM_core.py:1854-1858) against the oracle env played the
reference's way and oracle/maps_oracle.c, and its bookkeeping kernel rs_eval_step against a numpy restatement."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import c_oracle as co
from tests import parity_util as pu

pytestmark = pytest.mark.gpu

import radiation_ppo_b200 as rp  # noqa: E402
from radiation_ppo_b200 import _lib as L  # noqa: E402

DIRS = np.array([[-1, 0], [-1, 1], [0, 1], [1, 1], [1, 0], [1, -1], [0, -1], [-1, -1]], np.float64)
DIRS /= np.linalg.norm(DIRS, axis=1, keepdims=True)


def scenarios(k, S):
    sc = pu.load_golden("scenarios_v4")
    return {key: sc[f"obs{k}_{key}"][:S] for key in ("src", "det", "intensity", "bkg", "rects", "num_obs")}


def lattice64(o, scale):
    """the reference's float64 observation of a float32 env observation [A, 11] (x * scale on the lattice coordinate)"""
    o64 = np.asarray(o, np.float64).copy()
    o64[:, 1:3] = np.rint(o64[:, 1:3] / scale) * scale
    return o64


class Greedy:
    """Greedy towards the source (float32 arithmetic on the device) where `greedy_steps(t)`, else the action of
    `other(t, obs, actor)`; records every action it played.  jitter: agent a > 0 plays a random move at the steps
    t = a - 1 (mod 4).  The agents of an env start on one point, and two agents that propose the same cell collide and
    stay where they are (take_action R:876-946): a team that only plays greedy moves never leaves its start."""

    def __init__(self, ev, arr, greedy_steps, other=None, jitter=False):
        d = ev.env.device
        src = np.repeat(arr["src"], ev.runs, axis=0).astype(np.float64) / 2200.0
        self.src = torch.as_tensor(src, dtype=torch.float32, device=d)
        self.dirs = torch.as_tensor(DIRS, dtype=torch.float32, device=d)
        self.greedy_steps, self.other = greedy_steps, other
        self.t, self.log = 0, []
        self.jitter = None
        if jitter:
            T, N, A = ev.steps_per_episode, len(src), ev.env.number_agents
            tab = np.random.default_rng(7).integers(0, 8, size=(T, N, A)).astype(np.int32)
            t, ag = np.arange(T)[:, None], np.arange(A)[None, :]
            mask = (ag > 0) & ((t - ag + 1) % 4 == 0)
            self.jitter = (torch.as_tensor(tab, device=d), torch.as_tensor(mask[:, None, :], device=d))

    def actions(self, obs, actor=None):
        to = self.src[:, None, :] - obs[:, :, 1:3]
        a = (to @ self.dirs.T).argmax(dim=2).to(torch.int32)
        if not self.greedy_steps(self.t):
            a = self.other(self.t, obs, actor)
        if self.jitter is not None:
            a = torch.where(self.jitter[1][self.t], self.jitter[0][self.t], a)
        self.log.append(a.cpu().numpy())
        self.t += 1
        return a


class ScriptedTeam(Greedy):
    """The team policy of the oracle test: predictions are a function of the observation (NaN for the agents whose
    count is a multiple of 3); two steps in three greedy, the third the argmax of a fixed linear head on the actor stacks
    it is handed, with the per-agent jitter of Greedy.  Records the predictions of all envs, and the observation and stacks of the sampled envs."""

    def __init__(self, ev, arr, sample, seed):
        super().__init__(ev, arr, lambda t: t % 3 != 2, self.head, jitter=True)
        d = ev.env.device
        X = Y = 27
        self.Wa = torch.as_tensor(np.random.default_rng(seed).normal(size=(6 * X * Y, 8)), dtype=torch.float32, device=d)
        self.idx = torch.as_tensor(sample, device=d)
        self.preds, self.seen, self.resets = [], [], []

    def head(self, t, obs, actor):
        N, A = obs.shape[:2]
        return (actor.permute(0, 1, 3, 4, 2).reshape(N * A, -1) @ self.Wa).argmax(dim=1).to(torch.int32).view(N, A)

    def predict(self, obs):
        pred = (obs[..., 1:3] * 0.5 + 0.25)
        pred = torch.where((torch.remainder(obs[..., :1], 3) == 0), torch.full_like(pred, float("nan")), pred).contiguous()
        self.preds.append(pred.cpu().numpy())
        return pred

    def act(self, obs, actor, critic):
        self.seen.append((obs[self.idx].cpu().numpy(), actor[self.idx].cpu().numpy(), critic[self.idx].cpu().numpy()))
        a = self.actions(obs, actor)
        return a, torch.zeros(a.shape, device=a.device), torch.zeros(a.shape, device=a.device)

    def reset_state(self, mask):
        self.resets.append(mask)


def oracle_play(arr, R, A, k, log, ctr0, team_mode):
    """The recorded actions replayed in the oracle, the reference's bookkeeping per run (E:402-419): every run stops
    counting at its first terminal step.  Also returns the active mask before every step and the oracle observations."""
    N = len(arr["src"]) * R
    ob = co.OracleBatch(N, co.default_config(n_agents=A, obstruction_count=k, enforce=1), seed=123)
    rep = {key: np.repeat(v, R, axis=0) for key, v in arr.items()}
    ob.load_scenarios(rep["src"], rep["det"], rep["intensity"], rep["bkg"], rep["rects"], rep["num_obs"])
    active = np.ones(N, bool); success = np.zeros(N, bool); length = np.zeros(N, np.int32)
    ret, oob, finders = np.zeros((N, A)), np.zeros((N, A), np.int32), np.zeros(N, np.uint8)
    act_before, obs_before = [], []
    for t in range(len(log)):
        act_before.append(active.copy())
        obs_before.append(ob.outs["obs"][:, :A].copy())
        ob.step(log[t], ctr0 + t + 1)
        o, e = ob.outs, ob.envs
        r = o["reward"][:, :A] if team_mode == "individual" else np.repeat(o["team_reward"][:, None], A, 1)
        ret += np.where(active[:, None], r.astype(np.float32).astype(np.float64), 0.0)
        length += active
        oob += ((e["oob"][:, :A] != 0) & active[:, None]).astype(np.int32)
        done = o["done"][:, :A] != 0
        term = done.any(axis=1) & active
        finders[term] = (done[term] * (1 << np.arange(A))).sum(axis=1).astype(np.uint8)
        success |= term
        active &= ~term
    return dict(success=success, length=length, ret=ret, oob=oob, finders=finders, active=np.array(act_before),
                obs=np.array(obs_before))


@pytest.mark.parametrize("k", [0, 3, 5])
@pytest.mark.parametrize("team_mode", ["individual", "cooperative"])
@pytest.mark.parametrize("A", [1, 2, 4])
def test_run_team_matches_oracle_and_maps_oracle(A, team_mode, k):
    """run_team against the oracle env and MapsOracle: the stacks the policy read (sampled envs) equal the oracle's bit
    for bit while the run plays and stay frozen after it finished; success, lengths, every agent's return, out-of-bounds
    counts, finders and success_counter match the reference's per-run bookkeeping; the localisation error equals a
    float64 numpy restatement."""
    S, R, T = 32, 4, 120
    arr = scenarios(k, S)
    ev = rp.MonteCarloEvaluator(scenarios=arr, montecarlo_runs=R, steps_per_episode=T, obstruction_count=k, seed=123,
                                enforce_grid_boundaries=True, number_agents=A, team_mode=team_mode)
    N = S * R
    sample = np.sort(np.random.default_rng(k + 10 * A).choice(N, 8, replace=False))
    pol = ScriptedTeam(ev, arr, sample, seed=A)
    res = ev.run_team(pol)
    assert pol.resets == [None]
    steps = res.steps_played
    assert steps == len(pol.log) == len(pol.seen) and steps <= T
    orc = oracle_play(arr, R, A, k, pol.log, ev.env._ctr - steps, team_mode)
    success, length = orc["success"], orc["length"]

    np.testing.assert_array_equal(res.success.cpu().numpy().reshape(-1), success)
    np.testing.assert_array_equal(res.episode_length.cpu().numpy().reshape(-1), length)
    np.testing.assert_allclose(res.agent_return.cpu().numpy().reshape(N, A), orc["ret"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(res.episode_return.cpu().numpy().reshape(-1), orc["ret"][:, 0], rtol=0, atol=1e-9)
    np.testing.assert_array_equal(res.out_of_bounds.cpu().numpy().reshape(N, A), orc["oob"])
    np.testing.assert_array_equal(res.finders.cpu().numpy().reshape(-1), orc["finders"])
    np.testing.assert_array_equal(res.success_counter.cpu().numpy(), success.reshape(S, R).sum(1))
    assert success.mean() > 0.05 and res.completed_runs == R
    if steps < T:
        assert success.all()

    # the stacks the policy read vs MapsOracle fed the reference's way (the observation and prediction of each step
    # while the run plays); a NaN prediction leaves buffer i's prediction map as it was, which the oracle, that always
    # has a prediction, reproduces with the buffer's previous prediction (or one outside the map before the first)
    scale = ev.env.scale
    for j, n in enumerate(sample):
        oracles = [co.MapsOracle(A, T) for _ in range(A)]
        last = [(100.0, 100.0)] * A
        frozen = None
        for t in range(steps):
            obs_s, act_a, act_c = pol.seen[t]
            if t < length[n]:
                if t > 0:                                               # (the oracle's load writes no observation)
                    pu.compare_obs(obs_s[j:j + 1], orc["obs"][t][n:n + 1])
                o64 = lattice64(obs_s[j], scale)
                for i in range(A):
                    p = pol.preds[t][n, i]
                    if not np.isnan(p).any():
                        last[i] = (float(p[0]), float(p[1]))
                    want = oracles[i].observation_to_map(o64, i, last[i])
                    np.testing.assert_array_equal(np.concatenate([act_a[j][i], act_c[j][:1]], axis=0), want,
                                                  err_msg=f"env {n} agent {i} step {t}")
                frozen = (act_a[j], act_c[j])
            else:                                                       # finished: no longer updated
                np.testing.assert_array_equal(act_a[j], frozen[0], err_msg=f"env {n} step {t} after the end")
                np.testing.assert_array_equal(act_c[j], frozen[1], err_msg=f"env {n} step {t} after the end")

    # localisation error of the predictions made for the steps each run played
    src = np.repeat(arr["src"], R, axis=0).astype(np.float64)
    e_sum, e_n, e_last = np.zeros((N, A)), np.zeros((N, A), np.int64), np.full((N, A), np.nan)
    for t in range(steps):
        p = pol.preds[t].astype(np.float64)
        ok = ~np.isnan(p).any(axis=2) & orc["active"][t][:, None]
        e = np.hypot(p[..., 0] / scale - src[:, None, 0], p[..., 1] / scale - src[:, None, 1])
        e_sum += np.where(ok, e, 0.0)
        e_n += ok
        e_last = np.where(ok, e, e_last)
    assert e_n.min() < e_n.max() and (e_n > 0).any()
    with np.errstate(invalid="ignore"):
        np.testing.assert_allclose(res.loc_err_mean.cpu().numpy().reshape(N, A), e_sum / e_n, rtol=1e-13, atol=0)
    np.testing.assert_allclose(res.loc_err_final.cpu().numpy().reshape(N, A), e_last.astype(np.float32), rtol=1e-6, atol=0)
    s = res.summary()
    assert s["success_rate"] == pytest.approx(success.mean())
    assert s["median_loc_err_final"] == pytest.approx(float(np.nanmedian(e_last.astype(np.float32))), rel=1e-6)


def eval_step_numpy(st, reward, team, done, info, pred, src, scale, individual):
    """rs_eval_step restated on numpy copies of its state (dict of arrays, updated in place)."""
    act = st["active"] != 0
    A = done.shape[1]
    st["length"][act] += 1
    r = reward if individual else np.repeat(team[:, None], A, 1)
    st["ret"][act] += r[act].astype(np.float64)
    st["oob"][act] += (info[act] & L.I_OOB) != 0
    dn = (done != 0) & act[:, None]
    fin = dn.any(axis=1)
    st["success"][fin] = 1
    st["active"][fin] = 0
    st["finders"][fin] = (dn[fin] * (1 << np.arange(A))).sum(axis=1)
    st["n_active"][0] -= int(fin.sum())
    if pred is not None:
        p = pred.astype(np.float64)
        ok = ~np.isnan(p).any(axis=2) & act[:, None]
        e = np.hypot(p[..., 0] / scale - src[:, None, 0], p[..., 1] / scale - src[:, None, 1])
        st["loc_sum"] += np.where(ok, e, 0.0)
        st["loc_n"] += ok
        st["loc_last"] = np.where(ok, e.astype(np.float32), st["loc_last"])


@pytest.mark.parametrize("individual", [0, 1])
@pytest.mark.parametrize("N,A", [(1000, 1), (4099, 3), (1000, 8), (4099, 8)])
def test_eval_step_kernel_matches_numpy(N, A, individual):
    """rs_eval_step called several times in a row on random inputs (N not a multiple of 32, NaN predictions, envs
    inactive on entry, finders NULL for A = 3) against the numpy restatement; n_active stays active.sum()."""
    rng = np.random.default_rng(N + A + 7 * individual)
    d = torch.device("cuda")
    lib = L.load()
    scale = 1 / 2200.0
    st = dict(active=(rng.random(N) < 0.8).astype(np.uint8), success=np.zeros(N, np.uint8), length=np.zeros(N, np.int32),
              ret=rng.normal(size=(N, A)), oob=np.zeros((N, A), np.int32), finders=np.zeros(N, np.uint8),
              loc_sum=np.zeros((N, A)), loc_n=np.zeros((N, A), np.int32), loc_last=np.full((N, A), np.nan, np.float32))
    st["n_active"] = np.array([int(st["active"].sum())], np.int32)
    dev = {k: torch.as_tensor(v, device=d) for k, v in st.items()}
    no_finders = A == 3
    src = rng.integers(0, 2700, size=(N, 2)).astype(np.int32)
    src_d = torch.as_tensor(src, device=d)
    stream = C.c_void_p(torch.cuda.current_stream(d).cuda_stream)
    p = lambda x: None if x is None else C.c_void_p(x.data_ptr())     # noqa: E731
    for call in range(6):
        reward = rng.normal(size=(N, A)).astype(np.float32)
        team = rng.normal(size=N).astype(np.float32)
        done = (rng.random((N, A)) < 0.04).astype(np.uint8) * rng.integers(1, 3, size=(N, A)).astype(np.uint8)
        info = rng.integers(0, 32, size=(N, A)).astype(np.uint8)
        pred = rng.random((N, A, 2)).astype(np.float32) * 1.3 - 0.1
        pred[rng.random((N, A)) < 0.2, rng.integers(0, 2)] = np.nan
        pred_in = None if call == 2 else pred                          # a call without predictions
        ins = [torch.as_tensor(x, device=d) for x in (reward, team, done, info)]
        pd = None if pred_in is None else torch.as_tensor(pred_in, device=d)
        loc = (None,) * 3 if pd is None else (dev["loc_sum"], dev["loc_n"], dev["loc_last"])
        rc = lib.rs_eval_step(p(ins[0]), p(ins[1]), p(ins[2]), p(ins[3]), p(dev["active"]), p(dev["success"]),
                              p(dev["length"]), p(dev["ret"]), p(dev["oob"]), None if no_finders else p(dev["finders"]),
                              p(dev["n_active"]), p(pd), None if pd is None else p(src_d), scale, *[p(x) for x in loc],
                              N, A, individual, stream)
        assert rc == 0, lib.rs_last_error()
        eval_step_numpy(st, reward, team, done, info, pred_in, src.astype(np.float64), scale, individual)
        if no_finders:
            st["finders"][:] = 0
        got = {k: v.cpu().numpy() for k, v in dev.items()}
        for key in ("active", "success", "length", "oob", "finders", "n_active", "loc_n"):
            np.testing.assert_array_equal(got[key], st[key], err_msg=f"{key} after call {call}")
        np.testing.assert_array_equal(got["ret"], st["ret"], err_msg=f"ret after call {call}")
        np.testing.assert_allclose(got["loc_sum"], st["loc_sum"], rtol=1e-14, atol=0)
        np.testing.assert_allclose(got["loc_last"], st["loc_last"], rtol=1e-6, atol=0)
        assert int(got["n_active"][0]) == int(got["active"].sum())
    assert 0 < int(st["success"].sum()) and int(st["active"].sum()) > 0


@pytest.mark.parametrize("team_mode", ["individual", "cooperative"])
def test_run_team_agrees_with_run_on_the_same_actions(team_mode):
    """A team policy that ignores the stacks and plays the same actions as an obs-only policy: run_team gives run()'s
    success, episode_length and episode_return, on the same scenarios and seed."""
    S, R, T, A, k = 40, 4, 120, 2, 3
    arr = scenarios(k, S)
    kw = dict(scenarios=arr, montecarlo_runs=R, steps_per_episode=T, obstruction_count=k, seed=9,
              enforce_grid_boundaries=True, number_agents=A, team_mode=team_mode)
    ev1, ev2 = rp.MonteCarloEvaluator(**kw), rp.MonteCarloEvaluator(**kw)
    N = S * R
    table = torch.as_tensor(np.random.default_rng(3).integers(0, 8, size=(T, N, A)).astype(np.int32), device=ev1.env.device)
    other = lambda t, obs, actor: table[t]                             # noqa: E731
    g1 = Greedy(ev1, arr, lambda t: t % 2 == 0, other)
    g2 = Greedy(ev2, arr, lambda t: t % 2 == 0, other)

    class TeamOfG2:
        def predict(self, obs):
            return None

        def act(self, obs, actor, critic):
            return g2.actions(obs)

    r1 = ev1.run(lambda obs, t: g1.actions(obs))
    r2 = ev2.run_team(TeamOfG2())
    assert r2.loc_err_mean is None and r2.loc_err_final is None and "median_loc_err_final" not in r2.summary()
    for key in ("success", "episode_length", "episode_return", "success_counter"):
        assert torch.equal(getattr(r1, key), getattr(r2, key)), key
    assert float(r1.success.float().mean()) > 0.1


def test_early_stop_follows_the_lag_rule():
    """A policy that reaches the source quickly: steps_played is the first t + 1 with t % 8 == 7 at which no run was
    playing after step t - 4, below steps_per_episode, and the results equal those of early_stop=False."""
    S, R, T, A, k = 32, 4, 120, 2, 0
    arr = scenarios(k, S)
    kw = dict(scenarios=arr, montecarlo_runs=R, steps_per_episode=T, obstruction_count=k, seed=5,
              enforce_grid_boundaries=True, number_agents=A)
    res = {}
    for early in (True, False):
        ev = rp.MonteCarloEvaluator(**kw)
        g = Greedy(ev, arr, lambda t: True, jitter=True)

        class Team:
            def predict(self, obs):
                return (obs[..., 1:3] * 0.5 + 0.25).contiguous()

            def act(self, obs, actor, critic):
                return g.actions(obs)

        res[early] = ev.run_team(Team(), early_stop=early)
    r, full = res[True], res[False]
    assert full.steps_played == T
    length = full.episode_length.cpu().numpy().reshape(-1)
    assert bool(full.success.all())
    finished_by = lambda s: int((length <= s + 1).sum())                # noqa: E731  runs done after step s
    N = S * R
    want = next((t + 1 for t in range(7, T, 8) if finished_by(t - 4) == N), T)
    assert r.steps_played == want < T
    for key in ("success", "episode_length", "episode_return", "success_counter", "agent_return", "out_of_bounds",
                "finders", "loc_err_mean", "loc_err_final"):
        np.testing.assert_array_equal(getattr(r, key).cpu().numpy(), getattr(full, key).cpu().numpy(), err_msg=key)


def test_run_team_argument_errors():
    arr = scenarios(0, 4)
    kw = dict(scenarios=arr, montecarlo_runs=2, steps_per_episode=20, seed=1, enforce_grid_boundaries=True, number_agents=2)

    class Never:
        def predict(self, obs):
            raise AssertionError("not reached")

        act = predict

    with pytest.raises(ValueError, match="standardize"):
        rp.MonteCarloEvaluator(standardize=1, **kw).run_team(Never())
    ev = rp.MonteCarloEvaluator(**kw)
    for maps in (rp.BatchedMapsBuffer(9, 2, 20, environment_scale=ev.env.scale),
                 rp.BatchedMapsBuffer(8, 3, 20, environment_scale=ev.env.scale)):
        with pytest.raises(ValueError, match="maps must be"):
            ev.run_team(Never(), maps=maps)
