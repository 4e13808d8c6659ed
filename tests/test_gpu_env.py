"""GPU parity tests (pytest -m gpu): the CUDA env step / reset path, called through the product API and the C ABI,
against the oracle (oracle/radsearch_oracle.c) and the golden vectors recorded from the unmodified reference.

Bars (BASELINE.json north_star): bit-exact detector positions, collision / LOS / blocked / out-of-bounds flags,
termination, reset indices, Poisson counts (injected uniforms AND the shared Philox stream), rewards, best distances;
sensor values within 1e-5 relative in fp32."""
import numpy as np
import pytest
import torch

from oracle import c_oracle as co
from tests import parity_util as pu

pytestmark = pytest.mark.gpu

import radiation_ppo_b200 as rp  # noqa: E402
from radiation_ppo_b200 import _lib as L  # noqa: E402


def make_pair(n, A=1, oc=5, enforce=True, seed=11, env_id0=3, max_ep_len=120, **kw):
    env = rp.RadSearch(obstruction_count=oc, enforce_grid_boundaries=enforce, number_agents=A, num_envs=n, seed=seed,
                       env_id_offset=env_id0, steps_per_episode=max_ep_len, **kw)
    ob = co.OracleBatch(n, co.default_config(n_agents=A, obstruction_count=oc, enforce=int(enforce),
                                             max_ep_len=max_ep_len), seed=seed, env_id0=env_id0)
    ob.reset()          # the constructor reset used counter env._ctr
    return env, ob


@pytest.mark.parametrize("n,A,oc,enforce,T,idle", [(1024, 1, 5, True, 130, 0.0), (1024, 1, -1, False, 100, 0.0),
                                                   (512, 4, 5, True, 90, 0.15), (256, 1, 0, True, 40, 0.0),
                                                   (300, 2, 7, True, 70, 0.1), (37, 1, 3, False, 50, 0.0),
                                                   (480, 3, 4, True, 80, 0.1), (96, 5, 2, True, 40, 0.2), (50, 8, 3, True, 30, 0.1),
                                                   (200, 6, 4, True, 40, 0.1), (77, 7, 6, False, 40, 0.15)])
def test_rollout_matches_oracle(n, A, oc, enforce, T, idle):
    env, ob = make_pair(n, A, oc, enforce, seed=100 + n)
    v = pu.GpuView(env)
    pu.compare_state(v, ob, A)
    pu.compare_obs(v.obs, ob.outs["obs"][:, :A])
    rng = np.random.default_rng(n)
    seen = dict(los=0, sens=0, done=0)
    for t in range(T):
        acts = rng.integers(0, 8, size=(n, A))
        acts[rng.random((n, A)) < idle] = 8
        env.step_batch(torch.as_tensor(acts, dtype=torch.int32, device=env.device))
        ob.step(acts, env._ctr)
        v = pu.GpuView(env)
        pu.compare_state(v, ob, A)
        o, e = ob.outs, ob.envs
        pu.compare_obs(v.obs, o["obs"][:, :A])
        np.testing.assert_array_equal(v.reward, o["reward"][:, :A].astype(np.float32))
        np.testing.assert_array_equal(v.done, o["done"][:, :A])
        np.testing.assert_array_equal(v.team_reward, o["team_reward"].astype(np.float32))
        info_ref = e["oob"][:, :A] | (e["blocked"][:, :A] * 2) | (e["collision"][:, :A] * 4) | (e["los_blocked"][:, :A] * 8)
        np.testing.assert_array_equal(v.info & 15, info_ref)
        seen["los"] += int(((v.info & 8) != 0).sum()); seen["sens"] += int((v.obs[:, :, 3:] > 0).sum()); seen["done"] += int(v.done.sum())
        mask = (e["done"] == 1) | (e["ep_len"] == 120) | ((t + 1) % 45 == 0)
        if mask.any():
            newm = np.full(n, (t + 1) % 45 == 0)
            env.reset_batch(mask=torch.as_tensor(mask), new_obstacles=torch.as_tensor(newm))
            ob.reset(mask=mask, new_obstacles=newm)
            v = pu.GpuView(env)
            pu.compare_state(v, ob, A)
            pu.compare_obs(v.obs, ob.outs["obs"][:, :A], sel=np.where(mask)[0])
    assert seen["sens"] > 0 and (oc == 0 or seen["los"] > 0)


def test_auto_reset_follows_caller_rules():
    """train.py:394-405, 446-548 applied on the device: timeout, terminal, epoch end, reset indices, final obs."""
    n, A, T, ML = 2048, 1, 130, 40
    env, ob = make_pair(n, A, 5, True, seed=5, max_ep_len=ML, auto_reset=True)
    rng = np.random.default_rng(0)
    n_resets = 0
    for t in range(1, T + 1):
        acts = rng.integers(0, 8, size=(n, A))
        epoch_end = t % 60 == 0
        env.step_batch(torch.as_tensor(acts, dtype=torch.int32, device=env.device), epoch_end=epoch_end)
        ob.step(acts, env._ctr)
        e = ob.envs
        terminal, timeout = e["done"] == 1, e["ep_len"] == ML
        want = terminal * 1 | timeout * 2 | ((terminal | timeout | epoch_end) * 4)
        mask = (want & 4) != 0
        final = ob.outs["obs"][:, :A].copy()
        rew = ob.outs["reward"][:, :A].astype(np.float32).copy()
        if mask.any():
            ob.reset(mask=mask, new_obstacles=np.full(n, epoch_end))
        v = pu.GpuView(env)
        np.testing.assert_array_equal(v.ended, want)
        np.testing.assert_array_equal(v.reward, rew)
        pu.compare_obs(v.final_obs, final, sel=np.where(mask)[0])
        pu.compare_state(v, ob, A)
        np.testing.assert_array_equal(v.ep_len, e["ep_len"])
        # observation handed to the policy next: first obs of the new episode where reset, else the step's obs
        nxt = np.where(mask[:, None, None], ob.outs["obs"][:, :A], final)
        pu.compare_obs(v.obs, nxt)
        n_resets += int(mask.sum())
    assert n_resets > n


@pytest.mark.parametrize("name", list(pu.STEP_FILES))
def test_reference_records_replayed_on_gpu(name):
    """Every recorded call of the unmodified reference, replayed from its pre-state with its own uniforms injected."""
    g = pu.load_golden(name)
    kw = pu.STEP_FILES[name]
    A, n = kw["n_agents"], len(g["is_reset"])
    env = rp.RadSearch(obstruction_count=kw["obstruction_count"], enforce_grid_boundaries=bool(kw["enforce"]),
                       number_agents=A, num_envs=n, seed=1, k_max=7)
    dev = env.device
    u = torch.as_tensor(g["out_uniforms"], device=dev)
    env.load_scenarios(g["pre_src"], g["pre_det"][:, 0], g["pre_intensity"], g["pre_bkg"], g["pre_rects"][:, :7],
                       g["pre_num_obs"], uniforms=u)
    is_reset = g["is_reset"].astype(bool)
    v = pu.GpuView(env)
    r = np.where(is_reset)[0]
    if len(r):
        pu.compare_obs(v.obs, g["out_obs"], sel=r)
        np.testing.assert_array_equal(v.best[:, r].T, g["pre_best"][r])
    env._det.copy_(torch.as_tensor(g["pre_det"].transpose(1, 0, 2).copy(), device=dev))
    env._best.copy_(torch.as_tensor(g["pre_best"].T.copy(), device=dev))
    env._aflags.copy_(torch.as_tensor((g["pre_oob_count"] | (g["pre_blocked"] << 24)).T.copy(), device=dev))
    env._meta.copy_(torch.as_tensor(g["pre_num_obs"] | (g["pre_done"] << 8), device=dev))
    acts = np.where(is_reset[:, None], 8, g["out_actions"])
    env.step_batch(torch.as_tensor(acts, dtype=torch.int32, device=dev), uniforms=u)
    v = pu.GpuView(env)
    s = np.where(~is_reset)[0]
    pu.compare_obs(v.obs, g["out_obs"], sel=s)
    np.testing.assert_array_equal(v.reward[s], g["out_reward"][s].astype(np.float32))
    np.testing.assert_array_equal(v.done[s], g["out_done"][s])
    np.testing.assert_array_equal(v.team_reward[s], g["out_team_reward"][s].astype(np.float32))
    np.testing.assert_array_equal(v.det[:, s].transpose(1, 0, 2), g["out_det"][s])
    np.testing.assert_array_equal(v.best[:, s].T, g["out_best"][s])
    np.testing.assert_array_equal((v.aflags[:, s] & 0xFFFFFF).T, g["out_oob_count"][s])
    np.testing.assert_array_equal(((v.aflags[:, s] >> 24) & 1).T, g["out_blocked"][s])
    np.testing.assert_array_equal(((v.info[s] & 8) != 0).astype(int), g["out_los"][s])
    np.testing.assert_array_equal(((v.info[s] & 1) != 0).astype(int), g["out_oob"][s])
    assert not (v.status[s] & ~np.uint32(L.ST_LAMBDA_INF)).any()


def test_saved_evaluation_scenarios_against_oracle():
    """The reference's test_env_dict_obs*_v4 scenarios (inputs) through rs_load_scenarios + 30 steps vs the oracle."""
    sc = pu.load_golden("scenarios_v4")
    for k in (0, 1, 3, 5, 7):
        arr = {key: sc[f"obs{k}_{key}"] for key in ("src", "det", "intensity", "bkg", "rects", "num_obs")}
        n = len(arr["src"])
        env = rp.RadSearch(obstruction_count=k, enforce_grid_boundaries=True, num_envs=n, seed=77, k_max=7)
        env.load_scenarios(**arr)
        ob = co.OracleBatch(n, co.default_config(obstruction_count=k, enforce=1), seed=77)
        ob.load_scenarios(arr["src"], arr["det"], arr["intensity"], arr["bkg"], arr["rects"], arr["num_obs"])
        ob.step(None, env._ctr)
        ob.envs["iter_count"] = 0
        ob.envs["ep_len"] = 0
        # the probe draws from Philox domain 2 on the GPU (reset) and domain 0 in the oracle's step(None): compare
        # everything but the count here, the counts in the steps below
        v = pu.GpuView(env)
        np.testing.assert_array_equal(v.best[0], ob.envs["best"][:, 0])
        np.testing.assert_allclose(v.obs[:, 0, 1:], ob.outs["obs"][:, 0, 1:].astype(np.float32), rtol=1e-5)
        rng = np.random.default_rng(k)
        for t in range(30):
            acts = rng.integers(0, 8, size=(n, 1))
            env.step_batch(torch.as_tensor(acts, dtype=torch.int32, device=env.device))
            ob.step(acts, env._ctr)
            v = pu.GpuView(env)
            pu.compare_state(v, ob, 1)
            pu.compare_obs(v.obs, ob.outs["obs"][:, :1])


def test_poisson_philox_distribution_ks_against_numpy():
    """Counts drawn from the Philox stream (exact and fp32-acceptance samplers) vs numpy.random.Generator.poisson."""
    from scipy import stats

    sc = pu.load_golden("scenarios_v4")
    arr = {key: sc[f"obs0_{key}"][:1].repeat(40000, axis=0) for key in ("src", "det", "intensity", "bkg")}
    for lam_case in range(3):
        a = {k: v.copy() for k, v in arr.items()}
        if lam_case == 1:
            a["intensity"][:] = 1000000; a["bkg"][:] = 10
            a["det"][:] = a["src"] + np.array([1400, 1400])        # far: lambda ~ 515
        if lam_case == 2:
            a["det"][:] = a["src"] + np.array([110, 0]); a["intensity"][:] = 9999999   # lambda ~ 9.1e4
        d = (a["det"][0] - a["src"][0]).astype(float)
        lam = a["intensity"][0] / np.hypot(*d) + a["bkg"][0]
        ref = np.random.default_rng(0).poisson(lam, 200000)
        for fast in (False, True):
            env = rp.RadSearch(obstruction_count=0, enforce_grid_boundaries=True, num_envs=40000, seed=9 + lam_case,
                               fast_poisson=fast)
            env.load_scenarios(**a)
            counts = []
            for _ in range(3):
                env.step_batch(None)
                counts.append(env.obs[:, 0, 0].cpu().numpy())
            c = np.concatenate(counts)
            p = stats.ks_2samp(c, ref).pvalue
            assert p > 1e-3, (lam, fast, p)
            assert abs(c.mean() - lam) < 5 * np.sqrt(lam / len(c)), (lam, fast, c.mean())
            assert abs(c.var() / lam - 1) < 0.03, (lam, fast, c.var())


def test_poisson_alias_table_ks_against_numpy():
    """RS_F_FAST_POISSON with a blocked line of sight: the count is Poisson(bkg) for the integer background rate and comes
    from the alias tables (rs_poisson_alias.h) -- KS, mean and variance against numpy for the ends and the middle of the
    table's range, and for a rate outside it (PTRS fallback)."""
    from scipy import stats

    n = 40000
    for bkg in (10, 23, 50, 77):
        env = rp.RadSearch(obstruction_count=1, enforce_grid_boundaries=True, num_envs=n, seed=100 + bkg, fast_poisson=True)
        env.load_scenarios(src=np.tile([500, 500], (n, 1)), det=np.tile([1900, 500], (n, 1)), intensity=np.full(n, 5_000_000),
                           bkg=np.full(n, bkg), rects=np.tile([[1000, 300, 1300, 700]], (n, 1, 1)), num_obs=np.ones(n))
        counts = []
        for _ in range(3):
            env.step_batch(None)
            assert bool(((env.info_flags & L.I_LOS_BLOCKED) != 0).all())
            counts.append(env.obs[:, 0, 0].cpu().numpy())
        c = np.concatenate(counts)
        ref = np.random.default_rng(bkg).poisson(bkg, 300000)
        assert stats.ks_2samp(c, ref).pvalue > 1e-3, bkg
        assert abs(c.mean() - bkg) < 5 * np.sqrt(bkg / len(c)) and abs(c.var() / bkg - 1) < 0.03, (bkg, c.mean(), c.var())
        assert c.min() >= 0 and float(c.max()) < bkg + 12 * np.sqrt(bkg)


def test_single_env_gym_api_matches_reference_shapes():
    env = rp.RadSearch(obstruction_count=3, enforce_grid_boundaries=True, np_random=np.random.default_rng(2))
    obs, rew, done, info = env.reset()
    assert set(obs) == {0} and obs[0].shape == (11,) and obs[0].dtype == np.float64
    assert set(rew) == {"team_reward", "individual_reward"} and done == {0: False}
    assert set(info[0]) == {"out_of_bounds", "out_of_bounds_count", "blocked", "scale"}
    assert env.observation_space.shape[0] == 11 and env.detectable_directions == 8 and env.number_actions == 9
    assert env.search_area[2] == (2200.0, 2200.0) and env.max_dist == 2000.0 and env.scale == 1 / 2200.0
    x, y = env.agents[0].det_coords
    assert obs[0][1] == np.float32(x / 2200.0) and len(env.obs_coord) == 3
    obs2, rew2, done2, info2 = env.step({0: 4})
    x2, y2 = env.agents[0].det_coords
    assert (x2, y2) in ((x + 100, y), (x, y))
    assert rew2["individual_reward"][0] == round(rew2["individual_reward"][0], 2)
    o3 = env.step(-1)            # idle (R:620-623)
    assert env.agents[0].det_coords == (x2, y2) and env.iter_count == 2
    env.epoch_end = True
    env.reset()
    assert env.epoch_cnt == 2 and env.iter_count == 0
    with pytest.raises(ValueError):
        env.step("left")


def test_full_size_properties_65536_envs():
    """BASELINE config sizes: invariants that hold for every env (no oracle at this size)."""
    n = 65536
    env = rp.RadSearch(obstruction_count=5, enforce_grid_boundaries=True, num_envs=n, seed=3, auto_reset=True)
    g = torch.Generator(device=env.device).manual_seed(0)
    prev_best = env._best.clone()
    tot_reset = 0
    for t in range(1, 241):
        acts = torch.randint(0, 8, (n, 1), generator=g, device=env.device, dtype=torch.int32)
        obs, rew, team, done, info, ended = env.step_batch(acts, epoch_end=(t % 120 == 0))
        rs = (ended & 4) != 0
        # detector stays inside the arena, never strictly inside an obstruction; best is a running minimum
        det = env._det[0]
        assert bool(((det >= 0) & (det < 2700)).all())
        r = env._rects
        inside = ((r[:, :, 0] < det[None, :, 0]) & (det[None, :, 0] < r[:, :, 2]) & (r[:, :, 1] < det[None, :, 1]) &
                  (det[None, :, 1] < r[:, :, 3]))
        assert not bool(inside.any())
        keep = ~rs
        assert bool((env._best[0][keep] <= prev_best[0][keep]).all())
        prev_best = env._best.clone()
        # rewards are two-decimal values; +0.1 exactly when done or improved; done => reset scheduled
        r64 = rew.double()
        assert bool((((r64 * 100).round() / 100).float() == rew).all())
        assert bool((rs | ~(done[:, 0] != 0)).all())
        assert bool((obs[:, :, 3:] >= 0).all()) and bool((obs[:, :, 3:] <= 1).all()) and bool((obs[:, :, 0] >= 0).all())
        tot_reset += int(rs.sum())
    assert int((env.status & ~2).any()) == 0
    assert tot_reset >= 2 * n
    assert int(env.steps_in_episode.max()) <= 120


@pytest.mark.parametrize("n", [3000, 6000, 40000])
def test_reset_teaming_modes_match_oracle(n):
    """The reset kernel teams 32 / 8 / 1 lanes per env depending on how many envs reset: all three give the oracle's state."""
    env, ob = make_pair(n, 1, -1, True, seed=n)
    v = pu.GpuView(env)
    pu.compare_state(v, ob, 1)
    pu.compare_obs(v.obs, ob.outs["obs"][:, :1])
    env.reset_batch(new_obstacles=False)
    ob.reset(new_obstacles=np.zeros(n, np.uint8))
    v = pu.GpuView(env)
    pu.compare_state(v, ob, 1)
    pu.compare_obs(v.obs, ob.outs["obs"][:, :1])
    np.testing.assert_array_equal(v.best[0], ob.envs["best"][:, 0])


@pytest.mark.parametrize("oc", [1, 5, 7, -1])
def test_pruned_shortest_path_is_bit_identical_on_gpu(oc):
    n = 4096
    env, ob = make_pair(n, 1, oc, True, seed=900 + oc)
    rng = np.random.default_rng(oc + 3)
    rects = env._rects.cpu().numpy()
    num_obs = (env._meta & 0xFF).cpu().numpy()
    for rep in range(3):
        pts = rng.integers(0, 2700, size=(n, 2))
        for i in range(n):
            k = num_obs[i]
            if k and rng.random() < 0.6:
                r = rects[rng.integers(0, k), i]
                c = [(r[0], r[1]), (r[0], r[3]), (r[2], r[3]), (r[2], r[1])][rng.integers(0, 4)]
                pts[i] = (c[0] + rng.integers(-120, 121) * (rng.random() < 0.7), c[1] + rng.integers(-120, 121) * (rng.random() < 0.7))
            for kk in range(k):
                r = rects[kk, i]
                if r[0] < pts[i, 0] < r[2] and r[1] < pts[i, 1] < r[3]:
                    pts[i, 0] = r[0]
        pts = np.clip(pts, 0, 2699)
        a = env.shortest_path_to(torch.as_tensor(pts), 0).cpu().numpy()
        b = env.shortest_path_to(torch.as_tensor(pts), 1).cpu().numpy()
        c = np.array([ob.shortest_path(i, pts[i]) for i in range(n)])
        np.testing.assert_array_equal(a, b)
        np.testing.assert_array_equal(a, c)


@pytest.mark.parametrize("graph", [False, True])
def test_prefetched_resets_match_oracle(graph):
    """prefetch=True (side-stream rs_prepare, optionally replayed as a CUDA graph): same rollout as the oracle's
    synchronous resets -- reset indices, new scenarios, first observations, final observations, Philox counters."""
    n, A, T, ML = 4096, 1, 150, 25
    env, ob = make_pair(n, A, 5, True, seed=77, max_ep_len=ML, auto_reset=True, prefetch=True, use_cuda_graph=graph)
    rng = np.random.default_rng(0)
    n_resets = 0
    for t in range(1, T + 1):
        acts = rng.integers(0, 8, size=(n, A))
        epoch_end = t % 60 == 0
        env.step_batch(torch.as_tensor(acts, dtype=torch.int32, device=env.device), epoch_end=epoch_end)
        ob.step(acts, env._ctr)
        e = ob.envs
        terminal, timeout = e["done"] == 1, e["ep_len"] == ML
        want = terminal * 1 | timeout * 2 | ((terminal | timeout | epoch_end) * 4)
        mask = (want & 4) != 0
        final = ob.outs["obs"][:, :A].copy()
        rew = ob.outs["reward"][:, :A].astype(np.float32).copy()
        if mask.any():
            ob.reset(mask=mask, new_obstacles=np.full(n, epoch_end))
        v = pu.GpuView(env)
        np.testing.assert_array_equal(v.ended, want)
        np.testing.assert_array_equal(v.reward, rew)
        pu.compare_obs(v.final_obs, final, sel=np.where(mask)[0])
        pu.compare_state(v, ob, A)
        np.testing.assert_array_equal(v.ep_len, e["ep_len"])
        np.testing.assert_array_equal(env._epi.cpu().numpy(), e["episode"])
        nxt = np.where(mask[:, None, None], ob.outs["obs"][:, :A], final)
        pu.compare_obs(v.obs, nxt)
        n_resets += int(mask.sum())
    assert n_resets > 5 * n
    # explicit reset / scenario injection still work with the prefetch machinery around
    env.epoch_end = True
    env.reset()
    ob.reset()
    pu.compare_state(pu.GpuView(env), ob, A)


def test_full_size_batch_matches_oracle():
    """BASELINE configs[4]'s batch (131,072 envs, 5 obstructions) through the prefetch + CUDA-graph path, 60 steps with
    staggered episodes (~66 k resets): every output of every step and the full state against the oracle, Poisson counts
    included (numpy-exact sampler on the shared Philox stream).  tests/full_size_soak.py is the same loop for T = 480."""
    n, T, ML, A = 131072, 60, 120, 1
    env, ob = make_pair(n, A, 5, True, seed=777, env_id0=0, max_ep_len=ML, auto_reset=True, prefetch=True, use_cuda_graph=True)
    g = torch.Generator(device=env.device).manual_seed(1)
    stagger = torch.randint(0, ML, (n,), generator=g, device=env.device, dtype=torch.int32)
    env._meta.add_(stagger << 16)
    ob.envs["ep_len"] = stagger.cpu().numpy()
    rng = np.random.default_rng(1)
    resets = 0
    for t in range(1, T + 1):
        acts = rng.integers(0, 8, size=(n, A))
        env.step_batch(torch.as_tensor(acts, dtype=torch.int32, device=env.device))
        ob.step(acts, env._ctr)
        e, o = ob.envs, ob.outs
        terminal, timeout = e["done"] == 1, e["ep_len"] == ML
        want = terminal * 1 | timeout * 2 | ((terminal | timeout) * 4)
        mask = (want & 4) != 0
        final = o["obs"][:, :A].copy()
        rew = o["reward"][:, :A].astype(np.float32).copy()
        if mask.any():
            ob.reset(mask=mask, new_obstacles=np.zeros(n))
        v = pu.GpuView(env)
        np.testing.assert_array_equal(v.ended, want)
        np.testing.assert_array_equal(v.reward, rew)
        pu.compare_obs(v.final_obs, final, sel=np.where(mask)[0])
        pu.compare_obs(v.obs, np.where(mask[:, None, None], o["obs"][:, :A], final))
        pu.compare_state(v, ob, A)
        resets += int(mask.sum())
    assert resets > n // 4 and int((env.status & ~2).sum()) == 0


@pytest.mark.parametrize("period", [None, 10])
def test_step_block_equals_single_steps(period):
    """RadSearch.step_block (PREFETCH_PERIOD steps + the refill rs_prepare as ONE graph launch) against the same steps taken
    one by one: identical state, outputs and Philox counters, also when blocks and single steps are mixed; with the
    default block length and with `prefetch_period=10` (episodes that end before their refill is back take the
    synchronous reset: same state) against an env that prefetches in blocks of 4."""
    n, ML = 4096, 30
    kw = dict(obstruction_count=5, enforce_grid_boundaries=True, num_envs=n, seed=123, steps_per_episode=ML, auto_reset=True,
              prefetch=True, use_cuda_graph=True)
    a, b = rp.RadSearch(**kw, prefetch_period=period), rp.RadSearch(**kw)
    P = a.PREFETCH_PERIOD
    assert P == (period or 4) and b.PREFETCH_PERIOD == 4 and a.prefetch and a.use_cuda_graph
    rng = np.random.default_rng(2)
    for rnd in range(14):
        acts = torch.as_tensor(rng.integers(0, 8, size=(P, n, 1)), dtype=torch.int32, device=a.device)
        if rnd % 5 == 4:                                 # a block taken step by step on both (mixing the two paths)
            for i in range(P):
                a.step_batch(acts[i])
        else:
            a.step_block(acts)
        for i in range(P):
            b.step_batch(acts[i])
        assert a._ctr == b._ctr
        for name in ("obs", "reward", "done_flags", "info_flags", "ended", "final_obs", "_det", "_src", "_meta", "_best", "_epi"):
            np.testing.assert_array_equal(getattr(a, name).cpu().numpy(), getattr(b, name).cpu().numpy(), err_msg=f"{name} round {rnd}")
    assert int(a._epi.sum()) > 2 * n
    with pytest.raises(ValueError):
        a.step_batch(acts[0]); a.step_block(acts)        # not at a block boundary


def test_coord_noise_and_partial_action_dicts():
    """R:570-574 `coord_noise` perturbs the reported coordinates only (state and rewards unchanged); R:645-659 a dict
    action that names a subset of the agents steps only those and reports None for the others."""
    kw = dict(obstruction_count=3, enforce_grid_boundaries=True, np_random=np.random.default_rng(5), seed=77)
    a, b = rp.RadSearch(**kw), rp.RadSearch(**dict(kw, np_random=np.random.default_rng(5)))
    b.coord_noise = True
    for act in (2, 4, 6, 0, 3):
        oa, ra, da, _ = a.step(act)
        ob_, rb, db, _ = b.step(act)
        assert ra == rb and da == db and a.agents[0].det_coords == b.agents[0].det_coords
        assert oa[0][0] == ob_[0][0] and np.array_equal(oa[0][3:], ob_[0][3:])
        d = (ob_[0][1:3] - oa[0][1:3]) / a.scale
        assert np.all(d != 0) and np.all(np.abs(d) < 40)            # N(0, 5) on the coordinates
    env = rp.RadSearch(obstruction_count=2, enforce_grid_boundaries=True, number_agents=3, seed=9)
    before = [env.agents[i].det_coords for i in range(3)]
    obs, rew, done, info = env.step({1: 4})
    assert obs[0] is None and obs[2] is None and obs[1].shape == (11,)
    assert rew["individual_reward"][0] is None and rew["individual_reward"][1] == rew["team_reward"]
    assert done[0] is None and info[2] is None and info[1]["scale"] == env.scale
    after = [env.agents[i].det_coords for i in range(3)]
    assert after[0] == before[0] and after[2] == before[2]
    assert after[1] != before[1] or info[1]["blocked"] or info[1]["out_of_bounds"]
    with pytest.raises(ValueError):
        env.step({5: 1})


def test_prefetch_is_refused_for_episodes_shorter_than_a_block():
    """An env is listed for refill once per block of PREFETCH_PERIOD steps: with 2-step episodes the prefetch machinery is
    switched off (the results are those of the synchronous resets) instead of overrunning its lists."""
    n, T, ML = 1024, 24, 2
    env, ob = make_pair(n, 1, 5, True, seed=31, max_ep_len=ML, auto_reset=True, prefetch=True, use_cuda_graph=True)
    assert not env.prefetch and not env.use_cuda_graph
    rng = np.random.default_rng(1)
    for t in range(T):
        acts = rng.integers(0, 8, size=(n, 1))
        env.step_batch(torch.as_tensor(acts, dtype=torch.int32, device=env.device))
        ob.step(acts, env._ctr)
        e = ob.envs
        mask = (e["done"] == 1) | (e["ep_len"] == ML)
        if mask.any():
            ob.reset(mask=mask, new_obstacles=np.zeros(n))
        pu.compare_state(pu.GpuView(env), ob, 1)
    assert int((env.status & L.ST_REFILL_OVERFLOW).sum()) == 0


@pytest.mark.parametrize("graph", [False, True])
def test_step_host_matches_step_batch(graph):
    """RadSearch.step_host (pinned host actions in, one packed device->host copy out, the env's own stream) gives the
    results of step_batch, also with several env batches in flight."""
    n, T = 640, 40
    kw = dict(obstruction_count=5, enforce_grid_boundaries=True, num_envs=n, seed=5, auto_reset=True,
              steps_per_episode=25, prefetch=graph, use_cuda_graph=graph)
    ref = [rp.RadSearch(env_id_offset=r * n, **kw) for r in range(2)]
    hst = [rp.RadSearch(env_id_offset=r * n, **kw) for r in range(2)]
    hbs = [e.host_buffers() for e in hst]
    rng = np.random.default_rng(3)
    acts = rng.integers(0, 8, size=(T, 2, n, 1)).astype(np.int32)
    for t in range(T):
        for r in range(2):
            hbs[r].wait()
            hbs[r].actions.copy_(torch.as_tensor(acts[t, r]))
            hst[r].step_host(hbs[r])
        for r in range(2):
            ref[r].step_batch(torch.as_tensor(acts[t, r], device=ref[r].device))
            hb = hbs[r].wait()
            for name in ("obs", "reward", "team_reward", "done_flags", "info_flags", "ended"):
                np.testing.assert_array_equal(getattr(hb, name).numpy(), getattr(ref[r], name).cpu().numpy(), err_msg=name)
    # one agent: obs 44 + reward 4 + done / info / ended 3 bytes per env (the team reward equals the reward and is a host view)
    assert n * (44 + 4 + 3) <= hbs[0].d2h_bytes < n * (44 + 4 + 4 + 3) and hbs[0].h2d_bytes == n * 4


@pytest.mark.parametrize("mode,A,fast_path,n", [(1, 1, False, 2048), (2, 1, False, 2048), (1, 4, False, 2048),
                                                (1, 1, True, 2048), (1, 1, False, 37), (2, 3, False, 101), (2, 3, False, 2048)])
def test_fused_count_standardizer_matches_callers_order(mode, A, fast_path, n):
    """RsConfig.standardize (SURVEY 8a row a20): the count channel leaves rs_step / rs_reset as the per-episode running
    z-score the RAD-A2C caller computes with StatisticStandardization (RADTEAM_core.py:188-277; mode 2: StatBuff of
    test_environment/core.py:55-79 + clip 8) in train.py's order; the oracle restatement is pinned on the reference
    classes (tests/golden/ref_standardize.npz).  Bar: the float64 z-score rounded to fp32, bit for bit; running mean and
    M2 bit for bit; raw counts unchanged.  fast_path = prefetch + CUDA-graph replay (adopted resets)."""
    T, ML = 100, 30
    kw = dict(prefetch=True, use_cuda_graph=True) if fast_path else {}
    env, ob = make_pair(n, A, 4, True, seed=31, max_ep_len=ML, auto_reset=True, standardize=mode, **kw)
    so = pu.StandardizedOracle(ob, mode)
    so.after_reset()
    np.testing.assert_array_equal(env.obs[:, :, 0].cpu().numpy(), 0.0)
    np.testing.assert_array_equal(env.raw_count.cpu().numpy(), ob.outs["obs"][:, :A, 0].astype(np.float32))
    rng = np.random.default_rng(1)
    big = 0
    for t in range(1, T + 1):
        acts = rng.integers(0, 9, size=(n, A))
        env.step_batch(torch.as_tensor(acts, dtype=torch.int32, device=env.device))
        ob.step(acts, env._ctr)
        z = so.after_step()
        e = ob.envs
        mask = (e["done"] == 1) | (e["ep_len"] == ML)
        raw = ob.outs["obs"][:, :A, 0].copy()
        big += int((np.abs(z) > 3).sum())
        np.testing.assert_array_equal(env.final_obs[:, :, 0].cpu().numpy()[mask], z[mask].astype(np.float32))
        if mask.any():
            ob.reset(mask=mask, new_obstacles=np.zeros(n))
            z = so.after_reset(mask)
            raw = np.where(mask[:, None], ob.outs["obs"][:, :A, 0], raw)
        np.testing.assert_array_equal(env.obs[:, :, 0].cpu().numpy(), z.astype(np.float32))
        np.testing.assert_array_equal(env.raw_count.cpu().numpy(), raw.astype(np.float32))
        np.testing.assert_array_equal(env._st_mean.cpu().numpy().T, so.st.mean.reshape(n, A))
        np.testing.assert_array_equal(env._st_m2.cpu().numpy().T, so.st.m2.reshape(n, A))
    pu.compare_state(pu.GpuView(env), ob, A)
    assert big > 0


@pytest.mark.parametrize("n,A,oc,enforce,T,fast_path", [(16384, 1, 5, True, 240, True), (8192, 4, -1, True, 130, False),
                                                        (8192, 2, 7, False, 130, False), (4096, 8, 3, True, 60, False)])
def test_soak_rollout_with_auto_reset_matches_oracle(n, A, oc, enforce, T, fast_path):
    """Millions of env-steps against the oracle (every output of every step: observations, rewards, done / info / ended
    flags, final observations, full state after the resets), to catch rare geometric coincidences (a grazed corner on the
    source line was found this way).  fast_path = prefetched resets + CUDA-graph replay."""
    ML = 120
    kw = dict(prefetch=True, use_cuda_graph=True) if fast_path else {}
    env, ob = make_pair(n, A, oc, enforce, seed=4242 + n + A, max_ep_len=ML, auto_reset=True, **kw)
    rng = np.random.default_rng(n + A)
    g = torch.Generator(device=env.device).manual_seed(1)
    stagger = torch.randint(0, ML, (n,), generator=g, device=env.device, dtype=torch.int32)
    env._meta.add_(stagger << 16)                                    # stagger the episodes like a long-running rollout
    ob.envs["ep_len"] = stagger.cpu().numpy()
    resets = 0
    for t in range(1, T + 1):
        acts = rng.integers(0, 9 if A > 1 else 8, size=(n, A))
        epoch_end = t == T // 2
        env.step_batch(torch.as_tensor(acts, dtype=torch.int32, device=env.device), epoch_end=epoch_end)
        ob.step(acts, env._ctr)
        e, o = ob.envs, ob.outs
        terminal, timeout = e["done"] == 1, e["ep_len"] == ML
        want = terminal * 1 | timeout * 2 | ((terminal | timeout | epoch_end) * 4)
        mask = (want & 4) != 0
        final = o["obs"][:, :A].copy()
        rew, done = o["reward"][:, :A].astype(np.float32).copy(), o["done"][:, :A].copy()
        team = o["team_reward"].astype(np.float32).copy()
        info_ref = (e["oob"][:, :A] | (e["blocked"][:, :A] * 2) | (e["collision"][:, :A] * 4) | (e["los_blocked"][:, :A] * 8)).copy()
        if mask.any():
            ob.reset(mask=mask, new_obstacles=np.full(n, epoch_end))
        v = pu.GpuView(env)
        np.testing.assert_array_equal(v.ended, want)
        np.testing.assert_array_equal(v.reward, rew)
        np.testing.assert_array_equal(v.team_reward, team)
        np.testing.assert_array_equal(v.done, done)
        np.testing.assert_array_equal(v.info & 15, info_ref)
        pu.compare_obs(v.final_obs, final, sel=np.where(mask)[0])
        pu.compare_obs(v.obs, np.where(mask[:, None, None], o["obs"][:, :A], final))
        pu.compare_state(v, ob, A)
        np.testing.assert_array_equal(v.ep_len, e["ep_len"])
        resets += int(mask.sum())
    assert resets > n


def test_results_do_not_depend_on_how_envs_are_sharded():
    """SURVEY 8e: rank r owns the contiguous global env ids shard_range(total, r, world) and keys its Philox streams with
    them, so the shards of a 3-rank job reproduce the single-rank batch bit for bit (states, observations, rewards,
    reset points) -- no collective on the data path."""
    total, T = 1000, 70
    kw = dict(obstruction_count=-1, enforce_grid_boundaries=True, number_agents=2, seed=17, steps_per_episode=25,
              auto_reset=True)
    full = rp.RadSearch(num_envs=total, **kw)
    shards = []
    for r in range(3):
        lo, hi = rp.shard_range(total, r, 3)
        shards.append((lo, hi, rp.RadSearch(num_envs=hi - lo, env_id_offset=lo, **kw)))
    rng = np.random.default_rng(8)
    for t in range(T):
        acts = torch.as_tensor(rng.integers(0, 9, size=(total, 2)), dtype=torch.int32, device=full.device)
        full.step_batch(acts, epoch_end=(t == 40))
        for lo, hi, e in shards:
            e.step_batch(acts[lo:hi], epoch_end=(t == 40))
            for name in ("obs", "reward", "team_reward", "done_flags", "info_flags", "ended", "final_obs"):
                np.testing.assert_array_equal(getattr(e, name).cpu().numpy(), getattr(full, name)[lo:hi].cpu().numpy(), err_msg=name)
            np.testing.assert_array_equal(e._det.cpu().numpy(), full._det[:, lo:hi].cpu().numpy())
            np.testing.assert_array_equal(e._src.cpu().numpy(), full._src[lo:hi].cpu().numpy())
            np.testing.assert_array_equal(e._rects.cpu().numpy(), full._rects[:, lo:hi].cpu().numpy())


@pytest.mark.parametrize("n", [4096, 76032, 76001, 98464])
def test_fast_sampler_kernel_variants_match_oracle_except_counts(n):
    """fast_poisson=True selects other instantiations of the step kernel (64-register, 8 CTAs per SM; 256-env tiles on 256
    threads from 75776 envs up; 76001 envs end in a partial tile, staged without bulk copies; 98464 envs = 3077 tiles take the
    pipelined step1p_kernel, the one bench.py times, with a last CTA that is not full).  Everything but the Poisson counts (KS-tested elsewhere) must
    still equal the oracle bit for bit: positions, flags, shortest paths, rewards, termination, resets, sensors."""
    ML, T = 60, 90
    env, ob = make_pair(n, 1, 5, True, seed=2024, max_ep_len=ML, auto_reset=True, fast_poisson=True, prefetch=True,
                        use_cuda_graph=True)
    rng = np.random.default_rng(n)
    for t in range(1, T + 1):
        acts = rng.integers(0, 8, size=(n, 1))
        env.step_batch(torch.as_tensor(acts, dtype=torch.int32, device=env.device))
        ob.step(acts, env._ctr)
        e, o = ob.envs, ob.outs
        mask = (e["done"] == 1) | (e["ep_len"] == ML)
        final = o["obs"][:, :1].copy()
        rew, done = o["reward"][:, :1].astype(np.float32).copy(), o["done"][:, :1].copy()
        if mask.any():
            ob.reset(mask=mask, new_obstacles=np.zeros(n))
        v = pu.GpuView(env)
        np.testing.assert_array_equal(v.reward, rew)
        np.testing.assert_array_equal(v.done, done)
        np.testing.assert_array_equal((v.ended & 4) != 0, mask)
        nxt = np.where(mask[:, None, None], o["obs"][:, :1], final).astype(np.float32)
        np.testing.assert_array_equal(v.obs[:, :, 1:3], nxt[:, :, 1:3])
        np.testing.assert_allclose(v.obs[:, :, 3:], nxt[:, :, 3:], rtol=1e-5, atol=0)
        np.testing.assert_allclose(v.final_obs[mask][:, :, 3:], final[mask][:, :, 3:].astype(np.float32), rtol=1e-5, atol=0)
        assert (v.obs[:, :, 0] >= 0).all()
        pu.compare_state(v, ob, 1)


def test_wide_tile_kernel_with_standardizer_is_self_consistent():
    """The 256-env-tile instantiation (fast sampler, >= 75776 envs) with RsConfig.standardize: the z-scores it writes are
    the running standardisation of the raw counts it reports (checked with the oracle's standardiser on a sample of envs;
    the counts themselves come from the fp32-acceptance sampler and are KS-tested elsewhere)."""
    n, T, ML = 76032, 45, 20
    env = rp.RadSearch(obstruction_count=5, enforce_grid_boundaries=True, num_envs=n, seed=6, steps_per_episode=ML,
                       auto_reset=True, fast_poisson=True, standardize=1, prefetch=True, use_cuda_graph=True)
    sample = np.arange(0, n, 97)
    st = co.Standardizer(len(sample), 1)
    z = st.update_standardize(env.raw_count[sample, 0].cpu().numpy())
    np.testing.assert_array_equal(env.obs[sample, 0, 0].cpu().numpy(), z.astype(np.float32))
    rng = np.random.default_rng(0)
    for t in range(T):
        acts = torch.as_tensor(rng.integers(0, 8, size=(n, 1)), dtype=torch.int32, device=env.device)
        env.step_batch(acts)
        ended = ((env.ended & 4) != 0).cpu().numpy()[sample]
        # the step's own observation is in final_obs for the envs that were reset, in obs for the others; its raw count
        # is only kept for the latter, so the reset envs restart their statistics from the new first reading
        raw = env.raw_count[sample, 0].cpu().numpy()
        live = ~ended
        z = st.update_standardize(raw, mask=live)
        np.testing.assert_array_equal(env.obs[sample, 0, 0].cpu().numpy()[live], z[live].astype(np.float32))
        st.reset(ended)
        z0 = st.update_standardize(raw, mask=ended)
        np.testing.assert_array_equal(env.obs[sample, 0, 0].cpu().numpy()[ended], z0[ended].astype(np.float32))
    assert int((env.status & ~2).sum()) == 0
