"""CPU tests of the KERNEL SOURCE: radiation_ppo_b200/csrc/rs_env_impl.cuh compiled as host C++ (tests/emu) and compared
with the oracle and with the golden vectors of the reference.  This is a debugging aid for the GPU-less build container;
the real parity tests are the `-m gpu` ones that call the CUDA library through the C ABI."""
import numpy as np
import pytest

from oracle import c_oracle as co
from radiation_ppo_b200 import _lib as L
from tests import parity_util as pu
from tests.emu.harness import EmuEnv, make_config


compare_state, compare_obs = pu.compare_state, pu.compare_obs


_DEFAULT_RUNS = [(192, 1, 5, True, 130, 0.0), (128, 1, -1, False, 90, 0.0), (96, 3, 4, True, 80, 0.2),
                 (64, 1, 0, True, 40, 0.0), (48, 2, 7, True, 60, 0.1)]
# the RadSearch knobs the runs above leave at their defaults: count_law = 1 (inverse square), bbox / observation_area
# (offset origin with negative coordinates, a 1720 x 1720 arena just above the 1000 max-distance floor, arenas spanning
# +-16000 and +-16383), k_max above the obstruction count, and single-agent runs through the tile program
_KNOB_RUNS = {
    "count_law1": ((128, 1, 5, True, 100, 0.0), dict(count_law=1)),
    "offset_bbox": ((128, 1, 5, True, 100, 0.0), dict(bbox=(300, -200, 3300, 2900), obs_area=(150, 450))),
    "offset_bbox_free": ((128, 1, 5, False, 100, 0.0), dict(bbox=(300, -200, 3300, 2900), obs_area=(150, 450))),
    "offset_bbox_a3_count_law1": ((96, 3, 4, True, 80, 0.1), dict(bbox=(300, -200, 3300, 2900), obs_area=(150, 450),
                                                                   count_law=1)),
    "offset_bbox_tiled": ((128, 1, 3, True, 80, 0.0), dict(bbox=(300, -200, 3300, 2900), obs_area=(150, 450), tiled=True)),
    "tight_1720": ((64, 1, 7, True, 60, 0.0), dict(bbox=(0, 0, 1720, 1720))),
    "tight_1720_a2": ((64, 2, 7, True, 40, 0.1), dict(bbox=(0, 0, 1720, 1720))),
    "large_16000": ((64, 1, 5, True, 60, 0.0), dict(bbox=(-16000, -16000, 16000, 16000))),
    "large_16383": ((64, 1, 5, True, 60, 0.0), dict(bbox=(-16383, -16383, 16383, 16383))),
    "kmax8": ((128, 1, -1, True, 80, 0.0), dict(k_max=8)),
}


@pytest.mark.parametrize("n,A,oc,enforce,T,idle,knobs",
                         [pytest.param(*r, {}, id="-".join(str(x) for x in r)) for r in _DEFAULT_RUNS] +
                         [pytest.param(*r, kw, id=name) for name, (r, kw) in _KNOB_RUNS.items()])
def test_emulated_kernels_match_oracle_rollout(n, A, oc, enforce, T, idle, knobs):
    seed = 1000 + n
    knobs = dict(knobs)
    tiled = knobs.pop("tiled", False)
    geo = dict(bbox=knobs.get("bbox", (0, 0, 2700, 2700)), obs_area=knobs.get("obs_area", (200, 500)),
               count_law=knobs.get("count_law", 0))
    cfg = make_config(n_agents=A, obstruction_count=oc, enforce=enforce, k_max=knobs.get("k_max"), **geo)
    ob = co.OracleBatch(n, co.default_config(n_agents=A, obstruction_count=oc, enforce=int(enforce), **geo), seed=seed,
                        env_id0=7)
    em = EmuEnv(n, cfg, seed=seed, env_id0=7, tiled=tiled)
    em.reset(0, flags=L.F_NEW_OBSTACLES)
    ob.reset()
    compare_state(em, ob, A)
    compare_obs(em.obs, ob.outs["obs"][:, :A])
    rng = np.random.default_rng(seed)
    seen = dict(los=0, sens=0, done=0, blocked=0)
    for t in range(1, T + 1):
        acts = rng.integers(0, 8, size=(n, A))
        acts[rng.random((n, A)) < idle] = 8
        em.step(acts, t)
        ob.step(acts, t)
        compare_state(em, ob, A)
        o, e = ob.outs, ob.envs
        compare_obs(em.obs, o["obs"][:, :A])
        np.testing.assert_array_equal(em.reward, o["reward"][:, :A].astype(np.float32))
        np.testing.assert_array_equal(em.done, o["done"][:, :A])
        np.testing.assert_array_equal(em.team_reward, o["team_reward"].astype(np.float32))
        info_ref = e["oob"][:, :A] | (e["blocked"][:, :A] * 2) | (e["collision"][:, :A] * 4) | (e["los_blocked"][:, :A] * 8)
        np.testing.assert_array_equal(em.info & 15, info_ref)
        seen["los"] += int((em.info & 8).astype(bool).sum()); seen["sens"] += int((em.obs[:, :, 3:] > 0).sum())
        seen["done"] += int(em.done.sum()); seen["blocked"] += int((em.info & 2).astype(bool).sum())
        mask = (e["done"] == 1) | (e["ep_len"] == 120) | (t % 45 == 0)
        if mask.any():
            newm = np.full(n, t % 45 == 0)
            em.reset(t, mask=mask, new_mask=newm)
            ob.reset(mask=mask, new_obstacles=newm)
            compare_state(em, ob, A)
            compare_obs(em.obs, ob.outs["obs"][:, :A], sel=np.where(mask)[0])
    assert seen["sens"] > 0 and (oc == 0 or seen["los"] > 0)


def test_emulated_auto_reset_matches_caller_rules():
    n, A, T = 160, 1, 150
    cfg = make_config(n_agents=A, obstruction_count=5, enforce=True, max_ep_len=40)
    ocfg = co.default_config(n_agents=A, obstruction_count=5, enforce=1, max_ep_len=40)
    ob = co.OracleBatch(n, ocfg, seed=5)
    em = EmuEnv(n, cfg, seed=5)
    em.reset(0, flags=L.F_NEW_OBSTACLES)
    ob.reset()
    rng = np.random.default_rng(0)
    for t in range(1, T + 1):
        acts = rng.integers(0, 8, size=(n, A))
        epoch_end = t % 60 == 0
        em.step(acts, t, flags=L.F_AUTO_RESET | (L.F_EPOCH_END if epoch_end else 0))
        ob.step(acts, t)
        e = ob.envs
        terminal, timeout = e["done"] == 1, e["ep_len"] == 40
        want = terminal * 1 | timeout * 2 | ((terminal | timeout | epoch_end) * 4)
        np.testing.assert_array_equal(em.ended, want)
        mask = (want & 4) != 0
        final = ob.outs["obs"][:, :A].copy()
        assert em.reset_count[0] == mask.sum()
        assert sorted(em.reset_list[: mask.sum()]) == list(np.where(mask)[0])
        compare_obs(em.final_obs, final, sel=np.where(mask)[0])
        em.reset(t, flags=L.F_RESET_LIST | (L.F_NEW_OBSTACLES if epoch_end else 0))
        if mask.any():
            ob.reset(mask=mask, new_obstacles=np.full(n, epoch_end))
        compare_state(em, ob, A)
        np.testing.assert_array_equal(em.ep_len, e["ep_len"])


def _load_records_into_emu(g, kw):
    n, A = len(g["is_reset"]), kw["n_agents"]
    oc = kw["obstruction_count"]
    cfg = make_config(n_agents=A, obstruction_count=oc, enforce=bool(kw["enforce"]), k_max=7)
    em = EmuEnv(n, cfg)
    em.load_scenarios(g["pre_src"], g["pre_det"][:, 0], g["pre_intensity"], g["pre_bkg"], g["pre_rects"][:, :7],
                      g["pre_num_obs"], uniforms=g["out_uniforms"])
    return em


@pytest.mark.parametrize("name", list(pu.STEP_FILES))
def test_emulated_kernels_reproduce_reference_records(name):
    """Every recorded reference call, replayed from its recorded pre-state with the recorded uniforms."""
    g = pu.load_golden(name)
    kw = pu.STEP_FILES[name]
    A = kw["n_agents"]
    em = _load_records_into_emu(g, kw)
    is_reset = g["is_reset"].astype(bool)
    # reset records: load_scenarios already took the step(None) probe with the recorded uniforms
    r = np.where(is_reset)[0]
    if len(r):
        compare_obs(em.obs, g["out_obs"], sel=r)
        np.testing.assert_array_equal(em.best[:, r].T, g["pre_best"][r])
    # step records: restore the remaining pre-state (agents may stand at different places) and step
    for a in range(A):
        em.det[a] = g["pre_det"][:, a]
        em.best[a] = g["pre_best"][:, a]
        em.aflags[a] = g["pre_oob_count"][:, a] | (g["pre_blocked"][:, a] << 24)
    em.meta[:] = g["pre_num_obs"] | (g["pre_done"] << 8)
    em.step(np.where(is_reset[:, None], 8, g["out_actions"]), 1, uniforms=g["out_uniforms"])
    s = np.where(~is_reset)[0]
    compare_obs(em.obs, g["out_obs"], sel=s)
    np.testing.assert_array_equal(em.reward[s], g["out_reward"][s].astype(np.float32))
    np.testing.assert_array_equal(em.done[s], g["out_done"][s])
    np.testing.assert_array_equal(em.team_reward[s], g["out_team_reward"][s].astype(np.float32))
    np.testing.assert_array_equal(em.det[:, s].transpose(1, 0, 2), g["out_det"][s])
    np.testing.assert_array_equal(em.best[:, s].T, g["out_best"][s])
    np.testing.assert_array_equal((em.aflags[:, s] & 0xFFFFFF).T, g["out_oob_count"][s])
    np.testing.assert_array_equal(((em.aflags[:, s] >> 24) & 1).T, g["out_blocked"][s])
    np.testing.assert_array_equal(((em.info[s] & 8) != 0).astype(int), g["out_los"][s])
    np.testing.assert_array_equal(((em.info[s] & 1) != 0).astype(int), g["out_oob"][s])
    assert not (em.status[s] & ~np.uint32(L.ST_LAMBDA_INF)).any()


def _sp_probe_points(rng, em_rects, num_obs, n):
    """Points spread over the arena plus points hugging obstruction edges / corners (never strictly inside one)."""
    pts = rng.integers(0, 2700, size=(n, 2))
    for i in range(n):
        k = num_obs[i]
        if k and rng.random() < 0.6:
            r = em_rects[rng.integers(0, k), i]
            c = [(r[0], r[1]), (r[0], r[3]), (r[2], r[3]), (r[2], r[1])][rng.integers(0, 4)]
            pts[i] = (c[0] + rng.integers(-120, 121) * (rng.random() < 0.7), c[1] + rng.integers(-120, 121) * (rng.random() < 0.7))
        for kk in range(k):
            r = em_rects[kk, i]
            if r[0] < pts[i, 0] < r[2] and r[1] < pts[i, 1] < r[3]:
                pts[i, 0] = r[0]
    return np.clip(pts, 0, 2699)


@pytest.mark.parametrize("oc", [1, 3, 5, 7, -1])
def test_pruned_shortest_path_is_bit_identical(oc):
    """The step kernel's pruned search (tangent corners, float lower bounds, hint) == plain min over all corners ==
    the oracle's per-call Dijkstra, to the last bit of the float64 sum."""
    n = 1500
    cfg = make_config(obstruction_count=oc, enforce=True)
    em = EmuEnv(n, cfg, seed=321 + oc)
    em.reset(0, flags=L.F_NEW_OBSTACLES)
    ob = co.OracleBatch(n, co.default_config(obstruction_count=oc, enforce=1), seed=321 + oc)
    ob.reset()
    rng = np.random.default_rng(oc + 10)
    for rep in range(4):
        pts = _sp_probe_points(rng, em.rects, em.num_obs, n)
        a = em.query_sp(pts, 0)
        b = em.query_sp(pts, 1)
        c = np.array([ob.shortest_path(i, pts[i]) for i in range(n)])
        np.testing.assert_array_equal(a, b)
        np.testing.assert_array_equal(a, c)


@pytest.mark.parametrize("skip_some_prepares", [False, True])
def test_emulated_prefetch_gives_the_same_rollout(skip_some_prepares):
    """RS_F_PREFETCH: finished envs adopt the scenario rs_prepare computed ahead of time.  Because a scenario is a pure
    function of (seed, env id, episode number, obstructions) the rollout equals the oracle's synchronous resets,
    whether a prefetched scenario was ready or not."""
    n, A, T, ML = 200, 2, 170, 25
    cfg = make_config(n_agents=A, obstruction_count=4, enforce=True, max_ep_len=ML)
    ob = co.OracleBatch(n, co.default_config(n_agents=A, obstruction_count=4, enforce=1, max_ep_len=ML), seed=8)
    em = EmuEnv(n, cfg, seed=8)
    em.reset(0, flags=L.F_NEW_OBSTACLES)
    ob.reset()
    em.prepare()                                            # everybody's second episode
    assert (em.nx_seq == em.epi + 1).all()
    rng = np.random.default_rng(1)
    used_prefetch = used_sync = 0
    for t in range(1, T + 1):
        p = t & 1
        pf = L.F_PREFETCH | (L.F_PARITY1 if p else 0)
        acts = rng.integers(0, 8, size=(n, A))
        epoch_end = t % 70 == 0
        em.refill_count[p] = 0                              # the caller starts list p
        em.step(acts, t, flags=L.F_AUTO_RESET | pf | (L.F_EPOCH_END if epoch_end else 0))
        ob.step(acts, t)
        e = ob.envs
        mask = (e["done"] == 1) | (e["ep_len"] == ML) | epoch_end
        final = ob.outs["obs"][:, :A].copy()
        assert em.reset_count[0] == mask.sum()
        ready = (em.nx_seq == em.epi + 1) & mask & (not epoch_end)
        used_prefetch += int(ready.sum())
        used_sync += int(mask.sum() - ready.sum())
        compare_obs(em.final_obs, final, sel=np.where(mask)[0])
        em.reset(t, flags=L.F_RESET_LIST | pf | (L.F_NEW_OBSTACLES if epoch_end else 0))
        assert em.refill_count[p] == mask.sum()          # adopted or recomputed, every reset env awaits rs_prepare
        if mask.any():
            ob.reset(mask=mask, new_obstacles=np.full(n, epoch_end))
        compare_state(em, ob, A)
        np.testing.assert_array_equal(em.ep_len, e["ep_len"])
        np.testing.assert_array_equal(em.epi, e["episode"])
        nxt = np.where(mask[:, None, None], ob.outs["obs"][:, :A], final)
        compare_obs(em.obs, nxt)
        if not (skip_some_prepares and t % 3 == 0):
            em.prepare(flags=L.F_REFILL_LIST | (L.F_PARITY1 if p else 0))
    assert used_prefetch >= 3 * n
    assert (used_sync > n) if skip_some_prepares else True


def _clip_exact(px, py, qx, qy, x0, y0, x1, y1, closed):
    """Liang-Barsky in exact rationals: does the (open|closed) segment meet the (open|closed) rectangle?"""
    from fractions import Fraction as F
    lo, hi = F(0), F(1)
    for p0, d, a, b in ((px, qx - px, x0, x1), (py, qy - py, y0, y1)):
        if d == 0:
            if not ((a <= p0 <= b) if closed else (a < p0 < b)):
                return False
        else:
            t0, t1 = F(a - p0, d), F(b - p0, d)
            if t0 > t1:
                t0, t1 = t1, t0
            lo, hi = max(lo, t0), min(hi, t1)
    return lo <= hi if closed else lo < hi


def test_segment_rectangle_predicate_is_exact():
    """rs_device.cuh::seg_rect (separating axes on shared cross products) against exact rational clipping, on random
    and adversarial lattice inputs: corners, edges, axis-parallel and diagonal grazing segments."""
    from tests.emu.harness import emu
    lib = emu()
    rng = np.random.default_rng(11)
    n_checked = 0
    for it in range(6000):
        x0, y0 = (int(v) for v in rng.integers(-40, 40, 2))
        x1, y1 = x0 + int(rng.integers(1, 30)), y0 + int(rng.integers(1, 30))
        pool_x = [x0, x1, x0 - 1, x1 + 1, x0 + 1, x1 - 1, int(rng.integers(-60, 60)), int(rng.integers(-60, 60))]
        pool_y = [y0, y1, y0 - 1, y1 + 1, y0 + 1, y1 - 1, int(rng.integers(-60, 60)), int(rng.integers(-60, 60))]
        px, qx = (int(v) for v in rng.choice(pool_x, 2))
        py, qy = (int(v) for v in rng.choice(pool_y, 2))
        if (px, py) == (qx, qy):
            continue
        got = lib.emu_seg_rect(px, py, qx, qy, x0, y0, x1, y1)
        want = int(_clip_exact(px, py, qx, qy, x0, y0, x1, y1, False)) | (int(_clip_exact(px, py, qx, qy, x0, y0, x1, y1, True)) << 1)
        assert got == want, (px, py, qx, qy, x0, y0, x1, y1, got, want)
        n_checked += 1
    # arena-scale coordinates (products close to 2^30)
    for it in range(3000):
        x0, y0 = (int(v) for v in rng.integers(0, 2200, 2))
        x1, y1 = x0 + int(rng.integers(200, 500)), y0 + int(rng.integers(200, 500))
        px, py, qx, qy = (int(v) for v in rng.integers(-300, 3000, 4))
        if it % 3 == 0:
            px, py = x0, int(rng.integers(y0, y1 + 1))          # start on the left edge
        got = lib.emu_seg_rect(px, py, qx, qy, x0, y0, x1, y1)
        want = int(_clip_exact(px, py, qx, qy, x0, y0, x1, y1, False)) | (int(_clip_exact(px, py, qx, qy, x0, y0, x1, y1, True)) << 1)
        assert got == want, (px, py, qx, qy, x0, y0, x1, y1, got, want)
        n_checked += 1
    assert n_checked > 8000


@pytest.mark.parametrize("lam_case", [0, 1, 2, 3])
def test_emulated_fast_poisson_is_ks_equivalent_to_numpy(lam_case):
    """RS_F_FAST_POISSON (single-precision PTRS on the Philox stream, split into first proposal + full sampler by the
    step phases) against numpy.random.Generator.poisson: KS test, mean and variance."""
    from scipy import stats

    n = 30000
    src = np.tile(np.array([[400, 400]], np.int32), (n, 1))
    det, inten, bkg = src + np.array([1400, 1400], np.int32), np.full(n, 1000000, np.int32), np.full(n, 10, np.int32)
    if lam_case == 1:
        det, inten = src + np.array([110, 0], np.int32), np.full(n, 9999999, np.int32)       # lambda ~ 9.1e4
    if lam_case == 2:
        det, inten, bkg = src + np.array([900, 300], np.int32), np.full(n, 3000000, np.int32), np.full(n, 25, np.int32)
    if lam_case == 3:
        det, inten, bkg = src + np.array([1500, 1500], np.int32), np.full(n, 1000000, np.int32), np.full(n, 10, np.int32)
        inten[:] = 1000          # lambda ~ 10.5: just above the PTRS threshold
    d = (det[0] - src[0]).astype(float)
    lam = inten[0] / np.hypot(*d) + bkg[0]
    ref = np.random.default_rng(0).poisson(lam, 200000)
    cfg = make_config(n_agents=1, obstruction_count=0, enforce=True)
    em = EmuEnv(n, cfg, seed=21 + lam_case)
    em.load_scenarios(src, det, inten, bkg, np.zeros((n, 0, 4), np.int32), np.zeros(n, np.int32))
    counts = []
    for t in range(1, 4):
        em.step(None, t, flags=L.F_FAST_POISSON)
        counts.append(em.obs[:, 0, 0].copy())
    c = np.concatenate(counts)
    assert stats.ks_2samp(c, ref).pvalue > 1e-3, lam
    assert abs(c.mean() - lam) < 5 * np.sqrt(lam / len(c)), (lam, c.mean())
    assert abs(c.var() / lam - 1) < 0.03, (lam, c.var())


@pytest.mark.parametrize("mode,A", [(1, 1), (2, 1), (1, 3)])
def test_emulated_standardizer_follows_the_callers_order(mode, A):
    """RsConfig.standardize: obs[..., 0] is the per-episode running z-score the RAD-A2C caller computes (train.py:311,
    339, 436, 469, 509, 548) and raw_count keeps the Poisson count; the statistics restart with every reset, adopted
    (prefetch) or synchronous; final_obs carries the standardised last observation used for the bootstrap value."""
    n, T, ML = 96, 90, 30
    cfg = make_config(n_agents=A, obstruction_count=3, enforce=True, max_ep_len=ML, standardize=mode)
    ob = co.OracleBatch(n, co.default_config(n_agents=A, obstruction_count=3, enforce=1, max_ep_len=ML), seed=77)
    so = pu.StandardizedOracle(ob, mode)
    em = EmuEnv(n, cfg, seed=77)
    em.reset(0, flags=L.F_NEW_OBSTACLES)
    ob.reset()
    so.after_reset()
    np.testing.assert_array_equal(em.obs[:, :, 0], 0.0)                    # a first reading standardises to 0
    np.testing.assert_array_equal(em.raw_count, ob.outs["obs"][:, :A, 0].astype(np.float32))
    em.prepare()
    rng = np.random.default_rng(3)
    big = 0
    for t in range(1, T + 1):
        p = t & 1
        pf = L.F_PREFETCH | (L.F_PARITY1 if p else 0)
        acts = rng.integers(0, 9, size=(n, A))
        em.refill_count[p] = 0
        em.step(acts, t, flags=L.F_AUTO_RESET | pf)
        ob.step(acts, t)
        z = so.after_step()
        e = ob.envs
        mask = (e["done"] == 1) | (e["ep_len"] == ML)
        np.testing.assert_array_equal(em.raw_count, ob.outs["obs"][:, :A, 0].astype(np.float32))
        np.testing.assert_array_equal(em.final_obs[mask][:, :, 0], z[mask].astype(np.float32))
        big += int((np.abs(z) > 3).sum())
        em.reset(t, flags=L.F_RESET_LIST | pf)
        if mask.any():
            ob.reset(mask=mask, new_obstacles=np.zeros(n))
            z = so.after_reset(mask)
        np.testing.assert_array_equal(em.obs[:, :, 0], z.astype(np.float32))
        raw = np.where(mask[:, None], ob.outs["obs"][:, :A, 0], em.raw_count)
        np.testing.assert_array_equal(em.raw_count, raw.astype(np.float32))
        np.testing.assert_array_equal(em.st_mean.T, so.st.mean.reshape(n, A))
        np.testing.assert_array_equal(em.st_m2.T, so.st.m2.reshape(n, A))
        if t % 2:
            em.prepare(flags=L.F_REFILL_LIST | (L.F_PARITY1 if p else 0))
    assert big > 0


def test_division_through_the_reciprocal_equals_ieee_division():
    """rs_step1.cuh::div_const (x * (1/d), one exact-residual correction) against `/` for the two launch-constant divisors of
    the commit phase, and round2_fast (Python round(x, 2) with that division) against round2 and against Python itself."""
    import ctypes as C
    from tests.emu.harness import emu
    e = emu()
    rng = np.random.default_rng(0)
    for d in (2000.0, 100.0, 1732.0, 3.0):
        xs = np.concatenate([rng.uniform(-5000, 5000, 4_000_000), -0.5 * np.sqrt(rng.integers(1, 2 ** 24, 4_000_000).astype(np.float64)),
                             rng.integers(-400, 400, 1_000_000).astype(np.float64), np.array([0.0, -0.0, np.inf, -np.inf, 1e-310, 1e300])])
        assert e.emu_div_const_mismatches(xs.ctypes.data_as(C.c_void_p), len(xs), d) == 0, d
    for x in np.concatenate([rng.uniform(-2, 1, 200_000), (rng.integers(-200, 100, 2000) + 0.5) / 100.0, [0.125, -0.125, 0.005, -0.005, 0.1]]):
        a, b = e.emu_round2_fast(float(x)), e.emu_round2(float(x))
        assert a == b == round(float(x), 2), x


def test_division_by_the_reading_count_through_the_reciprocal_table_equals_ieee_division():
    """rs_rcp.cuh::div_count (the map standardiser's x / count: table reciprocal + one exact-residual correction) against `/`
    for every divisor of the table and operands of the magnitudes the standardiser sees (count differences and squared
    distances), plus zeros, tiny, huge and non-finite values."""
    import ctypes as C
    from tests.emu.harness import emu
    e = emu()
    rng = np.random.default_rng(5)
    xs = np.concatenate([rng.normal(0, 1, 1500) * 10.0 ** rng.integers(-12, 12, 1500), rng.integers(-10**7, 10**7, 500) / 3.0,
                         rng.integers(0, 10**6, 500).astype(np.float64),
                         np.array([0.0, -0.0, 1.0, -1.0, 5e-324, 2.2e-308, 1.7e308, -1.7e308, np.inf, -np.inf, np.nan])])
    ks = np.concatenate([np.arange(1, 4096), np.array([0, -3, 4096, 5000, 2**30])]).astype(np.int32)
    bad = e.emu_div_count_mismatches(xs.ctypes.data_as(C.c_void_p), len(xs), ks.ctypes.data_as(C.c_void_p), len(ks))
    assert bad == 0


def test_prepared_segment_predicates_are_exact():
    """rs_device.cuh::seg_open1 / seg_both1 / seg_cross_open1 (segment prepared once, corner cross products by multiply-adds,
    min / max compared without forming the corner values) against exact rational clipping, like seg_rect above."""
    from tests.emu.harness import emu
    lib = emu()
    rng = np.random.default_rng(12)
    n_checked = 0
    for it in range(9000):
        if it < 6000:
            x0, y0 = (int(v) for v in rng.integers(-40, 40, 2))
            x1, y1 = x0 + int(rng.integers(1, 30)), y0 + int(rng.integers(1, 30))
            pool_x = [x0, x1, x0 - 1, x1 + 1, x0 + 1, x1 - 1, int(rng.integers(-60, 60)), int(rng.integers(-60, 60))]
            pool_y = [y0, y1, y0 - 1, y1 + 1, y0 + 1, y1 - 1, int(rng.integers(-60, 60)), int(rng.integers(-60, 60))]
            px, qx = (int(v) for v in rng.choice(pool_x, 2))
            py, qy = (int(v) for v in rng.choice(pool_y, 2))
        else:                                                           # arena scale, up to the coordinate limit
            x0, y0 = (int(v) for v in rng.integers(-16000, 15000, 2))
            x1, y1 = x0 + int(rng.integers(200, 1300)), y0 + int(rng.integers(200, 1300))
            px, py, qx, qy = (int(v) for v in rng.integers(-16383, 16384, 4))
            if it % 3 == 0:
                px, py = x0, int(rng.integers(y0, y1 + 1))
        if (px, py) == (qx, qy):
            continue
        got = lib.emu_seg_prepared(px, py, qx, qy, x0, y0, x1, y1)
        want = int(_clip_exact(px, py, qx, qy, x0, y0, x1, y1, False)) | (int(_clip_exact(px, py, qx, qy, x0, y0, x1, y1, True)) << 1)
        assert got == want, (px, py, qx, qy, x0, y0, x1, y1, got, want)
        n_checked += 1
    assert n_checked > 8000
