"""Edge tests of the env step / reset / prefetch kernels (pytest -m gpu): every launch shape the dispatchers of
rs_kernels.cu select, driven with real actions against the oracle (oracle/radsearch_oracle.c), and built scenes that
reach the rare warp paths of the single-agent step kernel.

Bars (those of test_gpu_env.py): positions, flags, rewards, best distances, termination, reset indices, status bits and,
with the numpy-exact sampler, the Poisson counts bit for bit; sensor values within 1e-5 relative.  With fast_poisson
everything but the counts (KS-tested in test_gpu_env.py).

Launch shapes of rs_step (rs_kernels.cu) and launch_reset / rs_prepare, and the tests that run each one against the
oracle:

| launch shape                                  | chosen when                                  | test                                          |
|-----------------------------------------------|----------------------------------------------|-----------------------------------------------|
| step1_kernel<fast, KMAX=0, TB 128, OCC 7>     | A = 1, k_max = 0                             | test_single_agent_kmax_bucket_matches_oracle  |
| step1_kernel<fast, KMAX=3, OCC 7>             | A = 1, k_max 1-3                             | test_single_agent_kmax_bucket_matches_oracle  |
| step1_kernel<fast, KMAX=5, OCC 4>             | A = 1, k_max 4-5, N <= 148 * 4 * 128 = 75776 | test_kmax5_occupancy_switch_matches_oracle,   |
|                                               |                                              | test_pair_list_overflow_matches_oracle        |
| step1_kernel<fast, KMAX=5, OCC 7>             | A = 1, k_max 4-5, N > 75776                  | test_kmax5_occupancy_switch_matches_oracle    |
| step1_kernel<fast, KMAX=8, OCC 5>             | A = 1, k_max 6-8                             | test_single_agent_kmax_bucket_matches_oracle, |
|                                               |                                              | test_pair_list_overflow_matches_oracle        |
|   bulk copies, full CTAs / partial last CTA   | N % 4 == 0 (and aligned rows)                | sizes 512 / 516 of the bucket test            |
|   no bulk copies                              | N % 4 != 0                                   | size 389 of the bucket test                   |
| adoption inside step1_tile, rows of 4 k_max   | A = 1, prefetch                              | test_prefetch_adoption_at_every_row_stride,   |
|                                               |                                              | test_step_block_at_kmax8_matches_oracle       |
| reset_kernel<fast, 512, 1> (rs_prepare)       | 512 * 64 * k_max B <= 200 KB: k_max 0-6      | test_prefetch_adoption_at_every_row_stride    |
| reset_kernel<fast, 256, 2> (rs_prepare)       | k_max 7-8                                    | test_prefetch_adoption_at_every_row_stride,   |
|                                               |                                              | test_step_block_at_kmax8_matches_oracle       |
| reset_kernel<fast, 128, 1> (reset, 64 KB      | rs_reset / rs_load_scenarios at k_max = 8;   | test_reset_teaming_at_kmax8_matches_oracle    |
|   of scratch at k_max 8), 32 / 8 / 1 lanes    | <= 4096 / <= 32768 / more envs reset         |                                               |
| step_kernel<fast=true, E=64> (tile program)   | A = 2, fast_poisson                          | test_tile_program_fast_sampler_matches_oracle |
| step_kernel<fast=true, E=32>                  | A >= 3, fast_poisson                         | test_tile_program_fast_sampler_matches_oracle |
| step_kernel<*, E=32>, full row table          | A = 8, k_max = 8, standardize: 52 rows in =  | test_tile_program_full_row_table_standardizer |
|                                               | kMaxRowsIn, 48 out = kMaxRowsOut             |                                               |
"""
import numpy as np
import pytest
import torch

from oracle import c_oracle as co
from tests import parity_util as pu

pytestmark = pytest.mark.gpu

import radiation_ppo_b200 as rp  # noqa: E402
from radiation_ppo_b200 import _lib as L  # noqa: E402

HINT_SHIFT = 25
HINT_MASK = 31 << HINT_SHIFT
BIG_BEST = 1.0e9                          # a large finite running minimum: the next successful move sets best = sp


def make_pair(n, A=1, oc=5, enforce=True, seed=11, env_id0=3, max_ep_len=120, bbox=None, obs_area=None, count_law=0, **kw):
    geo, ogeo = {}, {}
    if bbox is not None:
        x0, y0, x1, y1 = bbox
        geo["bbox"] = ((x0, y0), (x1, y0), (x1, y1), (x0, y1))
        ogeo["bbox"] = bbox
    if obs_area is not None:
        geo["observation_area"] = obs_area
        ogeo["obs_area"] = obs_area
    env = rp.RadSearch(obstruction_count=oc, enforce_grid_boundaries=enforce, number_agents=A, num_envs=n, seed=seed,
                       env_id_offset=env_id0, steps_per_episode=max_ep_len, count_law=count_law, **geo, **kw)
    ob = co.OracleBatch(n, co.default_config(n_agents=A, obstruction_count=oc, enforce=int(enforce), max_ep_len=max_ep_len,
                                             count_law=count_law, **ogeo), seed=seed, env_id0=env_id0)
    ob.reset()
    return env, ob


def check_obs(got, ref64, counts, sel=None):
    if counts:
        pu.compare_obs(got, ref64, sel=sel)
        return
    ref = ref64.astype(np.float32)
    if sel is not None:
        got, ref = got[sel], ref[sel]
    np.testing.assert_array_equal(got[:, :, 1:3], ref[:, :, 1:3])
    np.testing.assert_allclose(got[:, :, 3:], ref[:, :, 3:], rtol=1e-5, atol=0)
    np.testing.assert_array_equal(got[:, :, 3:] == 0, ref[:, :, 3:] == 0)
    np.testing.assert_array_equal(got[:, :, 3:] == 1, ref[:, :, 3:] == 1)
    assert (got[:, :, 0] >= 0).all()


def auto_reset_rollout(env, ob, T, ML, counts=True, epoch_end_at=None, idle=0.0, seed=0, stagger=True, early_reject=False):
    """Soak-style rollout with the caller rules on the device: every output of every step and the full state after the
    resets against the oracle.  Returns (resets, resets left to the reset kernel) -- the latter only known without a
    CUDA graph (the graph's reset kernel empties the list).  early_reject: with prefetch, rs_prepare raises
    RS_ST_REJECT_CAP when it draws a scenario, i.e. before the oracle's reset of that episode (and also for a prepared
    scenario an epoch end discards): that bit may then be set early, every other bit must be equal."""
    n, A = ob.n, ob.A
    rng = np.random.default_rng(seed)
    if stagger:                                   # staggered episodes, like a long-running rollout
        st = rng.integers(0, ML, n).astype(np.int32)
        env._meta.add_(torch.as_tensor(st << 16, device=env.device))
        ob.envs["ep_len"] = st
    resets = listed = 0
    for t in range(1, T + 1):
        acts = rng.integers(0, 9 if A > 1 else 8, size=(n, A))
        acts[rng.random((n, A)) < idle] = 8
        epoch_end = t == epoch_end_at
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
        if early_reject:
            late = (e["status"] & L.ST_REJECT_CAP) & ~(v.status & L.ST_REJECT_CAP)
            assert not late.any()
            v.status = (v.status & ~np.uint32(L.ST_REJECT_CAP)) | (e["status"] & L.ST_REJECT_CAP)
        np.testing.assert_array_equal(v.ended, want, err_msg=f"step {t}")
        np.testing.assert_array_equal(v.reward, rew)
        np.testing.assert_array_equal(v.team_reward, team)
        np.testing.assert_array_equal(v.done, done)
        np.testing.assert_array_equal(v.info & 15, info_ref)
        check_obs(v.final_obs, final, counts, sel=np.where(mask)[0])
        check_obs(v.obs, np.where(mask[:, None, None], o["obs"][:, :A], final), counts)
        pu.compare_state(v, ob, A)
        np.testing.assert_array_equal(v.ep_len, e["ep_len"])
        resets += int(mask.sum())
        if not env.use_cuda_graph:
            listed += int(v.reset_count[0])
    return resets, listed


# ---- (a) the launch matrix ---------------------------------------------------------------------------------------------

BUCKETS = [(0, 0, True), (2, 2, False), (3, 3, True), (6, 6, True), (7, 7, False), (3, 8, True), (-1, 8, False), (7, 8, True)]


@pytest.mark.parametrize("fast", [False, True])
@pytest.mark.parametrize("n", [512, 516, 389])
@pytest.mark.parametrize("oc,k_max,enforce", BUCKETS)
def test_single_agent_kmax_bucket_matches_oracle(oc, k_max, enforce, n, fast):
    """step1_kernel<fast, KMAX, 128, OCC> for KMAX = 0 (k_max 0), 3 (k_max 2, 3) and 8 (k_max 6, 7, 8; also with fewer
    rectangles than the bucket holds: 3 or a random number in a k_max = 8 env): auto-reset rollouts with one epoch end.  n = 512:
    full 128-env CTAs with bulk copies; 516: bulk copies and a partial last CTA; 389: no bulk copies (N % 4 != 0)."""
    ML = 40
    env, ob = make_pair(n, 1, oc, enforce, seed=31 * n + k_max, max_ep_len=ML, auto_reset=True, k_max=k_max,
                        fast_poisson=fast)
    assert env._cfg.k_max == k_max
    resets, _ = auto_reset_rollout(env, ob, 70, ML, counts=not fast, epoch_end_at=35, seed=n + k_max)
    assert resets > n


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("oc,k_max", [(0, 0), (3, 3), (6, 6), (7, 7), (-1, 8)])
def test_prefetch_adoption_at_every_row_stride(oc, k_max, graph):
    """Prefetched episodes adopted inside step1_tile with source-distance rows of 4 k_max = 0, 12, 24, 28 and 32 entries
    (at most 28 filled), refilled by rs_prepare on 512-thread CTAs (k_max 0: no scratch at all; 3, 6) and on 256-thread
    CTAs (k_max 7, 8: 512 x 64 k_max B of scratch would exceed 200 KB); graph = the CUDA-graph replay of the step."""
    n, ML = 1000, 20
    env, ob = make_pair(n, 1, oc, True, seed=700 + k_max, max_ep_len=ML, auto_reset=True, prefetch=True,
                        use_cuda_graph=graph, k_max=k_max)
    assert env.prefetch and env.use_cuda_graph == graph
    resets, listed = auto_reset_rollout(env, ob, 90, ML, epoch_end_at=45, seed=k_max)
    assert resets > 3 * n
    if not graph:           # most episodes were adopted by the step kernel, not left to the reset kernel
        assert listed < resets // 2, (listed, resets)
    assert int((env.status & L.ST_REFILL_OVERFLOW).sum()) == 0


def test_step_block_at_kmax8_matches_oracle():
    """RadSearch.step_block at k_max = 8 (a random number of rectangles): step1_kernel<*, 8, 128, 5> with adoption, the straggler reset
    and rs_prepare on 256-thread CTAs in one graph; after every block the state and the block's last outputs against the
    oracle stepped one step at a time."""
    n, ML = 1000, 20
    env, ob = make_pair(n, 1, -1, True, seed=808, max_ep_len=ML, auto_reset=True, prefetch=True, use_cuda_graph=True, k_max=8)
    P = env.PREFETCH_PERIOD
    rng = np.random.default_rng(8)
    resets = 0
    for rnd in range(20):
        acts = rng.integers(0, 8, size=(P, n, 1))
        ctr0 = env._ctr
        env.step_block(torch.as_tensor(acts, dtype=torch.int32, device=env.device))
        for i in range(P):
            ob.step(acts[i], ctr0 + i + 1)
            e, o = ob.envs, ob.outs
            terminal, timeout = e["done"] == 1, e["ep_len"] == ML
            want = terminal * 1 | timeout * 2 | ((terminal | timeout) * 4)
            mask = (want & 4) != 0
            final = o["obs"][:, :1].copy()
            rew = o["reward"][:, :1].astype(np.float32).copy()
            if mask.any():
                ob.reset(mask=mask, new_obstacles=np.zeros(n))
            resets += int(mask.sum())
        assert env._ctr == ctr0 + P
        v = pu.GpuView(env)
        np.testing.assert_array_equal(v.ended, want, err_msg=f"block {rnd}")
        np.testing.assert_array_equal(v.reward, rew)
        pu.compare_obs(v.final_obs, final, sel=np.where(mask)[0])
        pu.compare_obs(v.obs, np.where(mask[:, None, None], ob.outs["obs"][:, :1], final))
        pu.compare_state(v, ob, 1)
        np.testing.assert_array_equal(v.ep_len, ob.envs["ep_len"])
        np.testing.assert_array_equal(env._epi.cpu().numpy(), ob.envs["episode"])
    assert resets > 3 * n


@pytest.mark.parametrize("n", [75776, 75780])
def test_kmax5_occupancy_switch_matches_oracle(n):
    """The KMAX = 5 bucket switches from step1_kernel<false, 5, 128, 4> (128 registers) to <false, 5, 128, 7> above
    148 x 4 x 128 = 75776 envs: the last size of the first and the first of the second (with a partial last CTA),
    numpy-exact sampler."""
    ML = 30
    env, ob = make_pair(n, 1, 5, True, seed=n, max_ep_len=ML, auto_reset=True)
    resets, _ = auto_reset_rollout(env, ob, 40, ML, seed=n)
    assert resets > n // 2


@pytest.mark.parametrize("fast_path", [False, True])
@pytest.mark.parametrize("A,n,oc", [(2, 1000, 5), (3, 601, 4), (8, 300, 7)])
def test_tile_program_fast_sampler_matches_oracle(A, n, oc, fast_path):
    """step_kernel<fast=true, E=64> (A = 2) and <fast=true, E=32> (A = 3, 8): the tile program with the fp32-acceptance
    sampler that bench.py times for multi-agent runs; everything but the counts against the oracle.  n = 601: no bulk
    copies.  fast_path = prefetch + CUDA-graph replay."""
    ML = 20
    kw = dict(prefetch=True, use_cuda_graph=True) if fast_path else {}
    env, ob = make_pair(n, A, oc, True, seed=50 + A, max_ep_len=ML, auto_reset=True, fast_poisson=True, **kw)
    resets, _ = auto_reset_rollout(env, ob, 60, ML, counts=False, epoch_end_at=30, seed=A, idle=0.1)
    assert resets > n


def test_tile_program_full_row_table_standardizer():
    """step_kernel<false, 32> with every row of its tables: A = 8, k_max = 8 (7 obstructions), standardize = 1 reads
    src, rad, meta, actions, 8 rectangle rows and 5 rows per agent (52 = kMaxRowsIn) and writes meta, obs, reward, team
    reward, done, info, ended, raw counts and 5 rows per agent (48 = kMaxRowsOut).  The z-scores bit for bit against the
    caller's running standardisation, as in test_fused_count_standardizer_matches_callers_order."""
    n, A, T, ML = 300, 8, 60, 25
    env, ob = make_pair(n, A, 7, True, seed=88, max_ep_len=ML, auto_reset=True, standardize=1, k_max=8)
    so = pu.StandardizedOracle(ob, 1)
    so.after_reset()
    np.testing.assert_array_equal(env.obs[:, :, 0].cpu().numpy(), 0.0)
    rng = np.random.default_rng(88)
    big = 0
    for t in range(1, T + 1):
        acts = rng.integers(0, 9, size=(n, A))
        env.step_batch(torch.as_tensor(acts, dtype=torch.int32, device=env.device))
        ob.step(acts, env._ctr)
        z = so.after_step()
        e = ob.envs
        mask = (e["done"] == 1) | (e["ep_len"] == ML)
        raw = ob.outs["obs"][:, :A, 0].copy()
        final = ob.outs["obs"][:, :A].copy()
        big += int((np.abs(z) > 3).sum())
        np.testing.assert_array_equal(env.final_obs[:, :, 0].cpu().numpy()[mask], z[mask].astype(np.float32))
        sel = np.where(mask)[0]
        fo = env.final_obs.cpu().numpy()[sel]
        np.testing.assert_array_equal(fo[:, :, 1:3], final[sel][:, :, 1:3].astype(np.float32))
        np.testing.assert_allclose(fo[:, :, 3:], final[sel][:, :, 3:].astype(np.float32), rtol=1e-5, atol=0)
        np.testing.assert_array_equal(env.reward.cpu().numpy(), ob.outs["reward"][:, :A].astype(np.float32))
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


@pytest.mark.parametrize("n", [3000, 6000, 40000])
def test_reset_teaming_at_kmax8_matches_oracle(n):
    """reset_kernel<false, 128, 1> with k_max = 8: 64 KB of scratch columns per CTA (above the 48 KB default), with 32,
    8 and 1 lanes per env for 3000, 6000 and 40000 envs reset; with and without new obstructions."""
    env, ob = make_pair(n, 1, -1, True, seed=n + 8, k_max=8)
    v = pu.GpuView(env)
    pu.compare_state(v, ob, 1)
    pu.compare_obs(v.obs, ob.outs["obs"][:, :1])
    for new in (False, True):
        env.reset_batch(new_obstacles=new)
        ob.reset(new_obstacles=np.full(n, new, np.uint8))
        v = pu.GpuView(env)
        pu.compare_state(v, ob, 1)
        pu.compare_obs(v.obs, ob.outs["obs"][:, :1])
    assert len(np.unique(v.num_obs)) >= 4


# ---- (b) built scenes for the rare paths --------------------------------------------------------------------------------

def marked_pairs(rects, num_obs, det, finite):
    """The marking rule of rs_step1.cuh::mark1 with an unusable hint (bound = inf), restated: corner c of rectangle k is
    marked iff it is tangent seen from det -- (x0,y0): ux*uy <= 0, (x0,y1): >= 0, (x1,y1): <= 0, (x1,y0): >= 0 with
    u = corner - det -- and its source distance dsrc is finite.  rects [n, K, 4], det [n, 2], finite [n, 4K] -> [n]."""
    n = len(det)
    out = np.zeros(n, np.int64)
    for k in range(rects.shape[1]):
        on = num_obs > k
        ux0, uy0 = rects[:, k, 0].astype(np.int64) - det[:, 0], rects[:, k, 1].astype(np.int64) - det[:, 1]
        ux1, uy1 = rects[:, k, 2].astype(np.int64) - det[:, 0], rects[:, k, 3].astype(np.int64) - det[:, 1]
        tang = [ux0 * uy0 <= 0, ux0 * uy1 >= 0, ux1 * uy1 <= 0, ux1 * uy0 >= 0]
        for c in range(4):
            out += on & tang[c] & finite[:, 4 * k + c]
    return out


def _corners(r):
    return [(r[0], r[1]), (r[0], r[3]), (r[2], r[3]), (r[2], r[1])]


def direct_segment(rects, num_obs, p, q):
    """No rectangle meets the open segment p-q in its interior: the single-agent kernel's `direct`."""
    return not any(co.seg_hits_open_rect(p, q, rects[k]) for k in range(num_obs))


def dense_scene(rng, n_rects, want_direct):
    """n_rects disjoint rectangles in the middle of the arena, source and detector outside them; the detector's segment
    to the source crosses a rectangle unless want_direct.  The detector shares its x and / or y with some rectangle
    edges in two scenes of three, which makes three or four of that rectangle's corners tangent instead of two: the
    marked counts then take every value from 2 n_rects up."""
    while True:
        rects = []
        while len(rects) < n_rects:
            w, h = (int(v) for v in rng.integers(120, 330, 2))
            x0, y0 = int(rng.integers(300, 2400 - w)), int(rng.integers(300, 2400 - h))
            r = (x0, y0, x0 + w, y0 + h)
            if all(r[0] > q[2] + 20 or q[0] > r[2] + 20 or r[1] > q[3] + 20 or q[1] > r[3] + 20 for q in rects):
                rects.append(r)
        src = (int(rng.integers(150, 2550)), int(rng.integers(150, 2550)))
        det = [int(rng.integers(150, 2550)), int(rng.integers(150, 2550))]
        align = int(rng.integers(0, 3))
        if align >= 1:
            det[0] = rects[int(rng.integers(n_rects))][int(rng.choice([0, 2]))]
        if align >= 2:
            det[1] = rects[int(rng.integers(n_rects))][int(rng.choice([1, 3]))]
        det = tuple(det)
        if any(r[0] - 5 <= p[0] <= r[2] + 5 and r[1] - 5 <= p[1] <= r[3] + 5 for r in rects for p in (src, det)):
            continue
        if np.hypot(src[0] - det[0], src[1] - det[1]) < 400:
            continue
        if direct_segment(rects, n_rects, det, src) == want_direct:
            return src, det, rects


def load_pair(n, A, k_max, src, det, rects, num_obs, fast=False, enforce=True, seed=5, count_law=0, bbox=None,
              intensity=None, bkg=None):
    rng = np.random.default_rng(seed)
    inten = intensity if intensity is not None else rng.integers(1_000_000, 10_000_000, n).astype(np.int32)
    bk = bkg if bkg is not None else rng.integers(10, 51, n).astype(np.int32)
    env, ob = make_pair(n, A, 0, enforce, seed=seed, k_max=k_max, fast_poisson=fast, count_law=count_law, bbox=bbox)
    env.load_scenarios(src, det, inten, bk, rects if k_max else None, num_obs)
    ob.load_scenarios(src, det, inten, bk, rects if k_max else np.zeros((n, 1, 4), np.int32), num_obs)
    ob.step(None, env._ctr)                         # the probe observation (counts from another Philox domain)
    ob.envs["iter_count"] = 0
    ob.envs["ep_len"] = 0
    v = pu.GpuView(env)
    np.testing.assert_array_equal(v.best[0], ob.envs["best"][:, 0])
    env._status.zero_()
    ob.envs["status"] = 0
    return env, ob


def set_hint(env, hint):
    """Write the corner hint of the next step (aflags bits 25-29) of every unit."""
    h = torch.as_tensor(np.broadcast_to(np.asarray(hint, np.int32), env._aflags.shape[1:]).copy(), device=env.device)
    env._aflags.copy_((env._aflags & ~HINT_MASK) | (h << HINT_SHIFT))


def set_best(env, ob, A, value):
    env._best.fill_(value)
    ob.envs["best"][:, :A] = value


def step_and_compare(env, ob, acts, counts):
    A = ob.A
    env.step_batch(torch.as_tensor(acts, dtype=torch.int32, device=env.device))
    ob.step(acts, env._ctr)
    v = pu.GpuView(env)
    o, e = ob.outs, ob.envs
    check_obs(v.obs, o["obs"][:, :A], counts)
    np.testing.assert_array_equal(v.reward, o["reward"][:, :A].astype(np.float32))
    np.testing.assert_array_equal(v.done, o["done"][:, :A])
    np.testing.assert_array_equal(v.team_reward, o["team_reward"].astype(np.float32))
    info_ref = e["oob"][:, :A] | (e["blocked"][:, :A] * 2) | (e["collision"][:, :A] * 4) | (e["los_blocked"][:, :A] * 8)
    np.testing.assert_array_equal(v.info & 15, info_ref)
    pu.compare_state(v, ob, A)
    return v


def compose_warps(rng, pool_counts, targets):
    """Lane assignment: for each warp, indices into the pool of obstructed scenes (-1 = a direct env, at random lanes)
    whose marked pairs add up to the target (None: all 32 lanes obstructed)."""
    out = []
    for tgt in targets:
        if tgt is None:
            out.append([int(i) for i in rng.choice(len(pool_counts), 32, replace=False)])
            continue
        for _ in range(1000):
            picks, r = [], tgt
            while r > 0:
                exact = np.where(pool_counts == r)[0]
                if len(exact) and rng.random() < 0.5 or r < pool_counts.min() * 2:
                    if not len(exact):
                        break
                    picks.append(int(rng.choice(exact)))
                    r = 0
                    break
                i = int(rng.integers(len(pool_counts)))
                picks.append(i)
                r -= int(pool_counts[i])
            if r == 0 and len(picks) < 32:
                break
        assert sum(int(pool_counts[i]) for i in picks) == tgt
        row = [-1] * 32
        for lane, i in zip(sorted(rng.choice(32, len(picks), replace=False)), picks):
            row[int(lane)] = i
        out.append(row)
    return out


@pytest.mark.parametrize("fast", [False, True])
@pytest.mark.parametrize("n_rects,k_max", [(5, 5), (7, 8)])
def test_pair_list_overflow_matches_oracle(n_rects, k_max, fast):
    """The pairs beyond kPairCap = 128 of a warp (rs_kernels.cu, step1_tile: evaluated by their own thread) in
    step1_kernel<*, 5, 128, 4> and <*, 8, 128, 5>.  Dense scenes with the source hidden, and hint corner 31 (unusable
    with at most 28 corners: the bound is infinite, so every tangent corner with a finite source distance is marked).
    Warps are composed so that they mark exactly 128, exactly 129 and several hundred pairs, asserted with the marking
    rule restated in numpy.  Then moves and idle steps with hint 31, and one idle step with a usable but poor hint (the
    visible corner farthest around).  best is set to 1e9 before the first two steps: after a step that moved (idle
    included: the reference counts it as a move, R:507-522) best is the shortest path itself, bit for bit."""
    rng = np.random.default_rng(100 * k_max + fast)
    pool = [dense_scene(rng, n_rects, False) for _ in range(120)]
    direct = [dense_scene(rng, n_rects, True) for _ in range(40)]
    pool_ob = co.OracleBatch(len(pool), co.default_config())
    pad = lambda r: np.array(r + [(0, 0, 0, 0)] * (k_max - len(r)), np.int32)   # noqa: E731
    pool_ob.load_scenarios(np.array([p[0] for p in pool]), np.array([p[1] for p in pool]), np.full(len(pool), 10 ** 6),
                           np.full(len(pool), 10), np.stack([pad(p[2]) for p in pool]), np.full(len(pool), n_rects))
    fin = np.array([[np.isfinite(pool_ob.shortest_path(i, c)) for r in p[2] for c in _corners(r)] + [False] * 4 * (k_max - n_rects)
                    for i, p in enumerate(pool)])
    pool_counts = marked_pairs(np.stack([pad(p[2]) for p in pool]), np.full(len(pool), n_rects), np.array([p[1] for p in pool]), fin)
    targets = [128, 129, None, 128, 129, None, 127, None]
    lanes = compose_warps(rng, pool_counts, targets)
    n = 32 * len(targets)
    scenes = []
    for row in lanes:
        for i in row:
            scenes.append(pool[i] if i >= 0 else direct[int(rng.integers(len(direct)))])
    src = np.array([s[0] for s in scenes], np.int32)
    det = np.array([s[1] for s in scenes], np.int32)
    rects = np.stack([pad(s[2]) for s in scenes])
    num_obs = np.full(n, n_rects, np.int32)
    env, ob = load_pair(n, 1, k_max, src, det, rects, num_obs, fast=fast, seed=k_max)
    # source distances of every corner: finite exactly where the oracle's shortest path is
    finite = np.array([[np.isfinite(ob.shortest_path(i, c)) for r in rects[i, :n_rects] for c in _corners(r)] +
                       [False] * 4 * (k_max - n_rects) for i in range(n)])
    np.testing.assert_array_equal(np.isfinite(env._dsrc.cpu().numpy()[:, :4 * n_rects]), finite[:, :4 * n_rects])

    def warp_pairs(d):
        direct_now = np.array([direct_segment(rects[i], n_rects, d[i], src[i]) for i in range(n)])
        return np.where(direct_now, 0, marked_pairs(rects, num_obs, d, finite)).reshape(-1, 32).sum(1)

    per_warp = warp_pairs(det)
    for w, tgt in enumerate(targets):
        if tgt is None:
            assert per_warp[w] > 2 * 128, per_warp
        else:
            assert per_warp[w] == tgt, (w, per_warp)
    counts = not fast
    # 1: idle with an unusable hint; best starts large, so every unit that is not done now holds best == sp
    set_hint(env, 31)
    set_best(env, ob, 1, BIG_BEST)
    step_and_compare(env, ob, np.full((n, 1), 8), counts)
    e = ob.envs
    live = e["done"] == 0
    assert live.sum() > n // 2
    np.testing.assert_array_equal(pu.GpuView(env).best[0][live], e["sp"][live, 0])
    np.testing.assert_array_equal(e["sp"][live, 0], [ob.shortest_path(i, e["det"][i, 0]) for i in np.where(live)[0]])
    # 2: moves, hint 31, best large again: where the move succeeded best is the new shortest path
    set_hint(env, 31)
    set_best(env, ob, 1, BIG_BEST)
    acts = rng.integers(0, 8, size=(n, 1))
    step_and_compare(env, ob, acts, counts)
    v = pu.GpuView(env)
    moved = ((v.info[:, 0] & L.I_MOVED) != 0) & (ob.envs["done"] == 0)
    assert moved.sum() > n // 3
    np.testing.assert_array_equal(v.best[0][moved], ob.envs["sp"][moved, 0])
    assert (warp_pairs(ob.envs["det"][:, 0]) > 128).sum() >= 3
    # 3: idle with a usable but poor hint: the visible corner with the longest path through it
    d = ob.envs["det"][:, 0]
    hint = np.full(n, 31, np.int32)
    for i in range(n):
        best_c, best_v = 31, -1.0
        for c in range(4 * n_rects):
            cx, cy = _corners(rects[i, c // 4])[c % 4]
            if finite[i, c] and direct_segment(rects[i], n_rects, d[i], (cx, cy)) and (cx, cy) != tuple(d[i]):
                val = ob.shortest_path(i, (cx, cy)) + np.hypot(cx - d[i, 0], cy - d[i, 1])
                if val > best_v:
                    best_c, best_v = c, val
        hint[i] = best_c
    assert (hint < 31).mean() > 0.9
    set_hint(env, hint)
    step_and_compare(env, ob, np.full((n, 1), 8), counts)
    # 4-7: random moves and idles, hint 31 before each
    for t in range(4):
        set_hint(env, 31)
        acts = rng.integers(0, 8, size=(n, 1))
        acts[rng.random((n, 1)) < 0.3] = 8
        step_and_compare(env, ob, acts, counts)


def edge_scenes():
    """Detector positions on obstruction edges: each corner and edge of R = (1000, 1000, 1300, 1400), the edge R shares
    with a touching rectangle, edges / corners of rectangles 60 from the arena walls, and a
    thin rectangle 20-50 from the left wall (a wall reading over an obstruction reading: RS_ST_WALL_ASSERT).  Returns rects [4, 4], source,
    and a list of (position, actions along the edge)."""
    rects = np.array([(1000, 1000, 1300, 1400), (1300, 1100, 1500, 1300), (60, 600, 400, 800), (2300, 2300, 2640, 2640),
                      (20, 1500, 50, 1700)], np.int32)
    src = (2000, 500)
    V, H = (2, 6), (0, 4)
    pos = [((1000, 1000), V + H), ((1000, 1400), V + H), ((1300, 1400), V + H), ((1300, 1000), V + H),
           ((1000, 1200), V), ((1150, 1000), H), ((1150, 1400), H), ((1300, 1050), V),
           ((1300, 1200), V), ((1300, 1100), V + H), ((1400, 1300), H), ((1400, 1100), H),
           ((60, 700), V), ((60, 600), V + H), ((200, 600), H), ((2640, 2400), V), ((2400, 2640), H), ((2640, 2640), V + H),
           ((50, 1600), V), ((50, 1500), V + H), ((100, 1600), V), ((35, 1700), H)]
    return rects, src, pos


@pytest.mark.parametrize("A", [1, 2, 4])
def test_on_edge_sensor_correction_and_wall_asserts(A):
    """Detectors standing on obstruction edges and corners (more than three rays read 1.0: correct_coords, the `fix`
    branch of step1_tile and of the tile program's phase_sense), on the edge two touching rectangles share, and on edges
    within 110 of the arena wall with enforce=True (RS_ST_WALL_ASSERT where the oracle raises it).  Idle steps and moves
    along the edge; sensors and status bits against the oracle.  A = 1: step1_kernel<false, 5, 128, 4>; A = 2, 4: the
    tile program; agents of an env start at different edge positions."""
    rects, src, pos = edge_scenes()
    plans = []
    for p, along in pos:
        for a in (8,) + along:
            plans.append((p, a))
    n = len(plans)
    rng = np.random.default_rng(A)
    det0 = np.array([p for p, _ in plans], np.int32)
    env, ob = load_pair(n, A, 5, np.tile(src, (n, 1)), det0, np.tile(rects, (n, 1, 1)), np.full(n, len(rects), np.int32),
                        seed=40 + A)
    # agent a > 0 starts at another edge position (from the same list), so the tile program sees several per env
    dets = np.zeros((n, A, 2), np.int32)
    first = np.zeros((n, A), np.int64)
    for a in range(A):
        idx = (np.arange(n) + 7 * a) % n
        dets[:, a] = det0[idx]
        first[:, a] = [plans[i][1] for i in idx]
    env._det.copy_(torch.as_tensor(dets.transpose(1, 0, 2).copy(), device=env.device))
    ob.envs["det"][:, :A] = dets
    set_best(env, ob, A, BIG_BEST)
    seen = 0
    for acts in (np.full((n, A), 8), first, np.full((n, A), 8), np.where(first == 8, 8, (first + 4) % 8), first,
                 rng.integers(0, 9, size=(n, A))):
        step_and_compare(env, ob, acts, counts=True)
        seen |= int(np.bitwise_or.reduce(ob.envs["status"]))
    assert seen & L.ST_WALL_ASSERT


def test_lambda_inf_and_coordinate_range_status():
    """RS_ST_LAMBDA_INF: a detector standing on the source (intensity / 0).  RS_ST_COORD_RANGE: a non-enforced arena
    reaching past 16383, detectors loaded at exactly +-16383 and +-16384 with their sources within 1000 (every product
    stays inside int32): the bit is set exactly for the envs whose detector ends a step outside [-16383, 16383] (the
    oracle does not model it), and everything else -- status bits excluded -- equals the oracle for the others."""
    n = 64
    rng = np.random.default_rng(3)
    src = rng.integers(500, 2000, size=(n, 2)).astype(np.int32)
    det = src.copy()                                  # on the source
    det[n // 2:] += rng.integers(-300, 300, size=(n // 2, 2)).astype(np.int32)
    env, ob = load_pair(n, 1, 0, src, det, None, np.zeros(n, np.int32), seed=9)
    step_and_compare(env, ob, np.full((n, 1), 8), counts=True)
    on_src = (ob.envs["det"][:, 0] == ob.envs["src"]).all(1)
    assert on_src.sum() >= n // 2
    np.testing.assert_array_equal((pu.GpuView(env).status & L.ST_LAMBDA_INF) != 0, on_src)

    edge = np.array([16383, 16384, -16383, -16384])
    det = np.zeros((n, 2), np.int32)
    det[:, 0] = edge[np.arange(n) % 4]
    det[:, 1] = rng.integers(-2000, 2000, n)
    det[n // 2:, [0, 1]] = det[n // 2:, [1, 0]]
    src = (det + rng.integers(-999, 1000, size=(n, 2)) * [[1, 1]]).astype(np.int32)
    src = np.clip(src, -16384, 16384)
    bbox = (-17000, -17000, 17000, 17000)
    env, ob = load_pair(n, 1, 0, src, det.astype(np.int32), None, np.zeros(n, np.int32), enforce=False, seed=10, bbox=bbox)
    ever_out = np.zeros(n, bool)
    for t in range(6):
        acts = rng.integers(0, 9, size=(n, 1))
        if t == 0:
            acts[:] = 8
        env.step_batch(torch.as_tensor(acts, dtype=torch.int32, device=env.device))
        ob.step(acts, env._ctr)
        v = pu.GpuView(env)
        d = ob.envs["det"][:, 0]
        ever_out |= (np.abs(d) > 16383).any(1)
        np.testing.assert_array_equal((v.status & L.ST_COORD_RANGE) != 0, ever_out, err_msg=f"step {t}")
        ok = ~ever_out
        assert ever_out.any() and ok.any()
        np.testing.assert_array_equal(v.det[0], d)
        pu.compare_obs(v.obs[ok], ob.outs["obs"][ok][:, :1])
        np.testing.assert_array_equal(v.best[0][ok], ob.envs["best"][ok, 0])
        np.testing.assert_array_equal(v.reward[ok], ob.outs["reward"][ok][:, :1].astype(np.float32))
        np.testing.assert_array_equal(v.done[ok], ob.outs["done"][ok][:, :1])
        np.testing.assert_array_equal(v.env_done[ok], ob.envs["done"][ok])
        np.testing.assert_array_equal(v.status[ok] & ~np.uint32(L.ST_COORD_RANGE), ob.envs["status"][ok])


# ---- (c) the configuration knobs ----------------------------------------------------------------------------------------

KNOBS = {
    "count_law1": dict(count_law=1),
    "offset_origin": dict(bbox=(300, -200, 3300, 2900), obs_area=(150, 450)),
    "tight_1720": dict(bbox=(0, 0, 1720, 1720), obs_area=(200, 500)),
    "large_16000": dict(bbox=(-16000, -16000, 16000, 16000), obs_area=(200, 500), count_law=1),
}


@pytest.mark.parametrize("prefetch", [False, True])
@pytest.mark.parametrize("A", [1, 3])
@pytest.mark.parametrize("knob", list(KNOBS))
def test_configuration_knobs_match_oracle(knob, A, prefetch):
    """count_law = 1 (inverse square) and non-default bbox / observation_area -- an offset origin with negative
    coordinates, a 1720 x 1720 arena whose search area is just above the 1000 max-distance floor (7 obstructions: the
    rejection sampling hits its cap, RS_ST_REJECT_CAP; with prefetch rs_prepare raises it when it draws the scenario,
    ahead of the reset), a +-16000 arena -- through the step, reset and prepare kernels:
    Params, wall sensors, out-of-bounds tests, search-area sampling, inv_scale and max_dist."""
    kw = KNOBS[knob]
    oc = 7 if knob == "tight_1720" else (-1 if A == 1 else 4)
    n, ML = 256 if A == 1 else 128, 20
    pf = dict(prefetch=True, use_cuda_graph=True) if prefetch else {}
    env, ob = make_pair(n, A, oc, True, seed=10 * list(KNOBS).index(knob) + A, max_ep_len=ML, auto_reset=True, **kw, **pf)
    auto_reset_rollout(env, ob, 60, ML, epoch_end_at=30, seed=A, idle=0.1 if A > 1 else 0.0,
                       early_reject=prefetch and knob == "tight_1720")
    if knob == "tight_1720":
        assert int((env.status & L.ST_REJECT_CAP).sum()) > 0


@pytest.mark.parametrize("fast", [False, True])
def test_inverse_square_law_near_the_source(fast):
    """count_law = 1 with the detector 1-110 from the source: lambda = intensity / d^2 + bkg up to ~1e7, the far end of
    the sampler (random rollouts stay below ~1e3).  Counts bit for bit with the numpy-exact sampler."""
    n = 256
    rng = np.random.default_rng(21)
    src = rng.integers(800, 1800, size=(n, 2)).astype(np.int32)
    ang = rng.uniform(0, 2 * np.pi, n)
    r = np.concatenate([np.arange(1, 11), rng.integers(1, 111, n - 10)])
    det = (src + np.stack([np.rint(r * np.cos(ang)), np.rint(r * np.sin(ang))], 1)).astype(np.int32)
    det[(det == src).all(1), 0] += 1
    inten = rng.integers(1_000_000, 10_000_000, n).astype(np.int32)
    env, ob = load_pair(n, 1, 0, src, det, None, np.zeros(n, np.int32), fast=fast, count_law=1, intensity=inten, seed=21)
    step_and_compare(env, ob, np.full((n, 1), 8), counts=not fast)
    lam = ob.outs["lam"][:, 0]
    assert lam.max() > 1e6
    if not fast:
        assert (pu.GpuView(env).obs[:, 0, 0] > 1e6).any()
