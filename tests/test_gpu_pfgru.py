"""GPU tests (pytest -m gpu) of the fused PFGRU localiser (rs_pfgru_predict / peek / restart, pfgru.FusedPFGRU) against
the float64 restatement of tests/pfgru_ref.py with the same Philox noise.  The argument errors, the module rejection and
the host build of the per-row body are CPU tests (test_pfgru_cabi.py).

Dispatch table of rs_pfgru.cu (DXP = d_in rounded up to 4 or 12, HMAX = H rounded up to 16, 32 or 64) and the shape of
test_instantiation_matches_float64 that runs each entry (d_in, H, K, W, resample, alpha):
  pfgru_kernel<4, 16>    (3, 16, 33, 1, 1, 0.05)
  pfgru_kernel<4, 32>    (3, 24, 40, 24, 1, 0.7)      the reference localiser
  pfgru_kernel<4, 64>    (4, 64, 64, 64, 1, 1.0)
  pfgru_kernel<12, 16>   (11, 1, 1, 64, 1, 0.7)
  pfgru_kernel<12, 32>   (5, 32, 32, 17, 0, 0.7)      no resampling
  pfgru_kernel<12, 64>   (11, 33, 64, 8, 1, 0.3)
Each runs restart, then predict twice and peek, at 1, 257 and 65 537 rows; every call starts from the kernel's own state
("teacher forced"), so errors do not compound.  The bar is 1e-5 absolute plus 1e-5 relative of float64 for particles,
log-weights and predictions; rows with a resampling draw within 2^-20 C_{K-1} of a prefix-sum boundary are left out and
counted (float32 and float64 may pick either neighbour there).  Elsewhere the drawn indices must equal float64's."""
import pytest
import torch

from tests import pfgru_ref as ref

pytestmark = pytest.mark.gpu

import radiation_ppo_b200 as rp  # noqa: E402
from radiation_ppo_b200 import _lib as L  # noqa: E402

DEV = torch.device("cuda:0")
INSTANTIATIONS = {"4-16": (3, 16, 33, 1, 1, 0.05), "4-32": (3, 24, 40, 24, 1, 0.7), "4-64": (4, 64, 64, 64, 1, 1.0),
                  "12-16": (11, 1, 1, 64, 1, 0.7), "12-32": (5, 32, 32, 17, 0, 0.7), "12-64": (11, 33, 64, 8, 1, 0.3)}
REFERENCE = INSTANTIATIONS["4-32"]


@pytest.fixture(autouse=True)
def full_fp32():
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def localiser(shape, rows, seed=0, row_id_offset=0, mseed=0, **kw):
    d, H, K, W, rs_, alpha = shape
    mods = ref.modules(d, H, W, seed=mseed, identity=True, device=DEV)
    return rp.FusedPFGRU(*mods, num_rows=rows, num_particles=K, resamp_alpha=alpha, resample=bool(rs_), seed=seed,
                         row_id_offset=row_id_offset, **kw), mods


def observations(n, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    obs = torch.randn(n, 11, device=DEV, generator=g)
    obs[:, :3] = torch.rand(n, 3, device=DEV, generator=g)
    return obs


def recover_indices(h, h1):
    """[R, K] index i with h1[i] == h[k] (the nearest one), in chunks"""
    out = []
    for a, b in zip(h.split(2048), h1.split(2048)):
        out.append(torch.cdist(a.double(), b.double()).argmin(dim=2))
    return torch.cat(out)


def check_step(loc, mods, shape, obs, h0, p0, ctr, got_h, got_p, got_pred, blk0=0, rows=None):
    """-> (worst error / bar, particles left out) of one step against float64; asserts the indices off the boundaries"""
    d, H, K, W, rs_, alpha = shape
    rows = torch.arange(loc.row_id_offset, loc.row_id_offset + loc.rows, device=DEV) if rows is None else rows
    want = ref.step(mods, obs, h0, p0, rows, loc.seed, ctr, K, alpha, bool(rs_), blk0)
    ok = ~want["near"].any(dim=1)
    errs = [ref.close(got_pred[ok], want["pred"][ok])]
    if got_h is not None:
        errs += [ref.close(got_h[ok], want["h"][ok]), ref.close(got_p[ok], want["p"][ok])]
        if rs_:
            idx = recover_indices(got_h[ok], want["h1"][ok])
            same = (idx == want["idx"][ok]) | (want["h1"][ok].gather(1, idx[:, :, None].expand(-1, -1, H)) ==
                                              want["h"][ok]).all(dim=2)      # twin particles may swap
            assert bool(same.all()), "resampling indices differ from float64 away from the boundaries"
    return max(errs), int(want["near"].sum())


@pytest.mark.parametrize("rows", [1, 257, 65537])
@pytest.mark.parametrize("name", list(INSTANTIATIONS))
def test_instantiation_matches_float64(name, rows):
    shape = INSTANTIATIONS[name]
    d, H, K, W, rs_, alpha = shape
    loc, mods = localiser(shape, rows, seed=0xABCDEF0123 + rows, row_id_offset=3 * rows, mseed=rows)
    ids = torch.arange(3 * rows, 4 * rows, device=DEV)
    torch.cuda.synchronize()
    # the constructor's restart: U[0, 1) from the restart blocks at counter 0, p = -log K
    h_want, p_want = ref.restart_state(ids, K, H, loc.seed, 0)
    assert torch.equal(loc.particles, h_want.float()) and ref.close(loc.log_weights, p_want, 1e-6, 0) <= 1.0
    worst, left_out = 0.0, 0
    for step in range(2):
        obs = observations(rows, seed=10 * rows + step)
        h0, p0 = loc.particles.clone(), loc.log_weights.clone()
        ctr = int(loc.ctr.item())
        assert ctr == step
        pred = loc.predict(obs).clone()
        e, n = check_step(loc, mods, shape, obs, h0, p0, ctr, loc.particles, loc.log_weights, pred)
        worst, left_out = max(worst, e), left_out + n
    assert int(loc.ctr.item()) == 2 and int(loc.ticket.item()) == 0
    # peek: the peek blocks on the current state, selected rows only; state, counter and other rows untouched
    obs = observations(rows, seed=7)
    h0, p0 = loc.particles.clone(), loc.log_weights.clone()
    mask = (torch.arange(rows, device=DEV) % 3 != 1).to(torch.uint8) * L.E_TIMEOUT
    loc.pred_peek.fill_(123.0)
    out = loc.peek(obs, mask=mask, mask_bits=L.E_TIMEOUT).clone()
    assert torch.equal(loc.particles, h0) and torch.equal(loc.log_weights, p0) and int(loc.ctr.item()) == 2
    sel = mask != 0
    assert bool((out[~sel] == 123.0).all())
    e, n = check_step(loc, mods, shape, obs[sel], h0[sel], p0[sel], 2, None, None, out[sel], ref.PEEK_BLOCK,
                      rows=torch.arange(3 * rows, 4 * rows, device=DEV)[sel])
    worst, left_out = max(worst, e), left_out + n
    # a masked restart at counter 2
    loc.reset_state(mask, L.E_TIMEOUT)
    h_want, p_want = ref.restart_state(ids, K, H, loc.seed, 2)
    assert torch.equal(loc.particles[sel], h_want.float()[sel]) and torch.equal(loc.particles[~sel], h0[~sel])
    assert ref.close(loc.log_weights[sel], p_want[sel], 1e-6, 0) <= 1.0 and torch.equal(loc.log_weights[~sel], p0[~sel])
    print(f"{name} rows={rows}: worst error / bar {worst:.3f}; {left_out} particles near a boundary left out")
    assert worst <= 1.0
    assert left_out <= max(1, rows * K // 1000)


def test_shards_and_repeats_are_bit_identical():
    shape = REFERENCE
    N, cut, seed = 4099, 1701, 31
    whole, mods = localiser(shape, N, seed=seed, mseed=4)
    parts = [rp.FusedPFGRU(*mods, num_rows=cut, seed=seed), rp.FusedPFGRU(*mods, num_rows=N - cut, seed=seed,
                                                                          row_id_offset=cut)]
    again, _ = localiser(shape, N, seed=seed, mseed=4)
    mask = (torch.arange(N, device=DEV) % 5 == 0).to(torch.uint8)
    for step in range(4):
        obs = observations(N, seed=step)
        want = whole.predict(obs).clone()
        got = torch.cat([p.predict(o).clone() for p, o in zip(parts, (obs[:cut], obs[cut:]))])
        assert torch.equal(got, want) and torch.equal(again.predict(obs), want)
        assert torch.equal(torch.cat([p.particles for p in parts]), whole.particles)
        assert torch.equal(torch.cat([p.log_weights for p in parts]), whole.log_weights)
        pk = whole.peek(obs, mask).clone()
        pk_parts = torch.cat([p.peek(o, m).clone() for p, o, m in zip(parts, (obs[:cut], obs[cut:]), (mask[:cut], mask[cut:]))])
        assert torch.equal(pk[mask != 0], pk_parts[mask != 0])
        for loc, m in ((whole, mask), (parts[0], mask[:cut]), (parts[1], mask[cut:]), (again, mask)):
            loc.reset_state(m)
        assert torch.equal(torch.cat([p.particles for p in parts]), whole.particles)
        assert torch.equal(again.particles, whole.particles)


def test_captured_predict_draws_fresh_noise():
    shape = REFERENCE
    N = 3000
    cap, mods = localiser(shape, N, seed=9, mseed=5)
    plain = rp.FusedPFGRU(*mods, num_rows=N, seed=9)
    obs = observations(N, seed=1)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        cap.predict(obs)                                            # ctr 0 (warm-up on the capture stream)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        cap.predict(obs)
    plain.predict(obs)
    preds = []
    for _ in range(3):
        g.replay()
        preds.append(cap.pred.clone())
        assert torch.equal(plain.predict(obs), cap.pred)
        assert torch.equal(plain.particles, cap.particles) and torch.equal(plain.log_weights, cap.log_weights)
    assert int(cap.ctr.item()) == 4 and int(cap.ticket.item()) == 0
    assert not torch.equal(preds[0], preds[1])


def test_last_row_ids_and_counter_over_two_to_the_32():
    shape = REFERENCE
    d, H, K, W, rs_, alpha = shape
    N = 513
    loc, mods = localiser(shape, N, seed=2 ** 63 + 5, row_id_offset=2 ** 32 - N, mseed=6)
    loc.ctr.fill_(2 ** 32 - 1)
    worst = 0.0
    for step in range(2):
        obs = observations(N, seed=20 + step)
        h0, p0 = loc.particles.clone(), loc.log_weights.clone()
        pred = loc.predict(obs).clone()
        e, _ = check_step(loc, mods, shape, obs, h0, p0, 2 ** 32 - 1 + step, loc.particles, loc.log_weights, pred)
        worst = max(worst, e)
    assert int(loc.ctr.item()) == 2 ** 32 + 1
    loc.reset_state(None)
    h_want, _ = ref.restart_state(torch.arange(2 ** 32 - N, 2 ** 32, device=DEV), K, H, loc.seed, 2 ** 32 + 1)
    assert torch.equal(loc.particles, h_want.float())
    assert worst <= 1.0


class Recording:
    """A RolloutPolicy around FusedGruPolicy that keeps every bootstrap observation and prediction"""

    def __init__(self, pol):
        self.pol, self.hidden_state, self.finals = pol, pol.hidden_state, []

    def act(self, obs, pred):
        return self.pol.act(obs, pred)

    def value(self, obs, pred):
        self.finals.append((obs.clone(), pred.clone()))
        return self.pol.value(obs, pred)

    def reset_state(self, mask):
        self.pol.reset_state(mask)


@pytest.mark.parametrize("mode", ["rows", "graph"])
def test_collector_epoch_with_the_localiser(mode):
    N, T, seed = 2048, 240, 17
    d, H, K, W, rs_, alpha = REFERENCE
    env = rp.RadSearch(obstruction_count=5, enforce_grid_boundaries=True, num_envs=N, seed=7, device=DEV, auto_reset=True,
                       steps_per_episode=120, prefetch=True, use_cuda_graph=mode == "graph", standardize=1)
    buf = rp.BatchedPPOBuffer(11, T, N, device=DEV, predictions=True)
    torch.manual_seed(3)
    gru, pi, v = torch.nn.GRUCell(13, 24).to(DEV), torch.nn.Linear(24, 8).to(DEV), torch.nn.Linear(24, 1).to(DEV)
    kw = dict(obs_in=env.obs.view(N, 11), action_out=env.action_buffer.view(N)) if mode == "graph" else {}
    pol = rp.FusedGruPolicy(gru, pi, v, num_rows=N, seed=seed, **kw)
    loc, mods = localiser(REFERENCE, N, seed=seed + 1, mseed=8)
    rec = Recording(pol)
    with pytest.raises(ValueError, match="pred_buf"):
        rp.RolloutCollector(env, rp.BatchedPPOBuffer(11, T, N, device=DEV), rec, mode=mode, localizer=loc)
    rp.RolloutCollector(env, buf, rec, mode=mode, localizer=loc).collect()
    torch.cuda.synchronize()
    assert not bool(buf.pred_buf.isnan().any())
    # the same localiser calls by hand, in the collector's order, reproduce pred_buf and the bootstrap predictions
    alone = rp.FusedPFGRU(*mods, num_rows=N, num_particles=K, resamp_alpha=alpha, seed=seed + 1)
    alone.reset_state(None)
    for t in range(T):
        assert torch.equal(alone.predict(buf.obs_buf[t]), buf.pred_buf[t]), t
        end = buf.end_buf[t]
        last = t == T - 1
        cut = torch.ones(N, dtype=torch.bool, device=DEV) if last else (end & L.E_TIMEOUT) != 0
        fobs, fpred = rec.finals[t]
        assert torch.equal(alone.peek(fobs, None if last else end, L.E_TIMEOUT)[cut], fpred[cut]), t
        if not last:
            alone.reset_state(end)
    # the torch modules on the stored predictions give the stored log-probabilities and bootstrap values
    h = torch.zeros(N, 24, device=DEV)
    dl = db = 0.0
    with torch.no_grad():
        for t in range(T):
            h = gru(torch.cat([buf.obs_buf[t], buf.pred_buf[t]], dim=1), h)
            lp = torch.log_softmax(pi(h), dim=-1)
            dl = max(dl, (lp.gather(1, buf.act_buf[t].long()[:, None])[:, 0] - buf.logp_buf[t]).abs().max().item())
            end = buf.end_buf[t]
            cut = ((end & L.E_TIMEOUT) != 0) if t < T - 1 else torch.ones(N, dtype=torch.bool, device=DEV)
            fobs, fpred = rec.finals[t]
            boot = v(gru(torch.cat([fobs, fpred], dim=1), h))[:, 0]
            db = max(db, (torch.where(cut, boot, 0.0) - buf.boot_buf[t]).abs().max().item())
            h = h * (end == 0)[:, None]
    print(f"{mode}: max |d logp| {dl:.2e}, |d boot| {db:.2e}")
    assert dl < 1e-4 and db < 1e-4
    assert int(((buf.end_buf & L.E_TIMEOUT) != 0).sum()) > 0
    buf.get()
    out = pol.loss_and_grad(buf, pred=buf.pred_buf, clip_ratio=0.0)
    assert out["clip_frac"].item() == 0.0


def test_evaluator_runs_the_localiser():
    from tests import parity_util as pu

    sc = pu.load_golden("scenarios_v4")
    S, R, k = 48, 5, 5
    arr = {key: sc[f"obs{k}_{key}"][:S] for key in ("src", "det", "intensity", "bkg", "rects", "num_obs")}
    N = S * R
    torch.manual_seed(12)
    gru, pi, v = torch.nn.GRUCell(13, 24).to(DEV), torch.nn.Linear(24, 8).to(DEV), torch.nn.Linear(24, 1).to(DEV)
    results, loops = [], []
    for by_hand in (False, True):
        ev = rp.MonteCarloEvaluator(scenarios=arr, montecarlo_runs=R, steps_per_episode=120, obstruction_count=k, seed=3,
                                    enforce_grid_boundaries=True)
        pol = rp.FusedGruPolicy(gru, pi, v, num_rows=N, seed=21)
        loc, _ = localiser(REFERENCE, N, seed=22, mseed=9)
        preds = []
        if by_hand:
            def policy(obs, t):
                if t == 0:
                    loc.reset_state(None)
                    pol.reset_state(None)
                p = loc.predict(obs)
                preds.append(p.clone())
                return pol.act(obs, p)[0]
            results.append(ev.run(policy))
        else:
            def recorded(obs, t):
                p = loc(obs, t)
                preds.append(p.clone())
                return p
            results.append(ev.run(pol, localizer=recorded))
        loops.append(preds)
    a, b = results
    for f in ("success", "episode_length", "episode_return", "success_counter"):
        assert torch.equal(getattr(a, f), getattr(b, f)), f
    assert len(loops[0]) == len(loops[1]) and all(torch.equal(x, y) for x, y in zip(*loops))
