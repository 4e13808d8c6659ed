"""GPU tests (pytest -m gpu) of the fused GRU actor-critic (rs_policy_act / rs_policy_value, policy.FusedGruPolicy)
against the torch modules it replaces: the GRU step, log-probabilities and values to float32 tolerance, the sampled actions
against Gumbel-max under the oracle's Philox uniforms, their distribution, sharding over row offsets, a whole collector
epoch in both modes, sync() after an optimiser step and the Monte-Carlo evaluator.  The module rejection and the argument
errors are CPU tests (test_policy_cabi.py)."""
import numpy as np
import pytest
import torch

from oracle import c_oracle as co
from tests import parity_util as pu

pytestmark = pytest.mark.gpu

import radiation_ppo_b200 as rp  # noqa: E402
from radiation_ppo_b200 import _lib as L  # noqa: E402

DEV = torch.device("cuda:0")
ATOL = 1e-5
# (d_in, H, P, V, activation): the bench shape, the reference defaults, the widest, the narrowest
SHAPES = {"bench": (11, 24, 0, 0, 0), "reference": (13, 24, 32, 32, 0), "widest": (11, 64, 64, 64, 1),
          "narrowest": (11, 1, 1, 1, 0)}


@pytest.fixture(autouse=True)
def full_fp32():
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def modules(d_in, H, P, V, act, seed=0):
    torch.manual_seed(seed)
    A = (torch.nn.Tanh, torch.nn.ReLU)[act]
    gru = torch.nn.GRUCell(d_in, H)
    pi = torch.nn.Linear(H, 8) if P == 0 else torch.nn.Sequential(torch.nn.Linear(H, P), A(), torch.nn.Linear(P, 8))
    v = torch.nn.Linear(H, 1) if V == 0 else torch.nn.Sequential(torch.nn.Linear(H, V), A(), torch.nn.Linear(V, 1))
    return gru.to(DEV), pi.to(DEV), v.to(DEV)


def torch_step(mods, obs, pred, h):
    gru, pi, v = mods
    x = obs if pred is None else torch.cat([obs, pred], dim=1)
    with torch.no_grad():
        h1 = gru(x, h)
        return h1, torch.log_softmax(pi(h1), dim=-1), v(h1)[:, 0]


def philox_np(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 on uint32 numpy arrays (checked against the oracle's in test_numpy_philox_matches_oracle)"""
    M = np.uint64(0xFFFFFFFF)
    c = [np.asarray(x, np.uint64) & M for x in (c0, c1, c2, c3)]
    k0, k1 = np.uint64(k0), np.uint64(k1)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        c = [((p1 >> np.uint64(32)) ^ c[1] ^ k0) & M, p1 & M, ((p0 >> np.uint64(32)) ^ c[3] ^ k1) & M, p0 & M]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & M, (k1 + np.uint64(0xBB67AE85)) & M
    return c


def gumbel(seed, rows, ctr):
    """[len(rows), 8] float64 Gumbel noise of rs_policy_act's counters (rows = global row ids, ctr = call counter)"""
    rows = np.asarray(rows, np.uint64)
    k0, k1 = seed & 0xFFFFFFFF, seed >> 32
    words = []
    for b in (0, 1):
        words += philox_np(rows, np.full_like(rows, (4 << 24) | b), np.full_like(rows, ctr & 0xFFFFFFFF),
                           np.full_like(rows, ctr >> 32), k0, k1)
    u = ((np.stack(words, axis=1) >> np.uint64(8)).astype(np.float64) + 0.5) * 2.0 ** -24
    return -np.log(-np.log(u))


def gumbel_max(lp, g):
    """(argmax, mask of rows whose top-two score gap is >= 1e-4) of float64 scores"""
    sc = lp.double().cpu().numpy() + g
    top = np.sort(sc, axis=1)
    return sc.argmax(axis=1), top[:, -1] - top[:, -2] >= 1e-4


def test_numpy_philox_matches_oracle():
    rng = np.random.default_rng(0)
    for _ in range(20):
        c = [int(x) for x in rng.integers(0, 2 ** 32, 4, dtype=np.uint64)]
        k = [int(x) for x in rng.integers(0, 2 ** 32, 2, dtype=np.uint64)]
        assert [int(w[0]) for w in philox_np(*[[x] for x in c], *k)] == co.philox(c, k)


def inputs(n, d_in, H, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    obs = torch.randn(n, 11, device=DEV, generator=g)
    obs[:, 0] *= 3.0
    pred = torch.rand(n, 2, device=DEV, generator=g) if d_in == 13 else None
    h = torch.rand(n, H, device=DEV, generator=g) * 2 - 1
    return obs, pred, h


@pytest.mark.parametrize("rows", [1, 1000, 65573])
@pytest.mark.parametrize("name", list(SHAPES))
def test_act_and_value_match_torch(name, rows):
    shape = SHAPES[name]
    mods = modules(*shape, seed=rows)
    pol = rp.FusedGruPolicy(*mods, num_rows=rows, seed=5)
    obs, pred, h0 = inputs(rows, shape[0], shape[1], seed=rows)
    pol.hidden_state.copy_(h0)
    action, value, logp = pol.act(obs, pred)
    h_ref, lp_ref, v_ref = torch_step(mods, obs, pred, h0)
    dh = (pol.hidden_state - h_ref).abs().max().item()
    dv = (value - v_ref).abs().max().item()
    dl = (logp - lp_ref.gather(1, action.long()[:, None])[:, 0]).abs().max().item()
    print(f"{name} rows={rows}: max |d hidden| {dh:.2e}, |d value| {dv:.2e}, |d logp| {dl:.2e}")
    assert dh < ATOL and dv < ATOL and dl < ATOL
    assert action.dtype == torch.int32 and int(action.min()) >= 0 and int(action.max()) < 8
    # the value pass on other observations: torch's value of GRUCell(obs2, h'), hidden left bit-unchanged
    obs2, pred2, _ = inputs(rows, shape[0], shape[1], seed=rows + 1)
    h1 = pol.hidden_state.clone()
    v2 = pol.value(obs2, pred2)
    assert torch.equal(pol.hidden_state, h1)
    _, _, v2_ref = torch_step(mods, obs2, pred2, h1)
    assert (v2 - v2_ref).abs().max().item() < ATOL


def test_sampling_is_gumbel_max_of_philox_noise():
    shape = SHAPES["reference"]
    N, seed = 8192, 0xDEADBEEF12345
    mods = modules(*shape, seed=1)
    pol = rp.FusedGruPolicy(*mods, num_rows=N, seed=seed, row_id_offset=777)
    obs, pred, h0 = inputs(N, 13, 24, seed=2)
    rows = np.arange(777, 777 + N)

    def check(ctr, action):
        _, lp, _ = torch_step(mods, obs, pred, h0)
        want, clear = gumbel_max(lp, gumbel(seed, rows, ctr))
        assert clear.mean() >= 0.999
        assert np.array_equal(action.cpu().numpy()[clear], want[clear])
        return action.cpu().numpy().copy()

    pol.hidden_state.copy_(h0)
    a0 = check(0, pol.act(obs, pred)[0])
    pol.hidden_state.copy_(h0)
    a1 = check(1, pol.act(obs, pred)[0])
    assert (a0 != a1).mean() > 0.5                                  # two calls draw different noise
    assert int(pol.ctr.item()) == 2 and int(pol.ticket.item()) == 0
    # a captured act replayed twice advances the counter as well
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        pol.act(obs, pred)                                          # ctr 2 (warm-up on the capture stream)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        pol.act(obs, pred)
    for ctr in (3, 4):
        pol.hidden_state.copy_(h0)
        g.replay()
        check(ctr, pol.action)
    assert int(pol.ctr.item()) == 5


def test_action_distribution_chi_square():
    from scipy import stats

    N = 1 << 20
    mods = modules(11, 4, 0, 0, 0)
    logits = torch.tensor([0.3, -1.2, 2.0, 0.0, -0.4, 1.1, -2.5, 0.7], device=DEV)
    with torch.no_grad():
        mods[1].weight.zero_()
        mods[1].bias.copy_(logits)
    pol = rp.FusedGruPolicy(*mods, num_rows=N, seed=2024)
    obs, _, _ = inputs(N, 11, 4, seed=3)
    action, _, logp = pol.act(obs)
    p = torch.softmax(logits.double(), 0).cpu().numpy()
    assert np.allclose(logp.cpu().numpy(), np.log(p)[action.cpu().numpy()], atol=1e-6)
    counts = np.bincount(action.cpu().numpy(), minlength=8)
    chi2, pval = stats.chisquare(counts, N * p)
    print(f"chi-square {chi2:.2f} (7 dof), p = {pval:.3f}")
    assert pval > 1e-3


def test_sharded_rows_match_one_policy():
    shape = SHAPES["bench"]
    N, seed = 4099, 11
    mods = modules(*shape, seed=4)
    whole = rp.FusedGruPolicy(*mods, num_rows=N, seed=seed)
    cut = 1701
    parts = [rp.FusedGruPolicy(*mods, num_rows=cut, seed=seed),
             rp.FusedGruPolicy(*mods, num_rows=N - cut, seed=seed, row_id_offset=cut)]
    _, _, h0 = inputs(N, 11, 24, seed=5)
    whole.hidden_state.copy_(h0)
    parts[0].hidden_state.copy_(h0[:cut])
    parts[1].hidden_state.copy_(h0[cut:])
    for step in range(3):
        obs, _, _ = inputs(N, 11, 24, seed=10 + step)
        got = [p.act(o) for p, o in zip(parts, (obs[:cut], obs[cut:]))]
        want = whole.act(obs)
        for i in range(3):
            assert torch.equal(torch.cat([got[0][i], got[1][i]]), want[i])
        assert torch.equal(torch.cat([p.hidden_state for p in parts]), whole.hidden_state)
        v = torch.cat([p.value(o) for p, o in zip(parts, (obs[:cut], obs[cut:]))])
        assert torch.equal(v, whole.value(obs))


class Recording:
    """A RolloutPolicy around FusedGruPolicy that keeps a copy of every bootstrap observation (final_obs)"""

    def __init__(self, pol):
        self.pol, self.hidden_state, self.finals = pol, pol.hidden_state, []

    def act(self, obs):
        return self.pol.act(obs)

    def value(self, obs):
        self.finals.append(obs.clone())
        return self.pol.value(obs)

    def reset_state(self, mask):
        self.pol.reset_state(mask)


@pytest.mark.parametrize("mode", ["rows", "graph"])
def test_collector_epoch_matches_torch_rerun(mode):
    N, T, seed = 2048, 240, 99
    env = rp.RadSearch(obstruction_count=5, enforce_grid_boundaries=True, num_envs=N, seed=7, device=DEV, auto_reset=True,
                       steps_per_episode=120, prefetch=True, use_cuda_graph=mode == "graph", standardize=1)
    buf = rp.BatchedPPOBuffer(11, T, N, device=DEV)
    mods = modules(*SHAPES["bench"], seed=6)
    kw = dict(obs_in=env.obs.view(N, 11), action_out=env.action_buffer.view(N)) if mode == "graph" else {}
    pol = rp.FusedGruPolicy(*mods, num_rows=N, seed=seed, **kw)
    rec = Recording(pol)
    rp.RolloutCollector(env, buf, rec, mode=mode).collect()
    torch.cuda.synchronize()
    gru, pi, v = mods
    h = torch.zeros(N, 24, device=DEV)
    dv = dl = db = 0.0
    matched = total = 0
    with torch.no_grad():
        for t in range(T):
            h = gru(buf.obs_buf[t], h)
            lp = torch.log_softmax(pi(h), dim=-1)
            act = buf.act_buf[t].long()
            dv = max(dv, (v(h)[:, 0] - buf.val_buf[t]).abs().max().item())
            dl = max(dl, (lp.gather(1, act[:, None])[:, 0] - buf.logp_buf[t]).abs().max().item())
            want, clear = gumbel_max(lp, gumbel(seed, np.arange(N), t))
            matched += int(np.sum(act.cpu().numpy()[clear] == want[clear]))
            total += int(clear.sum())
            assert clear.mean() >= 0.99
            end = buf.end_buf[t]
            cut = ((end & L.E_TIMEOUT) != 0) if t < T - 1 else torch.ones(N, dtype=torch.bool, device=DEV)
            boot = v(gru(rec.finals[t], h))[:, 0]
            db = max(db, (torch.where(cut, boot, 0.0) - buf.boot_buf[t]).abs().max().item())
            h = h * (end == 0)[:, None]
    print(f"{mode}: max |d val| {dv:.2e}, |d logp| {dl:.2e}, |d boot| {db:.2e}; actions {matched}/{total} clear rows")
    assert matched == total
    assert dv < 1e-4 and dl < 1e-4 and db < 1e-4
    assert int(((buf.end_buf & L.E_TIMEOUT) != 0).sum()) > 0                      # some trajectories were cut by the timeout


def test_sync_follows_the_optimiser():
    shape = SHAPES["reference"]
    N = 3000
    mods = modules(*shape, seed=8)
    pol = rp.FusedGruPolicy(*mods, num_rows=N, seed=1)
    obs, pred, h0 = inputs(N, 13, 24, seed=9)
    _, lp_old, v_old = torch_step(mods, obs, pred, h0)
    opt = torch.optim.Adam([p for m in mods for p in m.parameters()], lr=1e-2)
    x = torch.cat([obs, pred], dim=1)
    h1 = mods[0](x, h0)
    (mods[2](h1).square().mean() - torch.log_softmax(mods[1](h1), -1)[:, 3].mean()).backward()
    opt.step()
    _, lp_new, v_new = torch_step(mods, obs, pred, h0)
    assert (v_new - v_old).abs().max().item() > 1e-3
    for want_lp, want_v, do_sync in ((lp_old, v_old, False), (lp_new, v_new, True)):
        if do_sync:
            pol.sync()
        pol.hidden_state.copy_(h0)
        a, val, lp = pol.act(obs, pred)
        assert (val - want_v).abs().max().item() < ATOL
        assert (lp - want_lp.gather(1, a.long()[:, None])[:, 0]).abs().max().item() < ATOL


@pytest.mark.parametrize("A", [1, 2])
def test_monte_carlo_evaluator_runs_the_fused_policy(A):
    sc = pu.load_golden("scenarios_v4")
    S, R, k = 48, 5, 5
    arr = {key: sc[f"obs{k}_{key}"][:S] for key in ("src", "det", "intensity", "bkg", "rects", "num_obs")}
    results = []
    for stale in (False, True):
        ev = rp.MonteCarloEvaluator(scenarios=arr, montecarlo_runs=R, steps_per_episode=120, obstruction_count=k, seed=3,
                                    enforce_grid_boundaries=True, number_agents=A)
        mods = modules(*SHAPES["bench"], seed=12)
        pol = rp.FusedGruPolicy(*mods, num_rows=S * R * A, seed=21)
        if stale:                                # a stale hidden state must not matter: t == 0 restarts every row
            pol.hidden_state.fill_(0.75)

        def policy(obs, t):
            out = pol(obs, t)
            if t == 0:                           # h' = GRUCell(obs, 0)
                x = obs.reshape(-1, 11)
                h_ref, _, _ = torch_step(mods, x, None, torch.zeros(x.shape[0], 24, device=DEV))
                assert (pol.hidden_state - h_ref).abs().max().item() < ATOL
            return out

        results.append(ev.run(policy))
    a, b = results
    for f in ("success", "episode_length", "episode_return", "success_counter"):
        assert torch.equal(getattr(a, f), getattr(b, f)), f
