"""GPU tests (pytest -m gpu) of the fused PPO loss and gradient (rs_policy_ppo_grad, FusedGruPolicy.loss_and_grad)
against torch autograd of bench.py::ppo_update's loop (float64, and float32 with TF32 off): four shapes x M in {1, 1000,
8192} x T in {1, 37, 480} with path ends every <= 120 steps, column subsets (a team buffer's agent columns), skipped
rows, bit-identical repeats and CUDA-graph replay, accumulation into .grad, the weights after an optimiser step, and ten
Adam steps after a collector epoch against the same steps driven by torch.  Argument errors and the per-step math on the
host are CPU tests (test_policy_grad_cabi.py)."""
import copy

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import radiation_ppo_b200 as rp  # noqa: E402

DEV = torch.device("cuda:0")
SHAPES = {"bench": (11, 24, 0, 0, 0), "reference": (13, 24, 32, 32, 0), "widest": (11, 64, 64, 64, 1),
          "narrowest": (11, 1, 1, 1, 0)}
REL = 1e-4          # |g - g64|_inf <= REL |g64|_inf per parameter tensor
# ReLU heads: relu' jumps at 0, and a row whose hidden pre-activation lies within float32 rounding of 0 takes the other
# branch than float64 does, moving that head's gradient by one row's whole contribution.  Torch's own float32 update
# shows these flips (4e-5 from float64 at GRU(11->64) + 64/64 ReLU, M = 1000, T = 480), and float32 computations that
# round differently flip different rows, so for ReLU heads the bound is the larger of REL and 10x torch float32's error.
RELU_FLIP_FACTOR = 10.0


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


def params_of(mods):
    gru, pi, v = mods
    return [gru.weight_ih, gru.weight_hh, gru.bias_ih, gru.bias_hh] + list(pi.parameters()) + list(v.parameters())


def filled_buffer(T, N, seed, agents=None):
    """a BatchedPPOBuffer after get(): random rows, logp_old near the uniform policy's, path ends every <= 120 steps"""
    g = torch.Generator(device=DEV).manual_seed(seed)
    buf = rp.BatchedPPOBuffer(11, T, N if agents is None else N // agents, device=DEV, agents=agents)
    N = buf.N
    buf.obs_buf.copy_(torch.randn(T, N, 11, generator=g, device=DEV))
    buf.act_buf.copy_(torch.randint(0, 8, (T, N), generator=g, device=DEV).float())
    buf.adv_buf.copy_(torch.randn(T, N, generator=g, device=DEV))
    buf.ret_buf.copy_(torch.randn(T, N, generator=g, device=DEV))
    buf.logp_buf.copy_(np.log(1 / 8) + 0.3 * torch.randn(T, N, generator=g, device=DEV))
    length = torch.randint(1, 121, (N,), generator=g, device=DEV)
    phase = torch.randint(0, 120, (N,), generator=g, device=DEV)
    t = torch.arange(T, device=DEV)[:, None]
    end = ((t + phase) % length == length - 1) | (torch.rand(T, N, generator=g, device=DEV) < 0.01)
    buf.end_buf.copy_(end.to(torch.uint8) * torch.randint(1, 8, (T, N), generator=g, device=DEV).to(torch.uint8))
    pred = torch.rand(T, N, 2, generator=g, device=DEV)
    return buf, pred


def torch_update(mods, buf, pred, cols=None, dtype=torch.float64, clip=0.2, w_pi=1.0, w_v=0.5):
    """bench.py::ppo_update's loss on the gathered columns in torch autograd (rows with a bad column or action left out)
    -> (per-tensor gradients in float64, stats dict)"""
    gru, pi, v = (copy.deepcopy(m).to(dtype) for m in mods)
    T, N = buf.T, buf.N
    cols = torch.arange(N, device=DEV) if cols is None else cols.long()
    okc = (cols >= 0) & (cols < N)
    c = cols.clamp(0, N - 1)
    x = buf.obs_buf[:, c].to(dtype)
    if gru.input_size == 13:
        x = torch.cat([x, pred[:, c].to(dtype)], dim=2)
    act, adv, ret, logp_old, end = (b[:, c] for b in (buf.act_buf, buf.adv_buf, buf.ret_buf, buf.logp_buf, buf.end_buf))
    adv, ret, logp_old = adv.to(dtype), ret.to(dtype), logp_old.to(dtype)
    M = len(cols)
    h = torch.zeros(M, gru.hidden_size, device=DEV, dtype=dtype)
    loss = 0.0
    zero = torch.zeros((), device=DEV, dtype=dtype)
    st = torch.zeros(6, device=DEV, dtype=torch.float64)
    for t in range(T):
        h = gru(x[t], h)
        lsm = torch.log_softmax(pi(h), dim=-1)
        ok = okc & (act[t] > -1) & (act[t] < 8)
        lp = lsm.gather(1, torch.where(ok, act[t], 0.0).long()[:, None]).squeeze(1)
        ratio = torch.exp(lp - logp_old[t])
        surr = torch.minimum(ratio * adv[t], torch.clamp(ratio, 1 - clip, 1 + clip) * adv[t])
        val = v(h).squeeze(1)
        sq = (val - ret[t]) ** 2
        loss = loss - w_pi * torch.where(ok, surr, zero).sum() + w_v * torch.where(ok, sq, zero).sum()
        with torch.no_grad():
            okd = ok.double()
            st += torch.stack([-(surr * okd).sum(), (sq * okd).sum(), ((logp_old[t] - lp) * okd).sum(),
                               (-(lsm.exp() * lsm).sum(1) * okd).sum(), ((((ratio - 1).abs() > clip)) * okd).sum(),
                               (1 - okd).sum()]).double()
        h = h * (end[t] == 0)[:, None]
    loss = loss / (T * M)
    ps = params_of((gru, pi, v))
    grads = torch.autograd.grad(loss, ps)
    n = T * M - st[5]
    stats = dict(loss_pi=st[0] / (T * M), loss_v=st[1] / (T * M), approx_kl=st[2] / n, entropy=st[3] / n, clip_frac=st[4] / n,
                 skipped=st[5])
    return [gr.double() for gr in grads], stats


def fused_grads(pol, mods, buf, pred, cols=None, **kw):
    for p in params_of(mods):
        p.grad = None
    out = pol.loss_and_grad(buf, pred=pred if pol.d_in == 13 else None, columns=cols, **kw)
    return [p.grad.double().clone() for p in params_of(mods)], out


def worst(got, want):
    """max over tensors of |g - w|_inf / |w|_inf"""
    return max(((a - b).abs().max() / b.abs().max().clamp(min=1e-30)).item() for a, b in zip(got, want))


@pytest.mark.parametrize("T", [1, 37, 480])
@pytest.mark.parametrize("M", [1, 1000, 8192])
@pytest.mark.parametrize("name", list(SHAPES))
def test_gradient_matches_torch_autograd(name, M, T):
    shape = SHAPES[name]
    mods = modules(*shape, seed=M + T)
    buf, pred = filled_buffer(T, M, seed=3 * M + T)
    pol = rp.FusedGruPolicy(*mods, num_rows=M)
    got, out = fused_grads(pol, mods, buf, pred)
    g64, st64 = torch_update(mods, buf, pred)
    g32, _ = torch_update(mods, buf, pred, dtype=torch.float32)
    e64, e32, t32 = worst(got, g64), worst(got, g32), worst(g32, g64)
    print(f"{name} M={M} T={T}: fused vs f64 {e64:.2e}, vs f32 {e32:.2e}; torch f32 vs f64 {t32:.2e}")
    bound = max(REL, RELU_FLIP_FACTOR * t32) if shape[4] == 1 else REL
    assert e64 <= bound and e32 <= bound
    for k in ("loss_pi", "loss_v", "approx_kl", "entropy"):
        assert abs(out[k].item() - st64[k].item()) <= 1e-5 * max(1.0, abs(st64[k].item())), k
    assert abs(out["clip_frac"].item() - st64["clip_frac"].item()) <= 4.0 / (T * M)   # rows on the bound may flip
    assert out["skipped"].item() == 0
    assert abs(out["loss"].item() - (st64["loss_pi"] + 0.5 * st64["loss_v"]).item()) <= 1e-5 * max(1.0, abs(out["loss"].item()))


def test_column_subsets_and_team_agent_columns():
    T = 120
    for name, agents in (("bench", None), ("reference", 4)):
        shape = SHAPES[name]
        mods = modules(*shape, seed=4)
        buf, pred = filled_buffer(T, 4096, seed=9, agents=agents)
        N = buf.N
        g = torch.Generator(device=DEV).manual_seed(1)
        subsets = [torch.randperm(N, generator=g, device=DEV)[:1500], torch.randint(0, N, (777,), generator=g, device=DEV)]
        if agents:
            subsets += [torch.arange(N // agents, device=DEV) * agents + a for a in range(agents)]
        for cols in subsets:
            cols = cols.to(torch.int32)
            pol = rp.FusedGruPolicy(*mods, num_rows=len(cols))
            got, out = fused_grads(pol, mods, buf, pred, cols)
            want, st = torch_update(mods, buf, pred, cols)
            assert worst(got, want) <= REL, name
            assert abs(out["loss_pi"].item() - st["loss_pi"].item()) <= 1e-5


def test_skipped_rows_are_counted_and_left_out():
    T, N = 60, 512
    mods = modules(*SHAPES["bench"], seed=2)
    buf, pred = filled_buffer(T, N, seed=2)
    buf.act_buf[5, 7] = 8.0
    buf.act_buf[0, 100] = -1.0
    buf.act_buf[59, 3] = float("nan")
    cols = torch.arange(300, dtype=torch.int32, device=DEV)
    cols[10], cols[20], cols[299] = -1, N, 2 ** 30
    pol = rp.FusedGruPolicy(*mods, num_rows=300)
    got, out = fused_grads(pol, mods, buf, pred, cols)
    want, st = torch_update(mods, buf, pred, cols)
    assert out["skipped"].item() == st["skipped"].item() == 3 * T + 3
    assert worst(got, want) <= REL
    assert abs(out["approx_kl"].item() - st["approx_kl"].item()) <= 1e-6


def test_bit_identical_repeats_and_graph_replay():
    T, N = 96, 3000
    mods = modules(*SHAPES["reference"], seed=8)
    buf, pred = filled_buffer(T, N, seed=8)
    pol = rp.FusedGruPolicy(*mods, num_rows=N)
    first, out = fused_grads(pol, mods, buf, pred)
    again, _ = fused_grads(pol, mods, buf, pred)
    assert all(torch.equal(a, b) for a, b in zip(first, again))
    ps = params_of(mods)
    for p in ps:
        p.grad = None
    s = torch.cuda.Stream(device=DEV)
    s.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(s):
        pol.loss_and_grad(buf, pred=pred)          # warm-up: workspace and .grad exist before the capture
    torch.cuda.current_stream(DEV).wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for p in ps:
            p.grad.zero_()
        res = pol.loss_and_grad(buf, pred=pred)
    for _ in range(3):
        graph.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(p.grad.double(), a) for p, a in zip(ps, first))
        assert torch.equal(res["loss"], out["loss"]) and torch.equal(res["entropy"], out["entropy"])


def test_accumulates_into_grad_and_follows_the_optimiser():
    T, N = 50, 700
    mods = modules(*SHAPES["widest"], seed=5)
    buf, pred = filled_buffer(T, N, seed=5)
    pol = rp.FusedGruPolicy(*mods, num_rows=N)
    ps = params_of(mods)
    g, _ = fused_grads(pol, mods, buf, pred)
    base = [torch.randn_like(p) for p in ps]
    for p, b in zip(ps, base):
        p.grad = b.clone()
    pol.loss_and_grad(buf)
    assert all(torch.equal(p.grad, b + gi.float()) for p, b, gi in zip(ps, base, g))
    opt = torch.optim.Adam(ps, lr=1e-2)
    opt.step()                                     # no sync(): loss_and_grad repacks the weights itself
    got, _ = fused_grads(pol, mods, buf, pred)
    want, _ = torch_update(mods, buf, pred)
    assert worst(got, want) <= REL
    assert worst(got, g) > 1e-3                    # the weights moved


def test_adam_steps_after_a_collector_epoch_track_torch():
    """collect one epoch with the fused policy, get(), then 10 Adam steps on minibatches of 1024 columns driven by
    loss_and_grad, and the same 10 steps driven by the torch loop from the same start"""
    N, T = 4096, 240
    env = rp.RadSearch(obstruction_count=5, enforce_grid_boundaries=True, num_envs=N, seed=7, device=DEV, auto_reset=True,
                       steps_per_episode=120, prefetch=True, standardize=1)
    buf = rp.BatchedPPOBuffer(11, T, N, device=DEV)
    mods = modules(*SHAPES["bench"], seed=6)
    ref = tuple(copy.deepcopy(m) for m in mods)
    pol = rp.FusedGruPolicy(*mods, num_rows=N, seed=3)
    rp.RolloutCollector(env, buf, pol, mode="rows").collect()
    buf.get()
    opt, opt_ref = torch.optim.Adam(params_of(mods), lr=3e-4), torch.optim.Adam(params_of(ref), lr=3e-4)
    g = torch.Generator(device=DEV).manual_seed(0)
    for step in range(10):
        cols = torch.randperm(N, generator=g, device=DEV)[:1024].to(torch.int32)
        opt.zero_grad(set_to_none=True)
        out = pol.loss_and_grad(buf, columns=cols)
        opt.step()
        opt_ref.zero_grad(set_to_none=True)
        grads, st = torch_update(ref, buf, None, cols, dtype=torch.float32)
        for p, gr in zip(params_of(ref), grads):
            p.grad = gr.float()
        opt_ref.step()
        if step == 0:
            # fresh weights and the sampling policy's own log-probabilities: ratio 1 wherever the column's state was not
            # carried over from before the epoch
            assert out["approx_kl"].abs().item() < 1e-3
        assert abs(out["approx_kl"].item() - st["approx_kl"].item()) <= 1e-5
        assert abs(out["loss_pi"].item() - st["loss_pi"].item()) <= 1e-5
        assert abs(out["loss_v"].item() - st["loss_v"].item()) <= 1e-5 * max(1.0, st["loss_v"].item())
    # Adam divides by the gradient's running scale, so an entry whose gradient is ~0 may take a step of up to lr from
    # float32 noise alone: bound the worst entry by the 10 steps, and nearly every entry tightly
    for a, b in zip(params_of(mods), params_of(ref)):
        d = (a - b).abs().flatten().double()
        assert d.max().item() <= 10 * 3e-4 and torch.quantile(d, 0.99).item() <= 1e-5, "parameters drifted apart"
