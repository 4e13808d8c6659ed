"""Edge tests of the fused actor-critic kernels (pytest -m gpu): every instantiation the dispatchers of rs_policy.cu and
rs_policy_grad.cu select, named from torch.profiler's CUDA activity (fixture `dispatched`), and the gradient
kernel's group, flush and lane edges, against float64 references.

Bars: the gradient within REL of float64 autograd per tensor (test_gpu_policy_grad.py's bar) and, per entry, within
C_ENTRY * 2^-24 of the entry's mass (8 with tanh heads, 512 with ReLU heads), the sum over rows of |factor| * |input|
that the kernel adds in float32 (the float64 gradient of a cancelling entry is ~0, where only this bound tests anything);
the loss statistics within 1e-5; hidden, value and log-probability within 1e-5 of torch (TF32 off), the actions
Gumbel-max of the Philox noise on clear rows.
Rows whose float64 value lies within float32 rounding of a branch point -- a ReLU head unit's pre-activation near 0, a
ratio near the clip bounds -- take either branch, moving the gradient by that row's whole contribution: the references
find them first and the tests mark their action invalid (skipped by kernel and reference alike).

policy_grad_kernel<DXP, HMAX, NACC> (rs_policy_grad.cu dispatch): DXP 12 for d_in 11, 16 for d_in 13; NACC = packed
parameters per thread, from need = ceil(count / 512).  Every table shape runs in test_gradient_at_every_instantiation
(M = 2 * 16 * SMs + 5 columns, T = 65) and test_act_and_grad_kernels_agree_exactly; count is rs_policy_param_count.

| kernel      | chosen when                  | shapes (d_in, H, P, V): count                               |
|-------------|------------------------------|-------------------------------------------------------------|
| <*, 16, 8>  | H <= 16, need <= 8           | (11,1,1,1): 64, (11,16,63,62): 4092, (13,16,60,61): 4095     |
| <*, 16, 16> | H <= 16, need > 8            | (11,16,64,61): 4099, (13,16,64,64): 4249 (largest, H <= 16)  |
| <*, 32, 8>  | H 17..32, need <= 8          | (11,17,1,0): 1582, (11,27,5,23): 4096, (13,29,6,1): 4096     |
| <*, 32, 16> | H 17..32, need 9..16         | (11,17,56,58): 4097, (11,30,63,58): 8192, (13,17,55,54):     |
|             |                              | 4097, (13,32,63,32): 8192                                   |
| <*, 32, 32> | H 17..32, need > 16          | (11,32,42,63): 8193, (11,32,64,64): 9129, (13,31,63,42):     |
|             |                              | 8193, (13,32,64,64): 9321                                   |
| <*, 64, 16> | H 33..64, need <= 16         | (11,33,1,0): 4638, (11,37,53,5): 8192, (13,33,1,0): 4836,    |
|             |                              | (13,34,23,61): 8192                                         |
| <*, 64, 32> | H 33..64, need 17..32        | (11,34,42,44): 8193, (11,55,28,59): 16384, (13,34,54,24):    |
|             |                              | 8193, (13,53,64,29): 16384                                  |
| <*, 64, 48> | H 33..64, need > 32          | (11,52,50,59): 16385, (11,64,64,64): 23689, (13,51,64,46):   |
|             |                              | 16385, (13,64,64,64): 24073 (the largest network)           |

policy_kernel<DXP, HMAX> (rs_policy.cu dispatch, act and value): HMAX 16 for H <= 16, 32 for H <= 32, 64 above; all six
run in test_act_and_value_at_every_instantiation (the same shapes, 1, 257 and 400 003 rows: more rows than the grid holds
at once, so the grid-stride loop repeats) and test_act_and_grad_kernels_agree_exactly.

Gradient kernel edges and their tests:
  columns 1, 15, 16, 17, 16 SMs, 16 SMs + 1; invalid columns at warps that held a valid column in the CTA's earlier group;
  all columns invalid; duplicate columns                                       test_group_and_column_edges
  T = 1, 31, 32, 33, 64, 481 (float32 flushes at t % 32 == 0); an end at every step; no end in T = 2049
                                                                               test_time_and_path_end_edges, test_long_bptt
  paired columns with negated advantages (float64 gradient ~0); bench shape at M = 16 384, T = 480
                                                                               test_cancelling_columns, test_bench_shape_*
  w_pi = 0, w_v = 0, clip_ratio = 0, ratios e^+-30, logits of +-50            test_loss_parameter_edges, test_large_logits
Inference noise at the last row ids and across the 2^32 call counter: test_noise_at_counter_and_row_id_limits.
"""
import copy
import ctypes as C
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import radiation_ppo_b200 as rp  # noqa: E402
from radiation_ppo_b200 import _lib as L  # noqa: E402
from tests.test_gpu_policy import gumbel, gumbel_max, inputs, torch_step  # noqa: E402
from tests.test_gpu_policy_grad import (REL, RELU_FLIP_FACTOR, filled_buffer, modules, params_of,  # noqa: E402
                                        torch_update, worst)

DEV = torch.device("cuda:0")
ATOL = 1e-5
C_ENTRY = (8.0, 512.0)  # |g - g64| <= C_ENTRY[act] 2^-24 mass per entry, tanh / ReLU heads (see entry_ratio)
EPS = 2.0 ** -24
BRANCH_TOL = 1e-4      # relative distance from a branch point under which a row counts as ambiguous
BENCH = (11, 24, 0, 0, 0)
WIDE13 = (13, 33, 17, 64, 1)

# (gradient kernel (DXP, HMAX, NACC), shapes (d_in, H, P, V)) -- the table of the module docstring, in its order
TABLE = [((12, 16, 8), [(11, 1, 1, 1), (11, 16, 63, 62)]), ((12, 16, 16), [(11, 16, 64, 61)]),
         ((16, 16, 8), [(13, 16, 60, 61)]), ((16, 16, 16), [(13, 16, 64, 64)]),
         ((12, 32, 8), [(11, 17, 1, 0), (11, 27, 5, 23)]), ((12, 32, 16), [(11, 17, 56, 58), (11, 30, 63, 58)]),
         ((12, 32, 32), [(11, 32, 42, 63), (11, 32, 64, 64)]), ((16, 32, 8), [(13, 29, 6, 1)]),
         ((16, 32, 16), [(13, 17, 55, 54), (13, 32, 63, 32)]), ((16, 32, 32), [(13, 31, 63, 42), (13, 32, 64, 64)]),
         ((12, 64, 16), [(11, 33, 1, 0), (11, 37, 53, 5)]), ((12, 64, 32), [(11, 34, 42, 44), (11, 55, 28, 59)]),
         ((12, 64, 48), [(11, 52, 50, 59), (11, 64, 64, 64)]), ((16, 64, 16), [(13, 33, 1, 0), (13, 34, 23, 61)]),
         ((16, 64, 32), [(13, 34, 54, 24), (13, 53, 64, 29)]), ((16, 64, 48), [(13, 51, 64, 46), (13, 64, 64, 64)])]
# tanh and ReLU alternate down the table, so that every (DXP, HMAX) runs both activations
CASES = [(kern, shape + (i % 2,)) for i, (kern, shape) in enumerate((k, s) for k, ss in TABLE for s in ss)]
CASE_IDS = ["{}-{}-{}-{}-{}".format(*shape[:4], ("tanh", "relu")[shape[4]]) for _, shape in CASES]

KERNEL_NAME = re.compile(r"(policy(?:_grad)?_kernel<[^>]*>)")


@pytest.fixture(autouse=True)
def full_fp32():
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def sms():
    return torch.cuda.get_device_properties(DEV).multi_processor_count


def param_count(d, H, P, V):
    """policy_layout's packed count, restated"""
    return 3 * H * d + 3 * H * H + 6 * H + (8 * H + 8 if P == 0 else P * H + P + 8 * P + 8) + (H + 1 if V == 0 else V * H + 2 * V + 1)


def expected_kernels(d, H, P, V):
    """(gradient kernel, inference kernel) the dispatchers should pick"""
    need = -(-param_count(d, H, P, V) // 512)
    dxp = 12 if d == 11 else 16
    if H <= 16:
        hmax, nacc = 16, 8 if need <= 8 else 16
    elif H <= 32:
        hmax, nacc = 32, 8 if need <= 8 else 16 if need <= 16 else 32
    else:
        hmax, nacc = 64, 16 if need <= 16 else 32 if need <= 32 else 48
    return (dxp, hmax, nacc), (dxp, hmax)


def profile_dispatch():
    """Print (JSON) the policy kernels torch.profiler's CUDA activity names, in launch order, for one loss_and_grad, act and
    value call of every table shape.  The dispatchers pick a kernel from the network's config alone (not from M, T or the
    row count), so small calls name the kernels of the tests' calls.  Run in a child process by the fixture `dispatched`."""
    calls = []
    for _, shape in CASES:
        mods = modules(*shape, seed=1)
        pol = rp.FusedGruPolicy(*mods, num_rows=3, seed=1)
        buf, pred = filled_buffer(2, 5, seed=1)
        obs, pred1, _ = inputs(3, shape[0], shape[1], seed=1)
        calls.append((pol, mods, buf, pred, obs, pred1))
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for pol, mods, buf, pred, obs, pred1 in calls:
            fused(pol, mods, buf, pred)
            pol.act(obs, pred1)
            pol.value(obs, pred1)
        torch.cuda.synchronize()
    events = sorted(prof.events(), key=lambda e: e.time_range.start)
    print(json.dumps([m.group(1) for m in (KERNEL_NAME.search(e.name) for e in events) if m]))


@pytest.fixture(scope="module")
def dispatched():
    """{shape: [gradient kernel, act kernel, value kernel]} from profile_dispatch, run in a child process so that the
    test process opens no torch.profiler session.  With sessions opened in the pytest process next to this file's tests,
    later sessions in that process -- test_gpu_ppo_edges.py names the GAE kernels from them -- came back without CUDA
    kernel activity."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = "from tests.test_gpu_policy_edges import profile_dispatch; profile_dispatch()"
    run = subprocess.run([sys.executable, "-c", code], cwd=root, capture_output=True, text=True, timeout=600)
    assert run.returncode == 0, run.stderr[-4000:]
    names = json.loads(run.stdout.strip().splitlines()[-1])
    assert len(names) == 3 * len(CASES), names
    return {shape: names[3 * i:3 * i + 3] for i, (_, shape) in enumerate(CASES)}


def _keep(t):
    if t.requires_grad:
        t.retain_grad()


def _head(ps, i0, z, act, saved):
    """a Linear or Linear-act-Linear head on z in float64; records (weight index, bias index, output, input) per layer"""
    if len(ps) == 2:
        out = z @ ps[0].T + ps[1]
        _keep(out)
        saved.append((i0, i0 + 1, out, z))
        return out, None
    pre = z @ ps[0].T + ps[1]
    _keep(pre)
    saved.append((i0, i0 + 1, pre, z))
    a = torch.tanh(pre) if act == 0 else torch.relu(pre)
    out = a @ ps[2].T + ps[3]
    _keep(out)
    saved.append((i0 + 2, i0 + 3, out, a))
    return out, (pre, (z.abs() @ ps[0].abs().T + ps[1].abs()))


def _reference_chunk(mods, act, buf, pred, cols, norm, clip, w_pi, w_v, self_ratio, branches, dtype=torch.float64):
    T, N = buf.T, buf.N
    ps = [p.detach().to(dtype).clone().requires_grad_(not branches) for p in params_of(mods)]
    w_ih, w_hh, b_ih, b_hh = ps[:4]
    n_pi = len(list(mods[1].parameters()))
    pi_ps, v_ps = ps[4:4 + n_pi], ps[4 + n_pi:]
    okc = (cols >= 0) & (cols < N)
    c = cols.clamp(0, N - 1)
    x = buf.obs_buf[:, c].to(dtype)
    if mods[0].input_size == 13:
        x = torch.cat([x, pred[:, c].to(dtype)], dim=2)
    a_t, adv, ret, logp_old, end = (b[:, c] for b in (buf.act_buf, buf.adv_buf, buf.ret_buf, buf.logp_buf, buf.end_buf))
    adv, ret, logp_old = adv.to(dtype), ret.to(dtype), logp_old.to(dtype)
    H = mods[0].hidden_size
    h = torch.zeros(len(cols), H, device=DEV, dtype=dtype)
    zero = torch.zeros((), device=DEV, dtype=dtype)
    loss = 0.0
    saved = []
    st = torch.zeros(6, device=DEV, dtype=torch.float64)
    amb = torch.zeros(T, len(cols), device=DEV, dtype=torch.bool)
    for t in range(T):
        hp = h
        gi = x[t] @ w_ih.T + b_ih
        gh = hp @ w_hh.T + b_hh
        _keep(gi)
        _keep(gh)
        saved += [(0, 2, gi, x[t]), (1, 3, gh, hp)]
        ir, iz, i_n = gi.chunk(3, 1)
        hr, hz, hn = gh.chunk(3, 1)
        r, z = torch.sigmoid(ir + hr), torch.sigmoid(iz + hz)
        n = torch.tanh(i_n + r * hn)
        h = n + z * (hp - n)
        logits, pre_pi = _head(pi_ps, 4, h, act, saved)
        val, pre_v = _head(v_ps, 4 + n_pi, h, act, saved)
        val = val[:, 0]
        lsm = torch.log_softmax(logits, dim=-1)
        ok = okc & (a_t[t] > -1) & (a_t[t] < 8)
        lp = lsm.gather(1, torch.where(ok, a_t[t], 0.0).long()[:, None]).squeeze(1)
        lpo = lp.detach() if self_ratio else logp_old[t]
        ratio = torch.exp(lp - lpo)
        surr = torch.minimum(ratio * adv[t], torch.clamp(ratio, 1 - clip, 1 + clip) * adv[t])
        sq = (val - ret[t]) ** 2
        loss = loss - w_pi * torch.where(ok, surr, zero).sum() + w_v * torch.where(ok, sq, zero).sum()
        with torch.no_grad():
            okd = ok.to(dtype)
            st += torch.stack([-(surr * okd).sum(), (sq * okd).sum(), ((lpo - lp) * okd).sum(),
                               (-(lsm.exp() * lsm).sum(1) * okd).sum(), (((ratio - 1).abs() > clip) * okd).sum(),
                               (1 - okd).sum()]).double()
            if branches:
                for pre in (pre_pi, pre_v):
                    if pre is not None and act == 1:
                        amb[t] |= ((pre[0].abs() <= BRANCH_TOL * pre[1]).any(1))
                if not self_ratio:
                    for bound in (1 - clip, 1 + clip):
                        amb[t] |= (ratio - bound).abs() <= BRANCH_TOL * bound
        h = h * (end[t] == 0)[:, None]
    if branches:
        return None, None, st, amb
    (loss / norm).backward()
    grads = [p.grad for p in ps]
    mass = [torch.zeros_like(p) for p in ps]
    with torch.no_grad():
        for iw, ib, out, inp in saved:
            f = out.grad.abs() if out.grad is not None else torch.zeros_like(out)
            mass[iw] += f.T @ inp.abs()
            mass[ib] += f.sum(0)
    return grads, mass, st, amb


def reference(mods, act, buf, pred, cols=None, clip=0.2, w_pi=1.0, w_v=0.5, self_ratio=False, chunk=2048,
              dtype=torch.float64):
    """The PPO loss and its gradient in float64 (or dtype), the GRU written out (gi = x W_ih^T + b_ih, gh = h W_hh^T +
    b_hh) so that every packed parameter's factor is a retained gradient.  self_ratio: logp_old := the reference's own
    logp (ratio 1 exactly, as the kernels give for logp_old from rs_policy_act).  Columns run in chunks (the sum is over
    columns), so the autograd memory stays moderate.  -> (gradients, masses per tensor, stats dict like torch_update's)"""
    T, N = buf.T, buf.N
    cols = torch.arange(N, device=DEV) if cols is None else cols.to(DEV).long()
    M = len(cols)
    grads = mass = None
    st = torch.zeros(6, device=DEV, dtype=torch.float64)
    for c0 in range(0, M, chunk):
        g, m, s, _ = _reference_chunk(mods, act, buf, pred, cols[c0:c0 + chunk], T * M, clip, w_pi, w_v, self_ratio, False,
                                      dtype)
        grads = g if grads is None else [a + b for a, b in zip(grads, g)]
        mass = m if mass is None else [a + b for a, b in zip(mass, m)]
        st += s
    n = T * M - st[5]
    stats = dict(loss_pi=st[0] / (T * M), loss_v=st[1] / (T * M), approx_kl=st[2] / n, entropy=st[3] / n, clip_frac=st[4] / n,
                 skipped=st[5])
    return [g.detach().double() for g in grads], [m.double() for m in mass], stats


def mark_branch_rows(mods, act, buf, pred, clip=0.2, self_ratio=False, chunk=2048):
    """Set the action of every ambiguous row of the buffer (module docstring) to 8, so that both sides skip it."""
    T, N = buf.T, buf.N
    for c0 in range(0, N, chunk):
        cols = torch.arange(c0, min(N, c0 + chunk), device=DEV)
        *_, amb = _reference_chunk(mods, act, buf, pred, cols, 1.0, clip, 1.0, 0.5, self_ratio, True)
        buf.act_buf[:, c0:c0 + len(cols)][amb] = 8.0


def entry_ratio(got, want, mass, g32=None):
    """max over entries of |g - g64| / (2^-24 mass); an entry of zero mass must be exactly zero.  g32 (ReLU heads): the
    reference's own float32 gradient.  A ReLU unit whose pre-activation cancels to near 0 has an activation with a large
    relative float32 error that the mass (of |activation|) does not see, so with ReLU heads the bound is looser (C_ENTRY)
    and an entry may also be off by RELU_FLIP_FACTOR times the float32 reference's error (the per-tensor allowance of
    test_gpu_policy_grad.py, per entry).  Measured on a B200 (1000 W), worst over this file: 5.4 with tanh heads, 378 with ReLU
    heads; without the float32 flush every 32 steps the tanh worst is 14.8 (test_long_bptt)."""
    r = 0.0
    for i, (g, w, m) in enumerate(zip(got, want, mass)):
        err = (g - w).abs()
        scale = EPS * m
        if g32 is not None:
            scale = torch.maximum(scale, RELU_FLIP_FACTOR / C_ENTRY[1] * (g32[i] - w).abs())
        bad = (scale == 0) & (err > 0)
        assert not bad.any(), "a gradient entry with zero mass is nonzero"
        r = max(r, (err / scale.clamp(min=1e-300)).max().item())
    return r


def relu_f32(mods, act, buf, pred, cols=None, **kw):
    """the reference in float32 for ReLU heads (the allowance of entry_ratio), None for tanh"""
    return reference(mods, act, buf, pred, cols, dtype=torch.float32, **kw)[0] if act == 1 else None


def fused(pol, mods, buf, pred, cols=None, **kw):
    for p in params_of(mods):
        p.grad = None
    out = pol.loss_and_grad(buf, pred=pred if pol.d_in == 13 else None, columns=cols, **kw)
    return [p.grad.double().clone() for p in params_of(mods)], out


def check_gradient(what, mods, shape, buf, pred, cols=None, stats=True, **kw):
    """the fused gradient and statistics against the float64 reference, per tensor and per entry -> (fused out, ref stats)"""
    pol = rp.FusedGruPolicy(*mods, num_rows=1)
    got, out = fused(pol, mods, buf, pred, cols, **kw)
    ref_kw = {k: kw[k] for k in ("w_pi", "w_v") if k in kw}
    want, mass, st = reference(mods, shape[4], buf, pred, cols, clip=kw.get("clip_ratio", 0.2), **ref_kw)
    g32 = relu_f32(mods, shape[4], buf, pred, cols, clip=kw.get("clip_ratio", 0.2), **ref_kw)
    e64, er = worst(got, want), entry_ratio(got, want, mass, g32)
    bound = REL if g32 is None else max(REL, RELU_FLIP_FACTOR * worst(g32, want))
    print(f"{what}: per tensor {e64:.2e}, per entry {er:.2f} x 2^-24 mass")
    assert e64 <= bound, what
    assert er <= C_ENTRY[shape[4]], what
    assert out["skipped"].item() == st["skipped"].item()
    if stats:
        for k in ("loss_pi", "loss_v", "approx_kl", "entropy"):
            assert abs(out[k].item() - st[k].item()) <= 1e-5 * max(1.0, abs(st[k].item())), (what, k)
        assert abs(out["clip_frac"].item() - st["clip_frac"].item()) <= 1e-12, what
    assert int(pol.grad_ticket.item()) == 0
    return got, out, want, st


# --------------------------------------------------------------------------------------------------------------------
# 1. every instantiation


@pytest.mark.parametrize("kernel,shape", CASES, ids=CASE_IDS)
def test_gradient_at_every_instantiation(kernel, shape, dispatched):
    d, H, P, V, act = shape
    count = param_count(d, H, P, V)
    assert L.load().rs_policy_param_count(C.byref(L.RsPolicyConfig(d, H, P, V, act))) == count
    mods = modules(*shape, seed=count)
    assert sum(p.numel() for p in params_of(mods)) == count
    assert expected_kernels(d, H, P, V)[0] == kernel
    print(f"{shape}: {dispatched[shape]}")
    assert dispatched[shape][0] == "policy_grad_kernel<{}, {}, {}>".format(*kernel)
    M, T = 2 * 16 * sms() + 5, 65                 # every CTA walks >= 2 groups, the last one partial; flushes at 64, 32, 0
    buf, pred = filled_buffer(T, M, seed=count)
    mark_branch_rows(mods, act, buf, pred)
    got, out, want, st = check_gradient(f"{shape} count {count}", mods, shape, buf, pred)
    # the written-out reference is torch_update's loop
    g64, st64 = torch_update(mods, buf, pred)
    assert worst(want, g64) <= 1e-10
    for k in st64:
        assert abs(st[k].item() - st64[k].item()) <= 1e-10 * max(1.0, abs(st64[k].item())), k


@pytest.mark.parametrize("kernel,shape", CASES, ids=CASE_IDS)
def test_act_and_value_at_every_instantiation(kernel, shape, dispatched):
    d, H, P, V, act = shape
    mods = modules(*shape, seed=H + P + V)
    want_kernel = "policy_kernel<{}, {}>".format(*expected_kernels(d, H, P, V)[1])
    assert dispatched[shape][1:] == [want_kernel, want_kernel], dispatched[shape]
    for rows in (1, 257, 400_003):
        seed = 0x5EED0000 + rows
        pol = rp.FusedGruPolicy(*mods, num_rows=rows, seed=seed)
        obs, pred, h0 = inputs(rows, d, H, seed=rows)
        pol.hidden_state.copy_(h0)
        action, value, logp = pol.act(obs, pred)
        h_ref, lp_ref, v_ref = torch_step(mods, obs, pred, h0)
        dh = (pol.hidden_state - h_ref).abs().max().item()
        dv = (value - v_ref).abs().max().item()
        dl = (logp - lp_ref.gather(1, action.long()[:, None])[:, 0]).abs().max().item()
        print(f"{shape} rows={rows}: |d hidden| {dh:.2e}, |d value| {dv:.2e}, |d logp| {dl:.2e}")
        assert dh < ATOL and dv < ATOL and dl < ATOL
        want, clear = gumbel_max(lp_ref, gumbel(seed, np.arange(rows), 0))
        assert clear.mean() >= 0.99
        assert np.array_equal(action.cpu().numpy()[clear], want[clear])
        assert int(pol.ticket.item()) == 0 and int(pol.ctr.item()) == 1
        obs2, pred2, _ = inputs(rows, d, H, seed=rows + 1)
        h1 = pol.hidden_state.clone()
        v2 = pol.value(obs2, pred2)
        assert torch.equal(pol.hidden_state, h1)
        _, _, v2_ref = torch_step(mods, obs2, pred2, h1)
        assert (v2 - v2_ref).abs().max().item() < ATOL


# --------------------------------------------------------------------------------------------------------------------
# 2. the two kernels agree bit for bit


def act_rollout(mods, T, N, end, seed):
    """T steps of rs_policy_act from h = 0 with rs_rollout_post's restart h *= (end == 0) between steps, stored in a
    BatchedPPOBuffer: obs, action, logp, value; ret := value, logp_old := logp, random advantages -> (pol, buf, pred)"""
    d_in = mods[0].input_size
    pol = rp.FusedGruPolicy(*mods, num_rows=N, seed=seed)
    buf = rp.BatchedPPOBuffer(11, T, N, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(seed)
    buf.obs_buf.copy_(torch.randn(T, N, 11, generator=g, device=DEV))
    pred = torch.rand(T, N, 2, generator=g, device=DEV) if d_in == 13 else None
    buf.adv_buf.copy_(torch.randn(T, N, generator=g, device=DEV))
    buf.end_buf.copy_(end)
    for t in range(T):
        a, v, lp = pol.act(buf.obs_buf[t], None if pred is None else pred[t])
        buf.act_buf[t] = a.float()
        buf.logp_buf[t] = lp
        buf.val_buf[t] = v
        buf.ret_buf[t] = v
        pol.hidden_state.mul_((end[t] == 0).float()[:, None])
    return pol, buf, pred


def rollout_ends(T, N, seed):
    """random path ends, plus ends at t = 0, back to back, and at T - 1"""
    g = torch.Generator(device=DEV).manual_seed(seed)
    end = (torch.rand(T, N, generator=g, device=DEV) < 0.05).to(torch.uint8)
    end[0, ::3] = 1
    end[10:14, 1::5] = 2
    end[T - 1] = 1
    return end


def value_head_params(mods):
    return params_of(mods)[4 + len(list(mods[1].parameters())):]


@pytest.mark.parametrize("kernel,shape", CASES, ids=CASE_IDS)
def test_act_and_grad_kernels_agree_exactly(kernel, shape):
    """loss_and_grad recomputes rs_policy_act's logp and value bit for bit: at clip_ratio = 0 (lo = hi = 1) a row whose
    ratio is not exactly 1 counts as clipped, and ret = value gives v - ret = 0 exactly"""
    T, N = 70, 1000
    mods = modules(*shape[:5], seed=7 + shape[1])
    pol, buf, pred = act_rollout(mods, T, N, rollout_ends(T, N, seed=shape[1]), seed=shape[1] + 100)
    mark_branch_rows(mods, shape[4], buf, pred, clip=0.0, self_ratio=True)
    n_pi = len(list(mods[1].parameters()))
    got, out = fused(pol, mods, buf, pred, clip_ratio=0.0)
    assert out["clip_frac"].item() == 0.0
    assert out["approx_kl"].item() == 0.0
    assert out["loss_v"].item() == 0.0
    assert out["skipped"].item() == (buf.act_buf == 8).sum().item()
    assert all(torch.count_nonzero(g).item() == 0 for g in got[4 + n_pi:]), "value-head gradient is not exactly zero"
    want, mass, _ = reference(mods, shape[4], buf, pred, clip=0.0, w_v=0.0, self_ratio=True)
    g32 = relu_f32(mods, shape[4], buf, pred, clip=0.0, w_v=0.0, self_ratio=True)
    e64, er = worst(got, want), entry_ratio(got, want, mass, g32)
    print(f"{shape}: per tensor {e64:.2e}, per entry {er:.2f}")
    assert e64 <= (REL if g32 is None else max(REL, RELU_FLIP_FACTOR * worst(g32, want))) and er <= C_ENTRY[shape[4]]


@pytest.mark.parametrize("mode", ["rows", "graph"])
def test_collector_epoch_has_ratio_one_at_fresh_weights(mode):
    N, T = 2048, 240
    env = rp.RadSearch(obstruction_count=5, enforce_grid_boundaries=True, num_envs=N, seed=17, device=DEV, auto_reset=True,
                       steps_per_episode=120, prefetch=True, use_cuda_graph=mode == "graph", standardize=1)
    buf = rp.BatchedPPOBuffer(11, T, N, device=DEV)
    mods = modules(*BENCH, seed=16)
    kw = dict(obs_in=env.obs.view(N, 11), action_out=env.action_buffer.view(N)) if mode == "graph" else {}
    pol = rp.FusedGruPolicy(*mods, num_rows=N, seed=5, **kw)
    rp.RolloutCollector(env, buf, pol, mode=mode).collect()
    buf.get()
    out = pol.loss_and_grad(buf, clip_ratio=0.0)
    print(f"{mode}: clip_frac {out['clip_frac'].item()!r}, approx_kl {out['approx_kl'].item()!r}")
    assert out["clip_frac"].item() == 0.0 and out["approx_kl"].item() == 0.0


# --------------------------------------------------------------------------------------------------------------------
# 3. group and column edges, 4. time and path-end edges


@pytest.mark.parametrize("shape", [BENCH, WIDE13], ids=["bench", "13-33-17-64-relu"])
def test_group_and_column_edges(shape):
    T = 40
    S = sms()
    mods = modules(*shape, seed=21)
    g = torch.Generator(device=DEV).manual_seed(3)
    for M in (1, 15, 16, 17, 16 * S, 16 * S + 1):
        N = M + 7
        buf, pred = filled_buffer(T, N, seed=M)
        mark_branch_rows(mods, shape[4], buf, pred)
        cols = torch.randperm(N, generator=g, device=DEV)[:M].to(torch.int32)
        check_gradient(f"{shape} M={M}", mods, shape, buf, pred, cols)
    # groups SMs .. 2 SMs - 1 run on the CTAs of groups 0 .. SMs - 1 (one 512-thread CTA per SM): invalid columns at warps
    # that held a valid column in the CTA's first group must contribute nothing
    M = N = 2 * 16 * S
    buf, pred = filled_buffer(T, N, seed=5)
    mark_branch_rows(mods, shape[4], buf, pred)
    cols = torch.arange(M, dtype=torch.int32, device=DEV)
    bad = torch.tensor([-1, N, 2 ** 30], dtype=torch.int32, device=DEV)
    second = torch.arange(S, 2 * S, device=DEV)
    for i, w in enumerate((0, 7, 15)):
        cols[second * 16 + w] = bad[(second + i) % 3]
    _, out, _, _ = check_gradient(f"{shape} stale scratch", mods, shape, buf, pred, cols)
    valid = cols[(cols >= 0) & (cols < N)].long()
    assert out["skipped"].item() == 3 * S * T + (buf.act_buf[:, valid] == 8).sum().item()
    # every column invalid
    cols = bad.repeat(M // 3 + 1)[:M + 1]
    pol = rp.FusedGruPolicy(*mods, num_rows=1)
    got, out = fused(pol, mods, buf, pred, cols)
    assert all(torch.count_nonzero(x).item() == 0 for x in got)
    assert out["skipped"].item() == T * (M + 1)
    assert all(torch.isfinite(v).item() for v in out.values())
    # duplicate columns, in one group and across groups
    base = torch.randperm(N, generator=g, device=DEV)[:700]
    cols = torch.cat([base, base[:300], base.flip(0)[:40]]).to(torch.int32)
    check_gradient(f"{shape} duplicates", mods, shape, buf, pred, cols)


@pytest.mark.parametrize("T", [1, 31, 32, 33, 64, 481])
@pytest.mark.parametrize("shape", [BENCH, WIDE13], ids=["bench", "13-33-17-64-relu"])
def test_time_and_path_end_edges(shape, T):
    M = 16 * sms() + 1
    mods = modules(*shape, seed=T)
    buf, pred = filled_buffer(T, M, seed=T + 1)
    mark_branch_rows(mods, shape[4], buf, pred)
    check_gradient(f"{shape} T={T}", mods, shape, buf, pred)
    if T in (33, 481):
        buf.end_buf.fill_(1)                      # the carry is always 0
        mark_branch_rows(mods, shape[4], buf, pred)
        check_gradient(f"{shape} T={T}, an end at every step", mods, shape, buf, pred)


@pytest.mark.parametrize("shape", [BENCH, WIDE13], ids=["bench", "13-33-17-64-relu"])
def test_long_bptt(shape):
    """no path end in T = 2049 steps: BPTT through the whole column; one group, so one CTA's float32 sums carry it all"""
    T, M = 2049, 16
    mods = modules(*shape, seed=2049)
    buf, pred = filled_buffer(T, M, seed=2049)
    buf.end_buf.zero_()
    mark_branch_rows(mods, shape[4], buf, pred)
    check_gradient(f"{shape} T={T} no ends", mods, shape, buf, pred)


# --------------------------------------------------------------------------------------------------------------------
# 5. cancellation and the bench shape per entry


@pytest.mark.parametrize("shape", [BENCH, WIDE13], ids=["bench", "13-33-17-64-relu"])
def test_cancelling_columns(shape):
    """each column paired with a duplicate whose advantage is negated, ratio exactly 1 (logp_old from rs_policy_act) and
    w_v = 0: the float64 gradient is ~0, so the per-entry mass bound is the whole test"""
    T, K = 97, 16 * sms() + 3
    mods = modules(*shape, seed=31)
    _, half, pred = act_rollout(mods, T, K, rollout_ends(T, K, seed=4), seed=9)
    buf = rp.BatchedPPOBuffer(11, T, 2 * K, device=DEV)
    for name in ("obs_buf", "act_buf", "adv_buf", "ret_buf", "logp_buf", "end_buf"):
        src = getattr(half, name)
        getattr(buf, name).copy_(torch.cat([src, -src if name == "adv_buf" else src], dim=1))
    pred = None if pred is None else torch.cat([pred, pred], dim=1)
    mark_branch_rows(mods, shape[4], buf, pred, clip=0.0, self_ratio=True)
    # pairs side by side in the first half of the columns (one warp sum), in different CTAs' groups in the second
    i = torch.arange(K, device=DEV)
    cols = torch.cat([torch.stack([i[:K // 2], i[:K // 2] + K], 1).reshape(-1), i[K // 2:], i[K // 2:] + K]).to(torch.int32)
    pol = rp.FusedGruPolicy(*mods, num_rows=1)
    got, out = fused(pol, mods, buf, pred, cols, w_v=0.0)
    want, mass, _ = reference(mods, shape[4], buf, pred, cols, w_v=0.0, self_ratio=True)
    er = entry_ratio(got, want, mass, relu_f32(mods, shape[4], buf, pred, cols, w_v=0.0, self_ratio=True))
    scale = max(g.abs().max().item() for g in want) / max(m.max().item() for m in mass)
    print(f"{shape} cancelling: |g64|_inf / mass_inf {scale:.1e}, per entry {er:.2f} x 2^-24 mass")
    assert scale < 1e-12 and er <= C_ENTRY[shape[4]]
    assert out["clip_frac"].item() == 0.0


def test_bench_shape_per_entry_at_full_minibatch():
    T, M = 480, 16384
    mods = modules(*BENCH, seed=480)
    buf, pred = filled_buffer(T, M, seed=480)
    mark_branch_rows(mods, 0, buf, pred)
    check_gradient("bench M=16384 T=480", mods, BENCH, buf, pred)


# --------------------------------------------------------------------------------------------------------------------
# 6. loss-parameter edges


@pytest.mark.parametrize("variant", ["w_pi=0", "w_v=0", "clip=0", "ratio e+-30"])
@pytest.mark.parametrize("shape", [BENCH, WIDE13], ids=["bench", "13-33-17-64-relu"])
def test_loss_parameter_edges(shape, variant):
    T, M = 50, 1500
    mods = modules(*shape, seed=50)
    buf, pred = filled_buffer(T, M, seed=51)
    kw = {"w_pi=0": dict(w_pi=0.0), "w_v=0": dict(w_v=0.0), "clip=0": dict(clip_ratio=0.0), "ratio e+-30": {}}[variant]
    if variant == "ratio e+-30":
        sign = torch.randint(0, 2, (T, M), generator=torch.Generator(device=DEV).manual_seed(2), device=DEV) * 2 - 1
        buf.logp_buf.add_(30.0 * sign)
    mark_branch_rows(mods, shape[4], buf, pred, clip=kw.get("clip_ratio", 0.2))
    got, out, _, _ = check_gradient(f"{shape} {variant}", mods, shape, buf, pred, **kw)
    n_pi = len(list(mods[1].parameters()))
    if variant == "w_pi=0":
        assert all(torch.count_nonzero(g).item() == 0 for g in got[4:4 + n_pi])
    if variant == "w_v=0":
        assert all(torch.count_nonzero(g).item() == 0 for g in got[4 + n_pi:])
    if variant == "clip=0":
        assert out["clip_frac"].item() > 0.99
    if variant == "ratio e+-30":
        assert out["clip_frac"].item() == 1.0


@pytest.mark.parametrize("shape", [BENCH, WIDE13], ids=["bench", "13-33-17-64-relu"])
def test_large_logits(shape):
    """policy-head weights scaled so that the logits span about +-50: log_softmax far from uniform"""
    T, M = 40, 2000
    mods = modules(*shape, seed=60)
    obs, pred1, h0 = inputs(M, shape[0], shape[1], seed=61)
    last = mods[1] if shape[2] == 0 else mods[1][2]
    with torch.no_grad():
        h1 = mods[0](obs if pred1 is None else torch.cat([obs, pred1], 1), h0)
        span = mods[1](h1).abs().max().item()
        last.weight.mul_(50.0 / span)
        last.bias.mul_(50.0 / span)
    pol = rp.FusedGruPolicy(*mods, num_rows=M, seed=3)
    pol.hidden_state.copy_(h0)
    action, _, logp = pol.act(obs, pred1)
    gru, pi, v = (copy.deepcopy(m).double() for m in mods)
    x = (obs if pred1 is None else torch.cat([obs, pred1], 1)).double()
    with torch.no_grad():
        lg = pi(gru(x, h0.double()))
        lp = torch.log_softmax(lg, -1).gather(1, action.long()[:, None])[:, 0]
    scale = lg.abs().max(1).values
    rel = ((logp.double() - lp).abs() / scale).max().item()
    print(f"{shape}: logits up to {scale.max().item():.1f}, |d logp| / max |logit| {rel:.2e}")
    assert scale.max().item() > 40.0 and rel <= 1e-6
    buf, pred = filled_buffer(T, M, seed=62)
    mark_branch_rows(mods, shape[4], buf, pred)
    check_gradient(f"{shape} logits +-50", mods, shape, buf, pred)


# --------------------------------------------------------------------------------------------------------------------
# 7. inference noise edges


def test_noise_at_counter_and_row_id_limits():
    rows, seed = 3000, 0x0123456789ABCDEF
    mods = modules(*BENCH, seed=70)
    obs, _, h0 = inputs(rows, 11, 24, seed=71)
    _, lp_ref, _ = torch_step(mods, obs, None, h0)
    ids = np.arange(2 ** 32 - rows, 2 ** 32, dtype=np.uint64)                  # the last valid row ids
    pol = rp.FusedGruPolicy(*mods, num_rows=rows, seed=seed, row_id_offset=2 ** 32 - rows)
    pol.ctr.fill_(2 ** 32 - 1)                                                   # counter words (0xFFFFFFFF, 0), then (0, 1)
    for ctr in (2 ** 32 - 1, 2 ** 32):
        pol.hidden_state.copy_(h0)
        action = pol.act(obs)[0].cpu().numpy()
        want, clear = gumbel_max(lp_ref, gumbel(seed, ids, ctr))
        assert clear.mean() >= 0.99
        assert np.array_equal(action[clear], want[clear]), hex(ctr)
        assert int(pol.ticket.item()) == 0
    assert int(pol.ctr.item()) == 2 ** 32 + 1


# --------------------------------------------------------------------------------------------------------------------
# the returned statistics are fresh tensors


def test_returned_stats_are_not_overwritten_by_later_calls():
    T, N = 30, 600
    mods = modules(*BENCH, seed=80)
    buf, _ = filled_buffer(T, N, seed=80)
    other, _ = filled_buffer(T, N, seed=81)
    other.act_buf[3, :17] = 8.0                                                  # 17 skipped rows
    pol = rp.FusedGruPolicy(*mods, num_rows=N)
    first = pol.loss_and_grad(buf)
    kept = {k: v.item() for k, v in first.items()}
    second = pol.loss_and_grad(other)
    assert second["skipped"].item() == 17
    assert {k: v.item() for k, v in first.items()} == kept
    # under a CUDA graph every returned entry follows each replay
    eager = []
    for b in (buf, other):
        eager.append({k: v.item() for k, v in pol.loss_and_grad(b).items()})
    work = rp.FusedGruPolicy(*mods, num_rows=N)
    live, _ = filled_buffer(T, N, seed=82)
    s = torch.cuda.Stream(device=DEV)
    s.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(s):
        work.loss_and_grad(live)
    torch.cuda.current_stream(DEV).wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        res = work.loss_and_grad(live)
    for b, want in zip((buf, other), eager):
        for name in ("obs_buf", "act_buf", "adv_buf", "ret_buf", "logp_buf", "end_buf"):
            getattr(live, name).copy_(getattr(b, name))
        graph.replay()
        torch.cuda.synchronize()
        assert {k: v.item() for k, v in res.items()} == want
