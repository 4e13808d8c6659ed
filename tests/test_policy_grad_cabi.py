"""CPU tests of the fused PPO loss and gradient (rs_policy_ppo_grad, FusedGruPolicy.loss_and_grad), no GPU needed:
  * every argument error of rs_policy_ppo_grad and rs_policy_grad_workspace_bytes comes back as a negative return code with
    a message, before any launch; the workspace size against its formula;
  * the kernel's per-step math (rs_policy_grad.cuh), built for the host (tests/emu/policy_grad_emu.cpp) and run over whole
    columns, against float64 torch autograd of the same loss: eight shapes, path ends at t = 0, mid-column and at T-1,
    T = 1, ratios inside, outside, exactly at 1 +- eps and exactly 1, out-of-range columns and actions."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from radiation_ppo_b200 import _lib as L, build
from tests.test_policy_cabi import SHAPES, modules, packed

HERE = os.path.dirname(os.path.abspath(__file__))
DUMMY = C.c_void_p(256)          # non-NULL, never dereferenced: every call below fails its argument checks first


@pytest.fixture(scope="module")
def lib():
    build.build()
    return L.load()


def err(lib):
    return lib.rs_last_error().decode()


def test_argument_errors(lib):
    good = L.RsPolicyConfig(11, 24, 0, 0, 0)
    names = ("params", "obs", "pred", "act", "adv", "ret", "logp", "end", "columns", "T", "N", "M", "clip", "w_pi", "w_v",
             "grad", "stats", "workspace", "ticket")

    def call(cfg=good, **kw):
        a = dict.fromkeys(names, DUMMY)
        a.update(pred=None, columns=None, T=8, N=4, M=4, clip=0.2, w_pi=1.0, w_v=0.5)
        a.update(kw)
        rc = lib.rs_policy_ppo_grad(None if cfg is None else C.byref(cfg), *[a[n] for n in names], None)
        return rc, err(lib) if rc < 0 else ""

    f = "rs_policy_ppo_grad: "
    assert call(cfg=None) == (-1, f + "cfg is NULL")
    for bad in [(12, 24, 0, 0, 0), (11, 0, 0, 0, 0), (11, 65, 0, 0, 0), (11, 24, 65, 0, 0), (11, 24, 0, -1, 0), (11, 24, 0, 0, 2)]:
        rc, msg = call(cfg=L.RsPolicyConfig(*bad))
        assert rc == -1 and msg.startswith(f + "unsupported config"), bad
    for k in ("params", "obs", "act", "adv", "ret", "logp", "end"):
        assert call(**{k: None}) == (-1, f + "NULL buffer"), k
    assert call(cfg=L.RsPolicyConfig(13, 24, 32, 32, 0)) == (-1, f + "d_in = 13 needs pred")
    assert call(pred=DUMMY) == (-1, f + "pred given with d_in = 11")
    for k in ("T", "N", "M"):
        for v in (0, -3):
            assert call(**{k: v}) == (-1, f + "T, N and M must be positive"), (k, v)
    assert call(M=3) == (-1, f + "M must equal N without columns")
    for clip in (-0.1, 1.0, float("nan")):
        assert call(clip=clip) == (-1, f + "clip_ratio must be in [0, 1)"), clip
    for k in ("w_pi", "w_v"):
        assert call(**{k: float("inf")}) == (-1, f + "w_pi and w_v must be finite"), k
    for k in ("grad", "stats", "workspace", "ticket"):
        assert call(**{k: None}) == (-1, f + "NULL output / workspace / ticket"), k

    ws = lib.rs_policy_grad_workspace_bytes
    assert ws(None, 4, 4) == -1 and "unsupported config" in err(lib)
    assert ws(C.byref(L.RsPolicyConfig(11, 24, 0, 0, 3)), 4, 4) == -1 and "unsupported config" in err(lib)
    for T, M in ((0, 4), (4, 0), (-1, 4)):
        assert ws(C.byref(good), T, M) == -1 and err(lib) == "rs_policy_grad_workspace_bytes: T and M must be positive"


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("T,M", [(1, 1), (480, 16), (37, 65536), (480, 65536)])
def test_workspace_bytes(lib, shape, T, M):
    """stats partials (8 doubles) and float64 gradient partials (count rounded to 4) per 16-column group, then the hidden
    state of every step [T][M][H]"""
    cfg = L.RsPolicyConfig(*shape)
    count = lib.rs_policy_param_count(C.byref(cfg))
    groups = (M + 15) // 16
    want = groups * 64 + groups * 32 * ((count + 3) // 4) + 4 * T * M * shape[1]
    assert lib.rs_policy_grad_workspace_bytes(C.byref(cfg), T, M) == want


# ---- the per-step math on the host -------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("policy_grad_emu") / "libpolicy_grad_emu.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-I" + os.path.join(HERE, "emu"),
                    "-o", out, os.path.join(HERE, "emu", "policy_grad_emu.cpp")], check=True)
    e = C.CDLL(out)
    vp = C.c_void_p
    e.emu_policy_grad.restype = C.c_int
    e.emu_policy_grad.argtypes = [C.POINTER(L.RsPolicyConfig)] + [vp] * 9 + [C.c_int] * 3 + [C.c_double] * 3 + [vp] * 4
    e.emu_grad_entries.restype = C.c_int
    e.emu_grad_entries.argtypes = [C.POINTER(L.RsPolicyConfig), vp]
    return e


def _vp(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def rollout(rng, T, N, d_in, end_every=None):
    """random [T][N] buffer rows; path ends at t = 0, at T-1 and every few steps in between"""
    obs = rng.normal(size=(T, N, 11)).astype(np.float32)
    pred = rng.uniform(0, 1, size=(T, N, 2)).astype(np.float32) if d_in == 13 else None
    act = rng.integers(0, 8, size=(T, N)).astype(np.float32)
    adv = rng.normal(size=(T, N)).astype(np.float32)
    ret = rng.normal(size=(T, N)).astype(np.float32)
    logp = (np.log(1 / 8) + 0.3 * rng.normal(size=(T, N))).astype(np.float32)
    end = (rng.uniform(size=(T, N)) < (1.0 / end_every if end_every else 0.15)).astype(np.uint8)
    end[0, ::3] = 1
    end[T - 1, ::2] = 1
    return dict(obs=obs, pred=pred, act=act, adv=adv, ret=ret, logp=logp, end=end)


def emu_grad(e, shape, params, r, columns=None, clip=0.2, w_pi=1.0, w_v=0.5):
    T, N = r["act"].shape
    M = N if columns is None else len(columns)
    count = len(params)
    grad, stats = np.zeros(count), np.zeros(6)
    lp, ratio = np.full((T, M), np.nan, np.float32), np.full((T, M), np.nan, np.float32)
    cols = None if columns is None else np.ascontiguousarray(columns, np.int32)
    rc = e.emu_policy_grad(C.byref(L.RsPolicyConfig(*shape)), _vp(params), _vp(r["obs"]), _vp(r["pred"]), _vp(r["act"]),
                           _vp(r["adv"]), _vp(r["ret"]), _vp(r["logp"]), _vp(r["end"]), _vp(cols), T, N, M, clip, w_pi, w_v,
                           _vp(grad), _vp(stats), _vp(lp), _vp(ratio))
    assert rc == 0
    return grad, stats, lp, ratio


def torch_grad(mods, r, columns=None, clip=0.2, w_pi=1.0, w_v=0.5, ratio32=None, dtype=torch.float64):
    """the loss of bench.py::ppo_update in torch autograd (restart after a path end, h = 0 at t = 0) over the gathered
    columns; rows with an out-of-range column or action are left out.  ratio32 [T][M]: a float32 ratio per row that the
    reference takes as its value (ratio - (ratio - ratio32).detach(): exact, and the gradient still flows), so that
    ties and clip boundaries are decided on the same number as the kernel's.  -> (flat gradient, stats)"""
    gru0, pi0, v0 = mods
    gru = torch.nn.GRUCell(gru0.input_size, gru0.hidden_size).to(dtype)
    gru.load_state_dict({k: t.to(dtype) for k, t in gru0.state_dict().items()})
    import copy
    pi, v = copy.deepcopy(pi0).to(dtype), copy.deepcopy(v0).to(dtype)
    T, N = r["act"].shape
    cols = np.arange(N) if columns is None else np.asarray(columns)
    M = len(cols)
    okc = torch.as_tensor((cols >= 0) & (cols < N))
    c = np.clip(cols, 0, N - 1)
    g = lambda k: torch.as_tensor(r[k][:, c])                                         # noqa: E731
    x = g("obs").to(dtype)
    if r["pred"] is not None:
        x = torch.cat([x, g("pred").to(dtype)], dim=2)
    act, adv, ret, logp_old, end = g("act"), g("adv").to(dtype), g("ret").to(dtype), g("logp").to(dtype), g("end")
    lo, hi = float(np.float32(1 - clip)), float(np.float32(1 + clip))
    h = torch.zeros(M, gru.hidden_size, dtype=dtype)
    loss = 0.0
    st = np.zeros(6)
    for t in range(T):
        h = gru(x[t], h)
        lsm = torch.log_softmax(pi(h), dim=-1)
        ok = okc & (act[t] > -1) & (act[t] < 8)
        a = torch.where(ok, act[t], torch.zeros_like(act[t])).long()
        lp = lsm.gather(1, a[:, None]).squeeze(1)
        ratio = torch.exp(lp - logp_old[t])
        if ratio32 is not None:
            r32 = torch.as_tensor(np.nan_to_num(ratio32[t], nan=1.0), dtype=dtype)
            ratio = ratio - (ratio - r32).detach()
        surr = torch.minimum(ratio * adv[t], torch.clamp(ratio, lo, hi) * adv[t])
        val = v(h).squeeze(1)
        zero = torch.zeros((), dtype=dtype)
        loss = loss - w_pi * torch.where(ok, surr, zero).sum() + w_v * torch.where(ok, (val - ret[t]) ** 2, zero).sum()
        with torch.no_grad():
            okn = ok.numpy()
            st[0] -= surr[ok].sum().item()
            st[1] += ((val - ret[t]) ** 2)[ok].sum().item()
            st[2] += (logp_old[t] - lp)[ok].sum().item()
            st[3] -= (lsm.exp() * lsm).sum(1)[ok].sum().item()
            st[4] += ((ratio < lo) | (ratio > hi))[ok].sum().item()
            st[5] += (~okn).sum()
        h = h * (end[t] == 0)[:, None]
    loss = loss / (T * M)
    params = [gru.weight_ih, gru.weight_hh, gru.bias_ih, gru.bias_hh] + list(pi.parameters()) + list(v.parameters())
    grads = torch.autograd.grad(loss, params, allow_unused=True)
    flat = torch.cat([(torch.zeros_like(p) if gr is None else gr).reshape(-1) for p, gr in zip(params, grads)])
    return flat.detach().double().numpy(), st


def split(shape, flat):
    """per parameter tensor, in packing order"""
    mods = modules(*shape)
    ps = [mods[0].weight_ih, mods[0].weight_hh, mods[0].bias_ih, mods[0].bias_hh] + list(mods[1].parameters()) + \
        list(mods[2].parameters())
    out, off = [], 0
    for p in ps:
        out.append(flat[off:off + p.numel()])
        off += p.numel()
    return out


def assert_grad_close(shape, got, want, rel=1e-5):
    for i, (a, b) in enumerate(zip(split(shape, got), split(shape, want))):
        scale = max(np.abs(b).max(), 1e-30)
        assert np.abs(a - b).max() <= rel * scale + 1e-12, (shape, i, np.abs(a - b).max(), scale)


def test_parameters_map_to_distinct_products(emu, lib):
    for shape in SHAPES:
        cfg = L.RsPolicyConfig(*shape)
        count = lib.rs_policy_param_count(C.byref(cfg))
        ent = np.zeros(count, np.uint32)
        cw = emu.emu_grad_entries(C.byref(cfg), _vp(ent))
        # only bias_ih and bias_hh of the r and z gates share their product (both are da_r / da_z times 1)
        H, d = shape[1], shape[0]
        b_ih = 3 * H * d + 3 * H * H
        assert np.array_equal(ent[b_ih:b_ih + 2 * H], ent[b_ih + 3 * H:b_ih + 5 * H])
        assert len(np.unique(ent)) == count - 2 * H, shape
        assert (ent >> 16).max() < cw and (ent & 0xFFFF).max() < cw


@pytest.mark.parametrize("shape", SHAPES)
def test_columns_match_torch_autograd(emu, shape):
    mods = modules(*shape, seed=7 + sum(shape))
    params = packed(*mods)
    rng = np.random.default_rng(sum(shape))
    T, N = 23, 6
    r = rollout(rng, T, N, shape[0], end_every=5)
    cols = np.array([5, 0, 3, 3, -1, 6, 2, 1000], np.int32)      # repeats, and two columns out of range
    r["act"][4, 2] = 8.0
    r["act"][9, 5] = -1.0
    r["act"][11, 0] = np.nan
    r["act"][T - 1, 3] = 7.9                                      # truncated to 7, like torch's .long()
    for w_pi, w_v in ((1.0, 0.5), (1.0, 0.0), (0.0, 2.0)):
        grad, stats, _, ratio = emu_grad(emu, shape, params, r, cols, w_pi=w_pi, w_v=w_v)
        want, st_ref = torch_grad(mods, r, cols, w_pi=w_pi, w_v=w_v)
        assert_grad_close(shape, grad, want)
        # 3 columns out of range (-1, 6, 1000) x T rows, and one bad action in each of the gathered columns 2, 5, 0
        assert stats[5] == st_ref[5] == 3 * T + 3
        assert np.isnan(ratio[:, [4, 5, 7]]).all() and np.isnan(ratio[4, 6]) and not np.isnan(ratio[T - 1, 2])
        np.testing.assert_allclose(stats[:5], st_ref[:5], rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("shape", SHAPES[:4])
def test_single_step_and_no_ends(emu, shape):
    mods = modules(*shape, seed=3)
    params = packed(*mods)
    rng = np.random.default_rng(5)
    for T, clean in ((1, False), (40, True)):
        r = rollout(rng, T, 5, shape[0])
        if clean:
            r["end"][:] = 0
        grad, stats, _, _ = emu_grad(emu, shape, params, r)
        want, st_ref = torch_grad(mods, r)
        assert_grad_close(shape, grad, want)
        np.testing.assert_allclose(stats, st_ref, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("shape", [SHAPES[0], SHAPES[1], SHAPES[2]])
def test_ratio_exactly_one_and_at_the_clip_bounds(emu, shape):
    """logp_old = the kernel's own logp gives ratio exactly 1; a clip_ratio of ratio - 1 (1 - ratio) puts a row exactly on
    1 + eps (1 - eps).  Both signs of the advantage; the reference decides on the same float32 ratios."""
    mods = modules(*shape, seed=11)
    params = packed(*mods)
    rng = np.random.default_rng(17)
    T, N = 12, 8
    r = rollout(rng, T, N, shape[0], end_every=4)
    _, _, lp, _ = emu_grad(emu, shape, params, r)
    r["logp"][:, :4] = lp[:, :4]                                  # columns 0..3: ratio exactly 1
    r["adv"][::2, :] = -np.abs(r["adv"][::2, :])
    r["adv"][1::2, :] = np.abs(r["adv"][1::2, :])
    _, _, _, ratio = emu_grad(emu, shape, params, r)
    assert (ratio[:, :4] == 1.0).all()
    above = ratio[:, 4:][(ratio[:, 4:] > 1.01) & (ratio[:, 4:] < 1.9)]
    below = ratio[:, 4:][(ratio[:, 4:] < 0.99) & (ratio[:, 4:] > 0.1)]
    assert len(above) and len(below)
    for clip in (0.2, float(above[0]) - 1.0, 1.0 - float(below[0])):
        grad, stats, _, ratio = emu_grad(emu, shape, params, r, clip=clip)
        lo, hi = np.float32(1 - clip), np.float32(1 + clip)
        if clip != 0.2:
            assert ((ratio == lo) | (ratio == hi)).sum() >= 1
        want, st_ref = torch_grad(mods, r, clip=clip, ratio32=ratio)
        assert_grad_close(shape, grad, want)
        assert stats[4] == st_ref[4]
