"""CPU tests of the fused PFGRU localiser (rs_pfgru_*, radiation_ppo_b200/pfgru.py), no GPU needed:
  * every argument error of the entry points comes back as a negative return code with a message, before any launch;
  * the config struct's size, and rs_pfgru_param_count against the parameter count of the torch modules;
  * the unsupported modules and settings FusedPFGRU rejects with ValueError;
  * the kernel's per-row body (rs_pfgru.cuh), built for the host (tests/emu/pfgru_emu.cpp), against the float64
    restatement of tests/pfgru_ref.py with the same Philox noise: predict, peek and restart;
  * the Box-Muller rule against N(0, 1) (Kolmogorov-Smirnov) and the resampling index rule against q (chi-square)."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from radiation_ppo_b200 import _lib as L, build
from radiation_ppo_b200.pfgru import FusedPFGRU
from tests import pfgru_ref as ref

HERE = os.path.dirname(os.path.abspath(__file__))
DUMMY = C.c_void_p(256)          # non-NULL, never dereferenced: every call below fails its argument checks first

# (d_in, H, K, W, resample, alpha): the reference shape first; together they cover every (DXP, HMAX) instantiation
SHAPES = [(3, 24, 40, 24, 1, 0.7), (3, 1, 1, 1, 1, 0.7), (11, 64, 64, 64, 1, 0.05), (3, 24, 32, 1, 1, 1.0),
          (11, 24, 33, 64, 1, 0.7), (3, 64, 40, 24, 0, 0.7), (1, 17, 40, 8, 1, 0.3), (7, 33, 5, 3, 1, 1.0),
          (11, 1, 64, 64, 0, 0.05)]


@pytest.fixture(scope="module")
def lib():
    build.build()
    return L.load()


def err(lib):
    return lib.rs_last_error().decode()


def cfg_of(shape):
    return L.RsPfgruConfig(*shape)


def test_sizeof_pfgru_config(lib):
    assert lib.rs_sizeof_pfgru_config() == C.sizeof(L.RsPfgruConfig) == 24


@pytest.mark.parametrize("shape", SHAPES)
def test_param_count_matches_torch(lib, shape):
    d, H, K, W = shape[:4]
    n = sum(p.numel() for m in ref.modules(d, H, W) for p in m.parameters())
    assert lib.rs_pfgru_param_count(C.byref(cfg_of(shape))) == n


def test_argument_errors(lib):
    good = (3, 24, 40, 24, 1, 0.7)
    assert lib.rs_pfgru_param_count(None) < 0 and "unsupported config" in err(lib)
    bads = [(0, 24, 40, 24, 1, 0.7), (12, 24, 40, 24, 1, 0.7), (3, 0, 40, 24, 1, 0.7), (3, 65, 40, 24, 1, 0.7),
            (3, 24, 0, 24, 1, 0.7), (3, 24, 65, 24, 1, 0.7), (3, 24, 40, 0, 1, 0.7), (3, 24, 40, 65, 1, 0.7),
            (3, 24, 40, 24, -1, 0.7), (3, 24, 40, 24, 2, 0.7), (3, 24, 40, 24, 1, 0.0), (3, 24, 40, 24, 1, -0.5),
            (3, 24, 40, 24, 1, 1.0001), (3, 24, 40, 24, 1, float("nan"))]
    d = DUMMY
    for bad in bads:
        cfg = cfg_of(bad)
        assert lib.rs_pfgru_param_count(C.byref(cfg)) < 0 and "unsupported config" in err(lib), bad
        assert lib.rs_pfgru_predict(C.byref(cfg), d, d, d, d, d, 4, 0, 0, d, d, None) < 0
        assert "rs_pfgru_predict: unsupported config" in err(lib), bad
        assert lib.rs_pfgru_peek(C.byref(cfg), d, d, d, d, d, None, 0, 4, 0, 0, d, None) < 0
        assert "rs_pfgru_peek: unsupported config" in err(lib), bad
        assert lib.rs_pfgru_restart(C.byref(cfg), d, d, None, 0, 4, 0, 0, d, None) < 0
        assert "rs_pfgru_restart: unsupported config" in err(lib), bad

    def predict(cfg=good, **kw):
        a = dict(params=d, obs=d, particles=d, logw=d, pred=d, rows=4, row_id0=0, seed=0, ctr=d, ticket=d)
        a.update(kw)
        rc = lib.rs_pfgru_predict(None if cfg is None else C.byref(cfg_of(cfg)), *a.values(), None)
        return rc, err(lib) if rc < 0 else ""

    def peek(cfg=good, **kw):
        a = dict(params=d, obs=d, particles=d, logw=d, pred=d, mask=None, bits=0, rows=4, row_id0=0, seed=0, ctr=d)
        a.update(kw)
        rc = lib.rs_pfgru_peek(None if cfg is None else C.byref(cfg_of(cfg)), *a.values(), None)
        return rc, err(lib) if rc < 0 else ""

    def restart(cfg=good, **kw):
        a = dict(particles=d, logw=d, mask=None, bits=0, rows=4, row_id0=0, seed=0, ctr=d)
        a.update(kw)
        rc = lib.rs_pfgru_restart(None if cfg is None else C.byref(cfg_of(cfg)), *a.values(), None)
        return rc, err(lib) if rc < 0 else ""

    for fn, name in ((predict, "rs_pfgru_predict"), (peek, "rs_pfgru_peek"), (restart, "rs_pfgru_restart")):
        assert fn(cfg=None) == (-1, f"{name}: cfg is NULL")
        for k in ("particles", "logw"):
            assert fn(**{k: None}) == (-1, f"{name}: NULL state"), k
        assert fn(ctr=None) == (-1, f"{name}: NULL ctr")
        for rows in (0, -5):
            assert fn(rows=rows) == (-1, f"{name}: rows must be positive")
        assert fn(row_id0=2 ** 32 - 3, rows=4) == (-1, f"{name}: row_id0 + rows exceeds 2^32")
        assert fn(row_id0=2 ** 32 - 1, rows=2) == (-1, f"{name}: row_id0 + rows exceeds 2^32")
    for fn, name in ((predict, "rs_pfgru_predict"), (peek, "rs_pfgru_peek")):
        for k in ("params", "obs", "pred"):
            assert fn(**{k: None}) == (-1, f"{name}: NULL buffer"), k
    assert predict(ticket=None) == (-1, "rs_pfgru_predict: NULL ticket")


def test_unsupported_modules_are_rejected():
    H, d, W = 24, 3, 24
    lin = torch.nn.Linear
    seq = torch.nn.Sequential
    fz, fr, fn, fo, ho = ref.modules(d, H, W)
    good = dict(fc_z=fz, fc_r=fr, fc_n=fn, fc_obs=fo, hid_obs=ho)
    cases = [
        (dict(fc_z=torch.nn.GRUCell(d, H)), "fc_z: unsupported layer GRUCell"),
        (dict(fc_z=lin(H + 12, H)), "input size 12"),
        (dict(fc_z=lin(H, H)), "input size 0"),
        (dict(fc_z=lin(65 + d, 65)), "hidden size 65"),
        (dict(fc_z=lin(H + d, H, bias=False)), "fc_z: Linear without bias"),
        (dict(fc_r=lin(H + d + 1, H)), "fc_r: Linear(28, 24) where Linear(27, 24)"),
        (dict(fc_n=lin(H + d, H)), "fc_n: Linear(27, 24) where Linear(27, 48)"),
        (dict(fc_obs=lin(H + d, 2)), "fc_obs: Linear(27, 2) where Linear(27, 1)"),
        (dict(fc_r=seq(lin(H + d, H))), "fc_r: unsupported layer Sequential"),
        (dict(hid_obs=lin(H, 2)), "hid_obs: unsupported module Linear"),
        (dict(hid_obs=seq(lin(H, W), torch.nn.ReLU())), "Sequential of 2"),
        (dict(hid_obs=seq(lin(H, W), torch.nn.ReLU(), lin(W, 2), torch.nn.ReLU())), "Sequential of 4"),
        (dict(hid_obs=seq(lin(H, W), torch.nn.Tanh(), lin(W, 2))), "activation Tanh"),
        (dict(hid_obs=seq(lin(H, 65), torch.nn.ReLU(), lin(65, 2))), "hidden width 65"),
        (dict(hid_obs=seq(lin(H, W), torch.nn.ReLU(), lin(W, 3))), "Linear(24, 3) where Linear(24, 2)"),
        (dict(hid_obs=seq(lin(H + 1, W), torch.nn.ReLU(), lin(W, 2))), "Linear(25, 24) where Linear(24, 24)"),
        (dict(hid_obs=seq(torch.nn.Conv1d(H, W, 1), torch.nn.ReLU(), lin(W, 2))), "unsupported layer Conv1d"),
        (dict(fc_obs=lin(H + d, 1).double()), "float32"),
        (dict(activation="relu"), "activation 'relu' is unsupported"),
        (dict(num_particles=0), "num_particles 0"),
        (dict(num_particles=65), "num_particles 65"),
        (dict(resamp_alpha=0.0), "resamp_alpha 0.0"),
        (dict(resamp_alpha=1.5), "resamp_alpha 1.5"),
        (dict(num_rows=0), "num_rows"),
        (dict(num_rows=8, row_id_offset=2 ** 32 - 4), "num_rows"),
        (dict(device="cpu"), "CUDA device"),
    ]
    for change, msg in cases:
        kw = dict(good, num_rows=4, device="cuda:0")
        kw.update(change)
        with pytest.raises(ValueError, match=re.escape(msg)):
            FusedPFGRU(**kw)


# ---- the per-row body on the host -------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("pfgru_emu") / "libpfgru_emu.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-I" + os.path.join(HERE, "emu"),
                    "-o", out, os.path.join(HERE, "emu", "pfgru_emu.cpp")], check=True)
    e = C.CDLL(out)
    vp = C.c_void_p
    e.emu_pfgru_rows.restype = C.c_int
    e.emu_pfgru_rows.argtypes = [C.POINTER(L.RsPfgruConfig), vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_uint32,
                                 C.c_uint64, C.c_uint64, C.c_int]
    e.emu_pfgru_layout.restype = C.c_int
    e.emu_pfgru_layout.argtypes = [C.POINTER(L.RsPfgruConfig), vp]
    e.emu_pfgru_normals.restype = None
    e.emu_pfgru_normals.argtypes = [C.c_uint32, C.c_uint32, C.c_int, C.c_uint64, C.c_uint64, vp]
    e.emu_pfgru_pick.restype = None
    e.emu_pfgru_pick.argtypes = [vp, C.c_int, vp, C.c_int, vp]
    return e


def _vp(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def emu_call(e, shape, params, obs, part, logw, mode, row_id0=0, seed=0, ctr=0, mask=None, mask_bits=0):
    """-> (particles, log_weights, pred) after one call; pred NaN where nothing was written"""
    n = part.shape[0]
    part, logw = part.copy(), logw.copy()
    pred = np.full((n, 2), np.nan, np.float32)
    rc = e.emu_pfgru_rows(C.byref(cfg_of(shape)), _vp(params), _vp(obs), _vp(part), _vp(logw), _vp(pred), _vp(mask),
                          mask_bits, n, row_id0, seed, ctr, mode)
    assert rc == 0
    return part, logw, pred


def random_state(rng, n, K, H):
    obs = rng.normal(size=(n, 11)).astype(np.float32)
    obs[:, :3] = rng.uniform(0, 1, size=(n, 3))
    part = rng.uniform(0, 1, size=(n, K, H)).astype(np.float32)
    s = rng.normal(size=(n, K)) * 2
    logw = (s - np.log(np.exp(s).sum(axis=1, keepdims=True))).astype(np.float32)
    return obs, part, logw


def test_staging_fills_every_slot_once(lib, emu):
    for shape in SHAPES:
        cfg = cfg_of(shape)
        count = lib.rs_pfgru_param_count(C.byref(cfg))
        dst = np.zeros(count, np.int32)
        total = emu.emu_pfgru_layout(C.byref(cfg), _vp(dst))
        assert total >= count and total % 4 == 0
        assert dst.min() >= 0 and dst.max() < total and len(np.unique(dst)) == count, shape


def check_against_reference(shape, mods, got, obs, part, logw, rows, seed, ctr, blk0):
    d, H, K, W, rs_, alpha = shape
    want = ref.step(mods, torch.as_tensor(obs), torch.as_tensor(part), torch.as_tensor(logw), rows, seed, ctr, K, alpha,
                    bool(rs_), blk0)
    near = want["near"].any(dim=1).numpy()
    ok = ~near
    e_h = ref.close(got[0][ok], want["h"].numpy()[ok])
    e_p = ref.close(got[1][ok], want["p"].numpy()[ok])
    e_y = ref.close(got[2][ok], want["pred"].numpy()[ok])
    return e_h, e_p, e_y, int(want["near"].sum()), ok.mean()


@pytest.mark.parametrize("shape", SHAPES, ids=[str(s) for s in SHAPES])
def test_row_body_matches_float64(emu, shape):
    d, H, K, W, rs_, alpha = shape
    mods = ref.modules(d, H, W, seed=H + K)
    params = ref.packed(mods).numpy()
    rng = np.random.default_rng(K * 100 + H)
    n = 48 if K * H > 2000 else 96
    obs, part, logw = random_state(rng, n, K, H)
    seed, ctr, row0 = 0x0123_4567_89AB_CDEF + K, (1 << 32) - 1 + H, 5000 * K
    rows = torch.arange(row0, row0 + n)
    # predict: one step, state written
    got = emu_call(emu, shape, params, obs, part, logw, 0, row0, seed, ctr)
    e_h, e_p, e_y, n_near, frac = check_against_reference(shape, mods, got, obs, part, logw, rows, seed, ctr, 0)
    print(f"{shape}: predict max err/bar h {e_h:.3f} p {e_p:.3f} pred {e_y:.3f}; {n_near} draws near a boundary")
    assert max(e_h, e_p, e_y) <= 1.0 and frac >= 0.9
    # a second, teacher-forced step from the body's own state
    obs2 = random_state(rng, n, K, H)[0]
    got2 = emu_call(emu, shape, params, obs2, got[0], got[1], 0, row0, seed, ctr + 1)
    assert max(check_against_reference(shape, mods, got2, obs2, got[0], got[1], rows, seed, ctr + 1, 0)[:3]) <= 1.0
    # peek: the peek blocks, the state untouched, only the selected rows written
    mask = (np.arange(n) % 3 == 1).astype(np.uint8) * 4
    pk = emu_call(emu, shape, params, obs, part, logw, 1, row0, seed, ctr, mask, 4)
    assert np.array_equal(pk[0], part) and np.array_equal(pk[1], logw)
    sel = mask != 0
    assert np.isnan(pk[2][~sel]).all() and not np.isnan(pk[2][sel]).any()
    want = ref.step(mods, torch.as_tensor(obs), torch.as_tensor(part), torch.as_tensor(logw), rows, seed, ctr, K, alpha,
                    bool(rs_), ref.PEEK_BLOCK)
    ok = sel & ~want["near"].any(dim=1).numpy()
    assert ref.close(pk[2][ok], want["pred"].numpy()[ok]) <= 1.0
    if W > 4:                                                        # (a one-unit ReLU head may be dead in both)
        assert not np.array_equal(pk[2][sel], got[2][sel])        # peek draws its own noise
    # restart of the selected rows: U[0, 1) from the restart blocks, -log K
    rp_, rl, _ = emu_call(emu, shape, None, None, part, logw, 2, row0, seed, ctr, mask, 0)
    h_want, p_want = ref.restart_state(rows, K, H, seed, ctr)
    assert np.array_equal(rp_[sel], h_want.float().numpy()[sel]) and np.array_equal(rp_[~sel], part[~sel])
    assert np.allclose(rl[sel], p_want.numpy()[sel], rtol=0, atol=1e-6) and np.array_equal(rl[~sel], logw[~sel])
    assert rp_[sel].min() > 0.0 and rp_[sel].max() < 1.0


def test_restart_then_predict_matches_float64(emu):
    """the rollout's pattern: restart every row, then predict from that state"""
    shape = SHAPES[0]
    d, H, K, W, rs_, alpha = shape
    mods = ref.modules(d, H, W, seed=3)
    params = ref.packed(mods).numpy()
    n, seed = 64, 77
    obs, part, logw = random_state(np.random.default_rng(4), n, K, H)
    part, logw, _ = emu_call(emu, shape, None, None, part, logw, 2, 0, seed, 0)
    got = emu_call(emu, shape, params, obs, part, logw, 0, 0, seed, 0)
    e = check_against_reference(shape, mods, got, obs, part, logw, torch.arange(n), seed, 0, 0)
    assert max(e[:3]) <= 1.0


def test_box_muller_is_standard_normal(emu):
    from scipy import stats

    n_blocks = 1 << 15
    out = np.zeros(4 * n_blocks, np.float32)
    emu.emu_pfgru_normals(12345, 0, n_blocks, 3, 99, _vp(out))
    # the same words through the float64 rule: float32 accuracy everywhere, also where u is within 2^-24 of 1 (the
    # largest |ln u| error would come from rounding u to float32 there)
    u = ref.uniform(ref.words(torch.tensor([12345]), torch.arange(n_blocks), 99, 3))[0].numpy()
    r0, r1 = np.sqrt(-2 * np.log(u[:, 0])), np.sqrt(-2 * np.log(u[:, 2]))
    want = np.stack([r0 * np.cos(2 * np.pi * u[:, 1]), r0 * np.sin(2 * np.pi * u[:, 1]), r1 * np.cos(2 * np.pi * u[:, 3]),
                     r1 * np.sin(2 * np.pi * u[:, 3])], axis=1).reshape(-1)
    err = np.abs(out - want) / (1e-7 + 1e-6 * np.abs(want))
    print(f"Box-Muller: worst |float32 - float64| / (1e-7 + 1e-6 |eps|) = {err.max():.3f}")
    assert err.max() <= 1.0
    for i in range(4):                                                  # each word position on its own, then all
        assert stats.kstest(out[i::4], "norm").pvalue > 1e-3, i
    res = stats.kstest(out, "norm")
    print(f"KS D = {res.statistic:.2e}, p = {res.pvalue:.3f} over {out.size} draws")
    assert res.pvalue > 1e-3
    assert abs(np.corrcoef(out[0::4], out[1::4])[0, 1]) < 0.01        # the cos / sin pair is uncorrelated


def test_resampling_index_rule_follows_q(emu):
    from scipy import stats

    rng = np.random.default_rng(8)
    for K, alpha in ((40, 0.7), (33, 0.05), (64, 1.0), (1, 0.7)):
        p1 = rng.normal(size=K) * 2
        p1 = p1 - np.log(np.exp(p1).sum())
        q = (alpha * np.exp(p1) + (1 - alpha) / K).astype(np.float32)
        n = 400_000
        u = ((rng.integers(0, 2 ** 24, n) + 0.5) * 2.0 ** -24).astype(np.float32)
        idx = np.zeros(n, np.int32)
        emu.emu_pfgru_pick(_vp(q), K, _vp(u), n, _vp(idx))
        assert idx.min() >= 0 and idx.max() < K
        counts = np.bincount(idx, minlength=K)
        if K == 1:
            assert counts[0] == n
            continue
        chi2, pval = stats.chisquare(counts, n * q.astype(np.float64) / q.astype(np.float64).sum())
        print(f"K {K} alpha {alpha}: chi-square {chi2:.1f} ({K - 1} dof), p = {pval:.3f}")
        assert pval > 1e-3
        # the rule itself: the first i with u C_{K-1} < C_i
        C = np.cumsum(q, dtype=np.float32)
        t = u[:2000] * C[-1]
        assert np.array_equal(idx[:2000], np.minimum(np.searchsorted(C, t, side="right"), K - 1))
