"""CPU tests of the fused GRU actor-critic (rs_policy_*, radiation_ppo_b200/policy.py), no GPU needed:
  * every argument error of the three entry points comes back as a negative return code with a message, before any launch;
  * the config struct's size, and rs_policy_param_count against the parameter count of the torch modules;
  * the unsupported modules FusedGruPolicy rejects with ValueError;
  * the kernel's per-row body (rs_policy.cuh), built for the host (tests/emu/policy_emu.cpp), against torch on the CPU in
    float64 and its Gumbel-max sampling against the oracle's Philox."""
import ctypes as C
import copy
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from oracle import c_oracle as co
from radiation_ppo_b200 import _lib as L, build
from radiation_ppo_b200.policy import FusedGruPolicy

HERE = os.path.dirname(os.path.abspath(__file__))
DUMMY = C.c_void_p(256)          # non-NULL, never dereferenced: every call below fails its argument checks first

# (d_in, H, P, V, activation): the bench shape, the reference defaults, the widest, the narrowest, and mixed heads
SHAPES = [(11, 24, 0, 0, 0), (13, 24, 32, 32, 0), (11, 64, 64, 64, 1), (11, 1, 1, 1, 0), (13, 64, 0, 7, 1),
          (11, 13, 5, 0, 0), (13, 33, 17, 64, 1), (11, 16, 0, 16, 0)]


@pytest.fixture(scope="module")
def lib():
    build.build()
    return L.load()


def err(lib):
    return lib.rs_last_error().decode()


def modules(d_in, H, P, V, act, seed=0):
    torch.manual_seed(seed)
    A = (torch.nn.Tanh, torch.nn.ReLU)[act]
    gru = torch.nn.GRUCell(d_in, H)
    pi = torch.nn.Linear(H, 8) if P == 0 else torch.nn.Sequential(torch.nn.Linear(H, P), A(), torch.nn.Linear(P, 8))
    v = torch.nn.Linear(H, 1) if V == 0 else torch.nn.Sequential(torch.nn.Linear(H, V), A(), torch.nn.Linear(V, 1))
    return gru, pi, v


def packed(gru, pi, v):
    ps = [gru.weight_ih, gru.weight_hh, gru.bias_ih, gru.bias_hh] + list(pi.parameters()) + list(v.parameters())
    return torch.cat([p.detach().reshape(-1) for p in ps]).numpy().astype(np.float32)


def test_sizeof_policy_config(lib):
    assert lib.rs_sizeof_policy_config() == C.sizeof(L.RsPolicyConfig) == 20


@pytest.mark.parametrize("shape", SHAPES)
def test_param_count_matches_torch(lib, shape):
    gru, pi, v = modules(*shape)
    n = sum(p.numel() for m in (gru, pi, v) for p in m.parameters())
    assert lib.rs_policy_param_count(C.byref(L.RsPolicyConfig(*shape))) == n


def test_argument_errors(lib):
    good = L.RsPolicyConfig(11, 24, 0, 0, 0)
    assert lib.rs_policy_param_count(None) < 0 and "unsupported config" in err(lib)
    for bad in [(12, 24, 0, 0, 0), (11, 0, 0, 0, 0), (11, 65, 0, 0, 0), (11, 24, -1, 0, 0), (11, 24, 65, 0, 0),
                (11, 24, 0, -1, 0), (11, 24, 0, 65, 0), (11, 24, 0, 0, 2), (11, 24, 0, 0, -1)]:
        cfg = L.RsPolicyConfig(*bad)
        assert lib.rs_policy_param_count(C.byref(cfg)) < 0 and "unsupported config" in err(lib), bad
        assert lib.rs_policy_act(C.byref(cfg), *([DUMMY] * 7), 4, 0, 0, DUMMY, DUMMY, None) < 0
        assert "rs_policy_act: unsupported config" in err(lib), bad
        assert lib.rs_policy_value(C.byref(cfg), DUMMY, DUMMY, None, DUMMY, DUMMY, 4, None) < 0
        assert "rs_policy_value: unsupported config" in err(lib), bad

    d = DUMMY
    names = ("params", "obs", "pred", "hidden", "action", "value", "logp", "rows", "row_id0", "seed", "ctr", "ticket")

    def act(cfg=good, **kw):
        a = dict.fromkeys(names, d)
        a.update(pred=None, rows=4, row_id0=0, seed=0)
        a.update(kw)
        rc = lib.rs_policy_act(None if cfg is None else C.byref(cfg), *[a[n] for n in names], None)
        return rc, err(lib) if rc < 0 else ""

    def value(cfg=good, **kw):
        a = dict(params=d, obs=d, pred=None, hidden=d, value=d, rows=4)
        a.update(kw)
        rc = lib.rs_policy_value(None if cfg is None else C.byref(cfg), a["params"], a["obs"], a["pred"], a["hidden"],
                                 a["value"], a["rows"], None)
        return rc, err(lib) if rc < 0 else ""

    for fn in (act, value):
        name = "rs_policy_act" if fn is act else "rs_policy_value"
        assert fn(cfg=None) == (-1, f"{name}: cfg is NULL")
        for k in ("params", "obs", "hidden"):
            assert fn(**{k: None}) == (-1, f"{name}: NULL buffer"), k
        assert fn(cfg=L.RsPolicyConfig(13, 24, 32, 32, 0)) == (-1, f"{name}: d_in = 13 needs pred")
        assert fn(pred=d) == (-1, f"{name}: pred given with d_in = 11")
        for rows in (0, -5):
            assert fn(rows=rows) == (-1, f"{name}: rows must be positive")
        assert fn(value=None) == (-1, f"{name}: NULL output")
    for k in ("action", "logp"):
        assert act(**{k: None}) == (-1, "rs_policy_act: NULL output"), k
    for k in ("ctr", "ticket"):
        assert act(**{k: None}) == (-1, "rs_policy_act: NULL ctr / ticket"), k
    assert act(row_id0=2 ** 32 - 3, rows=4) == (-1, "rs_policy_act: row_id0 + rows exceeds 2^32")
    assert act(row_id0=2 ** 32 - 1, rows=2) == (-1, "rs_policy_act: row_id0 + rows exceeds 2^32")


def test_unsupported_modules_are_rejected():
    H = 24
    lin = lambda i, o: torch.nn.Linear(i, o)          # noqa: E731
    seq = lambda *m: torch.nn.Sequential(*m)          # noqa: E731
    gru, pi, v = torch.nn.GRUCell(11, H), lin(H, 8), lin(H, 1)
    cases = [
        ((torch.nn.GRUCell(12, H), pi, v), "input size 12"),
        ((torch.nn.GRUCell(11, 65), lin(65, 8), lin(65, 1)), "hidden size 65"),
        ((torch.nn.GRUCell(11, H, bias=False), pi, v), "without bias"),
        ((torch.nn.GRU(11, H), pi, v), "GRU"),
        ((torch.nn.LSTMCell(11, H), pi, v), "LSTMCell"),
        ((gru, lin(H, 4), v), "Linear(24, 4)"),
        ((gru, pi, lin(H, 2)), "Linear(24, 2)"),
        ((gru, torch.nn.Linear(H, 8, bias=False), v), "without bias"),
        ((gru, seq(lin(H, 32), torch.nn.Tanh(), lin(32, 32), torch.nn.Tanh(), lin(32, 8)), v), "Sequential of 5"),
        ((gru, seq(lin(H, 32), torch.nn.Sigmoid(), lin(32, 8)), v), "Sigmoid"),
        ((gru, seq(lin(H, 65), torch.nn.Tanh(), lin(65, 8)), v), "hidden width 65"),
        ((gru, seq(lin(H, 32), torch.nn.Tanh(), lin(32, 8)), seq(lin(H, 32), torch.nn.ReLU(), lin(32, 1))), "different activations"),
        ((gru, seq(torch.nn.Conv1d(H, 32, 1), torch.nn.Tanh(), lin(32, 8)), v), "Conv1d"),
        ((gru, pi, seq(lin(H, 32), torch.nn.Tanh(), lin(16, 1))), "Linear(16, 1) where Linear(32, 1)"),
        ((gru, pi, copy.deepcopy(v).double()), "float32"),
        ((torch.nn.GRUCell(11, H).half(), pi, v), "float32"),
        ((gru, torch.nn.Identity(), v), "Identity"),
    ]
    for mods, msg in cases:
        with pytest.raises(ValueError, match=re.escape(msg)):
            FusedGruPolicy(*mods, num_rows=4, device="cuda:0")
    with pytest.raises(ValueError, match="num_rows"):
        FusedGruPolicy(gru, pi, v, num_rows=0, device="cuda:0")
    with pytest.raises(ValueError, match="num_rows"):
        FusedGruPolicy(gru, pi, v, num_rows=8, row_id_offset=2 ** 32 - 4, device="cuda:0")
    with pytest.raises(ValueError, match="CUDA device"):
        FusedGruPolicy(gru, pi, v, num_rows=4, device="cpu")


# ---- the per-row body on the host -------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("policy_emu") / "libpolicy_emu.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-I" + os.path.join(HERE, "emu"),
                    "-o", out, os.path.join(HERE, "emu", "policy_emu.cpp")], check=True)
    e = C.CDLL(out)
    vp = C.c_void_p
    e.emu_policy_rows.restype = C.c_int
    e.emu_policy_rows.argtypes = [C.POINTER(L.RsPolicyConfig), vp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_uint32, C.c_uint64,
                                  C.c_uint64, C.c_int]
    e.emu_policy_layout.restype = C.c_int
    e.emu_policy_layout.argtypes = [C.POINTER(L.RsPolicyConfig), vp]
    return e


def _vp(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def emu_call(e, shape, params, obs, pred, hidden, act, row_id0=0, seed=0, ctr=0):
    n = obs.shape[0]
    h = hidden.copy()
    action, value, logp = np.full(n, -1, np.int32), np.full(n, np.nan, np.float32), np.full(n, np.nan, np.float32)
    rc = e.emu_policy_rows(C.byref(L.RsPolicyConfig(*shape)), _vp(params), _vp(obs), _vp(pred), _vp(h), _vp(action),
                           _vp(value), _vp(logp), n, row_id0, seed, ctr, int(act))
    assert rc == 0
    return h, action, value, logp


def torch_reference(mods, obs, pred, hidden):
    """float64 torch on the CPU: h', log_softmax of the policy head, value of h'"""
    gru, pi, v = (m.double() for m in (mods[0].__class__(mods[0].input_size, mods[0].hidden_size), mods[1], mods[2]))
    gru.load_state_dict({k: t.double() for k, t in mods[0].state_dict().items()})
    x = torch.as_tensor(obs, dtype=torch.float64)
    if pred is not None:
        x = torch.cat([x, torch.as_tensor(pred, dtype=torch.float64)], dim=1)
    with torch.no_grad():
        h1 = gru(x, torch.as_tensor(hidden, dtype=torch.float64))
        lp = torch.log_softmax(pi(h1), dim=-1)
        val = v(h1)[:, 0]
    return h1.numpy(), lp.numpy(), val.numpy()


def gumbel_reference(seed, row_ids, ctr):
    """g[m][k] in float64 from the oracle's Philox4x32-10 with the counters of rs_policy_act"""
    g = np.empty((len(row_ids), 8))
    key = [seed & 0xFFFFFFFF, seed >> 32]
    for i, r in enumerate(row_ids):
        words = co.philox([r, 4 << 24, ctr & 0xFFFFFFFF, ctr >> 32], key) + \
            co.philox([r, (4 << 24) | 1, ctr & 0xFFFFFFFF, ctr >> 32], key)
        u = ((np.array(words, np.uint64) >> np.uint64(8)).astype(np.float64) + 0.5) * 2.0 ** -24
        g[i] = -np.log(-np.log(u))
    return g


def random_inputs(rng, n, d_in, H):
    obs = rng.normal(size=(n, 11)).astype(np.float32)
    obs[:, 0] *= 3.0
    pred = rng.uniform(0, 1, size=(n, 2)).astype(np.float32) if d_in == 13 else None
    hidden = rng.uniform(-1, 1, size=(n, H)).astype(np.float32)
    return obs, pred, hidden


def test_staging_fills_every_slot_once(emu):
    for shape in SHAPES:
        cfg = L.RsPolicyConfig(*shape)
        count = L.load().rs_policy_param_count(C.byref(cfg))
        dst = np.zeros(count, np.int32)
        total = emu.emu_policy_layout(C.byref(cfg), _vp(dst))
        assert total >= count and total % 4 == 0
        assert dst.min() >= 0 and dst.max() < total and len(np.unique(dst)) == count, shape


@pytest.mark.parametrize("shape", SHAPES)
def test_row_body_matches_torch(emu, shape):
    mods = modules(*shape, seed=sum(shape))
    params = packed(*mods)
    rng = np.random.default_rng(sum(shape))
    n = 200
    obs, pred, hidden = random_inputs(rng, n, shape[0], shape[1])
    seed, ctr, row0 = 0x1234_5678_9ABC_DEF0 + shape[1], 7 + shape[2], 1000 * shape[1]
    h1, action, value, logp = emu_call(emu, shape, params, obs, pred, hidden, True, row0, seed, ctr)
    h_ref, lp_ref, v_ref = torch_reference(mods, obs, pred, hidden)
    assert np.abs(h1 - h_ref).max() < 1e-5
    assert np.abs(value - v_ref).max() < 1e-5
    assert np.abs(logp - lp_ref[np.arange(n), action]).max() < 1e-5
    # Gumbel-max under the oracle's uniforms, float64 scores, rows with a clear winner
    sc = lp_ref + gumbel_reference(seed, range(row0, row0 + n), ctr)
    top = np.sort(sc, axis=1)
    clear = top[:, -1] - top[:, -2] >= 1e-4
    assert clear.mean() >= 0.99
    assert np.array_equal(action[clear], sc.argmax(axis=1)[clear])
    # the value pass: the same value from the same (obs, h), hidden untouched
    h2, _, v2, _ = emu_call(emu, shape, params, obs, pred, hidden, False)
    assert np.array_equal(h2, hidden) and np.array_equal(v2, value)


def test_gumbel_noise_near_u_one(emu):
    """Philox words with x >> 8 close to 2^24 (u close to 1) give large finite Gumbel noise, not inf: with one logit far
    above the others, only such a word can take the action elsewhere.  Checked statistically: the argmax of 8 Gumbels
    over uniform logits is uniform."""
    shape = (11, 1, 0, 0, 0)
    mods = modules(*shape)
    with torch.no_grad():
        for p in mods[1].parameters():
            p.zero_()
    params = packed(*mods)
    n = 40000
    obs, _, hidden = random_inputs(np.random.default_rng(3), n, 11, 1)
    _, action, _, logp = emu_call(emu, shape, params, obs, None, hidden, True, 0, 99, 0)
    assert np.allclose(logp, -np.log(8.0), atol=1e-6)
    counts = np.bincount(action, minlength=8)
    assert counts.min() > 0.95 * n / 8 and counts.max() < 1.05 * n / 8
