"""GPU edge tests (pytest -m gpu) of the kernels whose outputs the PPO update consumes: every rs_gae variant and every
route of its auto-dispatch, the warp-scan's error bound, rs_adv_stats / rs_adv_normalize, rs_pack_rollout and
rs_episode_table.  The GAE kernels run on adversarial rollouts (every path-end byte code, ends at t = 0, at 8-step chunk
borders and back to back, NaN bootstrap values wherever none may be read, mixed magnitudes) into NaN-filled outputs with
sentinel words on both sides, so a skipped row, a stray read or a stray write cannot pass."""
import ctypes as C
import itertools
import math
import re

import numpy as np
import pytest
import torch

from oracle import c_oracle as co

pytestmark = pytest.mark.gpu

import radiation_ppo_b200 as rp  # noqa: E402
from radiation_ppo_b200 import _lib as L  # noqa: E402

PE_CODES = np.array([1, 2, 4, 5, 6, 255], np.uint8)     # non-zero path-end bytes (the step kernel's `ended` codes among them)
PAD = 32                                                  # sentinel floats on each side of an output (keeps 128-byte alignment)
SENTINEL = -1234.5678
SCAN_BYTES_PER_STEP = 8 * (3 * 4 + 1)                     # the scan stages [T][8] rew / val / boot floats and path-end bytes

COLS16, COLS8 = "gae_cols_kernel<16, 1>", "gae_cols_kernel<8, 7>"
TILE128, TILE64 = "gae_tile_kernel<128, 8, 3, 7>", "gae_tile_kernel<64, 8, 3, 14>"
WS128_3, WS128, WS64, WS224 = ("gae_tile_ws_kernel<128, 8, 3, 5>", "gae_tile_ws_kernel<128, 8, 6, 4>",
                               "gae_tile_ws_kernel<64, 8, 6, 7>", "gae_tile_ws_kernel<224, 8, 6, 2>")
TMAP128, TMAP224 = "gae_tmap_kernel<128, 8, 6, 4>", "gae_tmap_kernel<224, 8, 6, 2>"
SCAN = "gae_scan_kernel"
VARIANT_KERNEL = {1: COLS16, 3: COLS8, 4: COLS16, 7: TILE128, 8: WS128_3, 10: TILE64, 11: WS128, 12: WS64, 13: WS224,
                  14: TMAP128, 15: TMAP224}                # explicit variants at N <= 4096 (variant 1: no tile route below 16384)
EXPLICIT_T = [1, 2, 7, 8, 9, 24, 25, 48, 49, 97, 480, 481]  # partial chunks of 8 and ring wraps of 3 and 6 stages
EXPLICIT_N = [128, 256, 1152, 4096]                         # 128 and 1152: partial 224-column CTAs


def dev():
    return torch.device("cuda:0")


# ---- references -----------------------------------------------------------------------------------------------------
def gae_float64(rew, val, pe, boot, gamma=0.99, lam=0.90):
    """The recurrence of P:391-423 in float64, vectorised over columns, without the final rounding to float32."""
    T, N = rew.shape
    gl = gamma * lam
    adv, ret = np.empty((T, N)), np.empty((T, N))
    nv, na, nr = np.zeros(N), np.zeros(N), np.zeros(N)
    for t in range(T - 1, -1, -1):
        e = np.ones(N, bool) if t == T - 1 else pe[t] != 0
        b = np.where(e, boot[t], 0.0)
        nv, na, nr = np.where(e, b, nv), np.where(e, 0.0, na), np.where(e, b, nr)
        r, v = rew[t].astype(np.float64), val[t].astype(np.float64)
        a = (r + gamma * nv) - v + gl * na
        g = r + gamma * nr
        adv[t], ret[t] = a, g
        nv, na, nr = v, a, g
    return adv, ret


def assert_within_f32_ulp(got, ref64, what):
    """|got - ref64| <= spacing(float32(ref64)) + 1e-12 everywhere (NaN fails)."""
    err = np.abs(got.astype(np.float64) - ref64)
    tol = np.abs(np.spacing(ref64.astype(np.float32))).astype(np.float64) + 1e-12
    bad = ~(err <= tol)
    if bad.any():
        i = np.unravel_index(np.argmax(bad), bad.shape)
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} outside one float32 ulp, first at {i}: "
                             f"{got[i]!r} vs {ref64[i]!r} (tolerance {tol[i]:.3g})")


def fsum(x):
    """Correctly rounded float64 sum of a large array, streamed in chunks."""
    x = np.asarray(x, np.float64).ravel()
    return math.fsum(itertools.chain.from_iterable(c.tolist() for c in np.array_split(x, max(1, x.size >> 20))))


def two_pass_reference(x):
    x = np.asarray(x, np.float64)
    mean = fsum(x) / x.size
    return mean, math.sqrt(fsum((x - mean) ** 2) / x.size)


def episode_table_numpy(pe, offset):
    """(count[N], start[E], len[E]) of the trajectories of every column (an end where pe != 0 and at t = T-1), written
    from slot offset[n]."""
    T, N = pe.shape
    ends = pe != 0
    ends[T - 1] = True
    count = ends.sum(0).astype(np.int32)
    start = np.zeros(int(count.sum()), np.int32)
    length = np.zeros(int(count.sum()), np.int32)
    for n in range(N):
        ts = np.nonzero(ends[:, n])[0]
        first = np.concatenate([[0], ts[:-1] + 1])
        start[offset[n]:offset[n] + len(ts)] = n * T + first
        length[offset[n]:offset[n] + len(ts)] = ts + 1 - first
    return count, start, length


# ---- inputs and outputs -----------------------------------------------------------------------------------------------
def adversarial_pe(rng, T, N):
    """Path-end bytes drawn from {0, 1, 2, 4, 5, 6, 255}.  Every column plays one of five patterns: no interior end,
    sparse ends, ends at chunk borders (t % 8 in {0, 7}), a run of length-1 episodes, or an end at t = 0 plus dense ends.
    The byte of row T-1 is random: the kernels end every column there whatever it says."""
    t = np.arange(T)[:, None]
    kind = rng.integers(0, 5, N)
    u = rng.random((T, N), dtype=np.float32)
    run0, runlen = rng.integers(0, T, N), rng.integers(1, 40, N)
    end = ((kind == 1) & (u < 1 / 20)) | ((kind == 2) & ((t % 8 == 0) | (t % 8 == 7)) & (u < 0.7))
    end |= (kind == 3) & (((t >= run0) & (t < run0 + runlen)) | (u < 1 / 30))
    end |= (kind == 4) & ((t == 0) | (u < 1 / 8))
    end[T - 1] = rng.random(N) < 0.5
    return np.where(end, PE_CODES[rng.integers(0, len(PE_CODES), (T, N), dtype=np.int8)], np.uint8(0))


def adversarial_rollout(T, N, seed):
    rng = np.random.default_rng(seed)
    pe = adversarial_pe(rng, T, N)
    mags = np.array([1e-3, 1e-3, 1, 1, 1, 1, 1, 1, 1, 30], np.float32)
    rew = (rng.random((T, N), dtype=np.float32) * 1.6 - 1.5) * mags[rng.integers(0, 10, (T, N), dtype=np.int8)]
    rew[rng.random((T, N), dtype=np.float32) < 0.03] = 0.0
    val = rng.standard_normal((T, N), dtype=np.float32) * (mags * 0.3)[rng.integers(0, 10, (T, N), dtype=np.int8)]
    read = pe != 0
    read[T - 1] = True
    boot = np.where(read, rng.standard_normal((T, N), dtype=np.float32) * 3, np.float32(np.nan)).astype(np.float32)
    boot[read & (rng.random((T, N), dtype=np.float32) < 0.3)] = 0.0
    return rew, val, pe, boot


def to_dev(arrays, misaligned=False):
    """Device copies; with `misaligned`, rew is a contiguous view 4 bytes past an allocation."""
    d = dev()
    rew, val, pe, boot = (torch.as_tensor(np.ascontiguousarray(x), device=d) for x in arrays)
    if misaligned:
        r = torch.empty(rew.numel() + 1, device=d)[1:].view(rew.shape)
        r.copy_(rew)
        assert r.data_ptr() % 16 == 4
        rew = r
    return rew, val, pe, boot


def poisoned(shape):
    """(buffer, view): a NaN-filled [shape] view with PAD sentinel words before and after it."""
    n = math.prod(shape)
    buf = torch.full((n + 2 * PAD,), float("nan"), device=dev())
    buf[:PAD] = SENTINEL
    buf[-PAD:] = SENTINEL
    return buf, buf[PAD:PAD + n].view(shape)


def assert_sentinels(buf, what):
    assert bool((buf[:PAD] == SENTINEL).all()) and bool((buf[-PAD:] == SENTINEL).all()), f"{what}: sentinel overwritten"


def assert_bits(got, want, what):
    """Bit-identical float32 tensors (NaN in `got` fails)."""
    bad = got.view(torch.int32) != want.view(torch.int32)
    if bool(bad.any()):
        i = tuple(bad.nonzero()[0].tolist())
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} differ, first at {i}: "
                             f"{got[i].item()!r} vs {want[i].item()!r}")


KERNEL_NAME = re.compile(r"(gae_\w+?_kernel(?:<[^>]*>)?)")


def launched_gae_kernels(fn):
    """Names of the GAE kernels `fn` launched, from the CUDA activity of torch.profiler (demangled, e.g.
    'gae_tile_ws_kernel<224, 8, 6, 2>')."""
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [m.group(1) for m in (KERNEL_NAME.search(e.name) for e in prof.events()) if m]


def run_gae(inp, variant, gamma=0.99, lam=0.90, capture=False):
    """rs_gae into poisoned adv / ret with fp64 stats; checks the sentinels.  Returns (adv, ret, stats, kernels)."""
    rew, val, pe, boot = inp
    abuf, adv = poisoned(tuple(rew.shape))
    rbuf, ret = poisoned(tuple(rew.shape))
    stats = torch.zeros(2, dtype=torch.float64, device=dev())

    def call():
        rp.gae_advantages(rew, val, pe, boot, gamma, lam, adv=adv, ret=ret, stats=stats, variant=variant)

    kernels = None
    if capture:
        kernels = launched_gae_kernels(call)
    else:
        call()
    torch.cuda.synchronize()
    assert_sentinels(abuf, f"adv (variant {variant})")
    assert_sentinels(rbuf, f"ret (variant {variant})")
    return adv, ret, stats, kernels


def assert_stats(stats, adv, what):
    """stats = {sum, sum of squares} of the kernel's own float32 advantages, to 1e-12 of the sum of magnitudes."""
    a = adv.double()
    s = stats.cpu().numpy()
    for k, (want, scale) in enumerate(((a.sum().item(), a.abs().sum().item()), ((a * a).sum().item(), (a * a).sum().item()))):
        assert abs(s[k] - want) <= 1e-12 * scale, f"{what}: stats[{k}] = {s[k]!r}, want {want!r}"


_cache = {}


def case(T, N, seed=0):
    """Cached adversarial inputs on the device and the bit-exact float32 reference (co.gae) of one shape."""
    key = (T, N, seed)
    if key not in _cache:
        arrays = adversarial_rollout(T, N, seed=1000 * T + N + seed)
        a0, r0 = co.gae(*arrays)
        _cache[key] = (arrays, to_dev(arrays), torch.as_tensor(a0, device=dev()), torch.as_tensor(r0, device=dev()))
    return _cache[key]


# ---- 1. every explicit variant, bit for bit ---------------------------------------------------------------------------
@pytest.mark.parametrize("T", EXPLICIT_T)
@pytest.mark.parametrize("variant", sorted(VARIANT_KERNEL))
def test_gae_explicit_variant_is_bit_exact_on_adversarial_rollouts(variant, T):
    for N in EXPLICIT_N:
        _, inp, a0, r0 = case(T, N)
        capture = (T, N) == (480, 4096)
        adv, ret, stats, kernels = run_gae(inp, variant, capture=capture)
        what = f"variant {variant}, T={T}, N={N}"
        if capture:
            assert kernels == [VARIANT_KERNEL[variant]], (what, kernels)
        assert_bits(adv, a0, what + " adv")
        assert_bits(ret, r0, what + " ret")
        assert_stats(stats, adv, what)


# ---- 2. the auto-dispatch table -----------------------------------------------------------------------------------------
DISPATCH = [  # (T, N, rew misaligned, kernel under variant=0, kernel under variant=1)
    (480, 16383, False, SCAN, COLS16),          # scan: 49 920 B of shared memory (opt-in)
    (480, 16384, False, TMAP128, TMAP128),
    (480, 16385, False, COLS16, COLS16),
    (480, 32640, False, TMAP128, TMAP128),
    (480, 32768, False, WS224, WS224),
    (480, 75648, False, WS224, WS224),
    (480, 75776, False, TILE128, TILE128),
    (480, 75777, False, COLS8, COLS8),
    (480, 75776, True, COLS16, COLS16),
    (480, 65536, True, COLS16, COLS16),
    (1969, 1000, False, SCAN, COLS16),          # 204 776 B: the last T the auto route sends to the scan
    (1970, 1000, False, COLS16, COLS16),
]
DISPATCH_N_MAX = 75777


def dispatch_inputs(T, N):
    """T = 480 cases are column slices of one [480, 75777] rollout (columns are independent, so the reference slices too)."""
    if T != 480:
        arrays, _, a0, r0 = case(T, N)
        return arrays, a0, r0
    key = ("dispatch", T)
    if key not in _cache:
        arrays = adversarial_rollout(T, DISPATCH_N_MAX, seed=77)
        a0, r0 = co.gae(*arrays)
        _cache[key] = (arrays, torch.as_tensor(a0, device=dev()), torch.as_tensor(r0, device=dev()))
    arrays, a0, r0 = _cache[key]
    return [x[:, :N] for x in arrays], a0[:, :N], r0[:, :N]


@pytest.mark.parametrize("T,N,misaligned,auto_kernel,v1_kernel", DISPATCH,
                         ids=[f"T{t}-N{n}{'-misaligned' if m else ''}" for t, n, m, _, _ in DISPATCH])
def test_gae_dispatch_routes(T, N, misaligned, auto_kernel, v1_kernel):
    arrays, a0, r0 = dispatch_inputs(T, N)
    inp = to_dev(arrays, misaligned=misaligned)
    for variant, want in ((0, auto_kernel), (1, v1_kernel)):
        adv, ret, stats, kernels = run_gae(inp, variant, capture=True)
        what = f"variant {variant}, T={T}, N={N}{', misaligned' if misaligned else ''}"
        assert kernels == [want], (what, kernels)
        if want == SCAN:
            a64, r64 = gae_float64(*arrays)
            assert_within_f32_ulp(adv.cpu().numpy(), a64, what + " adv")
            assert_within_f32_ulp(ret.cpu().numpy(), r64, what + " ret")
        else:
            assert_bits(adv, a0, what + " adv")
            assert_bits(ret, r0, what + " ret")
        assert_stats(stats, adv, what)
        del adv, ret


# ---- 3. non-default discounting -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("gamma,lam", [(0.99, 0.95), (1.0, 1.0), (0.0, 0.5), (0.5, 0.0), (0.999, 0.97)])
def test_gae_discounting_parameters_are_bit_exact(gamma, lam):
    for T, N in ((97, 1152), (481, 4096)):
        arrays, inp, _, _ = case(T, N)
        a0, r0 = (torch.as_tensor(x, device=dev()) for x in co.gae(*arrays, gamma=gamma, lam=lam))
        for variant in (7, 3, 14):              # one tile, one register-pipelined and one tensor-map kernel
            adv, ret, stats, _ = run_gae(inp, variant, gamma=gamma, lam=lam)
            what = f"gamma={gamma}, lam={lam}, variant {variant}, T={T}, N={N}"
            assert_bits(adv, a0, what + " adv")
            assert_bits(ret, r0, what + " ret")
            assert_stats(stats, adv, what)


# ---- 4. the warp-scan's bound -------------------------------------------------------------------------------------------
def scan_t_max():
    return torch.cuda.get_device_properties(dev()).shared_memory_per_block_optin // SCAN_BYTES_PER_STEP


def scan_shapes():
    shapes = [(T, N) for T in EXPLICIT_T for N in EXPLICIT_N]
    shapes += [(T, N) for T, N, _, _, _ in DISPATCH if N < 16384]
    return shapes + [("max", 1001)]


@pytest.mark.parametrize("T,N", scan_shapes(), ids=[f"T{t}-N{n}" for t, n in scan_shapes()])
def test_gae_warp_scan_within_one_float32_ulp(T, N):
    """The scan (variant 2) re-associates the recurrence as fp64 affine maps: every output must stay within one float32
    ulp of the float64 recurrence, up to T = shared_memory_per_block_optin / 104 (the dynamic shared-memory opt-in)."""
    if T == "max":
        T = scan_t_max()
    arrays = dispatch_inputs(T, N)[0] if (T, N) == (480, 16383) else case(T, N)[0]
    adv, ret, stats, _ = run_gae(to_dev(arrays), 2)
    a64, r64 = gae_float64(*arrays)
    what = f"scan, T={T}, N={N}"
    assert_within_f32_ulp(adv.cpu().numpy(), a64, what + " adv")
    assert_within_f32_ulp(ret.cpu().numpy(), r64, what + " ret")
    assert_stats(stats, adv, what)


def test_gae_warp_scan_refuses_t_past_the_shared_memory_limit():
    T = scan_t_max() + 1
    inp = to_dev(adversarial_rollout(T, 8, seed=3))
    with pytest.raises(ValueError, match="T too large for the scan variant"):
        rp.gae_advantages(*inp, variant=2)


# ---- 5. advantage statistics and normalisation ------------------------------------------------------------------------
STATS_N = [1, 2, 3, 4, 5, 7, 1023, 1_212_416, 1_212_420, 31_457_283]   # 1 212 416 = 1184 blocks x 256 threads x 4


def stats_and_normalize(n, offset, x_host, std_rtol):
    """advantage_statistics against a math.fsum two-pass reference, then rs_adv_normalize bit for bit against numpy
    float32, on a view `offset` floats past a 16-byte boundary with sentinel words around it."""
    d = dev()
    buf = torch.full((4 + offset + n + 4,), SENTINEL, device=d)
    x = buf[4 + offset:4 + offset + n]
    x.copy_(torch.as_tensor(x_host, device=d))
    assert x.data_ptr() % 16 == 4 * offset
    mean, std = rp.advantage_statistics(x)
    m_ref, s_ref = two_pass_reference(x_host)
    what = f"n={n}, offset={offset}"
    assert math.isclose(mean.item(), m_ref, rel_tol=1e-12, abs_tol=0.0), (what, mean.item(), m_ref)
    assert math.isclose(std.item(), s_ref, rel_tol=std_rtol, abs_tol=0.0), (what, std.item(), s_ref)
    m32, s32 = mean.float(), std.float()
    rp.normalize_advantages_(x, m32.double(), s32.double())
    with np.errstate(invalid="ignore", divide="ignore"):
        want = (x_host - np.float32(m32.item())) / np.float32(s32.item())
    got = buf.cpu().numpy()
    assert (got[:4 + offset] == SENTINEL).all() and (got[4 + offset + n:] == SENTINEL).all(), what + ": sentinel overwritten"
    got = got[4 + offset:4 + offset + n]
    nan = np.isnan(want)
    np.testing.assert_array_equal(np.isnan(got), nan, err_msg=what)
    np.testing.assert_array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32), err_msg=what)


@pytest.mark.parametrize("offset", [0, 1, 2, 3])
@pytest.mark.parametrize("n", STATS_N)
def test_advantage_statistics_and_normalisation(n, offset):
    g = torch.Generator(device=dev()).manual_seed(n + offset)
    x = (torch.randn(n, generator=g, device=dev()) * 3 + 0.7).cpu().numpy()
    stats_and_normalize(n, offset, x, std_rtol=1e-12)


@pytest.mark.parametrize("offset", [0, 3])
@pytest.mark.parametrize("n", [5, 1023, 1_212_420, 31_457_283])
def test_advantage_statistics_centre_before_squaring(n, offset):
    """1000 + N(0, 1e-2) in float32: sum(x^2) / n - mean^2 would lose about 10 of the 16 digits of the variance; the
    two-pass form (centre on the mean, then square) keeps the std to 1e-9."""
    g = torch.Generator(device=dev()).manual_seed(7 * n + offset)
    x = (1000 + 1e-2 * torch.randn(n, generator=g, device=dev(), dtype=torch.float64)).float().cpu().numpy()
    stats_and_normalize(n, offset, x, std_rtol=1e-9)


# ---- 6. packing and the episode table ----------------------------------------------------------------------------------
def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream(dev()).cuda_stream)


@pytest.mark.parametrize("D", [1, 11, 18, 19, 40, 64])       # 16 x 32 x (D + 6) floats: above 48 KB from D = 19
def test_pack_rollout_is_a_concat_and_transpose(D):
    lib, d = L.load(), dev()
    rng = np.random.default_rng(D)
    for T, N in itertools.product([1, 31, 32, 33, 97], [1, 15, 16, 17, 50]):
        obs = rng.standard_normal((T, N, D), dtype=np.float32)
        cols = [rng.standard_normal((T, N), dtype=np.float32) for _ in range(4)]    # adv, ret, logp, act
        src = rng.standard_normal((T, N, 2), dtype=np.float32)
        for with_src in (True, False):
            dt = [torch.as_tensor(x, device=d) for x in (obs, *cols)]
            st = torch.as_tensor(src, device=d) if with_src else None
            W = D + 6
            buf = torch.full((N * T * W + PAD,), float("nan"), device=d)
            buf[-PAD:] = SENTINEL
            L.check(lib.rs_pack_rollout(*[_p(x) for x in dt], _p(st), _p(buf), T, N, D, _stream()), "rs_pack_rollout")
            got = buf.cpu().numpy()
            what = f"D={D}, T={T}, N={N}, src={with_src}"
            assert (got[-PAD:] == SENTINEL).all(), what + ": sentinel overwritten"
            tail = src if with_src else np.zeros((T, N, 2), np.float32)
            want = np.concatenate([obs, *[c[:, :, None] for c in cols], tail], axis=2).transpose(1, 0, 2).reshape(N * T, W)
            np.testing.assert_array_equal(got[:-PAD].reshape(N * T, W).view(np.uint32), want.view(np.uint32), err_msg=what)


def _pe_patterns(rng, T, N):
    rand = np.where(rng.random((T, N)) < 0.3, rng.integers(1, 256, (T, N)), 0).astype(np.uint8)
    first = np.zeros((T, N), np.uint8)
    first[0] = PE_CODES[rng.integers(0, len(PE_CODES), N)]
    return {"random": rand, "all_ones": np.ones((T, N), np.uint8), "all_zeros": np.zeros((T, N), np.uint8),
            "t0_only": first, "adversarial": adversarial_pe(rng, T, N)}


def test_episode_table_two_passes_against_numpy():
    """Counting pass, then the table pass from a non-prefix ep_offset (columns in reverse order); each pass leaves the
    other's outputs alone and nothing past the table is written."""
    lib, d = L.load(), dev()
    rng = np.random.default_rng(11)
    for T, N in itertools.product([1, 31, 32, 33, 97], [1, 15, 16, 17, 50, 129, 300]):
        for name, pe in _pe_patterns(rng, T, N).items():
            what = f"{name}, T={T}, N={N}"
            count_ref = ((pe != 0) | (np.arange(T) == T - 1)[:, None]).sum(0).astype(np.int32)
            offset = (np.cumsum(count_ref[::-1])[::-1] - count_ref).astype(np.int32)      # column N-1 first
            _, start_ref, len_ref = episode_table_numpy(pe, offset)
            E = len(start_ref)
            pe_d = torch.as_tensor(pe, device=d)
            count = torch.full((N,), -7, dtype=torch.int32, device=d)
            start = torch.full((E + PAD,), -5, dtype=torch.int32, device=d)
            length = torch.full((E + PAD,), -5, dtype=torch.int32, device=d)
            L.check(lib.rs_episode_table(_p(pe_d), T, N, _p(count), None, _p(start), _p(length), _stream()), "count")
            np.testing.assert_array_equal(count.cpu().numpy(), count_ref, err_msg=what)
            assert bool((start == -5).all()) and bool((length == -5).all()), what + ": the counting pass wrote the table"
            count.fill_(-9)
            off_d = torch.as_tensor(offset, device=d)
            L.check(lib.rs_episode_table(_p(pe_d), T, N, _p(count), _p(off_d), _p(start), _p(length), _stream()), "table")
            assert bool((count == -9).all()), what + ": the table pass wrote ep_count"
            s, ln = start.cpu().numpy(), length.cpu().numpy()
            np.testing.assert_array_equal(s[:E], start_ref, err_msg=what)
            np.testing.assert_array_equal(ln[:E], len_ref, err_msg=what)
            assert (s[E:] == -5).all() and (ln[E:] == -5).all(), what + ": written past the table"


def test_team_buffer_get_episodes_matches_restatement():
    """BatchedPPOBuffer(agents=3).get(episodes=True) over N*3 env-major columns: the normalised advantages, the packed
    rows and the episode table against numpy."""
    T, N, A, D = 33, 17, 3, 11
    d = dev()
    rng = np.random.default_rng(5)
    NA = N * A
    buf = rp.BatchedPPOBuffer(D, T, N, agents=A)
    obs = rng.standard_normal((T, NA, D), dtype=np.float32)
    act = rng.integers(0, 8, (T, NA)).astype(np.float32)
    adv, ret, logp = (rng.standard_normal((T, NA), dtype=np.float32) for _ in range(3))
    src = rng.standard_normal((T, NA, 2), dtype=np.float32)
    pe = adversarial_pe(rng, T, NA)
    for field, x in (("obs_buf", obs), ("act_buf", act), ("adv_buf", adv), ("ret_buf", ret), ("logp_buf", logp),
                     ("source_tar", src), ("end_buf", pe)):
        getattr(buf, field).copy_(torch.as_tensor(x, device=d))
    buf.ptr = T
    out = buf.get(episodes=True)
    m_ref, s_ref = two_pass_reference(adv)
    assert math.isclose(out["adv_mean"].item(), m_ref, rel_tol=1e-12) and math.isclose(out["adv_std"].item(), s_ref, rel_tol=1e-12)
    norm = (adv - np.float32(out["adv_mean"].item())) / np.float32(out["adv_std"].item())
    np.testing.assert_array_equal(out["adv"].cpu().numpy().view(np.uint32), norm.reshape(-1).view(np.uint32))
    want = np.concatenate([obs, norm[:, :, None], ret[:, :, None], logp[:, :, None], act[:, :, None], src], axis=2)
    want = want.transpose(1, 0, 2).reshape(NA * T, D + 6)
    np.testing.assert_array_equal(out["packed"].cpu().numpy().view(np.uint32), want.view(np.uint32))
    count = ((pe != 0) | (np.arange(T) == T - 1)[:, None]).sum(0)
    _, start_ref, len_ref = episode_table_numpy(pe, np.concatenate([[0], np.cumsum(count)[:-1]]).astype(np.int64))
    np.testing.assert_array_equal(out["ep_start"].cpu().numpy(), start_ref)
    np.testing.assert_array_equal(out["ep_len"].cpu().numpy(), len_ref)
