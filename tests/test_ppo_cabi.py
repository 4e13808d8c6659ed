"""CPU tests of the PPO-buffer entry points rs_gae, rs_adv_stats, rs_adv_normalize, rs_pack_rollout and rs_episode_table:
every argument error comes back as a negative return code with a message in rs_last_error(), before anything is launched."""
import ctypes as C

import pytest

from radiation_ppo_b200 import _lib as L, build

DUMMY = C.c_void_p(256)          # a non-NULL, 16-byte aligned pointer that is never dereferenced: every call below fails first
MISALIGNED = C.c_void_p(260)     # 4 bytes past a 16-byte boundary
ODD = C.c_void_p(258)            # not even 4-byte aligned


@pytest.fixture(scope="module")
def lib():
    build.build()
    return L.load()


def err(lib):
    return lib.rs_last_error().decode()


def test_gae_argument_errors(lib):
    d = DUMMY
    names = ("rew", "val", "pe", "boot", "adv", "ret", "T", "N", "gamma", "lam", "stats", "variant")

    def call(**kw):
        args = dict.fromkeys(names, d)
        args.update(T=480, N=4096, gamma=0.99, lam=0.9, stats=None, variant=0)
        args.update(kw)
        return lib.rs_gae(*[args[k] for k in names], None)

    for k in ("rew", "val", "pe", "boot", "adv", "ret"):
        assert call(**{k: None}) < 0 and "NULL buffer" in err(lib), k
    for kw in (dict(T=0), dict(T=-3), dict(N=0), dict(N=-128)):
        assert call(**kw) < 0 and "T and N must be positive" in err(lib), kw
    for v in (-1, 5, 6, 9, 16, 99, -2 ** 31):
        assert call(variant=v) < 0 and "unknown variant" in err(lib), v
    # the scan keeps T * 104 bytes in shared memory: 227 KB hold 2235 steps
    for t in (2236, 2 ** 31 - 1):
        assert call(variant=2, T=t, N=64) < 0 and "T too large for the scan variant" in err(lib), t
    # every tile variant needs whole 128-column tiles and 16-byte aligned rew / val / path_end
    for v in (7, 8, 10, 11, 12, 13, 14, 15):
        for n in (127, 129, 4100, 16383 + 128):
            assert call(variant=v, N=n) < 0 and "N % 128 == 0" in err(lib), (v, n)
        for k in ("rew", "val", "pe"):
            assert call(variant=v, **{k: MISALIGNED}) < 0 and "16-byte aligned" in err(lib), (v, k)


def test_adv_stats_and_normalize_argument_errors(lib):
    d = DUMMY
    for n in (0, -1, -(2 ** 40)):
        assert lib.rs_adv_stats(d, n, None, d, None) < 0 and "bad arguments" in err(lib), n
        assert lib.rs_adv_normalize(d, n, d, d, None) < 0 and "bad arguments" in err(lib), n
    assert lib.rs_adv_stats(None, 10, None, d, None) < 0 and "bad arguments" in err(lib)
    assert lib.rs_adv_stats(d, 10, None, None, None) < 0 and "bad arguments" in err(lib)
    for k in range(3):
        args = [d, d, d]
        args[k] = None
        assert lib.rs_adv_normalize(args[0], 10, args[1], args[2], None) < 0 and "bad arguments" in err(lib), k
    assert lib.rs_adv_stats(ODD, 10, None, d, None) < 0 and "not 4-byte aligned" in err(lib)
    assert lib.rs_adv_normalize(ODD, 10, d, d, None) < 0 and "not 4-byte aligned" in err(lib)


def test_pack_rollout_argument_errors(lib):
    d = DUMMY
    names = ("obs", "adv", "ret", "logp", "act", "src", "packed", "T", "N", "D")

    def call(**kw):
        args = dict.fromkeys(names, d)
        args.update(T=32, N=16, D=11)
        args.update(kw)
        return lib.rs_pack_rollout(*[args[k] for k in names], None)

    for k in ("obs", "adv", "ret", "logp", "act", "packed"):
        assert call(**{k: None}) < 0 and "NULL buffer" in err(lib), k
    for kw in (dict(T=0), dict(T=-1), dict(N=0), dict(N=-16), dict(D=0), dict(D=-1), dict(D=65), dict(D=1000)):
        assert call(**kw) < 0 and "bad T / N / D" in err(lib), kw


def test_episode_table_argument_errors(lib):
    d = DUMMY

    def call(pe=d, T=32, N=16, count=d, offset=None, start=None, length=None):
        return lib.rs_episode_table(pe, T, N, count, offset, start, length, None)

    for kw in (dict(pe=None), dict(T=0), dict(T=-1), dict(N=0), dict(N=-5)):
        assert call(**kw) < 0 and "bad arguments" in err(lib), kw
    assert call(count=None) < 0 and "counting pass needs ep_count" in err(lib)
    for kw in (dict(start=None, length=d), dict(start=d, length=None), dict(start=None, length=None)):
        assert call(offset=d, **kw) < 0 and "table pass needs ep_start / ep_len" in err(lib), kw
