"""CPU tests of the Monte-Carlo evaluation entry point rs_eval_step: every argument error comes back as a negative return
code with a message in rs_last_error(), before anything is launched."""
import ctypes as C

import pytest

from radiation_ppo_b200 import _lib as L, build

DUMMY = C.c_void_p(256)          # a non-NULL pointer that is never dereferenced: every call below fails its checks first


@pytest.fixture(scope="module")
def lib():
    build.build()
    return L.load()


def err(lib):
    return lib.rs_last_error().decode()


def test_eval_step_argument_errors(lib):
    d = DUMMY
    names = ("reward", "team", "done", "info", "active", "success", "length", "ep_return", "oob", "finders", "n_active",
             "pred", "src", "scale", "loc_sum", "loc_n", "loc_last", "n", "a", "individual")

    def call(**kw):
        # a bad call that every check but the one under test would accept (no prediction group unless asked for)
        args = dict.fromkeys(names, d)
        args.update(pred=None, src=None, scale=0.0, loc_sum=None, loc_n=None, loc_last=None, n=1000, a=4, individual=0)
        args.update(kw)
        return lib.rs_eval_step(*[args[k] for k in names], None)

    for bad in (0, -5):
        assert call(n=bad) < 0 and "n_env" in err(lib)
    for bad in (0, 9):
        assert call(a=bad) < 0 and "n_agents" in err(lib)
    assert call(team=None) < 0 and "team rewards need team_reward" in err(lib)
    assert call(reward=None, individual=1) < 0 and "individual rewards need reward" in err(lib)
    for k in ("done", "info", "active", "success", "length", "ep_return", "oob", "n_active"):
        assert call(**{k: None}) < 0 and "NULL buffer" in err(lib), k
    group = dict(pred=d, src=d, scale=1 / 2200, loc_sum=d, loc_n=d, loc_last=d)
    for k in ("src", "loc_sum", "loc_n", "loc_last"):
        assert call(**{**group, k: None}) < 0 and "pred needs" in err(lib), k
    for bad in (0.0, -1.0, float("nan")):
        assert call(**{**group, "scale": bad}) < 0 and "scale > 0" in err(lib), bad
