"""CPU tests of the RAD-TEAM epoch entry points (rs_rollout_pre_team, rs_rollout_post_team, rs_maps_replay): argument
errors come back as a negative return code with a message in rs_last_error(), before anything is launched.  Plus the
episode-table -> replay-range helper, which is plain tensor arithmetic."""
import ctypes as C

import pytest
import torch

from radiation_ppo_b200 import _lib as L, build
from radiation_ppo_b200.maps_buffer import episode_ranges

DUMMY = C.c_void_p(256)          # a non-NULL pointer that is never dereferenced: every call below fails its checks first


@pytest.fixture(scope="module")
def lib():
    build.build()
    return L.load()


def err(lib):
    return lib.rs_last_error().decode()


def maps_cfg():
    mc, ms = L.RsMapsConfig(), L.RsMapsState()
    mc.n_agents, mc.dim_x, mc.dim_y, mc.base, mc.log_cap, mc.resolution_accuracy, mc.scale = 4, 27, 27, 484, 492, 22.0, 1 / 2200
    ms.visit_lut = DUMMY.value
    return mc, ms


def test_rollout_pre_team_argument_errors(lib):
    f = lib.rs_rollout_pre_team
    d = DUMMY
    assert f(None, d, d, None, None, d, d, d, None, None, None, None, 11, 8, 2, None) < 0 and "NULL buffer" in err(lib)
    assert f(d, d, d, None, None, d, d, d, None, d, None, None, 11, 8, 2, None) < 0 and "src_row without src" in err(lib)
    assert f(d, d, d, None, None, d, d, d, None, None, None, d, 11, 8, 2, None) < 0 and "obs_row without obs" in err(lib)
    assert f(d, d, d, d, None, d, d, d, None, None, None, None, 11, 8, 2, None) < 0 and "pred without pred_row" in err(lib)
    assert f(d, d, d, None, None, d, d, d, None, None, None, None, 11, 0, 2, None) < 0 and "n_env" in err(lib)
    for bad in (0, 9):
        assert f(d, d, d, None, None, d, d, d, None, None, None, None, 11, 8, bad, None) < 0 and "n_agents" in err(lib)


def test_rollout_post_team_argument_errors(lib):
    f = lib.rs_rollout_post_team
    d = DUMMY

    def call(reward=d, team=d, ended=d, v_next=d, boot=d, hidden=None, hdim=0, stats=(None,) * 5, done=d, info=d,
             rew_row=d, n=8, a=2, individual=0):
        return f(reward, team, ended, done, info, v_next, boot, hidden, hdim, *stats, rew_row, d, n, a, individual, 0, None)

    assert call(ended=None) < 0 and "NULL buffer" in err(lib)
    assert call(v_next=None) < 0 and "NULL buffer" in err(lib)
    assert call(team=None) < 0 and "team_reward" in err(lib)
    assert call(reward=None, individual=1) < 0 and "individual rewards need reward" in err(lib)
    assert call(stats=(d, None, d, d, d)) < 0 and "episode statistics" in err(lib)
    assert call(stats=(d, d, d, d, d), info=None) < 0 and "episode statistics" in err(lib)
    assert call(n=0) < 0 and "bad sizes" in err(lib)
    assert call(hidden=d, hdim=0) < 0 and "bad sizes" in err(lib)
    for bad in (0, 9):
        assert call(a=bad) < 0 and "n_agents" in err(lib)


def test_maps_replay_argument_errors(lib):
    f = lib.rs_maps_replay
    d = DUMMY
    mc, ms = maps_cfg()

    def call(cfg=C.byref(mc), st=C.byref(ms), obs=d, pred=d, end=d, T=48, n_env=16, ranges=d, m=4, row0=d, actor=d,
             critic=d, status=d):
        return f(cfg, st, obs, pred, end, T, n_env, ranges, m, row0, actor, critic, status, None)

    assert call(cfg=None) < 0 and "NULL" in err(lib)
    assert call(st=None) < 0 and "NULL" in err(lib)
    assert call(T=0) < 0 and "positive" in err(lib)
    assert call(n_env=-3) < 0 and "positive" in err(lib)
    assert call(m=-1) < 0 and "m must be" in err(lib)
    assert call(obs=None) < 0 and "obs_rows" in err(lib)
    assert call(end=None) < 0 and "end_rows" in err(lib)
    for k in ("ranges", "row0", "actor", "critic", "status"):
        assert call(**{k: None}) < 0 and "is NULL" in err(lib), k
    assert call(m=0, ranges=None, row0=None, actor=None, critic=None, status=None) == 0      # nothing requested: no launch
    ms.visit_lut = None
    assert call() < 0 and "visit_lut" in err(lib)
    ms.visit_lut = d.value
    for field, value, what in (("n_agents", 9, "n_agents"), ("dim_x", 0, "dimensions"), ("log_cap", 2, "log_cap"),
                               ("scale", 0.0, "scale")):
        old = getattr(mc, field)
        setattr(mc, field, value)
        assert call() < 0 and what in err(lib), field
        setattr(mc, field, old)


def test_maps_log_cap_bounded_by_shared_memory(lib):
    """The update and replay kernels keep 4 sample tables of 10 bytes per reading (+ 16 bytes) in one block's shared
    memory, and sm_100 gives a block 227 KB (232448 bytes): log_cap 5810 is the largest that fits.  A larger one is an
    argument error of rs_maps_update, rs_maps_reset and rs_maps_replay, found before any CUDA call; 5810 passes the check
    (each call below then fails a later check, so nothing is launched)."""
    d = DUMMY
    mc, ms = maps_cfg()
    mc.n_agents = 8
    for k in ("actor", "critic", "log_cell", "log_val", "log_len", "last_cell", "last_pred", "std", "std_count", "status"):
        setattr(ms, k, d.value)

    def update(obs=d):
        return lib.rs_maps_update(C.byref(mc), C.byref(ms), obs, None, None, 0, 16, None)

    def reset():
        return lib.rs_maps_reset(C.byref(mc), C.byref(ms), None, 0, 16, None)

    def replay():
        return lib.rs_maps_replay(C.byref(mc), C.byref(ms), d, d, d, 48, 16, d, 4, d, d, d, d, None)

    for cap in (5811, 8192):
        mc.log_cap = cap
        for f in (update, reset, replay):
            assert f() < 0, (cap, f.__name__)
            assert "log_cap" in err(lib) and "5810" in err(lib) and "232448" in err(lib), (cap, f.__name__)
    mc.log_cap = 5810
    assert update(obs=None) < 0 and err(lib) == "obs is NULL"
    ms.status = None
    assert reset() < 0 and "NULL members" in err(lib)
    ms.visit_lut = None
    assert replay() < 0 and "visit_lut" in err(lib)


def test_episode_ranges_from_an_episode_table():
    """pack_episodes' table of an agents=2 buffer (columns n*2 + a, T = 10): every episode appears once per agent
    column; the ranges keep agent 0's, as (env, t0, t1)."""
    T, A = 10, 2
    # column 0 and 1 (env 0): episodes [0, 4), [4, 10); columns 2 and 3 (env 1): one episode [0, 10)
    ep_start = torch.tensor([0, 4, 10, 14, 20, 30], dtype=torch.int32)
    ep_len = torch.tensor([4, 6, 4, 6, 10, 10], dtype=torch.int32)
    r = episode_ranges(ep_start, ep_len, T, agents=A)
    assert r.dtype == torch.int32
    assert r.tolist() == [[0, 0, 3], [0, 4, 9], [1, 0, 9]]
    assert episode_ranges(ep_start[:2], ep_len[:2], T).tolist() == [[0, 0, 3], [0, 4, 9]]
