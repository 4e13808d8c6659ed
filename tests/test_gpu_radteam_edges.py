"""GPU tests (pytest -m gpu) of the RAD-TEAM kernels at every agent count A = 1..8 and at the map kernel's edge regimes.

- rs_rollout_pre_team / rs_rollout_post_team, called directly, against a numpy restatement and EpisodeStats.update;
- rs_maps_update / rs_maps_reset on constructed observation streams against MapsOracle (oracle/maps_oracle.c): cells
  holding hundreds of samples (several passes of the 32-wide compaction and rank selection), tied readings, cells with
  1, 2 and 3 samples (the median shortcut), agents sharing a cell in one call (the visit count), cells off the map,
  sample tables above 48 KB of shared memory and near the 227 KB limit, overfull tables, masked calls;
- rs_maps_replay against the live stacks of the same streams;
- the bound on the sample table that BatchedMapsBuffer enforces.
The streams are written directly (no env): coordinates are lattice integers times `scale`, readings integer-valued floats
from a small set including 0 (so medians tie), sensor channels zeros and several non-zero values."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import c_oracle as co
from tests.test_gpu_radteam import lattice64, maps_state

pytestmark = pytest.mark.gpu

import radiation_ppo_b200 as rp  # noqa: E402
import radiation_ppo_b200.maps_buffer as mbm  # noqa: E402
from radiation_ppo_b200 import _lib as L  # noqa: E402

SCALE = 1 / 2200.0
F32 = np.float32


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _dev():
    return torch.device("cuda", torch.cuda.current_device())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view({4: np.uint32, 8: np.uint64, 2: np.uint16, 1: np.uint8}[a.dtype.itemsize])


def assert_bits_equal(got, want, msg=""):
    np.testing.assert_array_equal(_bits(np.asarray(got)), _bits(np.asarray(want)), err_msg=msg)


# ---- (a) rs_rollout_pre_team / rs_rollout_post_team ----------------------------------------------------------------------

REWARDS = np.array([-1.0, -0.5, 0.0, 0.5, 1.0], F32)        # returns go negative and tie often
ENDED = np.array([0, 0, 0, 0, 1 | 4, 2 | 4, 4, 1 | 2 | 4], np.uint8)


def post_reference(A, individual, last_step, reward, team, ended, done, info, v_next, hidden, st):
    """rs_rollout_post_team restated: returns the rows and updates `hidden` / the statistics `st` (dict or None) in place."""
    N = ended.shape[0]
    r = reward if individual else np.repeat(team[:, None], A, 1)
    e = ended.astype(np.int64)
    cut = np.ones(N, bool) if last_step else (e & L.E_TIMEOUT) != 0
    rows = dict(rew=r.reshape(-1).astype(F32), end=np.repeat(ended, A),
                boot=np.where(np.repeat(cut, A), v_next.reshape(-1), F32(0)).astype(F32))
    if hidden is not None and not last_step:
        hidden[np.repeat(e != 0, A)] = 0.0
    if st is not None:
        steps = st["steps"] + 1
        ret = st["ret"] + r.astype(np.float64)
        over = (e & (L.E_TERMINAL | L.E_TIMEOUT)) != 0
        acc = st["acc"]
        acc[0] += over.sum()
        acc[3] += steps[over].sum()
        acc[4] += (done != 0).sum(0)
        acc[5] += ((info & L.I_OOB) != 0).sum(0)
        for b in range(A):
            acc[1, b] = math.fsum([acc[1, b]] + list(ret[over, b]))
            acc[2, b] = math.fsum([acc[2, b]] + list(ret[over, b] * ret[over, b]))
            if over.any():
                st["min"][b] = min(st["min"][b], ret[over, b].min())
                st["max"][b] = max(st["max"][b], ret[over, b].max())
        reset = (e & L.E_RESET) != 0
        st["ret"] = np.where(reset[:, None], 0.0, ret)
        st["steps"] = np.where(reset, 0, steps).astype(np.int32)
    return rows


def check_stats(A, ret, steps, acc, mn, mx, st, what):
    assert_bits_equal(ret.cpu().numpy(), st["ret"], f"{what}: ep_return")
    np.testing.assert_array_equal(steps.cpu().numpy(), st["steps"], err_msg=f"{what}: ep_steps")
    acc = acc.cpu().numpy()
    for k in (0, 3, 4, 5):                                            # counts: exact
        np.testing.assert_array_equal(acc[k], st["acc"][k], err_msg=f"{what}: acc[{k}]")
    np.testing.assert_allclose(acc[1:3], st["acc"][1:3], rtol=1e-12, atol=0, err_msg=f"{what}: sums")
    np.testing.assert_array_equal(mn.cpu().numpy(), st["min"], err_msg=f"{what}: min")
    np.testing.assert_array_equal(mx.cpu().numpy(), st["max"], err_msg=f"{what}: max")


@pytest.mark.parametrize("team_mode", ["individual", "cooperative"])
@pytest.mark.parametrize("A", range(1, 9))
def test_rollout_team_kernels_match_numpy(A, team_mode):
    """Several consecutive steps (ep_return / ep_steps carry over) at N = 1, 31, 257, 1000 (partial warps and blocks in the
    shuffle reduction), with every `ended` code, last_step 0 and 1, hidden state of dim 1 / 5 / none, statistics present
    and absent, predictions given and not (NaN rows), observation rows written or not.  Rows, hidden state, returns,
    step counts, counts, min and max are bit-exact; the atomically added sums within 1e-12; and the statistics equal
    EpisodeStats.update (the torch path) on the same inputs."""
    lib, dev = L.load(), _dev()
    individual = int(team_mode == "individual")
    rng = np.random.default_rng(1000 * A + individual)
    variants = [(h, s, p) for h in (None, 1, 5) for s in (True, False) for p in (True, False)]
    for N in (1, 31, 257, 1000):
        for v, (hdim, with_stats, with_pred) in enumerate(variants):
            with_obs = v % 2 == 0
            what = f"N={N} hidden={hdim} stats={with_stats} pred={with_pred} obs={with_obs}"
            NA = N * A
            hidden = None if hdim is None else torch.as_tensor(rng.uniform(0.5, 1.5, (NA, hdim)).astype(F32), device=dev)
            hid_ref = None if hidden is None else hidden.cpu().numpy()
            stats = rp.EpisodeStats(N, A, dev, team_mode=team_mode) if with_stats else None
            torch_stats = rp.EpisodeStats(N, A, dev, team_mode=team_mode)
            st = None if not with_stats else dict(ret=np.zeros((N, A)), steps=np.zeros(N, np.int32), acc=np.zeros((6, A)),
                                                   min=np.full(A, np.inf), max=np.full(A, -np.inf))
            fused = [_p(x) for x in (stats.fused_args() if with_stats else (None,) * 5)]
            for t in range(6):
                last = int(t % 3 == 2)
                # ---- pre: row t <- action / value / log-probability / prediction / source (/ observation) ----
                action = rng.integers(0, 9, (N, A)).astype(np.int32)
                val = rng.normal(size=(N, A)).astype(F32)
                logp = rng.normal(size=(N, A)).astype(F32)
                pred = rng.normal(size=(N, A, 2)).astype(F32) if with_pred else None
                src = rng.integers(0, 2700, (N, 2)).astype(np.int32)
                obs = rng.normal(size=(N, A, 11)).astype(F32)
                g = lambda x: None if x is None else torch.as_tensor(x, device=dev)       # noqa: E731
                rows = {k: torch.full(s, -7.0, device=dev) for k, s in
                        (("act", (NA,)), ("val", (NA,)), ("logp", (NA,)), ("pred", (NA, 2)), ("src", (NA, 2)),
                         ("obs", (NA, 11)), ("rew", (NA,)), ("boot", (NA,)))}
                rows["end"] = torch.full((NA,), 99, dtype=torch.uint8, device=dev)
                ins = [g(x) for x in (action, val, logp, pred, src, obs)]      # kept alive until the launch
                L.check(lib.rs_rollout_pre_team(*[_p(x) for x in ins[:5]],
                                                _p(rows["act"]), _p(rows["val"]), _p(rows["logp"]), _p(rows["pred"]),
                                                _p(rows["src"]), _p(ins[5]) if with_obs else None,
                                                _p(rows["obs"]) if with_obs else None, 11, N, A, _stream()),
                        "rs_rollout_pre_team")
                want_pred = pred.reshape(NA, 2) if with_pred else np.full((NA, 2), np.uint32(0x7fffffff)).view(F32)
                assert_bits_equal(rows["act"].cpu().numpy(), action.reshape(-1).astype(F32), f"{what}: act")
                assert_bits_equal(rows["val"].cpu().numpy(), val.reshape(-1), f"{what}: val")
                assert_bits_equal(rows["logp"].cpu().numpy(), logp.reshape(-1), f"{what}: logp")
                assert_bits_equal(rows["pred"].cpu().numpy(), want_pred, f"{what}: pred")
                assert_bits_equal(rows["src"].cpu().numpy(), np.repeat(src, A, 0).astype(F32), f"{what}: src")
                assert_bits_equal(rows["obs"].cpu().numpy(), obs.reshape(NA, 11) if with_obs else np.full((NA, 11), F32(-7)),
                                  f"{what}: obs")
                # ---- post: rewards / path ends / bootstrap / recurrent state / episode statistics ----
                reward = rng.choice(REWARDS, (N, A))
                team = rng.choice(REWARDS, N)
                ended = rng.choice(ENDED, N)
                done = (rng.random((N, A)) < 0.2).astype(np.uint8)
                info = rng.integers(0, 32, (N, A)).astype(np.uint8)
                v_next = rng.normal(size=(N, A)).astype(F32)
                tr = [g(x) for x in (reward, team, ended, done, info, v_next)]
                L.check(lib.rs_rollout_post_team(*[_p(x) for x in tr],
                                                 _p(rows["boot"]), _p(hidden), hdim or 0, *fused, _p(rows["rew"]),
                                                 _p(rows["end"]), N, A, individual, last, _stream()), "rs_rollout_post_team")
                want = post_reference(A, individual, last, reward, team, ended, done, info, v_next, hid_ref, st)
                w = f"{what} step {t}"
                assert_bits_equal(rows["rew"].cpu().numpy(), want["rew"], f"{w}: rew")
                np.testing.assert_array_equal(rows["end"].cpu().numpy(), want["end"], err_msg=f"{w}: end")
                assert_bits_equal(rows["boot"].cpu().numpy(), want["boot"], f"{w}: boot")
                if hidden is not None:
                    assert_bits_equal(hidden.cpu().numpy(), hid_ref, f"{w}: hidden")
                if with_stats:
                    check_stats(A, *stats.fused_args(), st, f"{w} kernel")
                    torch_stats.update(tr[0], tr[1], tr[3], tr[4], tr[2])
                    check_stats(A, *torch_stats.fused_args(), st, f"{w} EpisodeStats.update")


# ---- (b) rs_maps_update / rs_maps_reset ---------------------------------------------------------------------------------

VALS = np.array([0, 1, 2, 3, 5, 8], F32)          # readings: integer-valued, few distinct, 0 included -> tied medians
SENS = np.array([0.25, 0.5, 1.0], F32)            # non-zero sensor values: the last non-zero one must win
SCENARIOS = ("stack", "swap", "shortcut", "walk")


def episode_cells(rng, scen, A, n_calls, dims):
    """[n_calls, A, 2] integer grid cells of one episode (possibly off the map or negative)."""
    X, Y = dims
    if scen == "stack":                              # everyone idles in one cell: m = A * calls, far past 64
        return np.broadcast_to(rng.integers(0, [X, Y]), (n_calls, A, 2)).copy()
    if scen == "swap":                               # agents trade between 2 or 3 cells: several share a cell per call
        pool = rng.integers(0, [X, Y], size=(int(rng.integers(2, 4)), 2))
        return pool[rng.integers(0, len(pool), size=(n_calls, A))]
    if scen == "shortcut":                           # agent a on its own row, 1, 2, 3 calls per cell in turn
        js = np.concatenate([[j] * (j % 3 + 1) for j in range(n_calls)])[:n_calls]
        y0 = int(rng.integers(0, Y))
        out = np.empty((n_calls, A, 2), np.int64)
        for a in range(A):
            out[:, a, 0] = (3 * a) % X
            out[:, a, 1] = (y0 + js) % Y
        return out
    # random walk from near an edge of the map or of the wrapped negative cells: leaves the map, wraps
    lo, hi = np.array([-X - 3, -Y - 3]), np.array([X + 2, Y + 2])
    pos = np.clip(rng.choice([-X - 3, -3, X - 2], size=(A, 2)) + rng.integers(0, 5, size=(A, 2)), lo, hi)
    out = np.empty((n_calls, A, 2), np.int64)
    for k in range(n_calls):
        out[k] = pos
        pos = np.clip(pos + rng.integers(-1, 2, size=(A, 2)), lo, hi)
    return out


def lattice_coords(rng, cells):
    """float32 scaled coordinates whose int(x * 22) (truncated toward zero) is `cells` (cells of 100 lattice units)"""
    off = rng.integers(10, 91, size=cells.shape)
    lat = np.where(cells >= 0, cells * 100 + off, cells * 100 - off)
    return (lat * SCALE).astype(F32)


def make_obs(rng, cells):
    sh = cells.shape[:-1]
    obs = np.zeros(sh + (11,), F32)
    obs[..., 0] = rng.choice(VALS, size=sh)
    obs[..., 1:3] = lattice_coords(rng, cells)
    sens = rng.choice(SENS, size=sh + (8,))
    sens[rng.random(sh + (8,)) < 0.6] = 0.0
    obs[..., 3:] = sens
    return obs


def make_pred(rng, A, dims, pool):
    """[A, 2]: cells from a small per-env pool (the mark often stays), NaN rows (also a single NaN coordinate), off-map"""
    X, Y = dims
    pred = lattice_coords(rng, pool[rng.integers(0, len(pool), A)])
    u = rng.random(A)
    pred[u < 0.12] = np.nan
    pred[(u >= 0.12) & (u < 0.18), 1] = np.nan
    off = (u >= 0.18) & (u < 0.28)
    pred[off] = ((np.array([X, Y]) * 100 + 250) * SCALE * rng.choice([-1.2, 1.0], size=(int(off.sum()), 1))).astype(F32)
    return pred


def cells_of(xy, dims, ra, lattice):
    """the kernel's cell_of over [..., 2] float32 coordinates: flat cell or -1 (off the map)"""
    X, Y = dims
    v = xy.astype(np.float64)
    if lattice:                                                        # observations: the lattice coordinate recovered
        v = np.rint(v / SCALE) * SCALE
    with np.errstate(invalid="ignore"):
        c = np.trunc(v * ra)
    c = np.where(np.isnan(c), -(10 ** 6), c).astype(np.int64)
    cx, cy = c[..., 0], c[..., 1]
    cx = np.where(cx < 0, cx + X, cx)
    cy = np.where(cy < 0, cy + Y, cy)
    ok = (cx >= 0) & (cy >= 0) & (cx < X) & (cy < Y)
    return np.where(ok, cx * Y + cy, -1)


class Stream:
    """S policy calls for N envs of A agents, with episode ends, the final observations of the ended episodes (the
    bootstrap call) and their predictions.  Env n plays SCENARIOS[n % 4]; `endless` envs never end an episode."""

    def __init__(self, rng, N, A, ML, S, dims, endless=(), full_first=False, noise=False):
        X, Y = dims
        self.N, self.A, self.S = N, A, S
        self.obs = np.zeros((S, N, A, 11), F32)
        self.pred = np.zeros((S, N, A, 2), F32)
        self.fin_obs = np.zeros((S, N, A, 11), F32)
        self.fin_pred = np.zeros((S, N, A, 2), F32)
        self.end = np.zeros((S, N), np.uint8)                      # RS_E_* bits of the ended episodes (all with E_RESET)
        self.starts = [[] for _ in range(N)]
        for n in range(N):
            scen = SCENARIOS[n % 4]
            pool = rng.integers([-X, -Y], [X, Y], size=(3, 2))
            t = 0
            while t < S:
                if n in endless:
                    Lep = S
                elif full_first and t == 0:
                    Lep = ML
                else:
                    Lep = ML if rng.random() < 0.4 else int(rng.integers(1, ML + 1))
                Lep = min(Lep, S - t)
                cells = episode_cells(rng, scen, A, Lep + 1, dims)
                self.starts[n].append(t)
                self.obs[t:t + Lep, n] = make_obs(rng, cells[:Lep])
                for k in range(Lep):
                    self.pred[t + k, n] = make_pred(rng, A, dims, pool)
                e = t + Lep - 1
                if n not in endless:
                    self.fin_obs[e, n] = make_obs(rng, cells[Lep])
                    self.fin_pred[e, n] = make_pred(rng, A, dims, pool)
                    if Lep == ML:
                        self.end[e, n] = (2 | 4) if rng.random() < 0.7 else (1 | 2 | 4)
                    else:
                        self.end[e, n] = 4 if e == S - 1 else (1 | 4)
                t += Lep
        # the bootstrap / reset mask: codes without E_RESET elsewhere must not select (mask_bits = 4)
        self.mask = self.end.copy()
        if noise:
            k = (self.mask == 0) & (rng.random((S, N)) < 0.3)
            self.mask[k] = rng.choice(np.array([1, 2, 3], np.uint8), size=int(k.sum()))


def state_rows(mb, idx):
    """the raw bytes of every state tensor of the envs idx"""
    return [t[idx].contiguous().view(torch.uint8) for t in (
        mb._actor_store, mb._critic_store, mb._log_cell, mb._log_val, mb._log_len, mb._last_cell, mb._last_pred, mb._std,
        mb._std_count, mb.status)]


class MapsRun:
    """Drives a BatchedMapsBuffer through a Stream the way TeamRolloutCollector does (per step: update; for the ended
    episodes a bootstrap update and a reset, both masked by the end code & E_RESET) and checks every call: the envs not
    selected keep every state byte; the selected sampled envs' stacks equal MapsOracle (channels 1..6 and the critic) and
    the prediction rule (channel 0); status is exactly the RS_MS_* bits their calls earned."""

    def __init__(self, mb, st, sample, bufs=None, use_prediction=True):
        self.mb, self.st, self.A, self.dims = mb, st, mb.number_of_agents, mb.map_dimensions
        self.sample, self.bufs = list(sample), list(range(self.A)) if bufs is None else list(bufs)
        self.use_prediction = use_prediction
        ra = mb.resolution_accuracy
        self.ra = ra
        self.oracles = {n: {i: co.MapsOracle(self.A, mb.steps_per_episode, dims=self.dims, resolution_accuracy=ra)
                            for i in self.bufs} for n in self.sample}
        N = mb.num_envs
        self.last_pred = np.full((N, self.A), -1, np.int64)
        self.calls = np.zeros(N, np.int64)                 # calls since the last reset
        self.status = np.zeros(N, np.int64)
        self.cap = mb._cfg.log_cap
        self.checked = 0                                   # oracle comparisons made
        self.full_seen = np.zeros(N, bool)

    def update(self, obs, pred, mask, bits, sel, what):
        mb, dev, A, N = self.mb, self.mb.device, self.A, self.mb.num_envs
        unsel = torch.as_tensor(np.where(~sel)[0], device=dev)
        before = state_rows(mb, unsel)
        mb.update(torch.as_tensor(obs, device=dev), None if pred is None else torch.as_tensor(pred, device=dev),
                  mask=None if mask is None else torch.as_tensor(mask, device=dev), mask_bits=bits)
        for x, y in zip(before, state_rows(mb, unsel)):
            assert torch.equal(x, y), f"{what}: an env outside the mask changed"
        # the reference's bookkeeping of the selected envs
        self.calls[sel] += 1
        full = sel & (self.calls * A > self.cap)
        self.full_seen |= full
        self.status[full] |= L.MS_LOG_FULL
        oc = cells_of(obs[..., 1:3], self.dims, self.ra, lattice=True)
        self.status[sel & (oc < 0).any(1)] |= L.MS_CELL_RANGE
        if self.use_prediction and pred is not None:
            given = ~np.isnan(pred).any(-1)
            pc = cells_of(pred, self.dims, self.ra, lattice=False)
            upd = given & sel[:, None]
            self.last_pred[upd] = pc[upd]
            self.status[sel & (upd & (pc < 0)).any(1)] |= L.MS_PRED_RANGE
        np.testing.assert_array_equal(mb.status.cpu().numpy(), self.status, err_msg=f"{what}: status")
        # the sampled envs
        idx = [n for n in self.sample if sel[n]]
        if not idx:
            return
        actor = mb.actor_maps[idx].cpu().numpy()
        critic = mb.critic_maps[idx].cpu().numpy()
        X, Y = self.dims
        for j, n in enumerate(idx):
            w = f"{what} env {n} ({SCENARIOS[n % 4]}) call {self.calls[n]}"
            ch0 = np.zeros((A, X * Y), F32)
            for a in range(A):
                if self.last_pred[n, a] >= 0:
                    ch0[a, self.last_pred[n, a]] = 1.0
            np.testing.assert_array_equal(actor[j][:, 0].reshape(A, -1), ch0, err_msg=f"{w}: prediction map")
            for i in range(A):                                           # channels shared by every buffer and the critic
                np.testing.assert_array_equal(actor[j][i, 3:6], critic[j][1:4], err_msg=f"{w}: critic channels 1..3")
            if self.full_seen[n]:
                continue                                                 # the oracle's table is larger: compare until full
            o64 = lattice64(obs[n], SCALE)
            for i in self.bufs:
                p = (0.0, 0.0) if pred is None or np.isnan(pred[n, i]).any() else (float(pred[n, i, 0]), float(pred[n, i, 1]))
                want = self.oracles[n][i].observation_to_map(o64, i, p)
                np.testing.assert_array_equal(actor[j][i, 1:6], want[1:6], err_msg=f"{w}: buffer {i} channels 1..5")
                np.testing.assert_array_equal(critic[j][0], want[6], err_msg=f"{w}: combined locations")
                self.checked += 1

    def reset(self, mask, sel, what):
        mb, dev = self.mb, self.mb.device
        unsel = torch.as_tensor(np.where(~sel)[0], device=dev)
        before = state_rows(mb, unsel)
        mb.reset(mask=torch.as_tensor(mask, device=dev), mask_bits=L.E_RESET)
        for x, y in zip(before, state_rows(mb, unsel)):
            assert torch.equal(x, y), f"{what}: reset changed an env outside the mask"
        s = torch.as_tensor(np.where(sel)[0], device=dev)
        assert not mb._actor_store[s].any() and not mb._critic_store[s].any(), what
        assert not mb._log_len[s].any() and not mb._std[s].any() and not mb._std_count[s].any(), what
        assert bool((mb._last_cell[s] == -1).all()) and bool((mb._last_pred[s] == -1).all()), what
        self.calls[sel] = 0
        self.last_pred[sel] = -1
        self.full_seen[sel] = False
        for n in self.sample:
            if sel[n]:
                for o in self.oracles[n].values():
                    o.reset()

    def play(self, rng, masked=True, what=""):
        st, N = self.st, self.mb.num_envs
        self.mb.reset()
        for t in range(st.S):
            w = f"{what} step {t}"
            mask, bits, sel = None, 0, np.ones(N, bool)
            if masked and rng.random() < 0.7:
                bits = int(rng.choice([0, 2, 6]))
                mask = rng.integers(0, 8, N).astype(np.uint8)
                sel = (mask & (bits or 0xff)) != 0
            pred = None if rng.random() < 0.08 else st.pred[t]
            self.update(st.obs[t], pred, mask, bits, sel, w)
            ends = (st.mask[t] & L.E_RESET) != 0
            if ends.any():
                self.update(st.fin_obs[t], st.fin_pred[t], st.mask[t], L.E_RESET, ends, f"{w} bootstrap")
                self.reset(st.mask[t], ends, f"{w} reset")


def maps_run(A, ML, N, S, seed, sample=None, bufs=None, masked=True, use_prediction=True, endless=(), full_first=False,
             **kw):
    rng = np.random.default_rng(seed)
    mb = rp.BatchedMapsBuffer(N, A, ML, environment_scale=SCALE, use_prediction=use_prediction, **kw)
    st = Stream(rng, N, A, ML, S, mb.map_dimensions, endless=endless, full_first=full_first, noise=True)
    run = MapsRun(mb, st, range(N) if sample is None else sample, bufs, use_prediction)
    run.play(rng, masked, what=f"A={A} ML={ML}")
    assert run.checked > 0
    return run


@pytest.mark.parametrize("A", range(1, 9))
def test_maps_short_episodes_match_oracle(A):
    """Episodes of up to 24 steps, N = 4k + 3 envs (the last block is not full), random masks on most calls."""
    run = maps_run(A, 24, 35, 60, seed=A, sample=range(0, 35, 2))
    assert not run.full_seen.any()


@pytest.mark.parametrize("A", range(1, 9))
def test_maps_long_episodes_match_oracle(A):
    """Episodes of up to 200 steps: the stacked cells hold up to 201 * A samples; at A = 7 and 8 the sample tables need
    more than 48 KB of shared memory per block."""
    run = maps_run(A, 200, 11, 230, seed=50 + A, sample=range(8), full_first=True)
    assert not run.full_seen.any()


def test_maps_table_near_the_shared_memory_limit():
    """A = 8, one 720-step episode (+ the bootstrap call): 5768 readings in a table of 5784 (231 KB of the 227 KB a block
    may have), an env whose one cell holds them all; buffers 0 and 7 of three envs against the oracle."""
    run = maps_run(8, 720, 7, 720, seed=9, sample=[0, 1, 3], bufs=[0, 7], masked=False, full_first=True)
    assert run.mb._cfg.log_cap == 5784 and not run.full_seen.any()


@pytest.mark.parametrize("A", (3, 8))
def test_maps_without_prediction(A):
    """use_prediction=False: the prediction map stays zero whatever the predictions; the rest still matches."""
    run = maps_run(A, 24, 11, 50, seed=70 + A, use_prediction=False)
    assert not run.mb._actor_store[..., 0].any()


def test_maps_unenforced_147_grid_a8():
    """The 147 x 147 map of unenforced boundaries at A = 8 (random walks reach wrapped negative cells and leave the map)."""
    ra = mbm.calculate_resolution_accuracy(0.01, SCALE)
    run = maps_run(8, 120, 7, 130, seed=31, sample=[1, 3, 5], bufs=[0, 3, 7], resolution_accuracy=ra,
                   offset=SCALE * (500.0 + 120 * 100.0))
    assert run.mb.map_dimensions == (147, 147)


@pytest.mark.parametrize("A", (1, 5, 8))
def test_maps_overfull_table_flags_only_its_envs(A):
    """Envs 1, 6 and 8 never reset: after steps_per_episode + 3 calls their tables are full, RS_MS_LOG_FULL is set for
    them only (status is checked exactly at every call), and their stacks equal the oracle's until the call that
    overflows."""
    run = maps_run(A, 24, 11, 40, seed=90 + A, endless=(1, 6, 8), masked=False)
    assert [n for n in range(11) if run.status[n] & L.MS_LOG_FULL] == [1, 6, 8]


# ---- (c) rs_maps_replay ------------------------------------------------------------------------------------------------

def _store_equal(got, want):
    return torch.equal(got.contiguous().view(torch.int32), want.contiguous().view(torch.int32))


@pytest.mark.parametrize("ML", (24, 200))
@pytest.mark.parametrize("A", (3, 5, 7, 8))
def test_replay_matches_live_stacks(A, ML):
    """The streams of the map tests written into a BatchedPPOBuffer; the live updates run as the collector runs them, with
    a snapshot of the stacks at every step.  Replays of single rows (first, last and random rows of episodes), of whole
    episodes and of the whole epoch of some envs (episode starts inside the range) are bit-identical to the snapshots;
    the live state is left untouched.  ML = 200 at A = 7, 8: tables above 48 KB of shared memory."""
    rng = np.random.default_rng(10 * A + ML)
    N, S = 11, ML + ML // 2 + 7
    dev = _dev()
    mb = rp.BatchedMapsBuffer(N, A, ML, environment_scale=SCALE)
    st = Stream(rng, N, A, ML, S, mb.map_dimensions, full_first=True)
    buf = rp.BatchedPPOBuffer(11, S, N, agents=A)
    buf._obs_store[:S].copy_(torch.as_tensor(st.obs.reshape(S, N * A, 11)))
    buf.pred_buf.copy_(torch.as_tensor(st.pred.reshape(S, N * A, 2)))
    buf.end_buf.copy_(torch.as_tensor(np.repeat(st.end, A, axis=1)))
    mb.reset()
    snaps = []
    for t in range(S):
        mb.update(torch.as_tensor(st.obs[t], device=dev), torch.as_tensor(st.pred[t], device=dev))
        snaps.append((mb._actor_store.clone(), mb._critic_store.clone()))
        if st.end[t].any():
            m = torch.as_tensor(st.end[t], device=dev)
            mb.update(torch.as_tensor(st.fin_obs[t], device=dev), torch.as_tensor(st.fin_pred[t], device=dev), mask=m,
                      mask_bits=L.E_RESET)
            mb.reset(mask=m, mask_bits=L.E_RESET)
    before = maps_state(mb)

    def check(ranges, label):
        actor, critic, status = mb.replay(buf, torch.as_tensor(ranges, dtype=torch.int32))
        assert not (status.cpu().numpy() & L.MR_BAD_RANGE).any(), label
        a, c = actor.permute(0, 1, 3, 4, 2), critic.permute(0, 2, 3, 1)
        row = 0
        for n, t0, t1 in ranges:
            for t in range(t0, t1 + 1):
                assert _store_equal(a[row], snaps[t][0][n]), f"{label}: env {n} step {t} actor"
                assert _store_equal(c[row], snaps[t][1][n]), f"{label}: env {n} step {t} critic"
                row += 1
        assert row == actor.shape[0]

    singles, episodes = [], []
    for n in range(N):
        starts = st.starts[n]
        ends = [s - 1 for s in starts[1:]] + [S - 1]
        episodes += [[n, s, e] for s, e in zip(starts, ends)]
        rows = {0, S - 1, *starts, *ends, *rng.integers(0, S, 3).tolist()}
        singles += [[n, t, t] for t in sorted(rows)]
    check(singles, "single rows")
    check(episodes, "whole episodes")
    check([[n, 0, S - 1] for n in (0, 5, 10)], "whole epoch")
    for x, y in zip(before, maps_state(mb)):
        assert torch.equal(x, y)


# ---- the bound on the sample table ---------------------------------------------------------------------------------------

def test_maps_buffer_refuses_tables_beyond_shared_memory():
    """(steps_per_episode + 3) * number_of_agents readings must fit 5810: A = 8 allows 723 steps, not 724."""
    with pytest.raises(ValueError, match=r"steps_per_episode=724 with number_of_agents=8"):
        rp.BatchedMapsBuffer(3, 8, 724, environment_scale=SCALE)
    with pytest.raises(ValueError, match=r"steps_per_episode=5808 with number_of_agents=1"):
        rp.BatchedMapsBuffer(3, 1, 5808, environment_scale=SCALE)
    mb = rp.BatchedMapsBuffer(3, 8, 723, environment_scale=SCALE)
    assert mb._cfg.log_cap == 5808
    obs = make_obs(np.random.default_rng(0), np.full((3, 8, 2), 5))
    actor, _ = mb.update(torch.as_tensor(obs, device=mb.device))
    torch.cuda.synchronize()
    assert int(mb.status.sum()) == 0 and float(actor[:, :, 4].max()) > 0
