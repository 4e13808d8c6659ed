"""GPU tests (pytest -m gpu) of the RAD-TEAM epoch: TeamRolloutCollector (the multi-agent branch of train.py:321-571 with
the map observation in the loop, rs_rollout_pre_team / rs_rollout_post_team) against the oracle env stepped the
reference's way and oracle/maps_oracle.c, and BatchedMapsBuffer.replay (rs_maps_replay) against the stacks the policy
read during the collection."""
import numpy as np
import pytest
import torch

from oracle import c_oracle as co
from tests import parity_util as pu

pytestmark = pytest.mark.gpu

import radiation_ppo_b200 as rp  # noqa: E402
import radiation_ppo_b200.maps_buffer as mbm  # noqa: E402


def stacks_to_seven(actor, critic, i):
    """the reference's MapStack order for agent i's buffer: prediction, location, others, readings, visits, obstacles, combined"""
    return np.concatenate([actor[i], critic[:1]], axis=0)


def lattice64(o, scale):
    """the reference's float64 observation of a float32 env observation [A, 11] (x * scale on the lattice coordinate)"""
    o64 = np.asarray(o, np.float64).copy()
    o64[:, 1:3] = np.rint(o64[:, 1:3] / scale) * scale
    return o64


class Scripted:
    """A team policy whose prediction / action / value / log-probability are deterministic functions of its inputs (the
    actions come from a fixed table, one row per step).  It records what it was given for the sampled envs: the
    observation and prediction of every predict() call and the live stacks at every act() and value() call."""

    def __init__(self, maps, actions, sample, W):
        d = maps.device
        self.maps, self.acts, self.t = maps, torch.as_tensor(actions, device=d), 0
        self.idx = torch.as_tensor(sample, device=d)
        self.W = torch.as_tensor(W, device=d)
        N, A = maps.num_envs, maps.number_of_agents
        self.A = A
        self.hidden_state = torch.ones(N * A, 3, device=d)            # restarted in place by rs_rollout_post_team
        self.clear()

    def clear(self):
        self.pred_calls, self.act_snaps, self.boot_snaps, self.v_next = [], [], [], []

    def value_fn(self, critic):
        v = torch.tanh(0.01 * (critic * self.W).sum(dim=(1, 2, 3)))
        return (v[:, None] + 0.001 * torch.arange(self.A, device=v.device)).contiguous()

    def predict(self, obs):
        pred = (obs[..., 1:3] * 0.5 + 0.25).contiguous()
        self.pred_calls.append((obs[self.idx].cpu().numpy(), pred[self.idx].cpu().numpy()))
        return pred

    def act(self, obs, actor, critic):
        self.act_snaps.append((actor[self.idx].cpu().numpy(), critic[self.idx].cpu().numpy()))
        a = self.acts[self.t]
        self.t += 1
        v = self.value_fn(critic)
        return a, v, (-0.5 * v).contiguous()

    def value(self, critic):
        self.boot_snaps.append((self.maps.actor_maps[self.idx].cpu().numpy(), critic[self.idx].cpu().numpy()))
        v = self.value_fn(critic)
        self.v_next.append(v.cpu().numpy())
        return v

    def reset_state(self, mask):
        assert mask is None
        self.hidden_state.fill_(1.0)


def maps_state(mb):
    return [t.clone() for t in (mb._actor_store, mb._critic_store, mb._log_cell, mb._log_val, mb._log_len, mb._last_cell,
                                mb._last_pred, mb._std, mb._std_count, mb.status)]


def check_replay(mb, buf, pol, sample, T, rng):
    """replay of single rows and of whole episodes == the stacks the policy read (pol.act_snaps of this epoch); the live
    state is left byte-identical"""
    A = mb.number_of_agents
    before = maps_state(mb)
    end = buf.end_buf.cpu().numpy().reshape(T, -1, A)[:, :, 0]
    pairs = []
    for j, n in enumerate(sample):
        term = np.where(end[:, n] & 1)[0]
        starts = [0] + list(np.where(end[:-1, n] != 0)[0] + 1)
        pairs += [(j, 0), (j, T - 1), (j, int(rng.integers(0, T))), (j, int(starts[-1]))]
        if len(term):
            pairs.append((j, int(term[0])))                         # the last row of a terminal episode
    ranges = torch.as_tensor([[sample[j], t, t] for j, t in pairs], dtype=torch.int32)
    actor, critic, status = mb.replay(buf, ranges)
    assert int(status.abs().sum()) == 0
    a, c = actor.cpu().numpy(), critic.cpu().numpy()
    for k, (j, t) in enumerate(pairs):
        np.testing.assert_array_equal(a[k], pol.act_snaps[t][0][j], err_msg=f"single row env {sample[j]} step {t}")
        np.testing.assert_array_equal(c[k], pol.act_snaps[t][1][j], err_msg=f"single row env {sample[j]} step {t}")
    # whole episodes of the sampled envs, from the buffer's episode table
    _, ep_start, ep_len = buf.pack_episodes()
    rg = rp.episode_ranges(ep_start, ep_len, T, agents=A).cpu()
    rg = rg[torch.as_tensor(np.isin(rg[:, 0].numpy(), sample))]
    assert len(rg) >= len(sample) and int((rg[:, 2] - rg[:, 1] + 1).sum()) == T * len(sample)
    actor, critic, status = mb.replay(buf, rg)
    assert int(status.abs().sum()) == 0
    a, c = actor.cpu().numpy(), critic.cpu().numpy()
    row = 0
    for n, t0, t1 in rg.tolist():
        j = list(sample).index(n)
        for t in range(t0, t1 + 1):
            np.testing.assert_array_equal(a[row], pol.act_snaps[t][0][j], err_msg=f"episode row env {n} step {t}")
            np.testing.assert_array_equal(c[row], pol.act_snaps[t][1][j], err_msg=f"episode row env {n} step {t}")
            row += 1
    for x, y in zip(before, maps_state(mb)):
        assert torch.equal(x, y)


@pytest.mark.parametrize("A,mode,team_mode", [(1, "rows", "cooperative"), (1, "graph", "individual")] +
                         [(A, m, tm) for A in (2, 4) for m in ("rows", "graph") for tm in ("individual", "cooperative")] +
                         [(3, "rows", "individual"), (6, "graph", "cooperative"), (8, "rows", "cooperative"),
                          (8, "graph", "individual")])
def test_team_collector_epoch_matches_oracle_and_replay(A, mode, team_mode):
    """Two epochs of TeamRolloutCollector against the oracle env stepped the reference's way: observation rows, rewards per
    team mode, path ends in all A columns, actions, source coordinates, predictions, the bootstrap rule, GAE, the
    recurrent-state restart and the per-agent episode statistics; the live map stacks of sampled envs vs MapsOracle at
    every step and at the bootstrap call; then replay of single rows (first / last rows of episodes and of the epoch) and
    of whole episodes equals the stacks the policy read (and so the oracle's)."""
    N, T, ML = 512, 72, 24
    env = rp.RadSearch(obstruction_count=5, enforce_grid_boundaries=True, number_agents=A, num_envs=N, seed=77,
                       steps_per_episode=ML, auto_reset=True, prefetch=(mode == "graph"), use_cuda_graph=(mode == "graph"))
    ob = co.OracleBatch(N, co.default_config(n_agents=A, obstruction_count=5, enforce=1, max_ep_len=ML), seed=77)
    ob.reset()
    d = env.device
    rng = np.random.default_rng(11)
    sample = np.sort(rng.choice(N, 8, replace=False))
    mb = rp.BatchedMapsBuffer(N, A, ML, environment_scale=env.scale)
    X, Y = mb.map_dimensions
    W = rng.normal(size=(4, X, Y)).astype(np.float32)
    actions = rng.integers(0, 8, size=(2 * T, N, A)).astype(np.int32)
    pol = Scripted(mb, actions, sample, W)
    buf = rp.BatchedPPOBuffer(11, T, N, agents=A)
    stats = rp.EpisodeStats(N, A, d, team_mode=team_mode)
    col = rp.TeamRolloutCollector(env, buf, mb, pol, stats, mode=mode, team_mode=team_mode)
    oracles = {n: [co.MapsOracle(A, ML) for _ in range(A)] for n in sample}
    ep_ret, ep_len = np.zeros((N, A)), np.zeros(N, int)
    for epoch in range(2):
        cur = ob.outs["obs"][:, :A].copy()
        pol.clear()
        col.collect(gae_variant=1)
        obs_o = np.zeros((T, N, A, 11)); rew_o = np.zeros((T, N, A), np.float32)
        end_o = np.zeros((T, N), bool); cut_o = np.zeros((T, N), bool); src_o = np.zeros((T, N, 2), np.float32)
        rets, lens = [[] for _ in range(A)], [[] for _ in range(A)]
        done_count, oob_count, hid = np.zeros(A), np.zeros(A), np.ones(N)
        for t in range(T):
            obs_o[t] = cur
            src_o[t] = ob.envs["src"]
            last = t == T - 1
            ob.step(actions[epoch * T + t], env._ctr - (T - 1 - t))  # the Philox step counter the env used at that step
            e, o = ob.envs, ob.outs
            term, timeout = e["done"] == 1, e["ep_len"] == ML
            pe = term | timeout | last
            r = o["reward"][:, :A] if team_mode == "individual" else np.repeat(o["team_reward"][:, None], A, 1)
            rew_o[t] = r.astype(np.float32)
            end_o[t], cut_o[t] = pe, timeout | last
            ep_ret += rew_o[t].astype(np.float64)
            ep_len += 1
            over = term | timeout
            for a in range(A):
                rets[a] += list(ep_ret[over, a]); lens[a] += list(ep_len[over])
            done_count += (o["done"][:, :A] != 0).sum(0)
            oob_count += (e["oob"][:, :A] != 0).sum(0)
            ep_ret[pe] = 0.0; ep_len[pe] = 0
            if not last:
                hid = np.where(pe, 0.0, hid)
            if pe.any():
                ob.reset(mask=pe, new_obstacles=np.full(N, last))
            cur = ob.outs["obs"][:, :A].copy()
        NA = N * A
        pu.compare_obs(buf.obs_buf.cpu().numpy().reshape(T * N, A, 11), obs_o.reshape(T * N, A, 11))
        np.testing.assert_array_equal(buf.rew_buf.cpu().numpy(), rew_o.reshape(T, NA))
        np.testing.assert_array_equal(buf.end_buf.cpu().numpy() != 0, np.repeat(end_o, A, 1))
        np.testing.assert_array_equal(buf.act_buf.cpu().numpy(), actions[epoch * T:(epoch + 1) * T].reshape(T, NA))
        np.testing.assert_array_equal(buf.source_tar.cpu().numpy(), np.repeat(src_o, A, 1))
        obs_rows = buf.obs_buf.cpu().numpy()
        np.testing.assert_array_equal(buf.pred_buf.cpu().numpy(), obs_rows[:, :, 1:3] * np.float32(0.5) + np.float32(0.25))
        v_next = np.stack(pol.v_next).reshape(T, NA)
        np.testing.assert_array_equal(buf.boot_buf.cpu().numpy(), np.where(np.repeat(cut_o, A, 1), v_next, 0.0))
        np.testing.assert_array_equal(buf.logp_buf.cpu().numpy(), -0.5 * buf.val_buf.cpu().numpy())
        a0, r0 = co.gae(buf.rew_buf.cpu().numpy(), buf.val_buf.cpu().numpy(), np.repeat(end_o, A, 1).astype(np.uint8),
                        buf.boot_buf.cpu().numpy())
        np.testing.assert_array_equal(buf.adv_buf.cpu().numpy(), a0)
        np.testing.assert_array_equal(buf.ret_buf.cpu().numpy(), r0)
        np.testing.assert_array_equal(pol.hidden_state[:, 0].cpu().numpy(), np.repeat(hid, A))
        for a in range(A):                                            # per-agent views of the env-major columns
            v = buf.agent_view(a)
            np.testing.assert_array_equal(v["rew"].cpu().numpy(), rew_o[:, :, a])
        summ = {k: v.cpu().numpy() for k, v in stats.epoch_summary().items()}
        for a in range(A):
            assert int(summ["Episodes"][a]) == len(rets[a]) > 0
            np.testing.assert_allclose(summ["AverageEpRet"][a], np.mean(rets[a]), rtol=1e-9)
            np.testing.assert_allclose(summ["EpLen"][a], np.mean(lens[a]), rtol=1e-12)
            assert summ["MinEpRet"][a] == min(rets[a]) and summ["MaxEpRet"][a] == max(rets[a])
        np.testing.assert_array_equal(summ["DoneCount"], done_count)
        np.testing.assert_array_equal(summ["OutOfBound"], oob_count)

        # the live stacks of the sampled envs at every step and at the bootstrap call vs MapsOracle
        reset_rows = (buf.end_buf.cpu().numpy().reshape(T, N, A)[:, :, 0] & 4) != 0
        Wd = W.astype(np.float64)
        for t in range(T):
            (obs_s, pred_s), (act_a, act_c) = pol.pred_calls[2 * t], pol.act_snaps[t]
            (fin_s, fpred_s), (boot_a, boot_c) = pol.pred_calls[2 * t + 1], pol.boot_snaps[t]
            for j, n in enumerate(sample):
                o64 = lattice64(obs_s[j], env.scale)
                for i in range(A):
                    want = oracles[n][i].observation_to_map(o64, i, (float(pred_s[j, i, 0]), float(pred_s[j, i, 1])))
                    np.testing.assert_array_equal(stacks_to_seven(act_a[j], act_c[j], i), want, err_msg=f"env {n} step {t}")
                if reset_rows[t, n]:
                    o64 = lattice64(fin_s[j], env.scale)
                    for i in range(A):
                        want = oracles[n][i].observation_to_map(o64, i, (float(fpred_s[j, i, 0]), float(fpred_s[j, i, 1])))
                        np.testing.assert_array_equal(stacks_to_seven(boot_a[j], boot_c[j], i), want,
                                                      err_msg=f"bootstrap env {n} step {t}")
                    crit = np.stack([want[6], want[3], want[4], want[5]]).astype(np.float64)
                    v = np.tanh(0.01 * (crit * Wd).sum()) + 0.001 * np.arange(A)
                    np.testing.assert_allclose(pol.v_next[t][n], v, rtol=1e-5, atol=1e-5)
                    for b in oracles[n]:
                        b.reset()
        check_replay(mb, buf, pol, sample, T, rng)
        buf.get()
    assert int(mb.status.sum()) == 0 and int((env.status & ~2).sum()) == 0


class WalkDownLeft(Scripted):
    def __init__(self, maps, T, sample, W, seed):
        rng = np.random.default_rng(seed)
        N, A = maps.num_envs, maps.number_of_agents
        super().__init__(maps, rng.choice([0, 6, 7, 7], size=(T, N, A)).astype(np.int32), sample, W)

    def predict(self, obs):
        return (obs[..., 1:3] * 0.25 + 0.3).contiguous()              # inside the 147 x 147 map


def test_replay_unenforced_147_grid():
    """enforce_grid_boundaries=False (147 x 147 maps, wrapped negative cells, the configuration of
    test_maps_unenforced_boundaries_147_grid_and_status_flags): replay of whole episodes == the live stacks."""
    N, A, T = 256, 2, 60
    env = rp.RadSearch(obstruction_count=2, enforce_grid_boundaries=False, number_agents=A, num_envs=N, seed=3,
                       auto_reset=True)
    ra = mbm.calculate_resolution_accuracy(0.01, env.scale)
    offset = env.scale * (500.0 + 120 * 100.0)
    mb = rp.BatchedMapsBuffer(N, A, 120, resolution_accuracy=ra, offset=offset, environment_scale=env.scale)
    assert mb.map_dimensions == (147, 147)
    sample = np.arange(0, N, 32)
    pol = WalkDownLeft(mb, T, sample, np.ones((4, 147, 147), np.float32), seed=2)
    buf = rp.BatchedPPOBuffer(11, T, N, agents=A)
    rp.TeamRolloutCollector(env, buf, mb, pol).collect()
    assert bool((buf.obs_buf[..., 1:3] < 0).any())                     # some detectors crossed x < 0 / y < 0
    check_replay(mb, buf, pol, sample, T, np.random.default_rng(4))
    assert int(mb.status.sum()) == 0


def test_replay_bad_requests_are_flagged_not_faults():
    """Ranges outside the buffer get zero stacks and RS_MR_BAD_RANGE; an inverted range owns no rows and gets the bit;
    the valid ranges of the same launch are unaffected."""
    N, A, T, ML = 64, 2, 48, 24
    env = rp.RadSearch(obstruction_count=3, enforce_grid_boundaries=True, number_agents=A, num_envs=N, seed=21,
                       steps_per_episode=ML, auto_reset=True)
    mb = rp.BatchedMapsBuffer(N, A, ML, environment_scale=env.scale)
    X, Y = mb.map_dimensions
    pol = Scripted(mb, np.random.default_rng(0).integers(0, 8, size=(T, N, A)).astype(np.int32), np.arange(4),
                   np.ones((4, X, Y), np.float32))
    buf = rp.BatchedPPOBuffer(11, T, N, agents=A)
    rp.TeamRolloutCollector(env, buf, mb, pol).collect()
    req = [[0, 0, 5], [N, 0, 2], [-1, 1, 1], [3, -1, 2], [3, 40, T], [2, 5, 3], [1, 10, 20], [2, 30, 47]]
    good = [0, 6, 7]
    lens = [max(t1 - t0 + 1, 0) for _, t0, t1 in req]
    actor, critic, status = mb.replay(buf, torch.as_tensor(req, dtype=torch.int32))
    assert actor.shape[0] == sum(lens)
    st = status.cpu().numpy()
    assert [int(s) & rp._lib.MR_BAD_RANGE != 0 for s in st] == [i not in good for i in range(len(req))]
    a, c = actor.cpu().numpy(), critic.cpu().numpy()
    ga, gc, gs = mb.replay(buf, torch.as_tensor([req[i] for i in good], dtype=torch.int32))
    assert int(gs.abs().sum()) == 0
    ga, gc = ga.cpu().numpy(), gc.cpu().numpy()
    row0 = np.cumsum([0] + lens)
    g0 = np.cumsum([0] + [lens[i] for i in good])
    for i in range(len(req)):
        sl = slice(row0[i], row0[i] + lens[i])
        if i in good:
            k = good.index(i)
            np.testing.assert_array_equal(a[sl], ga[g0[k]:g0[k] + lens[i]])
            np.testing.assert_array_equal(c[sl], gc[g0[k]:g0[k] + lens[i]])
            assert float(np.abs(a[sl]).sum()) > 0
        else:
            assert not a[sl].any() and not c[sl].any()
    for j, (n, t0, t1) in enumerate([req[0], req[6], req[7]]):           # and equal to what the policy read
        if n in range(4):
            for t in range(t0, t1 + 1):
                k = good[j]
                np.testing.assert_array_equal(a[row0[k] + t - t0], pol.act_snaps[t][0][n])
