"""GPU parity tests (pytest -m gpu) of the GAE / returns / advantage-normalisation kernels and the PPOBuffer mirror."""
import numpy as np
import pytest
import torch

from oracle import c_oracle as co
from tests import parity_util as pu
from tests.test_gpu_ppo_edges import assert_within_f32_ulp, gae_float64

pytestmark = pytest.mark.gpu

import radiation_ppo_b200 as rp  # noqa: E402


def dev():
    return torch.device("cuda:0")


def run_gae(rew, val, end, boot, variant, stats=False):
    d = dev()
    s = torch.zeros(2, dtype=torch.float64, device=d) if stats else None
    adv, ret = rp.gae_advantages(torch.as_tensor(rew, device=d), torch.as_tensor(val, device=d),
                                 torch.as_tensor(end, device=d), torch.as_tensor(boot, device=d), stats=s, variant=variant)
    return adv.cpu().numpy(), ret.cpu().numpy(), (None if s is None else s.cpu().numpy())


@pytest.mark.parametrize("T,N", [(480, 1024), (96, 24), (480, 4099), (7, 3), (1, 1), (33, 9)])
def test_gae_thread_per_column_is_bit_exact(T, N):
    rew, val, end, boot = pu.synthetic_rollout(T, N, seed=T + N, max_ep=min(120, T))
    a0, r0 = co.gae(rew, val, end, boot)
    a1, r1, st = run_gae(rew, val, end, boot, variant=1, stats=True)
    np.testing.assert_array_equal(a1, a0)
    np.testing.assert_array_equal(r1, r0)
    np.testing.assert_allclose(st, [a0.astype(np.float64).sum(), (a0.astype(np.float64) ** 2).sum()], rtol=1e-12)


@pytest.mark.parametrize("variant", [7, 8, 10, 11, 12, 13, 14, 15])
@pytest.mark.parametrize("T,N", [(480, 1024), (96, 128), (481, 4096), (7, 256), (1, 128), (33, 384), (3, 128), (12, 128), (50, 1152)])
def test_gae_copy_engine_tiles_are_bit_exact(T, N, variant):
    """variants 7, 8, 10-15: the per-column recurrence fed by bulk-async or tensor-map tile copies (N % 128 == 0); same
    operation order as variant 1, hence bit-identical to the reference recurrence, incl. T not a multiple of the tile height."""
    rew, val, end, boot = pu.synthetic_rollout(T, N, seed=T + N, max_ep=min(120, T))
    a0, r0 = co.gae(rew, val, end, boot)
    a1, r1, st = run_gae(rew, val, end, boot, variant=variant, stats=True)
    np.testing.assert_array_equal(a1, a0)
    np.testing.assert_array_equal(r1, r0)
    np.testing.assert_allclose(st, [a0.astype(np.float64).sum(), (a0.astype(np.float64) ** 2).sum()], rtol=1e-12)


@pytest.mark.parametrize("T,N", [(480, 1024), (96, 24), (480, 1021), (7, 3), (1, 1), (33, 9), (1000, 64)])
def test_gae_warp_scan_within_tolerance(T, N):
    """fp32 outputs within one float32 ulp of the float64 recurrence (the scan re-associates the fp64 sums)."""
    rew, val, end, boot = pu.synthetic_rollout(T, N, seed=T * 3 + N, max_ep=min(120, T))
    a0, r0 = co.gae(rew, val, end, boot)
    a1, r1, st = run_gae(rew, val, end, boot, variant=2, stats=True)
    a64, r64 = gae_float64(rew, val, end, boot)
    assert_within_f32_ulp(a1, a64, "adv")
    assert_within_f32_ulp(r1, r64, "ret")
    assert (a1 != a0).mean() < 0.01          # in practice the fp32 roundings coincide almost everywhere
    a = a1.astype(np.float64)
    assert abs(st[0] - a.sum()) <= 1e-12 * np.abs(a).sum() and abs(st[1] - (a * a).sum()) <= 1e-12 * (a * a).sum()


def test_gae_golden_reference_ppobuffer():
    g = pu.load_golden("ref_gae")
    for variant in (1, 2):
        a, r, _ = run_gae(g["rew"], g["val"], g["end"], g["boot"], variant)
        if variant == 1:
            np.testing.assert_array_equal(a, g["adv"])
            np.testing.assert_array_equal(r, g["ret"])
        else:
            np.testing.assert_allclose(a, g["adv"], rtol=1e-5, atol=1e-6)
            np.testing.assert_allclose(r, g["ret"], rtol=1e-5, atol=1e-6)


def test_gae_full_size_properties():
    """Config 3 size (T=480, N=65536): linearity in the rewards and agreement of both variants; oracle on a slice."""
    T, N = 480, 65536
    d = dev()
    g = torch.Generator(device=d).manual_seed(1)
    rew = -0.5 * torch.rand(T, N, generator=g, device=d) * 1.5
    val = torch.randn(T, N, generator=g, device=d)
    end = (torch.rand(T, N, generator=g, device=d) < 1 / 90).to(torch.uint8)
    end[T - 1] = 1
    boot = torch.randn(T, N, generator=g, device=d) * end
    a1, r1 = rp.gae_advantages(rew, val, end, boot, variant=1)
    a2, r2 = rp.gae_advantages(rew, val, end, boot, variant=2)
    assert torch.allclose(a1, a2, rtol=1e-5, atol=1e-6) and torch.allclose(r1, r2, rtol=1e-5, atol=1e-6)
    # linearity: GAE(2*rew, 2*val, 2*boot) == 2*GAE(rew, val, boot) exactly (powers of two)
    a3, r3 = rp.gae_advantages(2 * rew, 2 * val, end, 2 * boot, variant=1)
    assert torch.equal(a3, 2 * a1) and torch.equal(r3, 2 * r1)
    sl = slice(1000, 1064)
    a0, r0 = co.gae(rew[:, sl].cpu().numpy(), val[:, sl].cpu().numpy(), end[:, sl].cpu().numpy(), boot[:, sl].cpu().numpy())
    np.testing.assert_array_equal(a1[:, sl].cpu().numpy(), a0)
    np.testing.assert_array_equal(r1[:, sl].cpu().numpy(), r0)


@pytest.mark.parametrize("offset", [0, 1, 3])
def test_advantage_normalisation_matches_reference_statistics(offset):
    """`offset`: a view that starts 4 / 12 bytes past a 16-byte boundary (the kernels read float4 behind a scalar head)."""
    d = dev()
    x = (torch.randn(480 * 1024 + 3 + offset, device=d) * 3 + 0.7)[offset:]
    assert x.data_ptr() % 16 == 4 * offset
    mean, std = rp.advantage_statistics(x)
    xs = x.cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(mean.item(), xs.mean(), rtol=1e-12)
    np.testing.assert_allclose(std.item(), xs.std(), rtol=1e-12)
    y = torch.empty(x.numel() + offset, device=d)[offset:]
    y.copy_(x)
    rp.normalize_advantages_(y, mean.float().double(), std.float().double())
    want = (x.cpu().numpy() - np.float32(xs.mean())) / np.float32(xs.std())        # float32 math as in P:446
    np.testing.assert_allclose(y.cpu().numpy(), want, rtol=2e-7, atol=1e-7)


# ---- the reference's own PPOBuffer unit tests (unit_tests/test_PPO.py), restated against the mirror -----------------
def manual_gae(gamma, lamb, rewards, values, last_val):          # unit_tests/test_PPO.py:156-191 (Helpers)
    n = len(rewards)
    adv = np.zeros(n + 1)
    last_adv, last_value = 0, last_val
    for t in reversed(range(n)):
        delta = rewards[t] + gamma * last_value - values[t]
        last_adv = delta + gamma * lamb * last_adv
        adv[t] = last_adv
        last_value = values[t]
    return adv[:-1]


def manual_rtg(rews, gamma):                                      # unit_tests/test_PPO.py:193-209
    out, acc = [], 0
    for r in reversed(rews):
        acc = r + acc * gamma
        out.insert(0, acc)
    return out


def test_ppobuffer_init_quick_reset_store():                      # unit_tests/test_PPO.py:300-453
    buf = rp.PPOBuffer(observation_dimension=11, max_size=2, max_episode_length=2, number_agents=2)
    buf.ptr = 1; buf.path_start_idx = 1; buf.episode_lengths_buffer.append(1)
    buf.quick_reset()
    assert buf.ptr == 0 and buf.path_start_idx == 0 and len(buf.episode_lengths_buffer) == 0
    obs = np.array([41.0, 0.42181818, 0.92181818, 0, 0, 0, 0, 0, 0, 0, 0], dtype=np.float32)
    src = np.array([788.0, 306.0])
    for i in range(2):
        buf.store(obs=obs, act=1, rew=-0.46, val=-0.26629042625427246, logp=-1.777620792388916, src=src,
                  full_observation={0: obs, 1: obs}, heatmap_stacks=None, terminal=False)
        assert buf.obs_buf.shape == (2, 11) and np.array_equal(buf.obs_buf[i], obs)
        assert buf.act_buf.shape == (2,) and buf.act_buf[i].item() == 1
        assert buf.rew_buf[i].item() == pytest.approx(-0.46) and buf.val_buf[i].item() == pytest.approx(-0.26629042625427246)
        assert buf.source_tar.shape == (2, 2) and np.array_equal(buf.source_tar[i], src)
        assert buf.logp_buf[i].item() == pytest.approx(-1.777620792388916) and buf.ptr == i + 1
    with pytest.raises(AssertionError):
        buf.store(obs=obs, act=1, rew=0, val=0, logp=0, src=src)
    buf.store_episode_length(7)
    assert buf.episode_lengths_buffer == [7]


def test_ppobuffer_gae_hardcoded_and_with_storage():              # unit_tests/test_PPO.py:462-571
    rewards = np.array([-0.46, -0.48, -0.46, -0.45, -0.45, -0.47, -0.48, -0.48, -0.48, -0.49])
    values = np.array([-0.26629043, -0.26634163, -0.26718464, -0.26631153, -0.26637784, -0.26601458, -0.26657045,
                       -0.2666973, -0.26680088, -0.26717135])
    last_val = -0.26717135
    buf = rp.PPOBuffer(observation_dimension=11, max_size=10, max_episode_length=2, number_agents=2)
    buf.rew_buf = rewards          # the reference test assigns numpy arrays straight into the fields
    buf.val_buf = values
    buf.ptr = 10
    buf.GAE_advantage_and_rewardsToGO(last_state_value=last_val)
    for want, got in zip(manual_rtg(np.append(rewards, last_val).tolist(), 0.99)[:-1], buf.ret_buf.tolist()):
        assert want == pytest.approx(got)
    for want, got in zip(manual_gae(0.99, 0.90, rewards, values, last_val), buf.adv_buf.tolist()):
        assert want == pytest.approx(got)
    assert buf.path_start_idx == 10
    buf = rp.PPOBuffer(observation_dimension=11, max_size=10, max_episode_length=2, number_agents=2)
    for i in range(3):
        buf.store(obs=np.zeros(11, np.float32), act=0, rew=rewards[i], val=values[i], logp=0, src=np.zeros((1, 2), np.float32))
    buf.GAE_advantage_and_rewardsToGO(last_state_value=values[2])
    for want, got in zip(manual_gae(0.99, 0.90, rewards[:3], values[:3], values[2]), buf.adv_buf.tolist()):
        assert want == pytest.approx(got)
    for want, got in zip(manual_rtg(np.append(rewards[:3], values[2]).tolist(), 0.99)[:-1], buf.ret_buf.tolist()):
        assert want == pytest.approx(got)


def test_ppobuffer_get_matches_reference_semantics():             # P:425-502, unit_tests/test_PPO.py:573-660
    rng = np.random.default_rng(0)
    T = 12
    buf = rp.PPOBuffer(observation_dimension=11, max_size=T, max_episode_length=5, number_agents=1)
    obs = rng.normal(size=(T, 11)).astype(np.float32)
    rew, val = rng.normal(size=T).astype(np.float32), rng.normal(size=T).astype(np.float32)
    for t in range(T):
        buf.store(obs=obs[t], act=t % 8, rew=rew[t], val=val[t], logp=-1.5, src=np.array([788.0, 306.0]))
        if t in (4, 9):
            buf.GAE_advantage_and_rewardsToGO(0.0)
            buf.store_episode_length(5)
    buf.GAE_advantage_and_rewardsToGO(float(val[-1]))
    adv_before = buf.adv_buf.copy()
    data = buf.get()
    assert buf.ptr == 0 and buf.path_start_idx == 0 and len(buf.episode_lengths_buffer) == 0
    assert set(data) == {"obs", "act", "ret", "adv", "logp", "loc_pred", "ep_len", "ep_form"}
    np.testing.assert_array_equal(data["obs"].cpu().numpy(), obs)
    np.testing.assert_array_equal(data["act"].cpu().numpy(), np.arange(T) % 8)
    want = (adv_before - np.float32(adv_before.astype(np.float64).mean())) / np.float32(adv_before.astype(np.float64).std())
    np.testing.assert_allclose(data["adv"].cpu().numpy(), want, rtol=1e-6, atol=1e-6)
    assert data["ep_len"].item() == 10 and len(data["ep_form"]) == 3
    assert [e[0].shape for e in data["ep_form"]] == [(5, 17), (5, 17), (2, 17)]


def test_batched_buffer_end_to_end_against_oracle():
    T, N = 64, 256
    rew, val, end, boot = pu.synthetic_rollout(T, N, seed=9, max_ep=30)
    d = dev()
    buf = rp.BatchedPPOBuffer(11, T, N)
    for t in range(T):
        buf.store_batch(torch.zeros(N, 11, device=d), torch.zeros(N, device=d), torch.as_tensor(rew[t], device=d),
                        torch.as_tensor(val[t], device=d), torch.zeros(N, device=d),
                        end=torch.as_tensor(end[t], device=d), boot=torch.as_tensor(boot[t], device=d))
    buf.finish_paths(variant=1)
    a0, r0 = co.gae(rew, val, end, boot)
    np.testing.assert_array_equal(buf.adv_buf.cpu().numpy(), a0)
    np.testing.assert_array_equal(buf.ret_buf.cpu().numpy(), r0)
    data = buf.get()
    m, s = a0.astype(np.float64).mean(), a0.astype(np.float64).std()
    np.testing.assert_allclose(data["adv"].cpu().numpy().reshape(T, N), (a0 - np.float32(m)) / np.float32(s), rtol=1e-6, atol=1e-6)
    assert data["obs"].shape == (T * N, 11) and buf.ptr == 0


def test_batched_buffer_second_epoch_without_bootstrap_rows_starts_clean():
    """store_batch with boot / end / src omitted must not inherit the previous epoch's rows (rs_gae reads boot[T-1]
    unconditionally): epoch 2, stored without boot, equals a fresh buffer fed the same data with boot = 0."""
    T, N = 32, 128
    d = dev()
    rew, val, end, boot = pu.synthetic_rollout(T, N, seed=4, max_ep=12)
    rew2, val2, _, _ = pu.synthetic_rollout(T, N, seed=5, max_ep=12)
    z = torch.zeros(N, device=d)
    buf = rp.BatchedPPOBuffer(11, T, N)
    for t in range(T):                                               # epoch 1: every optional row filled with non-zeros
        buf.store_batch(torch.zeros(N, 11, device=d), z, torch.as_tensor(rew[t], device=d), torch.as_tensor(val[t], device=d), z,
                        src=torch.ones(N, 2, device=d), end=torch.as_tensor(end[t], device=d),
                        boot=torch.as_tensor(boot[t], device=d) + 3.0)
    buf.finish_paths(variant=1)
    buf.get()
    for t in range(T):                                               # epoch 2: no boot / end / src
        buf.store_batch(torch.zeros(N, 11, device=d), z, torch.as_tensor(rew2[t], device=d), torch.as_tensor(val2[t], device=d), z)
    buf.finish_paths(variant=1)
    e0 = np.zeros((T, N), np.uint8); e0[-1] = 1
    a0, r0 = co.gae(rew2, val2, e0, np.zeros((T, N), np.float32))
    np.testing.assert_array_equal(buf.adv_buf.cpu().numpy(), a0)
    np.testing.assert_array_equal(buf.ret_buf.cpu().numpy(), r0)
    assert float(buf.source_tar.abs().sum()) == 0.0 and float(buf.boot_buf.abs().sum()) == 0.0


def test_batched_get_packs_the_reference_episode_tensors():
    """BatchedPPOBuffer.get(episodes=True) (rs_pack_rollout + rs_episode_table) against the `ep_form` tensors of the
    reference's PPOBuffer.get (P:425-502), one reference buffer per column (tests/golden/ref_get_epform.npz):
    row layout [obs | adv | ret | logp | act | source_tar], episode order and lengths, bit-exact (the advantage column is
    checked in the single-column buffers, where the reference's single-rank normalisation is the batched one)."""
    g = pu.load_golden("ref_get_epform")
    T, N, _ = g["obs"].shape
    d = dev()

    def fill(cols):
        buf = rp.BatchedPPOBuffer(11, T, len(cols))
        tt = lambda x: torch.as_tensor(np.ascontiguousarray(x), device=d)          # noqa: E731
        for t in range(T):
            buf.store_batch(tt(g["obs"][t, cols]), tt(g["act"][t, cols]), tt(g["rew"][t, cols]), tt(g["val"][t, cols]),
                            tt(g["logp"][t, cols]), src=tt(g["src"][t, cols]), end=tt(g["end"][t, cols]),
                            boot=tt(g["boot"][t, cols]))
        buf.finish_paths(variant=1)
        return buf

    data = fill(list(range(N))).get(episodes=True)
    packed = data["packed"].cpu().numpy().reshape(N, T, 17)
    np.testing.assert_array_equal(packed[:, :, :11], g["ep_rows"][:, :, :11])
    np.testing.assert_array_equal(packed[:, :, 12:], g["ep_rows"][:, :, 12:])
    es, el = data["ep_start"].cpu().numpy(), data["ep_len"].cpu().numpy()
    want_len = np.concatenate([g["ep_lens"][n][g["ep_lens"][n] > 0] for n in range(N)])
    want_start = np.concatenate([n * T + np.concatenate([[0], np.cumsum(g["ep_lens"][n][g["ep_lens"][n] > 0])[:-1]])
                                 for n in range(N)])
    np.testing.assert_array_equal(el, want_len)
    np.testing.assert_array_equal(es, want_start)
    for n in (0, 3):                                       # single column = the reference's single-rank buffer
        one = fill([n]).get(episodes=True)
        p1 = one["packed"].cpu().numpy()
        np.testing.assert_allclose(p1[:, 11], g["ep_rows"][n][:, 11], rtol=2e-6, atol=2e-6)
        np.testing.assert_array_equal(np.delete(p1, 11, axis=1), np.delete(g["ep_rows"][n], 11, axis=1))


def test_rollout_to_advantages_pipeline_matches_oracle():
    """BASELINE configs[2] as a parity case (scaled to what the oracle replays in seconds): a batched rollout with
    auto-reset feeds BatchedPPOBuffer.store_batch with the caller rules of train.py:446-491 (path end on terminal /
    timeout / epoch end; bootstrap V(last observation) unless terminal), then one rs_gae launch, the global advantage
    normalisation and the episode packing -- against the oracle env stepped the reference's way and the oracle GAE."""
    N, T, ML = 4096, 160, 40
    env = rp.RadSearch(obstruction_count=5, enforce_grid_boundaries=True, num_envs=N, seed=99, steps_per_episode=ML,
                       auto_reset=True, prefetch=True, use_cuda_graph=True)
    ob = co.OracleBatch(N, co.default_config(obstruction_count=5, enforce=1, max_ep_len=ML), seed=99)
    ob.reset()
    d = env.device
    buf = rp.BatchedPPOBuffer(11, T, N)
    rng = np.random.default_rng(5)
    w = torch.as_tensor(rng.normal(size=11).astype(np.float32), device=d)

    def value_fn(obs):                                   # a fixed "critic": any deterministic function of the observation
        x = obs.reshape(-1, 11).clone()
        x[:, 0] = torch.log1p(x[:, 0]) * 0.1
        return torch.tanh(x @ w)

    rew_o = np.zeros((T, N), np.float32); val_o = np.zeros((T, N), np.float32)
    end_o = np.zeros((T, N), np.uint8); boot_o = np.zeros((T, N), np.float32)
    obs = env.obs.clone()
    for t in range(T):
        acts = rng.integers(0, 8, size=(N, 1))
        val = value_fn(obs)
        val_o[t] = value_fn(torch.as_tensor(ob.outs["obs"][:, :1].astype(np.float32), device=d)).cpu().numpy()
        epoch_end = t == T - 1
        env.step_batch(torch.as_tensor(acts, dtype=torch.int32, device=d), epoch_end=epoch_end)
        ended = env.ended
        path_end = (ended & 4) != 0
        terminal = (ended & 1) != 0
        # bootstrap with V(last observation of the episode) unless the episode ended in a terminal state (train.py:462-487)
        boot = torch.where(path_end & ~terminal, value_fn(env.final_obs), torch.zeros(N, device=d))
        buf.store_batch(obs, torch.as_tensor(acts[:, 0], dtype=torch.float32, device=d), env.reward[:, 0], val,
                        torch.zeros(N, device=d), end=path_end, boot=boot)
        obs = env.obs.clone()
        # the oracle, the reference's way
        ob.step(acts, env._ctr)
        e = ob.envs
        term_o, timeout_o = e["done"] == 1, e["ep_len"] == ML
        pe = term_o | timeout_o | epoch_end
        rew_o[t] = ob.outs["reward"][:, 0].astype(np.float32)
        end_o[t] = pe
        fin = torch.as_tensor(ob.outs["obs"][:, :1].astype(np.float32), device=d)
        boot_o[t] = np.where(pe & ~term_o, value_fn(fin).cpu().numpy(), 0.0)
        if pe.any():
            ob.reset(mask=pe, new_obstacles=np.full(N, epoch_end))
    np.testing.assert_array_equal(buf.rew_buf.cpu().numpy(), rew_o)
    np.testing.assert_array_equal(buf.end_buf.cpu().numpy(), end_o)
    np.testing.assert_allclose(buf.val_buf.cpu().numpy(), val_o, rtol=1e-5, atol=1e-6)     # fp32 matmul on sensors within 1e-5
    np.testing.assert_allclose(buf.boot_buf.cpu().numpy(), boot_o, rtol=1e-5, atol=1e-6)
    buf.finish_paths()
    a0, r0 = co.gae(buf.rew_buf.cpu().numpy(), buf.val_buf.cpu().numpy(), end_o, buf.boot_buf.cpu().numpy())
    np.testing.assert_array_equal(buf.adv_buf.cpu().numpy(), a0)
    np.testing.assert_array_equal(buf.ret_buf.cpu().numpy(), r0)
    data = buf.get(episodes=True)
    es, el = data["ep_start"].cpu().numpy(), data["ep_len"].cpu().numpy()
    assert el.sum() == T * N and (el <= ML).all() and len(el) == int(end_o.sum())
    packed = data["packed"].cpu().numpy().reshape(N, T, 17)
    np.testing.assert_array_equal(packed[:, :, 12], r0.T)
    assert end_o.sum() > 4 * N


@pytest.mark.parametrize("mode", ["rows", "graph"])
def test_rollout_collector_zero_copy_epoch_matches_oracle(mode):
    """RolloutCollector (train.py:321-571 for a batched env): the step kernel stores observation t+1 / reward / path-end flags
    straight into the buffer rows (step_batch(out=); mode "graph": the captured step graph's fixed outputs are carried
    into the rows by the bookkeeping launches), rs_rollout_pre / rs_rollout_post do the caller-side bookkeeping --
    against the oracle env stepped the reference's way: every buffer row, the bootstrap rule (value of the next observation
    where the trajectory was cut by the timeout or the epoch's last step, else 0), the episode statistics, then GAE."""
    N, T, ML = 2048, 96, 24
    env = rp.RadSearch(obstruction_count=5, enforce_grid_boundaries=True, num_envs=N, seed=41, steps_per_episode=ML,
                       auto_reset=True, prefetch=True, use_cuda_graph=(mode == "graph"))
    ob = co.OracleBatch(N, co.default_config(obstruction_count=5, enforce=1, max_ep_len=ML), seed=41)
    ob.reset()
    d = env.device
    rng = np.random.default_rng(8)
    w = torch.as_tensor(rng.normal(size=11).astype(np.float32), device=d)
    actions = rng.integers(0, 8, size=(2 * T, N)).astype(np.int32)

    def value_fn(obs):
        x = obs.reshape(-1, 11).clone()
        x[:, 0] = torch.log1p(x[:, 0]) * 0.1
        return torch.tanh(x @ w)

    class Scripted:
        def __init__(self):
            self.t = 0
            self.acts = torch.as_tensor(actions, device=d)
            self.hidden_state = torch.ones(N, 3, device=d)            # restarted in place by rs_rollout_post
        def act(self, obs):
            a = self.acts[self.t]; self.t += 1
            v = value_fn(obs)
            return a, v, (-0.5 * v).contiguous()
        def value(self, obs):
            return value_fn(obs)
        def reset_state(self, mask):
            assert mask is None
            self.hidden_state.fill_(1.0)

    pol = Scripted()
    buf = rp.BatchedPPOBuffer(11, T, N)
    stats = rp.EpisodeStats(N, 1, d)
    col = rp.RolloutCollector(env, buf, pol, stats, mode=mode)
    ep_ret, ep_len = np.zeros(N), np.zeros(N, int)
    for epoch in range(2):
        first_obs = ob.outs["obs"][:, :1].astype(np.float32).copy()
        col.collect(gae_variant=1)
        obs_o = np.zeros((T, N, 11), np.float32); rew_o = np.zeros((T, N), np.float32)
        end_o = np.zeros((T, N), np.uint8); boot_o = np.zeros((T, N), np.float32); src_o = np.zeros((T, N, 2), np.float32)
        rets, lens, done_count, hid = [], [], 0, np.ones(N)
        cur = first_obs
        for t in range(T):
            obs_o[t] = cur[:, 0]
            src_o[t] = ob.envs["src"]
            acts = actions[epoch * T + t][:, None]
            last = t == T - 1
            ob.step(acts, env._ctr - (T - 1 - t))                 # the Philox step counter the env used at that step
            e = ob.envs
            term, timeout = e["done"] == 1, e["ep_len"] == ML
            pe = term | timeout | last
            rew_o[t] = ob.outs["reward"][:, 0].astype(np.float32)
            end_o[t] = pe
            fin = torch.as_tensor(ob.outs["obs"][:, :1].astype(np.float32), device=d)
            cut = np.full(N, True) if last else timeout
            boot_o[t] = np.where(cut, value_fn(fin).cpu().numpy(), 0.0)
            ep_ret += rew_o[t].astype(np.float64); ep_len += 1
            over = term | timeout
            rets += list(ep_ret[over]); lens += list(ep_len[over]); done_count += int(term.sum())
            ep_ret[pe] = 0.0; ep_len[pe] = 0
            if not last:
                hid = np.where(pe, 0.0, hid)
            if pe.any():
                ob.reset(mask=pe, new_obstacles=np.full(N, last))
            cur = ob.outs["obs"][:, :1].astype(np.float32).copy()
        pu.compare_obs(buf.obs_buf.cpu().numpy().reshape(T * N, 1, 11), obs_o.reshape(T * N, 1, 11))
        np.testing.assert_array_equal(buf.rew_buf.cpu().numpy(), rew_o)
        np.testing.assert_array_equal(buf.end_buf.cpu().numpy() != 0, end_o != 0)
        np.testing.assert_array_equal(buf.act_buf.cpu().numpy(), actions[epoch * T:(epoch + 1) * T].astype(np.float32))
        np.testing.assert_array_equal(buf.source_tar.cpu().numpy(), src_o)
        np.testing.assert_allclose(buf.boot_buf.cpu().numpy(), boot_o, rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(buf.logp_buf.cpu().numpy(), -0.5 * buf.val_buf.cpu().numpy(), rtol=0, atol=0)
        a0, r0 = co.gae(buf.rew_buf.cpu().numpy(), buf.val_buf.cpu().numpy(), (end_o != 0).astype(np.uint8), buf.boot_buf.cpu().numpy())
        np.testing.assert_array_equal(buf.adv_buf.cpu().numpy(), a0)
        np.testing.assert_array_equal(buf.ret_buf.cpu().numpy(), r0)
        np.testing.assert_array_equal(pol.hidden_state[:, 0].cpu().numpy(), hid)
        summ = stats.epoch_summary()
        assert int(summ["Episodes"][0]) == len(rets) and int(summ["DoneCount"][0]) == done_count
        np.testing.assert_allclose(float(summ["AverageEpRet"][0]), np.mean(rets), rtol=1e-9)
        np.testing.assert_allclose(float(summ["EpLen"][0]), np.mean(lens), rtol=1e-12)
        assert float(summ["MinEpRet"][0]) == min(rets) and float(summ["MaxEpRet"][0]) == max(rets)
        buf.get()
    assert int((env.status & ~2).sum()) == 0
