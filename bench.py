"""bench.py -- RadSearch env-steps/s (5 obstructions) on N B200s of one node, GAE GB/s, rooflines, the rollout pipeline,
and the CPU baselines.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--envs-per-gpu E] [--legs a,b,...]
                  [--dump-outputs DIR]
  torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" is one batched environment step of every env on every GPU: rs_step (move, obstruction collision, line of sight,
shortest path, expected counts, Philox + Poisson, 8 sensors, reward / terminal, caller rules) followed by rs_reset for the
envs that finished (auto-reset).  Headline workload = BASELINE.json configs[4]: 131,072 envs per GPU, 5 obstructions,
enforced boundaries, uniform random actions 0..7, episodes staggered so that ~1/120 of the envs reset at every step.
Weak scaling: envs shard independently over ranks, no data-path collective.

What the JSON line carries (rank 0 prints it):
  value / ms_per_step   device-resident env-steps/s over exactly K timed steps: one window bracketed by a barrier +
                        synchronize on both sides, its launches queued before its first kernel starts, timed with CUDA
                        events, MAX over ranks
  roofline              the step kernel alone against the HBM roofline (algorithmic bytes SURVEY.md 8d)
  exact_poisson         the same headline with the numpy-exact PTRS sampler instead of the KS-equivalent fast one
  sweep                 BASELINE configs[1] (1,024 envs, 1-5 obstructions) and configs[2]'s size (65,536 envs): per-launch
                        step-kernel time with L2 flushed in between, env-steps/s and roofline fraction
  gae                   rs_gae over [480, N] for N = 1,024 / 65,536 / 131,072: GB/s at 17 B per element vs the HBM peak
  pipeline              BASELINE configs[2]: 65,536 envs x T = 480, policy in the loop (stock PyTorch GRU(11 -> 24) + heads),
                        the step kernel storing straight into the rollout buffer, GAE, get(episodes=True), one PPO update;
                        with several ranks the section-8e collectives under NCCL, timed and checked
  maps                  BASELINE configs[3]: 16,384 envs x 4 agents, env step + map observation
  e2e                   the same metric through RadSearch.step_host with pinned HOST buffers, copies inside the timed region,
                        next to the measured ceiling of the device->host link
  cpu_baseline          the oracle's C port of the reference's per-env loop on the box's host cores (+ the reference's own
                        Python, timed in the build container, as secondary keys)

The inputs are seeded and the number of steps before and inside the timed window depends on the arguments only, so
`--dump-outputs DIR` (what the headline's last step handed its caller, see dump_outputs) can be compared between builds.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True                   # the benchmark runs from a built tree and leaves it as it found it

METRIC = "RadSearch env-steps/sec (5 obstructions)"
UNIT = "env-steps/s"
K_OBS = 5
BYTES_PER_ENV_STEP = 122 + 32 * K_OBS        # SURVEY.md 8(d): algorithmic bytes per env-step, single agent
GAE_BYTES_PER_ELEM = 17                      # SURVEY.md 8(d): rew 4 + val 4 + path_end 1 + adv 4 + ret 4
T_EPOCH = 480
PREROLL_STEPS = 20000                        # untimed steps before the timed window: ~0.6 s at 131,072 envs on a B200
GATE_CYCLES = 1000000                        # device sleep the timed window's launches queue behind: ~0.5 ms
DUMP_BYTES = 64 << 20                        # --dump-outputs writes at most this much
ALL_LEGS = ("exact", "sweep", "gae", "pipeline", "maps", "e2e", "cpu")


def measured_traffic(kernel: str, n_env: int):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture (profiles/)."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[kernel]
        if t.get("n_env", t.get("N")) == n_env:
            return t["dram_bytes_read"] + t["dram_bytes_write"]
    except Exception:
        pass
    return None


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


# ---------------------------------------------------------------------------------------------------------------------
# CPU arms
# ---------------------------------------------------------------------------------------------------------------------
def cpu_baseline(n_envs: int, T: int, threads: int):
    """The oracle's scalar per-env loop (reference semantics, OpenMP over envs) on the host cores."""
    from oracle import c_oracle as co

    ob = co.OracleBatch(n_envs, co.default_config(obstruction_count=K_OBS, enforce=1), seed=2, threads=threads)
    ob.reset()
    t0 = time.perf_counter()
    n, chk = ob.rollout(T, 1, epoch_end_last=False)
    dt = time.perf_counter() - t0
    return n / dt, dt, chk


def gae_lfilter_baseline(T: int, n_cols: int):
    """PPOBuffer.GAE_advantage_and_rewardsToGO's arithmetic (ppo.py:391-423: np.append, deltas, two scipy lfilter calls per
    trajectory, discount_cumsum ppo.py:62-85) over the columns of a [T, n_cols] rollout, one process."""
    import numpy as np
    from tests import parity_util as pu

    rew, val, end, boot = pu.synthetic_rollout(T, n_cols, seed=1, max_ep=120)
    t0 = time.perf_counter()
    pu.gae_numpy_reference(rew, val, end, boot)
    dt = time.perf_counter() - t0
    return GAE_BYTES_PER_ELEM * T * n_cols / dt / 1e9, dt


def reference_python_record():
    p = os.path.join(ROOT, "profiles", "r02_reference_python_baselines.json")
    try:
        d = json.load(open(p))
        d["kind"] = "reference-python, timed in the build container by tools/time_reference_python.py (not on this box)"
        return d
    except Exception:
        return None


def run_reference(args):
    """--impl reference: the CPU path (oracle port of the reference's per-env loop) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import c_oracle as co

    cores = os.cpu_count() or 1
    n = 16384                    # per step: enough envs per thread for the OpenMP loop to run at its best rate
    ob = co.OracleBatch(n, co.default_config(obstruction_count=K_OBS, enforce=1), seed=2, threads=cores)
    ob.reset()
    # one reference step = 16384 envs x `inner` steps: 8 (= 131072 env-steps, the GPU arm's units per step) unless the
    # requested number of steps would then run for more than ~90 s on these cores
    t0 = time.perf_counter()
    ob.rollout(2, 1, epoch_end_last=False)
    rate = 2 * n / (time.perf_counter() - t0)
    inner = int(max(1, min(8, rate * 90.0 / max(args.steps + args.warmup, 1) / n)))
    ctr = 3
    for _ in range(args.warmup):
        ob.rollout(inner, ctr, epoch_end_last=False); ctr += inner
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ob.rollout(inner, ctr, epoch_end_last=False); ctr += inner
    dt = time.perf_counter() - t0
    v = n * inner * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32+f64", "data": "synthetic",
            "config": {"workload": "RadSearch env step, 5 obstructions, enforced boundaries, random actions, auto-reset; "
                                   f"one step = {n} envs x {inner} steps = {n * inner} env-steps (the GPU arm's units per step)"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{n} envs x {inner * args.steps} steps, oracle/radsearch_oracle.c (scalar per-env loop, OpenMP)"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# GPU legs
# ---------------------------------------------------------------------------------------------------------------------
class Ctx:
    """What every leg needs: torch handles, rank info, helpers."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        import radiation_ppo_b200 as rp
        from radiation_ppo_b200 import _lib as L

        self.torch, self.dist, self.rp, self.L, self.args = torch, dist, rp, L, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device(f"cuda:{self.local_rank}"))
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device(f"cuda:{self.local_rank}")
        self.lib = L.load()
        self.peak, self.peak_src = measured_peak_gbs()
        self._flush = None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        t = self.torch.tensor(values, device=self.dev, dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()

    def flush_l2(self):
        """Write a buffer twice the size of L2 (126 MB): what ran before is out of the cache."""
        if self._flush is None:
            self._flush = self.torch.empty(256 << 20, dtype=self.torch.uint8, device=self.dev)
        self._flush.fill_(1)

    def event(self):
        return self.torch.cuda.Event(enable_timing=True)


def pick_period(K: int, episode_steps: int = 120) -> int:
    """Steps per prefetch block (= per CUDA-graph launch) for windows of K steps: the largest divisor of K up to 12 that
    leaves at least two blocks per window (K = 20 -> 10, 240 -> 12), so that a window is whole blocks."""
    cands = [p for p in range(1, 13) if K % p == 0 and 2 * p <= episode_steps]
    two = [p for p in cands if K // p >= 2]
    return max(two or cands or [4])


def make_ring(cx: Ctx, N: int, R: int, fast: bool, episode_steps: int, graph: bool = True, prefetch: bool = True,
              period: int = 0):
    torch, rp = cx.torch, cx.rp
    envs = []
    for r in range(R):
        e = rp.RadSearch(obstruction_count=K_OBS, enforce_grid_boundaries=True, num_envs=N, seed=2, device=cx.dev,
                         env_id_offset=(cx.rank * R + r) * N, auto_reset=True, fast_poisson=fast,
                         steps_per_episode=episode_steps, prefetch=prefetch, use_cuda_graph=graph and prefetch,
                         prefetch_period=period or None)
        # stagger the episodes: steady state of a training run (about 1/120 of the envs finish at every step)
        g = torch.Generator(device=cx.dev).manual_seed(1000 + cx.rank * R + r)
        e._meta.add_(torch.randint(0, min(episode_steps, 120), (N,), generator=g, device=cx.dev, dtype=torch.int32) << 16)
        torch.cuda.synchronize()
        e.capture_graphs()
        envs.append(e)
    return envs


def headline(cx: Ctx, envs, K: int, W: int, sample_clocks: bool):
    """Device-resident throughput of the ring of env batches over one timed window of K steps.  Batch r lives on its own
    stream, so that the short tail kernels of one batch (reset of finished envs) and the drain of its step kernel's last
    CTAs overlap the next batch's step kernel.  Whole blocks of PREFETCH_PERIOD steps are one CUDA-graph launch
    (RadSearch.step_block); a K that is not a multiple of the period runs step by step.  How many steps run before the
    timed window depends on K and W only, so the state the window leaves behind is the same from run to run."""
    torch = cx.torch
    R, N = len(envs), envs[0].num_envs
    P = envs[0].PREFETCH_PERIOD
    g = torch.Generator(device=cx.dev).manual_seed(7 + cx.rank)
    n_act = 8
    act_blocks = torch.randint(0, 8, (n_act, P, N, 1), generator=g, device=cx.dev, dtype=torch.int32)   # resident in HBM
    main = torch.cuda.current_stream(cx.dev)
    streams = [torch.cuda.Stream(device=cx.dev) for _ in range(R)] if R > 1 else [main]
    use_blocks = envs[0].use_cuda_graph and K % P == 0
    counter = [0]

    def window(k_steps):
        for st in streams:
            st.wait_stream(main)
        if use_blocks:
            for _ in range(k_steps // P):
                i = counter[0]; counter[0] += 1
                with torch.cuda.stream(streams[i % R]):
                    envs[i % R].step_block(act_blocks[i % n_act])
        else:
            for _ in range(k_steps):
                i = counter[0]; counter[0] += 1
                with torch.cuda.stream(streams[i % R]):
                    envs[i % R].step_batch(act_blocks[i % n_act, i % P], epoch_end=False)
        for st in streams:
            main.wait_stream(st)

    warm = -(-max(W, 3) // P) * P                        # warm-up: at least W steps, whole blocks
    window(warm)
    cx.barrier()
    sampler = ClockSampler(cx.local_rank)
    if sample_clocks and cx.rank == 0:
        sampler.start()
    # nvidia-smi samples every 100 ms: the same windows keep running (untimed) for PREROLL_STEPS steps in front of the timed
    # one, so that the clocks have settled and their samples are taken under this very load.  A step count, not a time:
    # the state at the end of the timed window must not depend on how fast the box ran.
    pre = 0
    while pre < PREROLL_STEPS:
        for _ in range(8):
            window(K)
            pre += K
        torch.cuda.synchronize()
    cx.barrier()
    # the window's launches queue up behind a short sleep on the main stream, so that its time is the GPU's for K steps
    # and not the host's launch latency after the barrier (~30 us on a B200, 5 % of a 20-step window at 131,072 envs)
    torch.cuda._sleep(GATE_CYCLES)
    e0, e1 = cx.event(), cx.event()
    e0.record()
    window(K)
    e1.record()
    cx.barrier()
    clocks = sampler.stop() if (sample_clocks and cx.rank == 0) else None
    ms = cx.max_over_ranks([e0.elapsed_time(e1)])[0]
    launches_per_step = (2 + 1.0 / P)
    return {"ms": ms, "warmup_steps": warm, "preroll_steps": pre,
            "value": N * cx.world * K / (ms / 1e3), "clocks": clocks, "launches": int(launches_per_step * K),
            "graph_launches": (K // P) if use_blocks else K,
            "mode": (f"one CUDA-graph launch per block of {P} steps" if use_blocks else "one CUDA-graph launch per step")
            if envs[0].use_cuda_graph else "stream launches"}


def dump_outputs(cx: Ctx, envs, out_dir: str):
    """Write what the headline's last step handed its caller: the six step outputs (obs, reward, team_reward, done_flags,
    info_flags, ended) of every env batch of the ring, each as DIR/<name>.npy in float32 with the batches concatenated
    along the env axis (row b * N + n = env n of batch b).  Above DUMP_BYTES in all, every array keeps the same fixed,
    seeded sample of rows, whose row numbers go to DIR/env_index.npy (float64)."""
    import numpy as np

    torch = cx.torch
    names = ("obs", "reward", "team_reward", "done_flags", "info_flags", "ended")
    arrays = {n: torch.cat([getattr(e, n) for e in envs]).float() for n in names}
    rows = len(envs) * envs[0].num_envs
    row_bytes = sum(a[0].numel() * 4 for a in arrays.values())
    budget = DUMP_BYTES - (64 << 10)                     # room for the .npy headers
    os.makedirs(out_dir, exist_ok=True)
    if rows * row_bytes > budget:
        idx = torch.randperm(rows, generator=torch.Generator().manual_seed(0))[:budget // (row_bytes + 8)].sort().values
        np.save(os.path.join(out_dir, "env_index.npy"), idx.double().numpy())
        arrays = {n: a[idx.to(a.device)] for n, a in arrays.items()}
    for n, a in arrays.items():
        np.save(os.path.join(out_dir, n + ".npy"), a.cpu().numpy())


def step_kernel_time(cx: Ctx, envs, groups: int, fast: bool):
    """CUDA events around the step kernel alone, on the stream it is launched on.  `back_to_back`: one launch per batch of
    the ring between an event pair (independent batches, same stream), time / launches; `single`: an event pair per
    launch (adds the event overhead of an otherwise empty stream)."""
    import ctypes as C

    torch, L, lib = cx.torch, cx.L, cx.lib
    R, N = len(envs), envs[0].num_envs
    g = torch.Generator(device=cx.dev).manual_seed(99 + cx.rank)
    acts = torch.randint(0, 8, (4, N, 1), generator=g, device=cx.dev, dtype=torch.int32)
    stream = C.c_void_p(torch.cuda.current_stream(cx.dev).cuda_stream)
    for e in envs:
        e._quiesce_prefetch()
    torch.cuda.synchronize()
    sflags = L.F_AUTO_RESET | L.F_DEVICE_CTR | (L.F_FAST_POISSON if fast else 0)     # DEVICE_CTR: no memset inside

    def launch_step(e, a, stream=stream):
        e._ctr += 1
        e._ctr_dev.fill_(e._ctr)
        e._reset_count.zero_()
        return lambda: L.check(lib.rs_step(
            C.byref(e._cfg), C.byref(e._st), C.c_void_p(a.data_ptr()), C.c_void_p(e.obs.data_ptr()),
            C.c_void_p(e.reward.data_ptr()), C.c_void_p(e.team_reward.data_ptr()), C.c_void_p(e.done_flags.data_ptr()),
            C.c_void_p(e.info_flags.data_ptr()), C.c_void_p(e.ended.data_ptr()), C.c_void_p(e.final_obs.data_ptr()), N,
            e.env_id_offset, e.seed, e._ctr, None, 0, sflags, stream), "rs_step")

    def launch_reset(e):
        L.check(lib.rs_reset(C.byref(e._cfg), C.byref(e._st), None, None, C.c_void_p(e.obs.data_ptr()), N,
                             e.env_id_offset, e.seed, e._ctr, None, 0, L.F_RESET_LIST | (L.F_FAST_POISSON if fast else 0),
                             stream), "rs_reset")
        e._ctr_dev_val = -1

    b2b, single = [], []
    for i in range(groups + 2):
        fns = [launch_step(e, acts[(i + j) % 4]) for j, e in enumerate(envs)]
        e0, e1 = cx.event(), cx.event()
        e0.record()
        for f in fns:
            f()
        e1.record()
        for e in envs:
            launch_reset(e)
        if i >= 2:
            b2b.append((e0, e1))
    for i in range(groups):
        e = envs[i % R]
        f = launch_step(e, acts[i % 4])
        e0, e1 = cx.event(), cx.event()
        e0.record()
        f()
        e1.record()
        launch_reset(e)
        single.append((e0, e1))
    # the same R launches, each on a stream of its own (how the block graphs run the ring's batches): what a launch costs
    # when the start and the tail of one launch overlap the others -- SM-time per launch rather than launch-to-drain time
    side = [torch.cuda.Stream(device=cx.dev) for _ in envs]
    conc = []
    for i in range(groups // 2 + 2):
        fns = []
        for j, e in enumerate(envs):
            fns.append(launch_step(e, acts[(i + j) % 4], C.c_void_p(side[j].cuda_stream)))
        torch.cuda.synchronize()
        e0, e1 = cx.event(), cx.event()
        e0.record()
        for sd in side:
            sd.wait_event(e0)
        done = []
        for sd, f in zip(side, fns):
            f()
            d = cx.event()
            d.record(sd)
            done.append(d)
        for d in done:
            torch.cuda.current_stream(cx.dev).wait_event(d)
        e1.record()
        for e in envs:
            launch_reset(e)
        if i >= 2:
            conc.append((e0, e1))
    for e in envs:
        e.prefetch_all()            # the raw calls above bypassed the prefetch bookkeeping: next episodes of every env again
    torch.cuda.synchronize()
    t_b2b = [a.elapsed_time(b) / R for a, b in b2b]
    t_single = [a.elapsed_time(b) for a, b in single]
    t_conc = [a.elapsed_time(b) / R for a, b in conc]
    return sum(t_b2b) / len(t_b2b), median(t_b2b), sum(t_single) / len(t_single), median(t_conc)


def sweep_leg(cx: Ctx, fast: bool):
    """Per-launch step-kernel time at the smaller BASELINE sizes, L2 flushed before every timed launch."""
    import ctypes as C

    torch, L, lib, rp = cx.torch, cx.L, cx.lib, cx.rp
    out = []
    for N, oc, label in ((1024, -1, "BASELINE configs[1]: 1,024 envs, 1-5 obstructions"),
                         (65536, K_OBS, "BASELINE configs[2] size: 65,536 envs, 5 obstructions")):
        e = rp.RadSearch(obstruction_count=oc, enforce_grid_boundaries=True, num_envs=N, seed=3, device=cx.dev,
                         auto_reset=True, fast_poisson=fast, steps_per_episode=120)
        g = torch.Generator(device=cx.dev).manual_seed(5)
        e._meta.add_(torch.randint(0, 120, (N,), generator=g, device=cx.dev, dtype=torch.int32) << 16)
        acts = torch.randint(0, 8, (4, N, 1), generator=g, device=cx.dev, dtype=torch.int32)
        for i in range(8):
            e.step_batch(acts[i % 4])
        stream = C.c_void_p(torch.cuda.current_stream(cx.dev).cuda_stream)
        flags = L.F_AUTO_RESET | (L.F_FAST_POISSON if fast else 0)
        evs = []
        for i in range(24):
            e._ctr += 1
            e._reset_count.zero_()
            cx.flush_l2()
            e0, e1 = cx.event(), cx.event()
            e0.record()
            L.check(lib.rs_step(C.byref(e._cfg), C.byref(e._st), C.c_void_p(acts[i % 4].data_ptr()), C.c_void_p(e.obs.data_ptr()),
                                C.c_void_p(e.reward.data_ptr()), C.c_void_p(e.team_reward.data_ptr()),
                                C.c_void_p(e.done_flags.data_ptr()), C.c_void_p(e.info_flags.data_ptr()),
                                C.c_void_p(e.ended.data_ptr()), C.c_void_p(e.final_obs.data_ptr()), N, e.env_id_offset,
                                e.seed, e._ctr, None, 0, flags | L.F_DEVICE_CTR * 0, stream), "rs_step")
            e1.record()
            L.check(lib.rs_reset(C.byref(e._cfg), C.byref(e._st), None, None, C.c_void_p(e.obs.data_ptr()), N,
                                 e.env_id_offset, e.seed, e._ctr, None, 0, L.F_RESET_LIST | (L.F_FAST_POISSON if fast else 0),
                                 stream), "rs_reset")
            evs.append((e0, e1))
        torch.cuda.synchronize()
        ms = median([a.elapsed_time(b) for a, b in evs[4:]])
        nbytes = int((122 * N + 32 * (e._meta & 0xFF).sum().item()))
        # rs_step with a host step counter clears the reset list with a 4-byte memset first: it is inside the event pair
        out.append({"workload": label, "n_envs": N, "kernel_ms": ms, "env_steps_per_s": N / (ms / 1e3),
                    "algorithmic_bytes_per_launch": nbytes, "achieved": nbytes / (ms / 1e3) / 1e9, "peak": cx.peak,
                    "unit": "GB/s", "frac": nbytes / (ms / 1e3) / 1e9 / cx.peak, "l2": "flushed before every timed launch",
                    "note": "latency-bound: fewer warps than the GPU holds" if N < 148 * 128 * 7 else ""})
        del e
    return out


def gae_leg(cx: Ctx, sizes):
    torch, rp = cx.torch, cx.rp
    out = []
    T = T_EPOCH
    g = torch.Generator(device=cx.dev).manual_seed(11)
    for N in sizes:
        rew = -0.5 * torch.rand(T, N, generator=g, device=cx.dev) * 1.5
        val = torch.randn(T, N, generator=g, device=cx.dev)
        end = (torch.rand(T, N, generator=g, device=cx.dev) < 1 / 100).to(torch.uint8)
        end[T - 1] = 1
        boot = torch.randn(T, N, generator=g, device=cx.dev) * end
        adv, ret = torch.empty_like(rew), torch.empty_like(rew)
        for _ in range(3):
            rp.gae_advantages(rew, val, end, boot, adv=adv, ret=ret, variant=0)
        evs = []
        for _ in range(12):
            cx.flush_l2()
            a, b = cx.event(), cx.event()
            a.record()
            rp.gae_advantages(rew, val, end, boot, adv=adv, ret=ret, variant=0)
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        ms = median([a.elapsed_time(b) for a, b in evs])
        gbs = GAE_BYTES_PER_ELEM * T * N / (ms / 1e3) / 1e9
        out.append({"T": T, "N": N, "ms": ms, "achieved": gbs, "peak": cx.peak, "unit": "GB/s", "frac": gbs / cx.peak,
                    "bytes_per_element": GAE_BYTES_PER_ELEM, "l2": "flushed before every timed launch",
                    "traffic": measured_traffic("gae_tile_kernel", N)})
        del rew, val, end, boot, adv, ret
    return out


class GruPolicy:
    """Stock PyTorch actor-critic for the pipeline leg: GRUCell(11 -> 24), a categorical head over the 8 moves and a value
    head (the shape of the reference's RAD-A2C core, algos/test_environment/core.py).  `act` / `value` run as captured CUDA
    graphs on static buffers; everything inside them is torch's own kernels (cuBLAS GEMMs, elementwise)."""

    def __init__(self, cx: Ctx, N: int, obs_dim: int = 11, hidden: int = 24, n_act: int = 8, final_obs=None, obs_in=None,
                 action_out=None):
        torch = cx.torch
        self.torch, self.N = torch, N
        torch.manual_seed(0)
        self.net = torch.nn.ModuleDict({"gru": torch.nn.GRUCell(obs_dim, hidden), "pi": torch.nn.Linear(hidden, n_act),
                                        "v": torch.nn.Linear(hidden, 1)}).to(cx.dev)
        self.h = torch.zeros(N, hidden, device=cx.dev)
        self.hidden_state = self.h                       # restarted in place by rs_rollout_post (RolloutCollector)
        # obs_in / action_out: the env's own observation and action buffers (graph mode: nothing is copied)
        self.obs_in = torch.zeros(N, obs_dim, device=cx.dev) if obs_in is None else obs_in
        self.final_obs = final_obs
        self.action = torch.zeros(N, dtype=torch.int32, device=cx.dev) if action_out is None else action_out
        self.val = torch.zeros(N, device=cx.dev)
        self.logp = torch.zeros(N, device=cx.dev)
        self.v_next = torch.zeros(N, device=cx.dev)
        self.g_act = self.g_val = None
        self._capture(cx)

    def _act_body(self):
        torch = self.torch
        with torch.no_grad():
            h = self.net["gru"](self.obs_in, self.h)
            self.h.copy_(h)
            logits = self.net["pi"](h)
            lp = torch.log_softmax(logits, dim=-1)
            # Gumbel-max sampling: stays on the device and inside the graph
            u = torch.rand_like(lp).clamp_(1e-10, 1.0)
            a = (lp - torch.log(-torch.log(u))).argmax(dim=-1)
            self.action.copy_(a)
            self.logp.copy_(lp.gather(1, a[:, None]).squeeze(1))
            self.val.copy_(self.net["v"](h).squeeze(1))

    def _val_body(self):
        torch = self.torch
        with torch.no_grad():
            h = self.net["gru"](self.final_obs, self.h)
            self.v_next.copy_(self.net["v"](h).squeeze(1))

    def _capture(self, cx):
        torch = self.torch
        s = torch.cuda.Stream(device=cx.dev)
        s.wait_stream(torch.cuda.current_stream(cx.dev))
        with torch.cuda.stream(s):
            for _ in range(3):
                self._act_body()
                self._val_body()
        torch.cuda.current_stream(cx.dev).wait_stream(s)
        torch.cuda.synchronize()
        self.g_act, self.g_val = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.g_act):
            self._act_body()
        with torch.cuda.graph(self.g_val):
            self._val_body()
        self.h.zero_()

    def act(self, obs):
        if obs.data_ptr() != self.obs_in.data_ptr():
            self.obs_in.copy_(obs)
        self.g_act.replay()
        return self.action, self.val, self.logp

    def value(self, obs):
        assert obs.data_ptr() == self.final_obs.data_ptr()
        self.g_val.replay()
        return self.v_next

    def reset_state(self, mask):
        if mask is None:
            self.h.zero_()
        else:
            self.h.masked_fill_(mask[:, None], 0.0)


def ppo_update(cx: Ctx, pol: GruPolicy, buf, data, opt, columns: int = 8192, chunk: int = 8192, clip: float = 0.2):
    """One PPO update on a minibatch of `columns` trajectories x T steps of the epoch's rollout (clipped policy loss + value
    loss, P:1150-1281 in spirit): the GRU is re-run over the T steps of those columns with its state restarted where a path
    ended, the gradients are averaged over ranks with ONE flattened all-reduce (dist.average_gradients = mpi_avg_grads),
    one Adam step.  Stock PyTorch, step by step: it is the consumer of the hot path, not part of it."""
    torch = cx.torch
    from radiation_ppo_b200 import dist as rdist

    T, N, D = buf.T, min(buf.N, columns), buf.D
    data = {k: (v.view(buf.T, buf.N, *v.shape[1:])[:, :N] if k in ("obs", "act", "adv", "ret", "logp") else v) for k, v in data.items()}
    data["end"] = data["end"][:, :N]
    obs = data["obs"]
    act = data["act"].long()
    adv, ret, logp_old = data["adv"], data["ret"], data["logp"]
    end = data["end"]
    opt.zero_grad(set_to_none=True)
    total = 0.0
    for c0 in range(0, N, chunk):
        sl = slice(c0, min(N, c0 + chunk))
        h = torch.zeros(sl.stop - sl.start, pol.h.shape[1], device=cx.dev)
        loss = 0.0
        for t in range(T):
            h = pol.net["gru"](obs[t, sl], h)
            lp = torch.log_softmax(pol.net["pi"](h), dim=-1).gather(1, act[t, sl, None]).squeeze(1)
            v = pol.net["v"](h).squeeze(1)
            ratio = torch.exp(lp - logp_old[t, sl])
            a = adv[t, sl]
            loss = loss - torch.minimum(ratio * a, torch.clamp(ratio, 1 - clip, 1 + clip) * a).sum() \
                + 0.5 * ((v - ret[t, sl]) ** 2).sum()
            h = h * (end[t, sl] == 0)[:, None]
        loss = loss / (T * N)
        loss.backward()
        total += float(loss.detach())
    t0 = cx.event(); t1 = cx.event()
    t0.record()
    rdist.average_gradients(pol.net.parameters())
    t1.record()
    opt.step()
    return total, (t0, t1)


def pipeline_leg(cx: Ctx, fast: bool, N: int = 65536, T: int = T_EPOCH, epochs: int = 2, do_update: bool = True,
                 mode: str = "graph"):
    """BASELINE configs[2]: rollout (policy -> env step storing into the buffer -> bootstrap) x T, GAE, get(episodes=True),
    one PPO update; train.py:321-571 with ppo.py:746 / 1150-1281 as the consumer."""
    torch, rp = cx.torch, cx.rp
    from radiation_ppo_b200 import dist as rdist

    env = rp.RadSearch(obstruction_count=K_OBS, enforce_grid_boundaries=True, num_envs=N, seed=4, device=cx.dev,
                       env_id_offset=cx.rank * N, auto_reset=True, fast_poisson=fast, steps_per_episode=120,
                       prefetch=True, use_cuda_graph=(mode == "graph"), standardize=1)
    buf = rp.BatchedPPOBuffer(11, T, N, device=cx.dev)
    if mode == "graph":
        pol = GruPolicy(cx, N, final_obs=env.final_obs.view(N, 11), obs_in=env.obs.view(N, 11),
                        action_out=env.action_buffer.view(N))
    else:
        pol = GruPolicy(cx, N, final_obs=env.final_obs.view(N, 11))
    if cx.world > 1:
        rdist.sync_params(pol.net)                                                   # train.py:250-256
    stats = rp.EpisodeStats(N, 1, cx.dev)
    col = rp.RolloutCollector(env, buf, pol, stats, mode=mode)
    opt = torch.optim.Adam(pol.net.parameters(), lr=3e-4)
    rec = []
    for ep in range(epochs):
        cx.barrier()
        ev = [cx.event() for _ in range(6)]
        ev[0].record()
        col.collect()                                     # T steps + rs_gae
        ev[1].record()
        data = buf.get(episodes=True)                     # adv statistics (2 all-reduces) + normalise + pack + episode table
        ev[2].record()
        summ = stats.epoch_summary()                      # episode statistics: one sum + one min + one max all-reduce
        ev[3].record()
        loss, (g0, g1) = ppo_update(cx, pol, buf, data, opt) if do_update else (0.0, (ev[3], ev[3]))
        ev[4].record()
        cx.barrier()
        ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(4)]
        rec.append({"rollout_gae_ms": ms[0], "get_ms": ms[1], "episode_stats_ms": ms[2], "update_ms": ms[3],
                    "grad_allreduce_us": 1e3 * g0.elapsed_time(g1), "loss": loss,
                    "episodes": float(summ["Episodes"][0]), "avg_ep_ret": float(summ["AverageEpRet"][0]),
                    "n_episodes_packed": int(data["ep_len"].numel())})
        del data                                          # the epoch's packed rows go back to the allocator before the next epoch
    # where a rollout step's GPU time goes: each stage between its own event pair, median over 24 steps (one stage at a time,
    # so the pieces do not overlap; the loop above runs them back to back)
    stage_us = {}
    if True:
        import ctypes as C
        L_, lib_ = cx.L, cx.lib
        stream = C.c_void_p(torch.cuda.current_stream(cx.dev).cuda_stream)
        pp = lambda t: None if t is None else C.c_void_p(t.data_ptr())      # noqa: E731
        rows, outs = buf.policy_rows(0), buf.step_outputs(0)
        env_obs, fin = env.obs.view(N, 11), env.final_obs.view(N, 11)

        def timed(fn, n=24):
            ts = []
            for _ in range(n):
                torch.cuda.synchronize()
                a, b = cx.event(), cx.event()
                a.record(); fn(); b.record()
                torch.cuda.synchronize()
                ts.append(1e3 * a.elapsed_time(b))
            return median(ts)

        stage_us["policy_act_us"] = timed(lambda: pol.act(env_obs if mode == "graph" else rows["obs"]))
        stage_us["policy_value_us"] = timed(lambda: pol.value(fin))
        stage_us["env_step_reset_us"] = timed(lambda: env.step_batch(pol.action))
        stage_us["bookkeeping_pre_post_us"] = timed(lambda: (
            L_.check(lib_.rs_rollout_pre(pp(pol.action), pp(pol.val), pp(pol.logp), pp(env._src), pp(rows["act"]), pp(rows["val"]),
                                         pp(rows["logp"]), pp(rows["src"]), pp(env.obs), pp(rows["obs"]), 11, N, stream), "pre"),
            L_.check(lib_.rs_rollout_post(pp(env.reward), pp(env.ended), pp(env.done_flags), pp(env.info_flags), pp(pol.v_next),
                                          pp(rows["boot"]), pp(pol.h), 24, None, None, None, None, None, pp(outs["reward"]),
                                          pp(outs["ended"]), N, 0, stream), "post")))
        stage_us["note"] = ("GPU time per stage of one rollout step; the policy is stock PyTorch (GRUCell + heads + Gumbel-max "
                            "sampling, replayed as CUDA graphs) and sets the pace of the rollout, not the env step")
    r = rec[-1]
    tot = cx.max_over_ranks([r["rollout_gae_ms"], r["rollout_gae_ms"] + r["get_ms"] + r["episode_stats_ms"] + r["update_ms"]])
    how = ("step kernel stores into the rollout buffer rows (no copies, stream launches)" if mode == "rows" else
           "captured step graph, rs_rollout_pre / rs_rollout_post carry its outputs into the buffer rows")
    out = {"mode": mode, "workload": f"{N} envs/GPU x T={T}, 5 obstructions, GRU(11->24) policy in the loop, count standardiser fused in the "
                       f"step kernel, {how}, GAE, get(episodes=True), "
                       "1 PPO update (one Adam step on a minibatch of 8,192 trajectories x 480 steps) (BASELINE configs[2])",
           "rollout_env_steps_per_s": N * cx.world * T / (tot[0] / 1e3),
           "pipeline_env_steps_per_s": N * cx.world * T / (tot[1] / 1e3),
           "us_per_rollout_step": 1e3 * r["rollout_gae_ms"] / T, "rollout_step_stages_us": stage_us, "stages_ms": r,
           "epochs_run": epochs,
           "status_flags_raised": int((env.status & ~2).ne(0).sum().item())}
    # ---- SURVEY 8e collectives on their own: timed over 20 calls each, results asserted -----------------------------------
    if cx.world > 1:
        dist = cx.dist
        params = [p for p in pol.net.parameters()]
        for p in params:
            p.grad = torch.full_like(p, float(cx.rank + 1))
        times = {}

        def timeit(name, fn):
            fn()
            torch.cuda.synchronize()
            ts = []
            for _ in range(20):
                cx.barrier()
                a, b = cx.event(), cx.event()
                a.record(); fn(); b.record()
                torch.cuda.synchronize()
                ts.append(1e3 * a.elapsed_time(b))
            times[name] = median(cx.max_over_ranks(ts))

        def grads():
            for p in params:
                p.grad.fill_(float(cx.rank + 1))
            rdist.average_gradients(params)
        timeit("average_gradients_us", grads)
        want = sum(range(1, cx.world + 1)) / cx.world
        assert all(torch.allclose(p.grad, torch.full_like(p.grad, want)) for p in params), "average_gradients is wrong"
        adv = buf.adv_buf
        timeit("advantage_statistics_us", lambda: rp.advantage_statistics(adv))
        mean, std = rp.advantage_statistics(adv)
        gathered = [torch.zeros(2, dtype=torch.float64, device=cx.dev) for _ in range(cx.world)]
        a64 = adv.double()
        dist.all_gather(gathered, torch.stack([a64.sum(), (a64 * a64).sum()]))
        s1 = sum(float(g[0]) for g in gathered); s2 = sum(float(g[1]) for g in gathered); n = adv.numel() * cx.world
        assert abs(float(mean) - s1 / n) < 1e-9 and abs(float(std) - (s2 / n - (s1 / n) ** 2) ** 0.5) < 1e-6, "advantage_statistics is wrong"
        st = {"a": torch.tensor(float(cx.rank), device=cx.dev), "b": torch.tensor(2.0, device=cx.dev)}
        timeit("reduce_episode_stats_us", lambda: rdist.reduce_episode_stats(st))
        red = rdist.reduce_episode_stats(st)
        assert float(red["a"]) == sum(range(cx.world)) and float(red["b"]) == 2.0 * cx.world, "reduce_episode_stats is wrong"
        timeit("sync_params_us", lambda: rdist.sync_params(pol.net))
        times["flat_gradient_bytes"] = int(sum(p.numel() for p in params) * 4)
        times["backend"] = "nccl"
        times["checked"] = True
        out["collectives_us"] = times
    del env, buf, pol, col
    torch.cuda.empty_cache()
    if mode == "graph" and cx.world == 1:
        # the zero-copy variant of the same rollout (rs_step stores into the buffer rows; plain stream launches)
        env = rp.RadSearch(obstruction_count=K_OBS, enforce_grid_boundaries=True, num_envs=N, seed=4, device=cx.dev,
                           auto_reset=True, fast_poisson=fast, steps_per_episode=120, prefetch=True, standardize=1)
        buf = rp.BatchedPPOBuffer(11, T, N, device=cx.dev)
        pol = GruPolicy(cx, N, final_obs=env.final_obs.view(N, 11))
        col = rp.RolloutCollector(env, buf, pol, rp.EpisodeStats(N, 1, cx.dev), mode="rows")
        ms = []
        for ep in range(2):
            torch.cuda.synchronize()
            a, b = cx.event(), cx.event()
            a.record(); col.collect(); b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
            buf.get()
        out["rows_mode"] = {"rollout_env_steps_per_s": N * T / (ms[-1] / 1e3), "us_per_rollout_step": 1e3 * ms[-1] / T,
                            "how": "rs_step stores observation / reward / path-end flags straight into the buffer rows"}
        del env, buf, pol, col
    return out


def maps_leg(cx: Ctx, fast: bool):
    """RAD-TEAM pipeline of BASELINE configs[3]: 16,384 envs x 4 agents, env step -> shared map observation."""
    torch, rp = cx.torch, cx.rp
    Nm, Am, Tm = 16384, 4, 120
    g = torch.Generator(device=cx.dev).manual_seed(21)
    menv = rp.RadSearch(obstruction_count=K_OBS, enforce_grid_boundaries=True, number_agents=Am, num_envs=Nm, seed=4,
                        device=cx.dev, auto_reset=True, fast_poisson=fast, prefetch=True, use_cuda_graph=True)
    mb = rp.BatchedMapsBuffer(Nm, Am, 120, environment_scale=menv.scale, device=cx.dev)
    macts = torch.randint(0, 8, (8, Nm, Am), generator=g, device=cx.dev, dtype=torch.int32)
    mpred = torch.rand(Nm, Am, 2, generator=g, device=cx.dev)

    def maps_step(i):
        mb.update(menv.obs, mpred)
        menv.step_batch(macts[i % 8])
        mb.reset(mask=menv.ended, mask_bits=4)

    for i in range(24):
        maps_step(i)
    torch.cuda.synchronize()
    mev = []
    p0, p1 = cx.event(), cx.event()
    p0.record()
    for i in range(Tm):
        a, b = cx.event(), cx.event()
        a.record()
        mb.update(menv.obs, mpred)
        b.record()
        menv.step_batch(macts[i % 8])
        mb.reset(mask=menv.ended, mask_bits=4)
        mev.append((a, b))
    p1.record()
    torch.cuda.synchronize()
    upd_ms = median([a.elapsed_time(b) for a, b in mev])
    # algorithmic bytes of one rs_maps_update call (DESIGN.md section 3): per env 44 A obs + the episode's sample table scan
    # (6 B per logged reading, (T/2 + 1) A on average) + 4 B x (6 A + 6) A scattered map stores
    alg = Nm * (44 * Am + 6 * (Tm // 2 + 1) * Am + 4 * (6 * Am + 6) * Am)
    traffic = measured_traffic("maps_update_kernel", Nm)
    line = {"workload": f"{Nm} envs x {Am} agents, 27x27 maps, env step + rs_maps_update + rs_maps_reset (BASELINE configs[3])",
            "update_ms": upd_ms, "agent_map_updates_per_s": Nm * Am / (upd_ms / 1e3),
            "pipeline_env_steps_per_s": Nm * Tm / (p0.elapsed_time(p1) / 1e3),
            "maps_status_flags": int(mb.status.sum().item()),
            "roofline": {"bound": "hbm", "kernel": "maps_update_kernel", "algorithmic_bytes_per_launch": alg,
                         "achieved": alg / (upd_ms / 1e3) / 1e9, "peak": cx.peak, "unit": "GB/s",
                         "frac": alg / (upd_ms / 1e3) / 1e9 / cx.peak, "traffic": traffic,
                         "traffic_over_algorithmic": (traffic / alg) if traffic else None}}
    del menv, mb
    return line


def e2e_leg(cx: Ctx, envs, K: int, W: int):
    """End to end through the public API with HOST buffers (pinned), copies inside the timed region.
    RadSearch.step_host: pinned host actions -> device, step + auto-reset, ALL step outputs -> pinned host in one transfer,
    on the env batch's own stream.  `pipelined`: the R env batches of the ring are driven round-robin, the host waiting for
    batch r's previous results before it sends batch r's next actions; `sync`: one batch at a time, host waits every step.
    link: a bare pinned cudaMemcpyAsync device->host of the same bytes per rank, all ranks at once -- the ceiling of this
    host's link for that transfer."""
    torch = cx.torch
    R, N = len(envs), envs[0].num_envs
    n_act = 8
    h_act = torch.randint(0, 8, (n_act, N, 1), dtype=torch.int32).pin_memory()
    hbs = [e.host_buffers() for e in envs]
    torch.cuda.synchronize()
    Ke = min(max(K, 40), 480)

    def run(k0, k1, depth_all):
        chk = 0
        for i in range(k0, k1):
            r = i % R
            hb = hbs[r]
            if depth_all:
                hb.wait()                                      # results of this batch's previous step are on the host
            envs[r].step_host(hb, actions=h_act[i % n_act])
            if not depth_all:
                hb.wait()
            chk += int(hb.ended[0])                            # the host touches the results
        for hb in hbs:
            hb.wait()
        return chk

    vals = {}
    for name, depth_all in (("sync", False), ("pipelined", True)):
        run(0, max(W, 8), depth_all)
        ts = []
        for rep in range(5):
            cx.barrier()
            t0 = time.perf_counter()
            run(W, W + Ke, depth_all)
            cx.barrier()
            ts.append(time.perf_counter() - t0)
        ts = cx.max_over_ranks(ts)
        vals[name] = N * cx.world * Ke / median(ts)
    # the link: the same number of bytes, device -> pinned host, nothing else running, all ranks concurrently
    nbytes = hbs[0].d2h_bytes
    src = torch.empty(nbytes, dtype=torch.uint8, device=cx.dev)
    dst = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    for _ in range(3):
        dst.copy_(src, non_blocking=True)
    ts = []
    for rep in range(5):
        cx.barrier()
        t0 = time.perf_counter()
        for _ in range(50):
            dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        cx.barrier()
        ts.append((time.perf_counter() - t0) / 50)
    t_copy = median(cx.max_over_ranks(ts))
    link_gbs = nbytes * cx.world / t_copy / 1e9
    mode = "pipelined" if vals["pipelined"] >= vals["sync"] else "sync"
    e2e_value = vals[mode]
    per_env = (hbs[0].d2h_bytes + hbs[0].h2d_bytes) / N
    return {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": hbs[0].h2d_bytes, "d2h_bytes_per_step": hbs[0].d2h_bytes,
            "steps": Ke, "schedule": mode + " (the faster of the two schedules measured)", "sync_value": vals["sync"],
            "pipelined_value": vals["pipelined"], "reps": 5,
            "link_gbs": link_gbs, "link_env_steps_per_s": N * cx.world / t_copy,
            "frac_of_link": e2e_value / (N * cx.world / t_copy),
            "note": f"RadSearch.step_host: pinned host actions -> device, step+reset, all outputs (obs, reward, done/info/ended "
                    f"flags; {per_env:.0f} B per env both ways) -> pinned host in one copy; link_gbs = bare pinned "
                    f"cudaMemcpyAsync device->host of the same {nbytes} bytes per rank, all ranks concurrently (aggregate); "
                    "frac_of_link = value / (envs per copy / copy time)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=240)
    ap.add_argument("--warmup", type=int, default=24)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=131072)
    ap.add_argument("--ring", type=int, default=4, help="env batches cycled so that each step's state comes from HBM")
    ap.add_argument("--exact-poisson", action="store_true", help="fp64 numpy-exact PTRS acceptance as the headline sampler")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="headline + step-kernel timing only (what the ncu passes replay)")
    ap.add_argument("--legs", default=",".join(ALL_LEGS), help="comma list of " + ",".join(ALL_LEGS))
    ap.add_argument("--no-prefetch", action="store_true", help="synchronous reset kernel after every step")
    ap.add_argument("--no-graph", action="store_true", help="plain stream launches instead of CUDA-graph replay")
    ap.add_argument("--episode-steps", type=int, default=120, help="steps_per_episode (120 = the reference's; a huge value "
                    "shows the throughput without resets)")
    ap.add_argument("--period", type=int, default=0, help="steps per prefetch block / graph launch (0 = pick_period(steps))")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write rank 0's step outputs of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    legs = set() if args.quick else {x for x in args.legs.split(",") if x}
    if args.no_cpu_baseline:
        legs.discard("cpu")

    cx = Ctx(args)
    torch = cx.torch
    N, K, W, R = args.envs_per_gpu, args.steps, max(args.warmup, 3), max(args.ring, 1)
    fast = not args.exact_poisson
    graph, prefetch = not (args.no_graph or args.no_prefetch), not args.no_prefetch

    period = args.period or pick_period(K, args.episode_steps)
    envs = make_ring(cx, N, R, fast, args.episode_steps, graph, prefetch, period)
    head = headline(cx, envs, K, W, sample_clocks=True)
    if args.dump_outputs and cx.rank == 0:
        dump_outputs(cx, envs, args.dump_outputs)
    k_mean, k_med, k_single, k_conc = step_kernel_time(cx, envs, 120, fast)
    achieved = BYTES_PER_ENV_STEP * N / (k_mean / 1e3) / 1e9
    state_mb = R * N * (BYTES_PER_ENV_STEP + 160 + 80 + 80) / 1e6
    status = int(sum(int((e.status & ~2).any()) for e in envs))

    if args.quick:
        if cx.rank == 0:
            print(json.dumps({"quick": True, "value": head["value"], "ms_per_step": head["ms"] / K, "kernel_ms": k_mean,
                              "kernel_ms_single_launch": k_single, "kernel_ms_concurrent": k_conc,
                              "frac": achieved / cx.peak}), flush=True)
        if cx.world > 1:
            cx.dist.destroy_process_group()
        return

    line = {
        "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": cx.world, "steps": K, "warmup": W,
        "ms_per_step": head["ms"] / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32+f64", "data": "synthetic",
        "timing": {"timed_steps": K, "window_ms": head["ms"], "warmup_steps": head["warmup_steps"],
                   "preroll_steps": head["preroll_steps"],
                   "rule": "one K-step window after the warm-up and pre-roll steps, bracketed by barrier + synchronize, "
                           "launches queued behind a device sleep before the start event, CUDA events, max over ranks"},
        "config": {"workload": f"RadSearch env step + auto-reset, {N} envs/GPU (BASELINE configs[4]), 5 obstructions, "
                               f"enforced boundaries, 1 agent, uniform random actions, staggered {args.episode_steps}-step episodes",
                   "envs_per_gpu": N, "obstructions": K_OBS,
                   "poisson": ("alias table for blocked lines of sight + fp32-acceptance PTRS (KS-equivalent to numpy)" if fast
                               else "numpy-exact PTRS"),
                   "l2": f"ring of {R} env batches ({state_mb:.0f} MB of state) cycled: every step reads its state from HBM",
                   "resets": ("next episodes prefetched by rs_prepare on a parallel graph branch / side stream"
                              if prefetch else "synchronous rs_reset after every step"),
                   "launch": head["mode"] + f", ring batches on {R} stream(s)",
                   "parallelism": f"env-sharded x{cx.world}, no data-path collective"},
        "roofline": {"bound": "hbm", "kernel": "step1_kernel", "achieved": achieved, "peak": cx.peak, "unit": "GB/s",
                     "frac": achieved / cx.peak, "traffic": measured_traffic("step1_kernel", N), "peak_source": cx.peak_src,
                     "algorithmic_bytes_per_launch": BYTES_PER_ENV_STEP * N,
                     "algorithmic_bytes_per_env_step": BYTES_PER_ENV_STEP, "kernel_ms": k_mean, "kernel_ms_median": k_med,
                     "kernel_ms_single_launch": k_single,
                     "kernel_ms_rule": f"CUDA events around {R} back-to-back launches (one per ring batch, same stream) / {R}, "
                                       "mean over 120 groups; single_launch = an event pair around every launch",
                     "kernel_env_steps_per_s": N / (k_mean / 1e3),
                     "kernel_ms_concurrent": k_conc,
                     "frac_concurrent": BYTES_PER_ENV_STEP * N / (k_conc / 1e3) / 1e9 / cx.peak,
                     "concurrent_rule": f"the same {R} launches, one stream each, between one event pair / {R} (median): "
                                        "SM-time per launch when launches overlap, as in the block graphs; `frac` stays the "
                                        "same-stream figure"},
        "gpu_launches": head["launches"], "graph_launches": head["graph_launches"], "clocks": head["clocks"],
        "status_flags_raised": status,
    }
    if "e2e" in legs:
        line["e2e"] = e2e_leg(cx, envs, K, W)
    if "exact" in legs and fast:
        for e in envs:
            e._quiesce_prefetch()
        envs_x = make_ring(cx, N, 2, False, args.episode_steps, graph, prefetch)
        hx = headline(cx, envs_x, K, W, sample_clocks=False)
        kx_mean, _, kx_single, _ = step_kernel_time(cx, envs_x, 40, False)
        line["exact_poisson"] = {"value": hx["value"], "ms_per_step": hx["ms"] / K, "kernel_ms": kx_mean,
                                 "frac": BYTES_PER_ENV_STEP * N / (kx_mean / 1e3) / 1e9 / cx.peak,
                                 "sampler": "numpy-exact PTRS (bit-identical counts to the oracle on the shared Philox stream)",
                                 "ring": 2}
        line["exact_poisson_value"] = hx["value"]
        del envs_x
    del envs
    torch.cuda.empty_cache()
    if "sweep" in legs and cx.world == 1:
        line["sweep"] = sweep_leg(cx, fast)
    if "gae" in legs:
        gl = gae_leg(cx, (1024, 65536, 131072) if cx.world == 1 else (131072,))
        line["gae"] = dict(gl[-1])
        line["gae"]["kernel"] = "rs_gae variant 0 (bulk-async tiles, per-column fp64 recurrence; warp-scan form for small N)"
        line["gae"]["sizes"] = gl
    if "pipeline" in legs:
        line["pipeline"] = pipeline_leg(cx, fast)
    if "maps" in legs and cx.world == 1:
        line["maps"] = maps_leg(cx, fast)
    if cx.rank == 0:
        if "cpu" in legs and cx.world == 1:
            cores = os.cpu_count() or 1
            import numpy as np
            from oracle import c_oracle as co
            Tg, Ng = T_EPOCH, 16384
            rg = np.random.default_rng(0)
            c_rew = (-0.5 * rg.uniform(0, 1.5, (Tg, Ng))).astype(np.float32)
            c_val = rg.normal(size=(Tg, Ng)).astype(np.float32)
            c_end = (rg.random((Tg, Ng)) < 0.01).astype(np.uint8); c_end[-1] = 1
            c_boot = (rg.normal(size=(Tg, Ng)) * c_end).astype(np.float32)
            co.gae(c_rew, c_val, c_end, c_boot, threads=cores)
            t0 = time.perf_counter()
            for _ in range(3):
                co.gae(c_rew, c_val, c_end, c_boot, threads=cores)
            dtg = (time.perf_counter() - t0) / 3
            if "gae" in line:
                line["gae"]["cpu_baseline"] = {"value": GAE_BYTES_PER_ELEM * Tg * Ng / dtg / 1e9, "unit": "GB/s", "cores": cores,
                                               "kind": "port", "sample": f"[{Tg}, {Ng}] rollout, oracle orc_gae (OpenMP over columns)"}
                lf, lf_dt = gae_lfilter_baseline(Tg, 256)
                line["gae"]["cpu_baseline_lfilter"] = {"value": lf, "unit": "GB/s", "cores": 1, "kind": "port (scipy.signal.lfilter "
                                                       "per trajectory, the reference's arithmetic ppo.py:391-423)",
                                                       "sample": f"[{Tg}, 256] rollout in {lf_dt:.2f}s, one process"}
            v1, dt1, _ = cpu_baseline(256, 60, cores)                 # calibrate
            n_s = max(256, min(16384, int(256 * 12.0 / max(dt1, 1e-3)) // 256 * 256))
            v, dt, _ = cpu_baseline(n_s, 60, cores)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"{n_s} envs x 60 steps in {dt:.1f}s, oracle/radsearch_oracle.c "
                                              "(scalar per-env loop with per-step Dijkstra, OpenMP over envs)"}
            ref = reference_python_record()
            if ref:
                line["cpu_baseline_reference_python"] = ref
        if "e2e" not in line:
            line["e2e"] = None
        print(json.dumps(line), flush=True)
    if cx.world > 1:
        cx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
