"""One RAD-TEAM epoch at BASELINE configs[3] (16,384 envs x 4 agents, 5 obstructions, enforced bounds, 120-step
episodes, T = 480) through TeamRolloutCollector with a scripted policy -- fixed random linear heads on the map stacks, so
that the collector's own cost is what is timed -- and BatchedMapsBuffer.replay of the epoch's stacks for the update.

  python tools/radteam_epoch.py --out <dir>                # full size, on a GPU
  python tools/radteam_epoch.py --size tiny --out <dir>    # rehearsal shapes (still needs a GPU to run)

Writes <out>/radteam_epoch.json:
  * the GPU name and power limit, read in the same run;
  * per-step stage times (CUDA events on the collector's stream, median over the timed epoch): maps update (predict +
    rs_maps_update), pre (rs_rollout_pre_team), env step, bootstrap (predict + masked rs_maps_update + value head), post
    (rs_rollout_post_team), maps reset; the policy's action head is timed as its own stage;
  * env-steps/s of a whole epoch (collect() incl. GAE, no events);
  * replay of (a) whole episodes and (b) single random rows: emitted rows/s and GB/s of the algorithmic bytes
    (4 (6A + 4) X Y per emitted row + 52 A per replayed call), set against a device-to-device copy rate measured in the
    same run (>= 1 GB, cudaMemcpyAsync through torch's copy_ of contiguous tensors; bytes read + written).
No GPU: the script fails.  It never falls back to another device.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SIZES = {   # envs, agents, steps per epoch, steps per episode, whole episodes replayed, single rows replayed, copy MB
    "full": dict(N=16384, A=4, T=480, ML=120, episodes=4096, rows=8192, copy_mb=2048),
    "tiny": dict(N=64, A=4, T=48, ML=24, episodes=32, rows=64, copy_mb=64),
}


def gpu_identity(torch):
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        power, clock = [x.strip() for x in q.stdout.strip().split(",")[:2]]
    except Exception as e:                                # noqa: BLE001 -- reported, not hidden
        power, clock = f"unavailable ({e})", None
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


class Heads:
    """Scripted team policy: fixed random linear heads.  act: logits = actor stack (as stored, [X, Y, 6]) @ Wa -> argmax
    over 8 moves, value = critic stack @ wc + agent offset; predict: sigmoid(obs[:, :, :3] @ Wp) (in the map)."""

    def __init__(self, torch, N, A, X, Y, dev, marks=None):
        g = torch.Generator(device=dev).manual_seed(5)
        self.t, self.N, self.A = torch, N, A
        self.Wa = torch.randn(X * Y * 6, 8, generator=g, device=dev) * 0.01
        self.wc = torch.randn(X * Y * 4, 1, generator=g, device=dev) * 0.01
        self.Wp = torch.randn(3, 2, generator=g, device=dev)
        self.off = torch.arange(A, device=dev, dtype=torch.float32) * 0.01
        self.marks = marks

    def _mark(self, name):
        if self.marks is not None:
            self.marks(name)

    def predict(self, obs):
        self._mark("predict")
        x = obs[..., :3].clone()
        x[..., 0] = self.t.log1p(x[..., 0]) * 0.1
        return self.t.sigmoid(x @ self.Wp).contiguous()

    def act(self, obs, actor, critic):
        self._mark("act")
        a_store = actor.permute(0, 1, 3, 4, 2).reshape(self.N * self.A, -1)      # the stored layout: no copy
        c_store = critic.permute(0, 2, 3, 1).reshape(self.N, -1)
        action = (a_store @ self.Wa).argmax(dim=1).to(self.t.int32).view(self.N, self.A)
        v = (c_store @ self.wc) + self.off
        self._mark("act_end")
        return action, v, (-0.5 * v).contiguous()

    def value(self, critic):
        v = (critic.permute(0, 2, 3, 1).reshape(self.N, -1) @ self.wc) + self.off
        self._mark("value_end")
        return v.contiguous()

    def reset_state(self, mask):
        pass


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--size", choices=sorted(SIZES), default="full")
    ap.add_argument("--out", required=True, help="directory that receives radteam_epoch.json")
    ap.add_argument("--mode", choices=("rows", "graph"), default="rows")
    args = ap.parse_args()
    sz = SIZES[args.size]
    N, A, T, ML = sz["N"], sz["A"], sz["T"], sz["ML"]
    X = Y = 27
    row_bytes = 4 * (6 * A + 4) * X * Y
    print(f"size {args.size}: {N} envs x {A} agents, T = {T}, {row_bytes} B of stacks per env and step", flush=True)

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("radteam_epoch.py measures on a CUDA device and none was found (no fallback)")
    import radiation_ppo_b200 as rp

    dev = torch.device("cuda:0")
    out = {"size": args.size, "mode": args.mode, **gpu_identity(torch),
           "workload": f"{N} envs x {A} agents, 5 obstructions, enforced bounds, {X}x{Y} maps, {ML}-step episodes, T = {T}"}

    env = rp.RadSearch(obstruction_count=5, enforce_grid_boundaries=True, number_agents=A, num_envs=N, seed=4, device=dev,
                       steps_per_episode=ML, auto_reset=True, prefetch=(args.mode == "graph"),
                       use_cuda_graph=(args.mode == "graph"))
    maps = rp.BatchedMapsBuffer(N, A, ML, environment_scale=env.scale, device=dev)
    buf = rp.BatchedPPOBuffer(11, T, N, agents=A, device=dev)
    stats = rp.EpisodeStats(N, A, dev)

    # ---- stage timing: events at the stage boundaries on the collector's stream -------------------------------------
    events, timing = [], [True]

    def mark(name):
        if not timing[0]:
            return
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        events.append((name, e))

    class TimedMaps:                       # the collector's maps, with events around update / reset
        def __init__(self, m):
            self.m, self.num_envs, self.number_of_agents = m, m.num_envs, m.number_of_agents
            self.n_update = 0

        def update(self, *a, **k):
            r = self.m.update(*a, **k)
            mark("update_end" if self.n_update % 2 == 0 else "boot_update_end")
            self.n_update += 1
            return r

        def reset(self, *a, **k):
            mark("reset")
            self.m.reset(*a, **k)
            mark("reset_end")

    class TimedEnv:                        # the env, with events around step_batch
        def __init__(self, e):
            self.__dict__["e"] = e

        def __getattr__(self, k):
            return getattr(self.e, k)

        def step_batch(self, *a, **k):
            mark("step")
            r = self.e.step_batch(*a, **k)
            mark("step_end")
            return r

    pol = Heads(torch, N, A, X, Y, dev, marks=mark)
    tmaps = TimedMaps(maps)
    col_t = rp.TeamRolloutCollector(TimedEnv(env), buf, tmaps, pol, stats, mode=args.mode)
    # the first predict of a step opens it; the second predict (bootstrap) follows step_end
    col_t.collect()                                     # warm-up epoch: every shape, the captured graphs
    torch.cuda.synchronize()
    events.clear()
    tmaps.n_update = 0
    col_t.collect()
    torch.cuda.synchronize()
    stages = {k: [] for k in ("maps_update", "policy_act", "pre", "env_step", "bootstrap_maps_and_value", "post", "maps_reset")}
    step, cur = [], []
    for name, e in events:                              # split the event list into steps (each opens with "predict")
        if name == "predict" and cur and cur[-1][0] == "reset_end":
            step.append(cur)
            cur = []
        cur.append((name, e))
    step.append(cur)
    for s in step:
        d = dict()
        for name, e in s:
            d.setdefault(name, e)
        boot_pred = [e for name, e in s if name == "predict"][1]
        el = lambda a, b: a.elapsed_time(b)              # noqa: E731
        stages["maps_update"].append(el(d["predict"], d["update_end"]))
        stages["policy_act"].append(el(d["act"], d["act_end"]))
        stages["pre"].append(el(d["act_end"], d["step"]))
        stages["env_step"].append(el(d["step"], d["step_end"]))
        stages["bootstrap_maps_and_value"].append(el(boot_pred, d["value_end"]))
        stages["post"].append(el(d["value_end"], d["reset"]))
        stages["maps_reset"].append(el(d["reset"], d["reset_end"]))
    assert len(step) == T, (len(step), T)
    out["stage_ms_median"] = {k: statistics.median(v) for k, v in stages.items()}
    out["stage_ms_mean"] = {k: sum(v) / len(v) for k, v in stages.items()}
    out["stage_note"] = ("intervals between events recorded on the stream at the stage boundaries: launch gaps the host "
                         "leaves inside a stage count towards it")

    # ---- whole epochs, no events ----------------------------------------------------------------------------------
    timing[0] = False
    col = col_t
    torch.cuda.synchronize()
    reps = 3
    t0 = time.perf_counter()
    for _ in range(reps):
        col.collect()
    t_enq = time.perf_counter()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / reps
    out["epoch_s"] = dt
    # the host's share: when enqueueing the epochs takes (almost) as long as running them, the host sets the pace
    out["epoch_host_enqueue_s"] = (t_enq - t0) / reps
    out["env_steps_per_s"] = N * T / dt
    out["agent_steps_per_s"] = N * A * T / dt
    out["maps_status_flags"] = int(maps.status.sum().item())

    # ---- HBM copy rate of this card, same run ------------------------------------------------------------------------
    nb = sz["copy_mb"] * 2 ** 20
    src = torch.empty(nb, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    dst.copy_(src)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    copy_gbs = 2 * nb * 10 / (e0.elapsed_time(e1) / 1e3) / 1e9
    out["d2d_copy"] = {"bytes_per_copy": nb, "GBps_read_plus_write": copy_gbs}
    del src, dst

    # ---- replay -------------------------------------------------------------------------------------------------------
    _, ep_start, ep_len = buf.pack_episodes()
    ranges_all = rp.episode_ranges(ep_start, ep_len, T, agents=A)
    g = torch.Generator(device="cpu").manual_seed(9)
    pick = torch.randperm(ranges_all.shape[0], generator=g)[:sz["episodes"]]
    ep_ranges = ranges_all[pick.to(ranges_all.device)].contiguous()
    rn = torch.randint(0, N, (sz["rows"],), generator=g)
    rt = torch.randint(0, T, (sz["rows"],), generator=g)
    row_ranges = torch.stack((rn, rt, rt), dim=1).to(torch.int32).to(dev)
    end = buf.end_buf.view(T, N, A)[:, :, 0].cpu().numpy() != 0

    def calls_of(rg):
        """replayed observation_to_map calls: whole range + the episode head before t0"""
        n = 0
        for e, t0, t1 in rg.tolist():
            s = t0
            while s > 0 and not end[s - 1, e]:
                s -= 1
            n += t1 - s + 1
        return n

    res = {}
    for label, rg in (("whole_episodes", ep_ranges), ("single_rows", row_ranges)):
        rows = int((rg[:, 2] - rg[:, 1] + 1).sum().item())
        store = (torch.empty(rows, A, X, Y, 6, device=dev), torch.empty(rows, X, Y, 4, device=dev))
        for _ in range(2):
            maps.replay(buf, rg, out=store)                 # warm-up
        torch.cuda.synchronize()
        e0.record()
        reps = 5
        for _ in range(reps):
            _, _, status = maps.replay(buf, rg, out=store)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        calls = calls_of(rg)
        alg = rows * row_bytes + calls * 52 * A
        res[label] = {"ranges": int(rg.shape[0]), "rows": rows, "replayed_calls": calls, "ms": ms,
                      "rows_per_s": rows / (ms / 1e3), "algorithmic_bytes": alg, "GBps": alg / (ms / 1e3) / 1e9,
                      "frac_of_measured_copy_rate": alg / (ms / 1e3) / 1e9 / copy_gbs,
                      "output_bytes": rows * row_bytes, "status_flags": int(status.abs().sum().item())}
        del store
    out["replay"] = res
    out["context"] = "data-sheet HBM3e bandwidth of a B200 at 1000 W: 7.7 TB/s (not reached here; the copy rate is the yardstick)"
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "radteam_epoch.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))
    print("wrote", path)


if __name__ == "__main__":
    main()
