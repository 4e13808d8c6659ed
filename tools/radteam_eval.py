"""Monte-Carlo evaluation of a RAD-TEAM policy (MonteCarloEvaluator.run_team) at batch scale: 1000 scenarios with 5
obstructions (seeded, from one batched reset), 25 runs each, 4 agents -- 25,000 envs, 27 x 27 maps (about 2 GB of map
stacks) -- played by the scripted linear-head policy of tools/radteam_epoch.py, so that the evaluator's own cost is what
is timed.

  python tools/radteam_eval.py --out <dir>                # full size, on a GPU
  python tools/radteam_eval.py --size tiny --out <dir>    # rehearsal shapes (still needs a GPU to run)

Writes <out>/radteam_eval.json:
  * the GPU name and power limit, read in the same run;
  * end to end (host clock around run_team, ending in a device synchronise): env-steps/s and runs/s, with the early stop
    and with all steps_per_episode steps played;
  * per-step stage intervals (CUDA events on the evaluator's stream, median over the steps of one run): predict + maps
    update, policy act, env step, bookkeeping (rs_eval_step);
  * rs_eval_step kernel time (CUDA events over many launches, every env playing) against the torch ops run() uses for
    its bookkeeping, timed the same way;
  * rs_maps_update time as a function of the fraction of runs still playing (the mask run_team passes).
No GPU: the script fails.  It never falls back to another device.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

SIZES = {   # scenarios, runs per scenario, agents, steps per episode, launches per kernel timing
    "full": dict(S=1000, R=25, A=4, ML=120, launches=2000),
    "tiny": dict(S=16, R=4, A=4, ML=40, launches=50),
}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--size", choices=sorted(SIZES), default="full")
    ap.add_argument("--out", required=True, help="directory that receives radteam_eval.json")
    args = ap.parse_args()
    sz = SIZES[args.size]
    S, R, A, ML = sz["S"], sz["R"], sz["A"], sz["ML"]
    N = S * R

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("radteam_eval.py measures on a CUDA device and none was found (no fallback)")
    import radiation_ppo_b200 as rp
    from radiation_ppo_b200 import _lib as L
    from radteam_epoch import Heads, gpu_identity

    dev = torch.device("cuda:0")
    X = Y = 27
    out = {"size": args.size, **gpu_identity(torch),
           "workload": f"{S} scenarios (5 obstructions, enforced bounds) x {R} runs = {N} envs x {A} agents, {X}x{Y} maps, "
                       f"{ML}-step episodes, scripted linear-head policy"}
    scen = rp.RadSearch(obstruction_count=5, enforce_grid_boundaries=True, num_envs=S, seed=17, device=dev).scenario_arrays()
    ev = rp.MonteCarloEvaluator(scenarios=scen, montecarlo_runs=R, steps_per_episode=ML, obstruction_count=5, seed=3,
                                device=dev, enforce_grid_boundaries=True, number_agents=A)
    env = ev.env
    maps = rp.BatchedMapsBuffer(N, A, ML, environment_scale=env.scale, device=dev)
    out["map_state_bytes"] = sum(t.numel() * t.element_size() for t in (
        maps._actor_store, maps._critic_store, maps._log_cell, maps._log_val))

    # ---- end to end, no events ---------------------------------------------------------------------------------------
    pol = Heads(torch, N, A, X, Y, dev)
    ev.run_team(pol, maps=maps)                                   # warm-up: every shape
    torch.cuda.synchronize()
    e2e = {}
    for label, early in (("early_stop", True), ("all_steps", False)):
        times, res = [], None
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = ev.run_team(pol, maps=maps, early_stop=early)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        dt = statistics.median(times)
        e2e[label] = {"s": dt, "s_all": times, "steps_played": res.steps_played, "env_steps_per_s": N * res.steps_played / dt,
                      "agent_steps_per_s": N * A * res.steps_played / dt, "runs_per_s": N / dt,
                      "success_rate": float(res.success.float().mean()), **{k: v for k, v in res.summary().items()}}
    out["end_to_end"] = e2e
    out["maps_status_flags"] = int(maps.status.sum().item())

    # ---- per-step stage intervals: events at the stage boundaries ------------------------------------------------------
    events = []

    def mark(name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        events.append((name, e))

    class TimedMaps:
        def __init__(self, m):
            self.m, self.num_envs, self.number_of_agents = m, m.num_envs, m.number_of_agents

        def update(self, *a, **k):
            r = self.m.update(*a, **k)
            mark("update_end")
            return r

        def reset(self, *a, **k):
            self.m.reset(*a, **k)

    class TimedEnv:
        def __init__(self, e):
            self.__dict__["e"] = e

        def __getattr__(self, k):
            return getattr(self.e, k)

        def step_batch(self, *a, **k):
            mark("step")
            r = self.e.step_batch(*a, **k)
            mark("step_end")
            return r

    pol_t = Heads(torch, N, A, X, Y, dev, marks=mark)
    ev.env = TimedEnv(env)
    try:
        res = ev.run_team(pol_t, maps=TimedMaps(maps), early_stop=False, on_step=lambda t, o, a: mark("eval_end"))
        torch.cuda.synchronize()
    finally:
        ev.env = env
    steps, cur = [], []
    for name, e in events:
        if name == "predict" and cur:
            steps.append(dict(cur))
            cur = []
        cur.append((name, e))
    steps.append(dict(cur))
    stages = {k: [] for k in ("predict_and_maps_update", "policy_act", "env_step", "eval_step")}
    for d in steps:
        stages["predict_and_maps_update"].append(d["predict"].elapsed_time(d["update_end"]))
        stages["policy_act"].append(d["act"].elapsed_time(d["act_end"]))
        stages["env_step"].append(d["step"].elapsed_time(d["step_end"]))
        stages["eval_step"].append(d["step_end"].elapsed_time(d["eval_end"]))
    assert len(steps) == ML, (len(steps), ML)
    out["stage_ms_median"] = {k: statistics.median(v) for k, v in stages.items()}
    out["stage_ms_mean"] = {k: sum(v) / len(v) for k, v in stages.items()}
    out["stage_note"] = ("all steps_per_episode steps; intervals between events recorded on the stream at the stage "
                         "boundaries: launch gaps the host leaves inside a stage count towards it")

    # ---- rs_eval_step vs the torch ops of run(), every env playing ----------------------------------------------------
    lib = L.load()
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    p = lambda x: None if x is None else C.c_void_p(x.data_ptr())         # noqa: E731
    z = lambda *s, dt: torch.zeros(*s, dtype=dt, device=dev)              # noqa: E731
    done0 = z(N, A, dt=torch.uint8)                                         # nobody finishes: the work stays the same
    pred = (torch.rand(N, A, 2, device=dev) * 0.8 + 0.1).contiguous()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_launch = sz["launches"]

    def time_launches(fn):
        for _ in range(20):
            fn()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(n_launch):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n_launch * 1e3                         # us per call

    active, success, finders = torch.ones(N, dtype=torch.uint8, device=dev), z(N, dt=torch.uint8), z(N, dt=torch.uint8)
    length, ret, oob = z(N, dt=torch.int32), z(N, A, dt=torch.float64), z(N, A, dt=torch.int32)
    n_active = torch.full((1,), N, dtype=torch.int32, device=dev)
    loc = (z(N, A, dt=torch.float64), z(N, A, dt=torch.int32), z(N, A, dt=torch.float32))
    kern = {}
    for label, pr in (("rs_eval_step_us", pred), ("rs_eval_step_no_pred_us", None)):
        lg = loc if pr is not None else (None,) * 3

        def call():
            L.check(lib.rs_eval_step(p(env.reward), p(env.team_reward), p(done0), p(env.info_flags), p(active), p(success),
                                     p(length), p(ret), p(oob), p(finders), p(n_active), p(pr), p(env._src) if pr is not None
                                     else None, env.scale, *[p(x) for x in lg], N, A, 0, stream), "rs_eval_step")
        kern[label] = time_launches(call)
    t_active, t_success = torch.ones(N, dtype=torch.bool, device=dev), torch.zeros(N, dtype=torch.bool, device=dev)
    t_len, t_ret = z(N, dt=torch.int32), z(N, dt=torch.float64)

    def torch_ops():                                                        # evaluate.py run(), its bookkeeping lines
        r = env.team_reward
        t_ret.add_(torch.where(t_active, r, torch.zeros_like(r)).double())
        t_len.add_(t_active.to(torch.int32))
        terminal = (done0 != 0).any(dim=1) & t_active
        t_success.logical_or_(terminal)
        t_active.logical_and_(~terminal)
    kern["torch_ops_of_run_us"] = time_launches(torch_ops)
    kern["note"] = ("device time per call from CUDA events over back-to-back calls (launch-bound at this size); the torch "
                    "ops keep agent 0's return only, rs_eval_step every agent's return, out-of-bounds counts, finders, the "
                    "count of runs playing and (first row) the localisation error")
    # algorithmic bytes of one rs_eval_step call with predictions, team rewards, every env playing: per env active r/w,
    # length r/w, source, team reward; per agent done, info, return r/w, out-of-bounds r/w, prediction, error sum r/w,
    # count r/w, last error
    kern["rs_eval_step_bytes"] = N * (2 + 8 + 8 + 4) + N * A * (1 + 1 + 16 + 8 + 8 + 16 + 8 + 4)
    out["bookkeeping"] = kern

    # ---- rs_maps_update vs the fraction of runs still playing ----------------------------------------------------------
    obs = env.obs
    pr = pol.predict(obs)
    g = torch.Generator(device="cpu").manual_seed(1)
    frac_ms = {}
    for frac in (1.0, 0.5, 0.25, 0.1, 0.0):
        mask = (torch.rand(N, generator=g) < frac).to(torch.uint8).to(dev)
        maps.reset()
        for _ in range(3):
            maps.update(obs, pr, mask=mask)
        reps = 20
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            maps.update(obs, pr, mask=mask)
        e1.record()
        torch.cuda.synchronize()
        frac_ms[str(frac)] = {"playing": int(mask.sum().item()), "ms": e0.elapsed_time(e1) / reps}
    out["maps_update_vs_fraction_playing"] = frac_ms
    maps.reset()

    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "radteam_eval.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))
    print("wrote", path)


if __name__ == "__main__":
    main()
