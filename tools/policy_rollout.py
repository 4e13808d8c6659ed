"""The fused GRU actor-critic (FusedGruPolicy: rs_policy_act / rs_policy_value) against the stock PyTorch policy it replaces,
in one GPU run:

  python tools/policy_rollout.py OUT_DIR [--size full|tiny]

Writes OUT_DIR/policy_rollout.json:
  * the GPU name, power limit and max SM clock, read in the same run;
  * kernel time of act and value (CUDA events over `launches` back-to-back calls after warm-up) at 65 536, 131 072 and
    16 384 x 4 rows for the bench shape GRU(11 -> 24) + linear heads and for the reference's defaults GRU(13 -> 24) +
    32-wide tanh heads, next to CUDA-graph replays of the same torch modules (the bodies of bench.GruPolicy); FMAs and
    bytes per row from the shape, the share of the FP32 FMA bound (SMs x 128 lanes x max SM clock) and of the HBM bound
    (7.7 TB/s, data sheet), and which of the two binds; the largest difference to the torch modules at each size;
  * collection: RolloutCollector at BASELINE configs[2] (65 536 envs x T = 480, 5 obstructions, standardize=1, prefetch),
    both modes, 2 epochs each, with the fused policy and with bench.GruPolicy over the same modules: env-steps/s of the
    second epoch's collect() (incl. GAE) and the per-stage GPU times of one step as bench.py's rollout_step_stages_us;
  * evaluation: MonteCarloEvaluator.run over 1000 seeded scenarios x 100 runs (single agent, 5 obstructions) with both
    policies (host clock around run(), ending in a device synchronise).
No GPU: the script fails.  It never falls back to another device.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

SIZES = {
    "full": dict(rows=[("65536", 65536), ("131072", 131072), ("16384x4", 16384 * 4)], launches=200, N=65536, T=480,
                 S=1000, R=100),
    "tiny": dict(rows=[("4096", 4096)], launches=20, N=4096, T=48, S=20, R=10),
}
HBM_BYTES_PER_S = 7.7e12     # HGX B200 data sheet, one GPU (a bound, not a measurement)


def shape_cost(d_in, H, P, V):
    """(FMAs, bytes) per row of act and of value: the products of GRUCell and heads; obs (+ pred) and hidden in, hidden /
    action / value / logp out"""
    gru = 3 * H * (d_in + H)
    pi = 8 * H if P == 0 else P * H + 8 * P
    v = H if V == 0 else V * H + V
    x_bytes = 4 * d_in
    return {"act_fma": gru + pi + v, "act_bytes": x_bytes + 8 * H + 12, "value_fma": gru + v, "value_bytes": x_bytes + 4 * H + 4}


class TorchGraph:
    """act / value of (gru, pi, v) as captured CUDA graphs on static buffers: the body of bench.GruPolicy for any shape"""

    def __init__(self, torch, mods, N, d_in, dev):
        self.torch, (self.gru, self.pi, self.v) = torch, mods
        self.x = torch.randn(N, d_in, device=dev)
        self.h = torch.zeros(N, mods[0].hidden_size, device=dev)
        self.action = torch.zeros(N, dtype=torch.int32, device=dev)
        self.val, self.logp, self.v_next = (torch.zeros(N, device=dev) for _ in range(3))
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            for _ in range(3):
                self._act(), self._value()
        torch.cuda.current_stream(dev).wait_stream(s)
        torch.cuda.synchronize()
        self.g_act, self.g_val = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.g_act):
            self._act()
        with torch.cuda.graph(self.g_val):
            self._value()

    def _act(self):
        torch = self.torch
        with torch.no_grad():
            h = self.gru(self.x, self.h)
            self.h.copy_(h)
            lp = torch.log_softmax(self.pi(h), dim=-1)
            u = torch.rand_like(lp).clamp_(1e-10, 1.0)
            a = (lp - torch.log(-torch.log(u))).argmax(dim=-1)
            self.action.copy_(a)
            self.logp.copy_(lp.gather(1, a[:, None]).squeeze(1))
            self.val.copy_(self.v(h).squeeze(1))

    def _value(self):
        with self.torch.no_grad():
            self.v_next.copy_(self.v(self.gru(self.x, self.h)).squeeze(1))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("out", help="directory that receives policy_rollout.json")
    ap.add_argument("--size", choices=sorted(SIZES), default="full")
    args = ap.parse_args()
    sz = SIZES[args.size]

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("policy_rollout.py measures on a CUDA device and none was found (no fallback)")
    import radiation_ppo_b200 as rp
    from radteam_epoch import gpu_identity

    import bench

    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda:0")
    ident = gpu_identity(torch)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    clock_mhz = float(str(ident["max_sm_clock"]).split()[0]) if ident["max_sm_clock"] else float("nan")
    fma_per_s = sms * 128 * clock_mhz * 1e6
    out = {"size": args.size, **ident, "sms": sms,
           "fp32_fma_bound_per_s": fma_per_s, "hbm_bound_bytes_per_s": HBM_BYTES_PER_S,
           "note": "kernel shares of peak: the larger of FMAs / FMA bound and bytes / HBM bound over the kernel time; the "
                   "inputs of one call (<= 40 MB) stay in the 126 MB L2 between back-to-back launches, so the HBM bound is "
                   "a floor, not what the kernel waits for"}

    def events_us(fn, n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(max(10, n // 10)):
            fn()
        torch.cuda.synchronize()
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return 1e3 * a.elapsed_time(b) / n

    # ---- kernel time ----------------------------------------------------------------------------------------------
    shapes = {"bench GRU(11->24), linear heads": (11, 24, 0, 0, 0),
              "reference defaults GRU(13->24), tanh heads 32 / 32": (13, 24, 32, 32, 0)}
    kern = []
    for sname, (d_in, H, P, V, act) in shapes.items():
        cost = shape_cost(d_in, H, P, V)
        for rname, n in sz["rows"]:
            torch.manual_seed(0)
            gru = torch.nn.GRUCell(d_in, H)
            pi = torch.nn.Linear(H, 8) if P == 0 else torch.nn.Sequential(torch.nn.Linear(H, P), torch.nn.Tanh(),
                                                                           torch.nn.Linear(P, 8))
            v = torch.nn.Linear(H, 1) if V == 0 else torch.nn.Sequential(torch.nn.Linear(H, V), torch.nn.Tanh(),
                                                                          torch.nn.Linear(V, 1))
            mods = [m.to(dev) for m in (gru, pi, v)]
            pol = rp.FusedGruPolicy(*mods, num_rows=n, seed=1)
            obs = torch.randn(n, 11, device=dev)
            pred = torch.rand(n, 2, device=dev) if d_in == 13 else None
            tg = TorchGraph(torch, mods, n, d_in, dev)
            tg.x.copy_(obs if pred is None else torch.cat([obs, pred], 1))
            # accuracy at this size: one act from a random hidden state against the torch modules
            h0 = torch.rand(n, H, device=dev) * 2 - 1
            pol.hidden_state.copy_(h0)
            a_, val_, lp_ = pol.act(obs, pred)
            with torch.no_grad():
                h1 = gru(tg.x, h0)
                lp_ref = torch.log_softmax(pi(h1), -1).gather(1, a_.long()[:, None])[:, 0]
                diffs = {"hidden": (pol.hidden_state - h1).abs().max().item(), "value": (val_ - v(h1)[:, 0]).abs().max().item(),
                         "logp": (lp_ - lp_ref).abs().max().item()}
            t_act = events_us(lambda: pol.act(obs, pred), sz["launches"])
            t_val = events_us(lambda: pol.value(obs, pred), sz["launches"])
            tt_act = events_us(tg.g_act.replay, sz["launches"])
            tt_val = events_us(tg.g_val.replay, sz["launches"])
            rec = {"shape": sname, "rows": rname, "n_rows": n, **cost, "max_abs_diff_vs_torch": diffs,
                   "fused_act_us": t_act, "fused_value_us": t_val, "torch_graph_act_us": tt_act, "torch_graph_value_us": tt_val}
            for k, t in (("act", t_act), ("value", t_val)):
                f = n * cost[f"{k}_fma"] / fma_per_s * 1e6
                b = n * cost[f"{k}_bytes"] / HBM_BYTES_PER_S * 1e6
                rec[f"{k}_fma_bound_us"], rec[f"{k}_hbm_bound_us"] = f, b
                rec[f"{k}_share_of_fma_bound"], rec[f"{k}_share_of_hbm_bound"] = f / t, b / t
                rec[f"{k}_binding_bound"] = "fp32 FMA" if f >= b else "HBM"
            kern.append(rec)
            print(json.dumps(rec), flush=True)
            del pol, tg
    out["kernels"] = kern

    # ---- collection: RolloutCollector at configs[2] -----------------------------------------------------------------
    cx = types.SimpleNamespace(torch=torch, dev=dev)
    N, T = sz["N"], sz["T"]
    coll = {}
    for mode in ("graph", "rows"):
        for which in ("torch", "fused"):
            env = rp.RadSearch(obstruction_count=5, enforce_grid_boundaries=True, num_envs=N, seed=4, device=dev,
                               auto_reset=True, fast_poisson=True, steps_per_episode=120, prefetch=True,
                               use_cuda_graph=(mode == "graph"), standardize=1)
            buf = rp.BatchedPPOBuffer(11, T, N, device=dev)
            kw = dict(obs_in=env.obs.view(N, 11), action_out=env.action_buffer.view(N)) if mode == "graph" else {}
            gp = bench.GruPolicy(cx, N, final_obs=env.final_obs.view(N, 11), **kw)
            pol = gp if which == "torch" else rp.FusedGruPolicy(gp.net["gru"], gp.net["pi"], gp.net["v"], num_rows=N, seed=4, **kw)
            col = rp.RolloutCollector(env, buf, pol, rp.EpisodeStats(N, 1, dev), mode=mode)
            ms = []
            for _ in range(2):
                torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); col.collect(); b.record()
                torch.cuda.synchronize()
                ms.append(a.elapsed_time(b))
                buf.get()
            env_obs, fin = env.obs.view(N, 11), env.final_obs.view(N, 11)
            rows0 = buf.policy_rows(0)

            def staged(fn, n=24):
                ts = []
                for _ in range(n):
                    torch.cuda.synchronize()
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record(); fn(); b.record()
                    torch.cuda.synchronize()
                    ts.append(1e3 * a.elapsed_time(b))
                return statistics.median(ts)

            stages = {"policy_act_us": staged(lambda: pol.act(env_obs if mode == "graph" else rows0["obs"])),
                      "policy_value_us": staged(lambda: pol.value(fin)),
                      "env_step_reset_us": staged(lambda: env.step_batch(pol.action.view(N, 1)))}
            coll[f"{mode}/{which}"] = {"epoch_ms": ms, "rollout_env_steps_per_s": N * T / (ms[-1] / 1e3),
                                       "us_per_rollout_step": 1e3 * ms[-1] / T, "rollout_step_stages_us": stages}
            print(mode, which, json.dumps(coll[f"{mode}/{which}"]), flush=True)
            del env, buf, gp, pol, col
            torch.cuda.empty_cache()
    out["collection"] = {"workload": f"{N} envs x T={T}, 5 obstructions, enforced bounds, standardize=1, prefetch, fast Poisson, "
                                     "GRU(11->24) + linear heads (bench.GruPolicy's modules), collect() incl. GAE, "
                                     "second of 2 epochs", **coll}

    # ---- evaluation: MonteCarloEvaluator.run -----------------------------------------------------------------------
    S, R = sz["S"], sz["R"]
    scen = rp.RadSearch(obstruction_count=5, enforce_grid_boundaries=True, num_envs=S, seed=17, device=dev).scenario_arrays()
    ev_out = {"workload": f"{S} seeded scenarios (5 obstructions, enforced bounds) x {R} runs = {S * R} envs, single agent, "
                          "120-step episodes, GRU(11->24) + linear heads; host clock around run(), median of 3"}
    for which in ("torch", "fused"):
        ev = rp.MonteCarloEvaluator(scenarios=scen, montecarlo_runs=R, steps_per_episode=120, obstruction_count=5, seed=3,
                                    device=dev, enforce_grid_boundaries=True)
        M = S * R
        gp = bench.GruPolicy(cx, M)
        if which == "fused":
            policy = rp.FusedGruPolicy(gp.net["gru"], gp.net["pi"], gp.net["v"], num_rows=M, seed=5)
        else:
            def policy(obs, t, gp=gp):
                if t == 0:
                    gp.reset_state(None)
                return gp.act(obs.view(M, 11))[0]
        ts, res = [], None
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = ev.run(policy)
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        steps = int(res.episode_length.sum())
        ev_out[which] = {"run_s": ts, "median_run_s": statistics.median(ts), "runs_per_s": M / statistics.median(ts),
                         "env_steps_played": steps, "summary": res.summary()}
        print("eval", which, json.dumps(ev_out[which]), flush=True)
        del ev, gp, policy
        torch.cuda.empty_cache()
    out["evaluation"] = ev_out

    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "policy_rollout.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", os.path.join(args.out, "policy_rollout.json"))


if __name__ == "__main__":
    main()
