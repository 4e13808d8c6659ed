"""The fused PPO loss and gradient (FusedGruPolicy.loss_and_grad: rs_policy_ppo_grad) against the stock autograd update
it replaces (the body of bench.py::ppo_update), in one GPU run:

  python tools/policy_update.py OUT_DIR [--size full|tiny]

Writes OUT_DIR/policy_update.json:
  * the GPU name, power limit and max SM clock, read in the same run;
  * for GRU(11 -> 24) + linear heads (the bench) and GRU(13 -> 24) + 32-wide tanh heads (the reference's defaults), at
    M = 8 192 and 65 536 columns x T = 480 of the same seeded rollout rows: the time of one gradient by the stock loop
    (bench.py's, 8 192 columns per chunk, loss.backward()) and by loss_and_grad, alternating, CUDA events; rows/s; the
    FMAs per row and the fp32 rate they make, the workspace bytes (both from the shapes); the largest difference per
    parameter tensor between the two gradients, relative to the tensor's largest entry;
  * one pipeline epoch at BASELINE configs[2] (65 536 envs x 480 steps): collect with FusedGruPolicy, get(episodes=True),
    the update on 8 192 columns (fused: loss_and_grad + Adam + sync; stock: the autograd loop + Adam), CUDA events.
No GPU: the script fails.  It never falls back to another device.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

SIZES = {"full": dict(Ms=[8192, 65536], T=480, reps=3, N_env=65536), "tiny": dict(Ms=[256], T=24, reps=1, N_env=1024)}
SHAPES = {"bench GRU(11->24), linear heads": (11, 24, 0, 0, 0), "reference GRU(13->24), 32/32 tanh heads": (13, 24, 32, 32, 0)}


def grad_fma_per_row(d_in, H, P, V):
    """FMAs of one (column, step) row: forward cell; backward: cell recomputed, heads forward, heads backward (dlogit /
    dv through the hidden layers into dL/dh), the cell's transposed products, and one FMA per parameter for the weight
    gradient's outer products"""
    cell = 3 * H * (d_in + H)
    heads_fwd = (8 * H if P == 0 else P * H + 8 * P) + (H if V == 0 else V * H + V)
    heads_back = (8 * H if P == 0 else 8 * P + P * H) + (H if V == 0 else V + V * H)
    params = 3 * H * d_in + 3 * H * H + 6 * H + (8 * H + 8 if P == 0 else P * H + P + 8 * P + 8) + \
        (H + 1 if V == 0 else V * H + 2 * V + 1)
    return 2 * cell + heads_fwd + heads_back + 3 * H * H + params


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("out", help="directory that receives policy_update.json")
    ap.add_argument("--size", choices=sorted(SIZES), default="full")
    args = ap.parse_args()
    sz = SIZES[args.size]

    import ctypes as C

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("policy_update.py measures on a CUDA device and none was found (no fallback)")
    import radiation_ppo_b200 as rp
    from radiation_ppo_b200 import _lib as L
    from radteam_epoch import gpu_identity

    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda:0")
    out = {"size": args.size, **gpu_identity(torch), "T": sz["T"], "cases": [], "note":
           "stock = bench.py::ppo_update's loop (GRUCell step by step through autograd, 8192 columns per chunk); fused = one "
           "rs_policy_ppo_grad launch plus the accumulation into .grad; both differentiate the same loss on the same rows"}
    ev = lambda: torch.cuda.Event(enable_timing=True)      # noqa: E731

    def timed_ms(fn):
        torch.cuda.synchronize()
        a, b = ev(), ev()
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    def stock_grad(mods, buf, pred, M, chunk=8192, clip=0.2):
        gru, pi, v = mods
        T = buf.T
        for m in mods:
            m.zero_grad(set_to_none=True)
        for c0 in range(0, M, chunk):
            sl = slice(c0, min(M, c0 + chunk))
            h = torch.zeros(sl.stop - sl.start, gru.hidden_size, device=dev)
            loss = 0.0
            for t in range(T):
                x = buf.obs_buf[t, sl] if pred is None else torch.cat([buf.obs_buf[t, sl], pred[t, sl]], dim=1)
                h = gru(x, h)
                lp = torch.log_softmax(pi(h), dim=-1).gather(1, buf.act_buf[t, sl].long()[:, None]).squeeze(1)
                val = v(h).squeeze(1)
                ratio = torch.exp(lp - buf.logp_buf[t, sl])
                a = buf.adv_buf[t, sl]
                loss = loss - torch.minimum(ratio * a, torch.clamp(ratio, 1 - clip, 1 + clip) * a).sum() \
                    + 0.5 * ((val - buf.ret_buf[t, sl]) ** 2).sum()
                h = h * (buf.end_buf[t, sl] == 0)[:, None]
            (loss / (T * M)).backward()

    def modules(d_in, H, P, V, act):
        torch.manual_seed(0)
        A = (torch.nn.Tanh, torch.nn.ReLU)[act]
        gru = torch.nn.GRUCell(d_in, H)
        pi = torch.nn.Linear(H, 8) if P == 0 else torch.nn.Sequential(torch.nn.Linear(H, P), A(), torch.nn.Linear(P, 8))
        v = torch.nn.Linear(H, 1) if V == 0 else torch.nn.Sequential(torch.nn.Linear(H, V), A(), torch.nn.Linear(V, 1))
        return gru.to(dev), pi.to(dev), v.to(dev)

    def params_of(mods):
        return [mods[0].weight_ih, mods[0].weight_hh, mods[0].bias_ih, mods[0].bias_hh] + list(mods[1].parameters()) + \
            list(mods[2].parameters())

    T = sz["T"]
    lib = L.load()
    for name, shape in SHAPES.items():
        for M in sz["Ms"]:
            g = torch.Generator(device=dev).manual_seed(M)
            buf = rp.BatchedPPOBuffer(11, T, M, device=dev)
            buf.obs_buf.copy_(torch.randn(T, M, 11, generator=g, device=dev))
            buf.act_buf.copy_(torch.randint(0, 8, (T, M), generator=g, device=dev).float())
            buf.adv_buf.copy_(torch.randn(T, M, generator=g, device=dev))
            buf.ret_buf.copy_(torch.randn(T, M, generator=g, device=dev))
            buf.logp_buf.copy_(-2.08 + 0.3 * torch.randn(T, M, generator=g, device=dev))
            buf.end_buf.copy_((torch.rand(T, M, generator=g, device=dev) < 1 / 60).to(torch.uint8))
            pred = torch.rand(T, M, 2, generator=g, device=dev) if shape[0] == 13 else None
            mods = modules(*shape)
            pol = rp.FusedGruPolicy(*mods, num_rows=M)
            ps = params_of(mods)

            def fused():
                for p in ps:
                    p.grad = None
                pol.loss_and_grad(buf, pred=pred)

            fused()
            stock_grad(mods, buf, pred, M)                              # warm-up of both
            stock_ms, fused_ms = [], []
            for _ in range(sz["reps"]):
                stock_ms.append(timed_ms(lambda: stock_grad(mods, buf, pred, M)))
                fused_ms.append(timed_ms(fused))
            stock_grad(mods, buf, pred, M)
            g_stock = [p.grad.clone() for p in ps]
            fused()
            diff = max(((p.grad - s).abs().max() / s.abs().max().clamp(min=1e-30)).item() for p, s in zip(ps, g_stock))
            # the kernel alone, back to back
            fused_kernel_ms = min(timed_ms(lambda: pol.loss_and_grad(buf, pred=pred)) for _ in range(sz["reps"]))
            fma = grad_fma_per_row(*shape[:4])
            f = min(fused_ms)
            rec = {"shape": name, "M": M, "T": T, "stock_ms": stock_ms, "fused_ms": fused_ms,
                   "fused_with_grad_accumulation_ms_min": f, "fused_back_to_back_ms_min": fused_kernel_ms,
                   "speedup_min_over_min": min(stock_ms) / f,
                   "stock_rows_per_s": T * M / (min(stock_ms) / 1e3), "fused_rows_per_s": T * M / (f / 1e3),
                   "fma_per_row": fma, "fused_fp32_fma_per_s": fma * T * M / (f / 1e3),
                   "fused_fp32_flop_per_s": 2 * fma * T * M / (f / 1e3),
                   "workspace_bytes": int(lib.rs_policy_grad_workspace_bytes(C.byref(pol.cfg), T, M)),
                   "max_rel_grad_diff_vs_stock": diff}
            print(json.dumps(rec), flush=True)
            out["cases"].append(rec)
            del buf, pol, mods, ps, g_stock
            torch.cuda.empty_cache()

    # one pipeline epoch with the fused policy in the loop, the update fused or stock on the same collected rows
    N = sz["N_env"]
    env = rp.RadSearch(obstruction_count=5, enforce_grid_boundaries=True, num_envs=N, seed=4, device=dev, auto_reset=True,
                       steps_per_episode=120, prefetch=True, standardize=1)
    buf = rp.BatchedPPOBuffer(11, T, N, device=dev)
    mods = modules(11, 24, 0, 0, 0)
    pol = rp.FusedGruPolicy(*mods, num_rows=N, seed=1)
    col = rp.RolloutCollector(env, buf, pol, rp.EpisodeStats(N, 1, dev), mode="rows")
    opt = torch.optim.Adam(params_of(mods), lr=3e-4)
    Mu = min(8192, N)
    cols = torch.arange(Mu, dtype=torch.int32, device=dev)
    epochs = []
    for ep in range(2):
        e = [ev() for _ in range(4)]
        torch.cuda.synchronize()
        e[0].record()
        col.collect()
        e[1].record()
        buf.get(episodes=True)
        e[2].record()
        opt.zero_grad(set_to_none=True)
        pol.loss_and_grad(buf, columns=cols)
        opt.step()
        pol.sync()
        e[3].record()
        torch.cuda.synchronize()
        epochs.append({"collect_gae_ms": e[0].elapsed_time(e[1]), "get_ms": e[1].elapsed_time(e[2]),
                       "fused_update_ms": e[2].elapsed_time(e[3])})
    sub = rp.BatchedPPOBuffer(11, T, Mu, device=dev)                    # the stock loop on the same 8192 columns
    for k in ("obs_buf", "act_buf", "adv_buf", "ret_buf", "logp_buf", "end_buf"):
        getattr(sub, k).copy_(getattr(buf, k)[:, :Mu])
    stock_update_ms = min(timed_ms(lambda: (stock_grad(mods, sub, None, Mu), opt.step())) for _ in range(2))
    last = epochs[-1]
    base = last["collect_gae_ms"] + last["get_ms"]
    out["pipeline_epoch"] = {
        "workload": f"{N} envs x T={T}, FusedGruPolicy in the loop (rows mode), get(episodes=True), one update on {Mu} "
                    "columns (gradient + Adam)", "epochs": epochs, "stock_update_ms": stock_update_ms,
        "pipeline_env_steps_per_s_fused_update": N * T / ((base + last["fused_update_ms"]) / 1e3),
        "pipeline_env_steps_per_s_stock_update": N * T / ((base + stock_update_ms) / 1e3),
        "collect_env_steps_per_s": N * T / (last["collect_gae_ms"] / 1e3)}
    print(json.dumps(out["pipeline_epoch"]), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "policy_update.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
