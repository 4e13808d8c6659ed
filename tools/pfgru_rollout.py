"""The fused PFGRU localiser (FusedPFGRU: rs_pfgru_predict / peek / restart) against the stock PyTorch cell it replaces,
in one GPU run, at the reference shape (K = 40 particles, H = 24, d_in = 3, hid_obs width 24, alpha = 0.7):

  python tools/pfgru_rollout.py OUT_DIR [--size full|tiny]

Writes OUT_DIR/r06_pfgru.json:
  * the GPU name, power limit and max SM clock, read in the same run, and the HBM bandwidth measured in the same run
    (device-to-device copies of 4 GiB);
  * the registers and spills of every kernel instantiation (nvcc -Xptxas -v on rs_pfgru.cu, into a temporary directory);
  * kernel time of predict (CUDA events over `launches` back-to-back calls after warm-up) at 65 536 and 131 072 rows; FMAs
    and bytes per row from the shape, the share of the FP32 FMA bound (SMs x 128 lanes x max SM clock) and of the measured
    HBM bandwidth, and which of the two binds; the largest difference to the float64 restatement at each size;
  * the stock torch cell (float32, the reference's PFGRUCell.forward with torch.multinomial resampling, batch-first) at the
    same rows, by the same events;
  * collection: RolloutCollector in graph mode, 65 536 envs x T = 480, 5 obstructions, standardize=1, prefetch, with
    FusedGruPolicy(GRUCell(13, 24), Linear(24, 8), Linear(24, 1)) and the fused localiser, and the same policy with the
    torch cell as localiser (predict and an all-rows bootstrap prediction per step), 2 epochs each: the second epoch.
No GPU: the script fails.  It never falls back to another device.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

SIZES = {
    "full": dict(rows=[65536, 131072], launches=200, N=65536, T=480),
    "tiny": dict(rows=[4096], launches=20, N=4096, T=48),
}
D_IN, H, K, W, ALPHA = 3, 24, 40, 24, 0.7


def shape_cost():
    """(FMAs, bytes) per row of predict: the products of the cell for K particles and of hid_obs; the state in and out,
    the observation's d_in columns in, the prediction out"""
    I = H + D_IN
    fma = K * (2 * H * I + 2 * H * I + I) + K * H + W * H + 2 * W      # gates, n, fc_obs; weighted mean; hid_obs
    return fma, 2 * 4 * K * (H + 1) + 4 * D_IN + 8


class TorchPFGRU:
    """The stock torch cell (PFGRUCell.forward, float32) over rows x K particles, with the FusedPFGRU interface"""

    def __init__(self, torch, mods, rows, dev):
        self.t = torch
        self.fz, self.fr, self.fn, self.fo, self.ho = mods
        self.rows = rows
        self.h = torch.rand(rows, K, H, device=dev)
        self.p = torch.full((rows, K), -float(torch.log(torch.tensor(float(K)))), device=dev)
        self.pred = torch.zeros(rows, 2, device=dev)

    def _step(self, obs):
        t = self.t
        x = obs.reshape(self.rows, 11)[:, None, :D_IN].expand(-1, K, -1)
        h0, p0 = self.h, self.p
        with t.no_grad():
            cat = t.cat([h0, x], dim=-1)
            z, r = t.sigmoid(self.fz(cat)), t.sigmoid(self.fr(cat))
            mu, var = t.split(self.fn(t.cat([r * h0, x], dim=-1)), H, dim=-1)
            n = t.tanh(mu + t.randn_like(var) * t.nn.functional.softplus(var))
            h1 = (1 - z) * n + z * h0
            p1 = self.fo(t.cat([h1, x], dim=-1))[..., 0] + p0
            p1 = p1 - t.logsumexp(p1, dim=1, keepdim=True)
            q = ALPHA * p1.exp() + (1 - ALPHA) / K
            idx = t.multinomial(q, K, replacement=True)
            h = t.gather(h1, 1, idx[:, :, None].expand(-1, -1, H))
            w = t.gather(p1, 1, idx).exp()
            p = t.log(w / (ALPHA * w + (1 - ALPHA) / K))
            p = p - t.logsumexp(p, dim=1, keepdim=True)
            pred = self.ho((p.exp()[:, :, None] * h).sum(dim=1))
        return h, p, pred

    def predict(self, obs=None, out=None):
        self.h, self.p, pred = self._step(obs)
        (self.pred if out is None else out).copy_(pred)
        return self.pred if out is None else out

    def peek(self, obs, mask=None, mask_bits=0):
        return self._step(obs)[2]

    def reset_state(self, mask=None, mask_bits=0):
        if mask is None:
            self.h.uniform_()
            self.p.fill_(-float(self.t.log(self.t.tensor(float(K)))))
        else:
            m = ((mask if mask_bits == 0 else mask & mask_bits).reshape(-1) != 0)
            self.h.copy_(self.t.where(m[:, None, None], self.t.rand_like(self.h), self.h))
            self.p.masked_fill_(m[:, None], -float(self.t.log(self.t.tensor(float(K)))))


def ptxas_report():
    nvcc = os.environ.get("NVCC", "nvcc")
    src = os.path.join(ROOT, "radiation_ppo_b200", "csrc", "rs_pfgru.cu")
    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-fmad=false", "-c",
                            "-Xptxas", "-v", src, "-o", os.path.join(d, "rs_pfgru.o")], capture_output=True, text=True)
    lines, out, name = r.stderr.splitlines(), {}, None
    for ln in lines:
        if "Compiling entry function" in ln:
            name = ln.split("'")[1]
            name = "pfgru_kernel<" + name.split("pfgru_kernelILi")[1].split("EEEv")[0].replace("ELi", ", ") + ">"
        elif name and "spill" in ln:
            out.setdefault(name, {})["spills"] = ln.strip()
        elif name and "Used" in ln and "registers" in ln:
            out.setdefault(name, {})["registers"] = int(ln.split("Used")[1].split("registers")[0])
    return out if out else {"error": r.stderr[-400:]}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("out", help="directory that receives r06_pfgru.json")
    ap.add_argument("--size", choices=sorted(SIZES), default="full")
    args = ap.parse_args()
    sz = SIZES[args.size]

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("pfgru_rollout.py measures on a CUDA device and none was found (no fallback)")
    import radiation_ppo_b200 as rp
    from radteam_epoch import gpu_identity

    from tests import pfgru_ref as ref

    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda:0")
    ident = gpu_identity(torch)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    clock_mhz = float(str(ident["max_sm_clock"]).split()[0]) if ident["max_sm_clock"] else float("nan")
    fma_per_s = sms * 128 * clock_mhz * 1e6

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

    src, dst = torch.empty(1 << 30, dtype=torch.float32, device=dev), torch.empty(1 << 30, dtype=torch.float32, device=dev)
    hbm = 2 * src.numel() * 4 / (events_us(lambda: dst.copy_(src), 20) * 1e-6)
    del src, dst
    torch.cuda.empty_cache()
    fma_row, bytes_row = shape_cost()
    out = {"size": args.size, **ident, "sms": sms, "fp32_fma_bound_per_s": fma_per_s,
           "hbm_measured_bytes_per_s": hbm, "shape": {"d_in": D_IN, "hidden": H, "particles": K, "obs_hidden": W,
                                                      "alpha": ALPHA, "resample": True},
           "fma_per_row": fma_row, "state_bytes_per_row": bytes_row, "ptxas": ptxas_report(),
           "note": "kernel shares of peak: FMAs / FMA bound and bytes / measured HBM bandwidth over the kernel time. The "
                   "state of 131 072 rows (42 MB) fits the 126 MB L2, so back-to-back predicts may read it from there; "
                   "the HBM bound is a floor"}
    print(json.dumps(out), flush=True)

    kern = []
    for n in sz["rows"]:
        mods = ref.modules(D_IN, H, W, seed=0, identity=True, device=dev)
        loc = rp.FusedPFGRU(*mods, num_rows=n, seed=1)
        obs = torch.rand(n, 11, device=dev)
        h0, p0 = loc.particles.clone(), loc.log_weights.clone()
        pred = loc.predict(obs).clone()
        want = ref.step(mods, obs, h0, p0, torch.arange(n, device=dev), 1, 0, K, ALPHA)
        ok = ~want["near"].any(dim=1)
        diffs = {"particles": (loc.particles[ok] - want["h"][ok]).abs().max().item(),
                 "log_weights": (loc.log_weights[ok] - want["p"][ok]).abs().max().item(),
                 "pred": (pred[ok] - want["pred"][ok]).abs().max().item(), "rows_left_out": int((~ok).sum())}
        del want
        tl = TorchPFGRU(torch, mods, n, dev)
        t_f = events_us(lambda: loc.predict(obs), sz["launches"])
        t_t = events_us(lambda: tl.predict(obs), max(20, sz["launches"] // 4))
        f, b = n * fma_row / fma_per_s * 1e6, n * bytes_row / hbm * 1e6
        rec = {"rows": n, "fused_predict_us": t_f, "torch_predict_us": t_t, "speedup_vs_torch": t_t / t_f,
               "fma_per_s": n * fma_row / (t_f * 1e-6), "bytes_per_s": n * bytes_row / (t_f * 1e-6),
               "fma_bound_us": f, "hbm_bound_us": b, "share_of_fma_bound": f / t_f, "share_of_hbm_bound": b / t_f,
               "binding_bound": "fp32 FMA" if f >= b else "HBM", "max_abs_diff_vs_float64": diffs}
        kern.append(rec)
        print(json.dumps(rec), flush=True)
        del loc, tl
        torch.cuda.empty_cache()
    out["kernels"] = kern

    N, T = sz["N"], sz["T"]
    coll = {}
    for which in ("fused", "torch"):
        env = rp.RadSearch(obstruction_count=5, enforce_grid_boundaries=True, num_envs=N, seed=4, device=dev,
                           auto_reset=True, fast_poisson=True, steps_per_episode=120, prefetch=True, use_cuda_graph=True,
                           standardize=1)
        buf = rp.BatchedPPOBuffer(11, T, N, device=dev, predictions=True)
        torch.manual_seed(0)
        gru, pi, v = torch.nn.GRUCell(13, H).to(dev), torch.nn.Linear(H, 8).to(dev), torch.nn.Linear(H, 1).to(dev)
        pol = rp.FusedGruPolicy(gru, pi, v, num_rows=N, seed=4, obs_in=env.obs.view(N, 11),
                                action_out=env.action_buffer.view(N))
        mods = ref.modules(D_IN, H, W, seed=0, identity=True, device=dev)
        loc = rp.FusedPFGRU(*mods, num_rows=N, seed=5) if which == "fused" else TorchPFGRU(torch, mods, N, dev)
        col = rp.RolloutCollector(env, buf, pol, rp.EpisodeStats(N, 1, dev), mode="graph", localizer=loc)
        ms = []
        for _ in range(2):
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); col.collect(); b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
            buf.get()
        coll[which] = {"epoch_ms": ms, "rollout_env_steps_per_s": N * T / (ms[-1] / 1e3), "us_per_rollout_step": 1e3 * ms[-1] / T}
        print(which, json.dumps(coll[which]), flush=True)
        del env, buf, pol, loc, col
        torch.cuda.empty_cache()
    out["collection"] = {"workload": f"{N} envs x T={T}, graph mode, 5 obstructions, enforced bounds, standardize=1, "
                                     "prefetch, fast Poisson, FusedGruPolicy GRUCell(13->24) + linear heads, collect() incl. "
                                     "GAE, second of 2 epochs", **coll}

    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r06_pfgru.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", os.path.join(args.out, "r06_pfgru.json"))


if __name__ == "__main__":
    main()
