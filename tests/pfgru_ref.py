"""TEST INFRASTRUCTURE ONLY -- a float64 torch restatement of one step of the PFGRU localiser (the rules of
include/radsearch_b200.h, RADA2C_core.py:215-307) with the kernel's Philox noise, on any torch device.  Shared by
tests/test_pfgru_cabi.py (host build of the per-row body) and tests/test_gpu_pfgru.py (the kernels)."""
from __future__ import annotations

import copy
import math

import numpy as np
import torch

M32 = 0xFFFFFFFF
DOMAIN = 5
RESAMPLE_BLOCK, PEEK_BLOCK, RESTART_BLOCK = 1024, 2048, 4096
NEAR = 2.0 ** -20          # a draw within NEAR * C_{K-1} of a prefix-sum boundary may pick either side in float32


def modules(d_in, H, W, seed=0, identity=False, device="cpu"):
    """fc_z, fc_r, fc_n, fc_obs, hid_obs as the reference builds them"""
    torch.manual_seed(seed)
    I = H + d_in
    lin = torch.nn.Linear
    hid = [lin(H, W), torch.nn.ReLU(), lin(W, 2)] + ([torch.nn.Identity()] if identity else [])
    return [m.to(device) for m in (lin(I, H), lin(I, H), lin(I, 2 * H), lin(I, 1), torch.nn.Sequential(*hid))]


def packed(mods):
    return torch.cat([p.detach().reshape(-1).float().cpu() for m in mods for p in m.parameters()])


def philox(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 on int64 torch tensors holding uint32 values (the low 64 bits of a product wrap exactly)"""
    c = [c0, c1, c2, c3]
    for _ in range(10):
        p0, p1 = c[0] * 0xD2511F53, c[2] * 0xCD9E8D57
        c = [((p1 >> 32) & M32) ^ c[1] ^ k0, p1 & M32, ((p0 >> 32) & M32) ^ c[3] ^ k1, p0 & M32]
        k0, k1 = (k0 + 0x9E3779B9) & M32, (k1 + 0xBB67AE85) & M32
    return c


def words(row_ids: torch.Tensor, blocks: torch.Tensor, seed: int, ctr: int) -> torch.Tensor:
    """[R, B, 4] int64: the Philox words of rows `row_ids` [R] and blocks `blocks` [B] of domain 5"""
    r = row_ids.to(torch.int64)[:, None].expand(-1, blocks.numel())
    b = (DOMAIN << 24) | blocks.to(device=r.device, dtype=torch.int64)[None, :].expand_as(r)
    f = lambda v: torch.full_like(r, v)                    # noqa: E731
    return torch.stack(philox(r, b, f(ctr & M32), f(ctr >> 32), seed & M32, (seed >> 32) & M32), dim=-1)


def uniform(x: torch.Tensor) -> torch.Tensor:
    return ((x >> 8).double() + 0.5) * 2.0 ** -24


def normals(row_ids, K, H, seed, ctr, blk0=0):
    """[R, K, H] float64 eps of the step: block blk0 + k*16 + j//4, Box-Muller on word pairs"""
    G = (H + 3) // 4
    blocks = torch.tensor([blk0 + k * 16 + g for k in range(K) for g in range(G)], device=row_ids.device)
    u = uniform(words(row_ids, blocks, seed, ctr)).view(-1, K, G, 4)
    r0, r1 = torch.sqrt(-2 * torch.log(u[..., 0])), torch.sqrt(-2 * torch.log(u[..., 2]))
    a0, a1 = 2 * math.pi * u[..., 1], 2 * math.pi * u[..., 3]
    eps = torch.stack([r0 * torch.cos(a0), r0 * torch.sin(a0), r1 * torch.cos(a1), r1 * torch.sin(a1)], dim=-1)
    return eps.view(-1, K, 4 * G)[:, :, :H]


def resample_uniforms(row_ids, K, seed, ctr, blk0=0):
    blocks = torch.arange(blk0 + RESAMPLE_BLOCK, blk0 + RESAMPLE_BLOCK + (K + 3) // 4, device=row_ids.device)
    return uniform(words(row_ids, blocks, seed, ctr)).view(-1, 4 * ((K + 3) // 4))[:, :K]


def restart_state(row_ids, K, H, seed, ctr):
    G = (H + 3) // 4
    blocks = torch.tensor([RESTART_BLOCK + k * 16 + g for k in range(K) for g in range(G)], device=row_ids.device)
    h = uniform(words(row_ids, blocks, seed, ctr)).view(-1, K, 4 * G)[:, :, :H]
    return h, torch.full((h.shape[0], K), -math.log(K), dtype=torch.float64, device=h.device)


def step(mods, obs, h0, p0, row_ids, seed, ctr, K, alpha, resample=True, blk0=0):
    """One step in float64.  obs [R, 11], h0 [R, K, H], p0 [R, K] -> dict(h, p, pred, h1, p1, idx, near): the new state,
    the prediction, the state before resampling, the drawn indices and the draws within NEAR of a boundary ([R, K] bool)."""
    fz, fr, fn, fo, ho = (copy.deepcopy(m).double() for m in mods)
    H = fz.out_features
    d = fz.in_features - H
    R = obs.shape[0]
    x = obs[:, :d].double()[:, None, :].expand(R, K, d)
    h0, p0 = h0.double(), p0.double()
    with torch.no_grad():
        hx = torch.cat([h0, x], dim=-1)
        z, r = torch.sigmoid(fz(hx)), torch.sigmoid(fr(hx))
        nn = fn(torch.cat([r * h0, x], dim=-1))
        mu, nu = nn[..., :H], nn[..., H:]
        eps = normals(row_ids, K, H, seed, ctr, blk0)
        n = torch.tanh(mu + eps * torch.nn.functional.softplus(nu))
        h1 = (1 - z) * n + z * h0
        p1 = torch.log_softmax(fo(torch.cat([h1, x], dim=-1))[..., 0] + p0, dim=1)
        a = float(np.float32(alpha))
        if resample:
            q = a * torch.exp(p1) + (1 - a) / K
            C = torch.cumsum(q, dim=1)
            t = resample_uniforms(row_ids, K, seed, ctr, blk0) * C[:, -1:]
            idx = torch.searchsorted(C, t, right=True).clamp(max=K - 1)
            near = ((t[:, :, None] - C[:, None, :]).abs() < NEAR * C[:, -1:, None]).any(dim=2)
            h = torch.gather(h1, 1, idx[:, :, None].expand(-1, -1, H))
            pi = torch.gather(p1, 1, idx)
            p = pi - torch.log(a * torch.exp(pi) + (1 - a) / K)
            p = p - torch.logsumexp(p, dim=1, keepdim=True)
        else:
            idx = torch.arange(K, device=h1.device)[None].expand(R, K)
            near = torch.zeros(R, K, dtype=torch.bool, device=h1.device)
            h, p = h1, p1
        pred = ho(torch.sum(torch.exp(p)[:, :, None] * h, dim=1))
    return dict(h=h, p=p, pred=pred, h1=h1, p1=p1, idx=idx, near=near)


def close(got, want, atol=1e-5, rtol=1e-5):
    """max of |got - want| / (atol + rtol |want|): <= 1 passes"""
    got, want = torch.as_tensor(got).double(), torch.as_tensor(want).double().to(torch.as_tensor(got).device)
    if got.numel() == 0:
        return 0.0
    return float(((got - want).abs() / (atol + rtol * want.abs())).max())
