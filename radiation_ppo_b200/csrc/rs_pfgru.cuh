// Per-row body of the fused PFGRU source localiser (rs_pfgru.cu): one step of the particle-filter GRU cell of PF-RNN (Ma et
// al. 2020) as RAD-A2C configures it (RADA2C_core.py:215-307: K particles, soft resampling with alpha, tanh), followed by
// the prediction head hid_obs, for one row of the batch, in float32 with explicit FMAs.
//
// One warp owns a row.  Its particles sit on the lanes (particle k on lane k % 32), and everything that crosses particles
// (log-softmax, prefix sums, the resampling gather, the weighted mean) goes through the warp's shared-memory scratch with
// fixed-order sums, so the result does not depend on scheduling.  The body is written as phases between warp barriers;
// under RS_HOST_EMU (tests/emu) the same phases run on the host, each for lane = 0..31 in turn, so the CPU tests check
// this arithmetic before any GPU time is spent.  A value that crosses a phase boundary lives in shared memory.
//
// Per row m, x = obs[m][0 .. d_in), particles h0_k in R^H and log-weights p0_k, k < K ([a | b]: hidden part first):
//   z = s(fc_z[h0 | x]), r = s(fc_r[h0 | x]), (mu, nu) = fc_n[r h0 | x], n = tanh(mu + eps softplus(nu)),
//   h1 = (1 - z) n + z h0, p1 = log_softmax(fc_obs[h1 | x] + p0) over k;
//   resampling: q = alpha exp(p1) + (1 - alpha) / K, i_k = the first i with u_k C_{K-1} < C_i (C the prefix sum of q),
//   h_k = h1_{i_k}, p_k = p1_{i_k} - log(alpha w + (1 - alpha) / K) with w = exp(p1_{i_k}), then p -= logsumexp(p);
//   pred = hid_obs(sum_k exp(p_k) h_k) = W2 relu(W1 mean + b1) + b2.
// A restart sets h_k ~ U[0, 1) per element and p_k = -log K.
//
// Noise: Philox4x32-10 (rs_policy.cuh), key = seed, counter (global row id, 5<<24 | block, ctr lo, ctr hi).  Every word x
// becomes the open uniform u = ((x >> 8) + 0.5) 2^-24.  Block numbers (24 bits), disjoint between the three calls:
//   predict   k*16 + g           eps of particle k, elements 4g .. 4g+3 (Box-Muller: eps_4g = sqrt(-2 ln u0) cos 2pi u1,
//                                eps_4g+1 = sqrt(-2 ln u0) sin 2pi u1, eps_4g+2 / eps_4g+3 the same of u2, u3)
//             1024 + k/4         the resampling uniform u_k = word k % 4
//   peek      2048 + the predict numbering (2048 .. 3087)
//   restart   4096 + k*16 + j/4  element j of particle k = word j % 4
// ctr is the localiser's call counter, advanced by predict alone.
//
// Weights arrive in torch's row-major order, packed by the caller:
//   fc_z.weight [H][H+d] | fc_z.bias [H] | fc_r.* | fc_n.weight [2H][H+d] | fc_n.bias [2H] | fc_obs.weight [1][H+d] |
//   fc_obs.bias [1] | hid_obs[0].weight [W][H] | hid_obs[0].bias [W] | hid_obs[2].weight [2][W] | hid_obs[2].bias [2]
// and are staged into a table (PfgruLayout) whose gate rows are [W_h (HP) | W_x (DXP)], whole float4s zero-filled past
// their width, so that the lanes read each weight with one 16-byte broadcast load.
#pragma once
#ifdef RS_HOST_EMU
#include "cuda_host_shim.h"
#else
#include <cuda_runtime.h>
#endif
#include <math.h>
#include <stdint.h>

#include "../../include/radsearch_b200.h"
#include "rs_policy.cuh"

#ifdef RS_HOST_EMU
// the phases of one warp, run lane by lane on the host
#define RS_PF_LANES for (int lane = 0; lane < 32; lane++)
#define RS_PF_SYNC() ((void)0)
static inline void sincospif(float x, float *s, float *c) {
    *s = (float)sin(M_PI * (double)x);
    *c = (float)cos(M_PI * (double)x);
}
#else
#define RS_PF_LANES for (int lane = (int)(threadIdx.x & 31u), once_ = 1; once_; once_ = 0)
#define RS_PF_SYNC() __syncwarp()
#endif

namespace rs {

constexpr int kPfgruMaxWidth = 64;       // d_in <= 11; H, W, K in 1..64
constexpr uint32_t kPfgruDomain = 5u;    // Philox counter domain (0..3 env step / reset / prefetch, 4 policy actions)
constexpr uint32_t kPfgruResampleBlock = 1024u, kPfgruPeekBlock = 2048u, kPfgruRestartBlock = 4096u;

struct PfgruLayout {
    int d_in, H, K, W, resample;
    float alpha;
    int DXP, HP, GW;              // padded input width, padded hidden width, gate row
    int off_z, off_r, off_n, off_o, off_b, off_w1, off_b1, off_w2, off_b2;
    int total;                    // floats of the staged table (a multiple of 4)
    int count;                    // floats of the packed torch buffer
    int HS;                       // particle stride in the scratch (odd: lane k's slot sits in bank k * HS % 32)
    int scratch;                  // floats of one warp's scratch (a multiple of 4)
};

__host__ __device__ inline bool pfgru_layout(const RsPfgruConfig &c, PfgruLayout &L) {
    if (c.d_in < 1 || c.d_in > 11 || c.hidden < 1 || c.hidden > kPfgruMaxWidth || c.particles < 1 ||
        c.particles > kPfgruMaxWidth || c.obs_hidden < 1 || c.obs_hidden > kPfgruMaxWidth || c.resample < 0 ||
        c.resample > 1 || !(c.alpha > 0.0f && c.alpha <= 1.0f))
        return false;
    const int H = c.hidden, d = c.d_in, K = c.particles, W = c.obs_hidden;
    L.d_in = d; L.H = H; L.K = K; L.W = W; L.resample = c.resample; L.alpha = c.alpha;
    L.DXP = round4(d);
    L.HP = round4(H);
    L.GW = L.HP + L.DXP;
    L.off_z = 0;
    L.off_r = H * L.GW;
    L.off_n = 2 * H * L.GW;
    L.off_o = 4 * H * L.GW;
    L.off_b = L.off_o + L.GW;                       // b_z [HP] | b_r [HP] | b_n [2HP] | b_obs, 3 pad
    L.off_w1 = L.off_b + 4 * L.HP + 4;              // hid_obs[0].weight transposed, [H][W]
    L.off_b1 = L.off_w1 + round4(H * W);
    L.off_w2 = L.off_b1 + round4(W);                // [2][W]
    L.off_b2 = L.off_w2 + round4(2 * W);
    L.total = L.off_b2 + 4;
    L.count = 2 * (H * (H + d) + H) + 2 * H * (H + d) + 2 * H + (H + d) + 1 + W * H + W + 2 * W + 2;
    L.HS = H | 1;
    // hb [K][HS] | rb [K][HS] | sc, ex, p1, cq, cc, pn [K] | idx [K] | mean [H] | hid [W]
    L.scratch = round4(2 * K * L.HS + 7 * K + H + W);
    return true;
}

// Where element s of the packed torch buffer goes in the staged table.
__host__ __device__ inline int pfgru_param_dst(const PfgruLayout &L, int s) {
    const int H = L.H, d = L.d_in, I = H + d, W = L.W;
    auto gate = [&](int base, int e) { const int row = e / I, c = e % I; return base + row * L.GW + (c < H ? c : L.HP + c - H); };
    if (s < H * I) return gate(L.off_z, s);
    s -= H * I;
    if (s < H) return L.off_b + s;
    s -= H;
    if (s < H * I) return gate(L.off_r, s);
    s -= H * I;
    if (s < H) return L.off_b + L.HP + s;
    s -= H;
    if (s < 2 * H * I) return gate(L.off_n, s);
    s -= 2 * H * I;
    if (s < 2 * H) return L.off_b + 2 * L.HP + s;
    s -= 2 * H;
    if (s < I) return gate(L.off_o, s);
    s -= I;
    if (s < 1) return L.off_b + 4 * L.HP;
    s -= 1;
    if (s < W * H) return L.off_w1 + (s % H) * W + s / H;
    s -= W * H;
    if (s < W) return L.off_b1 + s;
    s -= W;
    if (s < 2 * W) return L.off_w2 + s;
    return L.off_b2 + (s - 2 * W);
}

// ((x >> 8) + 0.5) 2^-24 rounded to float32 (to nearest even where it has 25 significant bits)
__device__ __forceinline__ float pfgru_uniform(uint32_t x) { return ((float)(x >> 8) + 0.5f) * 0x1p-24f; }

// four N(0, 1) draws of block `blk` by Box-Muller (see the header comment).  u = (i + 0.5) 2^-24 (i = x >> 8) needs 25
// significant bits for i >= 2^23, so it is never rounded to float32 here: ln u is taken as log1p(-(1 - u)) there, where
// 1 - u = (2^24 - i - 0.5) 2^-24 is exact (sqrt(-2 ln u) near u = 1 would turn the rounding into errors of 1e-5), and the
// angle 2 pi u as 2 pi (2u - 2) in sincospi's units, also exact.
__device__ __forceinline__ void pfgru_normal4(uint32_t row_id, uint32_t blk, uint64_t ctr, uint64_t seed, float e[4]) {
    uint32_t u[4];
    policy_philox(row_id, (kPfgruDomain << 24) | blk, (uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)seed,
                  (uint32_t)(seed >> 32), u);
#pragma unroll
    for (int b = 0; b < 2; b++) {
        const uint32_t i0 = u[2 * b] >> 8, i1 = u[2 * b + 1] >> 8;
        const float ln = i0 >= (1u << 23) ? log1pf(-((float)((1u << 24) - i0) - 0.5f) * 0x1p-24f)
                                          : logf(((float)i0 + 0.5f) * 0x1p-24f);
        const float r = sqrtf(-2.0f * ln);
        const float a = i1 >= (1u << 23) ? -((float)((1u << 24) - i1) - 0.5f) * 0x1p-23f : ((float)i1 + 0.5f) * 0x1p-23f;
        float s, c;
        sincospif(a, &s, &c);
        e[2 * b] = r * c;
        e[2 * b + 1] = r * s;
    }
}

__device__ __forceinline__ uint32_t pfgru_word(uint32_t row_id, uint32_t blk, int word, uint64_t ctr, uint64_t seed) {
    uint32_t u[4];
    policy_philox(row_id, (kPfgruDomain << 24) | blk, (uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)seed,
                  (uint32_t)(seed >> 32), u);
    return u[word];
}

// the first i in [0, K) with t < C_i (C non-decreasing); K - 1 when there is none
__device__ __forceinline__ int pfgru_pick(const float *C, int K, float t) {
    int lo = 0, hi = K - 1;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (t < C[mid]) hi = mid; else lo = mid + 1;
    }
    return lo;
}

__device__ __forceinline__ float pfgru_sigmoid(float v) { return 1.0f / (1.0f + expf(-v)); }
__device__ __forceinline__ float pfgru_softplus(float v) { return v > 20.0f ? v : log1pf(expf(v)); }

// One particle: hk (H floats of the scratch) holds h0 on entry and h1 on return, rk (H floats) receives r h0; returns
// fc_obs[h1 | x].  The input vectors sit in registers (h0, then r h0: indexed at compile time inside the dots); the outputs
// go four at a time, one Philox block per group of four.
template <int DXP, int HMAX>
__device__ __forceinline__ float pfgru_particle(const PfgruLayout &L, const float *__restrict__ w, const float (&x)[DXP],
                                                float *hk, float *rk, int k, uint32_t row_id, uint32_t blk0, uint64_t ctr,
                                                uint64_t seed) {
    const int H = L.H, HP = L.HP;
    float h[HMAX];
#pragma unroll
    for (int c = 0; c < HMAX; c++) h[c] = c < H ? hk[c] : 0.0f;
#pragma unroll 1
    for (int j0 = 0; j0 < H; j0 += 4) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int j = j0 + i;
            if (j < H) {
                const float *row = w + L.off_r + j * L.GW;
                const float r = pfgru_sigmoid(policy_dot(row, h, HP) + policy_dot(row + HP, x, DXP) + w[L.off_b + HP + j]);
                rk[j] = r * hk[j];
            }
        }
    }
    float rh[HMAX];
#pragma unroll
    for (int c = 0; c < HMAX; c++) rh[c] = c < H ? rk[c] : 0.0f;
#pragma unroll 1
    for (int j0 = 0; j0 < H; j0 += 4) {
        float eps[4];
        pfgru_normal4(row_id, blk0 + (uint32_t)(k * 16 + j0 / 4), ctr, seed, eps);
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int j = j0 + i;
            if (j < H) {
                const float *zr = w + L.off_z + j * L.GW, *mr = w + L.off_n + j * L.GW, *nr = w + L.off_n + (H + j) * L.GW;
                const float z = pfgru_sigmoid(policy_dot(zr, h, HP) + policy_dot(zr + HP, x, DXP) + w[L.off_b + j]);
                const float mu = policy_dot(mr, rh, HP) + policy_dot(mr + HP, x, DXP) + w[L.off_b + 2 * HP + j];
                const float nu = policy_dot(nr, rh, HP) + policy_dot(nr + HP, x, DXP) + w[L.off_b + 2 * HP + H + j];
                const float n = tanhf(fmaf(eps[i], pfgru_softplus(nu), mu));
                hk[j] = fmaf(z, hk[j] - n, n);
            }
        }
    }
#pragma unroll
    for (int c = 0; c < HMAX; c++) h[c] = c < H ? hk[c] : 0.0f;
    const float *orow = w + L.off_o;
    return policy_dot(orow, h, HP) + policy_dot(orow + HP, x, DXP) + w[L.off_b + 4 * HP];
}

// One row, by one warp.  s: the warp's scratch (L.scratch floats); part [K][H] / logw [K]: the row's state, read, and
// written back when write_state; pred: the row's two outputs.  blk0: 0 for predict, kPfgruPeekBlock for peek.
template <int DXP, int HMAX>
__device__ __forceinline__ void pfgru_row(const PfgruLayout &L, const float *__restrict__ w, float *s,
                                          const float *__restrict__ obs_row, float *part, float *logw, float *pred,
                                          bool write_state, uint32_t row_id, uint32_t blk0, uint64_t ctr, uint64_t seed) {
    const int H = L.H, K = L.K, HS = L.HS;
    float *hb = s, *rb = hb + K * HS, *sc = rb + K * HS, *ex = sc + K, *p1 = ex + K, *cq = p1 + K, *cc = cq + K, *pn = cc + K;
    int *idx = reinterpret_cast<int *>(pn + K);
    float *mb = reinterpret_cast<float *>(idx + K), *hid = mb + H;
    RS_PF_LANES {                                  // the state into the scratch, coalesced
        for (int e = lane; e < K * H; e += 32) hb[(e / H) * HS + e % H] = part[e];
        for (int k = lane; k < K; k += 32) sc[k] = logw[k];
    }
    RS_PF_SYNC();
    RS_PF_LANES {                                  // steps 1-4: h1 in place, sc = fc_obs[h1 | x] + p0
        float x[DXP];
#pragma unroll
        for (int c = 0; c < DXP; c++) x[c] = c < L.d_in ? obs_row[c] : 0.0f;
        for (int k = lane; k < K; k += 32)
            sc[k] += pfgru_particle<DXP, HMAX>(L, w, x, hb + k * HS, rb + k * HS, k, row_id, blk0, ctr, seed);
    }
    RS_PF_SYNC();
    RS_PF_LANES {
        float m = sc[0];
        for (int i = 1; i < K; i++) m = fmaxf(m, sc[i]);
        for (int k = lane; k < K; k += 32) ex[k] = expf(sc[k] - m);
    }
    RS_PF_SYNC();
    RS_PF_LANES {                                  // p1 = log_softmax(sc); q
        float m = sc[0], S = 0.0f;
        for (int i = 1; i < K; i++) m = fmaxf(m, sc[i]);
        for (int i = 0; i < K; i++) S += ex[i];
        const float lse = m + logf(S), a = L.alpha, b = (1.0f - L.alpha) / (float)K;
        for (int k = lane; k < K; k += 32) {
            p1[k] = sc[k] - lse;
            cq[k] = fmaf(a, expf(p1[k]), b);
        }
    }
    RS_PF_SYNC();
    if (L.resample) {
        RS_PF_LANES {                              // C_i = q_0 + ... + q_i, in particle order
            for (int i = lane; i < K; i += 32) {
                float c = 0.0f;
                for (int k = 0; k <= i; k++) c += cq[k];
                cc[i] = c;
            }
        }
        RS_PF_SYNC();
        RS_PF_LANES {                              // step 5: draw, gather index, corrected log-weight
            const float a = L.alpha, b = (1.0f - L.alpha) / (float)K, total = cc[K - 1];
            for (int k = lane; k < K; k += 32) {
                const float u = pfgru_uniform(pfgru_word(row_id, blk0 + kPfgruResampleBlock + (uint32_t)(k / 4), k % 4, ctr, seed));
                const int i = pfgru_pick(cc, K, u * total);
                idx[k] = i;
                pn[k] = p1[i] - logf(fmaf(a, expf(p1[i]), b));
            }
        }
    } else {
        RS_PF_LANES {
            for (int k = lane; k < K; k += 32) { idx[k] = k; pn[k] = p1[k]; }
        }
    }
    RS_PF_SYNC();
    RS_PF_LANES {
        float m = pn[0];
        for (int i = 1; i < K; i++) m = fmaxf(m, pn[i]);
        for (int k = lane; k < K; k += 32) ex[k] = expf(pn[k] - m);
    }
    RS_PF_SYNC();
    RS_PF_LANES {                                  // p = pn - logsumexp(pn), weight exp(p)
        float m = pn[0], S = 0.0f;
        for (int i = 1; i < K; i++) m = fmaxf(m, pn[i]);
        for (int i = 0; i < K; i++) S += ex[i];
        const float lse = m + logf(S);
        for (int k = lane; k < K; k += 32) {
            sc[k] = pn[k] - lse;
            cq[k] = expf(sc[k]);
        }
    }
    RS_PF_SYNC();
    RS_PF_LANES {                                  // step 6: weighted mean of the new particles; the new state out
        for (int j = lane; j < H; j += 32) {
            float v = 0.0f;
            for (int k = 0; k < K; k++) v = fmaf(cq[k], hb[idx[k] * HS + j], v);
            mb[j] = v;
        }
        if (write_state) {
            for (int e = lane; e < K * H; e += 32) part[e] = hb[idx[e / H] * HS + e % H];
            for (int k = lane; k < K; k += 32) logw[k] = sc[k];
        }
    }
    RS_PF_SYNC();
    RS_PF_LANES {                                  // hid_obs: Linear(H, W) -> ReLU
        const int W = L.W;
        for (int q = lane; q < W; q += 32) {
            float v = 0.0f;
            for (int j = 0; j < H; j++) v = fmaf(w[L.off_w1 + j * W + q], mb[j], v);
            hid[q] = fmaxf(v + w[L.off_b1 + q], 0.0f);
        }
    }
    RS_PF_SYNC();
    RS_PF_LANES {                                  // -> Linear(W, 2)
        if (lane < 2) {
            const int W = L.W;
            float v = 0.0f;
            for (int q = 0; q < W; q++) v = fmaf(w[L.off_w2 + lane * W + q], hid[q], v);
            pred[lane] = v + w[L.off_b2 + lane];
        }
    }
    RS_PF_SYNC();
}

// Step 7 for one row: h ~ U[0, 1) per element, p = -log K.
__device__ __forceinline__ void pfgru_restart_row(const PfgruLayout &L, float *part, float *logw, uint32_t row_id,
                                                  uint64_t ctr, uint64_t seed) {
    const int H = L.H, K = L.K;
    RS_PF_LANES {
        for (int e = lane; e < K * H; e += 32) {
            const int k = e / H, j = e % H;
            part[e] = pfgru_uniform(pfgru_word(row_id, kPfgruRestartBlock + (uint32_t)(k * 16 + j / 4), j % 4, ctr, seed));
        }
        const float p = -logf((float)K);
        for (int k = lane; k < K; k += 32) logw[k] = p;
    }
}

}  // namespace rs
