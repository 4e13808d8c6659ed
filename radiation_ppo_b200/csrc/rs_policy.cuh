// Per-row body of the fused GRU actor-critic inference (rs_policy.cu): torch.nn.GRUCell(d_in, H) -> policy head over the 8
// moves (log_softmax, Gumbel-max sampling) and value head, one row of the batch per call, in float32.
//
// Compiles as host C++ too (RS_HOST_EMU, tests/emu): the CPU tests compare this body with torch and with the oracle's
// Philox before any GPU time is spent.
//
// Weights arrive in torch's row-major order, packed by the caller:
//   weight_ih [3H][d_in] | weight_hh [3H][H] | bias_ih [3H] | bias_hh [3H] | policy head | value head
//   policy head: P = 0 -> W [8][H], b [8];  P > 0 -> W1 [P][H], b1 [P], W2 [8][P], b2 [8]
//   value head:  V = 0 -> W [1][H], b [1];  V > 0 -> W1 [V][H], b1 [V], W2 [1][V], b2 [1]
// and are staged into a padded table (PolicyLayout) whose rows are whole float4s, zero-filled past their width, so that
// every product reads its weights with 16-byte shared-memory loads that all lanes of a warp share (broadcast).
#pragma once
#ifdef RS_HOST_EMU
#include "cuda_host_shim.h"
#else
#include <cuda_runtime.h>
#endif
#include <math.h>
#include <stdint.h>

#include "../../include/radsearch_b200.h"

namespace rs {

// Philox4x32-10, the generator of rs_device.cuh (which holds out-of-line definitions and so belongs to rs_kernels.cu alone)
__device__ __forceinline__ void policy_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                                              uint32_t out[4]) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

constexpr int kPolicyActions = 8;        // the policy's action space (main.py:545)
constexpr int kPolicyMaxWidth = 64;      // H, P, V in 1..64
constexpr uint32_t kPolicyDomain = 4u;   // Philox counter domain of the action noise (0..3: env step, reset, prefetch)

__host__ __device__ __forceinline__ int round4(int v) { return (v + 3) & ~3; }

// Offsets (floats) of the staged table.  GRU unit j owns one record of RJ floats: for each gate g = r, z, n a row
// [W_ig[j] (DXP) | W_hg[j] (HP)], then [b_ir b_iz b_in 0 | b_hr b_hz b_hn 0].
struct PolicyLayout {
    int d_in, H, P, V, act;
    int DXP, HP, GW, RJ;      // padded input width, padded hidden width, gate row, GRU record
    int pi_off, pi_rec;       // policy head: P = 0 -> [W[k] (HP)] x 8 then b[8]; P > 0 -> [W1[p] (HP) | b1 0 0 0 | W2[0..8][p]] x P, b2[8]
    int v_off, v_rec;         // value head:  V = 0 -> [W (HP) | b 0 0 0];  V > 0 -> [W1[q] (HP) | b1 W2[q] 0 0] x V, [b2 0 0 0]
    int total;                // floats of the staged table
    int count;                // floats of the packed torch buffer
};

__host__ __device__ inline bool policy_layout(const RsPolicyConfig &c, PolicyLayout &L) {
    if ((c.d_in != 11 && c.d_in != 13) || c.hidden < 1 || c.hidden > kPolicyMaxWidth || c.pi_hidden < 0 ||
        c.pi_hidden > kPolicyMaxWidth || c.v_hidden < 0 || c.v_hidden > kPolicyMaxWidth || c.activation < 0 ||
        c.activation > 1)
        return false;
    const int H = c.hidden, P = c.pi_hidden, V = c.v_hidden;
    L.d_in = c.d_in; L.H = H; L.P = P; L.V = V; L.act = c.activation;
    L.DXP = round4(c.d_in);
    L.HP = round4(H);
    L.GW = L.DXP + L.HP;
    L.RJ = 3 * L.GW + 8;
    L.pi_off = H * L.RJ;
    L.pi_rec = P == 0 ? L.HP : L.HP + 4 + kPolicyActions;
    L.v_off = L.pi_off + (P == 0 ? kPolicyActions : P) * L.pi_rec + kPolicyActions;
    L.v_rec = L.HP + 4;
    L.total = L.v_off + (V == 0 ? 1 : V) * L.v_rec + (V == 0 ? 0 : 4);
    L.count = 3 * H * c.d_in + 3 * H * H + 6 * H +
              (P == 0 ? kPolicyActions * H + kPolicyActions : P * H + P + kPolicyActions * P + kPolicyActions) +
              (V == 0 ? H + 1 : V * H + V + V + 1);
    return true;
}

// Where element s of the packed torch buffer goes in the staged table.
__host__ __device__ inline int policy_param_dst(const PolicyLayout &L, int s) {
    const int H = L.H, d = L.d_in;
    if (s < 3 * H * d) { const int row = s / d; return (row % H) * L.RJ + (row / H) * L.GW + s % d; }
    s -= 3 * H * d;
    if (s < 3 * H * H) { const int row = s / H; return (row % H) * L.RJ + (row / H) * L.GW + L.DXP + s % H; }
    s -= 3 * H * H;
    if (s < 3 * H) return (s % H) * L.RJ + 3 * L.GW + s / H;
    s -= 3 * H;
    if (s < 3 * H) return (s % H) * L.RJ + 3 * L.GW + 4 + s / H;
    s -= 3 * H;
    const int P = L.P;
    if (P == 0) {
        if (s < kPolicyActions * H) return L.pi_off + (s / H) * L.pi_rec + s % H;
        s -= kPolicyActions * H;
        if (s < kPolicyActions) return L.pi_off + kPolicyActions * L.pi_rec + s;
        s -= kPolicyActions;
    } else {
        if (s < P * H) return L.pi_off + (s / H) * L.pi_rec + s % H;
        s -= P * H;
        if (s < P) return L.pi_off + s * L.pi_rec + L.HP;
        s -= P;
        if (s < kPolicyActions * P) return L.pi_off + (s % P) * L.pi_rec + L.HP + 4 + s / P;
        s -= kPolicyActions * P;
        if (s < kPolicyActions) return L.pi_off + P * L.pi_rec + s;
        s -= kPolicyActions;
    }
    const int V = L.V;
    if (V == 0) return L.v_off + (s < H ? s : L.HP);
    if (s < V * H) return L.v_off + (s / H) * L.v_rec + s % H;
    s -= V * H;
    if (s < V) return L.v_off + s * L.v_rec + L.HP;
    s -= V;
    if (s < V) return L.v_off + s * L.v_rec + L.HP + 1;
    return L.v_off + V * L.v_rec;
}

__device__ __forceinline__ float policy_sigmoid(float v) { return 1.0f / (1.0f + expf(-v)); }
__device__ __forceinline__ float policy_act_fn(float v, int act) { return act ? fmaxf(v, 0.0f) : tanhf(v); }

// sum_k w[k] * v[k] over the padded width, in float4 steps (zero padding past `width`)
template <int N>
__device__ __forceinline__ float policy_dot(const float *__restrict__ w, const float (&v)[N], int width) {
    const float4 *w4 = reinterpret_cast<const float4 *>(w);
    float a = 0.0f, b = 0.0f;
#pragma unroll
    for (int c = 0; c < N / 4; c++) {
        if (4 * c < width) {
            const float4 q = w4[c];
            a = fmaf(q.x, v[4 * c], a);
            b = fmaf(q.y, v[4 * c + 1], b);
            a = fmaf(q.z, v[4 * c + 2], a);
            b = fmaf(q.w, v[4 * c + 3], b);
        }
    }
    return a + b;
}

// -log(-log u) of u = ((x >> 8) + 0.5) * 2^-24, the Gumbel noise of one Philox word.  -log u is taken as -log1p(u - 1)
// for u >= 1/2, where u - 1 is exact in float32, so that u close to 1 keeps its precision (float32 u would round to 1).
__device__ __forceinline__ float policy_gumbel(uint32_t x) {
    const uint32_t i = x >> 8;
    const float e = i >= (1u << 23) ? -log1pf(-((float)((1u << 24) - i) - 0.5f) * 0x1p-24f)
                                    : -logf(((float)i + 0.5f) * 0x1p-24f);
    return -logf(e);
}

struct PolicyOut {
    int action;
    float logp, value;
};

// One row.  w: the staged table; x: obs row (d_in = 11) with pred appended (d_in = 13); hs / hstride: this row's hidden
// state (H floats, element j at hs[j * hstride]), read as h and overwritten with h' = GRUCell(x, h).  With `act` the
// policy head runs and the action is sampled with the Philox words of (row_id, ctr, seed); the value head always runs.
template <int DXP, int HMAX>
__device__ __forceinline__ PolicyOut policy_row(const PolicyLayout &L, const float *__restrict__ w, const float (&x)[DXP],
                                                float *hs, int hstride, bool act, uint32_t row_id, uint64_t ctr,
                                                uint64_t seed) {
    const int H = L.H, HP = L.HP;
    float h[HMAX];
#pragma unroll
    for (int k = 0; k < HMAX; k++) h[k] = k < H ? hs[k * hstride] : 0.0f;
    // GRUCell (torch's gate order r, z, n): r = s(W_ir x + b_ir + W_hr h + b_hr), z likewise,
    // n = tanh(W_in x + b_in + r (W_hn h + b_hn)), h' = n + z (h - n)
    for (int j = 0; j < H; j++) {
        const float *rec = w + j * L.RJ;
        const float4 bi = *reinterpret_cast<const float4 *>(rec + 3 * L.GW);
        const float4 bh = *reinterpret_cast<const float4 *>(rec + 3 * L.GW + 4);
        const float xr = policy_dot(rec, x, DXP), hr = policy_dot(rec + L.DXP, h, HP);
        const float xz = policy_dot(rec + L.GW, x, DXP), hz = policy_dot(rec + L.GW + L.DXP, h, HP);
        const float xn = policy_dot(rec + 2 * L.GW, x, DXP), hn = policy_dot(rec + 2 * L.GW + L.DXP, h, HP);
        const float r = policy_sigmoid((xr + bi.x) + (hr + bh.x));
        const float z = policy_sigmoid((xz + bi.y) + (hz + bh.y));
        const float n = tanhf((xn + bi.z) + r * (hn + bh.z));
        const float hj = hs[j * hstride];
        hs[j * hstride] = fmaf(z, hj - n, n);
    }
#pragma unroll
    for (int k = 0; k < HMAX; k++) h[k] = k < H ? hs[k * hstride] : 0.0f;   // h'
    PolicyOut o{0, 0.0f, 0.0f};
    // value head
    {
        const float *vw = w + L.v_off;
        if (L.V == 0) {
            o.value = policy_dot(vw, h, HP) + vw[HP];
        } else {
            float v = 0.0f;
            for (int q = 0; q < L.V; q++) {
                const float *rec = vw + q * L.v_rec;
                v = fmaf(rec[HP + 1], policy_act_fn(policy_dot(rec, h, HP) + rec[HP], L.act), v);
            }
            o.value = v + vw[L.V * L.v_rec];
        }
    }
    if (!act) return o;
    // policy head -> logits
    float lg[kPolicyActions];
    const float *pw = w + L.pi_off;
    if (L.P == 0) {
#pragma unroll
        for (int k = 0; k < kPolicyActions; k++) lg[k] = policy_dot(pw + k * L.pi_rec, h, HP) + pw[kPolicyActions * L.pi_rec + k];
    } else {
#pragma unroll
        for (int k = 0; k < kPolicyActions; k++) lg[k] = 0.0f;
        for (int p = 0; p < L.P; p++) {
            const float *rec = pw + p * L.pi_rec;
            const float a = policy_act_fn(policy_dot(rec, h, HP) + rec[HP], L.act);
            const float4 w0 = *reinterpret_cast<const float4 *>(rec + HP + 4);
            const float4 w1 = *reinterpret_cast<const float4 *>(rec + HP + 8);
            lg[0] = fmaf(w0.x, a, lg[0]); lg[1] = fmaf(w0.y, a, lg[1]); lg[2] = fmaf(w0.z, a, lg[2]); lg[3] = fmaf(w0.w, a, lg[3]);
            lg[4] = fmaf(w1.x, a, lg[4]); lg[5] = fmaf(w1.y, a, lg[5]); lg[6] = fmaf(w1.z, a, lg[6]); lg[7] = fmaf(w1.w, a, lg[7]);
        }
#pragma unroll
        for (int k = 0; k < kPolicyActions; k++) lg[k] += pw[L.P * L.pi_rec + k];
    }
    // log_softmax (max-subtracted log-sum-exp)
    float m = lg[0];
#pragma unroll
    for (int k = 1; k < kPolicyActions; k++) m = fmaxf(m, lg[k]);
    float s = 0.0f;
#pragma unroll
    for (int k = 0; k < kPolicyActions; k++) s += expf(lg[k] - m);
    const float lse = m + logf(s);
    // Gumbel-max: the first index of the maximum of logp_k + g_k, g_k from Philox counter (row, 4<<24 | b, ctr), key seed
    uint32_t u[kPolicyActions];
    policy_philox(row_id, kPolicyDomain << 24, (uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)seed, (uint32_t)(seed >> 32), u);
    policy_philox(row_id, (kPolicyDomain << 24) | 1u, (uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)seed,
                  (uint32_t)(seed >> 32), u + 4);
    float best = lg[0] - lse + policy_gumbel(u[0]);
    int a = 0;
#pragma unroll
    for (int k = 1; k < kPolicyActions; k++) {
        const float sc = lg[k] - lse + policy_gumbel(u[k]);
        if (sc > best) { best = sc; a = k; }
    }
    float la = lg[0];
#pragma unroll
    for (int k = 1; k < kPolicyActions; k++) la = a == k ? lg[k] : la;
    o.action = a;
    o.logp = la - lse;
    return o;
}

}  // namespace rs
