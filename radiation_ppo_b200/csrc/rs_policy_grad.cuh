// Per-step math of the fused PPO loss and gradient of the GRU actor-critic (rs_policy_grad.cu): the forward step of one
// rollout column, and the backward step that recomputes that step's gates and heads from the stored hidden states and
// leaves the factors of its weight-gradient outer products in the column's scratch.
//
// Compiles as host C++ too (RS_HOST_EMU, tests/emu/policy_grad_emu.cpp): the CPU tests run whole columns through these
// functions and compare with float64 torch autograd.  On the device one warp owns a column and calls every function with
// (i0, is) = (lane, 32); the host calls them with (0, 1).  pg_sync() orders the phases of a column (__syncwarp).
//
// Column scratch (floats from the column's base, every block a whole number of float4s, zero past its width):
//   U  [x (DXP) | h_{t-1} as the cell read it (HP) | h_t (HP) | a_pi (P) | a_v (V) | 1 0 0 0]   inputs of the products
//   F  [da_r | da_z | da_n | dg (HP each) | dlogit (8) | dpre_pi (P) | dv 0 0 0 | dpre_v (V)]    their factors
//   S  [dh_direct (HP) | carry (HP) | logits (8) | value 0 0 0]
// Packed parameter s accumulates sum over (t, column) of F[f(s)] * U[u(s)] (grad_entry), so the weight gradient of a
// step is one fixed pass over the parameters, whatever the config.
#pragma once
#include "rs_policy.cuh"

namespace rs {

constexpr int kGradStats = 6;   // sum -min(surr), sum (v - ret)^2, sum (logp_old - logp), sum entropy, clipped rows, skipped rows

#ifdef RS_HOST_EMU
inline void pg_sync() {}
#else
__device__ __forceinline__ void pg_sync() { __syncwarp(); }
#endif

struct GradLayout {
    int ux, uhp, uh, uapi, uav, uone;            // U
    int far, faz, fan, fg, fdlg, fdpi, fdv, fdpv; // F
    int sdh, scarry, slg;                        // S
    int CW;                                      // column stride
};

__host__ __device__ inline void grad_layout(const PolicyLayout &L, GradLayout &G) {
    const int HP = L.HP;
    G.ux = 0;
    G.uhp = L.DXP;
    G.uh = G.uhp + HP;
    G.uapi = G.uh + HP;
    G.uav = G.uapi + round4(L.P);
    G.uone = G.uav + round4(L.V);
    G.far = G.uone + 4;
    G.faz = G.far + HP;
    G.fan = G.faz + HP;
    G.fg = G.fan + HP;
    G.fdlg = G.fg + HP;
    G.fdpi = G.fdlg + kPolicyActions;
    G.fdv = G.fdpi + round4(L.P);
    G.fdpv = G.fdv + 4;
    G.sdh = G.fdpv + round4(L.V);
    G.scarry = G.sdh + HP;
    G.slg = G.scarry + HP;
    G.CW = G.slg + 12;
}

// (f << 16) | u of packed parameter s: its gradient is the sum of F[f] * U[u] (offsets from the column's base)
__host__ __device__ inline uint32_t grad_entry(const PolicyLayout &L, const GradLayout &G, int s) {
    const int H = L.H, d = L.d_in;
    // gate g = r, z, n of the input side (da_r, da_z, da_n) and of the hidden side (da_r, da_z, dg)
    auto gi = [&](int g) { return g == 0 ? G.far : g == 1 ? G.faz : G.fan; };
    auto gh = [&](int g) { return g == 0 ? G.far : g == 1 ? G.faz : G.fg; };
    int f, u;
    if (s < 3 * H * d) {
        f = gi(s / d / H) + (s / d) % H; u = G.ux + s % d;
    } else if ((s -= 3 * H * d) < 3 * H * H) {
        f = gh(s / H / H) + (s / H) % H; u = G.uhp + s % H;
    } else if ((s -= 3 * H * H) < 3 * H) {
        f = gi(s / H) + s % H; u = G.uone;
    } else if ((s -= 3 * H) < 3 * H) {
        f = gh(s / H) + s % H; u = G.uone;
    } else {
        s -= 3 * H;
        const int P = L.P, V = L.V, A = kPolicyActions;
        const int pi = P == 0 ? A * H + A : P * H + P + A * P + A;
        if (s < pi) {
            if (P == 0) {
                if (s < A * H) { f = G.fdlg + s / H; u = G.uh + s % H; } else { f = G.fdlg + s - A * H; u = G.uone; }
            } else if (s < P * H) {
                f = G.fdpi + s / H; u = G.uh + s % H;
            } else if ((s -= P * H) < P) {
                f = G.fdpi + s; u = G.uone;
            } else if ((s -= P) < A * P) {
                f = G.fdlg + s / P; u = G.uapi + s % P;
            } else {
                f = G.fdlg + s - A * P; u = G.uone;
            }
        } else {
            s -= pi;
            if (V == 0) {
                f = G.fdv; u = s < H ? G.uh + s : G.uone;
            } else if (s < V * H) {
                f = G.fdpv + s / H; u = G.uh + s % H;
            } else if ((s -= V * H) < V) {
                f = G.fdpv + s; u = G.uone;
            } else if ((s -= V) < V) {
                f = G.fdv; u = G.uav + s;
            } else {
                f = G.fdv; u = G.uone;
            }
        }
    }
    return ((uint32_t)f << 16) | (uint32_t)u;
}

// one step's row of the rollout
struct PgRow {
    float act, adv, ret, logp_old;
};
// loss constants: clip bounds as torch.clamp sees them in float32, w_pi / (T M), 2 w_v / (T M)
struct PgConsts {
    float lo, hi, kpi, kv;
};

template <int N>
__device__ __forceinline__ void pg_load(const float *__restrict__ src, float (&v)[N]) {
    const float4 *s4 = reinterpret_cast<const float4 *>(src);
#pragma unroll
    for (int c = 0; c < N / 4; c++) {
        const float4 q = s4[c];
        v[4 * c] = q.x; v[4 * c + 1] = q.y; v[4 * c + 2] = q.z; v[4 * c + 3] = q.w;
    }
}

struct GruGates {
    float r, z, n, g;   // g = W_hn h + b_hn, the term r scales
};

// unit j of torch's GRUCell with the expressions of policy_row, so that the forward pass reproduces rs_policy_act's h'
template <int DXP, int HMAX>
__device__ __forceinline__ GruGates pg_gates(const PolicyLayout &L, const float *__restrict__ w, const float (&x)[DXP],
                                             const float (&h)[HMAX], int j) {
    const float *rec = w + j * L.RJ;
    const float4 bi = *reinterpret_cast<const float4 *>(rec + 3 * L.GW);
    const float4 bh = *reinterpret_cast<const float4 *>(rec + 3 * L.GW + 4);
    const float xr = policy_dot(rec, x, DXP), hr = policy_dot(rec + L.DXP, h, L.HP);
    const float xz = policy_dot(rec + L.GW, x, DXP), hz = policy_dot(rec + L.GW + L.DXP, h, L.HP);
    const float xn = policy_dot(rec + 2 * L.GW, x, DXP), hn = policy_dot(rec + 2 * L.GW + L.DXP, h, L.HP);
    GruGates o;
    o.r = policy_sigmoid((xr + bi.x) + (hr + bh.x));
    o.z = policy_sigmoid((xz + bi.y) + (hz + bh.y));
    o.g = hn + bh.z;
    o.n = tanhf((xn + bi.z) + o.r * o.g);
    return o;
}

// U.x <- [obs | pred | 0], U.h_{t-1} <- hprev (NULL: zeros, the restart), U.h_t <- ht (NULL: left alone)
template <int DXP>
__device__ __forceinline__ void pg_inputs(const PolicyLayout &L, const GradLayout &G, float *col, const float *obs,
                                          const float *pred, const float *hprev, const float *ht, int i0, int is) {
    for (int k = i0; k < DXP; k += is)
        col[G.ux + k] = k < RS_OBS_DIM ? obs[k] : k < L.d_in ? pred[k - RS_OBS_DIM] : 0.0f;
    for (int k = i0; k < L.H; k += is) {
        col[G.uhp + k] = hprev ? hprev[k] : 0.0f;
        if (ht) col[G.uh + k] = ht[k];
    }
}

// forward cell: U.h_t <- GRUCell(U.x, U.h_{t-1}), also to hout (the workspace row of step t)
template <int DXP, int HMAX>
__device__ __forceinline__ void pg_cell(const PolicyLayout &L, const GradLayout &G, const float *__restrict__ w, float *col,
                                        float *hout, int i0, int is) {
    float x[DXP], h[HMAX];
    pg_load(col + G.ux, x);
    pg_load(col + G.uhp, h);
    for (int j = i0; j < L.H; j += is) {
        const GruGates q = pg_gates<DXP, HMAX>(L, w, x, h, j);
        const float hj = fmaf(q.z, col[G.uhp + j] - q.n, q.n);
        col[G.uh + j] = hj;
        hout[j] = hj;
    }
}

// heads from U.h_t: the hidden layers (a_pi, a_v), then the 8 logits and the value into S
template <int HMAX>
__device__ __forceinline__ void pg_heads(const PolicyLayout &L, const GradLayout &G, const float *__restrict__ w, float *col,
                                         int i0, int is) {
    float h[HMAX];
    pg_load(col + G.uh, h);
    const int HP = L.HP, P = L.P, V = L.V;
    const float *pw = w + L.pi_off, *vw = w + L.v_off;
    for (int i = i0; i < P + V; i += is) {
        if (i < P) {
            const float *rec = pw + i * L.pi_rec;
            col[G.uapi + i] = policy_act_fn(policy_dot(rec, h, HP) + rec[HP], L.act);
        } else {
            const float *rec = vw + (i - P) * L.v_rec;
            col[G.uav + i - P] = policy_act_fn(policy_dot(rec, h, HP) + rec[HP], L.act);
        }
    }
    pg_sync();
    for (int k = i0; k <= kPolicyActions; k += is) {
        float o;
        if (k < kPolicyActions) {
            if (P == 0) {
                o = policy_dot(pw + k * L.pi_rec, h, HP) + pw[kPolicyActions * L.pi_rec + k];
            } else {
                o = 0.0f;
                for (int p = 0; p < P; p++) o = fmaf(pw[p * L.pi_rec + HP + 4 + k], col[G.uapi + p], o);
                o += pw[P * L.pi_rec + k];
            }
        } else if (V == 0) {
            o = policy_dot(vw, h, HP) + vw[HP];
        } else {
            o = 0.0f;
            for (int q = 0; q < V; q++) o = fmaf(vw[q * L.v_rec + HP + 1], col[G.uav + q], o);
            o += vw[V * L.v_rec];
        }
        col[G.slg + k] = o;
    }
}

// The loss of one row from the logits and value in S: its diagnostics into st, and dL/dlogit, dL/dv into F.  A row whose
// action is outside 0..7 contributes nothing (zero factors) and is counted.  Gradient conventions of torch autograd:
// minimum splits a tie evenly (inside the clip range ratio * A == clamp(ratio) * A, so both halves carry A there), clamp
// passes the gradient on the closed interval.  logp is policy_row's, so fresh weights give ratio 1 exactly.  Returns
// (logp, ratio) of the row, NaN for a skipped one.
struct PgLossOut {
    float lp, ratio;
};
__device__ __forceinline__ PgLossOut pg_loss(const GradLayout &G, float *col, const PgRow &r, const PgConsts &k, double *st) {
    float *dlg = col + G.fdlg;
    if (!(r.act > -1.0f && r.act < (float)kPolicyActions)) {   // also NaN; otherwise truncated like torch's .long()
        for (int i = 0; i < kPolicyActions; i++) dlg[i] = 0.0f;
        col[G.fdv] = 0.0f;
        st[5] += 1.0;
        return PgLossOut{NAN, NAN};
    }
    const int a = (int)r.act;
    const float *lg = col + G.slg;
    float m = lg[0];
    for (int i = 1; i < kPolicyActions; i++) m = fmaxf(m, lg[i]);
    float s = 0.0f;
    for (int i = 0; i < kPolicyActions; i++) s += expf(lg[i] - m);
    const float lse = m + logf(s);
    const float lp = lg[a] - lse;
    const float ratio = expf(lp - r.logp_old);
    const float s1 = ratio * r.adv, s2 = fminf(fmaxf(ratio, k.lo), k.hi) * r.adv;
    const float g1 = s1 < s2 ? 1.0f : s1 == s2 ? 0.5f : 0.0f;
    const bool inside = ratio >= k.lo && ratio <= k.hi;
    const float dratio = -(g1 * r.adv + (inside ? (1.0f - g1) * r.adv : 0.0f));
    const float glp = k.kpi * dratio * ratio;
    double ent = 0.0;
    for (int i = 0; i < kPolicyActions; i++) {
        const float li = lg[i] - lse, p = expf(li);
        ent -= (double)p * (double)li;
        dlg[i] = (i == a ? glp : 0.0f) - p * glp;
    }
    const float diff = lg[kPolicyActions] - r.ret;
    col[G.fdv] = k.kv * diff;
    st[0] -= (double)fminf(s1, s2);
    st[1] += (double)diff * (double)diff;
    st[2] += (double)r.logp_old - (double)lp;
    st[3] += ent;
    st[4] += (ratio < k.lo || ratio > k.hi) ? 1.0 : 0.0;
    return PgLossOut{lp, ratio};
}

__device__ __forceinline__ float pg_act_grad(float a, int act) { return act ? (a > 0.0f ? 1.0f : 0.0f) : 1.0f - a * a; }

// hidden head layers: dpre = (W2^T dlogit or W2 dv) * act'(a)
__device__ __forceinline__ void pg_heads_back(const PolicyLayout &L, const GradLayout &G, const float *__restrict__ w,
                                              float *col, int i0, int is) {
    const int HP = L.HP, P = L.P, V = L.V;
    for (int i = i0; i < P + V; i += is) {
        if (i < P) {
            const float *rec = w + L.pi_off + i * L.pi_rec + HP + 4;
            float d = 0.0f;
            for (int k = 0; k < kPolicyActions; k++) d = fmaf(rec[k], col[G.fdlg + k], d);
            col[G.fdpi + i] = d * pg_act_grad(col[G.uapi + i], L.act);
        } else {
            const int q = i - P;
            col[G.fdpv + q] = col[G.fdv] * w[L.v_off + q * L.v_rec + HP + 1] * pg_act_grad(col[G.uav + q], L.act);
        }
    }
}

// unit j: delta = dL/dh_t (heads + the carry from step t+1), then the cell's backward from the recomputed gates:
// F.da_r, da_z, da_n, dg, and S.dh_direct = delta z
template <int DXP, int HMAX>
__device__ __forceinline__ void pg_cell_back(const PolicyLayout &L, const GradLayout &G, const float *__restrict__ w,
                                             float *col, int i0, int is) {
    float x[DXP], h[HMAX];
    pg_load(col + G.ux, x);
    pg_load(col + G.uhp, h);
    const int P = L.P, V = L.V;
    const float *pw = w + L.pi_off, *vw = w + L.v_off;
    for (int j = i0; j < L.H; j += is) {
        float d = col[G.scarry + j];
        if (P == 0) {
            for (int k = 0; k < kPolicyActions; k++) d = fmaf(pw[k * L.pi_rec + j], col[G.fdlg + k], d);
        } else {
            for (int p = 0; p < P; p++) d = fmaf(pw[p * L.pi_rec + j], col[G.fdpi + p], d);
        }
        if (V == 0) {
            d = fmaf(vw[j], col[G.fdv], d);
        } else {
            for (int q = 0; q < V; q++) d = fmaf(vw[q * L.v_rec + j], col[G.fdpv + q], d);
        }
        const GruGates q = pg_gates<DXP, HMAX>(L, w, x, h, j);
        const float dn = d * (1.0f - q.z), dz = d * (col[G.uhp + j] - q.n);
        const float dan = dn * (1.0f - q.n * q.n);
        const float dg = dan * q.r;
        const float dar = dan * q.g * (q.r * (1.0f - q.r));
        const float daz = dz * (q.z * (1.0f - q.z));
        col[G.far + j] = dar;
        col[G.faz + j] = daz;
        col[G.fan + j] = dan;
        col[G.fg + j] = dg;
        col[G.sdh + j] = d * q.z;
    }
}

// carry to step t-1: dh_direct + W_hr^T da_r + W_hz^T da_z + W_hn^T dg, zero where the cell restarted (keep = 0)
__device__ __forceinline__ void pg_carry(const PolicyLayout &L, const GradLayout &G, const float *__restrict__ w, float *col,
                                         bool keep, int i0, int is) {
    const int H = L.H;
    for (int k = i0; k < H; k += is) {
        float a = col[G.sdh + k], b = 0.0f, c = 0.0f;
        for (int j = 0; j < H; j++) {
            const float *rec = w + j * L.RJ + L.DXP + k;
            a = fmaf(rec[0], col[G.far + j], a);
            b = fmaf(rec[L.GW], col[G.faz + j], b);
            c = fmaf(rec[2 * L.GW], col[G.fg + j], c);
        }
        col[G.scarry + k] = keep ? a + b + c : 0.0f;
    }
}

}  // namespace rs
