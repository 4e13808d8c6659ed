// TEST INFRASTRUCTURE ONLY -- host build of the fused PPO gradient's per-step math (radiation_ppo_b200/csrc/
// rs_policy_grad.cuh): whole columns run forward and backward through the same functions the kernel's warps call, one
// column at a time with (i0, is) = (0, 1), and the weight gradient summed in float64 from the same (factor, input) pairs.
// Used by tests/test_policy_grad_cabi.py to compare the kernel math with float64 torch autograd where no GPU exists.
#define RS_HOST_EMU 1
#include "../../radiation_ppo_b200/csrc/rs_policy_grad.cuh"

#include <vector>

template <int DXP, int HMAX>
static void columns_body(const rs::PolicyLayout &L, const rs::GradLayout &G, const float *w, const float *obs,
                         const float *pred, const float *act, const float *adv, const float *ret, const float *logp,
                         const uint8_t *end, const int32_t *columns, int T, int N, int M, const rs::PgConsts &k,
                         double *grad, double *stats, float *lp_out, float *ratio_out) {
    const int H = L.H;
    std::vector<uint32_t> entry(L.count);
    for (int s = 0; s < L.count; s++) entry[s] = rs::grad_entry(L, G, s);
    std::vector<float4> buf((G.CW + 3) / 4);
    float *col = reinterpret_cast<float *>(buf.data());
    std::vector<float> hs((size_t)T * H);
    for (int m = 0; m < M; m++) {
        const int n = columns ? columns[m] : m;
        if (n < 0 || n >= N) {
            stats[5] += T;
            continue;
        }
        for (int i = 0; i < G.CW; i++) col[i] = 0.0f;
        col[G.uone] = 1.0f;
        for (int t = 0; t < T; t++) {
            const size_t row = (size_t)t * N + n;
            const bool keep = t > 0 && end[row - N] == 0;
            rs::pg_inputs<DXP>(L, G, col, obs + row * RS_OBS_DIM, pred ? pred + row * 2 : nullptr, keep ? col + G.uh : nullptr,
                               nullptr, 0, 1);
            rs::pg_cell<DXP, HMAX>(L, G, w, col, hs.data() + (size_t)t * H, 0, 1);
        }
        for (int t = T - 1; t >= 0; t--) {
            const size_t row = (size_t)t * N + n;
            const bool keep = t > 0 && end[row - N] == 0;
            const float *ht = hs.data() + (size_t)t * H;
            rs::pg_inputs<DXP>(L, G, col, obs + row * RS_OBS_DIM, pred ? pred + row * 2 : nullptr, keep ? ht - H : nullptr, ht,
                               0, 1);
            rs::pg_heads<HMAX>(L, G, w, col, 0, 1);
            const rs::PgLossOut o = rs::pg_loss(G, col, rs::PgRow{act[row], adv[row], ret[row], logp[row]}, k, stats);
            if (lp_out) lp_out[(size_t)t * M + m] = o.lp;
            if (ratio_out) ratio_out[(size_t)t * M + m] = o.ratio;
            rs::pg_heads_back(L, G, w, col, 0, 1);
            rs::pg_cell_back<DXP, HMAX>(L, G, w, col, 0, 1);
            rs::pg_carry(L, G, w, col, keep, 0, 1);
            for (int s = 0; s < L.count; s++) grad[s] += (double)col[entry[s] >> 16] * (double)col[entry[s] & 0xFFFFu];
        }
    }
}

// grad (float64, count) and stats (6 doubles) are overwritten; lp_out / ratio_out ([T][M], nullable) get each row's
// logp and ratio (NaN where the row is skipped or its column is out of range: left untouched)
extern "C" int emu_policy_grad(const RsPolicyConfig *cfg, const float *params, const float *obs, const float *pred,
                               const float *act, const float *adv, const float *ret, const float *logp, const uint8_t *end,
                               const int32_t *columns, int T, int N, int M, double clip_ratio, double w_pi, double w_v,
                               double *grad, double *stats, float *lp_out, float *ratio_out) {
    rs::PolicyLayout L;
    if (!rs::policy_layout(*cfg, L)) return -1;
    rs::GradLayout G;
    rs::grad_layout(L, G);
    std::vector<float4> table((L.total + 3) / 4, float4{0.0f, 0.0f, 0.0f, 0.0f});
    float *w = reinterpret_cast<float *>(table.data());
    for (int s = 0; s < L.count; s++) w[rs::policy_param_dst(L, s)] = params[s];
    const double c = 1.0 / ((double)T * (double)M);
    const rs::PgConsts k{(float)(1.0 - clip_ratio), (float)(1.0 + clip_ratio), (float)(w_pi * c), (float)(2.0 * w_v * c)};
    for (int s = 0; s < L.count; s++) grad[s] = 0.0;
    for (int q = 0; q < rs::kGradStats; q++) stats[q] = 0.0;
#define RS_EMU_COLS(DXP_, HMAX_) \
    columns_body<DXP_, HMAX_>(L, G, w, obs, pred, act, adv, ret, logp, end, columns, T, N, M, k, grad, stats, lp_out, ratio_out)
    if (L.d_in == 11) {
        if (L.H <= 16) RS_EMU_COLS(12, 16); else if (L.H <= 32) RS_EMU_COLS(12, 32); else RS_EMU_COLS(12, 64);
    } else {
        if (L.H <= 16) RS_EMU_COLS(16, 16); else if (L.H <= 32) RS_EMU_COLS(16, 32); else RS_EMU_COLS(16, 64);
    }
#undef RS_EMU_COLS
    return 0;
}

// the (factor, input) pair of every packed parameter, so that a test can check that no two parameters share one
extern "C" int emu_grad_entries(const RsPolicyConfig *cfg, uint32_t *entry) {
    rs::PolicyLayout L;
    if (!rs::policy_layout(*cfg, L)) return -1;
    rs::GradLayout G;
    rs::grad_layout(L, G);
    for (int s = 0; s < L.count; s++) entry[s] = rs::grad_entry(L, G, s);
    return G.CW;
}
