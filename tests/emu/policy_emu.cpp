// TEST INFRASTRUCTURE ONLY -- host build of the fused policy's per-row body (radiation_ppo_b200/csrc/rs_policy.cuh): the
// staging of the packed weights and one loop iteration per CUDA thread, on host memory.  Used by tests/test_policy_cabi.py
// to compare the kernel math with torch on the CPU and the sampling with the oracle's Philox where no GPU exists.
#define RS_HOST_EMU 1
#include "../../radiation_ppo_b200/csrc/rs_policy.cuh"

#include <vector>

template <int DXP, int HMAX>
static void rows_body(const rs::PolicyLayout &L, const float *w, const float *obs, const float *pred, float *hidden,
                      int32_t *action, float *value, float *logp, int rows, uint32_t row_id0, uint64_t seed, uint64_t ctr,
                      bool act) {
    std::vector<float> tmp(L.H);
    for (int m = 0; m < rows; m++) {
        float x[DXP];
        for (int k = 0; k < DXP; k++)
            x[k] = k < RS_OBS_DIM ? obs[(size_t)m * RS_OBS_DIM + k] : k < L.d_in ? pred[(size_t)m * 2 + (k - RS_OBS_DIM)] : 0.0f;
        float *hs = hidden + (size_t)m * L.H;
        if (!act) {                                 // the value pass leaves hidden alone
            for (int j = 0; j < L.H; j++) tmp[j] = hs[j];
            hs = tmp.data();
        }
        const rs::PolicyOut o = rs::policy_row<DXP, HMAX>(L, w, x, hs, 1, act, row_id0 + (uint32_t)m, ctr, seed);
        value[m] = o.value;
        if (act) {
            action[m] = o.action;
            logp[m] = o.logp;
        }
    }
}

extern "C" int emu_policy_rows(const RsPolicyConfig *cfg, const float *params, const float *obs, const float *pred,
                               float *hidden, int32_t *action, float *value, float *logp, int rows, uint32_t row_id0,
                               uint64_t seed, uint64_t ctr, int act) {
    rs::PolicyLayout L;
    if (!rs::policy_layout(*cfg, L)) return -1;
    std::vector<float4> table((L.total + 3) / 4, float4{0.0f, 0.0f, 0.0f, 0.0f});
    float *w = reinterpret_cast<float *>(table.data());
    for (int s = 0; s < L.count; s++) w[rs::policy_param_dst(L, s)] = params[s];
#define RS_EMU_ROWS(DXP_, HMAX_) rows_body<DXP_, HMAX_>(L, w, obs, pred, hidden, action, value, logp, rows, row_id0, seed, ctr, act != 0)
    if (L.d_in == 11) {
        if (L.H <= 16) RS_EMU_ROWS(12, 16); else if (L.H <= 32) RS_EMU_ROWS(12, 32); else RS_EMU_ROWS(12, 64);
    } else {
        if (L.H <= 16) RS_EMU_ROWS(16, 16); else if (L.H <= 32) RS_EMU_ROWS(16, 32); else RS_EMU_ROWS(16, 64);
    }
#undef RS_EMU_ROWS
    return 0;
}

// the table's size and the destination of every packed element, so that a test can check that the staging is a bijection
// onto the non-padding slots
extern "C" int emu_policy_layout(const RsPolicyConfig *cfg, int32_t *dst) {
    rs::PolicyLayout L;
    if (!rs::policy_layout(*cfg, L)) return -1;
    if (dst)
        for (int s = 0; s < L.count; s++) dst[s] = rs::policy_param_dst(L, s);
    return L.total;
}
