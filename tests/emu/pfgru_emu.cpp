// TEST INFRASTRUCTURE ONLY -- host build of the fused PFGRU localiser's per-row body (radiation_ppo_b200/csrc/rs_pfgru.cuh):
// the staging of the packed weights, and the warp phases of one row run lane by lane on host memory.  Used by
// tests/test_pfgru_cabi.py to compare the kernel's arithmetic with a float64 restatement where no GPU exists.
#define RS_HOST_EMU 1
#include "../../radiation_ppo_b200/csrc/rs_pfgru.cuh"

#include <vector>

template <int DXP, int HMAX>
static void rows_body(const rs::PfgruLayout &L, const float *w, const float *obs, float *particles, float *logw, float *pred,
                      const uint8_t *mask, int mask_bits, int rows, uint32_t row_id0, uint64_t seed, uint64_t ctr, int mode) {
    std::vector<float> scratch(L.scratch);
    for (int m = 0; m < rows; m++) {
        if (mask && (mask_bits ? (mask[m] & mask_bits) == 0 : mask[m] == 0)) continue;
        float *part = particles + (size_t)m * L.K * L.H, *lw = logw + (size_t)m * L.K;
        if (mode == 2)
            rs::pfgru_restart_row(L, part, lw, row_id0 + (uint32_t)m, ctr, seed);
        else
            rs::pfgru_row<DXP, HMAX>(L, w, scratch.data(), obs + (size_t)m * RS_OBS_DIM, part, lw, pred + (size_t)m * 2,
                                     mode == 0, row_id0 + (uint32_t)m, mode == 0 ? 0u : rs::kPfgruPeekBlock, ctr, seed);
    }
}

// mode 0 predict, 1 peek, 2 restart (the counter is passed by value: the host build does not advance it)
extern "C" int emu_pfgru_rows(const RsPfgruConfig *cfg, const float *params, const float *obs, float *particles, float *logw,
                              float *pred, const uint8_t *mask, int mask_bits, int rows, uint32_t row_id0, uint64_t seed,
                              uint64_t ctr, int mode) {
    rs::PfgruLayout L;
    if (!rs::pfgru_layout(*cfg, L)) return -1;
    std::vector<float4> table(L.total / 4, float4{0.0f, 0.0f, 0.0f, 0.0f});
    float *w = reinterpret_cast<float *>(table.data());
    if (params)
        for (int s = 0; s < L.count; s++) w[rs::pfgru_param_dst(L, s)] = params[s];
#define RS_EMU_ROWS(DXP_, HMAX_) \
    rows_body<DXP_, HMAX_>(L, w, obs, particles, logw, pred, mask, mask_bits, rows, row_id0, seed, ctr, mode)
    if (L.DXP == 4) {
        if (L.H <= 16) RS_EMU_ROWS(4, 16); else if (L.H <= 32) RS_EMU_ROWS(4, 32); else RS_EMU_ROWS(4, 64);
    } else {
        if (L.H <= 16) RS_EMU_ROWS(12, 16); else if (L.H <= 32) RS_EMU_ROWS(12, 32); else RS_EMU_ROWS(12, 64);
    }
#undef RS_EMU_ROWS
    return 0;
}

// the table's size and the destination of every packed element, so that a test can check that the staging is a bijection
extern "C" int emu_pfgru_layout(const RsPfgruConfig *cfg, int32_t *dst) {
    rs::PfgruLayout L;
    if (!rs::pfgru_layout(*cfg, L)) return -1;
    if (dst)
        for (int s = 0; s < L.count; s++) dst[s] = rs::pfgru_param_dst(L, s);
    return L.total;
}

// the Box-Muller normals of blocks blk0 .. blk0 + n - 1 of one row, four per block
extern "C" void emu_pfgru_normals(uint32_t row_id, uint32_t blk0, int n, uint64_t ctr, uint64_t seed, float *out) {
    for (int b = 0; b < n; b++) rs::pfgru_normal4(row_id, blk0 + (uint32_t)b, ctr, seed, out + 4 * b);
}

// the resampling index rule: C = the float32 prefix sum of q in particle order, idx[i] = pfgru_pick(C, K, u[i] C_{K-1})
extern "C" void emu_pfgru_pick(const float *q, int K, const float *u, int n, int32_t *idx) {
    std::vector<float> C(K);
    float c = 0.0f;
    for (int k = 0; k < K; k++) C[k] = c += q[k];
    for (int i = 0; i < n; i++) idx[i] = rs::pfgru_pick(C.data(), K, u[i] * C[K - 1]);
}
