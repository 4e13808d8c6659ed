// Fused PFGRU source localiser inference (pfgru.FusedPFGRU): one launch runs the particle-filter GRU step, the soft
// resampling and the prediction head for every row of the batch, where the stock PyTorch cell costs six linear layers,
// more than a dozen elementwise launches and a torch.multinomial per call.
//   rs_pfgru_predict  one step on the state, written back in place, prediction out; advances the call counter
//   rs_pfgru_peek     the same step on the current state of the selected rows, prediction out, nothing else written: the
//                     source prediction that goes with a bootstrap value (T:462-487)
//   rs_pfgru_restart  fresh particles for the selected rows (init_hidden, T:326, 509-511)
// One warp per row (rs_pfgru.cuh); each CTA stages the weights into shared memory once and its warps walk rows
// grid-stride.  The products are plain float32 FMAs with accurate expf / logf / tanhf: no TF32, no tensor cores.
// T: = /root/reference/algos/multiagent/train.py
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdio>

#include "../../include/radsearch_b200.h"
#include "rs_error.h"
#include "rs_pfgru.cuh"

namespace {

constexpr int kMaxWarps = 8;
enum Mode { kPredict = 0, kPeek = 1, kRestart = 2 };

// HMAX <= 32: at most 128 registers, so that two CTAs (16 rows) share an SM
template <int DXP, int HMAX>
__global__ void __launch_bounds__(kMaxWarps * 32, HMAX <= 32 ? 2 : 1) pfgru_kernel(rs::PfgruLayout L, const float *__restrict__ params,
                                                               const float *__restrict__ obs, float *particles, float *logw,
                                                               float *__restrict__ pred, const uint8_t *__restrict__ mask,
                                                               int mask_bits, int rows, uint32_t row_id0, uint64_t seed,
                                                               uint64_t *ctr, uint32_t *ticket, int mode) {
    extern __shared__ float4 smem4[];
    float *w = reinterpret_cast<float *>(smem4);
    if (mode != kRestart) {
        for (int i = threadIdx.x; i < L.total; i += blockDim.x) w[i] = 0.0f;
        __syncthreads();
        for (int s = threadIdx.x; s < L.count; s += blockDim.x) w[rs::pfgru_param_dst(L, s)] = params[s];
    }
    // every CTA reads the counter before it takes its ticket, so the last CTA's increment comes after all reads
    const uint64_t c = *ctr;
    __syncthreads();
    const int warps = blockDim.x >> 5, warp = threadIdx.x >> 5;
    float *scratch = w + L.total + warp * L.scratch;
    const int KH = L.K * L.H;
    for (int m = blockIdx.x * warps + warp; m < rows; m += gridDim.x * warps) {
        if (mask) {
            const int b = mask[m];
            if (mask_bits ? (b & mask_bits) == 0 : b == 0) continue;
        }
        float *part = particles + (size_t)m * KH, *lw = logw + (size_t)m * L.K;
        if (mode == kRestart)
            rs::pfgru_restart_row(L, part, lw, row_id0 + (uint32_t)m, c, seed);
        else
            rs::pfgru_row<DXP, HMAX>(L, w, scratch, obs + (size_t)m * RS_OBS_DIM, part, lw, pred + (size_t)m * 2,
                                     mode == kPredict, row_id0 + (uint32_t)m, mode == kPredict ? 0u : rs::kPfgruPeekBlock, c,
                                     seed);
    }
    if (mode == kPredict) {
        // the last CTA to finish advances the counter, so that every call -- and every replay of a captured call -- draws
        // fresh noise (the pattern of rs_policy_act)
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            if (atomicAdd(ticket, 1u) == gridDim.x - 1) {
                *ticket = 0u;
                *reinterpret_cast<unsigned long long *>(ctr) += 1ull;
            }
        }
    }
}

template <int DXP, int HMAX>
int launch(const rs::PfgruLayout &L, const float *params, const float *obs, float *particles, float *logw, float *pred,
           const uint8_t *mask, int mask_bits, int rows, uint32_t row_id0, uint64_t seed, uint64_t *ctr, uint32_t *ticket,
           int mode, cudaStream_t s) {
    auto kern = pfgru_kernel<DXP, HMAX>;
    int dev = 0, sms = 0, optin = 0, per_sm = 0;
    cudaError_t e;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return (int)e;
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return (int)e;
    if ((e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev)) != cudaSuccess) return (int)e;
    // as many warps (rows in flight) per CTA as the scratch allows next to the weights, at most kMaxWarps
    const size_t table = sizeof(float) * (mode == kRestart ? 0 : (size_t)L.total), per_warp = sizeof(float) * (size_t)L.scratch;
    int warps = mode == kRestart ? kMaxWarps : (int)(((size_t)optin - table) / per_warp);
    warps = warps < kMaxWarps ? warps : kMaxWarps;
    if (warps < 1) return rs_set_error("rs_pfgru: the weights and one warp's scratch exceed the shared memory of a block");
    const size_t smem = mode == kRestart ? 0 : table + per_warp * warps;
    if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return (int)e;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 32 * warps, smem)) != cudaSuccess) return (int)e;
    const long long need = ((long long)rows + warps - 1) / warps, cap = (long long)sms * (per_sm > 0 ? per_sm : 1);
    const int grid = (int)(need < cap ? need : cap);
    kern<<<grid, 32 * warps, smem, s>>>(L, params, obs, particles, logw, pred, mask, mask_bits, rows, row_id0, seed, ctr,
                                        ticket, mode);
    return (int)cudaGetLastError();
}

int dispatch(const rs::PfgruLayout &L, const float *params, const float *obs, float *particles, float *logw, float *pred,
             const uint8_t *mask, int mask_bits, int rows, uint32_t row_id0, uint64_t seed, uint64_t *ctr, uint32_t *ticket,
             int mode, void *stream) {
    cudaStream_t s = static_cast<cudaStream_t>(stream);
#define RS_PFGRU_LAUNCH(DXP_, HMAX_) \
    launch<DXP_, HMAX_>(L, params, obs, particles, logw, pred, mask, mask_bits, rows, row_id0, seed, ctr, ticket, mode, s)
    if (L.DXP == 4) {
        if (L.H <= 16) return RS_PFGRU_LAUNCH(4, 16);
        if (L.H <= 32) return RS_PFGRU_LAUNCH(4, 32);
        return RS_PFGRU_LAUNCH(4, 64);
    }
    if (L.H <= 16) return RS_PFGRU_LAUNCH(12, 16);
    if (L.H <= 32) return RS_PFGRU_LAUNCH(12, 32);
    return RS_PFGRU_LAUNCH(12, 64);
#undef RS_PFGRU_LAUNCH
}

int check_common(const char *fn, const RsPfgruConfig *cfg, rs::PfgruLayout &L, const float *particles, const float *logw,
                 int rows, uint32_t row_id0, const uint64_t *ctr) {
    auto fail = [&](const char *what) {
        char msg[200];
        std::snprintf(msg, sizeof msg, "%s: %s", fn, what);
        return rs_set_error(msg);
    };
    if (!cfg) return fail("cfg is NULL");
    if (!rs::pfgru_layout(*cfg, L))
        return fail("unsupported config (d_in 1..11; hidden, particles, obs_hidden 1..64; resample 0 or 1; alpha in (0, 1])");
    if (!particles || !logw) return fail("NULL state");
    if (!ctr) return fail("NULL ctr");
    if (rows < 1) return fail("rows must be positive");
    if ((uint64_t)row_id0 + (uint64_t)rows > (1ull << 32)) return fail("row_id0 + rows exceeds 2^32");
    return 0;
}

}  // namespace

extern "C" {

int rs_pfgru_param_count(const RsPfgruConfig *cfg) {
    rs::PfgruLayout L;
    if (!cfg || !rs::pfgru_layout(*cfg, L))
        return rs_set_error("rs_pfgru_param_count: unsupported config (d_in 1..11; hidden, particles, obs_hidden 1..64; "
                            "resample 0 or 1; alpha in (0, 1])");
    return L.count;
}

int rs_pfgru_predict(const RsPfgruConfig *cfg, const float *params, const float *obs, float *particles, float *log_weights,
                     float *pred_out, int32_t rows, uint32_t row_id0, uint64_t seed, uint64_t *ctr, uint32_t *ticket,
                     void *stream) {
    rs::PfgruLayout L;
    if (int rc = check_common("rs_pfgru_predict", cfg, L, particles, log_weights, rows, row_id0, ctr)) return rc;
    if (!params || !obs || !pred_out) return rs_set_error("rs_pfgru_predict: NULL buffer");
    if (!ticket) return rs_set_error("rs_pfgru_predict: NULL ticket");
    return dispatch(L, params, obs, particles, log_weights, pred_out, nullptr, 0, rows, row_id0, seed, ctr, ticket, kPredict,
                    stream);
}

int rs_pfgru_peek(const RsPfgruConfig *cfg, const float *params, const float *obs, const float *particles,
                  const float *log_weights, float *pred_out, const uint8_t *mask, int32_t mask_bits, int32_t rows,
                  uint32_t row_id0, uint64_t seed, const uint64_t *ctr, void *stream) {
    rs::PfgruLayout L;
    if (int rc = check_common("rs_pfgru_peek", cfg, L, particles, log_weights, rows, row_id0, ctr)) return rc;
    if (!params || !obs || !pred_out) return rs_set_error("rs_pfgru_peek: NULL buffer");
    // peek reads the state and the counter and never writes them
    return dispatch(L, params, obs, const_cast<float *>(particles), const_cast<float *>(log_weights), pred_out, mask,
                    mask_bits, rows, row_id0, seed, const_cast<uint64_t *>(ctr), nullptr, kPeek, stream);
}

int rs_pfgru_restart(const RsPfgruConfig *cfg, float *particles, float *log_weights, const uint8_t *mask, int32_t mask_bits,
                     int32_t rows, uint32_t row_id0, uint64_t seed, const uint64_t *ctr, void *stream) {
    rs::PfgruLayout L;
    if (int rc = check_common("rs_pfgru_restart", cfg, L, particles, log_weights, rows, row_id0, ctr)) return rc;
    return dispatch(L, nullptr, nullptr, particles, log_weights, nullptr, mask, mask_bits, rows, row_id0, seed,
                    const_cast<uint64_t *>(ctr), nullptr, kRestart, stream);
}

int rs_sizeof_pfgru_config(void) { return (int)sizeof(RsPfgruConfig); }

}  // extern "C"
