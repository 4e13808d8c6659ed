// Fused GRU actor-critic inference for the collection and evaluation loops (policy.FusedGruPolicy): one launch runs the
// recurrent cell, both heads and the action sampling for every row of the batch, where the stock PyTorch module costs a
// dozen cuBLAS / elementwise launches.
//   rs_policy_act    GRUCell step (hidden updated in place), log_softmax of the policy head, Gumbel-max sample, value of h'
//   rs_policy_value  the value of the next observation under the current hidden state, hidden untouched: the bootstrap
//                    of the trajectories that were cut (T:462-487)
// One thread per row; each CTA stages the weights into shared memory once and walks rows grid-stride.  The products are
// plain float32 FMAs (K = 11..64, N <= 192 per row): the tensor cores' TF32 would move the log-probabilities away from
// the torch module that recomputes them in the PPO ratio.
// T: = /root/reference/algos/multiagent/train.py
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdio>

#include "../../include/radsearch_b200.h"
#include "rs_error.h"
#include "rs_policy.cuh"

namespace {

constexpr int kBlock = 256;

// Shared memory: the staged table (PolicyLayout.total floats), then each thread's hidden state, element j of thread t at
// [j * kBlock + t] (conflict-free).
size_t policy_smem(const rs::PolicyLayout &L) { return sizeof(float) * ((size_t)L.total + (size_t)L.H * kBlock); }

template <int DXP, int HMAX>
__global__ void __launch_bounds__(kBlock) policy_kernel(rs::PolicyLayout L, const float *__restrict__ params,
                                                        const float *__restrict__ obs, const float *__restrict__ pred,
                                                        float *__restrict__ hidden, int32_t *__restrict__ action,
                                                        float *__restrict__ value, float *__restrict__ logp, int rows,
                                                        uint32_t row_id0, uint64_t seed, uint64_t *ctr, uint32_t *ticket,
                                                        int act) {
    constexpr int DIN = DXP == 12 ? 11 : 13;
    extern __shared__ float4 smem4[];
    float *w = reinterpret_cast<float *>(smem4);
    for (int i = threadIdx.x; i < L.total; i += kBlock) w[i] = 0.0f;
    __syncthreads();
    for (int s = threadIdx.x; s < L.count; s += kBlock) w[rs::policy_param_dst(L, s)] = params[s];
    // every CTA reads the counter before it takes its ticket, so the last CTA's increment comes after all reads
    const uint64_t c = act ? *ctr : 0ull;
    __syncthreads();
    float *hs = w + L.total + threadIdx.x;
    const int H = L.H;
    for (int m = blockIdx.x * kBlock + threadIdx.x; m < rows; m += gridDim.x * kBlock) {
        float x[DXP];
#pragma unroll
        for (int k = 0; k < DXP; k++)
            x[k] = k < RS_OBS_DIM ? obs[(size_t)m * RS_OBS_DIM + k] : k < DIN ? pred[(size_t)m * 2 + (k - RS_OBS_DIM)] : 0.0f;
        const float *hm = hidden + (size_t)m * H;
        for (int j = 0; j < H; j++) hs[j * kBlock] = hm[j];
        const rs::PolicyOut o = rs::policy_row<DXP, HMAX>(L, w, x, hs, kBlock, act != 0, row_id0 + (uint32_t)m, c, seed);
        value[m] = o.value;
        if (act) {
            float *hw = hidden + (size_t)m * H;
            for (int j = 0; j < H; j++) hw[j] = hs[j * kBlock];
            action[m] = o.action;
            logp[m] = o.logp;
        }
    }
    if (act) {
        // the last CTA to finish advances the counter, so that every call -- and every replay of a captured call -- draws
        // fresh noise (the pattern of rs_reset's RS_F_BUMP_CTR)
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
int launch(const rs::PolicyLayout &L, const float *params, const float *obs, const float *pred, float *hidden,
           int32_t *action, float *value, float *logp, int rows, uint32_t row_id0, uint64_t seed, uint64_t *ctr,
           uint32_t *ticket, int act, cudaStream_t s) {
    auto kern = policy_kernel<DXP, HMAX>;
    const size_t smem = policy_smem(L);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    int dev = 0, sms = 0, per_sm = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return (int)e;
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return (int)e;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kBlock, smem)) != cudaSuccess) return (int)e;
    const long long need = ((long long)rows + kBlock - 1) / kBlock, cap = (long long)sms * (per_sm > 0 ? per_sm : 1);
    const int grid = (int)(need < cap ? need : cap);
    kern<<<grid, kBlock, smem, s>>>(L, params, obs, pred, hidden, action, value, logp, rows, row_id0, seed, ctr, ticket, act);
    return (int)cudaGetLastError();
}

int dispatch(const rs::PolicyLayout &L, const float *params, const float *obs, const float *pred, float *hidden,
             int32_t *action, float *value, float *logp, int rows, uint32_t row_id0, uint64_t seed, uint64_t *ctr,
             uint32_t *ticket, int act, void *stream) {
    cudaStream_t s = static_cast<cudaStream_t>(stream);
#define RS_POLICY_LAUNCH(DXP_, HMAX_) \
    launch<DXP_, HMAX_>(L, params, obs, pred, hidden, action, value, logp, rows, row_id0, seed, ctr, ticket, act, s)
    if (L.d_in == 11) {
        if (L.H <= 16) return RS_POLICY_LAUNCH(12, 16);
        if (L.H <= 32) return RS_POLICY_LAUNCH(12, 32);
        return RS_POLICY_LAUNCH(12, 64);
    }
    if (L.H <= 16) return RS_POLICY_LAUNCH(16, 16);
    if (L.H <= 32) return RS_POLICY_LAUNCH(16, 32);
    return RS_POLICY_LAUNCH(16, 64);
#undef RS_POLICY_LAUNCH
}

int check_common(const char *fn, const RsPolicyConfig *cfg, rs::PolicyLayout &L, const float *params, const float *obs,
                 const float *pred, const float *hidden, int rows) {
    auto fail = [&](const char *what) {
        char msg[160];
        std::snprintf(msg, sizeof msg, "%s: %s", fn, what);
        return rs_set_error(msg);
    };
    if (!cfg) return fail("cfg is NULL");
    if (!rs::policy_layout(*cfg, L))
        return fail("unsupported config (d_in 11 or 13; hidden 1..64; pi_hidden / v_hidden 0..64; activation 0 or 1)");
    if (!params || !obs || !hidden) return fail("NULL buffer");
    if (cfg->d_in == 13 && !pred) return fail("d_in = 13 needs pred");
    if (cfg->d_in == 11 && pred) return fail("pred given with d_in = 11");
    if (rows < 1) return fail("rows must be positive");
    return 0;
}

}  // namespace

extern "C" {

int rs_policy_param_count(const RsPolicyConfig *cfg) {
    rs::PolicyLayout L;
    if (!cfg || !rs::policy_layout(*cfg, L))
        return rs_set_error("rs_policy_param_count: unsupported config (d_in 11 or 13; hidden 1..64; pi_hidden / v_hidden "
                            "0..64; activation 0 or 1)");
    return L.count;
}

int rs_policy_act(const RsPolicyConfig *cfg, const float *params, const float *obs, const float *pred, float *hidden,
                  int32_t *action, float *value, float *logp, int rows, uint32_t row_id0, uint64_t seed, uint64_t *ctr,
                  uint32_t *ticket, void *stream) {
    rs::PolicyLayout L;
    if (int rc = check_common("rs_policy_act", cfg, L, params, obs, pred, hidden, rows)) return rc;
    if (!action || !value || !logp) return rs_set_error("rs_policy_act: NULL output");
    if (!ctr || !ticket) return rs_set_error("rs_policy_act: NULL ctr / ticket");
    if ((uint64_t)row_id0 + (uint64_t)rows > (1ull << 32)) return rs_set_error("rs_policy_act: row_id0 + rows exceeds 2^32");
    return dispatch(L, params, obs, pred, hidden, action, value, logp, rows, row_id0, seed, ctr, ticket, 1, stream);
}

int rs_policy_value(const RsPolicyConfig *cfg, const float *params, const float *obs, const float *pred,
                    const float *hidden, float *value, int rows, void *stream) {
    rs::PolicyLayout L;
    if (int rc = check_common("rs_policy_value", cfg, L, params, obs, pred, hidden, rows)) return rc;
    if (!value) return rs_set_error("rs_policy_value: NULL output");
    // the value pass reads hidden and never writes it
    return dispatch(L, params, obs, pred, const_cast<float *>(hidden), nullptr, value, nullptr, rows, 0, 0, nullptr, nullptr,
                    0, stream);
}

int rs_sizeof_policy_config(void) { return (int)sizeof(RsPolicyConfig); }

}  // extern "C"
