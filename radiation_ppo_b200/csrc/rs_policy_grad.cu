// Fused PPO loss and backpropagation-through-time gradient of the GRU actor-critic (policy.FusedGruPolicy.loss_and_grad):
// one launch runs the recurrent cell forward over the T steps of a minibatch of rollout columns, then backward over the
// same steps, and sums the gradient of every packed parameter, where torch autograd launches a few dozen kernels per step
// in each direction.
//
// A CTA of 16 warps owns 16 consecutive minibatch columns at a time (a group; groups g = blockIdx.x, + gridDim.x, ...):
// one warp per column, lane l handling GRU units / head units l, l + 32.  The weights are staged once per CTA into the
// padded table of rs_policy.cuh.  Per column and step (rs_policy_grad.cuh):
//   forward,  t = 0 .. T-1   GRUCell with the restart rule of rs_rollout_post (the cell reads h_{t-1} (1 - end[t-1]),
//                            h_{-1} = 0); h_t to the workspace [T][M][H]
//   backward, t = T-1 .. 0   recompute the heads from h_t and the gates from (x_t, h_{t-1}); the loss's dL/dlogit, dL/dv;
//                            the heads' and the cell's backward; the carry dL/dh_{t-1}, zero across a restart
// After each backward step the CTA's 512 threads add the step's outer products of its 16 columns into the weight
// gradient: thread i owns the packed parameters i, i + 512, ... in registers, so the sums need no atomics.  Each CTA then
// keeps a float64 partial (its float32 sums are flushed there every 32 steps), and the last CTA (ticket) sums the
// partials in CTA order: the result is bit-identical from call to
// call and under graph replay.  float32 FMAs with accurate expf / tanhf / logf, as in rs_policy.cu: no TF32.
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>
#include <cstdio>

#include "../../include/radsearch_b200.h"
#include "rs_error.h"
#include "rs_policy_grad.cuh"

namespace {

constexpr int kCols = 16;                 // columns per CTA, one warp each
constexpr int kBlock = 32 * kCols;
constexpr int kStatStride = 8;            // doubles per CTA in the statistics partials
constexpr int kFlush = 32;               // backward steps a thread sums in float32 before it adds to its float64 partial

struct GradArgs {
    rs::PolicyLayout L;
    rs::GradLayout G;
    rs::PgConsts k;
    const float *params, *obs, *pred, *act, *adv, *ret, *logp;
    const uint8_t *end;
    const int32_t *columns;
    int T, N, M, groups, count4;
    float *grad;
    double *stats;
    double *part_stats;   // [grid][kStatStride]
    double *part;         // [grid][count4]
    float *hs;            // [T][M][H]
    uint32_t *ticket;
};

// workspace: statistics partials | gradient partials | hidden states, one partial slot per group (grid <= groups)
struct Workspace {
    size_t stats_off, part_off, hs_off, bytes;
};

Workspace workspace_layout(const rs::PolicyLayout &L, int T, int M) {
    const size_t groups = ((size_t)M + kCols - 1) / kCols;
    Workspace w;
    w.stats_off = 0;
    w.part_off = w.stats_off + groups * kStatStride * sizeof(double);
    w.hs_off = w.part_off + groups * (size_t)rs::round4(L.count) * sizeof(double);
    w.bytes = w.hs_off + (size_t)T * (size_t)M * (size_t)L.H * sizeof(float);
    return w;
}

size_t grad_smem(const rs::PolicyLayout &L, const rs::GradLayout &G) {
    return sizeof(float) * ((size_t)L.total + (size_t)kCols * G.CW);
}

template <int DXP, int HMAX, int NACC>
__global__ void __launch_bounds__(kBlock, 1) policy_grad_kernel(const GradArgs a) {
    const rs::PolicyLayout &L = a.L;
    const rs::GradLayout &G = a.G;
    extern __shared__ float4 smem4[];
    __shared__ double st_sh[kCols][rs::kGradStats];
    __shared__ bool last;
    float *w = reinterpret_cast<float *>(smem4);
    for (int i = threadIdx.x; i < L.total; i += kBlock) w[i] = 0.0f;
    __syncthreads();
    for (int s = threadIdx.x; s < L.count; s += kBlock) w[rs::policy_param_dst(L, s)] = a.params[s];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, H = L.H, T = a.T, N = a.N, M = a.M;
    float *scr = w + L.total;
    float *col = scr + warp * G.CW;
    // the parameters this thread sums; past the count, a pair of padding slots that stay zero
    uint32_t idx[NACC];
    float acc[NACC];
    const uint32_t pad = ((uint32_t)(G.uone + 1) << 16) | (uint32_t)(G.uone + 1);
#pragma unroll
    for (int i = 0; i < NACC; i++) {
        const int s = threadIdx.x + i * kBlock;
        idx[i] = s < L.count ? rs::grad_entry(L, G, s) : pad;
        acc[i] = 0.0f;
    }
    double *st = st_sh[warp];   // the column's diagnostics, summed by lane 0
    if (lane < rs::kGradStats) st[lane] = 0.0;
    // this CTA's float64 partial of the gradient: each thread owns its entries, so it adds there without atomics.  Its
    // address lives in shared memory, reloaded after the step's barrier, so that it takes no register in the step loop.
    __shared__ double *part_sh;
    if (threadIdx.x == 0) part_sh = a.part + (size_t)blockIdx.x * a.count4;
#pragma unroll
    for (int i = 0; i < NACC; i++) {
        const int s = threadIdx.x + i * kBlock;
        if (s < L.count) a.part[(size_t)blockIdx.x * a.count4 + s] = 0.0;
    }
    __syncthreads();

    for (int g = blockIdx.x; g < a.groups; g += gridDim.x) {
        const int m = g * kCols + warp;
        int n = -1;
        if (m < M) {
            n = a.columns ? a.columns[m] : m;
            if (n < 0 || n >= N) {
                if (lane == 0) st[5] += (double)T;
                n = -1;
            }
        }
        // a column without work keeps all-zero factors: its products add nothing
        for (int i = lane; i < G.CW; i += 32) col[i] = 0.0f;
        __syncwarp();
        if (lane == 0) col[G.uone] = 1.0f;
        if (n >= 0) {
            for (int t = 0; t < T; t++) {
                const size_t row = (size_t)t * N + n;
                const bool keep = t > 0 && a.end[row - N] == 0;
                rs::pg_inputs<DXP>(L, G, col, a.obs + row * RS_OBS_DIM, a.pred ? a.pred + row * 2 : nullptr,
                                   keep ? col + G.uh : nullptr, nullptr, lane, 32);
                __syncwarp();
                rs::pg_cell<DXP, HMAX>(L, G, w, col, a.hs + ((size_t)t * M + m) * H, lane, 32);
                __syncwarp();
            }
        }
        for (int t = T - 1; t >= 0; t--) {
            if (n >= 0) {
                const size_t row = (size_t)t * N + n;
                const bool keep = t > 0 && a.end[row - N] == 0;
                const float *ht = a.hs + ((size_t)t * M + m) * H;
                rs::pg_inputs<DXP>(L, G, col, a.obs + row * RS_OBS_DIM, a.pred ? a.pred + row * 2 : nullptr,
                                   keep ? ht - (size_t)M * H : nullptr, ht, lane, 32);
                __syncwarp();
                rs::pg_heads<HMAX>(L, G, w, col, lane, 32);
                __syncwarp();
                if (lane == 0) rs::pg_loss(G, col, rs::PgRow{a.act[row], a.adv[row], a.ret[row], a.logp[row]}, a.k, st);
                __syncwarp();
                rs::pg_heads_back(L, G, w, col, lane, 32);
                __syncwarp();
                rs::pg_cell_back<DXP, HMAX>(L, G, w, col, lane, 32);
                __syncwarp();
                rs::pg_carry(L, G, w, col, keep, lane, 32);
            }
            __syncthreads();
#pragma unroll
            for (int i = 0; i < NACC; i++) {
                const float *f = scr + (idx[i] >> 16), *u = scr + (idx[i] & 0xFFFFu);
                float v = acc[i];
#pragma unroll
                for (int c = 0; c < kCols; c++) v = fmaf(f[c * G.CW], u[c * G.CW], v);
                acc[i] = v;
            }
            // a float32 sum runs over at most kFlush steps x 16 columns: long float32 sums lose the gradient of a
            // parameter whose per-row products largely cancel
            if (t % kFlush == 0) {
                double *pp = part_sh;
#pragma unroll
                for (int i = 0; i < NACC; i++) {
                    const int s = threadIdx.x + i * kBlock;
                    if (s < L.count) pp[s] += (double)acc[i];
                    acc[i] = 0.0f;
                }
            }
            __syncthreads();
        }
    }

    if (threadIdx.x < rs::kGradStats) {
        double v = 0.0;
        for (int c = 0; c < kCols; c++) v += st_sh[c][threadIdx.x];
        a.part_stats[(size_t)blockIdx.x * kStatStride + threadIdx.x] = v;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(a.ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    // the last CTA: every partial in CTA order
    for (int s = threadIdx.x; s < L.count; s += kBlock) {
        double v = 0.0;
        for (unsigned b = 0; b < gridDim.x; b++) v += __ldcg(a.part + (size_t)b * a.count4 + s);
        a.grad[s] = (float)v;
    }
    if (threadIdx.x < rs::kGradStats) {
        double v = 0.0;
        for (unsigned b = 0; b < gridDim.x; b++) v += __ldcg(a.part_stats + (size_t)b * kStatStride + threadIdx.x);
        a.stats[threadIdx.x] = v;
    }
    if (threadIdx.x == 0) *a.ticket = 0u;
}

template <int DXP, int HMAX, int NACC>
int launch(GradArgs a, cudaStream_t s) {
    auto kern = policy_grad_kernel<DXP, HMAX, NACC>;
    const size_t smem = grad_smem(a.L, a.G);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    int dev = 0, sms = 0, per_sm = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return (int)e;
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return (int)e;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kBlock, smem)) != cudaSuccess) return (int)e;
    const long long cap = (long long)sms * (per_sm > 0 ? per_sm : 1);
    const int grid = (int)(a.groups < cap ? a.groups : cap);
    kern<<<grid, kBlock, smem, s>>>(a);
    return (int)cudaGetLastError();
}

// NACC = parameters per thread, rounded up to the classes each hidden width can need (H <= 16: up to 4 249 parameters,
// H <= 32: 9 321, H <= 64: 4 860 .. 24 073)
template <int DXP>
int dispatch(const GradArgs &a, cudaStream_t s) {
    const int need = (a.L.count + kBlock - 1) / kBlock;
    if (a.L.H <= 16) return need <= 8 ? launch<DXP, 16, 8>(a, s) : launch<DXP, 16, 16>(a, s);
    if (a.L.H <= 32) return need <= 8 ? launch<DXP, 32, 8>(a, s) : need <= 16 ? launch<DXP, 32, 16>(a, s) : launch<DXP, 32, 32>(a, s);
    return need <= 16 ? launch<DXP, 64, 16>(a, s) : need <= 32 ? launch<DXP, 64, 32>(a, s) : launch<DXP, 64, 48>(a, s);
}

}  // namespace

extern "C" {

int64_t rs_policy_grad_workspace_bytes(const RsPolicyConfig *cfg, int32_t T, int32_t M) {
    rs::PolicyLayout L;
    if (!cfg || !rs::policy_layout(*cfg, L))
        return rs_set_error("rs_policy_grad_workspace_bytes: unsupported config (d_in 11 or 13; hidden 1..64; pi_hidden / "
                            "v_hidden 0..64; activation 0 or 1)");
    if (T < 1 || M < 1) return rs_set_error("rs_policy_grad_workspace_bytes: T and M must be positive");
    return (int64_t)workspace_layout(L, T, M).bytes;
}

int rs_policy_ppo_grad(const RsPolicyConfig *cfg, const float *params, const float *obs, const float *pred, const float *act,
                       const float *adv, const float *ret, const float *logp, const uint8_t *end, const int32_t *columns,
                       int32_t T, int32_t N, int32_t M, double clip_ratio, double w_pi, double w_v, float *grad,
                       double *stats, void *workspace, uint32_t *ticket, void *stream) {
    auto fail = [](const char *what) {
        char msg[160];
        std::snprintf(msg, sizeof msg, "rs_policy_ppo_grad: %s", what);
        return rs_set_error(msg);
    };
    GradArgs a;
    if (!cfg) return fail("cfg is NULL");
    if (!rs::policy_layout(*cfg, a.L))
        return fail("unsupported config (d_in 11 or 13; hidden 1..64; pi_hidden / v_hidden 0..64; activation 0 or 1)");
    if (!params || !obs || !act || !adv || !ret || !logp || !end) return fail("NULL buffer");
    if (cfg->d_in == 13 && !pred) return fail("d_in = 13 needs pred");
    if (cfg->d_in == 11 && pred) return fail("pred given with d_in = 11");
    if (T < 1 || N < 1 || M < 1) return fail("T, N and M must be positive");
    if (!columns && M != N) return fail("M must equal N without columns");
    if (!(clip_ratio >= 0.0 && clip_ratio < 1.0)) return fail("clip_ratio must be in [0, 1)");
    if (!std::isfinite(w_pi) || !std::isfinite(w_v)) return fail("w_pi and w_v must be finite");
    if (!grad || !stats || !workspace || !ticket) return fail("NULL output / workspace / ticket");
    rs::grad_layout(a.L, a.G);
    const double c = 1.0 / ((double)T * (double)M);
    // torch.clamp(ratio, 1 - clip, 1 + clip) on float32 rounds its bounds to float32
    a.k = rs::PgConsts{(float)(1.0 - clip_ratio), (float)(1.0 + clip_ratio), (float)(w_pi * c), (float)(2.0 * w_v * c)};
    a.params = params; a.obs = obs; a.pred = pred; a.act = act; a.adv = adv; a.ret = ret; a.logp = logp; a.end = end;
    a.columns = columns;
    a.T = T; a.N = N; a.M = M;
    a.groups = (M + kCols - 1) / kCols;
    a.count4 = rs::round4(a.L.count);
    const Workspace ws = workspace_layout(a.L, T, M);
    char *base = static_cast<char *>(workspace);
    a.part_stats = reinterpret_cast<double *>(base + ws.stats_off);
    a.part = reinterpret_cast<double *>(base + ws.part_off);
    a.hs = reinterpret_cast<float *>(base + ws.hs_off);
    a.grad = grad; a.stats = stats; a.ticket = ticket;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    return cfg->d_in == 11 ? dispatch<12>(a, s) : dispatch<16>(a, s);
}

}  // extern "C"
