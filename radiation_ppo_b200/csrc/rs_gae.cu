// GAE-lambda advantages + rewards-to-go over a [T][N] rollout buffer, and the advantage statistics / normalisation.
// P: = /root/reference/algos/multiagent/ppo.py  (GAE_advantage_and_rewardsToGO P:391-423, discount_cumsum P:62-85,
// get() normalisation P:445-446; statistics algos/multiagent/rl_tools/mpi_tools.py:71-95).
//
// Per column n, scanning t = T-1 .. 0 (SURVEY.md Appendix C), everything in fp64 like scipy's lfilter:
//   end   = path_end[t][n] || t == T-1
//   nv,na,nr = end ? (boot, 0, boot) : (val[t+1], adv[t+1], ret[t+1])
//   adv[t] = (rew + gamma*nv) - val + (gamma*lam)*na ;  ret[t] = rew + gamma*nr
#include <cuda.h>
#include <algorithm>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdio>

#include "../../include/radsearch_b200.h"
#include "rs_error.h"

namespace {

// ------------------------------------------------------------------------------------------------------------------
// variant 1: one thread per column, U loads in flight per array (coalesced over n).  Bit-identical to the reference's
// float64 recurrence (same operation order, no fused multiply-add: the file is compiled with -fmad=false).
// ------------------------------------------------------------------------------------------------------------------
constexpr int kColsBlock = 128;

template <int U, int MINB>
__global__ void __launch_bounds__(kColsBlock, MINB) gae_cols_kernel(const float *__restrict__ rew, const float *__restrict__ val,
                                                                    const uint8_t *__restrict__ pe, const float *__restrict__ boot,
                                                                    float *__restrict__ adv, float *__restrict__ ret, int T, int N,
                                                                    double gamma, double gl, double *stats) {
    const int n = blockIdx.x * kColsBlock + threadIdx.x;
    double s1 = 0.0, s2 = 0.0;
    if (n < N) {
        double nv = 0.0, na = 0.0, nr = 0.0;
        float r[U], v[U], r2[U], v2[U];
        uint8_t e[U], e2[U];
        // software pipeline: the loads of chunk i+1 are issued before the dependent fp64 chain of chunk i runs
#pragma unroll
        for (int j = 0; j < U; j++) {
            const int t = T - 1 - j;
            if (t >= 0) {
                const size_t i = (size_t)t * N + n;
                r[j] = __ldcs(rew + i); v[j] = __ldcs(val + i); e[j] = __ldcs(pe + i);
            }
        }
        for (int t0 = T - 1; t0 >= 0; t0 -= U) {
#pragma unroll
            for (int j = 0; j < U; j++) {
                const int t = t0 - U - j;
                if (t >= 0) {
                    const size_t i = (size_t)t * N + n;
                    r2[j] = __ldcs(rew + i); v2[j] = __ldcs(val + i); e2[j] = __ldcs(pe + i);
                }
            }
#pragma unroll
            for (int j = 0; j < U; j++) {
                const int t = t0 - j;
                if (t >= 0) {
                    const size_t i = (size_t)t * N + n;
                    if (e[j] || t == T - 1) {
                        const double b = (double)__ldcs(boot + i);
                        nv = b; na = 0.0; nr = b;
                    }
                    const double rr = (double)r[j], vv = (double)v[j];
                    const double delta = (rr + gamma * nv) - vv;
                    const double a = delta + gl * na;
                    const double g = rr + gamma * nr;
                    const float af = (float)a;
                    __stcs(adv + i, af);
                    __stcs(ret + i, (float)g);
                    s1 += (double)af;
                    s2 += (double)af * (double)af;
                    nv = vv; na = a; nr = g;
                }
            }
#pragma unroll
            for (int j = 0; j < U; j++) { r[j] = r2[j]; v[j] = v2[j]; e[j] = e2[j]; }
        }
    }
    if (stats) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s1 += __shfl_down_sync(0xffffffffu, s1, o);
            s2 += __shfl_down_sync(0xffffffffu, s2, o);
        }
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(stats, s1);
            atomicAdd(stats + 1, s2);
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// variants 7 / 10: the same per-column recurrence (same operation order: bit-identical to variant 1) fed by the copy engine.
// A CTA owns 128 columns; the [U rows][128 columns] tiles of rew / val / path_end travel HBM -> shared memory as
// bulk-async copies (cp.async.bulk + mbarrier, one 512-byte / 128-byte run per row) through a ring of S stages issued S
// chunks ahead, so the threads spend their instructions on the fp64 chain instead of on address arithmetic and on
// holding loads in registers; the (rare) bootstrap values of a chunk are requested one chunk ahead, as soon as its
// path_end flags have landed, instead of inside the dependent chain.
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t g_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void g_bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     g_smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(g_smem_u32(mbar))
                 : "memory");
}
__device__ __forceinline__ void g_mbar_wait(uint64_t *mbar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "GAE_WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra GAE_WAIT_DONE;\n"
        "bra GAE_WAIT_LOOP;\n"
        "GAE_WAIT_DONE:\n"
        "}\n" ::"r"(g_smem_u32(mbar)),
        "r"(parity)
        : "memory");
}

// U consecutive steps (t_hi, t_hi-1, ...) of one column, values already in registers.  A whole chunk runs as straight-line
// code: the end-of-path restart is a select, not a branch, so the compiler overlaps the rows and only the one-operation
// recurrences (a, g, the two sums) stay serial.  Same operations per element as variant 1: bit-identical.
template <int U>
__device__ __forceinline__ void gae_rows(const float (&rj)[U], const float (&vj)[U], const uint8_t (&ej)[U], const float (&bc)[U],
                                         bool last_step_first, int t_hi, int N, size_t n, float *__restrict__ adv,
                                         float *__restrict__ ret, double gamma, double gl, double &nv, double &na, double &nr,
                                         double &s1, double &s2) {
    if (t_hi - (U - 1) >= 0) {
        float *pa = adv + (size_t)t_hi * N + n, *pr = ret + (size_t)t_hi * N + n;
#pragma unroll
        for (int j = 0; j < U; j++) {
            const bool e = ej[j] != 0 || (last_step_first && j == 0);
            const double b = (double)bc[j];
            nv = e ? b : nv; na = e ? 0.0 : na; nr = e ? b : nr;
            const double rr = (double)rj[j], vv = (double)vj[j];
            const double delta = (rr + gamma * nv) - vv;
            const double a = delta + gl * na;
            const double g = rr + gamma * nr;
            const float af = (float)a;
            __stcs(pa, af);
            __stcs(pr, (float)g);
            pa -= N; pr -= N;
            s1 += (double)af;
            s2 += (double)af * (double)af;
            nv = vv; na = a; nr = g;
        }
    } else {
#pragma unroll
        for (int j = 0; j < U; j++) {
            const int t = t_hi - j;
            if (t >= 0) {
                if (ej[j] || (last_step_first && j == 0)) {
                    const double b = (double)bc[j];
                    nv = b; na = 0.0; nr = b;
                }
                const double rr = (double)rj[j], vv = (double)vj[j];
                const double delta = (rr + gamma * nv) - vv;
                const double a = delta + gl * na;
                const double g = rr + gamma * nr;
                const float af = (float)a;
                const size_t i = (size_t)t * N + n;
                __stcs(adv + i, af);
                __stcs(ret + i, (float)g);
                s1 += (double)af;
                s2 += (double)af * (double)af;
                nv = vv; na = a; nr = g;
            }
        }
    }
}

template <int C, int U, int S, int MINB>
__global__ void __launch_bounds__(C, MINB) gae_tile_kernel(const float *__restrict__ rew, const float *__restrict__ val,
                                                                    const uint8_t *__restrict__ pe, const float *__restrict__ boot,
                                                                    float *__restrict__ adv, float *__restrict__ ret, int T, int N,
                                                                    double gamma, double gl, double *stats) {
    __shared__ __align__(128) float s_rew[S][U][C];
    __shared__ __align__(128) float s_val[S][U][C];
    __shared__ __align__(128) uint8_t s_pe[S][U][C];
    __shared__ __align__(8) uint64_t full[S];
    const int tid = threadIdx.x;
    const int n0 = blockIdx.x * C, n = n0 + tid;
    const int chunks = (T + U - 1) / U;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < S; s++)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(g_smem_u32(full + s)), "r"(1) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // chunk c = steps T-1-c*U .. T-1-c*U-(U-1) (row j of the tile = step T-1-c*U-j), rows below step 0 are absent
    auto issue = [&](int c) {
        const int st = c % S, t_hi = T - 1 - c * U, rows = min(U, t_hi + 1);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(g_smem_u32(full + st)),
                     "r"((uint32_t)rows * (uint32_t)(C * 9))
                     : "memory");
        for (int j = 0; j < rows; j++) {
            const size_t g = (size_t)(t_hi - j) * N + n0;
            g_bulk_g2s(&s_rew[st][j][0], rew + g, C * 4, full + st);
            g_bulk_g2s(&s_val[st][j][0], val + g, C * 4, full + st);
            g_bulk_g2s(&s_pe[st][j][0], pe + g, C, full + st);
        }
    };
    if (tid == 0)
        for (int c = 0; c < S && c < chunks; c++) issue(c);

    double nv = 0.0, na = 0.0, nr = 0.0, s1 = 0.0, s2 = 0.0;
    float bc[U], bn[U];
    // bootstrap values of chunk 0 (every column ends at T-1)
    g_mbar_wait(full + 0, 0);
#pragma unroll
    for (int j = 0; j < U; j++) {
        const int t = T - 1 - j;
        bc[j] = 0.0f;
        if (t >= 0 && (s_pe[0][j][tid] || t == T - 1)) bc[j] = __ldcs(boot + (size_t)t * N + n);
    }
    for (int c = 0; c < chunks; c++) {
        const int st = c % S, t_hi = T - 1 - c * U;
        if (c + 1 < chunks) {                           // the next chunk has landed long ago: ask for its bootstrap values
            const int sn = (c + 1) % S;
            g_mbar_wait(full + sn, (uint32_t)((c + 1) / S) & 1u);
#pragma unroll
            for (int j = 0; j < U; j++) {
                const int t = t_hi - U - j;
                bn[j] = 0.0f;
                if (t >= 0 && s_pe[sn][j][tid]) bn[j] = __ldcs(boot + (size_t)t * N + n);
            }
        }
        {
            float rj[U], vj[U];
            uint8_t ej[U];
#pragma unroll
            for (int j = 0; j < U; j++) { rj[j] = s_rew[st][j][tid]; vj[j] = s_val[st][j][tid]; ej[j] = s_pe[st][j][tid]; }
            gae_rows<U>(rj, vj, ej, bc, c == 0, t_hi, N, (size_t)n, adv, ret, gamma, gl, nv, na, nr, s1, s2);
        }
#pragma unroll
        for (int j = 0; j < U; j++) bc[j] = bn[j];
        __syncthreads();                                // everybody is done with stage st: refill it
        if (tid == 0 && c + S < chunks) issue(c + S);
    }
    if (stats) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s1 += __shfl_down_sync(0xffffffffu, s1, o);
            s2 += __shfl_down_sync(0xffffffffu, s2, o);
        }
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(stats, s1);
            atomicAdd(stats + 1, s2);
        }
    }
}

// variants 8 / 11 / 12 / 13: variant 7 with a producer warp.  Warp 4 only refills stages (it waits on the stage's `empty` barrier, which
// the 128 consumer threads arrive on when they are done reading it), so no CTA-wide barrier sits in the consumers' loop
// and the four consumer warps drift apart by up to S chunks.
template <int C, int U, int S, int MINB>
__global__ void __launch_bounds__(C + 32, MINB) gae_tile_ws_kernel(const float *__restrict__ rew, const float *__restrict__ val,
                                                                  const uint8_t *__restrict__ pe, const float *__restrict__ boot,
                                                                  float *__restrict__ adv, float *__restrict__ ret, int T, int N,
                                                                  double gamma, double gl, double *stats) {
    // dynamic shared memory: [S][U][C] rew | val | path_end, then the barriers.  C columns per CTA (C consumer threads + the
    // producer warp); the last CTA may own fewer (a multiple of 32: N % 128 == 0), its spare threads only keep the barriers
    extern __shared__ __align__(128) unsigned char ws_smem[];
    typedef float (*TileF)[U][C];
    typedef uint8_t (*TileB)[U][C];
    TileF s_rew = reinterpret_cast<TileF>(ws_smem);
    TileF s_val = reinterpret_cast<TileF>(ws_smem + sizeof(float) * S * U * C);
    TileB s_pe = reinterpret_cast<TileB>(ws_smem + 2 * sizeof(float) * S * U * C);
    uint64_t *full = reinterpret_cast<uint64_t *>(ws_smem + 9 * S * U * C);
    uint64_t *empty = full + S;
    const int tid = threadIdx.x;
    const int n0 = blockIdx.x * C, n = n0 + tid;
    const int cols = min(C, N - n0);
    const int chunks = (T + U - 1) / U;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < S; s++) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(g_smem_u32(full + s)), "r"(1) : "memory");
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(g_smem_u32(empty + s)), "r"(C) : "memory");
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid >= C) {                                     // ---- producer warp: lane j moves row j of the tile --------------
        const int lane = tid - C;
        for (int c = 0; c < chunks; c++) {
            const int st = c % S, t_hi = T - 1 - c * U, rows = min(U, t_hi + 1);
            if (c >= S) g_mbar_wait(empty + st, (uint32_t)(c / S - 1) & 1u);
            if (lane == 0)
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(g_smem_u32(full + st)),
                             "r"((uint32_t)rows * (uint32_t)(cols * 9))
                             : "memory");
            __syncwarp();
            if (lane < rows) {
                const size_t g = (size_t)(t_hi - lane) * N + n0;
                g_bulk_g2s(&s_rew[st][lane][0], rew + g, cols * 4, full + st);
                g_bulk_g2s(&s_val[st][lane][0], val + g, cols * 4, full + st);
                g_bulk_g2s(&s_pe[st][lane][0], pe + g, cols, full + st);
            }
        }
        return;
    }
    const bool active = tid < cols;
    double nv = 0.0, na = 0.0, nr = 0.0, s1 = 0.0, s2 = 0.0;
    float bc[U], bn[U];
    g_mbar_wait(full + 0, 0);
#pragma unroll
    for (int j = 0; j < U; j++) {
        const int t = T - 1 - j;
        bc[j] = 0.0f;
        if (active && t >= 0 && (s_pe[0][j][tid] || t == T - 1)) bc[j] = __ldcs(boot + (size_t)t * N + n);
    }
    for (int c = 0; c < chunks; c++) {
        const int st = c % S, t_hi = T - 1 - c * U;
        if (c + 1 < chunks) {
            const int sn = (c + 1) % S;
            g_mbar_wait(full + sn, (uint32_t)((c + 1) / S) & 1u);
#pragma unroll
            for (int j = 0; j < U; j++) {
                const int t = t_hi - U - j;
                bn[j] = 0.0f;
                if (active && t >= 0 && s_pe[sn][j][tid]) bn[j] = __ldcs(boot + (size_t)t * N + n);
            }
        }
        float rj[U], vj[U];
        uint8_t ej[U];
#pragma unroll
        for (int j = 0; j < U; j++) { rj[j] = s_rew[st][j][tid]; vj[j] = s_val[st][j][tid]; ej[j] = s_pe[st][j][tid]; }
        asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(g_smem_u32(empty + st)) : "memory");   // stage read
        if (active) gae_rows<U>(rj, vj, ej, bc, c == 0, t_hi, N, (size_t)n, adv, ret, gamma, gl, nv, na, nr, s1, s2);
#pragma unroll
        for (int j = 0; j < U; j++) bc[j] = bn[j];
    }
    if (stats) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s1 += __shfl_down_sync(0xffffffffu, s1, o);
            s2 += __shfl_down_sync(0xffffffffu, s2, o);
        }
        if ((threadIdx.x & 31) == 0 && active) {
            atomicAdd(stats, s1);
            atomicAdd(stats + 1, s2);
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// variants 14 / 15: the producer-warp form fed by TENSOR-MAP copies.  One cp.async.bulk.tensor.2d request moves a whole
// [U rows][C columns] box of an array, so a chunk costs the copy engine 3 requests instead of 3 U row copies (the row form
// spends ~40-80 cycles of the SM's copy unit per request: at mid sizes that, not HBM, paces the kernel).  Rows of a box are
// in ascending step order (row r of chunk c = step t_hi - (U-1) + r); rows below step 0 and columns beyond N are zero-
// filled by the unit and still counted by the barrier, so every chunk expects the full box.  Same operation order per
// column as variant 1: bit-identical.
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void g_tmap_2d(void *dst, const CUtensorMap *tm, int x, int y, uint64_t *mbar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                     g_smem_u32(dst)),
                 "l"(reinterpret_cast<uint64_t>(tm)), "r"(x), "r"(y), "r"(g_smem_u32(mbar))
                 : "memory");
}

template <int C, int U, int S, int MINB>
__global__ void __launch_bounds__(C + 32, MINB) gae_tmap_kernel(const __grid_constant__ CUtensorMap tm_rew,
                                                               const __grid_constant__ CUtensorMap tm_val,
                                                               const __grid_constant__ CUtensorMap tm_pe,
                                                               const float *__restrict__ boot, float *__restrict__ adv,
                                                               float *__restrict__ ret, int T, int N, double gamma, double gl,
                                                               double *stats) {
    extern __shared__ __align__(128) unsigned char ws_smem[];
    typedef float (*TileF)[U][C];
    typedef uint8_t (*TileB)[U][C];
    TileF s_rew = reinterpret_cast<TileF>(ws_smem);
    TileF s_val = reinterpret_cast<TileF>(ws_smem + sizeof(float) * S * U * C);
    TileB s_pe = reinterpret_cast<TileB>(ws_smem + 2 * sizeof(float) * S * U * C);
    uint64_t *full = reinterpret_cast<uint64_t *>(ws_smem + 9 * S * U * C);
    uint64_t *empty = full + S;
    const int tid = threadIdx.x;
    const int n0 = blockIdx.x * C, n = n0 + tid;
    const int chunks = (T + U - 1) / U;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < S; s++) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(g_smem_u32(full + s)), "r"(1) : "memory");
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(g_smem_u32(empty + s)), "r"(C) : "memory");
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid >= C) {                                     // ---- producer warp: one lane, three requests per chunk -----------
        if (tid == C) {
            for (int c = 0; c < chunks; c++) {
                const int st = c % S, y0 = T - 1 - c * U - (U - 1);
                if (c >= S) g_mbar_wait(empty + st, (uint32_t)(c / S - 1) & 1u);
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(g_smem_u32(full + st)),
                             "r"((uint32_t)(U * C * 9))
                             : "memory");
                g_tmap_2d(&s_rew[st][0][0], &tm_rew, n0, y0, full + st);
                g_tmap_2d(&s_val[st][0][0], &tm_val, n0, y0, full + st);
                g_tmap_2d(&s_pe[st][0][0], &tm_pe, n0, y0, full + st);
            }
        }
        return;
    }
    const bool active = n < N;
    double nv = 0.0, na = 0.0, nr = 0.0, s1 = 0.0, s2 = 0.0;
    float bc[U], bn[U];
    g_mbar_wait(full + 0, 0);
#pragma unroll
    for (int j = 0; j < U; j++) {
        const int t = T - 1 - j;
        bc[j] = 0.0f;
        if (active && t >= 0 && (s_pe[0][U - 1 - j][tid] || t == T - 1)) bc[j] = __ldcs(boot + (size_t)t * N + n);
    }
    for (int c = 0; c < chunks; c++) {
        const int st = c % S, t_hi = T - 1 - c * U;
        if (c + 1 < chunks) {
            const int sn = (c + 1) % S;
            g_mbar_wait(full + sn, (uint32_t)((c + 1) / S) & 1u);
#pragma unroll
            for (int j = 0; j < U; j++) {
                const int t = t_hi - U - j;
                bn[j] = 0.0f;
                if (active && t >= 0 && s_pe[sn][U - 1 - j][tid]) bn[j] = __ldcs(boot + (size_t)t * N + n);
            }
        }
        float rj[U], vj[U];
        uint8_t ej[U];
#pragma unroll
        for (int j = 0; j < U; j++) {
            rj[j] = s_rew[st][U - 1 - j][tid]; vj[j] = s_val[st][U - 1 - j][tid]; ej[j] = s_pe[st][U - 1 - j][tid];
        }
        asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(g_smem_u32(empty + st)) : "memory");   // stage read
        if (active) gae_rows<U>(rj, vj, ej, bc, c == 0, t_hi, N, (size_t)n, adv, ret, gamma, gl, nv, na, nr, s1, s2);
#pragma unroll
        for (int j = 0; j < U; j++) bc[j] = bn[j];
    }
    if (stats) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s1 += __shfl_down_sync(0xffffffffu, s1, o);
            s2 += __shfl_down_sync(0xffffffffu, s2, o);
        }
        if ((threadIdx.x & 31) == 0 && (s1 != 0.0 || s2 != 0.0)) {
            atomicAdd(stats, s1);
            atomicAdd(stats + 1, s2);
        }
    }
}

// tensor map of a row-major [T][N] array with [U][C] boxes; the driver entry point is looked up through the runtime, so
// the library does not link against libcuda
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
bool make_tmap(CUtensorMap *tm, const void *base, bool bytes, int T, int N, int U, int C) {
    static EncodeTiledFn encode = nullptr;
    if (!encode) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn) return false;
        encode = reinterpret_cast<EncodeTiledFn>(fn);
    }
    const cuuint64_t dims[2] = {(cuuint64_t)N, (cuuint64_t)T};
    const cuuint64_t strides[1] = {(cuuint64_t)N * (bytes ? 1 : 4)};
    const cuuint32_t box[2] = {(cuuint32_t)C, (cuuint32_t)U};
    const cuuint32_t estr[2] = {1, 1};
    return encode(tm, bytes ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void *>(base), dims,
                  strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// ------------------------------------------------------------------------------------------------------------------
// variant 2 (small N): a CTA stages an 8-column tile [T][8] in shared memory with full-sector loads; warp w owns column
// w and its 32 lanes split T into contiguous chunks.  Each lane folds its chunk into the affine map
// x_start = B + M * x_after, the maps are combined across lanes with a warp-shuffle (Kogge-Stone) suffix scan, and a
// second pass over the chunk applies the carried-in values.  Agrees with variant 1 to ~1e-15 relative in fp64.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kTileCols = 8;
constexpr int kScanBlock = 32 * kTileCols;

__global__ void __launch_bounds__(kScanBlock) gae_scan_kernel(const float *__restrict__ rew, const float *__restrict__ val,
                                                              const uint8_t *__restrict__ pe, const float *__restrict__ boot,
                                                              float *__restrict__ adv, float *__restrict__ ret, int T, int N,
                                                              double gamma, double gl, double *stats) {
    extern __shared__ __align__(16) unsigned char smem[];
    float *s_rew = reinterpret_cast<float *>(smem);              // [T][8]  (becomes adv)
    float *s_val = s_rew + (size_t)T * kTileCols;                // [T][8]
    float *s_boot = s_val + (size_t)T * kTileCols;               // [T][8]  (becomes ret)
    uint8_t *s_pe = reinterpret_cast<uint8_t *>(s_boot + (size_t)T * kTileCols);   // [T][8]
    const int n0 = blockIdx.x * kTileCols;
    const int tid = threadIdx.x;
    // stage: 8 consecutive threads read one 32-byte row segment
    {
        const int c = tid & (kTileCols - 1);
        const bool ok = n0 + c < N;
        for (int t = tid / kTileCols; t < T; t += kScanBlock / kTileCols) {
            const size_t i = (size_t)t * N + n0 + c;
            const int j = t * kTileCols + c;
            s_rew[j] = ok ? __ldcs(rew + i) : 0.f;
            s_val[j] = ok ? __ldcs(val + i) : 0.f;
            const uint8_t e = ok ? __ldcs(pe + i) : (uint8_t)1;
            s_pe[j] = (uint8_t)(e || t == T - 1);
            s_boot[j] = (ok && (e || t == T - 1)) ? __ldcs(boot + i) : 0.f;
        }
    }
    __syncthreads();
    const int w = tid >> 5, lane = tid & 31;
    const int L = (T + 31) / 32;
    const int t_lo = lane * L, t_hi = min(T, t_lo + L) - 1;      // chunk [t_lo, t_hi]; empty if t_lo > t_hi
    // pass 1: fold the chunk into (Ma, Ba) for advantages and (Mr, Br) for returns
    double Ma = 1.0, Ba = 0.0, Mr = 1.0, Br = 0.0;
    for (int t = t_hi; t >= t_lo; t--) {
        const int j = t * kTileCols + w;
        const bool e = s_pe[j];
        const double r = (double)s_rew[j], v = (double)s_val[j];
        const double nv = e ? (double)s_boot[j] : (double)s_val[j + kTileCols];
        const double delta = (r + gamma * nv) - v;
        // x_t = b_t + c_t * x_{t+1};  new map = (b_t + c_t*B, c_t*M)
        const double ca = e ? 0.0 : gl, cr = e ? 0.0 : gamma;
        const double br = e ? r + gamma * (double)s_boot[j] : r;
        Ba = delta + ca * Ba; Ma = ca * Ma;
        Br = br + cr * Br; Mr = cr * Mr;
    }
    // suffix scan over lanes: lane l needs the value at the start of chunk l+1, assuming zero after the last chunk
    double Sa_M = Ma, Sa_B = Ba, Sr_M = Mr, Sr_B = Br;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double oMa = __shfl_down_sync(0xffffffffu, Sa_M, o), oBa = __shfl_down_sync(0xffffffffu, Sa_B, o);
        const double oMr = __shfl_down_sync(0xffffffffu, Sr_M, o), oBr = __shfl_down_sync(0xffffffffu, Sr_B, o);
        if (lane + o < 32) {
            Sa_B = Sa_B + Sa_M * oBa; Sa_M = Sa_M * oMa;
            Sr_B = Sr_B + Sr_M * oBr; Sr_M = Sr_M * oMr;
        }
    }
    double na = __shfl_down_sync(0xffffffffu, Sa_B, 1), nr = __shfl_down_sync(0xffffffffu, Sr_B, 1);
    if (lane == 31) { na = 0.0; nr = 0.0; }
    // pass 2: apply
    double s1 = 0.0, s2 = 0.0;
    for (int t = t_hi; t >= t_lo; t--) {
        const int j = t * kTileCols + w;
        const bool e = s_pe[j];
        const double r = (double)s_rew[j], v = (double)s_val[j];
        const double b = (double)s_boot[j];
        const double nv = e ? b : (double)s_val[j + kTileCols];
        if (e) { na = 0.0; nr = b; }
        const double delta = (r + gamma * nv) - v;
        const double a = delta + gl * na;
        const double g = r + gamma * nr;
        na = a; nr = g;
        const float af = (float)a;
        s1 += (double)af; s2 += (double)af * (double)af;
        s_rew[j] = af;            // adv (rew[t] is not read again by this warp: later t only)
        s_boot[j] = (float)g;     // ret
    }
    // NOTE: s_val[j + 8] (t+1) is read by the lane that owns t, which may be a different lane than the owner of t+1;
    // values in s_val are never overwritten, s_rew/s_boot of step t are only read by the owner of t.
    __syncthreads();
    {
        const int c = tid & (kTileCols - 1);
        if (n0 + c < N) {
            for (int t = tid / kTileCols; t < T; t += kScanBlock / kTileCols) {
                const size_t i = (size_t)t * N + n0 + c;
                const int j = t * kTileCols + c;
                __stcs(adv + i, s_rew[j]);
                __stcs(ret + i, s_boot[j]);
            }
        }
    }
    if (stats) {
        if (n0 + w >= N) { s1 = 0.0; s2 = 0.0; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s1 += __shfl_down_sync(0xffffffffu, s1, o);
            s2 += __shfl_down_sync(0xffffffffu, s2, o);
        }
        if (lane == 0) {
            atomicAdd(stats, s1);
            atomicAdd(stats + 1, s2);
        }
    }
}

// `head` = elements in front of the first 16-byte boundary (0..3; handled one by one like the tail)
__global__ void __launch_bounds__(256) adv_stats_kernel(const float *__restrict__ x0, long long n0, int head, const double *center,
                                                        double *stats) {
    const double c = center ? *center : 0.0;
    double s1 = 0.0, s2 = 0.0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    if (blockIdx.x == 0 && threadIdx.x < head) {
        const double a = (double)x0[threadIdx.x] - c;
        s1 += a; s2 += a * a;
    }
    const float *x = x0 + head;
    const long long n = n0 - head;
    const long long n4 = n >> 2;
    const float4 *x4 = reinterpret_cast<const float4 *>(x);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        const float4 v = __ldcs(x4 + i);
        const double a = (double)v.x - c, b = (double)v.y - c, d = (double)v.z - c, e = (double)v.w - c;
        s1 += (a + b) + (d + e);
        s2 += (a * a + b * b) + (d * d + e * e);
    }
    for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const double a = (double)x[i] - c;
        s1 += a; s2 += a * a;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s1 += __shfl_down_sync(0xffffffffu, s1, o);
        s2 += __shfl_down_sync(0xffffffffu, s2, o);
    }
    __shared__ double sh1[8], sh2[8];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { sh1[w] = s1; sh2[w] = s2; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0;
        for (int i = 0; i < 8; i++) { a += sh1[i]; b += sh2[i]; }
        atomicAdd(stats, a);
        atomicAdd(stats + 1, b);
    }
}

__global__ void __launch_bounds__(256) adv_normalize_kernel(float *__restrict__ x0, long long n0, int head, const double *mean,
                                                            const double *std) {
    const float m = (float)*mean, s = (float)*std;      // (adv_buf - adv_mean) / adv_std on a float32 buffer P:446
    const long long stride = (long long)gridDim.x * blockDim.x;
    if (blockIdx.x == 0 && threadIdx.x < head) x0[threadIdx.x] = __fdiv_rn(x0[threadIdx.x] - m, s);
    float *x = x0 + head;
    const long long n = n0 - head;
    const long long n4 = n >> 2;
    float4 *x4 = reinterpret_cast<float4 *>(x);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        float4 v = x4[i];
        v.x = __fdiv_rn(v.x - m, s); v.y = __fdiv_rn(v.y - m, s); v.z = __fdiv_rn(v.z - m, s); v.w = __fdiv_rn(v.w - m, s);
        x4[i] = v;
    }
    for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        x[i] = __fdiv_rn(x[i] - m, s);
}

}  // namespace

extern "C" {

int rs_gae(const float *rew, const float *val, const uint8_t *path_end, const float *boot, float *adv, float *ret,
           int32_t T, int32_t N, double gamma, double lam, double *stats, int32_t variant, void *stream) {
    if (!rew || !val || !path_end || !boot || !adv || !ret) return rs_set_error("rs_gae: NULL buffer");
    if (T <= 0 || N <= 0) return rs_set_error("rs_gae: T and N must be positive");
    if (variant < 0 || variant > 15 || variant == 5 || variant == 6 || variant == 9) return rs_set_error("rs_gae: unknown variant");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const double gl = gamma * lam;
    const size_t scan_smem = (size_t)T * kTileCols * (3 * sizeof(float) + 1);
    if (variant == 0) variant = (N < 16384 && scan_smem <= 200 * 1024) ? 2 : 1;
    if (variant == 2) {
        if (scan_smem > 227 * 1024) return rs_set_error("rs_gae: T too large for the scan variant");
        if (scan_smem > 48 * 1024) {
            const cudaError_t e = cudaFuncSetAttribute(gae_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)scan_smem);
            if (e != cudaSuccess) return (int)e;
        }
        const int grid = (N + kTileCols - 1) / kTileCols;
        gae_scan_kernel<<<grid, kScanBlock, scan_smem, s>>>(rew, val, path_end, boot, adv, ret, T, N, gamma, gl, stats);
    } else {
        const int grid = (N + kColsBlock - 1) / kColsBlock;
        // 16 loads in flight per array when there are few columns; 8 (<= 72 registers, 7 CTAs per SM) when the columns
        // would otherwise not all be resident in one wave (N = 131072: 886 threads per SM)
        const bool tile_ok = (N % kColsBlock) == 0 && ((reinterpret_cast<uintptr_t>(rew) | reinterpret_cast<uintptr_t>(val) |
                                                        reinterpret_cast<uintptr_t>(path_end)) & 15) == 0;
        if (variant >= 7 && variant <= 15 && !tile_ok) return rs_set_error("rs_gae: the tile variants need N % 128 == 0 and 16-byte aligned arrays");
        // auto: the copy-engine variants whenever the tiles are whole and fill the GPU (measured on B200, T = 480:
        // N = 131072 -> 4.9 TB/s with the plain ring, N = 65536 -> 3.4 TB/s with the producer warp; register-pipelined
        // loads 3.9 / 2.7 TB/s)
        if (variant == 0 || variant == 1) {
            if (tile_ok && (long long)N >= 148LL * 128 * 4) variant = 7;
            else if (tile_ok && N >= 32768) variant = 13;     // 224-column CTAs, 2 per SM: N / 224 CTAs spread evenly
            else if (tile_ok && N >= 16384) variant = 14;     // 128-column CTAs fed by tensor-map copies
        }
        if (variant == 7)
            gae_tile_kernel<128, 8, 3, 7><<<grid, kColsBlock, 0, s>>>(rew, val, path_end, boot, adv, ret, T, N, gamma, gl, stats);
        else if (variant == 10)
            gae_tile_kernel<64, 8, 3, 14><<<N / 64, 64, 0, s>>>(rew, val, path_end, boot, adv, ret, T, N, gamma, gl, stats);
        else if (variant == 8)
            gae_tile_ws_kernel<128, 8, 3, 5><<<grid, kColsBlock + 32, 9 * 3 * 8 * kColsBlock + 2 * 3 * 8, s>>>(rew, val, path_end, boot, adv, ret, T, N, gamma, gl, stats);
        else if (variant == 11 || variant == 12 || variant == 13) {
            // 6 stages of 8 rows: mid-size rollouts (N < 75776 columns) do not fill the SMs with CTAs, so each CTA keeps more
            // bytes in flight instead.  11: 128 columns per CTA (54 KB of tiles, 4 CTAs per SM); 12: 64 columns (7 per SM);
            // 13: 224 columns (95 KB, 2 per SM) -- the widths differ in how evenly N / width CTAs spread over 148 SMs
            // (N = 65536: 512 CTAs = 3.46 per SM at width 128, 293 = 1.98 per SM at width 224)
#define RS_GAE_WS(CW, MINB)                                                                                                \
    do {                                                                                                                   \
        constexpr int sm = 9 * 6 * 8 * CW + 2 * 6 * 8;                                                                     \
        const cudaError_t e = cudaFuncSetAttribute(gae_tile_ws_kernel<CW, 8, 6, MINB>,                                     \
                                                   cudaFuncAttributeMaxDynamicSharedMemorySize, sm);                       \
        if (e != cudaSuccess) return (int)e;                                                                               \
        gae_tile_ws_kernel<CW, 8, 6, MINB><<<(N + CW - 1) / CW, CW + 32, sm, s>>>(rew, val, path_end, boot, adv, ret, T, N, \
                                                                              gamma, gl, stats);                          \
    } while (0)
            if (variant == 11) RS_GAE_WS(128, 4);
            else if (variant == 12) RS_GAE_WS(64, 7);
            else RS_GAE_WS(224, 2);
#undef RS_GAE_WS
        } else if (variant == 14 || variant == 15) {
            alignas(64) CUtensorMap tr, tv, tp;
#define RS_GAE_TMAP(CW, MINB)                                                                                              \
    do {                                                                                                                   \
        if (!make_tmap(&tr, rew, false, T, N, 8, CW) || !make_tmap(&tv, val, false, T, N, 8, CW) ||                        \
            !make_tmap(&tp, path_end, true, T, N, 8, CW))                                                                  \
            return rs_set_error("rs_gae: cuTensorMapEncodeTiled failed");                                                  \
        constexpr int sm = 9 * 6 * 8 * CW + 2 * 6 * 8;                                                                     \
        const cudaError_t e = cudaFuncSetAttribute(gae_tmap_kernel<CW, 8, 6, MINB>,                                        \
                                                   cudaFuncAttributeMaxDynamicSharedMemorySize, sm);                       \
        if (e != cudaSuccess) return (int)e;                                                                               \
        gae_tmap_kernel<CW, 8, 6, MINB><<<(N + CW - 1) / CW, CW + 32, sm, s>>>(tr, tv, tp, boot, adv, ret, T, N, gamma, gl, \
                                                                           stats);                                        \
    } while (0)
            if (variant == 14) RS_GAE_TMAP(128, 4);
            else RS_GAE_TMAP(224, 2);
#undef RS_GAE_TMAP
        } else if (variant == 3 || (variant != 4 && (long long)grid > 148LL * 4))
            gae_cols_kernel<8, 7><<<grid, kColsBlock, 0, s>>>(rew, val, path_end, boot, adv, ret, T, N, gamma, gl, stats);
        else
            gae_cols_kernel<16, 1><<<grid, kColsBlock, 0, s>>>(rew, val, path_end, boot, adv, ret, T, N, gamma, gl, stats);
    }
    return (int)cudaGetLastError();
}

int rs_adv_stats(const float *x, int64_t n, const double *center, double *stats, void *stream) {
    if (!x || !stats || n <= 0) return rs_set_error("rs_adv_stats: bad arguments");
    long long blocks = (n / 4 + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    if (blocks < 1) blocks = 1;
    if (reinterpret_cast<uintptr_t>(x) & 3) return rs_set_error("rs_adv_stats: x is not 4-byte aligned");
    const int head = (int)std::min<long long>(n, (long long)(((16 - (reinterpret_cast<uintptr_t>(x) & 15)) & 15) / 4));
    adv_stats_kernel<<<(int)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, (long long)n, head, center, stats);
    return (int)cudaGetLastError();
}

int rs_adv_normalize(float *x, int64_t n, const double *mean, const double *std, void *stream) {
    if (!x || !mean || !std || n <= 0) return rs_set_error("rs_adv_normalize: bad arguments");
    long long blocks = (n / 4 + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    if (blocks < 1) blocks = 1;
    if (reinterpret_cast<uintptr_t>(x) & 3) return rs_set_error("rs_adv_normalize: x is not 4-byte aligned");
    const int head = (int)std::min<long long>(n, (long long)(((16 - (reinterpret_cast<uintptr_t>(x) & 15)) & 15) / 4));
    adv_normalize_kernel<<<(int)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, (long long)n, head, mean, std);
    return (int)cudaGetLastError();
}

}  // extern "C"
