// Batched PPOBuffer.get() (SURVEY.md 8f-4): the per-step rows the reference stacks for its episode tensors and the
// episode segmentation, for the [T][N] rollout buffer.
// P: = /root/reference/algos/multiagent/ppo.py
//   get() P:425-502: np.hstack((obs_buf, adv, ret, logp, act, source_tar)) P:456-465, then one slice per episode P:468-486
//
// The reference slices ONE trajectory buffer (one env) by episode lengths.  In the batched buffer column n plays that
// env, so the episode-major order is column-major: row n*T + t.  rs_pack_rollout is therefore a fused concat + tiled
// transpose ([T][N][*] -> [N][T][D+6]): reads coalesced along N, staged in shared memory, written as contiguous
// 32-step x (D+6)-float runs; every episode is then one contiguous slice of `packed`, described by rs_episode_table.
// HBM bound: 4*(D+6) bytes read + 4*(D+6) bytes written per [t][n] element (136 B at D = 11).
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/radsearch_b200.h"
#include "rs_error.h"

namespace {

constexpr int kTT = 32, kTN = 16, kPackBlock = 256;

__global__ void __launch_bounds__(kPackBlock) pack_rollout_kernel(const float *__restrict__ obs, const float *__restrict__ adv,
                                                                  const float *__restrict__ ret, const float *__restrict__ logp,
                                                                  const float *__restrict__ act, const float *__restrict__ src,
                                                                  float *__restrict__ packed, int T, int N, int D) {
    extern __shared__ float tile[];                      // [kTN][kTT][W]
    const int W = D + 6;
    const int t0 = blockIdx.y * kTT, n0 = blockIdx.x * kTN;
    const int tt = min(kTT, T - t0), tn = min(kTN, N - n0);
    // observations: for a fixed step the tile's columns are one contiguous run of tn*D floats
    for (int i = threadIdx.x; i < tt * tn * D; i += kPackBlock) {
        const int t = i / (tn * D), r = i - t * tn * D, n = r / D, d = r - n * D;
        tile[(n * kTT + t) * W + d] = obs[((size_t)(t0 + t) * N + n0) * D + r];
    }
    for (int i = threadIdx.x; i < tt * tn; i += kPackBlock) {
        const int t = i / tn, n = i - t * tn;
        const size_t g = (size_t)(t0 + t) * N + n0 + n;
        float *row = tile + (n * kTT + t) * W + D;
        row[0] = adv[g]; row[1] = ret[g]; row[2] = logp[g]; row[3] = act[g];
        row[4] = src ? src[2 * g] : 0.0f;
        row[5] = src ? src[2 * g + 1] : 0.0f;
    }
    __syncthreads();
    // column n of the tile: tt*W contiguous floats of `packed`
    for (int i = threadIdx.x; i < tn * tt * W; i += kPackBlock) {
        const int n = i / (tt * W), r = i - n * tt * W;
        packed[((size_t)(n0 + n) * T + t0) * W + r] = tile[n * kTT * W + r];
    }
}

// pass 1 (ep_offset == nullptr): ep_count[n] = trajectories of column n (a path end at t, or t == T-1).
// pass 2: their start rows / lengths in time order, written from slot ep_offset[n].
__global__ void episode_table_kernel(const uint8_t *__restrict__ path_end, int T, int N, int32_t *ep_count,
                                     const int32_t *ep_offset, int32_t *ep_start, int32_t *ep_len) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    int cnt = 0, start = 0;
    const int base = ep_offset ? ep_offset[n] : 0;
    for (int t = 0; t < T; t++) {
        if (path_end[(size_t)t * N + n] || t == T - 1) {
            if (ep_offset) {
                ep_start[base + cnt] = n * T + start;
                ep_len[base + cnt] = t + 1 - start;
            }
            cnt++;
            start = t + 1;
        }
    }
    if (!ep_offset) ep_count[n] = cnt;
}

}  // namespace

extern "C" {

int rs_pack_rollout(const float *obs, const float *adv, const float *ret, const float *logp, const float *act,
                    const float *src, float *packed, int32_t T, int32_t N, int32_t D, void *stream) {
    if (!obs || !adv || !ret || !logp || !act || !packed) return rs_set_error("rs_pack_rollout: NULL buffer");
    if (T <= 0 || N <= 0 || D <= 0 || D > 64) return rs_set_error("rs_pack_rollout: bad T / N / D");
    const dim3 grid((N + kTN - 1) / kTN, (T + kTT - 1) / kTT);
    const size_t smem = (size_t)kTN * kTT * (D + 6) * sizeof(float);
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(pack_rollout_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
    }
    pack_rollout_kernel<<<grid, kPackBlock, smem, static_cast<cudaStream_t>(stream)>>>(obs, adv, ret, logp, act, src, packed,
                                                                                      T, N, D);
    return (int)cudaGetLastError();
}

int rs_episode_table(const uint8_t *path_end, int32_t T, int32_t N, int32_t *ep_count, const int32_t *ep_offset,
                     int32_t *ep_start, int32_t *ep_len, void *stream) {
    if (!path_end || T <= 0 || N <= 0) return rs_set_error("rs_episode_table: bad arguments");
    if (!ep_offset && !ep_count) return rs_set_error("rs_episode_table: the counting pass needs ep_count");
    if (ep_offset && (!ep_start || !ep_len)) return rs_set_error("rs_episode_table: the table pass needs ep_start / ep_len");
    episode_table_kernel<<<(N + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(path_end, T, N, ep_count, ep_offset,
                                                                                        ep_start, ep_len);
    return (int)cudaGetLastError();
}

}  // extern "C"
