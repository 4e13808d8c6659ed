// Caller-side bookkeeping of the batched rollout (SURVEY.md 8a row a19: the rules train.py applies around env.step), fused
// into two elementwise launches per step so that a rollout of N environments costs a handful of launches per step instead
// of a few dozen tiny tensor operations:
//   rs_rollout_pre   before the env step: the policy's action / state value / log-probability and the source coordinates of
//                    step t go into row t of the rollout buffer (PPOBuffer.store P:339-381; T:416-428)
//   rs_rollout_post  after the env step: bootstrap value of the trajectories that were cut (T:462-487), restart of the
//                    recurrent state of the envs whose episode ended (T:509-511), EpRet / EpLen / DoneCount / OutOfBound
//                    bookkeeping (T:361-391, 493-527) -- what rollout_stats.EpisodeStats.update does with tensor ops
// rs_rollout_pre_team / rs_rollout_post_team are the same two launches for A agents per environment (the RAD-TEAM
// branch): columns are env-major (column n*A + a, the memory order of the env's [N][A] outputs), the env-level inputs
// (source coordinates, team reward, path-end byte, episode length) are broadcast to the A columns of their env.  The
// single-agent entry points run the same kernels with A = 1.
// T: = /root/reference/algos/multiagent/train.py, P: = /root/reference/algos/multiagent/ppo.py
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/radsearch_b200.h"
#include "rs_error.h"

namespace {

// one thread per column i = n * A + a
__global__ void __launch_bounds__(256) rollout_pre_kernel(const int32_t *__restrict__ action, const float *__restrict__ val,
                                                          const float *__restrict__ logp, const float *__restrict__ pred,
                                                          const int32_t *__restrict__ src, float *__restrict__ act_row,
                                                          float *__restrict__ val_row, float *__restrict__ logp_row,
                                                          float *__restrict__ pred_row, float *__restrict__ src_row,
                                                          const float *__restrict__ obs, float *__restrict__ obs_row, int obs_dim,
                                                          int n, int n_agents) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (obs_row)        // the observation the policy just saw -> row t (a caller whose env step writes into fixed buffers)
        for (int j = i; j < n * obs_dim; j += gridDim.x * 256) obs_row[j] = obs[j];
    if (i >= n) return;
    act_row[i] = (float)action[i];
    val_row[i] = val[i];
    logp_row[i] = logp[i];
    if (pred_row)       // the source prediction the maps were updated with (NaN = none): what a replay of the maps needs
        reinterpret_cast<float2 *>(pred_row)[i] =
            pred ? reinterpret_cast<const float2 *>(pred)[i] : make_float2(__int_as_float(0x7fffffff), __int_as_float(0x7fffffff));
    if (src_row) {
        const int2 s = reinterpret_cast<const int2 *>(src)[n_agents == 1 ? i : i / n_agents];
        reinterpret_cast<float2 *>(src_row)[i] = make_float2((float)s.x, (float)s.y);
    }
}

__device__ __forceinline__ void atomic_min_f64(double *p, double v) {
    unsigned long long *q = reinterpret_cast<unsigned long long *>(p);
    unsigned long long old = *q;
    while (__longlong_as_double((long long)old) > v) {
        const unsigned long long seen = atomicCAS(q, old, (unsigned long long)__double_as_longlong(v));
        if (seen == old) break;
        old = seen;
    }
}
__device__ __forceinline__ void atomic_max_f64(double *p, double v) {
    unsigned long long *q = reinterpret_cast<unsigned long long *>(p);
    unsigned long long old = *q;
    while (__longlong_as_double((long long)old) < v) {
        const unsigned long long seen = atomicCAS(q, old, (unsigned long long)__double_as_longlong(v));
        if (seen == old) break;
        old = seen;
    }
}

// One thread per environment, its A columns n * A + a in a loop.  reward [N][A] (its own reward per agent) or team_reward
// [N] (shared by the A agents) feeds the reward row and the returns; ended / ep_steps are per environment; ep_return [N][A],
// acc [6][A], ep_min / ep_max [A].
template <int A>
__global__ void __launch_bounds__(256) rollout_post_kernel(const float *__restrict__ reward, const float *__restrict__ team_reward,
                                                           const uint8_t *__restrict__ ended, const uint8_t *__restrict__ done,
                                                           const uint8_t *__restrict__ info, const float *__restrict__ v_next,
                                                           float *__restrict__ boot_row, float *__restrict__ hidden, int hidden_dim,
                                                           double *__restrict__ ep_return, int32_t *__restrict__ ep_steps,
                                                           double *acc, double *ep_min, double *ep_max, float *__restrict__ rew_row,
                                                           uint8_t *__restrict__ end_row, int n, int last_step) {
    const int env = blockIdx.x * 256 + threadIdx.x;
    double a[A][6];                                          // per agent: episodes, sum EpRet, sum EpRet^2, sum EpLen, DoneCount, OutOfBound
#pragma unroll
    for (int b = 0; b < A; b++)
#pragma unroll
        for (int k = 0; k < 6; k++) a[b][k] = 0.0;
    if (env < n) {
        const int e = ended[env];
        // T:462-487: a trajectory cut by the timeout, or by the epoch's last step, is bootstrapped with V(next observation)
        const bool cut = last_step ? true : (e & RS_E_TIMEOUT) != 0;
        const bool reset = (e & RS_E_RESET) != 0;                            // env.reset() follows T:530-535
        const int steps = ep_return ? ep_steps[env] + 1 : 0;
#pragma unroll
        for (int b = 0; b < A; b++) {
            const int i = env * A + b;
            const float r = team_reward ? team_reward[env] : reward ? reward[i] : 0.0f;   // T:361-375
            if (rew_row) rew_row[i] = r;                     // (a caller whose env step writes into fixed buffers)
            if (end_row) end_row[i] = (uint8_t)e;
            boot_row[i] = cut ? v_next[i] : 0.0f;
            if (hidden && !last_step && e != 0)                              // T:509-511
                for (int h = 0; h < hidden_dim; h++) hidden[(size_t)i * hidden_dim + h] = 0.0f;
            if (ep_return) {
                const double ret = ep_return[i] + (double)r;                 // T:361-375
                a[b][4] = done[i] != 0;                                      // T:388-391
                a[b][5] = (info[i] & RS_I_OOB) != 0;                         // T:378-384
                if (e & (RS_E_TERMINAL | RS_E_TIMEOUT)) {                    // episode_over T:394-400, logged T:493-500
                    a[b][0] = 1.0; a[b][1] = ret; a[b][2] = ret * ret; a[b][3] = (double)steps;
                    atomic_min_f64(ep_min + b, ret);
                    atomic_max_f64(ep_max + b, ret);
                }
                ep_return[i] = reset ? 0.0 : ret;
            }
        }
        if (ep_return) ep_steps[env] = reset ? 0 : steps;
    }
    if (acc) {
#pragma unroll
        for (int b = 0; b < A; b++)
#pragma unroll
            for (int k = 0; k < 6; k++) {
                double v = a[b][k];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
                if ((threadIdx.x & 31) == 0 && v != 0.0) atomicAdd(acc + k * A + b, v);
            }
    }
}

template <int A>
void launch_post(const float *reward, const float *team_reward, const uint8_t *ended, const uint8_t *done, const uint8_t *info,
                 const float *v_next, float *boot_row, float *hidden, int hidden_dim, double *ep_return, int32_t *ep_steps,
                 double *acc, double *ep_min, double *ep_max, float *rew_row, uint8_t *end_row, int n, int last_step,
                 cudaStream_t stream) {
    rollout_post_kernel<A><<<(n + 255) / 256, 256, 0, stream>>>(reward, team_reward, ended, done, info, v_next, boot_row, hidden,
                                                                hidden_dim, ep_return, ep_steps, ep_return ? acc : nullptr,
                                                                ep_min, ep_max, rew_row, end_row, n, last_step);
}

}  // namespace

extern "C" {

int rs_rollout_pre(const int32_t *action, const float *val, const float *logp, const int32_t *src, float *act_row,
                   float *val_row, float *logp_row, float *src_row, const float *obs, float *obs_row, int32_t obs_dim,
                   int32_t n, void *stream) {
    if (!action || !val || !logp || !act_row || !val_row || !logp_row) return rs_set_error("rs_rollout_pre: NULL buffer");
    if (src_row && !src) return rs_set_error("rs_rollout_pre: src_row without src");
    if (obs_row && (!obs || obs_dim <= 0)) return rs_set_error("rs_rollout_pre: obs_row without obs");
    if (n <= 0) return rs_set_error("rs_rollout_pre: n must be positive");
    rollout_pre_kernel<<<(n + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        action, val, logp, nullptr, src, act_row, val_row, logp_row, nullptr, src_row, obs, obs_row, obs_dim, n, 1);
    return (int)cudaGetLastError();
}

int rs_rollout_post(const float *reward, const uint8_t *ended, const uint8_t *done, const uint8_t *info, const float *v_next,
                    float *boot_row, float *hidden, int32_t hidden_dim, double *ep_return, int32_t *ep_steps, double *acc,
                    double *ep_min, double *ep_max, float *rew_row, uint8_t *end_row, int32_t n, int32_t last_step,
                    void *stream) {
    if (!ended || !v_next || !boot_row) return rs_set_error("rs_rollout_post: NULL buffer");
    if (rew_row && !reward) return rs_set_error("rs_rollout_post: rew_row without reward");
    if (ep_return && (!reward || !done || !info || !ep_steps || !acc || !ep_min || !ep_max))
        return rs_set_error("rs_rollout_post: episode statistics need reward / done / info / ep_steps / acc / ep_min / ep_max");
    if (n <= 0 || (hidden && hidden_dim <= 0)) return rs_set_error("rs_rollout_post: bad sizes");
    launch_post<1>(reward, nullptr, ended, done, info, v_next, boot_row, hidden, hidden_dim, ep_return, ep_steps, acc, ep_min,
                   ep_max, rew_row, end_row, n, last_step, static_cast<cudaStream_t>(stream));
    return (int)cudaGetLastError();
}

int rs_rollout_pre_team(const int32_t *action, const float *val, const float *logp, const float *pred, const int32_t *src,
                        float *act_row, float *val_row, float *logp_row, float *pred_row, float *src_row, const float *obs,
                        float *obs_row, int32_t obs_dim, int32_t n_env, int32_t n_agents, void *stream) {
    if (!action || !val || !logp || !act_row || !val_row || !logp_row) return rs_set_error("rs_rollout_pre_team: NULL buffer");
    if (src_row && !src) return rs_set_error("rs_rollout_pre_team: src_row without src");
    if (obs_row && (!obs || obs_dim <= 0)) return rs_set_error("rs_rollout_pre_team: obs_row without obs");
    if (pred && !pred_row) return rs_set_error("rs_rollout_pre_team: pred without pred_row");
    if (n_env <= 0) return rs_set_error("rs_rollout_pre_team: n_env must be positive");
    if (n_agents < 1 || n_agents > RS_MAX_A) return rs_set_error("rs_rollout_pre_team: n_agents out of range [1, 8]");
    const int n = n_env * n_agents;
    rollout_pre_kernel<<<(n + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        action, val, logp, pred, src, act_row, val_row, logp_row, pred_row, src_row, obs, obs_row, obs_dim, n, n_agents);
    return (int)cudaGetLastError();
}

int rs_rollout_post_team(const float *reward, const float *team_reward, const uint8_t *ended, const uint8_t *done,
                         const uint8_t *info, const float *v_next, float *boot_row, float *hidden, int32_t hidden_dim,
                         double *ep_return, int32_t *ep_steps, double *acc, double *ep_min, double *ep_max, float *rew_row,
                         uint8_t *end_row, int32_t n_env, int32_t n_agents, int32_t individual, int32_t last_step,
                         void *stream) {
    if (!ended || !v_next || !boot_row) return rs_set_error("rs_rollout_post_team: NULL buffer");
    const float *r = individual ? reward : team_reward;
    if ((rew_row || ep_return) && !r)
        return rs_set_error(individual ? "rs_rollout_post_team: individual rewards need reward"
                                       : "rs_rollout_post_team: team rewards need team_reward");
    if (ep_return && (!done || !info || !ep_steps || !acc || !ep_min || !ep_max))
        return rs_set_error("rs_rollout_post_team: episode statistics need done / info / ep_steps / acc / ep_min / ep_max");
    if (n_env <= 0 || (hidden && hidden_dim <= 0)) return rs_set_error("rs_rollout_post_team: bad sizes");
    if (n_agents < 1 || n_agents > RS_MAX_A) return rs_set_error("rs_rollout_post_team: n_agents out of range [1, 8]");
    const float *rw = individual ? reward : nullptr, *tr = individual ? nullptr : team_reward;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
#define RS_POST(A_) launch_post<A_>(rw, tr, ended, done, info, v_next, boot_row, hidden, hidden_dim, ep_return, ep_steps, acc, \
                                    ep_min, ep_max, rew_row, end_row, n_env, last_step, s)
    switch (n_agents) {
        case 1: RS_POST(1); break;
        case 2: RS_POST(2); break;
        case 3: RS_POST(3); break;
        case 4: RS_POST(4); break;
        case 5: RS_POST(5); break;
        case 6: RS_POST(6); break;
        case 7: RS_POST(7); break;
        default: RS_POST(8); break;
    }
#undef RS_POST
    return (int)cudaGetLastError();
}

}  // extern "C"
