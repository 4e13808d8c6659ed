// Per-step bookkeeping of the batched Monte-Carlo evaluation (evaluate.py, MonteCarloEvaluator.run_team), fused into one
// elementwise launch: what EpisodeRunner.run keeps per run around env.step (E:402-419) -- episode length, the returns of
// every agent under the team mode, out-of-bounds counts, success and the agents that reached the source -- plus the count
// of runs still playing, which the host reads with a lag to stop early without draining the pipeline, and, optionally,
// the localisation error of the source prediction the policy made for the step.
// E: = /root/reference/algos/multiagent/evaluate.py
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/radsearch_b200.h"
#include "rs_error.h"

namespace {

// One thread per environment, its A agents unrolled.  Environments whose active byte is 0 on entry are not touched.
template <int A>
__global__ void __launch_bounds__(256) eval_step_kernel(const float *__restrict__ reward, const float *__restrict__ team_reward,
                                                        const uint8_t *__restrict__ done, const uint8_t *__restrict__ info,
                                                        uint8_t *__restrict__ active, uint8_t *__restrict__ success,
                                                        int32_t *__restrict__ length, double *__restrict__ ep_return,
                                                        int32_t *__restrict__ oob, uint8_t *__restrict__ finders,
                                                        int32_t *n_active, const float *__restrict__ pred,
                                                        const int32_t *__restrict__ src, double scale,
                                                        double *__restrict__ loc_err_sum, int32_t *__restrict__ loc_err_n,
                                                        float *__restrict__ loc_err_last, int n) {
    const int env = blockIdx.x * 256 + threadIdx.x;
    bool finished = false;
    if (env < n && active[env]) {
        length[env] += 1;
        const float tr = team_reward ? team_reward[env] : 0.0f;
        double sx = 0.0, sy = 0.0;
        if (pred) {
            const int2 s = reinterpret_cast<const int2 *>(src)[env];
            sx = (double)s.x;
            sy = (double)s.y;
        }
        unsigned mask = 0;
#pragma unroll
        for (int a = 0; a < A; a++) {
            const int i = env * A + a;
            ep_return[i] += (double)(reward ? reward[i] : tr);              // E:402-409: float32 rewards summed in fp64
            oob[i] += (info[i] & RS_I_OOB) != 0;
            if (done[i]) mask |= 1u << a;                                    // E:415-419
            if (pred) {
                const float2 p = reinterpret_cast<const float2 *>(pred)[i];
                if (p.x == p.x && p.y == p.y) {                              // NaN = no prediction for this agent
                    const double e = hypot((double)p.x / scale - sx, (double)p.y / scale - sy);
                    loc_err_sum[i] += e;
                    loc_err_n[i] += 1;
                    loc_err_last[i] = (float)e;
                }
            }
        }
        if (mask) {
            success[env] = 1;
            active[env] = 0;
            if (finders) finders[env] = (uint8_t)mask;
            finished = true;
        }
    }
    // one atomic per warp for the envs that finished this step (the lanes past n take part with `finished` false)
    const unsigned b = __ballot_sync(0xffffffffu, finished);
    if ((threadIdx.x & 31) == 0 && b) atomicSub(n_active, __popc(b));
}

template <int A>
void launch_eval(const float *reward, const float *team_reward, const uint8_t *done, const uint8_t *info, uint8_t *active,
                 uint8_t *success, int32_t *length, double *ep_return, int32_t *oob, uint8_t *finders, int32_t *n_active,
                 const float *pred, const int32_t *src, double scale, double *loc_err_sum, int32_t *loc_err_n,
                 float *loc_err_last, int n, cudaStream_t stream) {
    eval_step_kernel<A><<<(n + 255) / 256, 256, 0, stream>>>(reward, team_reward, done, info, active, success, length, ep_return,
                                                             oob, finders, n_active, pred, src, scale, loc_err_sum, loc_err_n,
                                                             loc_err_last, n);
}

}  // namespace

extern "C" {

int rs_eval_step(const float *reward, const float *team_reward, const uint8_t *done, const uint8_t *info, uint8_t *active,
                 uint8_t *success, int32_t *length, double *ep_return, int32_t *oob, uint8_t *finders, int32_t *n_active,
                 const float *pred, const int32_t *src, double scale, double *loc_err_sum, int32_t *loc_err_n,
                 float *loc_err_last, int32_t n_env, int32_t n_agents, int32_t individual, void *stream) {
    if (n_env <= 0) return rs_set_error("rs_eval_step: n_env must be positive");
    if (n_agents < 1 || n_agents > RS_MAX_A) return rs_set_error("rs_eval_step: n_agents out of range [1, 8]");
    if (individual ? !reward : !team_reward)
        return rs_set_error(individual ? "rs_eval_step: individual rewards need reward"
                                       : "rs_eval_step: team rewards need team_reward");
    if (!done || !info || !active || !success || !length || !ep_return || !oob || !n_active)
        return rs_set_error("rs_eval_step: NULL buffer (done / info / active / success / length / ep_return / oob / n_active)");
    if (pred && (!src || !loc_err_sum || !loc_err_n || !loc_err_last || !(scale > 0.0)))
        return rs_set_error("rs_eval_step: pred needs src / loc_err_sum / loc_err_n / loc_err_last and scale > 0");
    const float *rw = individual ? reward : nullptr, *tr = individual ? nullptr : team_reward;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
#define RS_EVAL(A_) launch_eval<A_>(rw, tr, done, info, active, success, length, ep_return, oob, finders, n_active, pred, src, \
                                    scale, loc_err_sum, loc_err_n, loc_err_last, n_env, s)
    switch (n_agents) {
        case 1: RS_EVAL(1); break;
        case 2: RS_EVAL(2); break;
        case 3: RS_EVAL(3); break;
        case 4: RS_EVAL(4); break;
        case 5: RS_EVAL(5); break;
        case 6: RS_EVAL(6); break;
        case 7: RS_EVAL(7); break;
        default: RS_EVAL(8); break;
    }
#undef RS_EVAL
    return (int)cudaGetLastError();
}

}  // extern "C"
