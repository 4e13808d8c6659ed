/* radsearch_b200 -- C ABI of the B200-native RadSearch env-step / reset / GAE path.
 *
 * This is the drop-in boundary (SURVEY.md 8b): plain pointers and sizes, no torch types.  Every buffer is owned by
 * the caller (PyTorch allocates them; pass tensor.data_ptr()); the library allocates nothing persistent, keeps no
 * mutable global state, never synchronises the host, and every launch is CUDA-graph capturable on `stream`.
 *
 * Return convention: 0 ok; <0 argument error (text in rs_last_error(), thread-local); >0 a cudaError_t.
 * Per-environment soft failures are OR-ed into RsState.status[n] (RS_ST_*), never abort.
 *
 * Reference interfaces replaced (R = /root/reference/gym_rad_search/gym_rad_search/envs/rad_search_env.py,
 * P = /root/reference/algos/multiagent/ppo.py, T = /root/reference/algos/multiagent/train.py):
 *   rs_step            R:443-728   RadSearch.step (agent_step, take_action R:876-946, is_intersect R:1133-1146,
 *                                  obstruction_sensors R:1172-1261, correct_coords R:1263-1306) + caller rules T:394-405
 *   rs_reset           R:730-797   RadSearch.reset (create_obs R:948-1011, sample_source_loc_pos R:1013-1131)
 *   rs_load_scenarios  R:799-874   RadSearch.refresh_environment
 *   rs_gae             P:391-423   PPOBuffer.GAE_advantage_and_rewardsToGO (discount_cumsum P:62-85)
 *   rs_adv_normalize   P:445-446   advantage normalisation in PPOBuffer.get (statistics: mpi_tools.py:71-95)
 *   RsConfig.standardize           per-episode running z-score of the count channel, fused into rs_step / rs_reset:
 *                                  StatisticStandardization.update/standardize (algos/multiagent/NeuralNetworkCores/
 *                                  RADTEAM_core.py:188-277) in the call order of train.py:305-311, 333-341, 436, 469, 509, 548;
 *                                  mode 2 = StatBuff (algos/test_environment/core.py:55-79) + clip to [-8, 8]
 *                                  (algos/test_environment/ppo.py:502, 518)
 *   rs_pfgru_predict / _peek / _restart   PFGRUCell.forward of the RAD-A2C source localiser
 *                                  (RADA2C_core.py:215-307) and init_hidden, for T:326, 345-353, 470-477, 509-511
 */
#ifndef RADSEARCH_B200_H
#define RADSEARCH_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RS_VERSION 3
#define RS_OBS_DIM 11            /* [count, x/2200, y/2200, 8 proximity sensors]            R:591-593 */
#define RS_MAX_K 8               /* obstruction slots (env allows 0..7)                     R:317     */
#define RS_MAX_A 8               /* agents per environment                                            */

/* rs_step / rs_reset flags */
#define RS_F_AUTO_RESET 1        /* apply T:394-405: timeout at max_ep_len, schedule a reset on done/timeout      */
#define RS_F_EPOCH_END 2         /* this is the last step of the epoch: schedule every env, new obstructions T:484 */
#define RS_F_RESET_LIST 4        /* rs_reset: reset the envs rs_step scheduled (RsState.reset_list / reset_count)  */
#define RS_F_NEW_OBSTACLES 8     /* rs_reset: draw new obstructions for every env being reset (env.epoch_end)      */
#define RS_F_FAST_POISSON 16     /* Philox path only: fp32 acceptance test in the PTRS sampler (KS-equivalent)     */
#define RS_F_PREFETCH 32         /* an env whose next episode was prefetched (RsState.nx_*, rs_prepare) adopts it    */
                                 /* with a few copies instead of recomputing it: rs_step does so for the envs it     */
                                 /* schedules (single agent), rs_reset for the envs of its work list; every env that  */
                                 /* starts an episode is appended to refill list `parity` (RS_F_ZERO_REFILL starts a  */
                                 /* list, rs_prepare drains it)                                                      */
#define RS_F_REFILL_LIST 64      /* rs_prepare: prepare the envs of refill list `parity`; else all envs            */
#define RS_F_DEVICE_CTR 128      /* read the step counter from RsState.ctr_dev (CUDA-graph replay); rs_bump_ctr     */
#define RS_F_PARITY1 256         /* which of the two refill lists rs_step / rs_reset push to (rs_prepare drains)    */
#define RS_F_BUMP_CTR 512        /* rs_reset: the last CTA to finish does what rs_bump_ctr does (needs RsState.ticket) */
#define RS_F_ZERO_REFILL 1024    /* rs_step: start refill list `parity` (refill_count[parity] = 0) before the resets   */

/* info[n][a] bits */
#define RS_I_OOB 1               /* Agent.out_of_bounds     R:919, 931 */
#define RS_I_BLOCKED 2           /* Agent.obstacle_blocking R:937 (sticky)                   */
#define RS_I_COLLISION 4         /* Agent.collision         R:909                            */
#define RS_I_LOS_BLOCKED 8       /* Agent.intersect         R:495                            */
#define RS_I_MOVED 16            /* take_action returned True                               */

/* ended[n] bits (caller rules T:394-405) */
#define RS_E_TERMINAL 1          /* any agent reported done this step                       */
#define RS_E_TIMEOUT 2           /* steps_in_episode == max_ep_len                          */
#define RS_E_RESET 4             /* a reset was scheduled for this env                      */

/* status[n] bits */
#define RS_ST_REJECT_CAP 1u      /* a rejection-sampling loop hit its cap (reference: MAX_CREATION_TRIES / hang)   */
#define RS_ST_LAMBDA_INF 2u      /* detector exactly on the source: intensity/0 (reference raises)                 */
#define RS_ST_UNIFORMS_OUT 4u    /* injected uniform stream exhausted                                              */
#define RS_ST_CORRECT_MISS 8u    /* correct_coords would never terminate (reference hangs)                         */
#define RS_ST_WALL_ASSERT 16u    /* `assert dists[i] == 0.0` in obstruction_sensors would fire                     */
#define RS_ST_COORD_RANGE 32u    /* |coordinate| > 16383: outside the exact-int32 geometry range                   */
#define RS_ST_REFILL_OVERFLOW 64u /* more resets in one block of steps than a refill list holds (the env was not listed   */
                                 /* and takes the synchronous reset path next time)                                     */

/* Environment constants (dataclass fields R:320-390 that the hot path reads). */
typedef struct RsConfig {
    int32_t bbox[4];             /* x0,y0,x1,y1                                default 0,0,2700,2700  R:321-325 */
    int32_t obs_area[2];         /* observation_area                           default 200,500        R:326     */
    int32_t enforce;             /* enforce_grid_boundaries                                           R:329     */
    int32_t n_agents;            /* number_agents                                                     R:353     */
    int32_t obstruction_count;   /* -1 random 1..5, 0..7 fixed                                        R:328     */
    int32_t count_law;           /* 0 = reference (intensity/distance + bkg, R:498-502), 1 = inverse square     */
    int32_t max_ep_len;          /* steps_per_episode                           default 120           T:394     */
    int32_t k_max;               /* obstruction slots allocated in RsState (>= max num_obs)                     */
    int32_t standardize;         /* 0 off; 1: obs[..][0] = (count - mean) / max(std, 1) with the per-episode running   */
                                 /* (Welford) sample statistics that include this reading (RADTEAM_core.py:215-265);   */
                                 /* 2: StatBuff rule (std == 0 -> 1) and the value clipped to [-8, 8].  Needs          */
                                 /* RsState.st_mean / st_m2; the raw count goes to RsState.raw_count when not NULL.     */
} RsConfig;

/* Structure-of-arrays environment state in HBM; N = envs on this rank, A = n_agents, K = k_max.  All device pointers. */
typedef struct RsState {
    int32_t *src;                /* [N][2]    source x,y                                                        */
    int32_t *rad;                /* [N][2]    intensity, background                                             */
    int32_t *rects;              /* [K][N][4] x0,y0,x1,y1 (16-byte rows; slot k of env n at (k*N+n)*4)          */
    int32_t *meta;               /* [N]       num_obs | done<<8 | (rectangles holding the source strictly inside)<<9 | ep_len<<16 */
    int32_t *det;                /* [A][N][2] detector x,y                                                      */
    double *best;                /* [A][N]    Agent.prev_det_dist (running minimum of the shortest-path length)  */
    int32_t *aflags;             /* [A][N]    out_of_bounds_count | obstacle_blocking<<24 | search seed corner<<25 */
    double *dsrc;                /* [N][4K]   shortest-path length source -> obstruction corner c (inf if none), env-major */
                                 /*           (a unit gathers its own row on demand)                                          */
    uint32_t *vis;               /* [4K][N]   corner-to-corner visibility bit masks                              */
    uint32_t *status;            /* [N]       RS_ST_* bits, sticky until cleared by the caller                   */
    int32_t *reset_list;         /* [N]       envs scheduled for reset by the last rs_step                       */
    int32_t *reset_count;        /* [1]                                                                          */
    uint32_t *epi;               /* [N]       episode sequence number: keys the reset draws (seed, env id, episode)  */
    /* prefetched next episode (optional, RS_F_PREFETCH; NULL otherwise) */
    int32_t *nx_src;             /* [N][2]                                                                        */
    int32_t *nx_det;             /* [N][2]    all agents start at the same point (R:771-773)                       */
    int32_t *nx_rad;             /* [N][2]    intensity, background | (corner of the initial shortest path << 8)   */
    double *nx_best;             /* [N]                                                                           */
    double *nx_dsrc;             /* [N][4K]   source-distance row of the prefetched episode                            */
    float *nx_obs;               /* [N][A][11] first observation of the prefetched episode                        */
    uint32_t *nx_seq;            /* [N]       episode number the prefetched scenario belongs to (0 = none)         */
    int32_t *refill_list;        /* [2][N]    envs whose prefetched scenario was consumed (two lists, ping-pong)   */
    int32_t *refill_count;       /* [2]                                                                           */
    uint64_t *ctr_dev;           /* [1]       device-side step counter (RS_F_DEVICE_CTR)                           */
    /* per-episode running statistics of the count channel (optional, RsConfig.standardize != 0; NULL otherwise).      */
    /* The number of readings seen is meta.ep_len + 1 (the reset observation, then one per step).                       */
    double *st_mean;             /* [A][N]    running mean                                RADTEAM_core.py:198         */
    double *st_m2;               /* [A][N]    aggregated squared distance from the mean   RADTEAM_core.py:200         */
    float *raw_count;            /* [N][A]    the unstandardised count of the last observation (output, nullable)     */
    uint32_t *ticket;            /* [1]       CTA completion counter of rs_reset (RS_F_BUMP_CTR), zero between launches   */
    float *dsf;                  /* [N][4K]   dsrc rounded DOWN to float (written by rs_reset / rs_load_scenarios with dsrc):  */
                                 /*           the single-agent step kernel prunes the shortest-path search on this table and   */
                                 /*           reads dsrc itself only for the corners that survive (k_max > 0)                  */
    float *nx_dsf;               /* [N][4K]   the same for the prefetched episode (with nx_dsrc)                              */
} RsState;

/* One environment step for n_env environments (all agents).  actions[N][A] in 0..8 (8 = idle), or NULL for the
 * reference's step(None) probe.  Outputs (any may be NULL except obs): obs[N][A][11] f32, reward[N][A] f32,
 * team_reward[N] f32, done[N][A] u8, info[N][A] u8 (RS_I_*), ended[N] u8 (RS_E_*), final_obs[N][A][11] f32 (written
 * only for envs that were scheduled for reset).  uniforms: NULL = Philox4x32-10 stream keyed (seed, env_id0+n, agent,
 * step_ctr); else [N][A][n_uniforms] doubles consumed in order by the Poisson sampler (numpy next_double stream). */
int rs_step(const RsConfig *cfg, const RsState *st, const int32_t *actions, float *obs, float *reward,
            float *team_reward, uint8_t *done, uint8_t *info, uint8_t *ended, float *final_obs, int32_t n_env,
            uint32_t env_id0, uint64_t seed, uint64_t step_ctr, const double *uniforms, int32_t n_uniforms,
            int32_t flags, void *stream);

/* Reset (re-sample source, detector, intensities; obstructions too where requested) and write the initial
 * observation.  Which envs: flags&RS_F_RESET_LIST -> those scheduled by rs_step; else reset_mask[N] (NULL = all).
 * New obstructions: flags&RS_F_NEW_OBSTACLES -> all of them; else new_obstacles_mask[N] (NULL = none). */
int rs_reset(const RsConfig *cfg, const RsState *st, const uint8_t *reset_mask, const uint8_t *new_obstacles_mask,
             float *obs, int32_t n_env, uint32_t env_id0, uint64_t seed, uint64_t step_ctr, const double *uniforms,
             int32_t n_uniforms, int32_t flags, void *stream);

/* Prefetch: compute the NEXT episode (number epi[n]+1) of the selected envs into RsState.nx_* without touching the
 * running episode.  The scenario is a pure function of (seed, env id, episode number, obstructions), so an env that
 * takes it from the prefetch buffer and one that is reset by rs_reset get identical state.  Intended to run on a side
 * stream / parallel graph branch next to rs_step.  flags: RS_F_REFILL_LIST (+RS_F_PARITY1) or all envs. */
int rs_prepare(const RsConfig *cfg, const RsState *st, int32_t n_env, uint32_t env_id0, uint64_t seed, int32_t flags,
               void *stream);

/* *RsState.ctr_dev += 1 and *reset_count = 0 (one thread): the tail of a captured rs_step / rs_reset sequence, so that a
 * CUDA-graph replay advances the Philox step counter and starts the next step with an empty reset list (rs_step with
 * RS_F_DEVICE_CTR does not zero it itself). */
int rs_bump_ctr(const RsState *st, void *stream);

/* Scenario injection: src[N][2], det[N][2], intensity[N], bkg[N], rects[N][k_in][4] (x0,y0,x1,y1), num_obs[N] -- all
 * int32 device arrays.  Builds the per-episode tables and writes the initial observation (a step(None) probe). */
int rs_load_scenarios(const RsConfig *cfg, const RsState *st, const int32_t *src, const int32_t *det,
                      const int32_t *intensity, const int32_t *bkg, const int32_t *rects, int32_t k_in,
                      const int32_t *num_obs, float *obs, int32_t n_env, uint32_t env_id0, uint64_t seed,
                      uint64_t step_ctr, const double *uniforms, int32_t n_uniforms, void *stream);

/* Shortest-path length source -> pts[n] (int32 [N][2], device) for every env, by the step kernel's pruned search
 * (R:491-493 semantics); out: double [N].  variant 0 = the step kernel's pruned search, 1 = plain min over all corners. */
int rs_query_shortest_path(const RsConfig *cfg, const RsState *st, const int32_t *pts, double *out, int32_t n_env,
                           int32_t variant, void *stream);

/* GAE-lambda advantages and rewards-to-go over a [T][N] rollout.  path_end[t][n] != 0 where the caller finished a
 * trajectory after step t; boot[t][n] = bootstrap value passed there (read only where path_end or t == T-1).
 * stats (nullable): double[2] device accumulators += {sum(adv), sum(adv^2)} (zero them first).
 * variant (defined: 0-4, 7, 8, 10-15; any other number is an argument error): 0 auto; 1 thread-per-column recurrence in the
 * reference's operation order (bit-exact vs scipy's lfilter), fed by bulk-async tile copies when N % 128 == 0 and the
 * arrays are 16-byte aligned, else by register-pipelined loads; 2 warp-shuffle scan along T (small N; each output within
 * one float32 ulp of the float64 recurrence; T * 104 bytes of shared memory, at most 227 KB).  3 / 4 force the 8- / 16-deep
 * register-pipelined form, 7 the 3-stage tile ring, 10 the same ring over 64-column tiles, 8 / 11 the producer-warp form
 * with 3 x 8 and 6 x 8 rows in flight, 12 / 13 that form over 64- / 224-column tiles, 14 / 15 the producer-warp form fed
 * by tensor-map (2-D TMA) copies over 128- / 224-column tiles -- all bit-identical to variant 1.  Variants 7-15 need whole
 * tiles (N % 128 == 0, 16-byte aligned rew / val / path_end).  Auto, with whole tiles: N >= 75776 -> 7, N >= 32768 -> 13,
 * N >= 16384 -> 14; N < 16384 with T * 104 <= 200 KB -> 2; otherwise the register-pipelined form, 8-deep when N > 75776.
 * Variant 1 is auto without the scan. */
int rs_gae(const float *rew, const float *val, const uint8_t *path_end, const float *boot, float *adv, float *ret,
           int32_t T, int32_t N, double gamma, double lam, double *stats, int32_t variant, void *stream);

/* stats[0] += sum(x - c), stats[1] += sum((x - c)^2) over n floats, fp64 accumulation; c = *center (device double,
 * NULL = 0).  Two calls give the reference's two-pass mean / population std (mpi_tools.py:71-95) with an all-reduce
 * of the two scalars in between when the envs are sharded over ranks. */
int rs_adv_stats(const float *x, int64_t n, const double *center, double *stats, void *stream);

/* x[i] = (x[i] - *mean) / *std   (device doubles)                                                     P:446 */
int rs_adv_normalize(float *x, int64_t n, const double *mean, const double *std, void *stream);

/* ---- batched PPOBuffer.get (SURVEY.md 8f-4; P:425-502) -----------------------------------------------------------
 * packed[n*T + t][0..D+5] = [obs[t][n][0..D-1], adv, ret, logp, act, source_tar x, y]: the rows of the reference's
 * np.hstack (P:456-465) in episode-major order -- column n of the rollout is one env's trajectory buffer, so every
 * episode is one contiguous slice of `packed` (P:468-486).  obs [T][N][D], adv/ret/logp/act [T][N], src [T][N][2]
 * (nullable: zeros), all f32. */
int rs_pack_rollout(const float *obs, const float *adv, const float *ret, const float *logp, const float *act,
                    const float *src, float *packed, int32_t T, int32_t N, int32_t D, void *stream);
/* Episode segmentation of the [T][N] rollout (a trajectory ends where path_end != 0 and at t = T-1).  Two passes:
 * ep_offset == NULL -> ep_count[n] = trajectories of column n; then, with ep_offset[n] = exclusive prefix sum of
 * ep_count, ep_start[e] = first row of episode e in `packed` (n*T + t_first) and ep_len[e], in (column, time) order. */
int rs_episode_table(const uint8_t *path_end, int32_t T, int32_t N, int32_t *ep_count, const int32_t *ep_offset,
                     int32_t *ep_start, int32_t *ep_len, void *stream);

/* ---- caller-side bookkeeping of a batched rollout (SURVEY.md 8a row a19; T:359-527), two elementwise launches per step ---
 * rs_rollout_pre, before the env step of time t: act_row[n] = action[n], val_row / logp_row = the policy's state value and
 * log-probability, src_row[n][2] = the source coordinates (nullable) -- row t of the rollout buffer (PPOBuffer.store P:339-381).
 * rs_rollout_post, after it: boot_row[n] = v_next[n] where the trajectory was cut (ended & RS_E_TIMEOUT, or every env when
 * last_step != 0), else 0 (T:462-487); hidden[n][0..hidden_dim) = 0 where ended != 0 and not last_step (T:509-511; nullable);
 * episode statistics (nullable as a group): ep_return[n] += reward[n], ep_steps[n] += 1, acc[0..5] += {episodes over by a
 * terminal state or the timeout, sum / sum of squares of their returns, sum of their lengths, done flags, out-of-bounds
 * flags}, *ep_min / *ep_max = extreme returns, then return and length restart where a reset was scheduled (T:361-391,
 * 493-535).  All arrays device, [n] unless noted.
 * A caller whose env step stores into the rollout buffer's rows itself (rs_step's output pointers = the rows) passes NULL
 * for obs_row / rew_row / end_row; one that replays a captured step graph with fixed output buffers has these two launches
 * copy them: obs[n][obs_dim] -> obs_row (the observation of step t), reward -> rew_row, ended -> end_row. */
int rs_rollout_pre(const int32_t *action, const float *val, const float *logp, const int32_t *src, float *act_row,
                   float *val_row, float *logp_row, float *src_row, const float *obs, float *obs_row, int32_t obs_dim,
                   int32_t n, void *stream);
int rs_rollout_post(const float *reward, const uint8_t *ended, const uint8_t *done, const uint8_t *info, const float *v_next,
                    float *boot_row, float *hidden, int32_t hidden_dim, double *ep_return, int32_t *ep_steps, double *acc,
                    double *ep_min, double *ep_max, float *rew_row, uint8_t *end_row, int32_t n, int32_t last_step,
                    void *stream);
/* The same two launches for n_agents (1..8) agents per environment (RAD-TEAM, T:321-571 multi-agent branch).  Columns are
 * env-major, column n*A + a, the memory order of rs_step's [N][A] outputs.
 * rs_rollout_pre_team: act_row / val_row / logp_row [N*A] <- action / val / logp [N][A]; pred_row [N*A][2] <- pred [N][A][2]
 * (the PFGRU's source prediction; NULL pred writes NaN = none; pred_row nullable); src_row [N*A][2] <- src[n] broadcast to
 * the env's A columns (nullable); obs_row [N*A][obs_dim] <- obs as in rs_rollout_pre (nullable).
 * rs_rollout_post_team: rew_row[n*A + a] = individual ? reward[n][a] : team_reward[n] (T:361-375; nullable);
 * end_row[n*A + a] = ended[n] (nullable); boot_row[n*A + a] = v_next[n][a] where the trajectory was cut, else 0;
 * hidden [N*A][hidden_dim] restarted where ended[n] != 0 and not last_step; episode statistics (nullable as a group) with
 * ep_return [N][A] f64 (returns of the same reward rule), ep_steps [N], acc [6][A], ep_min / ep_max [A]. */
int rs_rollout_pre_team(const int32_t *action, const float *val, const float *logp, const float *pred, const int32_t *src,
                        float *act_row, float *val_row, float *logp_row, float *pred_row, float *src_row, const float *obs,
                        float *obs_row, int32_t obs_dim, int32_t n_env, int32_t n_agents, void *stream);
int rs_rollout_post_team(const float *reward, const float *team_reward, const uint8_t *ended, const uint8_t *done,
                         const uint8_t *info, const float *v_next, float *boot_row, float *hidden, int32_t hidden_dim,
                         double *ep_return, int32_t *ep_steps, double *acc, double *ep_min, double *ep_max, float *rew_row,
                         uint8_t *end_row, int32_t n_env, int32_t n_agents, int32_t individual, int32_t last_step,
                         void *stream);

/* ---- caller-side bookkeeping of the batched Monte-Carlo evaluation (algos/multiagent/evaluate.py:333-475), one elementwise
 * launch per step ------------------------------------------------------------------------------------------------------
 * rs_eval_step, after the env step (auto-reset off), for every env n with active[n] != 0 on entry (the others are not
 * touched): length[n] += 1; ep_return[n][a] += individual ? reward[n][a] : team_reward[n] (float32 rewards summed in
 * float64, E:402-409); oob[n][a] += (info[n][a] & RS_I_OOB) != 0; when any done[n][a] != 0 (E:415-419): success[n] = 1,
 * active[n] = 0, finders[n] = bit mask of those agents (nullable) and *n_active -= 1 (one atomic per warp).
 * Localisation error (an addition, not a field of the reference's MonteCarloResults; nullable as a group): where pred
 * [N][A][2] (the policy's source prediction of the step in scaled coordinates) is not NaN, e = hypot(pred / scale - src)
 * in fp64 cm with src [N][2] int32 and scale = the env's coordinate scale; loc_err_sum[n][a] += e, loc_err_n[n][a] += 1,
 * loc_err_last[n][a] = (float)e.  active / success / finders u8 [N], length i32 [N], ep_return f64 [N][A], oob i32 [N][A],
 * n_active i32 [1], loc_err_sum f64 / loc_err_n i32 / loc_err_last f32 [N][A]. */
int rs_eval_step(const float *reward, const float *team_reward, const uint8_t *done, const uint8_t *info, uint8_t *active,
                 uint8_t *success, int32_t *length, double *ep_return, int32_t *oob, uint8_t *finders, int32_t *n_active,
                 const float *pred, const int32_t *src, double scale, double *loc_err_sum, int32_t *loc_err_n,
                 float *loc_err_last, int32_t n_env, int32_t n_agents, int32_t individual, void *stream);

/* ---- RAD-TEAM map observation (SURVEY.md 8f-1) ---------------------------------------------------------------------
 * MapsBuffer.observation_to_map (algos/multiagent/NeuralNetworkCores/RADTEAM_core.py:532-616 with its helpers :101-182
 * IntensityEstimator, :188-277 StatisticStandardization, :322-365 log-scale normalisation, :692-932 map updates) for
 * every agent's buffer of every environment, on persistent dense map stacks updated in place; MapsBuffer.reset
 * (:513-523) for the environments that start a new episode.  Module switches as shipped (PFGRU on, simple / radiation
 * normalisation off). */
#define RS_MS_CELL_RANGE 1u      /* an agent's grid cell lies outside the map (the reference raises IndexError)          */
#define RS_MS_LOG_FULL 2u        /* more readings in an episode than log_cap: the call's readings were not recorded      */
#define RS_MS_PRED_RANGE 4u      /* a source prediction lies outside the map (the reference raises IndexError)           */

typedef struct RsMapsConfig {
    int32_t n_agents;            /* A                                                                    :437      */
    int32_t dim_x, dim_y;        /* map_dimensions (27 x 27 with enforced boundaries, 147 x 147 without) :60-66    */
    int32_t base;                /* (steps_per_episode + 1) * A: base of the visit-count normalisation   :500      */
    int32_t log_cap;             /* readings an episode can record per environment (>= base + A, <= 5810: the     */
                                 /* kernels keep 4 tables in one block's shared memory, 40 * log_cap + 16 bytes,  */
                                 /* and sm_100 allows 227 KB)                                                     */
    int32_t use_prediction;      /* PFGRU: maintain the source prediction map                            :39       */
    double resolution_accuracy;  /* resolution_multiplier / scale (22.0)                                 :69-70    */
    double scale;                /* the environment's coordinate scale 1 / search_area_max  rad_search_env.py:435  */
} RsMapsConfig;

typedef struct RsMapsState {     /* caller-owned device memory; X = dim_x, Y = dim_y, cell = x * Y + y              */
    float *actor;                /* [N][A][X][Y][6] per buffer, channel innermost (channels_last): prediction, own location,    */
                                 /*                 others, readings, visits, obstacles                              :1799-1823 */
    float *critic;               /* [N][X][Y][4]    combined locations, readings, visits, obstacles (same in all A buffers) :1825-1832 */
    uint16_t *log_cell;          /* [N][log_cap]    sample table of the IntensityEstimator: cell of reading i (0xffff = none) */
    float *log_val;              /* [N][log_cap]                                                value of reading i  */
    int32_t *log_len;            /* [N]                                                                             */
    int32_t *last_cell;          /* [N][A]          tools.last_coords (-1 = none)                        :369      */
    int32_t *last_pred;          /* [N][A]          tools.last_prediction of buffer a (-1 = none)        :371      */
    double *std;                 /* [N][2]          tools.standardizer: mean, M2                         :198-200  */
    int32_t *std_count;          /* [N]                                                                  :207      */
    const float *visit_lut;      /* [log_cap + 1]   normalize_incremental_logscale(2 i, base, 2) for i = 0..log_cap :356-360 */
                                 /*                 (the shadow counter :464 is 2 x the cell's samples recorded so far)      */
    uint32_t *status;            /* [N]             RS_MS_* bits                                                    */
} RsMapsState;

/* observation_to_map for all A buffers of the selected environments: mask[N] u8 (NULL = all), env n is selected when
 * mask[n] & mask_bits != 0 (mask_bits 0 = any non-zero byte; pass rs_step's ended[] with RS_E_RESET to follow the env's
 * auto-resets without an intermediate mask).  obs[N][A][11] f32 as
 * written by rs_step / rs_reset (raw counts); loc_pred[N][A][2] f32 = the source location predicted for agent a's
 * buffer in scaled coordinates (NULL or NaN = none). */
int rs_maps_update(const RsMapsConfig *cfg, const RsMapsState *st, const float *obs, const float *loc_pred,
                   const uint8_t *mask, int32_t mask_bits, int32_t n_env, void *stream);
/* MapsBuffer.reset for the selected environments (mask NULL = all). */
int rs_maps_reset(const RsMapsConfig *cfg, const RsMapsState *st, const uint8_t *mask, int32_t mask_bits, int32_t n_env,
                  void *stream);
/* Map stacks for the PPO update, rebuilt from a rollout buffer instead of stored (one step's stacks are 4*(6A+4)*X*Y
 * bytes per env; the inputs of the calls that made them are 52*A).  For each range i = (n, t0, t1) of ranges[m][3]
 * (device), rows out_row0[i] .. out_row0[i] + t1 - t0 of out_actor [R][A][X][Y][6] / out_critic [R][X][Y][4] receive the
 * stacks rs_maps_update had produced when the policy read env n's observation of step t = t0..t1: the calls on
 * obs_rows[s..t] with pred_rows[s..t], s = 1 + the last path end before t in column n*A of end_rows (or 0).  A range
 * may cross path ends; the replay restarts there.  obs_rows [T+1][N][A][11] (row t = what the policy saw at step t),
 * pred_rows [T][N][A][2] (NaN = none; NULL = no predictions), end_rows [T][N*A] (the rollout buffer's path-end bytes).
 * st: only visit_lut is read; nothing of the live state is read or written.  out_status[i] = the RS_MS_* bits of the
 * replayed calls | RS_MR_BAD_RANGE when n is outside [0, N) or t0..t1 leaves [0, T) (its rows are zeroed) or t1 < t0
 * (it owns no rows). */
#define RS_MR_BAD_RANGE 8u
int rs_maps_replay(const RsMapsConfig *cfg, const RsMapsState *st, const float *obs_rows, const float *pred_rows,
                   const uint8_t *end_rows, int32_t T, int32_t n_env, const int32_t *ranges, int32_t m,
                   const int64_t *out_row0, float *out_actor, float *out_critic, uint32_t *out_status, void *stream);
int rs_sizeof_maps_config(void);
int rs_sizeof_maps_state(void);

/* ---- fused GRU actor-critic inference (the RAD-A2C core, algos/test_environment/core.py) ----------------------------
 * torch.nn.GRUCell(d_in, hidden) -> policy head over the 8 moves and value head, one thread per row m of the batch (env-
 * major n*A + a for multi-agent batches), float32 throughout (no tensor cores).  params: the packed weights in torch's
 * row-major order, weight_ih [3H][d_in] | weight_hh [3H][H] | bias_ih | bias_hh | policy head (W1, b1, W2, b2, or W, b)
 * | value head (the same), rs_policy_param_count floats.  obs [rows][11], pred [rows][2] (the last two input columns, only
 * with d_in = 13, NULL otherwise), hidden [rows][H]. */
typedef struct RsPolicyConfig {
    int32_t d_in;                /* 11, or 13 (obs + a caller-supplied source prediction)                         */
    int32_t hidden;              /* H, 1..64                                                                      */
    int32_t pi_hidden;           /* 0 = Linear(H, 8); P in 1..64 = Linear(H, P), activation, Linear(P, 8)          */
    int32_t v_hidden;            /* 0 = Linear(H, 1); V in 1..64 = Linear(H, V), activation, Linear(V, 1)          */
    int32_t activation;          /* 0 tanh, 1 relu (both heads)                                                   */
} RsPolicyConfig;
/* floats in the packed buffer; < 0 for a config outside the ranges above */
int rs_policy_param_count(const RsPolicyConfig *cfg);
/* hidden <- GRUCell(x, hidden) in place (torch's gate order r, z, n; h' = n + z (h - n)); value = value head of h';
 * logp = log_softmax of the policy head at the sampled action; action (int32) = the first index of the maximum of
 * logp_k + g_k, g_k = -log(-log u_k), u_k = ((x_k >> 8) + 0.5) 2^-24 for the 8 words x_k of Philox4x32-10 with key seed
 * and counters (row_id0 + m, 4<<24 | b, *ctr lo, *ctr hi), b = 0, 1.  ctr: device uint64, read by every CTA and advanced
 * by one by the last CTA to finish (ticket: device uint32, zero between launches), so a captured call draws fresh noise
 * on every replay.  row_id0 + rows <= 2^32: the global row id makes the actions independent of how rows shard. */
int rs_policy_act(const RsPolicyConfig *cfg, const float *params, const float *obs, const float *pred, float *hidden,
                  int32_t *action, float *value, float *logp, int rows, uint32_t row_id0, uint64_t seed, uint64_t *ctr,
                  uint32_t *ticket, void *stream);
/* value = value head of GRUCell(x, hidden), hidden not written: the bootstrap value of the next observation (T:462-487). */
int rs_policy_value(const RsPolicyConfig *cfg, const float *params, const float *obs, const float *pred,
                    const float *hidden, float *value, int rows, void *stream);
int rs_sizeof_policy_config(void);

/* ---- PPO loss and gradient of the same actor-critic (the update's forward and backpropagation through time) --------
 * One launch: the clipped PPO loss of M columns x T steps of a BatchedPPOBuffer, in its own [T][N] layout, and its exact
 * gradient with respect to every packed parameter.  obs [T][N][11], pred [T][N][2] (d_in = 13 only), act [T][N] (float
 * action indices), adv [T][N] (normalised), ret, logp [T][N], end [T][N] (uint8 path ends).  columns: int32 [M], the
 * buffer columns of the minibatch (NULL: all of them, M = N).  Column m starts from h = 0 at t = 0 and step t reads
 * h_{t-1} (1 - end[t-1]), the restart rule of rs_rollout_post.  With c = 1 / (T M), rho = exp(logp(a) - logp_old) and
 * eps = clip_ratio,
 *     L = w_pi c sum -min(rho A, clamp(rho, 1 - eps, 1 + eps) A) + w_v c sum (v - ret)^2
 * and grad (rs_policy_param_count floats, overwritten) = dL/dparams with torch autograd's conventions (minimum splits a
 * tie evenly, clamp passes the gradient on the closed interval).  stats (8 doubles, [0..5] written): sum -min(...),
 * sum (v - ret)^2, sum (logp_old - logp), sum of the policy's entropy, rows with |rho - 1| > eps, and rows skipped (a
 * column index outside 0..N-1 skips its T rows; an action outside 0..7 its row; skipped rows add nothing).  workspace:
 * rs_policy_grad_workspace_bytes, device memory (the hidden states of every step, [T][M][H] floats, and per-CTA
 * partials); ticket: device uint32, zero between launches.  No host synchronisation; CUDA-graph capturable; the result
 * is bit-identical from call to call. */
int64_t rs_policy_grad_workspace_bytes(const RsPolicyConfig *cfg, int32_t T, int32_t M);
int rs_policy_ppo_grad(const RsPolicyConfig *cfg, const float *params, const float *obs, const float *pred, const float *act,
                       const float *adv, const float *ret, const float *logp, const uint8_t *end, const int32_t *columns,
                       int32_t T, int32_t N, int32_t M, double clip_ratio, double w_pi, double w_v, float *grad,
                       double *stats, void *workspace, uint32_t *ticket, void *stream);

/* ---- fused PFGRU source localiser inference (the particle-filter GRU of RAD-A2C, RADA2C_core.py:215-307) -----------
 * One warp per row m of the batch (env-major n*A + a), float32 throughout (no tensor cores).  State: particles
 * [rows][K][H] and log_weights [rows][K], float32.  x = obs[m][0 .. d_in) (obs [rows][11]).  One step, with [a | b] the
 * concatenation hidden part first:
 *   z = sigmoid(fc_z[h0 | x]), r = sigmoid(fc_r[h0 | x]), (mu, nu) = fc_n[r h0 | x] (first H outputs mu, next H nu),
 *   n = tanh(mu + eps softplus(nu)), eps ~ N(0, 1) per element, h1 = (1 - z) n + z h0,
 *   p1 = log_softmax(fc_obs[h1 | x] + p0) over the K particles;
 *   resample = 1: q = alpha exp(p1) + (1 - alpha) / K, i_k = the first i with u_k C_{K-1} < C_i (C the prefix sum of q in
 *   particle order), h_k = h1[i_k], p_k = p1[i_k] - log(alpha w + (1 - alpha) / K), w = exp(p1[i_k]), p -= logsumexp(p);
 *   resample = 0: h = h1, p = p1;
 *   pred = hid_obs(sum_k exp(p_k) h_k), hid_obs = Linear(H, W) -> ReLU -> Linear(W, 2).
 * params: fc_z.weight, fc_z.bias, fc_r.*, fc_n.*, fc_obs.*, hid_obs[0].*, hid_obs[2].*, torch row-major,
 * rs_pfgru_param_count floats.
 * Noise: Philox4x32-10 with key seed and counter (row_id0 + m, 5<<24 | block, *ctr lo, *ctr hi); every word x gives the
 * uniform ((x >> 8) + 0.5) 2^-24.  Blocks: predict eps of particle k, elements 4g..4g+3: k*16 + g (Box-Muller: eps_4g =
 * sqrt(-2 ln u0) cos 2pi u1, eps_4g+1 = sqrt(-2 ln u0) sin 2pi u1, eps_4g+2/3 the same of u2, u3); predict u_k: 1024 + k/4,
 * word k%4; peek: 2048 + the predict blocks; restart element j of particle k: 4096 + k*16 + j/4, word j%4.  ctr: device
 * uint64, read by all three calls and advanced by one by the last CTA of a predict (ticket: device uint32, zero between
 * launches), so a captured predict draws fresh noise on every replay.  row_id0 + rows <= 2^32: the global row id makes
 * the results independent of how rows shard.  mask[rows] u8 (NULL = all rows): row m is selected when mask[m] &
 * mask_bits != 0 (mask_bits 0 = any non-zero byte).  All calls are asynchronous and CUDA-graph capturable. */
typedef struct RsPfgruConfig {
    int32_t d_in;                /* input columns taken from the observation, 1..11 (the reference: 3)              */
    int32_t hidden;              /* H, 1..64                                                                      */
    int32_t particles;           /* K, 1..64                                                                      */
    int32_t obs_hidden;          /* W, the hidden width of hid_obs, 1..64                                         */
    int32_t resample;            /* 1: soft resampling after every step, 0: none                                  */
    float alpha;                 /* soft-resampling alpha, (0, 1]                                                 */
} RsPfgruConfig;
/* floats in the packed buffer; < 0 for a config outside the ranges above */
int rs_pfgru_param_count(const RsPfgruConfig *cfg);
/* one step of every row: the state is replaced in place, pred_out [rows][2] written */
int rs_pfgru_predict(const RsPfgruConfig *cfg, const float *params, const float *obs, float *particles, float *log_weights,
                     float *pred_out, int32_t rows, uint32_t row_id0, uint64_t seed, uint64_t *ctr, uint32_t *ticket,
                     void *stream);
/* the same step on the current state of the selected rows, pred_out written for those rows only; the state and ctr are
 * not written */
int rs_pfgru_peek(const RsPfgruConfig *cfg, const float *params, const float *obs, const float *particles,
                  const float *log_weights, float *pred_out, const uint8_t *mask, int32_t mask_bits, int32_t rows,
                  uint32_t row_id0, uint64_t seed, const uint64_t *ctr, void *stream);
/* restart of the selected rows: h ~ U[0, 1) per element, p = -log K */
int rs_pfgru_restart(const RsPfgruConfig *cfg, float *particles, float *log_weights, const uint8_t *mask, int32_t mask_bits,
                     int32_t rows, uint32_t row_id0, uint64_t seed, const uint64_t *ctr, void *stream);
int rs_sizeof_pfgru_config(void);

const char *rs_last_error(void);
int rs_version(void);
/* sizeof checks for the binding */
int rs_sizeof_config(void);
int rs_sizeof_state(void);

#ifdef __cplusplus
}
#endif
#endif
