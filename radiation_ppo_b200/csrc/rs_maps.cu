// RAD-TEAM map observation on the device (SURVEY.md 8f-1): MapsBuffer.observation_to_map for every agent's buffer of
// every environment in one launch, on PERSISTENT dense map stacks in HBM that are updated sparsely in place.
// M: = /root/reference/algos/multiagent/NeuralNetworkCores/RADTEAM_core.py
//   observation_to_map M:532-616, _inflate_coordinates M:692-715, _update_* M:748-932, IntensityEstimator M:101-182,
//   StatisticStandardization M:188-277, normalize_incremental_logscale M:322-365, reset / _clear_maps M:513-530, 618-667
//
// The reference keeps one MapsBuffer per agent and feeds each of them the SAME observation dict every step, so the
// readings / visit-count / obstacle / combined-location maps, the sample table and the running standardiser are
// identical in the A buffers of an environment: they are computed once per environment and written to the agents'
// actor stacks and to the (shared) critic stack.  Only the agent's own location, the others' locations and the source
// prediction differ per buffer.
//
// One warp per environment.  Per call and environment the work is: the episode's sample table (<= (T+1)*A readings, 6
// bytes each) staged into shared memory, per agent a compaction + rank selection among the samples of its cell, and
// ~6*A*A scattered 4-byte STORES -- the location counts are recomputed from the agents' recorded cells and the visit
// counter from the sample table, so no map is ever read back.  Bound by the random 32-byte-sector traffic of those stores
// (every partially written sector is filled from DRAM first): the stacks are therefore stored CHANNEL-INNERMOST
// ([X][Y][6], torch's channels_last), so that the 4-5 values a call writes for one cell of one buffer share one or two
// sectors instead of one sector per channel plane (round 1: 117 sector fills per call and environment, now ~50).  The
// dense stacks are never rewritten; the policy's convolutions read them where they lie (channels_last is cuDNN's
// native layout).
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/radsearch_b200.h"
#include "rs_error.h"
#include "rs_rcp.cuh"

namespace {

constexpr int kWarpsPerBlock = 4;
constexpr int kBlock = 32 * kWarpsPerBlock;
// Dynamic shared memory of maps_update_kernel / maps_replay_kernel: per warp the sample table (value, cell) and the
// compaction scratch, 10 bytes per reading.  A block of sm_100 gets at most 227 KB, so log_cap <= 5810.
constexpr size_t kMaxSmemPerBlock = 227 * 1024;
constexpr int kMaxLogCap =
    (int)((kMaxSmemPerBlock - 16) / (kWarpsPerBlock * (2 * sizeof(float) + sizeof(uint16_t))));
#define RS_LOG_CAP_MSG "log_cap out of range [n_agents, 5810]: 40 * log_cap + 16 bytes of shared memory per block " \
                       "exceed the 227 KB (232448 bytes) of sm_100"
static_assert(kMaxLogCap == 5810, "RS_LOG_CAP_MSG names the limit");

size_t maps_smem_bytes(int log_cap) {
    return (size_t)kWarpsPerBlock * log_cap * (2 * sizeof(float) + sizeof(uint16_t)) + 16;
}

__device__ __forceinline__ int cell_of(const RsMapsConfig &c, double vx, double vy) {
    // int(v * resolution_accuracy) M:704-713, then numpy indexing: negative indices wrap once
    int cx = (int)(vx * c.resolution_accuracy), cy = (int)(vy * c.resolution_accuracy);
    if (cx < 0) cx += c.dim_x;
    if (cy < 0) cy += c.dim_y;
    if (cx < 0 || cy < 0 || cx >= c.dim_x || cy >= c.dim_y) return -1;
    return cx * c.dim_y + cy;
}

// The per-environment state of the map observation between two calls.  maps_update_kernel keeps it in HBM (RsMapsState)
// and holds it here for the duration of a call; maps_replay_kernel keeps it here (and the sample table in shared memory)
// for a whole replayed episode.  rec / last_pred are per lane (lane b: agent b); the rest is the same on every lane.
struct MapsCallState {
    int len;                 // readings in the sample table
    double mean, m2;         // tools.standardizer
    int cnt;
    int rec, last_pred;      // tools.last_coords[b] / buffer b's last prediction cell (-1 = none)
};

// One observation_to_map call of environment n for all its A buffers (M:532-616), by one warp.  obs: the env's [A][11]
// row; loc_pred: its [A][2] row or NULL; s_cell / s_val: the sample table staged in shared memory (st.len entries), and
// log_cell / log_val its copy in HBM (NULL: none); scratch: log_cap floats of shared memory; actor: the env's [A][X][Y][6]
// stacks, critic its [X][Y][4] stack.  The call only STORES into the stacks.  Returns the RS_MS_* bits of this lane.
__device__ __forceinline__ uint32_t maps_call(const RsMapsConfig &c, const float *__restrict__ visit_lut, const float *obs,
                                              const float *loc_pred, uint16_t *log_cell, float *log_val, uint16_t *s_cell,
                                              float *s_val, float *scratch, float *actor_env, float *critic, int lane,
                                              MapsCallState &st) {
    const int A = c.n_agents, XY = c.dim_x * c.dim_y;
    uint32_t status = 0;
    int len = st.len, cnt = st.cnt, rec = st.rec;
    double mean = st.mean, m2 = st.m2;

    // ---- this call's observations: lane a holds agent a -----------------------------------------------------------
    int my_cell = -1, my_pred = -1;
    float my_count = 0.0f, my_obst = 0.0f;
    bool my_has_obst = false, pred_given = false;
    if (lane < A) {
        const float *o = obs + (size_t)lane * RS_OBS_DIM;
        my_count = o[0];
        // the env writes x * scale rounded to fp32; the reference's float64 observation is recovered from the lattice
        // coordinate (exact: the fp32 error is 1e-4 of a lattice step)
        const double x = rint((double)o[1] / c.scale), y = rint((double)o[2] / c.scale);
        my_cell = cell_of(c, x * c.scale, y * c.scale);
        if (my_cell < 0) status |= RS_MS_CELL_RANGE;
#pragma unroll
        for (int d = 3; d < RS_OBS_DIM; d++) {                             // M:929-932: the last non-zero detection wins
            const float v = o[d];
            if (v != 0.0f) { my_obst = v; my_has_obst = true; }
        }
        if (c.use_prediction && loc_pred) {
            const float px = loc_pred[(size_t)lane * 2], py = loc_pred[(size_t)lane * 2 + 1];
            if (px == px && py == py) {                                    // NaN = no prediction for this buffer
                pred_given = true;
                my_pred = cell_of(c, (double)px, (double)py);
                if (my_pred < 0) status |= RS_MS_PRED_RANGE;
            }
        }
    }

    // ---- M:541-545: every agent's reading joins the sample table before any estimate -----------------------------------
    if (len + A <= c.log_cap) {
        if (lane < A) {
            const uint16_t cell16 = (uint16_t)(my_cell < 0 ? 0xffff : my_cell);
            if (log_cell) {
                log_cell[len + lane] = cell16;
                log_val[len + lane] = my_count;
            }
            s_cell[len + lane] = cell16;
            s_val[len + lane] = my_count;
        }
        len += A;
    } else {
        status |= RS_MS_LOG_FULL;
    }
    __syncwarp();

    // stacks are stored cell-major, channel innermost ([X][Y][6] / [X][Y][4]): the values one call writes for a cell of
    // a buffer share a 32-byte sector or two instead of one sector per channel plane
    float *actor = actor_env + (size_t)(lane < A ? lane : 0) * 6 * XY;   // lane a' owns buffer a'
#define ACT(ch, cell) actor[(size_t)(cell) * 6 + (ch)]
#define CRI(ch, cell) critic[(size_t)(cell) * 4 + (ch)]

    // ---- source prediction map of buffer a' (PFGRU) M:564-568, 748-766: the old mark (a 1) goes, the new one is set ------
    if (pred_given) {
        if (st.last_pred >= 0 && st.last_pred != my_pred) ACT(0, st.last_pred) = 0.0f;
        if (my_pred >= 0) ACT(0, my_pred) = 1.0f;      // outside the map (the reference raises): old mark cleared, none set
        st.last_pred = my_pred;
    }

    // ---- agents in dict order M:547-604 ---------------------------------------------------------------------------------
    // The location maps hold small integer counts that are functions of the recorded cells (lane b: rec), so their new
    // values are computed from those instead of read-modify-written: the loop issues stores only.
    for (int a = 0; a < A; a++) {
        const int cc = __shfl_sync(0xffffffffu, my_cell, a);
        if (cc < 0) continue;
        const float obst = __shfl_sync(0xffffffffu, my_obst, a);
        const bool has_obst = __shfl_sync(0xffffffffu, (int)my_has_obst, a) != 0;
        const int last = __shfl_sync(0xffffffffu, rec, a);
        if (lane == a) rec = cc;

        // median of the samples of this cell (IntensityEstimator.get_estimate M:160-167): compact them, then select by rank
        int m = 0;
        for (int i0 = 0; i0 < len; i0 += 32) {
            const int i = i0 + lane;
            const bool hit = i < len && s_cell[i] == (uint16_t)cc;
            const unsigned b = __ballot_sync(0xffffffffu, hit);
            if (hit) scratch[m + __popc(b & ((1u << lane) - 1u))] = s_val[i];
            m += __popc(b);
        }
        __syncwarp();
        const int k1 = (m - 1) >> 1, k2 = m >> 1;
        float r1, r2;                                                       // readings are >= 0
        if (m == 0) {                                                       // (only when the sample table is full: RS_MS_LOG_FULL)
            r1 = r2 = -1.0f;
        } else if (m <= 2) {
            // a cell the agent has visited once or twice (most calls: agents keep moving): the median is the sample or the
            // mean of the two -- no rank selection (m is the same on every lane: it comes from ballots)
            const float s0 = scratch[0], s1 = scratch[m - 1];
            r1 = fminf(s0, s1);
            r2 = fmaxf(s0, s1);
        } else {
            uint32_t b1 = 0u, b2 = 0u;                                      // the selected values as bit patterns (>= 0: ordered)
            for (int i = lane; i < m; i += 32) {
                const float v = scratch[i];
                int rank = 0;
                for (int j = 0; j < m; j++) {
                    const float u = scratch[j];
                    rank += (u < v) || (u == v && j < i);
                }
                if (rank == k1) b1 = __float_as_uint(v);
                if (rank == k2) b2 = __float_as_uint(v);
            }
            r1 = __uint_as_float(__reduce_max_sync(0xffffffffu, b1));       // exactly one lane holds each rank
            r2 = __uint_as_float(__reduce_max_sync(0xffffffffu, b2));
        }
        __syncwarp();                                                       // scratch is reused by the next agent
        const double est = ((double)r1 + (double)r2) / 2.0;                 // statistics.median

        // StatisticStandardization.update + standardize M:215-265 (same numbers on every lane)
        cnt += 1;
        double sd = 1.0;
        if (cnt == 1) mean = est;
        else {
            const double mean_new = mean + div_count(est - mean, cnt);
            m2 = m2 + (est - mean) * (est - mean_new);
            mean = mean_new;
            sd = fmax(sqrt(div_count(m2, cnt - 1)), 1.0);
        }
        const float z = (float)((est - mean) / sd);

        // visit counts M:886-916: the shadow counter (2 per earlier visit of the cell) equals twice the number of the cell's
        // samples recorded before this agent's turn: all of them minus this call's readings of agents a..A-1 there
        const int later = __popc(__ballot_sync(0xffffffffu, lane < A && lane >= a && my_cell == cc));
        const float vis = visit_lut[max(m - later, 0)];

        // agents recorded at the old / new cell after this move
        const int n_cc = __popc(__ballot_sync(0xffffffffu, lane < A && rec == cc));
        const int n_last = __popc(__ballot_sync(0xffffffffu, lane < A && last >= 0 && rec == last));
        if (lane < A) {
            if (lane == a) {                                                // own location map M:812-830
                if (last >= 0 && last != cc) ACT(1, last) = 0.0f;
                ACT(1, cc) = 1.0f;
            } else {                                                        // others' locations M:832-848: agents != a'
                if (last >= 0) ACT(2, last) = (float)(n_last - (rec == last));
                ACT(2, cc) = (float)(n_cc - (rec == cc));
            }
            ACT(3, cc) = z;                                                 // readings map M:884
            ACT(4, cc) = vis;                                               // visit counts map M:906
            if (has_obst) ACT(5, cc) = obst;                                // obstacles map M:929-932
        }
        if (lane == 0) {                                                    // the critic's stack (same in every buffer)
            if (last >= 0) CRI(0, last) = (float)n_last;                    // combined locations M:786-810
            CRI(0, cc) = (float)n_cc;
            CRI(1, cc) = z;
            CRI(2, cc) = vis;
            if (has_obst) CRI(3, cc) = obst;
        }
    }
#undef ACT
#undef CRI
    st.len = len;
    st.cnt = cnt;
    st.rec = rec;
    st.mean = mean;
    st.m2 = m2;
    return status;
}

__global__ void __launch_bounds__(kBlock) maps_update_kernel(const __grid_constant__ RsMapsConfig c,
                                                             const __grid_constant__ RsMapsState S, const float *obs,
                                                             const float *loc_pred, const uint8_t *mask, int mask_bits,
                                                             int n_env) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int n = blockIdx.x * kWarpsPerBlock + w;
    if (n >= n_env || (mask && !(mask[n] & mask_bits))) return;            // whole warps leave together
    // per warp: the episode's sample table (values, cells) and the compaction scratch
    float *s_val = reinterpret_cast<float *>(smem_raw) + (size_t)w * 2 * c.log_cap;
    float *scratch = s_val + c.log_cap;
    uint16_t *s_cell = reinterpret_cast<uint16_t *>(reinterpret_cast<float *>(smem_raw) + (size_t)kWarpsPerBlock * 2 * c.log_cap) +
                       (size_t)w * c.log_cap;
    const int A = c.n_agents, XY = c.dim_x * c.dim_y;

    // ---- everything the call reads from HBM is requested up front (one round of latency) ------------------------------
    uint16_t *log_cell = S.log_cell + (size_t)n * c.log_cap;
    float *log_val = S.log_val + (size_t)n * c.log_cap;
    MapsCallState st;
    st.len = S.log_len[n];
    st.mean = S.std[2 * (size_t)n];
    st.m2 = S.std[2 * (size_t)n + 1];
    st.cnt = S.std_count[n];
    st.rec = -1;
    st.last_pred = -1;
    if (lane < A) {
        st.rec = S.last_cell[(size_t)n * A + lane];
        st.last_pred = S.last_pred[(size_t)n * A + lane];
    }
    const int last_pred0 = st.last_pred;
#pragma unroll 4
    for (int i = lane; i < st.len; i += 32) {
        s_cell[i] = log_cell[i];
        s_val[i] = log_val[i];
    }

    uint32_t status = maps_call(c, S.visit_lut, obs + (size_t)n * A * RS_OBS_DIM,
                                loc_pred ? loc_pred + (size_t)n * A * 2 : nullptr, log_cell, log_val, s_cell, s_val, scratch,
                                S.actor + (size_t)n * A * 6 * XY, S.critic + (size_t)n * 4 * XY, lane, st);
    if (lane < A) {
        S.last_cell[(size_t)n * A + lane] = st.rec;
        if (st.last_pred != last_pred0) S.last_pred[(size_t)n * A + lane] = st.last_pred;
    }
    if (lane == 0) {
        S.log_len[n] = st.len;
        S.std[2 * (size_t)n] = st.mean;
        S.std[2 * (size_t)n + 1] = st.m2;
        S.std_count[n] = st.cnt;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) status |= __shfl_xor_sync(0xffffffffu, status, o);
    if (lane == 0 && status) S.status[n] |= status;
}

// Dense copy / zeroing of one output row of the replay (16-byte accesses when the row allows them).  A copy issues 8
// loads per lane before their stores: one warp moves a whole row, so the loads in flight are what sets its rate.
__device__ __forceinline__ void row_fill(float *dst, const float *src, size_t cnt, int lane) {
    if ((cnt & 3) == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0 && (!src || (reinterpret_cast<uintptr_t>(src) & 15) == 0)) {
        float4 *d4 = reinterpret_cast<float4 *>(dst);
        const float4 *s4 = reinterpret_cast<const float4 *>(src);
        const size_t n4 = cnt / 4;
        if (!src) {
            const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
            for (size_t i = lane; i < n4; i += 32) d4[i] = z4;
            return;
        }
        size_t i = lane;
        for (; i + 7 * 32 < n4; i += 8 * 32) {
            float4 v[8];
#pragma unroll
            for (int k = 0; k < 8; k++) v[k] = s4[i + k * 32];
#pragma unroll
            for (int k = 0; k < 8; k++) d4[i + k * 32] = v[k];
        }
        for (; i < n4; i += 32) d4[i] = s4[i];
    } else {
        for (size_t i = lane; i < cnt; i += 32) dst[i] = src ? src[i] : 0.0f;
    }
}

// The map stacks the policy read at steps t0..t1 of env n, rebuilt from the rollout buffer: one warp per requested range.
// The first row is built by replaying the calls of rows s..t0 (s: the first row of t0's episode) into the zeroed output row;
// every following row is the previous output row (dense copy) plus the sparse stores of its own call, or a zeroed row and
// a restarted state where an episode starts inside the range.  The sample table lives in shared memory, the rest of the
// state in registers: nothing of the live RsMapsState but the visit-count table is read.
__global__ void __launch_bounds__(kBlock) maps_replay_kernel(const __grid_constant__ RsMapsConfig c, const float *visit_lut,
                                                             const float *obs_rows, const float *pred_rows,
                                                             const uint8_t *end_rows, int T, int n_env, const int32_t *ranges,
                                                             int m, const int64_t *out_row0, float *out_actor,
                                                             float *out_critic, uint32_t *out_status) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int r = blockIdx.x * kWarpsPerBlock + w;
    if (r >= m) return;
    float *s_val = reinterpret_cast<float *>(smem_raw) + (size_t)w * 2 * c.log_cap;
    float *scratch = s_val + c.log_cap;
    uint16_t *s_cell = reinterpret_cast<uint16_t *>(reinterpret_cast<float *>(smem_raw) + (size_t)kWarpsPerBlock * 2 * c.log_cap) +
                       (size_t)w * c.log_cap;
    const int A = c.n_agents, XY = c.dim_x * c.dim_y, NA = n_env * A;
    const size_t actor_row = (size_t)A * 6 * XY, critic_row = (size_t)4 * XY;
    const int n = ranges[3 * (size_t)r], t0 = ranges[3 * (size_t)r + 1], t1 = ranges[3 * (size_t)r + 2];
    const int64_t row0 = out_row0[r];
    if (t1 < t0) {                                                          // inverted: owns no rows
        if (lane == 0) out_status[r] = RS_MR_BAD_RANGE;
        return;
    }
    if (n < 0 || n >= n_env || t0 < 0 || t1 >= T) {                         // outside the buffer: zero rows
        for (int64_t k = 0; k <= (int64_t)t1 - t0; k++) {
            row_fill(out_actor + (size_t)(row0 + k) * actor_row, nullptr, actor_row, lane);
            row_fill(out_critic + (size_t)(row0 + k) * critic_row, nullptr, critic_row, lane);
        }
        if (lane == 0) out_status[r] = RS_MR_BAD_RANGE;
        return;
    }
    // s: 1 + the last path end before t0 in column n*A (all agents of an env end together), or 0
    int s = 0;
    for (int hi = t0 - 1; hi >= 0; hi -= 32) {
        const int t = hi - lane;
        const bool e = t >= 0 && end_rows[(size_t)t * NA + (size_t)n * A] != 0;
        const unsigned b = __ballot_sync(0xffffffffu, e);
        if (b) { s = hi - (__ffs(b) - 1) + 1; break; }                      // lowest lane = latest row
    }
    uint32_t status = 0;
    MapsCallState st;
    float *act = out_actor + (size_t)row0 * actor_row, *cri = out_critic + (size_t)row0 * critic_row;
    for (int t = s; t <= t1; t++) {
        if (t == s || (t > t0 && end_rows[(size_t)(t - 1) * NA + (size_t)n * A] != 0)) {   // an episode starts: reset
            if (t > t0) {
                act += actor_row;
                cri += critic_row;
            }
            row_fill(act, nullptr, actor_row, lane);
            row_fill(cri, nullptr, critic_row, lane);
            st.len = 0; st.mean = 0.0; st.m2 = 0.0; st.cnt = 0; st.rec = -1; st.last_pred = -1;
        } else if (t > t0) {                                                // the next row starts as a copy of this one
            row_fill(act + actor_row, act, actor_row, lane);
            row_fill(cri + critic_row, cri, critic_row, lane);
            act += actor_row;
            cri += critic_row;
        }
        __syncwarp();
        status |= maps_call(c, visit_lut, obs_rows + ((size_t)t * NA + (size_t)n * A) * RS_OBS_DIM,
                            pred_rows ? pred_rows + ((size_t)t * NA + (size_t)n * A) * 2 : nullptr, nullptr, nullptr, s_cell,
                            s_val, scratch, act, cri, lane, st);
        __syncwarp();
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) status |= __shfl_xor_sync(0xffffffffu, status, o);
    if (lane == 0) out_status[r] = status;
}

// MapsBuffer.reset M:513-523 (+ ConversionTools.reset M:378-385) for the selected environments: one warp zeroes the
// environment's stacks with 16-byte stores
__global__ void __launch_bounds__(kBlock) maps_reset_kernel(const __grid_constant__ RsMapsConfig c,
                                                            const __grid_constant__ RsMapsState S, const uint8_t *mask,
                                                            int mask_bits, int n_env) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int n = blockIdx.x * kWarpsPerBlock + w;
    if (n >= n_env || (mask && !(mask[n] & mask_bits))) return;
    const int A = c.n_agents, XY = c.dim_x * c.dim_y;
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    {
        float *p = S.actor + (size_t)n * A * 6 * XY;
        const size_t cnt = (size_t)A * 6 * XY;
        if ((cnt & 3) == 0 && (reinterpret_cast<uintptr_t>(p) & 15) == 0)
            for (size_t i = lane; i < cnt / 4; i += 32) reinterpret_cast<float4 *>(p)[i] = z4;
        else
            for (size_t i = lane; i < cnt; i += 32) p[i] = 0.0f;
    }
    {
        float *p = S.critic + (size_t)n * 4 * XY;
        const size_t cnt = (size_t)4 * XY;
        if ((reinterpret_cast<uintptr_t>(p) & 15) == 0)
            for (size_t i = lane; i < cnt / 4; i += 32) reinterpret_cast<float4 *>(p)[i] = z4;
        else
            for (size_t i = lane; i < cnt; i += 32) p[i] = 0.0f;
    }
    if (lane < A) {
        S.last_cell[(size_t)n * A + lane] = -1;
        S.last_pred[(size_t)n * A + lane] = -1;
    }
    if (lane == 0) {
        S.log_len[n] = 0;
        S.std[2 * (size_t)n] = 0.0;
        S.std[2 * (size_t)n + 1] = 0.0;
        S.std_count[n] = 0;
    }
}

int check_maps(const RsMapsConfig *c, const RsMapsState *s, int32_t n_env) {
    if (!c || !s) return rs_set_error("maps cfg/state is NULL");
    if (n_env <= 0) return rs_set_error("n_env must be positive");
    if (c->n_agents < 1 || c->n_agents > RS_MAX_A) return rs_set_error("n_agents out of range [1, 8]");
    if (c->dim_x < 1 || c->dim_y < 1 || (int64_t)c->dim_x * c->dim_y > 65535) return rs_set_error("map dimensions out of range");
    if (c->log_cap < c->n_agents || c->log_cap > kMaxLogCap) return rs_set_error(RS_LOG_CAP_MSG);
    if (c->base < 2) return rs_set_error("base must be >= 2");
    if (!(c->resolution_accuracy > 0) || !(c->scale > 0)) return rs_set_error("resolution_accuracy / scale must be positive");
    if (!s->actor || !s->critic || !s->log_cell || !s->log_val || !s->log_len || !s->last_cell ||
        !s->last_pred || !s->std || !s->std_count || !s->visit_lut || !s->status)
        return rs_set_error("RsMapsState has NULL members");
    return 0;
}

}  // namespace

extern "C" {

int rs_maps_update(const RsMapsConfig *cfg, const RsMapsState *st, const float *obs, const float *loc_pred,
                   const uint8_t *mask, int32_t mask_bits, int32_t n_env, void *stream) {
    if (int rc = check_maps(cfg, st, n_env)) return rc;
    if (!obs) return rs_set_error("obs is NULL");
    const int grid = (n_env + kWarpsPerBlock - 1) / kWarpsPerBlock;
    const size_t smem = maps_smem_bytes(cfg->log_cap);
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(maps_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
    }
    maps_update_kernel<<<grid, kBlock, smem, static_cast<cudaStream_t>(stream)>>>(*cfg, *st, obs, loc_pred, mask,
                                                                                  mask_bits ? mask_bits : 0xff, n_env);
    return (int)cudaGetLastError();
}

int rs_maps_reset(const RsMapsConfig *cfg, const RsMapsState *st, const uint8_t *mask, int32_t mask_bits, int32_t n_env,
                  void *stream) {
    if (int rc = check_maps(cfg, st, n_env)) return rc;
    const int grid = (n_env + kWarpsPerBlock - 1) / kWarpsPerBlock;
    maps_reset_kernel<<<grid, kBlock, 0, static_cast<cudaStream_t>(stream)>>>(*cfg, *st, mask, mask_bits ? mask_bits : 0xff,
                                                                              n_env);
    return (int)cudaGetLastError();
}

int rs_maps_replay(const RsMapsConfig *cfg, const RsMapsState *st, const float *obs_rows, const float *pred_rows,
                   const uint8_t *end_rows, int32_t T, int32_t n_env, const int32_t *ranges, int32_t m,
                   const int64_t *out_row0, float *out_actor, float *out_critic, uint32_t *out_status, void *stream) {
    if (!cfg || !st) return rs_set_error("rs_maps_replay: maps cfg/state is NULL");
    if (n_env <= 0 || T <= 0) return rs_set_error("rs_maps_replay: T and n_env must be positive");
    if (m < 0) return rs_set_error("rs_maps_replay: m must be >= 0");
    if (cfg->n_agents < 1 || cfg->n_agents > RS_MAX_A) return rs_set_error("rs_maps_replay: n_agents out of range [1, 8]");
    if (cfg->dim_x < 1 || cfg->dim_y < 1 || (int64_t)cfg->dim_x * cfg->dim_y > 65535)
        return rs_set_error("rs_maps_replay: map dimensions out of range");
    if (cfg->log_cap < cfg->n_agents || cfg->log_cap > kMaxLogCap) return rs_set_error("rs_maps_replay: " RS_LOG_CAP_MSG);
    if (!(cfg->resolution_accuracy > 0) || !(cfg->scale > 0))
        return rs_set_error("rs_maps_replay: resolution_accuracy / scale must be positive");
    if (!st->visit_lut) return rs_set_error("rs_maps_replay: RsMapsState.visit_lut is NULL");
    if (!obs_rows || !end_rows) return rs_set_error("rs_maps_replay: obs_rows / end_rows is NULL");
    if (m == 0) return 0;
    if (!ranges || !out_row0 || !out_actor || !out_critic || !out_status)
        return rs_set_error("rs_maps_replay: ranges / out_row0 / out_actor / out_critic / out_status is NULL");
    const int grid = (m + kWarpsPerBlock - 1) / kWarpsPerBlock;
    const size_t smem = maps_smem_bytes(cfg->log_cap);
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(maps_replay_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
    }
    maps_replay_kernel<<<grid, kBlock, smem, static_cast<cudaStream_t>(stream)>>>(
        *cfg, st->visit_lut, obs_rows, pred_rows, end_rows, T, n_env, ranges, m, out_row0, out_actor, out_critic, out_status);
    return (int)cudaGetLastError();
}

int rs_sizeof_maps_config(void) { return (int)sizeof(RsMapsConfig); }
int rs_sizeof_maps_state(void) { return (int)sizeof(RsMapsState); }

}  // extern "C"
