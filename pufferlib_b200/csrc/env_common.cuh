// env_common.cuh -- the device-resident multi-env handle shared by all env kinds.
//
// One pb_env holds N env instances of one kind on one GPU: per-env state as SoA arrays in HBM (a few bytes per
// env; reloaded each step because the policy forward sits between steps), the `done` flags the vectoriser
// consults (vector.py:147), EpisodeStats accumulators (postprocess.py:22-54) and the device-side statistics.
#pragma once
#include "pb_common.cuh"

constexpr int PB_STAT_SLOTS = 256;

struct pb_env_vtable {
    int (*reset)(pb_env*, uint64_t seed, const pb_env_out*, cudaStream_t);
    int (*step)(pb_env*, const int64_t* actions, const pb_env_out*, cudaStream_t);
    void (*destroy)(pb_env*);
};

struct pb_env {
    pb_env_config cfg;
    pb_env_info info;
    const pb_env_vtable* vt;
    bool was_reset;
    // common device arrays [N]
    uint8_t* d_done;         // env.done: previous row was terminal -> reset on next send
    double* d_ep_return;     // running episode return (fp64 like the python-float sum of the reference)
    int32_t* d_ep_length;
    double* d_row_return;    // values of the episode that ended on the most recent step (valid where terminal)
    int32_t* d_row_length;
    float* d_row_score;
    double* d_stats;         // [PB_STAT_SLOTS][4] episodes, sum return, sum length, sum score (slot = warp hash:
                             // same-address atomics serialise in L2, spreading them keeps the step kernel flat)
    double* h_stats_pinned;  // [PB_STAT_SLOTS][4] pinned staging for pb_env_stats_read
    // where the previous call wrote the observations (snake / pong carry state in the obs rows)
    const void* cur_obs;
    int64_t cur_obs_stride;
    // truncations (always 0) and masks (always 1) are constants: a step rewrites them only into buffers it has not
    // filled before (saves two scattered [N] stores per env per step)
    const void* const_trunc;
    const void* const_masks;
    bool write_const;
    int32_t n_heads;         // MultiDiscrete kinds: action heads (0 = Discrete(info.num_actions)); actions are [N][n_heads]
    int32_t nvec[8];
    void* kind;              // kind-specific state
};

int pb_env_alloc_common(pb_env* env);
void pb_env_free_common(pb_env* env);

int pb_squared_create(pb_env* env);
int pb_breakout_create(pb_env* env);
int pb_snake_create(pb_env* env);
int pb_pong_create(pb_env* env);
int pb_spaces_create(pb_env* env);

struct EpisodeAcc {
    double* ep_return;
    int32_t* ep_length;
    double* row_return;
    int32_t* row_length;
    float* row_score;
    double* stats;
};

#ifdef __CUDACC__
// EpisodeStats bookkeeping for one env on one step (called by every env-step kernel, one lane per env).
// `finished`: this step ended the episode; `reset_row`: this step was an auto-reset (no reward accounted,
// postprocess.py:18-20 clears the accumulators).

__device__ __forceinline__ void episode_update(const EpisodeAcc& acc, int64_t e, bool active, bool reset_row,
                                               double reward, bool finished, float score) {
    double ret = 0.0;
    int len = 0;
    if (active) {
        if (reset_row) {
            acc.ep_return[e] = 0.0;
            acc.ep_length[e] = 0;
        } else {
            ret = acc.ep_return[e] + reward;
            len = acc.ep_length[e] + 1;
            acc.ep_return[e] = ret;
            acc.ep_length[e] = len;
            if (finished) {
                acc.row_return[e] = ret;
                acc.row_length[e] = len;
                acc.row_score[e] = score;
            }
        }
    }
    // warp-aggregated statistics: one atomic per warp and quantity
    const bool fin = active && !reset_row && finished;
    const unsigned m = __ballot_sync(0xffffffffu, fin);
    if (m) {
        double r = fin ? ret : 0.0, l = fin ? (double)len : 0.0, s = fin ? (double)score : 0.0;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            r += __shfl_xor_sync(0xffffffffu, r, off);
            l += __shfl_xor_sync(0xffffffffu, l, off);
            s += __shfl_xor_sync(0xffffffffu, s, off);
        }
        if ((threadIdx.x & 31) == 0) {
            const unsigned gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
            double* slot = acc.stats + 4 * ((gw * 2654435761u) >> 24);   // 256 slots, multiplicative hash of the warp id
            atomicAdd(slot + 0, (double)__popc(m));
            atomicAdd(slot + 1, r);
            atomicAdd(slot + 2, l);
            atomicAdd(slot + 3, s);
        }
    }
}

#endif

static inline EpisodeAcc pb_episode_acc(const pb_env* env) {
    return EpisodeAcc{env->d_ep_return, env->d_ep_length, env->d_row_return, env->d_row_length, env->d_row_score,
                      env->d_stats};
}
