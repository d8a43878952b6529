/* pufferlib_b200.h -- C ABI of libpuffer_b200.so: the B200 (sm_100a) env-step + PPO-rollout hot path.
 *
 * This is the drop-in boundary for PufferLib's vectorised env step / rollout / GAE / minibatch path.
 * Every entry point below names the reference interface it replaces (paths under /root/reference).
 * The reference has no C ABI of its own on this path: its native seams are the `PufferEnv` buffer-injection
 * protocol (pufferlib/environment.py:1-21 + vector.py:97-110) and two Cython functions
 * (c_gae.pyx:11 `compute_gae`, pufferlib/extensions.pyx:19,32 `emulate`/`nativize`); the rest is Python
 * (vector.py Serial/Multiprocessing send/recv, clean_pufferl.py Experience.store/sort_training_data/flatten_batch).
 *
 * Conventions
 *   - Plain C: pointers, sizes, POD structs.  No torch / C++ types cross this boundary.
 *   - Unless a parameter is suffixed `_host`, every data pointer is a DEVICE pointer owned by the caller
 *     (e.g. `tensor.data_ptr()`); the library owns only the opaque `pb_env` handle and its internal state.
 *   - `stream` is a `cudaStream_t` passed as `void*` (NULL = legacy default stream).  All work is enqueued
 *     asynchronously on it; nothing here synchronises the device unless documented.
 *   - Every function returns 0 on success or a negative `PB_ERR_*`; `pb_last_error()` gives the message of the
 *     calling thread's last failure.  No exceptions, no CPU fallback: without a CUDA device calls fail with
 *     PB_ERR_CUDA.
 *   - One host thread per GPU drives a handle; the library creates no threads and is re-entrant per handle.
 *
 * Rollout layout ("arrival order", identical to the reference's Experience tensors when every mask is True and
 * agent_ids == arange(N), clean_pufferl.py:390-397,436-450): row index = t*N + e for step t, env e.
 * "Sorted order" (what Experience.sort_training_data produces, clean_pufferl.py:452-464) is f = e*H + t; on the
 * device that permutation is arithmetic, no index tensor exists.
 */
#ifndef PUFFERLIB_B200_H
#define PUFFERLIB_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PB_ABI_VERSION 1

enum {
    PB_OK = 0,
    PB_ERR_INVALID = -1,   /* bad argument (maps to APIUsageError / ValueError on the Python side) */
    PB_ERR_CUDA = -2,      /* CUDA runtime failure or no device (RuntimeError) */
    PB_ERR_STATE = -3,     /* call order violated, e.g. step before reset (APIUsageError, emulation.py:198-201) */
    PB_ERR_UNSUPPORTED = -4
};

enum { PB_ENV_SQUARED = 0, PB_ENV_BREAKOUT = 1, PB_ENV_SNAKE = 2, PB_ENV_PONG = 3, PB_ENV_SPACES = 4 };
enum { PB_DTYPE_F32 = 0, PB_DTYPE_U8 = 1 };

typedef struct pb_env pb_env; /* opaque: N env instances resident on one GPU */

typedef struct {
    int32_t kind;             /* PB_ENV_* */
    int32_t num_envs;         /* N: env instances (== agents) on this GPU */
    int32_t device;           /* CUDA device ordinal */
    int32_t reserved;
    int64_t env_index_offset; /* global index of local env 0 (multi-GPU shards seed by GLOBAL index) */
    int32_t iparam[8];        /* kind-specific, 0 = default:
                                 SQUARED : [0]=distance_to_target (default 3; ocean/environment.py:28)
                                 BREAKOUT: [0]=max_ticks (default 4096)
                                 SNAKE   : [0]=max_ticks (default 1024)
                                 PONG    : [0]=max_score (default 5) [1]=max_ticks (default 4096)
                                 SPACES  : none */
} pb_env_config;

typedef struct {
    int32_t obs_dtype;    /* PB_DTYPE_* */
    int32_t obs_ndim;
    int32_t obs_shape[4];
    int64_t obs_bytes;    /* bytes of one agent's observation (O) */
    int32_t num_actions;  /* Discrete(n); 0 for MultiDiscrete kinds (pb_env_action_nvec) */
    int32_t num_envs;
    float obs_low, obs_high; /* Box bounds */
} pb_env_info;

/* Where one reset/step call writes its results.  With a time-major rollout tensor the caller passes
 * obs = rollout_obs + t*N*O, obs_stride = O, rewards = rollout_rewards + t*N, dones_f32 = rollout_dones + t*N:
 * the env kernel then stores straight into rollout row t (replaces buf.observations[row][:] = ob,
 * emulation.py:158-164, plus the obs/reward/done part of Experience.store, clean_pufferl.py:442-447). */
typedef struct {
    void* obs;            /* env e writes obs_bytes at (char*)obs + e*obs_stride */
    int64_t obs_stride;   /* bytes between consecutive envs' rows (>= obs_bytes) */
    float* rewards;       /* [N] fp32                          (buf.rewards,     emulation.py:219-221) */
    uint8_t* terminals;   /* [N] bool as one byte               (buf.terminals)   */
    uint8_t* truncations; /* [N] bool, always 0 for these envs  (buf.truncations); constants: written by reset, and by */
    uint8_t* masks;       /* [N] bool, always 1 (buf.masks)       a step only into buffers other than the previous call's */
    float* dones_f32;     /* optional [N]: terminal as 0.f/1.f  (Experience.dones, clean_pufferl.py:395,447); may be NULL */
} pb_env_out;

const char* pb_last_error(void);
int pb_abi_version(void);
int pb_device_count(int* out_count);
/* number of CUDA kernels this library has launched in this process (host-side counter; used by bench.py's
 * `gpu_launches`).  Kernels replayed by a CUDA graph are not counted again. */
uint64_t pb_launch_count(void);

/* -- environments ---------------------------------------------------------------------------------------------
 * Replaces: the backend constructor instantiating N envs (vector.py:79), Serial.async_reset (vector.py:112-135),
 * Serial.send's per-env `if env.done: reset() else: step()` loop (vector.py:137-156), the GymnasiumPufferEnv
 * buffer writes (emulation.py:169-228) and EpisodeStats (postprocess.py:8-54), for the device-native env kinds. */
int pb_env_create(const pb_env_config* cfg, pb_env** out);
int pb_env_destroy(pb_env* env);
int pb_env_get_info(const pb_env* env, pb_env_info* out);
/* MultiDiscrete action space of the kind (emulation.py:115-120 turns a Dict / Tuple of Discrete into MultiDiscrete):
 * nvec_out[0..n_heads) = head sizes, the rest of the 8 entries 0.  Discrete kinds report n_heads = 0. */
int pb_env_action_nvec(const pb_env* env, int32_t* nvec_out /*[8]*/, int32_t* n_heads_out);

/* vector.py:112-135: (re)seed env i with seed + env_index_offset + i (make_seeds, vector.py:639-641), reset it and
 * write the reset rows (r=0, terminal=False, truncation=False, mask=True; emulation.py:187-192). */
int pb_env_reset(pb_env* env, uint64_t seed, const pb_env_out* out, void* stream);

/* vector.py:137-156: envs whose previous row was terminal reset (action ignored, reset row written), all others
 * step with actions[e] (int64, Discrete) or actions[e][0..n_heads) (int64 [N][n_heads], MultiDiscrete kinds).
 * PB_ERR_STATE before the first reset.  `actions` is validated on the device only by clamping (each column) into
 * [0, num_actions) / [0, nvec[h]) -- the host layer does the reference's first-send action_space.contains check
 * (vector.py:36-39). */
int pb_env_step(pb_env* env, const int64_t* actions, const pb_env_out* out, void* stream);

/* Snake step kernel variant for A/B measurements: lanes per env, 4 (default) or 16 (round 1); bit-identical results. */
int pb_snake_set_variant(int32_t lanes_per_env);

/* Episode statistics (EpisodeStats, postprocess.py:22-54).
 * pb_env_episode_rows: per-env values of the episode that ENDED on the most recent step -- valid where that
 * step's terminals[e] != 0: episode_return (fp64 sum), episode_length, score.  Pointers are device arrays [N]
 * owned by the handle (read-only for the caller, overwritten by the next step).
 * pb_env_stats_read: {episodes finished, sum episode_return, sum episode_length, sum score} accumulated on the
 * device since the last read with clear != 0; copies 4 doubles to host memory and synchronises `stream`. */
int pb_env_episode_rows(pb_env* env, const double** episode_return, const int32_t** episode_length,
                        const float** score);
int pb_env_stats_read(pb_env* env, double* out4_host, int clear, void* stream);

/* -- rollout ---------------------------------------------------------------------------------------------------
 * Replaces the policy-output part of Experience.store (clean_pufferl.py:443-446): one fused copy of value /
 * logprob / action [N] into row t of the time-major rollout tensors (pass row pointers base + t*N). */
int pb_rollout_store(const float* value, const float* logprob, const int64_t* action, float* values_row,
                     float* logprobs_row, int64_t* actions_row, int64_t n, void* stream);

/* Copy N obs rows between strided row sets (carry-over of the boundary observation into row 0 of the next
 * rollout; the masked gather `obs[ptr:end] = obs[indices]` of clean_pufferl.py:442 with an all-True mask). */
int pb_copy_rows(const void* src, int64_t src_stride, void* dst, int64_t dst_stride, int64_t row_bytes,
                 int64_t n_rows, void* stream);

/* -- GAE -------------------------------------------------------------------------------------------------------
 * Replaces sort_training_data + the three numpy gathers + c_gae.compute_gae (clean_pufferl.py:163-169,
 * c_gae.pyx:11-32): ONE backward chain over the whole sorted batch f = e*H + t, crossing env boundaries exactly
 * as the reference does, A[B-1] = 0.  Inputs are the arrival-order (time-major [H][N]) rollout tensors; the
 * kernel reads them transposed.  Outputs are in sorted order: advantages[f] (== advantages_np) and, if non-NULL,
 * returns_sorted[f] = advantages[f] + values[t*N+e].  num_envs = 1 gives the reference's flat signature.
 * fp32; element arithmetic keeps c_gae.pyx's association, only the scan tree reorders it (<= 1e-5 relative).
 * `workspace`: pb_gae_workspace_bytes(...) bytes, zero-filled once by the caller; left zeroed by every call. */
size_t pb_gae_workspace_bytes(int64_t num_envs, int64_t horizon);
int pb_gae(const float* rewards, const float* values, const float* dones, float* advantages,
           float* returns_sorted, int64_t num_envs, int64_t horizon, float gamma, float gae_lambda,
           void* workspace, size_t workspace_bytes, void* stream);
/* pb_gae with an additional advantages output in ARRIVAL (time-major, row t*N + e) order -- the order the rollout
 * tensors and the zero-copy minibatch slabs are in, so the update can consume it without a re-ordering pass.  Either
 * advantages output may be null.  Time-major output: horizon in {128, 256, 512} and num_envs % 4 == 0
 * (pb_gae_time_major_supported). */
int pb_gae_time_major_supported(int64_t num_envs, int64_t horizon);
/* Tile-kernel variant for A/B measurements: 0 (default) chosen by horizon, 2 double-buffered tiles + coalesced outputs,
 * 3 single-buffered tiles, 1 the kernel of round 1.  Results are bit-identical. */
int pb_gae_set_variant(int32_t variant);
int pb_gae_tm(const float* rewards, const float* values, const float* dones, float* advantages, float* returns_sorted,
              float* advantages_time_major, int64_t num_envs, int64_t horizon, float gamma, float gae_lambda,
              void* workspace, size_t workspace_bytes, void* stream);

/* -- minibatch construction --------------------------------------------------------------------------------------
 * Replaces Experience.flatten_batch (clean_pufferl.py:466-482) for the scalar tensors.  Segment k (bptt
 * consecutive sorted rows) goes to minibatch k % n_mb, row k / n_mb (clean_pufferl.py:455-460,473-475).
 * Outputs are dense [n_mb][rows][bptt].  returns_np (optional) reproduces clean_pufferl.py:476 literally:
 * returns_np[i] = advantages_sorted[i] + values_arrival[i].  Any output pointer may be NULL. */
int pb_flatten_batch(const int64_t* actions, const float* logprobs, const float* dones, const float* values,
                     const float* advantages_sorted, int64_t* b_actions, float* b_logprobs, float* b_dones,
                     float* b_values, float* b_advantages, float* b_returns, float* returns_np,
                     int64_t num_envs, int64_t horizon, int64_t n_mb, int64_t rows, int64_t bptt, void* stream);

/* Replaces `b_obs = obs[b_idxs_obs]` (clean_pufferl.py:477) for minibatches [mb_begin, mb_begin+mb_count):
 * dst is dense [mb_count][rows][bptt][row_bytes]; src is the arrival-order obs tensor [H][N][row_bytes].
 * Rows >= 4 KiB and 16-byte aligned go through TMA bulk copies (global->shared->global). */
int pb_minibatch_gather(const void* obs, void* dst, int64_t row_bytes, int64_t num_envs, int64_t horizon,
                        int64_t n_mb, int64_t rows, int64_t bptt, int64_t mb_begin, int64_t mb_count,
                        void* stream);

/* Replaces the per-minibatch advantage normalisation of train (clean_pufferl.py:211-213), for n_mb minibatches
 * at once: out[m] = (adv[m] - mean_m) / (std_m + 1e-8), std unbiased (N-1).  in/out are [n_mb][mb_size] and may
 * alias.  `workspace`: pb_adv_norm_workspace_bytes(...) bytes (no initialisation required). */
size_t pb_adv_norm_workspace_bytes(int64_t n_mb, int64_t mb_size);
int pb_adv_norm(const float* adv, float* out, int64_t n_mb, int64_t mb_size, void* workspace,
                size_t workspace_bytes, void* stream);

/* -- image observation pack --------------------------------------------------------------------------------------
 * Replaces the frame-stack materialisation inside `self.obs[:] = ob` for (S, 84, 84) uint8 observations
 * (emulation.py:161-162 on a LazyFrames of S frames; atari/environment.py:37-39): for each env,
 * obs_out[e][0..S-2] = prev_obs[e][1..S-1], obs_out[e][S-1] = new_frames[e]; where reset_mask[e] != 0 all S slots
 * are filled with new_frames[e] (gymnasium FrameStack.reset).  frame_bytes % 16 == 0; staged through shared
 * memory with TMA bulk copies (cp.async.bulk).  Strides are bytes between consecutive envs. */
int pb_image_pack(const void* new_frames, int64_t frame_stride, const void* prev_obs, int64_t prev_stride,
                  void* obs_out, int64_t out_stride, const uint8_t* reset_mask, int64_t num_envs,
                  int64_t frame_bytes, int32_t stack, void* stream);

/* -- fused sampling epilogue (SURVEY §8f-1) ----------------------------------------------------------------------
 * Replaces sample_logits (pufferlib/frameworks/cleanrl.py:25-47) for one Discrete head when sampling:
 * normalised = logits - logsumexp; action ~ Categorical(softmax) drawn with a counter-based RNG
 * (seed, offset + *offset_dev, row) -- offset_dev (optional device counter) keeps replays of a captured CUDA
 * graph on fresh random numbers; logprob = normalised[action]; entropy = -sum p*log p.  Optionally also writes
 * action/logprob/value into rollout row pointers (the pb_rollout_store copy, fused).  logits: fp32 rows of n_act
 * values, `logits_stride` floats apart (>= n_act; lets both heads come out of one GEMM); value: one float per row,
 * `value_stride` floats apart. */
int pb_sample_logits(const float* logits, int64_t logits_stride, int64_t n, int32_t n_act, uint64_t seed,
                     uint64_t offset, const uint64_t* offset_dev, int64_t* actions, float* logprobs, float* entropies,
                     const float* value, int64_t value_stride, float* values_row, float* logprobs_row,
                     int64_t* actions_row, void* stream);

/* -- PPO minibatch loss, forward + backward --------------------------------------------------------------------------
 * Replaces the loss block of train (clean_pufferl.py:202-238) and the action-given branch of sample_logits
 * (frameworks/cleanrl.py:25-47) for one Discrete head, for a minibatch of m rows: one pass computes
 *   stats8[0..5] = SUMS over rows of {max(pg1,pg2), max(v_unclipped, v_clipped) (no 0.5 yet), entropy, -logratio,
 *                  (ratio-1)-logratio, |ratio-1| > clip_coef}                      (fp64; caller divides by m)
 * and the analytic gradients of  loss = mean(pg) - ent_coef*mean(entropy) + vf_coef*0.5*mean(v)  with respect to the
 * logits [m][n_act] and the value [m] (already scaled by 1/m), following ATen's tie rules for maximum / clamp.
 * `advantages` are the (already normalised, clean_pufferl.py:211-213) minibatch advantages.  Strides in floats. */
int pb_ppo_loss(const float* logits, int64_t logits_stride, const float* value, int64_t value_stride,
                const int64_t* actions, const float* old_logprobs, const float* advantages, const float* returns,
                const float* old_values, int64_t m, int32_t n_act, float clip_coef, int32_t clip_vloss,
                float vf_clip_coef, float vf_coef, float ent_coef, float* grad_logits, int64_t grad_logits_stride,
                float* grad_value, int64_t grad_value_stride, double* stats8, void* stream);

/* -- MultiDiscrete heads (sampling + PPO loss) ----------------------------------------------------------------------
 * pb_sample_logits_multi replaces sample_logits (pufferlib/frameworks/cleanrl.py:25-47) for a LIST of logits, one per
 * head of a MultiDiscrete space (models.Default's decoder ModuleList, pufferlib/models.py:29-38, 57-59), when sampling:
 * per head logsumexp and an inverse-CDF draw on the counter-based uniform of (seed, offset + *offset_dev, row, head);
 * actions [n][n_heads] int64, logprob = sum over heads, entropy = sum over heads; the optional row stores are those of
 * pb_sample_logits (actions_row is [n][n_heads]).  The head term of the RNG key vanishes for head 0, so nvec = {k}
 * reproduces pb_sample_logits bit for bit.  The logits of one row are the heads' columns one after another, logits_stride
 * floats apart (the packed [M, 8] head output: all heads | value | zero padding).  nvec_host: HOST array of n_heads
 * (<= 16) sizes with sum <= 64.
 * pb_ppo_loss_multi is pb_ppo_loss (the loss block of clean_pufferl.py:202-238) with newlogprob = sum_h normalized_h[a_h]
 * and entropy = sum_h H_h: same six fp64 statistics, ATen tie rules and gradient layout (gradient columns follow the
 * logit columns; a packed [m][8] gradient row -- grad_value == grad_logits + sum(nvec), both strides 8 -- is written
 * whole, zero padding included).  actions: [m][n_heads] int64, clamped per head into [0, nvec[h]). */
int pb_sample_logits_multi(const float* logits, int64_t logits_stride, int64_t n, const int32_t* nvec_host, int32_t n_heads,
                           uint64_t seed, uint64_t offset, const uint64_t* offset_dev, int64_t* actions, float* logprobs,
                           float* entropies, const float* value, int64_t value_stride, float* values_row,
                           float* logprobs_row, int64_t* actions_row, void* stream);
int pb_ppo_loss_multi(const float* logits, int64_t logits_stride, const float* value, int64_t value_stride,
                      const int64_t* actions, const float* old_logprobs, const float* advantages, const float* returns,
                      const float* old_values, int64_t m, const int32_t* nvec_host, int32_t n_heads, float clip_coef,
                      int32_t clip_vloss, float vf_clip_coef, float vf_coef, float ent_coef, float* grad_logits,
                      int64_t grad_logits_stride, float* grad_value, int64_t grad_value_stride, double* stats8,
                      void* stream);

/* -- fused rollout-time policy step --------------------------------------------------------------------------------
 * For models.Default with 128 input features and 128 hidden units (pufferlib/models.py:12-62): encoder Linear + ReLU,
 * both heads, sample_logits (frameworks/cleanrl.py:25-47) and the value / logprob / action row stores of
 * Experience.store (clean_pufferl.py:443-446) in ONE launch per env step; the hidden layer never leaves the SM
 * (mma.sync TF32 tensor-core tiles, fp32 accumulate).  w_heads / b_heads: the 8-row padded head matrix
 * (n_act logits | value | zeros).  w_enc is consumed as TF32: the tensor core ignores the low 13 mantissa bits, so pass
 * it pre-rounded (cvt.rna) for round-to-nearest products.  Sampling: counter-based inverse CDF on (seed, *counter_dev, row).  With a non-null
 * ticket_dev (one zero-initialised uint32 owned by the caller) the last CTA to finish advances *counter_dev by 1, so a
 * captured rollout graph needs no separate counter update per env step. */
int pb_policy_mlp_sample(const float* obs, int64_t obs_stride, const float* w_enc, const float* b_enc,
                         const float* w_heads, const float* b_heads, int64_t m, int32_t in_features, int32_t hidden_size,
                         int32_t n_act, uint64_t seed, uint64_t* counter_dev, uint32_t* ticket_dev, int64_t* actions,
                         float* logprobs, float* values, float* entropies, void* stream);

/* -- persistent rollout (env steps with the policy in the loop) -------------------------------------------------------
 * The H-iteration body of clean_pufferl.evaluate (clean_pufferl.py:84-124: recv -> policy -> store -> send) for a
 * breakout handle and models.Default (128 features, 128 hidden, n_act <= 4) in ONE launch: a CTA owns 128 envs for all
 * `horizon` steps, env state in registers, observation tile in shared memory feeding both the TMA store to the rollout
 * tensor and the tcgen05 encoder GEMM (W_enc resident in shared memory), heads + sampling + value / logprob / action row
 * stores by the env's own thread.  Rollout tensors are time-major [horizon * N] (row t*N + e); row 0 takes reward / done
 * from the carry buffers (the vecenv's own buffers, pb_env_out with dones_f32), the step that closes the rollout writes
 * the carry buffers (obs / rewards / terminals / dones_f32) -- the bound-rollout convention of vector.B200.  Sampling:
 * the counter-based inverse CDF of pb_policy_mlp_sample with step counters *counter_dev .. *counter_dev + horizon - 1;
 * *counter_dev is advanced by `horizon`.  num_envs must be a multiple of 128. */
int pb_rollout_breakout_mlp(pb_env* env, int32_t horizon, float* obs, float* rewards, float* dones, float* values,
                            float* logprobs, int64_t* actions, const pb_env_out* carry, const float* w_enc,
                            const float* b_enc, const float* w_heads, const float* b_heads, int32_t n_act, uint64_t seed,
                            uint64_t* counter_dev, void* stream);

/* Validation hook: relu(h) [N][128] and the head outputs [N][8] of step 0 of the following rollouts (null: off). */
int pb_rollout_debug_buffers(float* hidden, float* out);

/* -- policy tail backward ---------------------------------------------------------------------------------------------
 * For models.Default (pufferlib/models.py:12-62: Linear+ReLU encoder, action head + value head): everything of the
 * backward pass after the encoder GEMM, in ONE pass over the hidden layer instead of five ATen launches:
 *   dpre[m][H]      = (dout[m][0..7] @ w_heads[8][H]) * (hidden > 0)                  (heads dX + ReLU backward)
 *   grads_out       = [ dW_heads (8*H) | db_enc (H) = column sums of dpre | db_heads (8) = column sums of dout ]
 * dout holds the loss gradient w.r.t. the 8 padded head outputs (n_act logits, the value, zero padding), row stride
 * dout_stride floats.  Deterministic (two-stage partial sums).  H = 128.  Pointers 16-byte aligned. */
size_t pb_mlp_tail_workspace_bytes(int64_t m, int32_t hidden_size);
int pb_mlp_tail_backward(const float* dout, int64_t dout_stride, const float* w_heads, const float* hidden, int64_t m,
                         int32_t hidden_size, float* dpre, float* grads_out, void* workspace, size_t workspace_bytes,
                         void* stream);

/* -- fused minibatch update (forward + PPO loss + backward) -------------------------------------------------------------
 * One minibatch of clean_pufferl.train (clean_pufferl.py:186-244) for models.Default (pufferlib/models.py:12-62) with
 * 128 fp32 input features, 128 hidden units and <= 7 actions, up to and including the gradients, in ONE persistent
 * tcgen05 kernel (+ a small deterministic partial-sum kernel): encoder GEMM and dW_enc = dPre^T x on the 5th-gen tensor
 * cores (kind::tf32, fp32 accumulation in TMEM), heads / pb_ppo_loss row math / ReLU backward in the epilogue warps.
 * The observations are read from HBM once; hidden and dPre never leave the SM.
 *   x            n_slabs slabs of slab_rows rows x 128 features, row stride ldx floats; slab s starts slab_stride_rows rows
 *                after slab s-1 (the zero-copy minibatch view of the time-major rollout; n_slabs = 1: a plain matrix)
 *   w_heads/b_heads  the 8-row padded head matrix of pb_pack_heads (n_act logit rows | value row | zeros)
 *   actions .. old_values   per-row tensors; slab s starts at element s * row_slab_stride (row_slab_stride = slab_rows:
 *                slab-major copies; = the rollout's slab distance: the arrival-order rollout tensors themselves, no copies)
 *   adv_norm     nullable device (mean, 1/(std + 1e-8)) applied to `advantages` on the fly (clean_pufferl.py:211-213);
 *   returns      nullable: advantages (raw) + old_values is used (clean_pufferl.py:476-481)
 *   grad_flat    [128*128 + 8*128 + 128 + 8]: dW_enc | dW_heads | db_enc | db_heads  (what pb_clip_adam consumes)
 *   stats8       the six loss sums of pb_ppo_loss (zeroed here)
 *   dpre_out     must be NULL (anything else returns PB_ERR_UNSUPPORTED): dW_enc = dPre^T x is always accumulated inside
 *                the kernel, and dPre is never written to memory
 *   dbg_*        nullable dumps of relu(h) [M][128], dPre [M][128], dOut [M][8] for validation. */
size_t pb_mlp_update_workspace_bytes(void);
/* the reduce step of pb_mlp_update_fused also leaves the sum of squares of the whole gradient it wrote as
 * pb_mlp_update_sumsq_parts() doubles at byte pb_mlp_update_sumsq_offset() of the workspace: input of pb_clip_adam_parts */
size_t pb_mlp_update_sumsq_offset(void);
int32_t pb_mlp_update_sumsq_parts(void);
/* profiling hook: SM-clock stamps of tiles 8..11, [grid][18 warps][4][8] int64; NULL switches it off */
int pb_mlp_update_debug_clock(long long* buf);
int pb_mlp_update_fused(const float* x, int64_t ldx, int64_t slab_rows, int64_t slab_stride_rows, int32_t n_slabs,
                        const float* w_enc, const float* b_enc, const float* w_heads, const float* b_heads,
                        const int64_t* actions, const float* old_logprobs, const float* advantages, const float* returns,
                        const float* old_values, const float* adv_norm, int64_t row_slab_stride, int32_t n_act,
                        float clip_coef, int32_t clip_vloss, float vf_clip_coef,
                        float vf_coef, float ent_coef, float* grad_flat, double* stats8, void* workspace,
                        size_t workspace_bytes, float* dpre_out, float* dbg_hidden, float* dbg_dpre, float* dbg_dout,
                        void* stream);

/* Advantage statistics of the zero-copy slab minibatches from ARRIVAL-order advantages (pb_gae_tm): minibatch mb = slabs
 * g * n_minibatches + mb (g < n_slabs) of slab_rows consecutive rows.  norm_out[mb] = (mean, 1 / (unbiased std + 1e-8)),
 * the constants of clean_pufferl.py:211-213, which pb_mlp_update_fused applies on the fly.
 * workspace: pb_adv_norm_workspace_bytes(n_minibatches, slab_rows * n_slabs). */
int pb_adv_stats_slabs(const float* advantages_time_major, int64_t slab_rows, int32_t n_slabs, int32_t n_minibatches,
                       float* norm_out, void* workspace, size_t workspace_bytes, void* stream);

/* -- optimizer step for small policies -------------------------------------------------------------------------------
 * clip_grad_norm_ + Adam of clean_pufferl.py:240-244 (torch.nn.utils.clip_grad_norm_(params, max_grad_norm);
 * optimizer.step() with torch.optim.Adam(eps=1e-5)) in ONE single-CTA launch for up to 1 Mi parameters in up to 8
 * tensors.  Gradients are first multiplied by grad_scale (1/world_size after a sum all-reduce), the global L2 norm
 * gives coef = min(max_grad_norm / (norm + 1e-6), 1) (max_grad_norm <= 0: no clipping), then per element
 *   m += (1-b1)(g-m);  v = b2 v + (1-b2) g^2;  step += 1;  p -= lr/(1-b1^step) * m / (sqrt(v)/sqrt(1-b2^step) + eps)
 * on the optimizer's own state tensors (`step` is torch's per-parameter fp32 device scalar).  lr_dev (nullable)
 * overrides lr with a device scalar (CUDA-graph replays read the annealed value).  total_norm_out: nullable. */
typedef struct pb_adam_tensor {
    float* param;
    float* exp_avg;
    float* exp_avg_sq;
    float* step;
    const float* grad;
    int64_t numel;
} pb_adam_tensor;
int pb_clip_adam(const pb_adam_tensor* tensors, int32_t n_tensors, float max_grad_norm, float grad_scale, float lr,
                 const float* lr_dev, float beta1, float beta2, float eps, float* total_norm_out, void* stream);

/* -- gradient all-reduce over NVLink peer memory (multi-GPU, one node; SURVEY §8e: the reference has no distributed path) --
 * Each rank allocates one buffer (pb_peer_alloc: cudaMalloc + IPC handle), exchanges the 64-byte handles through the
 * host (torch.distributed), maps every peer's buffer (pb_peer_open) and fills a pb_peer_comm.  pb_peer_allreduce sums a
 * flat fp32 buffer in place over all ranks inside ONE single-CTA kernel: copy to the own peer-visible slot, raise a flag
 * in every peer's buffer, wait for all flags, add all ranks' slots in rank order with direct NVLink loads (identical
 * bits on every rank).  No host involvement per call: it can be captured in a CUDA graph.  pb_clip_adam_peer is
 * pb_clip_adam with that all-reduce of the flat gradient buffer fused in front (all `grad` pointers of the tensors must
 * lie inside grad_flat[0..grad_flat_numel)); pass grad_scale = 1/world for the mean. */
#define PB_PEER_MAX_RANKS 8
typedef struct pb_peer_comm {
    int32_t world, rank;
    void* base[PB_PEER_MAX_RANKS]; /* rank r's buffer as mapped in THIS process (base[rank] = the own allocation) */
    uint64_t* epoch;               /* one zero-initialised device uint64 owned by the caller (calls made so far) */
    int64_t capacity;              /* floats per gradient slot */
} pb_peer_comm;
size_t pb_peer_buffer_bytes(int64_t capacity_floats);
int pb_peer_alloc(size_t bytes, void** ptr_out, void* handle64_out);
int pb_peer_open(const void* handle64, void** ptr_out);
int pb_peer_close(void* ptr);
int pb_peer_free(void* ptr);
int pb_peer_allreduce(const pb_peer_comm* comm, float* flat, int64_t n, void* stream);
/* Multi-CTA forms (the single-CTA calls above stay for callers without partial sums of squares): pb_peer_allreduce_parts
 * sums flat[0..n) over the ranks with pb_peer_slices() CTAs and writes that many partial sums of squares of the result;
 * pb_clip_adam_parts is pb_clip_adam with the norm taken from n_parts partial sums of squares of the summed, unscaled
 * gradient; it advances *peer_epoch (nullable: the communicator's counter) for the all-reduce that preceded it.  One optimizer
 * step may be in flight per device at a time (device-wide ticket counters). */
int pb_peer_allreduce_parts(const pb_peer_comm* comm, float* flat, int64_t n, double* sumsq_parts, void* stream);
int32_t pb_peer_slices(void);
typedef struct pb_head_pack {   /* optional tail of pb_clip_adam_parts: pb_pack_heads (without the encoder copy) on the updated parameters */
    const float* w_dec;
    const float* b_dec;
    const float* w_val;
    const float* b_val;
    float* w_cat;
    float* b_cat;
    int32_t n_act;
    int32_t hid;
} pb_head_pack;
int pb_clip_adam_parts(const pb_adam_tensor* tensors, int32_t n_tensors, float max_grad_norm, float grad_scale, float lr,
                       const float* lr_dev, float beta1, float beta2, float eps, float* total_norm_out,
                       const double* sumsq_parts, int32_t n_parts, unsigned long long* peer_epoch, const pb_head_pack* pack,
                       void* stream);
/* pb_peer_allreduce_parts + pb_clip_adam_parts as ONE kernel (pb_peer_slices() CTAs with a grid barrier between the exchange
 * and the update): the multi-GPU optimizer step of the captured update graph.  sumsq_scratch: pb_peer_slices() doubles. */
int pb_clip_adam_peer_parts(const pb_adam_tensor* tensors, int32_t n_tensors, float max_grad_norm, float grad_scale, float lr,
                            const float* lr_dev, float beta1, float beta2, float eps, float* total_norm_out,
                            const pb_peer_comm* comm, float* grad_flat, int64_t grad_flat_numel, double* sumsq_scratch,
                            const pb_head_pack* pack, void* stream);
int pb_clip_adam_peer(const pb_adam_tensor* tensors, int32_t n_tensors, float max_grad_norm, float grad_scale, float lr,
                      const float* lr_dev, float beta1, float beta2, float eps, float* total_norm_out,
                      const pb_peer_comm* comm, float* grad_flat, int64_t grad_flat_numel, void* stream);

/* The 8-row head matrix of models.Default (pufferlib/models.py:33-38: decoder rows | value_head row | zero padding),
 * its bias, and (optionally) the encoder weight rounded to TF32, in one launch: the operands pb_policy_mlp_sample,
 * pb_mlp_tail_backward and the 8-column head GEMM consume. */
int pb_pack_heads(const float* w_dec, const float* b_dec, const float* w_val, const float* b_val, int32_t n_act,
                  int32_t hidden_size, float* w_cat, float* b_cat, const float* w_enc, float* w_enc_tf32,
                  int64_t enc_numel, void* stream);

/* -- structured observation pack / unpack (SURVEY §8 row a-4) --------------------------------------------------------
 * Replaces, for N samples at once, `emulate` / `nativize` (pufferlib/extensions.pyx:19-30, 32-49): leaf tensors
 * [N][nbytes[k]] <-> C-aligned records [N][record_bytes] whose layout is `np.dtype(..., align=True)` of the space
 * (pufferlib/emulation.py:68-80; computed by the host layer).  Padding bytes are packed as zero.  `leaves_host` is a
 * HOST array of n_leaves DEVICE pointers.  Up to 32 leaves. */
typedef struct {
    int32_t n_leaves;
    int32_t record_bytes;
    int32_t offset[32]; /* byte offset of leaf k inside a record */
    int32_t nbytes[32]; /* byte size of leaf k */
} pb_struct_layout;
int pb_struct_pack(const pb_struct_layout* layout, const void* const* leaves_host, void* records, int64_t record_stride,
                   int64_t n, void* stream);
int pb_struct_unpack(const pb_struct_layout* layout, const void* records, int64_t record_stride,
                     void* const* leaves_host, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PUFFERLIB_B200_H */
