// env_spaces.cu -- N instances of ocean.Spaces behind vector.Serial semantics, on the device (sm_100a).
//
// Restatement of (paths under /root/reference/pufferlib/):
//   environments/ocean/ocean.py:356-404   Spaces: Dict obs {image float32[5][5], flat int8[5]}, Dict actions
//                                         {image, flat} of Discrete(2); every step is terminal; reward 0.5 per head
//                                         whose action equals [sum(obs part) > 0]; step returns the reset observation
//   emulation.py:68-80, 115-120           obs record = np.dtype(align=True) of the Dict with gymnasium's sorted keys:
//                                         flat int8[5] @0, pad, image f32[5][5] @8, 108 bytes; actions MultiDiscrete([2,2])
//                                         with column 0 = flat, column 1 = image
//   postprocess.py:8-54                   EpisodeStats: episode_return = reward, episode_length = 1, score = reward
//   vector.py:112-156, 639-641            Serial: `if env.done: reset() else: step()` per send
// The reference draws from numpy's process-global stream (randn / randint), which has no per-env device form; the
// observations come from the counter-based rand32 of oracle/SPEC_spaces.md: reset k of env e uses draws
// 30k .. 30k+29 of seed_e = seed + global env index.  Image values are multiples of 1/128, so the sign of their sum is
// exact in any summation order and the device agrees with oracle/spaces.py bit for bit.
//
// One thread per env regenerates its observation from (seed_e, k) -- the per-env state is the reset count alone --
// stages the 27 words of its record in shared memory, and the block then writes its rows with consecutive threads
// on consecutive words (one contiguous span when the rows are packed).
#include "env_common.cuh"

namespace {

constexpr int SP_THREADS = 128;
constexpr int SP_WORDS = 27;   // 108-byte record

struct SpacesState {
    uint32_t* d_k;          // [N] reset count since async_reset (selects the draws of the current observation)
    uint64_t seed_base;     // seed + env_index_offset of the last async_reset
};

struct SpOut {
    uint8_t* obs;
    int64_t obs_stride;
    float* rewards;
    uint8_t* terminals;
    uint8_t* truncations;
    uint8_t* masks;
    float* dones_f32;
    bool write_const;
};

__device__ __forceinline__ uint32_t rand32(uint64_t seed_e, uint64_t ctr) {
    return pb_mix32(seed_e * 0x9E3779B97F4A7C15ull + ctr * 0xD1B54A32D192ED03ull);
}

// mode 0: reset rows for every env (async_reset); mode 1: vectoriser send (reset-or-step)
template <int MODE>
__global__ void __launch_bounds__(SP_THREADS) k_spaces(SpacesState st, int n, const int64_t* __restrict__ actions,
                                                       uint8_t* done, SpOut out, EpisodeAcc acc) {
    __shared__ uint32_t s_rec[SP_THREADS * SP_WORDS];
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = e < n;
    bool reset_row = true, terminal = false;
    float reward = 0.f;
    if (active) {
        uint32_t k = 0;
        if (MODE == 1) {
            k = st.d_k[e];
            if (done[e]) ++k;                  // vector.py:147-149: reset, action ignored
            else reset_row = false;
        }
        const uint64_t seed_e = st.seed_base + (uint64_t)e;
        const uint64_t ctr0 = (uint64_t)k * 30u;
        uint32_t* rec = s_rec + threadIdx.x * SP_WORDS;
        int image_sum = 0;                     // in units of 1/128
        for (int j = 0; j < 25; ++j) {
            const uint32_t r = rand32(seed_e, ctr0 + j);
            const int v = (int)(r & 255u) + (int)((r >> 8) & 255u) + (int)((r >> 16) & 255u) + (int)(r >> 24) - 510;
            image_sum += v;
            rec[2 + j] = __float_as_uint((float)v * (1.0f / 128.0f));
        }
        uint32_t w0 = 0, w1 = 0;
        int flat_sum = 0;
        for (int j = 0; j < 5; ++j) {
            const int f = (int)(rand32(seed_e, ctr0 + 25 + j) % 3u) - 1;
            flat_sum += f;
            const uint32_t b = (uint32_t)(uint8_t)(int8_t)f;
            if (j < 4) w0 |= b << (8 * j);
            else w1 = b;
        }
        rec[0] = w0;
        rec[1] = w1;
        if (!reset_row) {                      // ocean.py:391-404
            int64_t a_flat = actions[2 * (int64_t)e], a_image = actions[2 * (int64_t)e + 1];
            a_flat = a_flat < 0 ? 0 : (a_flat > 1 ? 1 : a_flat);
            a_image = a_image < 0 ? 0 : (a_image > 1 ? 1 : a_image);
            if ((image_sum > 0) == (a_image == 1)) reward += 0.5f;
            if ((flat_sum > 0) == (a_flat == 1)) reward += 0.5f;
            terminal = true;
        }
        if (MODE == 1) st.d_k[e] = k;
        else st.d_k[e] = 0;
        done[e] = terminal ? 1 : 0;
        out.rewards[e] = reward;
        out.terminals[e] = terminal ? 1 : 0;
        if (out.write_const) out.truncations[e] = 0;
        if (out.write_const) out.masks[e] = 1;
        if (out.dones_f32) out.dones_f32[e] = terminal ? 1.f : 0.f;
    }
    episode_update(acc, e, active, reset_row, (double)reward, terminal, reward);
    __syncthreads();
    const int e0 = blockIdx.x * blockDim.x;
    const int rows = min(SP_THREADS, n - e0);
    for (int w = threadIdx.x; w < rows * SP_WORDS; w += SP_THREADS) {
        const int r = w / SP_WORDS, c = w - r * SP_WORDS;
        *reinterpret_cast<uint32_t*>(out.obs + (int64_t)(e0 + r) * out.obs_stride + 4 * c) = s_rec[w];
    }
}

int spaces_launch(pb_env* env, int mode, const int64_t* actions, const pb_env_out* out, cudaStream_t s) {
    SpacesState* st = (SpacesState*)env->kind;
    const int n = env->cfg.num_envs;
    PB_REQUIRE(out->obs_stride % 4 == 0 && ((uintptr_t)out->obs & 3) == 0, PB_ERR_INVALID,
               "spaces: obs pointer/stride must be 4-byte aligned");
    SpOut o{(uint8_t*)out->obs, out->obs_stride, out->rewards, out->terminals, out->truncations, out->masks,
            out->dones_f32, env->write_const};
    const int blocks = (int)pb_ceil_div(n, SP_THREADS);
    if (mode == 0)
        k_spaces<0><<<blocks, SP_THREADS, 0, s>>>(*st, n, actions, env->d_done, o, pb_episode_acc(env));
    else
        k_spaces<1><<<blocks, SP_THREADS, 0, s>>>(*st, n, actions, env->d_done, o, pb_episode_acc(env));
    PB_LAUNCH_CHECK();
    return PB_OK;
}

int spaces_reset(pb_env* env, uint64_t seed, const pb_env_out* out, cudaStream_t s) {
    SpacesState* st = (SpacesState*)env->kind;
    st->seed_base = seed + (uint64_t)env->cfg.env_index_offset;
    return spaces_launch(env, 0, nullptr, out, s);
}

int spaces_step(pb_env* env, const int64_t* actions, const pb_env_out* out, cudaStream_t s) {
    return spaces_launch(env, 1, actions, out, s);
}

void spaces_destroy(pb_env* env) {
    SpacesState* st = (SpacesState*)env->kind;
    if (!st) return;
    cudaFree(st->d_k);
    delete st;
    env->kind = nullptr;
}

const pb_env_vtable SPACES_VT = {spaces_reset, spaces_step, spaces_destroy};

}  // namespace

int pb_spaces_create(pb_env* env) {
    SpacesState* st = new SpacesState();
    env->kind = st;
    env->vt = &SPACES_VT;
    const size_t n = (size_t)env->cfg.num_envs;
    PB_CUDA(cudaMalloc(&st->d_k, n * sizeof(uint32_t)));
    PB_CUDA(cudaMemset(st->d_k, 0, n * sizeof(uint32_t)));
    env->info.obs_dtype = PB_DTYPE_U8;
    env->info.obs_ndim = 1;
    env->info.obs_shape[0] = 108;
    env->info.obs_bytes = 108;
    env->info.num_actions = 0;                 // MultiDiscrete: pb_env_action_nvec
    env->info.obs_low = 0.f;
    env->info.obs_high = 255.f;
    env->n_heads = 2;
    env->nvec[0] = 2;                          // flat
    env->nvec[1] = 2;                          // image
    return PB_OK;
}
