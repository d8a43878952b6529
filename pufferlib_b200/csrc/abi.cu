// abi.cu -- C-ABI plumbing of libpuffer_b200.so: error strings, env handle lifecycle and dispatch.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include "env_common.cuh"

static thread_local char g_err[512] = "";

void pb_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

unsigned long long g_pb_launches = 0;

extern "C" const char* pb_last_error(void) { return g_err; }
extern "C" uint64_t pb_launch_count(void) { return g_pb_launches; }
extern "C" int pb_abi_version(void) { return PB_ABI_VERSION; }

extern "C" int pb_device_count(int* out_count) {
    PB_REQUIRE(out_count, PB_ERR_INVALID, "pb_device_count: null pointer");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        pb_set_error("cudaGetDeviceCount: %s", cudaGetErrorString(e));
        *out_count = 0;
        return PB_ERR_CUDA;
    }
    *out_count = n;
    return PB_OK;
}

int pb_env_alloc_common(pb_env* env) {
    const size_t n = (size_t)env->cfg.num_envs;
    PB_CUDA(cudaMalloc(&env->d_done, n));
    PB_CUDA(cudaMalloc(&env->d_ep_return, n * sizeof(double)));
    PB_CUDA(cudaMalloc(&env->d_ep_length, n * sizeof(int32_t)));
    PB_CUDA(cudaMalloc(&env->d_row_return, n * sizeof(double)));
    PB_CUDA(cudaMalloc(&env->d_row_length, n * sizeof(int32_t)));
    PB_CUDA(cudaMalloc(&env->d_row_score, n * sizeof(float)));
    PB_CUDA(cudaMalloc(&env->d_stats, PB_STAT_SLOTS * 4 * sizeof(double)));
    PB_CUDA(cudaMallocHost(&env->h_stats_pinned, PB_STAT_SLOTS * 4 * sizeof(double)));
    PB_CUDA(cudaMemset(env->d_done, 1, n));  // GymnasiumPufferEnv starts with done = True (emulation.py:129)
    PB_CUDA(cudaMemset(env->d_ep_return, 0, n * sizeof(double)));
    PB_CUDA(cudaMemset(env->d_ep_length, 0, n * sizeof(int32_t)));
    PB_CUDA(cudaMemset(env->d_row_return, 0, n * sizeof(double)));
    PB_CUDA(cudaMemset(env->d_row_length, 0, n * sizeof(int32_t)));
    PB_CUDA(cudaMemset(env->d_row_score, 0, n * sizeof(float)));
    PB_CUDA(cudaMemset(env->d_stats, 0, PB_STAT_SLOTS * 4 * sizeof(double)));
    return PB_OK;
}

void pb_env_free_common(pb_env* env) {
    cudaFree(env->d_done);
    cudaFree(env->d_ep_return);
    cudaFree(env->d_ep_length);
    cudaFree(env->d_row_return);
    cudaFree(env->d_row_length);
    cudaFree(env->d_row_score);
    cudaFree(env->d_stats);
    if (env->h_stats_pinned) cudaFreeHost(env->h_stats_pinned);
}

extern "C" int pb_env_create(const pb_env_config* cfg, pb_env** out) {
    PB_REQUIRE(cfg && out, PB_ERR_INVALID, "pb_env_create: null pointer");
    *out = nullptr;
    PB_REQUIRE(cfg->num_envs >= 1, PB_ERR_INVALID, "num_envs must be at least 1");  // vector.py:578-579
    PB_REQUIRE(cfg->kind >= PB_ENV_SQUARED && cfg->kind <= PB_ENV_SPACES, PB_ERR_INVALID, "unknown env kind %d",
               cfg->kind);
    int ndev = 0;
    PB_CUDA(cudaGetDeviceCount(&ndev));
    PB_REQUIRE(cfg->device >= 0 && cfg->device < ndev, PB_ERR_CUDA, "CUDA device %d not available (%d devices)",
               cfg->device, ndev);
    PB_CUDA(cudaSetDevice(cfg->device));
    pb_env* env = (pb_env*)calloc(1, sizeof(pb_env));
    PB_REQUIRE(env, PB_ERR_CUDA, "out of host memory");
    env->cfg = *cfg;
    int rc = pb_env_alloc_common(env);
    if (rc == PB_OK) {
        switch (cfg->kind) {
            case PB_ENV_SQUARED: rc = pb_squared_create(env); break;
            case PB_ENV_BREAKOUT: rc = pb_breakout_create(env); break;
            case PB_ENV_SNAKE: rc = pb_snake_create(env); break;
            case PB_ENV_PONG: rc = pb_pong_create(env); break;
            case PB_ENV_SPACES: rc = pb_spaces_create(env); break;
        }
    }
    if (rc != PB_OK) {
        if (env->vt && env->vt->destroy) env->vt->destroy(env);
        pb_env_free_common(env);
        free(env);
        return rc;
    }
    env->info.num_envs = cfg->num_envs;
    *out = env;
    return PB_OK;
}

extern "C" int pb_env_destroy(pb_env* env) {
    if (!env) return PB_OK;
    cudaSetDevice(env->cfg.device);
    if (env->vt && env->vt->destroy) env->vt->destroy(env);
    pb_env_free_common(env);
    free(env);
    return PB_OK;
}

extern "C" int pb_env_get_info(const pb_env* env, pb_env_info* out) {
    PB_REQUIRE(env && out, PB_ERR_INVALID, "pb_env_get_info: null pointer");
    *out = env->info;
    return PB_OK;
}

extern "C" int pb_env_action_nvec(const pb_env* env, int32_t* nvec_out, int32_t* n_heads_out) {
    PB_REQUIRE(env && nvec_out && n_heads_out, PB_ERR_INVALID, "pb_env_action_nvec: null pointer");
    for (int h = 0; h < 8; ++h) nvec_out[h] = h < env->n_heads ? env->nvec[h] : 0;
    *n_heads_out = env->n_heads;
    return PB_OK;
}

static int check_out(const pb_env* env, const pb_env_out* out, const char* who) {
    PB_REQUIRE(out && out->obs && out->rewards && out->terminals && out->truncations && out->masks, PB_ERR_INVALID,
               "%s: obs/rewards/terminals/truncations/masks pointers are required", who);
    PB_REQUIRE(out->obs_stride >= env->info.obs_bytes, PB_ERR_INVALID, "%s: obs_stride %lld < obs_bytes %lld", who,
               (long long)out->obs_stride, (long long)env->info.obs_bytes);
    return PB_OK;
}

extern "C" int pb_env_reset(pb_env* env, uint64_t seed, const pb_env_out* out, void* stream) {
    PB_REQUIRE(env, PB_ERR_INVALID, "pb_env_reset: null handle");
    int rc = check_out(env, out, "pb_env_reset");
    if (rc) return rc;
    PB_CUDA(cudaSetDevice(env->cfg.device));
    env->write_const = true;
    rc = env->vt->reset(env, seed, out, (cudaStream_t)stream);
    if (rc == PB_OK) {
        env->was_reset = true;
        env->const_trunc = out->truncations;
        env->const_masks = out->masks;
        env->cur_obs = out->obs;
        env->cur_obs_stride = out->obs_stride;
    }
    return rc;
}

extern "C" int pb_env_step(pb_env* env, const int64_t* actions, const pb_env_out* out, void* stream) {
    PB_REQUIRE(env, PB_ERR_INVALID, "pb_env_step: null handle");
    PB_REQUIRE(env->was_reset, PB_ERR_STATE, "step() called before reset()");  // emulation.py:198-199
    PB_REQUIRE(actions, PB_ERR_INVALID, "pb_env_step: null actions");
    int rc = check_out(env, out, "pb_env_step");
    if (rc) return rc;
    PB_CUDA(cudaSetDevice(env->cfg.device));
    env->write_const = out->truncations != env->const_trunc || out->masks != env->const_masks;
    rc = env->vt->step(env, actions, out, (cudaStream_t)stream);
    if (rc == PB_OK) {
        env->const_trunc = out->truncations;
        env->const_masks = out->masks;
        env->cur_obs = out->obs;
        env->cur_obs_stride = out->obs_stride;
    }
    return rc;
}

extern "C" int pb_env_episode_rows(pb_env* env, const double** episode_return, const int32_t** episode_length,
                                   const float** score) {
    PB_REQUIRE(env, PB_ERR_INVALID, "pb_env_episode_rows: null handle");
    if (episode_return) *episode_return = env->d_row_return;
    if (episode_length) *episode_length = env->d_row_length;
    if (score) *score = env->d_row_score;
    return PB_OK;
}

extern "C" int pb_env_stats_read(pb_env* env, double* out4_host, int clear, void* stream) {
    PB_REQUIRE(env && out4_host, PB_ERR_INVALID, "pb_env_stats_read: null pointer");
    cudaStream_t s = (cudaStream_t)stream;
    PB_CUDA(cudaSetDevice(env->cfg.device));
    const size_t bytes = PB_STAT_SLOTS * 4 * sizeof(double);
    PB_CUDA(cudaMemcpyAsync(env->h_stats_pinned, env->d_stats, bytes, cudaMemcpyDeviceToHost, s));
    if (clear) PB_CUDA(cudaMemsetAsync(env->d_stats, 0, bytes, s));
    PB_CUDA(cudaStreamSynchronize(s));
    for (int k = 0; k < 4; ++k) out4_host[k] = 0.0;
    for (int slot = 0; slot < PB_STAT_SLOTS; ++slot)
        for (int k = 0; k < 4; ++k) out4_host[k] += env->h_stats_pinned[slot * 4 + k];
    return PB_OK;
}

// cudaDevAttrMultiProcessorCount of the current device, cached per device ordinal
int pb_num_sms() {
    static int cache[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (!cache[dev]) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n < 1) n = 148;
        cache[dev] = n;
    }
    return cache[dev];
}
