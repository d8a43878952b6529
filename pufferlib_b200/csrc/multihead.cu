// multihead.cu -- sampling epilogue and PPO loss for MultiDiscrete action spaces (several Discrete heads), sm_100a.
//
// Replaces, for a list of logits (/root/reference/pufferlib/frameworks/cleanrl.py:25-47 with `logits` a list, the
// models.Default decoder ModuleList of pufferlib/models.py:29-38, 57-59):
//   per head h: normalized_h = logits_h - logsumexp(logits_h);  action_h ~ Categorical(softmax(normalized_h))
//   logprob = sum_h normalized_h[action_h];  entropy = sum_h H_h
// and the loss block of clean_pufferl.py:202-238 with that logprob / entropy.  The logits of one row are the heads'
// columns one after another (nvec[0] of head 0, then head 1, ...), `logits_stride` floats per row: the packed [M, 8]
// output of models.Default.forward_packed (all heads | value | zero padding) is read in place.
//
// One thread per row, heads in a loop; a head's logits are re-read from L1 instead of being held in registers, so no
// head size limit beyond sum(nvec) <= 64.  Per head the arithmetic is pb_sample_logits / pb_ppo_loss expression for
// expression, and the RNG key (seed, offset, row, head) adds head * K_HEAD, which vanishes for head 0: nvec = [n]
// reproduces pb_sample_logits bit for bit.
#include "pb_common.cuh"

namespace {

constexpr int MH_MAX_HEADS = 16;
constexpr int MH_MAX_SUM = 64;
constexpr int MH_THREADS = 256;
constexpr uint64_t K_HEAD = 0x9FB21C651E98DF25ull;

struct Heads {
    int n;
    int total;                    // sum of nvec
    int size[MH_MAX_HEADS];
    int base[MH_MAX_HEADS];       // first column of head h
};

__global__ void __launch_bounds__(MH_THREADS) k_sample_multi(const float* __restrict__ logits, int64_t lstride, int64_t n,
                                                           Heads hd, uint64_t seed, uint64_t offset,
                                                           const uint64_t* __restrict__ offset_dev, int64_t* actions,
                                                           float* logprobs, float* entropies, const float* value,
                                                           int64_t vstride, float* values_row, float* logprobs_row,
                                                           int64_t* actions_row) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (offset_dev) offset += *offset_dev;
    const float* row = logits + i * lstride;
    float lp_sum = 0.f, ent_sum = 0.f;
    for (int h = 0; h < hd.n; ++h) {
        const float* l = row + hd.base[h];
        const int na = hd.size[h];
        float m = -INFINITY;
        for (int k = 0; k < na; ++k) m = fmaxf(m, __ldg(l + k));
        float sum = 0.f;
        for (int k = 0; k < na; ++k) sum += expf(__ldg(l + k) - m);
        const float lse = m + logf(sum);
        const uint32_t r = pb_mix32(seed * 0x9E3779B97F4A7C15ull + offset * 0xD1B54A32D192ED03ull +
                                    (uint64_t)i * 0x2545F4914F6CDD1Dull + (uint64_t)h * K_HEAD);
        const float u = (float)(r >> 8) * (1.0f / 16777216.0f);
        float cdf = 0.f, ent = 0.f, lp_a = 0.f;
        int a = -1;
        for (int k = 0; k < na; ++k) {
            const float nl = __ldg(l + k) - lse;
            const float pk = expf(nl);
            ent -= pk * fmaxf(nl, -3.4028234663852886e38f);
            cdf += pk;
            if (a < 0 && u < cdf) { a = k; lp_a = nl; }
        }
        if (a < 0) {  // rounding left cdf a hair below u: take the last action with non-zero probability
            for (int k = na - 1; k >= 0; --k)
                if (__ldg(l + k) - lse > -80.f) { a = k; lp_a = __ldg(l + k) - lse; break; }
            if (a < 0) { a = na - 1; lp_a = __ldg(l + a) - lse; }
        }
        lp_sum = h == 0 ? lp_a : lp_sum + lp_a;
        ent_sum = h == 0 ? ent : ent_sum + ent;
        if (actions) actions[i * hd.n + h] = a;
        if (actions_row) actions_row[i * hd.n + h] = a;
    }
    if (logprobs) logprobs[i] = lp_sum;
    if (entropies) entropies[i] = ent_sum;
    if (logprobs_row) logprobs_row[i] = lp_sum;
    if (values_row && value) values_row[i] = value[i * vstride];
}

struct PpoMultiParams {
    const float* logits; int64_t lstride;
    const float* value; int64_t vstride;
    const int64_t* actions;       // [m][heads]
    const float* old_logprobs;
    const float* adv;
    const float* returns;
    const float* old_values;
    float* grad_logits; int64_t glstride;
    float* grad_value; int64_t gvstride;
    double* stats;
    int64_t m;
    float clip, vclip, vf_coef, ent_coef;
    int clip_vloss;
    int zero_pad_to;              // > 0: packed rows, columns total+1 .. zero_pad_to-1 of grad_logits are written as zero
};

__global__ void __launch_bounds__(MH_THREADS) k_ppo_loss_multi(PpoMultiParams p, Heads hd) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double s_pg = 0, s_v = 0, s_ent = 0, s_okl = 0, s_kl = 0, s_clip = 0;
    if (i < p.m) {
        const float* row = p.logits + i * p.lstride;
        float lse_h[MH_MAX_HEADS], ent_h[MH_MAX_HEADS];
        int a_h[MH_MAX_HEADS];
        float newlogprob = 0.f, entropy = 0.f;
        for (int h = 0; h < hd.n; ++h) {
            const float* l = row + hd.base[h];
            const int na = hd.size[h];
            float mx = -INFINITY;
            for (int k = 0; k < na; ++k) mx = fmaxf(mx, l[k]);
            float sum = 0.f;
            for (int k = 0; k < na; ++k) sum += expf(l[k] - mx);
            const float lse = mx + logf(sum);
            int a = (int)p.actions[i * hd.n + h];
            a = a < 0 ? 0 : (a >= na ? na - 1 : a);
            float ent = 0.f, nl_a = 0.f;
            for (int k = 0; k < na; ++k) {
                const float nl = l[k] - lse, pk = expf(nl);
                ent -= pk * nl;
                if (k == a) nl_a = nl;
            }
            lse_h[h] = lse; ent_h[h] = ent; a_h[h] = a;
            newlogprob = h == 0 ? nl_a : newlogprob + nl_a;
            entropy = h == 0 ? ent : entropy + ent;
        }
        const float logratio = newlogprob - p.old_logprobs[i];
        const float ratio = expf(logratio);
        const float adv = p.adv[i];
        const float pg1 = -adv * ratio;
        const float rc = fminf(fmaxf(ratio, 1.f - p.clip), 1.f + p.clip);
        const float pg2 = -adv * rc;
        const float pg = fmaxf(pg1, pg2);
        // ATen tie rules: maximum() splits the gradient on ties, clamp() passes it inside the inclusive bounds
        const float in_range = (ratio >= 1.f - p.clip && ratio <= 1.f + p.clip) ? 1.f : 0.f;
        float g_ratio;
        if (pg1 > pg2) g_ratio = -adv;
        else if (pg1 < pg2) g_ratio = -adv * in_range;
        else g_ratio = 0.5f * (-adv) + 0.5f * (-adv * in_range);
        const float inv_m = 1.0f / (float)p.m;
        const float g_nlp = g_ratio * ratio * inv_m;          // d loss / d newlogprob (the same for every head)
        const float v = p.value[i * p.vstride], ret = p.returns[i];
        const float dv = v - ret;
        float vl, g_v;
        if (p.clip_vloss) {
            const float ov = p.old_values[i];
            const float d = v - ov;
            const float dc = fminf(fmaxf(d, -p.vclip), p.vclip);
            const float vc = ov + dc;
            const float vu = dv * dv, vcl = (vc - ret) * (vc - ret);
            vl = fmaxf(vu, vcl);
            const float v_in = (d >= -p.vclip && d <= p.vclip) ? 1.f : 0.f;
            const float gu = 2.f * dv, gc = 2.f * (vc - ret) * v_in;
            g_v = vu > vcl ? gu : (vu < vcl ? gc : 0.5f * (gu + gc));
        } else {
            vl = dv * dv;
            g_v = 2.f * dv;
        }
        p.grad_value[i * p.gvstride] = 0.5f * p.vf_coef * g_v * inv_m;
        // d loss / d logit_{h,j} = g_nlp * (delta_{j,a_h} - p_{h,j}) + ent_coef/M * p_{h,j} * (nl_{h,j} + H_h)
        const float g_ent = p.ent_coef * inv_m;
        float* grow = p.grad_logits + i * p.glstride;
        for (int h = 0; h < hd.n; ++h) {
            const float* l = row + hd.base[h];
            float* g = grow + hd.base[h];
            for (int k = 0; k < hd.size[h]; ++k) {
                const float z = l[k] - lse_h[h];
                const float pk = expf(z);
                g[k] = g_nlp * ((k == a_h[h] ? 1.f : 0.f) - pk) + g_ent * pk * (z + ent_h[h]);
            }
        }
        for (int c = hd.total + 1; c < p.zero_pad_to; ++c) grow[c] = 0.f;
        s_pg = pg; s_v = vl; s_ent = entropy; s_okl = -logratio; s_kl = (ratio - 1.f) - logratio;
        s_clip = fabsf(ratio - 1.f) > p.clip ? 1.0 : 0.0;
    }
    // block reduction of the six sums (fp64), one atomic per block and statistic
    __shared__ double sh[6][MH_THREADS / 32];
    double vals[6] = {s_pg, s_v, s_ent, s_okl, s_kl, s_clip};
#pragma unroll
    for (int q = 0; q < 6; ++q) {
        double x = vals[q];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) x += __shfl_xor_sync(0xffffffffu, x, off);
        if ((threadIdx.x & 31) == 0) sh[q][threadIdx.x >> 5] = x;
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        double t = 0;
        for (int w = 0; w < MH_THREADS / 32; ++w) t += sh[threadIdx.x][w];
        atomicAdd(p.stats + threadIdx.x, t);
    }
}

int make_heads(const int32_t* nvec_host, int32_t n_heads, Heads* hd, const char* who) {
    PB_REQUIRE(nvec_host, PB_ERR_INVALID, "%s: null nvec", who);
    PB_REQUIRE(n_heads >= 1 && n_heads <= MH_MAX_HEADS, PB_ERR_UNSUPPORTED, "%s: n_heads must be in [1, %d]", who,
               MH_MAX_HEADS);
    hd->n = n_heads;
    hd->total = 0;
    for (int h = 0; h < n_heads; ++h) {
        PB_REQUIRE(nvec_host[h] >= 1, PB_ERR_INVALID, "%s: nvec[%d] = %d must be positive", who, h, nvec_host[h]);
        hd->size[h] = nvec_host[h];
        hd->base[h] = hd->total;
        hd->total += nvec_host[h];
        PB_REQUIRE(hd->total <= MH_MAX_SUM, PB_ERR_UNSUPPORTED, "%s: sum(nvec) must be at most %d", who, MH_MAX_SUM);
    }
    for (int h = n_heads; h < MH_MAX_HEADS; ++h) hd->size[h] = hd->base[h] = 0;
    return PB_OK;
}

}  // namespace

extern "C" int pb_sample_logits_multi(const float* logits, int64_t logits_stride, int64_t n, const int32_t* nvec_host,
                                      int32_t n_heads, uint64_t seed, uint64_t offset, const uint64_t* offset_dev,
                                      int64_t* actions, float* logprobs, float* entropies, const float* value,
                                      int64_t value_stride, float* values_row, float* logprobs_row, int64_t* actions_row,
                                      void* stream) {
    PB_REQUIRE(n >= 0, PB_ERR_INVALID, "pb_sample_logits_multi: negative n");
    Heads hd;
    int rc = make_heads(nvec_host, n_heads, &hd, "pb_sample_logits_multi");
    if (rc) return rc;
    if (n == 0) return PB_OK;
    PB_REQUIRE(logits, PB_ERR_INVALID, "pb_sample_logits_multi: null logits");
    PB_REQUIRE(!values_row || value, PB_ERR_INVALID, "pb_sample_logits_multi: values_row given without value");
    PB_REQUIRE(logits_stride >= hd.total, PB_ERR_INVALID, "pb_sample_logits_multi: logits_stride < sum(nvec)");
    k_sample_multi<<<(unsigned)pb_ceil_div(n, MH_THREADS), MH_THREADS, 0, (cudaStream_t)stream>>>(
        logits, logits_stride, n, hd, seed, offset, offset_dev, actions, logprobs, entropies, value, value_stride,
        values_row, logprobs_row, actions_row);
    PB_LAUNCH_CHECK();
    return PB_OK;
}

extern "C" int pb_ppo_loss_multi(const float* logits, int64_t logits_stride, const float* value, int64_t value_stride,
                                 const int64_t* actions, const float* old_logprobs, const float* advantages,
                                 const float* returns, const float* old_values, int64_t m, const int32_t* nvec_host,
                                 int32_t n_heads, float clip_coef, int32_t clip_vloss, float vf_clip_coef, float vf_coef,
                                 float ent_coef, float* grad_logits, int64_t grad_logits_stride, float* grad_value,
                                 int64_t grad_value_stride, double* stats8, void* stream) {
    PB_REQUIRE(m >= 1, PB_ERR_INVALID, "pb_ppo_loss_multi: m must be positive");
    Heads hd;
    int rc = make_heads(nvec_host, n_heads, &hd, "pb_ppo_loss_multi");
    if (rc) return rc;
    PB_REQUIRE(logits && value && actions && old_logprobs && advantages && returns && grad_logits && grad_value && stats8,
               PB_ERR_INVALID, "pb_ppo_loss_multi: null pointer");
    PB_REQUIRE(!clip_vloss || old_values, PB_ERR_INVALID, "pb_ppo_loss_multi: clip_vloss needs old_values");
    PB_REQUIRE(logits_stride >= hd.total && grad_logits_stride >= hd.total && value_stride >= 1 && grad_value_stride >= 1,
               PB_ERR_INVALID, "pb_ppo_loss_multi: bad strides");
    cudaStream_t s = (cudaStream_t)stream;
    PB_CUDA(cudaMemsetAsync(stats8, 0, 8 * sizeof(double), s));
    // packed [m][8] rows (heads | value | zero padding): the kernel writes the whole gradient row
    const bool packed = grad_logits_stride == 8 && hd.total + 1 <= 8 && grad_value == grad_logits + hd.total &&
                        grad_value_stride == 8;
    PpoMultiParams p{logits, logits_stride, value, value_stride, actions, old_logprobs, advantages, returns, old_values,
                     grad_logits, grad_logits_stride, grad_value, grad_value_stride, stats8, m, clip_coef, vf_clip_coef,
                     vf_coef, ent_coef, clip_vloss, packed ? 8 : 0};
    k_ppo_loss_multi<<<(unsigned)pb_ceil_div(m, MH_THREADS), MH_THREADS, 0, s>>>(p, hd);
    PB_LAUNCH_CHECK();
    return PB_OK;
}
