// mlp_update.cu -- the whole minibatch forward + PPO loss + backward of models.Default in ONE persistent
// tcgen05 kernel: the observations are read from HBM once, `hidden` / `dPre` never leave the SM.
//
// Replaces, per minibatch of clean_pufferl.train (the reference's clean_pufferl.py:186-244; policy = its
// pufferlib/models.py:12-62 with 128 input features, 128 hidden units, <= 7 actions), the chain
//     hidden = relu(x W_enc^T + b_enc)            (cuBLAS GEMM, writes 268 MB at M = 524288)
//     out    = hidden W_heads^T + b_heads         (cuBLAS GEMM, reads hidden)
//     pb_ppo_loss(out) -> dOut, statistics        (csrc/ppo_loss.cu)
//     pb_mlp_tail_backward(dOut, hidden) -> dPre, dW_heads, db_enc, db_heads      (csrc/mlp_tail.cu, reads hidden, writes dPre)
//     dW_enc = dPre^T x                           (split-K cuBLAS GEMM, reads dPre and x)
// which streams `hidden` / `dPre` through HBM five times (1.9 GB, ~350 us per minibatch).  Here the algorithmic traffic is
// x once (268 MB) + 28 B of per-row scalars (ncu: 287 MB of DRAM traffic per launch).
//
// k_mlp_update_xt (DESIGN.md 3b): warp 0 TMA producer, warp 1 single-thread tcgen05.mma issue + TMEM allocation, warps
// 2..17 epilogue.  Every x tile is loaded ONCE, K-major SWIZZLE_128B, and feeds three tensor-core products:
//     h[row][hid]       = x . W_enc^T       SS MMA, two accumulator stages in tensor memory
//     x^T[feat][row]    = I . x^T           SS MMA: A = an 8 KB "sliding identity" (no-swizzle K-major), B = the same x tile
//     dW^T[feat][hid]  += x^T . dPre        TS MMA: A = that accumulator (lanes = feat, columns = rows), B = dPre written by the
//                                           epilogue as K-major SWIZZLE_128B blocks [128 hid][32 rows] (one per row quadrant)
// The dW product contracts over rows, so x has to enter it transposed.  The tensor core takes transposed (MN-major) 32-bit
// operands from shared memory only in the SWIZZLE_128B_BASE32B layout, which would mean a second load of every tile in a
// second layout.  Instead the second product writes x^T into tensor memory, where a TS MMA reads it as its A operand.  It
// is exact (every product is with 1.0 or 0.0) and runs on a tensor pipe with slack (validated on hardware by
// tests/experimental/check_umma_transpose.py).  The identity is one 8x8 block at core matrix 15 of a 32-matrix strip of
// zeros; MMA k starts (15 - k) core matrices into the strip, so row group k of A sees the identity and every other row
// group zeros: one 8 KB buffer serves all 16 K-steps.  The shared memory a second x tile would take holds a whole tile of
// dPre instead, so the epilogue never waits for the tensor core inside a tile, and there is room for 16 epilogue warps
// (4 per scheduler: row quadrant q x column quarter c) that do all per-element products on mma.sync fragments.
// TMEM: [0,256) two forward accumulators, [256,384) x^T, [384,512) dW^T.  The dW_enc^T accumulator lives across all
// tiles of a CTA; per-CTA partials go to a workspace and k_update_reduce sums them deterministically into the flat
// gradient buffer [dW_enc (hid x feat) | dW_heads (8 x hid) | db_enc | db_heads] of clean_pufferl._DefaultMLPUpdate,
// leaving per-block sums of squares for pb_clip_adam_parts.
//
// Descriptor encodings were validated on hardware with csrc/experimental/umma_probe.cu (tests/experimental/
// check_umma_probe.py, check_umma_transpose.py).  Every mbarrier wait is bounded (tma.cuh: __trap instead of a hang).
#include <cuda.h>
#include <stdlib.h>

#include "pb_common.cuh"
#include "tma.cuh"

namespace {

constexpr int TILE_M = 128, HID = 128, FEAT = 128, NO = 8;
constexpr int KBLK = 32;                               // floats per 128-byte swizzle row
constexpr int KBLK_BYTES = TILE_M * KBLK * 4;          // 16 KiB: one [128 rows][32 floats] box
constexpr int TILE_BYTES = 4 * KBLK_BYTES;             // 64 KiB
constexpr int TMEM_COLS = 512;
constexpr int TAIL = NO * HID + HID + NO;              // dW_heads | db_enc | db_heads

struct FusedParams {
    const int64_t* actions;
    const float* old_logprobs;
    const float* adv;
    const float* returns;      // nullable: returns = advantages (raw) + old_values (clean_pufferl.py:476-481)
    const float* old_values;
    const float* adv_norm;     // nullable: (mean, 1 / (std + 1e-8)) of this minibatch's raw advantages (:211-213)
    int64_t row_slab_stride;   // per-row arrays: slab s starts at element s * row_slab_stride (slab_rows: slab-major)
    int64_t m;                 // rows of the minibatch (all slabs): the 1/M of the loss means
    int64_t slab_rows;         // R
    int64_t slab_stride_rows;  // distance between slab starts, in rows of the x tensor map
    int tiles_per_slab, n_tiles;
    int n_act;
    float clip, vclip, vf_coef, ent_coef;
    int clip_vloss;
    float* part_dw;            // [grid][FEAT][HID]
    float* part_tail;          // [grid][TAIL]
    double* stats;             // [8]
    float* dbg_hidden;         // nullable [m][128]
    float* dbg_dpre;           // nullable [m][128]
    float* dbg_dout;           // nullable [m][8]
    const float* w_heads;      // [8][128], b_enc [128], b_heads [8] in global memory
    const float* b_enc;
    const float* b_heads;
    long long* dbg_clk;        // profiling only: [grid][18 warps][4 tiles][8 events] SM clock stamps of tiles 8..11
};

__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// K-major SWIZZLE_128B descriptor (PTX ISA tcgen05 shared-memory descriptor; cute/arch/mma_sm100_desc.hpp): start>>4 |
// LBO>>4 <<16 | SBO>>4 <<32 | version 1 <<46 | layout 2 <<61, with LBO unused (1) and SBO = 1024 B between 8-row groups.
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFF) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor: D fmt F32 (1<<4) | A TF32 (2<<7) | B TF32 (2<<10) | both K-major (bits 15, 16 clear) | N>>3 <<17 |
// M>>4 <<24.  Used by all three products (M = N = 128).
constexpr uint32_t IDESC_FWD = (1u << 4) | (2u << 7) | (2u << 10) | ((HID >> 3) << 17) | ((TILE_M >> 4) << 24);

__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
    asm volatile(   // A operand from tensor memory: lanes = rows (M), columns = K
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(b_desc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&r)[32]) {
    uint32_t u[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
          "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15]), "=r"(u[16]),
          "=r"(u[17]), "=r"(u[18]), "=r"(u[19]), "=r"(u[20]), "=r"(u[21]), "=r"(u[22]), "=r"(u[23]), "=r"(u[24]),
          "=r"(u[25]), "=r"(u[26]), "=r"(u[27]), "=r"(u[28]), "=r"(u[29]), "=r"(u[30]), "=r"(u[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) r[i] = __uint_as_float(u[i]);
}

__device__ __forceinline__ uint32_t to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}

// The row math of k_ppo_loss (csrc/ppo_loss.cu, the statement of the math; clean_pufferl.py:202-238 +
// frameworks/cleanrl.py:25-47) with FOUR lanes per row: lane `sub` (0..3) of the row owns outputs sub and sub + 4 (logits
// below n_act, the value at index n_act); row-wide maxima / sums go through width-4 shuffles.  Every lane of the warp must
// call it (shuffles).  Returns dOut of the two owned outputs (already scaled by 1/M) and the six per-row statistics.
struct RowStats { float pg, v, ent, okl, kl, clipped; };
__device__ __forceinline__ RowStats ppo_row_sub(float z_lo, float z_hi, int sub, int lane, const FusedParams& p, int act,
                                                float old_lp, float adv, float ret, float old_v, float& g_lo, float& g_hi) {
    const unsigned full = 0xffffffffu;
    const int n = p.n_act;
    const bool lo_ok = sub < n, hi_ok = sub + 4 < n;
    float mx = fmaxf(lo_ok ? z_lo : -INFINITY, hi_ok ? z_hi : -INFINITY);
    mx = fmaxf(mx, __shfl_xor_sync(full, mx, 1));
    mx = fmaxf(mx, __shfl_xor_sync(full, mx, 2));
    float sum = (lo_ok ? expf(z_lo - mx) : 0.f) + (hi_ok ? expf(z_hi - mx) : 0.f);
    sum += __shfl_xor_sync(full, sum, 1);
    sum += __shfl_xor_sync(full, sum, 2);
    const float lse = mx + logf(sum);
    const float nl_lo = z_lo - lse, nl_hi = z_hi - lse;
    const float pk_lo = lo_ok ? expf(nl_lo) : 0.f, pk_hi = hi_ok ? expf(nl_hi) : 0.f;
    float ent = -(lo_ok ? pk_lo * nl_lo : 0.f) - (hi_ok ? pk_hi * nl_hi : 0.f);
    ent += __shfl_xor_sync(full, ent, 1);
    ent += __shfl_xor_sync(full, ent, 2);
    const int a = act < 0 ? 0 : (act >= n ? n - 1 : act);
    const int base = lane & ~3;
    const float nl_a = __shfl_sync(full, (a >> 2) ? nl_hi : nl_lo, base | (a & 3));
    const float v_new = __shfl_sync(full, (n >> 2) ? z_hi : z_lo, base | (n & 3));
    const float logratio = nl_a - old_lp;
    const float ratio = expf(logratio);
    const float pg1 = -adv * ratio;
    const float rc = fminf(fmaxf(ratio, 1.f - p.clip), 1.f + p.clip);
    const float pg2 = -adv * rc;
    const float pg = fmaxf(pg1, pg2);
    const float in_range = (ratio >= 1.f - p.clip && ratio <= 1.f + p.clip) ? 1.f : 0.f;
    float g_ratio;
    if (pg1 > pg2) g_ratio = -adv;
    else if (pg1 < pg2) g_ratio = -adv * in_range;
    else g_ratio = 0.5f * (-adv) + 0.5f * (-adv * in_range);
    const float inv_m = 1.0f / (float)p.m;
    const float g_nlp = g_ratio * ratio * inv_m;
    const float dv = v_new - ret;
    float vl, g_v;
    if (p.clip_vloss) {
        const float d = v_new - old_v;
        const float dc = fminf(fmaxf(d, -p.vclip), p.vclip);
        const float vc = old_v + dc;
        const float vu = dv * dv, vcl = (vc - ret) * (vc - ret);
        vl = fmaxf(vu, vcl);
        const float v_in = (d >= -p.vclip && d <= p.vclip) ? 1.f : 0.f;
        const float gu = 2.f * dv, gc = 2.f * (vc - ret) * v_in;
        g_v = vu > vcl ? gu : (vu < vcl ? gc : 0.5f * (gu + gc));
    } else {
        vl = dv * dv;
        g_v = 2.f * dv;
    }
    const float gv_out = 0.5f * p.vf_coef * g_v * inv_m;
    const float g_ent = p.ent_coef * inv_m;
    g_lo = lo_ok ? g_nlp * ((sub == a ? 1.f : 0.f) - pk_lo) + g_ent * pk_lo * (nl_lo + ent) : 0.f;
    g_hi = hi_ok ? g_nlp * ((sub + 4 == a ? 1.f : 0.f) - pk_hi) + g_ent * pk_hi * (nl_hi + ent) : 0.f;
    if (sub == n) g_lo = gv_out;
    if (sub + 4 == n) g_hi = gv_out;
    RowStats s;
    s.pg = pg; s.v = vl; s.ent = ent; s.okl = -logratio; s.kl = (ratio - 1.f) - logratio;
    s.clipped = fabsf(ratio - 1.f) > p.clip ? 1.f : 0.f;
    return s;
}

// Shared memory (byte offsets) and tensor memory (columns) of k_mlp_update_xt; the header comment describes the products.
constexpr int X2_THREADS = 576;                          // warp 0 TMA, warp 1 MMA, warps 2..17 epilogue
constexpr int X2_W = 0, X2_XK = TILE_BYTES, X2_G = 2 * TILE_BYTES;     // W_enc | x tile | 4 dPre blocks of 16 KiB
constexpr int X2_XCH = 3 * TILE_BYTES;                   // [4 q][4 c][32 rows][10]: partial head sums (8 used; 10 = bank spread)
constexpr int X2_XCH_ROW = 10, X2_XCH_Q = 4 * 32 * X2_XCH_ROW;
constexpr int X2_ID = X2_XCH + 4 * X2_XCH_Q * 4;         // sliding identity: 2 strips of 32 core matrices
constexpr int X2_DO = X2_ID + 8192;                      // [4 q][32 rows][9]: dOut of the tile (8 used)
constexpr int X2_DO_ROW = 9, X2_DO_Q = 320;
constexpr int X2_BE = X2_DO + 4 * X2_DO_Q * 4;           // b_enc [128]
constexpr int X2_BAR = X2_BE + 512;
constexpr int X2_TOTAL = X2_BAR + 256;
constexpr int X2_TMEM_XT = 256, X2_TMEM_DW = 384;
constexpr int X2_ID_GROUP = 128, X2_ID_STRIP = 32 * X2_ID_GROUP;
static_assert(X2_TOTAL <= 232448, "shared memory budget");

// no-swizzle K-major descriptor: 8-row x 16-byte core matrices, LBO = distance between the two core matrices of a K = 8
// slice, SBO = distance between 8-row groups
__device__ __forceinline__ uint64_t desc_nosw(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
           (1ull << 46);
}

// Layout of a dPre block (K-major SWIZZLE_128B, [128 hidden units][32 rows of the quadrant]): element (hidden unit n, row l)
// sits at byte  n * 128 + (((l >> 2) ^ (n & 7)) << 4) + ((l & 3) << 2)  -- hidden unit n = MN row of 128 B, the quadrant's rows
// along K in 16-byte pieces XORed with n & 7.  The epilogue's addresses (st_row, ha_base, wb_base) are instances of it.

// mma.sync m16n8k8 TF32 with all four A registers: a0 (g, t)  a1 (g + 8, t)  a2 (g, t + 4)  a3 (g + 8, t + 4);
// b0 (k = t, n = g)  b1 (k = t + 4, n = g);  c0 c1 (g, 2t + {0,1})  c2 c3 (g + 8, 2t + {0,1})      [g = lane >> 2, t = lane & 3]
__device__ __forceinline__ void mma_tf32_full(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

template <int REGS, bool CLK>
__global__ void __maxnreg__(REGS)
k_mlp_update_xt(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w, const FusedParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + X2_BAR);
    uint64_t* w_full = bars;
    uint64_t* xk_full = bars + 1;         // x tile landed
    uint64_t* xk_empty = bars + 2;        // ... read by the forward AND the transposing MMAs
    uint64_t* h_full = bars + 3;          // [2] forward accumulator complete
    uint64_t* h_empty = bars + 5;         // [2] read by the 16 epilogue warps
    uint64_t* dp_full = bars + 7;         // [4] dPre block of row quadrant q written (4 warps)
    uint64_t* dp_empty = bars + 11;       // [4] ... consumed by its dW MMAs
    uint64_t* dw_done = bars + 15;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        mbar_init(w_full, 1);
        mbar_init(xk_full, 1);
        mbar_init(xk_empty, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&h_full[i], 1);
            mbar_init(&h_empty[i], 16);
        }
        for (int i = 0; i < 4; ++i) {
            mbar_init(&dp_full[i], 4);
            mbar_init(&dp_empty[i], 1);
        }
        mbar_init(dw_done, 1);
        mbar_fence_init();
    }
    // sliding identity: strip s (features 4s..4s+3 of a K = 8 slice) is 32 core matrices of 8 rows x 16 B, all zero except
    // number 15, whose row r holds a 1 at column r - 4s.  MMA k reads from (15 - k) core matrices in: row group k of A sees
    // the identity block, every other row group zeros.
    for (int i = threadIdx.x; i < 8192 / 16; i += X2_THREADS) reinterpret_cast<uint4*>(smem + X2_ID)[i] = make_uint4(0, 0, 0, 0);
    if (threadIdx.x < HID) reinterpret_cast<float*>(smem + X2_BE)[threadIdx.x] = p.b_enc[threadIdx.x];
    __syncthreads();
    if (threadIdx.x < 8) {
        const int r = threadIdx.x;
        *reinterpret_cast<float*>(smem + X2_ID + (r >> 2) * X2_ID_STRIP + 15 * X2_ID_GROUP + r * 16 + (r & 3) * 4) = 1.0f;
    }
    fence_proxy_async_smem();
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"((uint32_t)TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int n_my = (p.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    auto stamp = [&](int it, int ev) {
        if (CLK && p.dbg_clk && lane == 0 && it >= 8 && it < 12) p.dbg_clk[(((int64_t)blockIdx.x * 18 + warp) * 4 + (it - 8)) * 8 + ev] = clock64();
    };

    // epilogue warp (q, c): TMEM lane quadrant q (tile rows 32q..32q+31), hidden units 32c..32c+31
    float acc_wh[2][4];                  // dW_heads[head 2t + (i & 1)][32c + 16mb + 8(i >> 1) + g] (this warp's rows)
    float st[6] = {0, 0, 0, 0, 0, 0};    // per-thread statistics of <= 28 tiles: fp32 here, fp64 across threads
    float acc_be[4] = {0.f, 0.f, 0.f, 0.f};   // db_enc[32c + 8nb + (lane >> 2)], this lane's 8 rows of every tile
    float acc_bh2[2] = {0.f, 0.f};       // db_heads[lane & 3], [(lane & 3) + 4] over this lane's rows
#pragma unroll
    for (int mb = 0; mb < 2; ++mb) acc_wh[mb][0] = acc_wh[mb][1] = acc_wh[mb][2] = acc_wh[mb][3] = 0.f;

    if (warp == 0) {
        if (lane == 0) {
            mbar_expect_tx(w_full, TILE_BYTES);
            for (int kb = 0; kb < 4; ++kb) tma_load_2d(smem + X2_W + kb * KBLK_BYTES, &map_w, kb * KBLK, 0, w_full);
            for (int it = 0; it < n_my; ++it) {
                const int tile = (int)blockIdx.x + it * (int)gridDim.x;
                const int64_t row0 = (int64_t)(tile / p.tiles_per_slab) * p.slab_stride_rows +
                                     (int64_t)(tile % p.tiles_per_slab) * TILE_M;
                stamp(it, 0);
                mbar_wait(xk_empty, (uint32_t)((it & 1) ^ 1));
                stamp(it, 1);
                mbar_expect_tx(xk_full, TILE_BYTES);
                for (int kb = 0; kb < 4; ++kb) tma_load_2d(smem + X2_XK + kb * KBLK_BYTES, &map_x, kb * KBLK, (int)row0, xk_full);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t w_addr = smem_u32(smem + X2_W), xk_addr = smem_u32(smem + X2_XK);
            const uint32_t g_addr = smem_u32(smem + X2_G), id_addr = smem_u32(smem + X2_ID);
            auto forward = [&](int it) {
                const int s = it & 1, ph = (it >> 1) & 1;
                stamp(it, 0);
                mbar_wait(&h_empty[s], ph ^ 1);
                stamp(it, 1);
                mbar_wait(xk_full, (uint32_t)(it & 1));
                stamp(it, 2);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(s * HID);
#pragma unroll
                for (int kb = 0; kb < 4; ++kb)
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        umma_tf32(d_tmem, desc_kmajor(xk_addr + kb * KBLK_BYTES + k * 32),
                                  desc_kmajor(w_addr + kb * KBLK_BYTES + k * 32), IDESC_FWD, (kb | k) ? 1u : 0u);
                umma_commit(&h_full[s]);
            };
            auto transpose = [&]() {     // x^T of the tile in the x buffer (the dW MMAs of the previous tile were issued before)
#pragma unroll
                for (int kb = 0; kb < 4; ++kb)
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        umma_tf32(tmem_base + X2_TMEM_XT,
                                  desc_nosw(id_addr + (15 - (4 * kb + k)) * X2_ID_GROUP, X2_ID_STRIP, X2_ID_GROUP),
                                  desc_kmajor(xk_addr + kb * KBLK_BYTES + k * 32), IDESC_FWD, (kb | k) ? 1u : 0u);
                umma_commit(xk_empty);   // the x tile may be overwritten: the next load starts
            };
            mbar_wait(w_full, 0);
            forward(0);
            transpose();
            for (int it = 0; it < n_my; ++it) {
                if (it + 1 < n_my) forward(it + 1);
#pragma unroll 1
                for (int q = 0; q < 4; ++q) {
                    mbar_wait(&dp_full[q], (uint32_t)(it & 1));
                    stamp(it, 3 + q);
                    tc_fence_after();
#pragma unroll
                    for (int k = 0; k < 4; ++k)      // K = 8 tile rows per MMA
                        umma_tf32_ts(tmem_base + X2_TMEM_DW, tmem_base + (uint32_t)(X2_TMEM_XT + 32 * q + 8 * k),
                                     desc_kmajor(g_addr + q * KBLK_BYTES + k * 32), IDESC_FWD, (it | q | k) ? 1u : 0u);
                    umma_commit(&dp_empty[q]);
                }
                if (it + 1 < n_my) transpose();
                stamp(it, 7);
            }
            umma_commit(dw_done);
        }
    } else {
        // ================= epilogue: all per-element products on the warp-level tensor core path (mma.sync, TF32 operands
        // = the raw fp32 bits, low mantissa bits ignored like the UMMA products; fp32 accumulation -- the precision class of
        // torch.set_float32_matmul_precision('high'), clean_pufferl.py:22).  Thread = row only for the TMEM read and the ReLU;
        // everything else works on mma fragments of the warp's [32 rows][32 hidden units] block staged in its part of the
        // dPre block.  The m / n / k indices of the three products are PERMUTED so that every fragment a lane needs is a run
        // of 4 or 8 consecutive rows of one hidden unit (one or two 16-byte pieces of the K-major block: LDS.128 / STS.128),
        // and so that the relu(h) fragments of the dW_heads product sit exactly where the g^T accumulators need their mask.
        const int q = warp & 3, c = (warp - 2) >> 2;
        const int g = lane >> 2, t = lane & 3;
        uint8_t* mine = smem + X2_G + q * KBLK_BYTES + 32 * c * 128;   // hidden units 32c..32c+31 x the quadrant's 32 rows
        float* xch = reinterpret_cast<float*>(smem + X2_XCH) + q * X2_XCH_Q;              // [4 c][32 rows][10]
        float* dos = reinterpret_cast<float*>(smem + X2_DO) + q * X2_DO_Q;                // [32 rows][9]
        const float4* be4 = reinterpret_cast<const float4*>(smem + X2_BE) + 8 * c;
        // W_heads fragments of this column quarter (TF32), resident in registers:
        //   heads   out[row][a] = sum_j rh[row][j] W[a][j]:  B[k][n = a], k = t + 4h <-> hidden unit 8kb + 2t + h
        //   g^T     g[j][row]   = sum_a W[a][j] dO[row][a]:  A[m][k = a], m = g + 8h <-> hidden unit 16mb + 8h + g
        uint32_t hb[4][2], ga[2][4];
#pragma unroll
        for (int kb = 0; kb < 4; ++kb) {
            hb[kb][0] = to_tf32(p.w_heads[g * HID + 32 * c + 8 * kb + 2 * t]);
            hb[kb][1] = to_tf32(p.w_heads[g * HID + 32 * c + 8 * kb + 2 * t + 1]);
        }
#pragma unroll
        for (int mb = 0; mb < 2; ++mb) {
            ga[mb][0] = to_tf32(p.w_heads[t * HID + 32 * c + 16 * mb + g]);
            ga[mb][1] = to_tf32(p.w_heads[t * HID + 32 * c + 16 * mb + g + 8]);
            ga[mb][2] = to_tf32(p.w_heads[(t + 4) * HID + 32 * c + 16 * mb + g]);
            ga[mb][3] = to_tf32(p.w_heads[(t + 4) * HID + 32 * c + 16 * mb + g + 8]);
        }
        // addresses inside the warp's part of the dPre block (see g_off), hoisted out of the tile loop
        uint8_t* const st_row = mine + ((lane & 3) << 2);       // thread = row: element (hidden unit k, row lane) at k * 128 + piece ((lane >> 2) ^ (k & 7))
        uint8_t* ha_base[2];                                    // heads A: hidden unit 8kb + 2t + h, rows 4g..4g+3 (one piece)
#pragma unroll
        for (int h = 0; h < 2; ++h) ha_base[h] = mine + (2 * t + h) * 128 + ((g ^ (2 * t + h)) << 4);
        uint8_t* wb_base[2];                                    // dW_heads B / g^T C: hidden unit 8nb + g, rows 8t..8t+3 | 8t+4..8t+7
#pragma unroll
        for (int e = 0; e < 2; ++e) wb_base[e] = mine + g * 128 + ((((2 * t + e) ^ g)) << 4);

        // the loss: warp c evaluates rows 8c..8c+7 of the quadrant, four lanes per row (ppo_row_sub)
        const int lr = 8 * c + (lane >> 2), sub = lane & 3;
        const float bh_lo = p.b_heads[sub], bh_hi = p.b_heads[sub + 4];
        // per-row scalars of the loss rows, loaded ONE TILE AHEAD with volatile loads issued right after the second barrier
        // (plain loads get sunk to their first use by the compiler, which puts their HBM latency back on the critical path)
        struct RowIn { int act; float old_lp, adv, ret, old_v; bool valid; };
        const float adv_mean = p.adv_norm ? p.adv_norm[0] : 0.f, adv_rstd = p.adv_norm ? p.adv_norm[1] : 1.f;
        const bool need_old_v = p.clip_vloss || !p.returns;
        auto ldg_f32 = [](const float* ptr) { float v; asm volatile("ld.global.f32 %0, [%1];" : "=f"(v) : "l"(ptr)); return v; };
        auto ldg_s64 = [](const int64_t* ptr) { long long v; asm volatile("ld.global.s64 %0, [%1];" : "=l"(v) : "l"(ptr)); return v; };
        auto load_row = [&](int it) {
            RowIn r;
            r.act = 0; r.old_lp = 0.f; r.adv = 0.f; r.ret = 0.f; r.old_v = 0.f; r.valid = false;
            if (it >= n_my) return r;
            const int tile = (int)blockIdx.x + it * (int)gridDim.x;
            const int slab = tile / p.tiles_per_slab, tis = tile - slab * p.tiles_per_slab;
            const int64_t lrow = (int64_t)tis * TILE_M + 32 * q + lr;
            r.valid = lrow < p.slab_rows;
            const int64_t ri = (int64_t)slab * p.row_slab_stride + lrow;     // position in the per-row arrays
            if (r.valid) {
                r.act = (int)ldg_s64(p.actions + ri);
                r.old_lp = ldg_f32(p.old_logprobs + ri);
                r.adv = ldg_f32(p.adv + ri);
                if (need_old_v) r.old_v = ldg_f32(p.old_values + ri);
                if (p.returns) r.ret = ldg_f32(p.returns + ri);
            }
            return r;
        };
        RowIn row = load_row(0);
        for (int it = 0; it < n_my; ++it) {
            const int s = it & 1, ph = (it >> 1) & 1;
            // debug dumps only: slab-major position of tile row 0 of this quadrant, rows of the slab left in the tile
            int64_t dbg_row0 = 0, rows_left = 32;
            if (p.dbg_hidden || p.dbg_dout || p.dbg_dpre) {
                const int tile = (int)blockIdx.x + it * (int)gridDim.x;
                dbg_row0 = (int64_t)(tile / p.tiles_per_slab) * p.slab_rows + (int64_t)(tile % p.tiles_per_slab) * TILE_M + 32 * q;
                rows_left = p.slab_rows - ((int64_t)(tile % p.tiles_per_slab) * TILE_M + 32 * q);
            }

            // ---- 1. h -> relu(h + b_enc) into the warp's part of the dPre block (K-major: [hidden unit][row])
            stamp(it, 0);
            mbar_wait(&h_full[s], ph);
            stamp(it, 1);
            tc_fence_after();
            {
                float v[32];
                tmem_ld32(tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(s * HID + 32 * c), v);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&h_empty[s]);                      // the accumulator stage is free already
                mbar_wait(&dp_empty[q], (uint32_t)((it & 1) ^ 1));            // the dW MMAs of the previous tile have read the block
                stamp(it, 2);
#pragma unroll
                for (int k4 = 0; k4 < 8; ++k4) {
                    const float4 b = be4[k4];
                    v[4 * k4] = fmaxf(v[4 * k4] + b.x, 0.f);
                    v[4 * k4 + 1] = fmaxf(v[4 * k4 + 1] + b.y, 0.f);
                    v[4 * k4 + 2] = fmaxf(v[4 * k4 + 2] + b.z, 0.f);
                    v[4 * k4 + 3] = fmaxf(v[4 * k4 + 3] + b.w, 0.f);
                }
#pragma unroll
                for (int k = 0; k < 32; ++k) *reinterpret_cast<float*>(st_row + ((((lane >> 2) ^ (k & 7))) << 4) + k * 128) = v[k];
                if (p.dbg_hidden && lane < rows_left) {
#pragma unroll
                    for (int k = 0; k < 32; k += 4)
                        *reinterpret_cast<float4*>(p.dbg_hidden + (dbg_row0 + lane) * HID + 32 * c + k) = make_float4(v[k], v[k + 1], v[k + 2], v[k + 3]);
                }
            }
            __syncwarp();

            // ---- 2. this quarter's share of the head products.  m = g + 8h of block mb <-> row 4g + 2mb + h
            {
                float hp[2][4];
#pragma unroll
                for (int mb = 0; mb < 2; ++mb) hp[mb][0] = hp[mb][1] = hp[mb][2] = hp[mb][3] = 0.f;
#pragma unroll
                for (int kb = 0; kb < 4; ++kb) {
                    const float4 lo = *reinterpret_cast<const float4*>(ha_base[0] + kb * 1024);   // hidden unit 8kb + 2t
                    const float4 hi = *reinterpret_cast<const float4*>(ha_base[1] + kb * 1024);   // hidden unit 8kb + 2t + 1
                    const uint32_t a0[4] = {__float_as_uint(lo.x), __float_as_uint(lo.y), __float_as_uint(hi.x), __float_as_uint(hi.y)};
                    const uint32_t a1[4] = {__float_as_uint(lo.z), __float_as_uint(lo.w), __float_as_uint(hi.z), __float_as_uint(hi.w)};
                    mma_tf32_full(hp[0], a0, hb[kb][0], hb[kb][1]);
                    mma_tf32_full(hp[1], a1, hb[kb][0], hb[kb][1]);
                }
#pragma unroll
                for (int mb = 0; mb < 2; ++mb) {
                    *reinterpret_cast<float2*>(xch + (c * 32 + 4 * g + 2 * mb) * X2_XCH_ROW + 2 * t) = make_float2(hp[mb][0], hp[mb][1]);
                    *reinterpret_cast<float2*>(xch + (c * 32 + 4 * g + 2 * mb + 1) * X2_XCH_ROW + 2 * t) = make_float2(hp[mb][2], hp[mb][3]);
                }
            }
            stamp(it, 3);
            asm volatile("bar.sync %0, 128;" ::"r"(1 + q) : "memory");
            stamp(it, 4);

            // ---- 3. the loss row math on the summed head outputs -> dOut tile of the quadrant
            {
                float z_lo = bh_lo, z_hi = bh_hi;
#pragma unroll
                for (int cq = 0; cq < 4; ++cq) {                                    // fixed order
                    z_lo += xch[(cq * 32 + lr) * X2_XCH_ROW + sub];
                    z_hi += xch[(cq * 32 + lr) * X2_XCH_ROW + sub + 4];
                }
                const float ret = p.returns ? row.ret : row.adv + row.old_v;       // returns = raw advantages + old values (:476-481)
                const float adv = (row.adv - adv_mean) * adv_rstd;
                float g_lo, g_hi;
                const RowStats rs = ppo_row_sub(z_lo, z_hi, sub, lane, p, row.act, row.old_lp, adv, ret, row.old_v, g_lo, g_hi);
                if (!row.valid) g_lo = g_hi = 0.f;
                if (row.valid && sub == 0) {
                    st[0] += rs.pg; st[1] += rs.v; st[2] += rs.ent; st[3] += rs.okl; st[4] += rs.kl; st[5] += rs.clipped;
                }
                acc_bh2[0] += g_lo;
                acc_bh2[1] += g_hi;
                dos[lr * X2_DO_ROW + sub] = g_lo;
                dos[lr * X2_DO_ROW + sub + 4] = g_hi;
                if (p.dbg_dout && row.valid) {
                    p.dbg_dout[(dbg_row0 + lr) * 8 + sub] = g_lo;
                    p.dbg_dout[(dbg_row0 + lr) * 8 + sub + 4] = g_hi;
                }
            }
            stamp(it, 5);
            asm volatile("bar.sync %0, 128;" ::"r"(1 + q) : "memory");
            stamp(it, 6);

            // ---- 4. per 16 hidden units (block mb):
            //         g^T[hidden unit][row] = W^T . dO^T        n = 2t' + j of block nb' <-> row 8t' + 2nb' + j
            //         dW_heads^T += rh^T . dO                   k = t + 4j of block ks  <-> row 8t + 2ks + j,  m = g + 8h <-> unit 16mb + 8h + g
            //      the rh fragments of the second product sit exactly where the first one's accumulators need their mask, and
            //      dPre goes back to the same places: no lane touches another lane's elements in this step
            {
                uint32_t gb[4][2], bfr[4][2];
#pragma unroll
                for (int nb = 0; nb < 4; ++nb) {                 // dO as B[k = head][n = row] (g^T) and as B[k = row][n = head] (dW_heads^T)
                    const int rn = 8 * (g >> 1) + 2 * nb + (g & 1);
                    gb[nb][0] = __float_as_uint(dos[rn * X2_DO_ROW + t]);
                    gb[nb][1] = __float_as_uint(dos[rn * X2_DO_ROW + t + 4]);
                    bfr[nb][0] = __float_as_uint(dos[(8 * t + 2 * nb) * X2_DO_ROW + g]);
                    bfr[nb][1] = __float_as_uint(dos[(8 * t + 2 * nb + 1) * X2_DO_ROW + g]);
                }
#pragma unroll
                for (int mb = 0; mb < 2; ++mb) {
                    float gt[4][4];                              // [nb'][2h + j]: hidden unit 16mb + 8h + g, row 8t + 2nb' + j
#pragma unroll
                    for (int nb = 0; nb < 4; ++nb) {
                        gt[nb][0] = gt[nb][1] = gt[nb][2] = gt[nb][3] = 0.f;
                        mma_tf32_full(gt[nb], ga[mb], gb[nb][0], gb[nb][1]);
                    }
                    float4 lo[2], hi[2];
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        lo[h] = *reinterpret_cast<const float4*>(wb_base[0] + (2 * mb + h) * 1024);   // rows 8t .. 8t+3
                        hi[h] = *reinterpret_cast<const float4*>(wb_base[1] + (2 * mb + h) * 1024);   // rows 8t+4 .. 8t+7
                    }
                    // A[m = g + 8h][k = t + 4j] = rh[row 8t + 2ks + j][hidden unit 16mb + 8h + g]
                    const uint32_t a0[4] = {__float_as_uint(lo[0].x), __float_as_uint(lo[1].x), __float_as_uint(lo[0].y), __float_as_uint(lo[1].y)};
                    const uint32_t a1[4] = {__float_as_uint(lo[0].z), __float_as_uint(lo[1].z), __float_as_uint(lo[0].w), __float_as_uint(lo[1].w)};
                    const uint32_t a2[4] = {__float_as_uint(hi[0].x), __float_as_uint(hi[1].x), __float_as_uint(hi[0].y), __float_as_uint(hi[1].y)};
                    const uint32_t a3[4] = {__float_as_uint(hi[0].z), __float_as_uint(hi[1].z), __float_as_uint(hi[0].w), __float_as_uint(hi[1].w)};
                    mma_tf32_full(acc_wh[mb], a0, bfr[0][0], bfr[0][1]);
                    mma_tf32_full(acc_wh[mb], a1, bfr[1][0], bfr[1][1]);
                    mma_tf32_full(acc_wh[mb], a2, bfr[2][0], bfr[2][1]);
                    mma_tf32_full(acc_wh[mb], a3, bfr[3][0], bfr[3][1]);
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const float4 d0 = make_float4(lo[h].x > 0.f ? gt[0][2 * h] : 0.f, lo[h].y > 0.f ? gt[0][2 * h + 1] : 0.f,
                                                      lo[h].z > 0.f ? gt[1][2 * h] : 0.f, lo[h].w > 0.f ? gt[1][2 * h + 1] : 0.f);
                        const float4 d1 = make_float4(hi[h].x > 0.f ? gt[2][2 * h] : 0.f, hi[h].y > 0.f ? gt[2][2 * h + 1] : 0.f,
                                                      hi[h].z > 0.f ? gt[3][2 * h] : 0.f, hi[h].w > 0.f ? gt[3][2 * h + 1] : 0.f);
                        *reinterpret_cast<float4*>(wb_base[0] + (2 * mb + h) * 1024) = d0;
                        *reinterpret_cast<float4*>(wb_base[1] + (2 * mb + h) * 1024) = d1;
                        acc_be[2 * mb + h] += ((d0.x + d0.y) + (d0.z + d0.w)) + ((d1.x + d1.y) + (d1.z + d1.w));
                        if (p.dbg_dpre) {
                            const float dv[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
#pragma unroll
                            for (int r8 = 0; r8 < 8; ++r8)
                                if (8 * t + r8 < rows_left) p.dbg_dpre[(dbg_row0 + 8 * t + r8) * HID + 32 * c + 16 * mb + 8 * h + g] = dv[r8];
                        }
                    }
                }
            }
            row = load_row(it + 1);          // (volatile loads: issued here, where few registers are live)
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&dp_full[q]);
            stamp(it, 7);
        }
        // ---- the dW^T accumulator: TMEM lane = feature, column = hidden unit
        mbar_wait(dw_done, 0);
        tc_fence_after();
        {
            float v[32];
            float* pd = p.part_dw + ((int64_t)blockIdx.x * FEAT + 32 * q + lane) * HID + 32 * c;
            tmem_ld32(tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(X2_TMEM_DW + 32 * c), v);
#pragma unroll
            for (int k = 0; k < 32; k += 4) *reinterpret_cast<float4*>(pd + k) = make_float4(v[k], v[k + 1], v[k + 2], v[k + 3]);
        }
#pragma unroll
        for (int k = 0; k < 6; ++k) {          // statistics: the sub == 0 lanes hold this warp's rows
            double x = (double)st[k];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) x += __shfl_xor_sync(0xffffffffu, x, off);
            if (lane == 0) atomicAdd(p.stats + k, x);
        }
        // db_enc: the four lanes of a hidden unit (t = 0..3) hold its 4 x 8 rows; db_heads: the eight lanes with the same sub
#pragma unroll
        for (int nb = 0; nb < 4; ++nb) {
            acc_be[nb] += __shfl_xor_sync(0xffffffffu, acc_be[nb], 1);
            acc_be[nb] += __shfl_xor_sync(0xffffffffu, acc_be[nb], 2);
        }
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int off = 4; off < 32; off <<= 1) acc_bh2[j] += __shfl_xor_sync(0xffffffffu, acc_bh2[j], off);
    }

    // ================= CTA reduction of the small gradients =================
    tc_fence_before();
    __syncthreads();                           // every role is done: all MMAs retired, the x tile is scratch now
    if (warp >= 2) {
        const int q = warp & 3, c = (warp - 2) >> 2, g = lane >> 2, t = lane & 3;
        float* red = reinterpret_cast<float*>(smem + X2_XK);
        float* mine_r = red + q * TAIL;
#pragma unroll
        for (int nb = 0; nb < 4; ++nb) {
            mine_r[(2 * t) * HID + 32 * c + 8 * nb + g] = acc_wh[nb >> 1][2 * (nb & 1)];
            mine_r[(2 * t + 1) * HID + 32 * c + 8 * nb + g] = acc_wh[nb >> 1][2 * (nb & 1) + 1];
            if (t == 0) mine_r[NO * HID + 32 * c + 8 * nb + g] = acc_be[nb];
        }
        if (lane < 4) {                        // db_heads partial of this warp's rows: [16 warps][8] behind the four TAIL rows
            red[4 * TAIL + (warp - 2) * NO + lane] = acc_bh2[0];
            red[4 * TAIL + (warp - 2) * NO + lane + 4] = acc_bh2[1];
        }
    }
    __syncthreads();
    {
        const float* red = reinterpret_cast<const float*>(smem + X2_XK);   // [4 quadrants][TAIL] | [16 warps][8] db_heads partials
        float* pt = p.part_tail + (int64_t)blockIdx.x * TAIL;
        for (int j = threadIdx.x; j < TAIL; j += X2_THREADS) {
            float v;
            if (j < NO * HID + HID) {
                v = red[j] + red[TAIL + j] + red[2 * TAIL + j] + red[3 * TAIL + j];
            } else {
                v = 0.f;
                for (int w = 0; w < 16; ++w) v += red[4 * TAIL + w * NO + (j - NO * HID - HID)];
            }
            pt[j] = v;
        }
    }
    if (warp == 1)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS)
                     : "memory");
}

// Deterministic sum of the per-CTA partials into the flat gradient buffer:
//   gflat = [ dW_enc[hid][feat] (transposed from the partials' [feat][hid]) | dW_heads 8 x hid | db_enc | db_heads ]
// Block = 64 outputs x 4 partial groups; consecutive threads read consecutive partial elements (coalesced).
__global__ void __launch_bounds__(256) k_update_reduce(const float* __restrict__ part_dw, const float* __restrict__ part_tail,
                                                       int n_parts, float* __restrict__ gflat, double* __restrict__ sumsq_part) {
    __shared__ float sh[4][64];
    __shared__ double sq[2];
    const int e = blockIdx.x * 64 + (threadIdx.x & 63), grp = threadIdx.x >> 6;
    constexpr int NDW = FEAT * HID;
    float s = 0.f;
    if (e < NDW + TAIL) {
        const float* src = e < NDW ? part_dw + e : part_tail + (e - NDW);
        const int64_t stride = e < NDW ? NDW : TAIL;
#pragma unroll 4
        for (int pidx = grp; pidx < n_parts; pidx += 4) s += src[(int64_t)pidx * stride];
    }
    sh[grp][threadIdx.x & 63] = s;
    __syncthreads();
    if (grp == 0) {                           // warps 0 and 1
        float tot = 0.f;
        if (e < NDW + TAIL) {
            tot = sh[0][threadIdx.x] + sh[1][threadIdx.x] + sh[2][threadIdx.x] + sh[3][threadIdx.x];
            if (e < NDW) gflat[(e % HID) * FEAT + e / HID] = tot;      // partial element (f, j) -> dW_enc[j][f]
            else gflat[e] = tot;
        }
        // sum of squares of this block's 64 gradient elements: the global-norm pass of the optimizer step becomes a sum of
        // gridDim.x doubles (pb_clip_adam_parts), in a fixed order
        double d = (double)tot * (double)tot;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) d += __shfl_xor_sync(0xffffffffu, d, off);
        if ((threadIdx.x & 31) == 0) sq[threadIdx.x >> 5] = d;
    }
    __syncthreads();
    if (threadIdx.x == 0) sumsq_part[blockIdx.x] = sq[0] + sq[1];
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int make_map2(EncodeTiledFn fn, CUtensorMap* map, const float* base, int64_t rows, int64_t row_stride_floats) {
    const cuuint64_t dims[2] = {(cuuint64_t)FEAT, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)row_stride_floats * 4};
    const cuuint32_t box[2] = {(cuuint32_t)KBLK, (cuuint32_t)TILE_M};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    PB_REQUIRE(r == CUDA_SUCCESS, PB_ERR_CUDA, "cuTensorMapEncodeTiled failed: %d", (int)r);
    return PB_OK;
}

int num_sms() { return pb_num_sms(); }

long long* g_dbg_clk = nullptr;

}  // namespace

extern "C" int pb_mlp_update_debug_clock(long long* buf) {     // profiling hook: see FusedParams::dbg_clk; nullptr = off
    g_dbg_clk = buf;
    return PB_OK;
}

constexpr int REDUCE_BLOCKS = (FEAT * HID + TAIL + 63) / 64;

// workspace: per-CTA partials [SMs][FEAT * HID + TAIL] floats | REDUCE_BLOCKS doubles (sums of squares of the gradient)
extern "C" size_t pb_mlp_update_sumsq_offset(void) {
    return (((size_t)num_sms() * (FEAT * HID + TAIL) * sizeof(float)) + 15) & ~(size_t)15;
}
extern "C" int32_t pb_mlp_update_sumsq_parts(void) { return REDUCE_BLOCKS; }
extern "C" size_t pb_mlp_update_workspace_bytes(void) {
    return pb_mlp_update_sumsq_offset() + REDUCE_BLOCKS * sizeof(double);
}

extern "C" int pb_mlp_update_fused(const float* x, int64_t ldx, int64_t slab_rows, int64_t slab_stride_rows, int32_t n_slabs,
                                   const float* w_enc, const float* b_enc, const float* w_heads, const float* b_heads,
                                   const int64_t* actions, const float* old_logprobs, const float* advantages,
                                   const float* returns, const float* old_values, const float* adv_norm,
                                   int64_t row_slab_stride, int32_t n_act, float clip_coef,
                                   int32_t clip_vloss, float vf_clip_coef, float vf_coef, float ent_coef, float* grad_flat,
                                   double* stats8, void* workspace, size_t workspace_bytes, float* dpre_out,
                                   float* dbg_hidden, float* dbg_dpre, float* dbg_dout, void* stream) {
    PB_REQUIRE(!dpre_out, PB_ERR_UNSUPPORTED,
               "pb_mlp_update_fused: dpre_out must be NULL (dW_enc is always formed inside the kernel; dPre is not written out)");
    PB_REQUIRE(x && w_enc && b_enc && w_heads && b_heads && actions && old_logprobs && advantages && grad_flat && stats8 &&
                   workspace && (returns || old_values),
               PB_ERR_INVALID, "pb_mlp_update_fused: null pointer");
    PB_REQUIRE(n_slabs == 1 || row_slab_stride >= slab_rows, PB_ERR_INVALID, "pb_mlp_update_fused: row slabs overlap");
    PB_REQUIRE(slab_rows >= 1 && n_slabs >= 1 && n_act >= 1 && n_act <= 7 && (!clip_vloss || old_values), PB_ERR_INVALID,
               "pb_mlp_update_fused: bad sizes (slab_rows %lld, n_slabs %d, n_act %d)", (long long)slab_rows, n_slabs, n_act);
    PB_REQUIRE(ldx >= FEAT && ldx % 4 == 0 && ((uintptr_t)x & 15) == 0 && ((uintptr_t)w_enc & 15) == 0, PB_ERR_INVALID,
               "pb_mlp_update_fused: x / w_enc must be 16-byte aligned, ldx a multiple of 4 floats");
    PB_REQUIRE(n_slabs == 1 || slab_stride_rows >= slab_rows, PB_ERR_INVALID, "pb_mlp_update_fused: slabs overlap");
    PB_REQUIRE(workspace_bytes >= pb_mlp_update_workspace_bytes(), PB_ERR_INVALID, "pb_mlp_update_fused: workspace too small");
    PB_REQUIRE(!dbg_hidden || dbg_dpre, PB_ERR_INVALID, "pb_mlp_update_fused: dbg_hidden needs dbg_dpre");
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qr;
    PB_REQUIRE(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr) == cudaSuccess && fn &&
                   qr == cudaDriverEntryPointSuccess,
               PB_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
    const int64_t tiles_per_slab = (slab_rows + TILE_M - 1) / TILE_M;
    const int64_t n_tiles = tiles_per_slab * n_slabs;
    const int64_t map_rows = (int64_t)(n_slabs - 1) * slab_stride_rows + slab_rows;
    PB_REQUIRE(n_tiles <= 0x7FFFFFFF && map_rows <= 0x7FFFFFFF, PB_ERR_UNSUPPORTED, "pb_mlp_update_fused: too many rows");
    alignas(64) CUtensorMap map_x, map_w;
    int rc = make_map2((EncodeTiledFn)fn, &map_x, x, map_rows, ldx);
    if (rc == PB_OK) rc = make_map2((EncodeTiledFn)fn, &map_w, w_enc, HID, FEAT);
    if (rc != PB_OK) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    const int grid = n_tiles < num_sms() ? (int)n_tiles : num_sms();
    FusedParams p;
    p.actions = actions; p.old_logprobs = old_logprobs; p.adv = advantages; p.returns = returns; p.old_values = old_values;
    p.adv_norm = adv_norm; p.row_slab_stride = n_slabs > 1 ? row_slab_stride : slab_rows;
    p.m = slab_rows * n_slabs; p.slab_rows = slab_rows; p.slab_stride_rows = n_slabs > 1 ? slab_stride_rows : slab_rows;
    p.tiles_per_slab = (int)tiles_per_slab; p.n_tiles = (int)n_tiles; p.n_act = n_act;
    p.clip = clip_coef; p.vclip = vf_clip_coef; p.vf_coef = vf_coef; p.ent_coef = ent_coef; p.clip_vloss = clip_vloss;
    p.part_dw = (float*)workspace; p.part_tail = (float*)workspace + (size_t)num_sms() * FEAT * HID;
    p.dbg_clk = g_dbg_clk;
    p.w_heads = w_heads; p.b_enc = b_enc; p.b_heads = b_heads;
    p.stats = stats8; p.dbg_hidden = dbg_hidden; p.dbg_dpre = dbg_dpre; p.dbg_dout = dbg_dout;
    PB_CUDA(cudaMemsetAsync(stats8, 0, 8 * sizeof(double), s));
    static bool attr_set = false;
    if (!attr_set) {
        PB_CUDA(cudaFuncSetAttribute(k_mlp_update_xt<96, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, X2_TOTAL));
        PB_CUDA(cudaFuncSetAttribute(k_mlp_update_xt<96, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, X2_TOTAL));
        attr_set = true;
    }
    // 18 warps = 5 on two of the four schedulers: 16384 registers / (5 x 32) caps the kernel at 96 per thread
    if (p.dbg_clk) k_mlp_update_xt<96, true><<<grid, X2_THREADS, X2_TOTAL, s>>>(map_x, map_w, p);
    else k_mlp_update_xt<96, false><<<grid, X2_THREADS, X2_TOTAL, s>>>(map_x, map_w, p);
    PB_LAUNCH_CHECK();
    k_update_reduce<<<REDUCE_BLOCKS, 256, 0, s>>>(p.part_dw, p.part_tail, grid, grad_flat,
                                                  reinterpret_cast<double*>((char*)workspace + pb_mlp_update_sumsq_offset()));
    PB_LAUNCH_CHECK();
    return PB_OK;
}
