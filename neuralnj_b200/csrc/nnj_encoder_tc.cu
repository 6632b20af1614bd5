// nnj_encoder_tc.cu — the MSA encoder's per-token work on tcgen05 (precision bf16x3).
//
// The residual stream is kept SITE-MAJOR inside the encoder (token t = c*R + r for site c, taxon r) in the tile-planar layout of
// xs_off (nnj_internal.h): a tile of 128 consecutive tokens is one contiguous 32 KB block, every 16-byte column chunk a plane of
// its own, and the head-major row-attention planes [B,H,C,R*8] are written in 16-byte pieces that are contiguous across the lanes.  Between two tied row attentions everything is
// per token or per site, so one layer is three fused kernels (msa_modules.py:62-125):
//   k_enc_rowqkv_tc   LN1 + q|k|v projection of the tied row attention (axial_attention.py:75-82) -> bf16 hi/lo planes
//   k_enc_colblock_tc row out_proj + residual (:116), LN2 + column q|k|v (:211-214), per-site attention over taxa (:216-234),
//                     column out_proj + residual (:236) — x is read once and written once
//   k_enc_ffn_tc      LN3 + fc1 + GELU + fc2 + residual (msa_modules.py:144-151), hidden activations never leave the SM
// Every contraction is a split-bf16 UMMA (hi*hi + hi*lo + lo*hi, fp32 accumulation in TMEM); weights sit in shared memory as
// ready-made SWIZZLE_128B images (EncTcW); A operands are written by the threads that produced them (LayerNorm output, the
// attention context, the GELU output).  256 threads: warp w owns TMEM lane quarter w & 3 (row = 32*(w&3) + lane) and column
// half w >> 2, so a token row is handled by two threads that exchange only the LayerNorm statistics.
#include "nnj_internal.h"
#include "nnj_tc.cuh"

namespace nnj {

constexpr int ET_THREADS = 256;

__device__ __forceinline__ void copy_img(uint8_t* dst, const uint4* __restrict__ src, int bytes) {
    for (int i = threadIdx.x; i < (bytes >> 4); i += blockDim.x) reinterpret_cast<uint4*>(dst)[i] = __ldg(src + i);
}

// LayerNorm(64) (eps 1e-5, biased variance) of a row held as two 32-value halves by threads (row, hf = 0/1).  The halves are
// combined with the pairwise (Chan) update, so the result has two-pass quality.  Contains one __syncthreads.
__device__ __forceinline__ void ln_half(float (&v)[32], float2* part, int row, int hf, const float* __restrict__ g, const float* __restrict__ bta) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 32; ++k) s += v[k];
    const float mh = s * (1.0f / 32.0f);
    float m2 = 0.f;
#pragma unroll
    for (int k = 0; k < 32; ++k) { const float d = v[k] - mh; m2 = fmaf(d, d, m2); }
    part[hf * 128 + row] = make_float2(mh, m2);
    __syncthreads();
    const float2 o = part[(hf ^ 1) * 128 + row];
    const float mean = 0.5f * (mh + o.x), dm = mh - o.x;
    const float var = (m2 + o.y + dm * dm * 16.0f) * (1.0f / 64.0f);
    const float rstd = 1.0f / sqrtf(var + 1e-5f);
#pragma unroll
    for (int k = 0; k < 32; k += 4) {
        const float4 g4 = *reinterpret_cast<const float4*>(g + hf * 32 + k), b4 = *reinterpret_cast<const float4*>(bta + hf * 32 + k);
        v[k] = (v[k] - mean) * rstd * g4.x + b4.x;
        v[k + 1] = (v[k + 1] - mean) * rstd * g4.y + b4.y;
        v[k + 2] = (v[k + 2] - mean) * rstd * g4.z + b4.z;
        v[k + 3] = (v[k + 3] - mean) * rstd * g4.w + b4.w;
    }
}

// this thread's 32 values -> chunks hf*4 .. hf*4+3 of row `row` of the A operand
__device__ __forceinline__ void a_store32(uint8_t* a_hi, uint8_t* a_lo, int row, int hf, const float (&v)[32]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) a_store8(a_hi, a_lo, row, hf * 4 + j, &v[j * 8]);
}

// all threads: make the freshly written A operand visible to the tensor core, then one elected lane of warp 0 issues
#define ET_PUBLISH_A()      \
    do {                    \
        fence_async_smem(); \
        tc_fence_before();  \
        __syncthreads();    \
    } while (0)

// ------------------------------------------------------------------ K1: LN1 + row q|k|v -> planes
struct RowQkvArgs {
    const float* x; size_t x_tree_stride;      // site-major [B][C][R][64]
    int R, C, B, tiles_per_tree;
    const uint4* w_img;                         // EncTcW::row_qkv (48 KB)
    const float *ln_g, *ln_b, *qkvb;
    float q_scale; const uint8_t* mask;
    __nv_bfloat16 *qh, *ql, *kh, *kl, *vh, *vl; // [B,H,C,R*8]
    int one;                                    // NNJ_PREC_BF16: hi * hi products only, the lo planes are neither used nor written
};

constexpr int K1_W = 49152;
constexpr int K1_SMEM = 1024 + K1_W + 32768 + (192 + 128) * 4 + 2048 + 64;

__global__ void __launch_bounds__(ET_THREADS, 2) k_enc_rowqkv_tc(const RowQkvArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* sm = smem_align1024(smem_raw);
    uint8_t* w_s = sm;
    uint8_t* a_hi = sm + K1_W;
    uint8_t* a_lo = a_hi + 16384;
    float* s_bias = reinterpret_cast<float*>(a_lo + 16384);   // q|k|v biases [192]
    float* s_g = s_bias + 192;
    float* s_b = s_g + 64;
    float2* part = reinterpret_cast<float2*>(s_b + 64);
    uint64_t* bar = reinterpret_cast<uint64_t*>(part + 256);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, hf = warp >> 2, row = q * 32 + lane;
    if (tid == 0) { mbar_init(bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    if (warp == 0) tmem_alloc(tmem_slot, 256);
    copy_img(w_s, a.w_img, K1_W);
    if (tid < 192) s_bias[tid] = a.qkvb[tid];
    if (tid < 64) { s_g[tid] = a.ln_g[tid]; s_b[tid] = a.ln_b[tid]; }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16);
    const uint32_t idesc = umma_idesc_bf16(128, 192);
    const int T = a.R * a.C, KD = a.R * DH;
    const int n_work = a.B * a.tiles_per_tree;
    uint32_t it = 0;
    for (int w = blockIdx.x; w < n_work; w += gridDim.x, ++it) {
        const int b = w / a.tiles_per_tree, tile = w - b * a.tiles_per_tree;
        const int t = tile * 128 + row;
        const bool valid = t < T;
        const int c = valid ? t / a.R : 0, r = t - c * a.R;
        const float qs = (valid && a.mask && a.mask[(size_t)b * a.C + c]) ? 0.f : a.q_scale;   // axial_attention.py:81-82 (loaded with the tile, used after the UMMA)
        float v[32];
        if (valid) {
            const float* xp = a.x + (size_t)b * a.x_tree_stride + xs_off((size_t)t, hf * 8);
#pragma unroll
            for (int k = 0; k < 8; ++k) { const float4 f = ld4(xp + k * 512); v[4 * k] = f.x; v[4 * k + 1] = f.y; v[4 * k + 2] = f.z; v[4 * k + 3] = f.w; }
        } else {
#pragma unroll
            for (int k = 0; k < 32; ++k) v[k] = 0.f;
        }
        ln_half(v, part, row, hf, s_g, s_b);
        a_store32(a_hi, a_lo, row, hf, v);
        ET_PUBLISH_A();
        if (warp == 0) {
            tc_fence_after();
            if (elect_one()) {
                umma_split_k64(tmem_base, smem_u32(a_hi), smem_u32(a_lo), smem_u32(w_s), smem_u32(w_s) + K1_W / 2, idesc, 0u, a.one);
                umma_commit(bar);
            }
            __syncwarp();
        }
        mbar_wait(bar, it & 1);
        tc_fence_after();
#pragma unroll
        for (int p = 0; p < 3; ++p) {
            uint32_t acc[32];
            tmem_ld32(t_row + p * 64 + hf * 32, acc);
            if (valid) {
                __nv_bfloat16* ph = p == 0 ? a.qh : (p == 1 ? a.kh : a.vh);
                __nv_bfloat16* pl = p == 0 ? a.ql : (p == 1 ? a.kl : a.vl);
                const float s = p == 0 ? qs : 1.0f;
#pragma unroll
                for (int hh = 0; hh < 4; ++hh) {
                    float o[8];
#pragma unroll
                    for (int d = 0; d < 8; ++d) o[d] = (__uint_as_float(acc[hh * 8 + d]) + s_bias[p * 64 + hf * 32 + hh * 8 + d]) * s;
                    uint4 hi4, lo4;
                    split2(o[0], o[1], hi4.x, lo4.x);
                    split2(o[2], o[3], hi4.y, lo4.y);
                    split2(o[4], o[5], hi4.z, lo4.z);
                    split2(o[6], o[7], hi4.w, lo4.w);
                    const size_t off = (((size_t)b * H + hf * 4 + hh) * a.C + c) * KD + (size_t)r * DH;
                    *reinterpret_cast<uint4*>(ph + off) = hi4;
                    if (!a.one) *reinterpret_cast<uint4*>(pl + off) = lo4;
                }
            }
        }
        tc_fence_before();   // TMEM reads of this tile are ordered before the next tile's UMMA by the __syncthreads in between
    }
    __syncthreads();
    if (warp == 0) { tc_fence_after(); tmem_dealloc(tmem_base, 256); }
}

// ------------------------------------------------------------------ K3: LN3 + fc1 + GELU + fc2 + residual
struct FfnTcArgs {
    float* x; size_t x_tree_stride;             // site-major, updated in place
    int T, B, tiles_per_tree;
    const uint4 *w1, *w2;                       // EncTcW images (64 KB each)
    const float *ln_g, *ln_b, *b1, *b2;
    int one;                                    // NNJ_PREC_BF16: hi * hi products only
};

constexpr int K3_THREADS = 512;             // 16 warps: TMEM lane quarter q = warp & 3 (row = 32 q + lane), column quarter cq = warp >> 2 (16 of every 64 columns)
constexpr int K3_SMEM = 1024 + 2 * 65536 + (256 + 64 + 128) * 4 + 4096 + 64;
__device__ __forceinline__ void ln_quarter(float (&v)[16], float2* part, int row, int cq, const float* __restrict__ g, const float* __restrict__ bta);


__global__ void __launch_bounds__(K3_THREADS, 1) k_enc_ffn_tc(const FfnTcArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* sm = smem_align1024(smem_raw);
    uint8_t* w1_s = sm;                       // hi 32 KB | lo 32 KB   ([256][64])
    uint8_t* w2_s = sm + 65536;               // hi: 4 K-chunks of 8 KB | lo: 4 K-chunks
    float* s_b1 = reinterpret_cast<float*>(sm + 131072);
    float* s_b2 = s_b1 + 256;
    float* s_g = s_b2 + 64;
    float* s_b = s_g + 64;
    float2* part = reinterpret_cast<float2*>(s_b + 64);            // [4][128]
    uint64_t* bars = reinterpret_cast<uint64_t*>(part + 512);   // d1_done, c0_done, c1_done, d2_done, a_ready[2], a0_ready
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 7);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, cq = warp >> 2, row = q * 32 + lane;
    if (tid == 0) {
        for (int i = 0; i < 4; ++i) mbar_init(bars + i, 1);
        mbar_init(bars + 4, K3_THREADS / 32); mbar_init(bars + 5, K3_THREADS / 32); mbar_init(bars + 6, K3_THREADS / 32);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) tmem_alloc(tmem_slot, 512);
    copy_img(w1_s, a.w1, 65536);
    copy_img(w2_s, a.w2, 65536);
    if (tid < 256) s_b1[tid] = a.b1[tid];
    if (tid < 64) { s_b2[tid] = a.b2[tid]; s_g[tid] = a.ln_g[tid]; s_b[tid] = a.ln_b[tid]; }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t t_d1 = tmem_base, t_d2 = tmem_base + 256, t_a = tmem_base + 320, t_a0 = tmem_base + 448;   // D1 256 | D2 64 | GELU chunk operand 2 x (hi 32 | lo 32) | LN3(x) operand (hi 32 | lo 32)
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    const uint32_t id_d1 = umma_idesc_bf16(128, 256), id_d2 = umma_idesc_bf16(128, 64);
    const int n_work = a.B * a.tiles_per_tree;
    uint32_t it = 0;
    // this thread's 16 values of its token row, loaded one tile ahead (the global-load latency hides behind the previous tile's GEMMs)
    auto load_row = [&](int w, float4 (&dst)[4]) {
        const int b = w / a.tiles_per_tree, tile = w - b * a.tiles_per_tree;
        const int t = tile * 128 + row;
        if (w < n_work && t < a.T) {
            const float* xp = a.x + (size_t)b * a.x_tree_stride + xs_off((size_t)t, cq * 4);
#pragma unroll
            for (int k = 0; k < 4; ++k) dst[k] = ld4(xp + k * 512);
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) dst[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    float4 xnext[4];
    load_row(blockIdx.x, xnext);
    for (int w = blockIdx.x; w < n_work; w += gridDim.x, ++it) {
        const uint32_t par = it & 1;
        const int b = w / a.tiles_per_tree, tile = w - b * a.tiles_per_tree;
        const int t = tile * 128 + row;
        const bool valid = t < a.T;
        float* xp = a.x + (size_t)b * a.x_tree_stride + xs_off((size_t)t, cq * 4);
        float xr[16], v[16];
#pragma unroll
        for (int k = 0; k < 4; ++k) { xr[4 * k] = xnext[k].x; xr[4 * k + 1] = xnext[k].y; xr[4 * k + 2] = xnext[k].z; xr[4 * k + 3] = xnext[k].w; }
        load_row(w + gridDim.x, xnext);
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] = xr[k];
        ln_quarter(v, part, row, cq, s_g, s_b);
        {   // LN3(x) -> bf16 hi / lo in tensor memory: A operand of fc1
            uint32_t hh[8], ll[8];
#pragma unroll
            for (int k = 0; k < 16; k += 2) split2(v[k], v[k + 1], hh[k >> 1], ll[k >> 1]);
            tmem_st8(t_a0 + lane_off + cq * 8, hh);
            tmem_st8(t_a0 + lane_off + 32 + cq * 8, ll);
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bars + 6);
        }
        if (warp == 0) {   // hidden pre-activations D1 [128 x 256] = LN3(x) . fc1^T
            mbar_wait(bars + 6, par);
            tc_fence_after();
            if (elect_one()) {
                const uint32_t wh = umma_desc_lo(smem_u32(w1_s)), wl = umma_desc_lo(smem_u32(w1_s) + 32768);
                if (a.one) {
                    umma_ts<false>(t_d1, t_a0, wh, id_d1);
#pragma unroll
                    for (int kk = 1; kk < 4; ++kk) umma_ts<true>(t_d1, t_a0 + kk * 8, wh + kk * 2, id_d1);
                } else {
                    umma_ts<false>(t_d1, t_a0 + 32, wh, id_d1);      // small terms first
                    umma_ts<true>(t_d1, t_a0, wl, id_d1);
                    umma_ts<true>(t_d1, t_a0, wh, id_d1);
#pragma unroll
                    for (int kk = 1; kk < 4; ++kk) {
                        umma_ts<true>(t_d1, t_a0 + 32 + kk * 8, wh + kk * 2, id_d1);
                        umma_ts<true>(t_d1, t_a0 + kk * 8, wl + kk * 2, id_d1);
                        umma_ts<true>(t_d1, t_a0 + kk * 8, wh + kk * 2, id_d1);
                    }
                }
                umma_commit(bars + 0);
            }
            __syncwarp();
        }
        mbar_wait(bars + 0, par);
        tc_fence_after();
#pragma unroll 1
        for (int ch = 0; ch < 4; ++ch) {
            // GELU chunk ch -> bf16 hi / lo straight into TENSOR MEMORY (row = this thread's lane, two bf16 per column): the fc2 UMMA
            // reads its A operand from there (42 clk per 128 x 64 x 16 instead of 75 from shared memory) and the hand-off is an
            // mbarrier arrive per warp, not a block-wide barrier.  The operand buffer of chunk ch was last read by the UMMA of chunk ch-2.
            if (ch >= 2) { mbar_wait(bars + 1 + (ch - 2), par); tc_fence_after(); }
            uint32_t acc[16];
            tmem_ld16_nw(t_d1 + lane_off + ch * 64 + cq * 16, acc);
            tmem_ld_wait();
            uint32_t hh[8], ll[8];
#pragma unroll
            for (int k = 0; k < 16; k += 2) {      // packed fp32x2 math: hidden units (k, k+1) share every FMA-pipe instruction
                const float2 gl = gelu_fast2(fadd2(make_float2(__uint_as_float(acc[k]), __uint_as_float(acc[k + 1])),
                                                   *reinterpret_cast<const float2*>(s_b1 + ch * 64 + cq * 16 + k)));
                split2(gl.x, gl.y, hh[k >> 1], ll[k >> 1]);
            }
            const uint32_t ta = t_a + (ch & 1) * 64;
            tmem_st8(ta + lane_off + cq * 8, hh);
            tmem_st8(ta + lane_off + 32 + cq * 8, ll);
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bars + 4 + (ch & 1));
            if (warp == 0) {   // D2 [128 x 64] += GELU chunk . fc2[:, 64 ch .. 64 ch + 63]^T
                mbar_wait(bars + 4 + (ch & 1), (2 * it + (ch >> 1)) & 1);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t wh = umma_desc_lo(smem_u32(w2_s) + ch * 8192), wl = umma_desc_lo(smem_u32(w2_s) + 32768 + ch * 8192);
                    if (a.one) {
                        if (ch == 0) umma_ts<false>(t_d2, ta, wh, id_d2); else umma_ts<true>(t_d2, ta, wh, id_d2);
#pragma unroll
                        for (int kk = 1; kk < 4; ++kk) umma_ts<true>(t_d2, ta + kk * 8, wh + kk * 2, id_d2);
                    } else {
                        if (ch == 0) umma_ts<false>(t_d2, ta + 32, wh, id_d2); else umma_ts<true>(t_d2, ta + 32, wh, id_d2);   // small terms first
                        umma_ts<true>(t_d2, ta, wl, id_d2);
                        umma_ts<true>(t_d2, ta, wh, id_d2);
#pragma unroll
                        for (int kk = 1; kk < 4; ++kk) {
                            umma_ts<true>(t_d2, ta + 32 + kk * 8, wh + kk * 2, id_d2);
                            umma_ts<true>(t_d2, ta + kk * 8, wl + kk * 2, id_d2);
                            umma_ts<true>(t_d2, ta + kk * 8, wh + kk * 2, id_d2);
                        }
                    }
                    if (ch == 0) umma_commit(bars + 1);
                    else if (ch == 1) umma_commit(bars + 2);
                    else if (ch == 3) umma_commit(bars + 3);
                }
                __syncwarp();
            }
        }
        mbar_wait(bars + 3, par);
        tc_fence_after();
        {
            uint32_t acc[16];
            tmem_ld16_nw(t_d2 + lane_off + cq * 16, acc);
            tmem_ld_wait();
            if (valid) {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    st4(xp + k * 512, make_float4(xr[4 * k] + __uint_as_float(acc[4 * k]) + s_b2[cq * 16 + 4 * k],
                                                xr[4 * k + 1] + __uint_as_float(acc[4 * k + 1]) + s_b2[cq * 16 + 4 * k + 1],
                                                xr[4 * k + 2] + __uint_as_float(acc[4 * k + 2]) + s_b2[cq * 16 + 4 * k + 2],
                                                xr[4 * k + 3] + __uint_as_float(acc[4 * k + 3]) + s_b2[cq * 16 + 4 * k + 3]));
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 0) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
}

// ------------------------------------------------------------------ K2: row out_proj + residual, LN2, column attention block
// 512 threads.  In the projection stages warp w owns TMEM lane quarter w & 3 (row = 32*(w&3) + lane) and column quarter cq = w >> 2
// (16 columns = heads 2cq, 2cq+1), i.e. four threads per token row.  A tile holds s = 128 / rb whole sites, each in a block of
// rb = 32 / 64 / 128 rows (the power of two >= R).  In the attention stage a warp owns one (site, head) UNIT and a lane RPL = rb / 32
// query rows of it (lane, lane + 32, ...): every K / V row of the unit is fetched once per warp (a broadcast LDS.128) and serves all
// RPL rows of every lane.  Round 1 mapped (row, two heads) to a thread: 8 LDS.128 per key and THREAD, and the kernel sat on the
// shared-memory pipe (l1tex 73 %, 15 k of the 27 k clocks of a tile in this loop); q goes through shared memory now as well.
struct ColBlkArgs {
    float* x; size_t x_tree_stride;             // site-major, updated in place
    int R, C, B, rb_shift, groups_per_tree;     // rb = 1 << rb_shift rows per site block, s = 128 >> rb_shift sites per tile
    const float* ctx;                            // tied row-attention context fp32 [B,H,C,R*8]
    const uint4* w_img;                          // EncTcW::row_o | col_qkv | col_o, contiguous (80 KB)
    const float *rob, *ln_g, *ln_b, *qkvb, *cob;
    float q_scale_log2e; const uint8_t* mask;
    int one;                                     // NNJ_PREC_BF16: hi * hi products only in the three projections
};

constexpr int K2_THREADS = 512;
constexpr int K2_W = 81920;
constexpr int CB_LDK = 68;                     // fp32 row pitch of the q / K / V tiles: lanes = consecutive rows move 16 B each without bank conflicts
constexpr int K2_SMEM = 1024 + K2_W + 32768 + 3 * 128 * CB_LDK * 4 + (64 + 192 + 64 + 128) * 4 + 4096 + 64;

__device__ __forceinline__ float dot8(const float2 (&q)[4], float4 k0, float4 k1) {
    float2 acc = fmul2(q[0], make_float2(k0.x, k0.y));
    acc = ffma2(q[1], make_float2(k0.z, k0.w), acc);
    acc = ffma2(q[2], make_float2(k1.x, k1.y), acc);
    acc = ffma2(q[3], make_float2(k1.z, k1.w), acc);
    return acc.x + acc.y;
}

// LayerNorm(64) of a row held as four 16-value quarters by threads (row, cq = 0..3); quarters combined pairwise (Chan), in the
// same fixed order by all four threads.  Contains one __syncthreads.
__device__ __forceinline__ void ln_quarter(float (&v)[16], float2* part, int row, int cq, const float* __restrict__ g, const float* __restrict__ bta) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) s += v[k];
    const float mq = s * (1.0f / 16.0f);
    float m2 = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) { const float d = v[k] - mq; m2 = fmaf(d, d, m2); }
    part[cq * 128 + row] = make_float2(mq, m2);
    __syncthreads();
    const float2 p0 = part[row], p1 = part[128 + row], p2 = part[256 + row], p3 = part[384 + row];
    const float d01 = p0.x - p1.x, d23 = p2.x - p3.x;
    const float m01 = 0.5f * (p0.x + p1.x), m23 = 0.5f * (p2.x + p3.x);
    const float s01 = p0.y + p1.y + d01 * d01 * 8.0f, s23 = p2.y + p3.y + d23 * d23 * 8.0f;
    const float mean = 0.5f * (m01 + m23), dm = m01 - m23;
    const float var = (s01 + s23 + dm * dm * 16.0f) * (1.0f / 64.0f);
    const float rstd = 1.0f / sqrtf(var + 1e-5f);
#pragma unroll
    for (int k = 0; k < 16; k += 4) {
        const float4 g4 = *reinterpret_cast<const float4*>(g + cq * 16 + k), b4 = *reinterpret_cast<const float4*>(bta + cq * 16 + k);
        v[k] = (v[k] - mean) * rstd * g4.x + b4.x;
        v[k + 1] = (v[k + 1] - mean) * rstd * g4.y + b4.y;
        v[k + 2] = (v[k + 2] - mean) * rstd * g4.z + b4.z;
        v[k + 3] = (v[k + 3] - mean) * rstd * g4.w + b4.w;
    }
}

__device__ __forceinline__ void a_store16(uint8_t* a_hi, uint8_t* a_lo, int row, int cq, const float (&v)[16]) {
    a_store8(a_hi, a_lo, row, cq * 2, &v[0]);
    a_store8(a_hi, a_lo, row, cq * 2 + 1, &v[8]);
}

#ifdef NNJ_COL_TRACE
// stage timeline of CTA 0 (thread 0), first 32 work items: debug builds only (scratch/col_trace.py)
__device__ long long g_col_trace[32 * 16];
#define COL_STAMP(i) do { if (threadIdx.x == 0 && blockIdx.x == 0 && trace_it < 32) g_col_trace[trace_it * 16 + (i)] = clock64(); } while (0)
#else
#define COL_STAMP(i) do { } while (0)
#endif

// Attention of RPL query rows (one head) over the R keys of their site: chunked online softmax (logits carry log2 e, probabilities
// are exp2; the running maximum moves - and the accumulators are rescaled - once per CH keys, not per key).
template <int RPL, int CH>
__device__ __forceinline__ void col_attend(const float* __restrict__ qb, const float* __restrict__ kb, const float* __restrict__ vb, int R, int lane,
                                           float (&o)[RPL][8]) {
    float2 q[RPL][4], acc[RPL][4];
    float m[RPL], l[RPL];
#pragma unroll
    for (int k = 0; k < RPL; ++k) {
        const float4 q0 = ld4(qb + (lane + 32 * k) * CB_LDK), q1 = ld4(qb + (lane + 32 * k) * CB_LDK + 4);
        q[k][0] = make_float2(q0.x, q0.y); q[k][1] = make_float2(q0.z, q0.w); q[k][2] = make_float2(q1.x, q1.y); q[k][3] = make_float2(q1.z, q1.w);
        m[k] = -INFINITY; l[k] = 0.f;
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[k][e] = make_float2(0.f, 0.f);
    }
    int j0 = 0;
    for (; j0 + CH <= R; j0 += CH) {
        float s[RPL][CH];
#pragma unroll
        for (int u = 0; u < CH; ++u) {
            const float4 k0 = ld4(kb + (j0 + u) * CB_LDK), k1 = ld4(kb + (j0 + u) * CB_LDK + 4);
#pragma unroll
            for (int k = 0; k < RPL; ++k) s[k][u] = dot8(q[k], k0, k1);
        }
#pragma unroll
        for (int k = 0; k < RPL; ++k) {
            float n = m[k];
#pragma unroll
            for (int u = 0; u < CH; ++u) n = fmaxf(n, s[k][u]);
            const float f = ex2_approx(m[k] - n);          // 0 on the first chunk (m = -inf), 1 when the maximum stays
            l[k] *= f; m[k] = n;
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[k][e] = fmul2(acc[k][e], splat2(f));
        }
#pragma unroll
        for (int u = 0; u < CH; ++u) {
            const float4 v0 = ld4(vb + (j0 + u) * CB_LDK), v1 = ld4(vb + (j0 + u) * CB_LDK + 4);
#pragma unroll
            for (int k = 0; k < RPL; ++k) {
                const float p = ex2_approx(s[k][u] - m[k]);
                l[k] += p;
                acc[k][0] = ffma2(splat2(p), make_float2(v0.x, v0.y), acc[k][0]); acc[k][1] = ffma2(splat2(p), make_float2(v0.z, v0.w), acc[k][1]);
                acc[k][2] = ffma2(splat2(p), make_float2(v1.x, v1.y), acc[k][2]); acc[k][3] = ffma2(splat2(p), make_float2(v1.z, v1.w), acc[k][3]);
            }
        }
    }
#pragma unroll 1
    for (; j0 < R; ++j0) {                                   // the R % CH last keys, one at a time
        const float4 k0 = ld4(kb + j0 * CB_LDK), k1 = ld4(kb + j0 * CB_LDK + 4);
        const float4 v0 = ld4(vb + j0 * CB_LDK), v1 = ld4(vb + j0 * CB_LDK + 4);
#pragma unroll
        for (int k = 0; k < RPL; ++k) {
            const float s = dot8(q[k], k0, k1);
            const float n = fmaxf(m[k], s);
            const float f = ex2_approx(m[k] - n), p = ex2_approx(s - n);
            m[k] = n;
            l[k] = fmaf(l[k], f, p);
            acc[k][0] = ffma2(splat2(p), make_float2(v0.x, v0.y), fmul2(acc[k][0], splat2(f))); acc[k][1] = ffma2(splat2(p), make_float2(v0.z, v0.w), fmul2(acc[k][1], splat2(f)));
            acc[k][2] = ffma2(splat2(p), make_float2(v1.x, v1.y), fmul2(acc[k][2], splat2(f))); acc[k][3] = ffma2(splat2(p), make_float2(v1.z, v1.w), fmul2(acc[k][3], splat2(f)));
        }
    }
#pragma unroll
    for (int k = 0; k < RPL; ++k) {
        const float inv = 1.0f / l[k];
#pragma unroll
        for (int e = 0; e < 4; ++e) { o[k][2 * e] = acc[k][e].x * inv; o[k][2 * e + 1] = acc[k][e].y * inv; }
    }
}

// ---- tensor-path attention (R <= 64).  q | k | v of the tile sit in shared memory as bf16 hi / lo planes [128 rows][64] (128 B per row,
// the 16-byte chunk of head h stored at h ^ (row & 7): the A-operand swizzle, conflict-free for the fragment loads below).
constexpr int K2_PLANE = 128 * 128;
// One (site, head, 16-query-row block): S = Q K^T [16 x 8 NT], softmax over the R keys in registers (the C fragments of two key blocks
// ARE the A fragment of the next m16n8k16), O = P V, normalised and written as bf16 hi / lo into the A operand of the column
// out-projection.  The 3-product bf16 split costs two instructions per 8 keys in Q K^T - the head dimension is 8, so the K = 16 of one
// instruction holds [q_hi | q_lo] . [k_hi | k_hi], a second one [q_hi | 0] . [k_lo | 0] - and three per 16 keys in P V.
// NT = ceil(R / 8) key blocks is a template constant: no predication inside.
template <int NT>
__device__ __forceinline__ void col_attend_mma(const uint8_t* __restrict__ pl, uint8_t* __restrict__ a_hi, uint8_t* __restrict__ a_lo, int row_base, int mt, int h, int R,
                                               int lane) {
    const int g = lane >> 2, t = lane & 3;
    const int r0 = row_base + mt * 16 + g;                                  // rows r0 and r0 + 8; row & 7 = g for both
    const uint32_t sw = (uint32_t)(((h ^ g) << 4) + t * 4);
    const uint8_t* qp = pl + r0 * 128 + sw;
    const uint32_t qh0 = *reinterpret_cast<const uint32_t*>(qp), qh1 = *reinterpret_cast<const uint32_t*>(qp + 1024);
    const uint32_t ql0 = *reinterpret_cast<const uint32_t*>(qp + K2_PLANE), ql1 = *reinterpret_cast<const uint32_t*>(qp + K2_PLANE + 1024);
    const uint8_t* kp = pl + 2 * K2_PLANE + (row_base + g) * 128 + sw;      // key rows 8 n + g
    float sc[NT][4];
#pragma unroll
    for (int n = 0; n < NT; ++n) {
        const uint32_t kh = *reinterpret_cast<const uint32_t*>(kp + n * 1024), kl = *reinterpret_cast<const uint32_t*>(kp + K2_PLANE + n * 1024);
        sc[n][0] = 0.f; sc[n][1] = 0.f; sc[n][2] = 0.f; sc[n][3] = 0.f;
        mma_m16n8k16(sc[n], {qh0, qh1, 0u, 0u}, kl, 0u);        // q_hi . k_lo (small term first)
        mma_m16n8k16(sc[n], {qh0, qh1, ql0, ql1}, kh, kh);      // q_hi . k_hi + q_lo . k_hi
    }
    {   // keys >= R do not exist (only the last key block can hold them)
        const int j = (NT - 1) * 8 + 2 * t;
        if (j >= R) { sc[NT - 1][0] = -INFINITY; sc[NT - 1][2] = -INFINITY; }
        if (j + 1 >= R) { sc[NT - 1][1] = -INFINITY; sc[NT - 1][3] = -INFINITY; }
    }
    float m_a = fmaxf(sc[0][0], sc[0][1]), m_b = fmaxf(sc[0][2], sc[0][3]);
#pragma unroll
    for (int n = 1; n < NT; ++n) { m_a = fmaxf(m_a, fmaxf(sc[n][0], sc[n][1])); m_b = fmaxf(m_b, fmaxf(sc[n][2], sc[n][3])); }
    m_a = fmaxf(m_a, __shfl_xor_sync(0xffffffffu, m_a, 1)); m_a = fmaxf(m_a, __shfl_xor_sync(0xffffffffu, m_a, 2));
    m_b = fmaxf(m_b, __shfl_xor_sync(0xffffffffu, m_b, 1)); m_b = fmaxf(m_b, __shfl_xor_sync(0xffffffffu, m_b, 2));
    float2 l_a = make_float2(0.f, 0.f), l_b = make_float2(0.f, 0.f);
    float o0[4] = {0.f, 0.f, 0.f, 0.f}, o1[4] = {0.f, 0.f, 0.f, 0.f};      // two accumulators: alternate 16-key steps
    // lane l supplies row l & 7 of matrix l >> 3: matrices 0, 1 = v_hi of two consecutive key blocks, 2, 3 = v_lo of the same
    const uint32_t vaddr = smem_u32(pl) + (uint32_t)((4 + ((lane >> 4) & 1)) * K2_PLANE + (row_base + ((lane >> 3) & 1) * 8 + (lane & 7)) * 128 + ((h ^ (lane & 7)) << 4));
#pragma unroll
    for (int n2 = 0; n2 < (NT + 1) / 2; ++n2) {
        uint32_t vf[4];      // v_hi(2 n2), v_hi(2 n2 + 1), v_lo(2 n2), v_lo(2 n2 + 1)
        ldsm_x4_t(vf, vaddr + n2 * 2048);
        uint32_t ph[4], pw[4];                                  // P hi / lo as the A fragment: [row g | row g+8] of block 2 n2, then of block 2 n2 + 1
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int n = 2 * n2 + e;
            if (n < NT) {
                const float2 da = fsub2(make_float2(sc[n][0], sc[n][1]), splat2(m_a)), db = fsub2(make_float2(sc[n][2], sc[n][3]), splat2(m_b));
                const float2 pa = make_float2(ex2_approx(da.x), ex2_approx(da.y)), pb = make_float2(ex2_approx(db.x), ex2_approx(db.y));
                l_a = fadd2(l_a, pa); l_b = fadd2(l_b, pb);
                split2(pa.x, pa.y, ph[2 * e], pw[2 * e]);
                split2(pb.x, pb.y, ph[2 * e + 1], pw[2 * e + 1]);
            } else {                                            // NT odd: the second block of the last step does not exist
                ph[2 * e] = 0u; ph[2 * e + 1] = 0u; pw[2 * e] = 0u; pw[2 * e + 1] = 0u;
            }
        }
        float (&o)[4] = (n2 & 1) ? o1 : o0;
        mma_m16n8k16(o, pw, vf[0], vf[1]);      // P_lo . V_hi
        mma_m16n8k16(o, ph, vf[2], vf[3]);      // P_hi . V_lo
        mma_m16n8k16(o, ph, vf[0], vf[1]);      // P_hi . V_hi
    }
    float s_a = l_a.x + l_a.y, s_b = l_b.x + l_b.y;
    s_a += __shfl_xor_sync(0xffffffffu, s_a, 1); s_a += __shfl_xor_sync(0xffffffffu, s_a, 2);
    s_b += __shfl_xor_sync(0xffffffffu, s_b, 1); s_b += __shfl_xor_sync(0xffffffffu, s_b, 2);
    const float i_a = 1.0f / s_a, i_b = 1.0f / s_b;
    uint32_t oh, ol;
    split2((o0[0] + o1[0]) * i_a, (o0[1] + o1[1]) * i_a, oh, ol);
    *reinterpret_cast<uint32_t*>(a_hi + r0 * 128 + sw) = oh;
    *reinterpret_cast<uint32_t*>(a_lo + r0 * 128 + sw) = ol;
    split2((o0[2] + o1[2]) * i_b, (o0[3] + o1[3]) * i_b, oh, ol);
    *reinterpret_cast<uint32_t*>(a_hi + (r0 + 8) * 128 + sw) = oh;
    *reinterpret_cast<uint32_t*>(a_lo + (r0 + 8) * 128 + sw) = ol;
}

// NT = 0: CUDA-core attention (col_attend, 64 < R <= 128); NT > 0: tensor-path attention with NT = ceil(R / 8) key blocks (R <= 64)
template <int RPL, int NT>
__global__ void __launch_bounds__(K2_THREADS, 1) k_enc_colblock_tc(const ColBlkArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* sm = smem_align1024(smem_raw);
    uint8_t* w_ro = sm;                        // row out_proj   hi 8 KB | lo 8 KB
    uint8_t* w_qkv = sm + 16384;               // column q|k|v   hi 24 KB | lo 24 KB
    uint8_t* w_co = sm + 65536;                // column out_proj
    uint8_t* a_hi = sm + K2_W;
    uint8_t* a_lo = a_hi + 16384;
    float* qsm = reinterpret_cast<float*>(a_lo + 16384);   // NT = 0: [128][CB_LDK] fp32 q (scaled), then K, then V
    uint8_t* pl = a_lo + 16384;                            // NT > 0: planes q_hi | q_lo | k_hi | k_lo | v_hi | v_lo (same region)
    float* ks = qsm + 128 * CB_LDK;
    float* vs = ks + 128 * CB_LDK;
    float* s_rob = vs + 128 * CB_LDK;
    float* s_qkvb = s_rob + 64;
    float* s_cob = s_qkvb + 192;
    float* s_g = s_cob + 64;
    float* s_b = s_g + 64;
    float2* part = reinterpret_cast<float2*>(s_b + 64);   // [4][128]
    uint64_t* bar = reinterpret_cast<uint64_t*>(part + 512);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, cq = warp >> 2, row = q * 32 + lane;
    if (tid == 0) { mbar_init(bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    if (warp == 0) tmem_alloc(tmem_slot, 256);
    for (int i = tid; i < (K2_W >> 4); i += K2_THREADS) reinterpret_cast<uint4*>(sm)[i] = __ldg(a.w_img + i);
    if (tid < 192) s_qkvb[tid] = a.qkvb[tid];
    if (tid < 64) { s_rob[tid] = a.rob[tid]; s_cob[tid] = a.cob[tid]; s_g[tid] = a.ln_g[tid]; s_b[tid] = a.ln_b[tid]; }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t t_o = tmem_base, t_qkv = tmem_base + 64;          // [128 x 64] projections | [128 x 192] q|k|v
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    const uint32_t id64 = umma_idesc_bf16(128, 64), id192 = umma_idesc_bf16(128, 192);
    const int R = a.R, KD = a.R * DH;
    constexpr int rb_shift = RPL == 1 ? 5 : (RPL == 2 ? 6 : 7);
    constexpr int rb = 1 << rb_shift, s_tile = 128 >> rb_shift;
    const int si = row >> rb_shift, r = row & (rb - 1);
    const int n_work = a.B * a.groups_per_tree;
    // this thread's piece of work item w: 16 values of the row-attention context (heads 2cq, 2cq+1), 16 of x, the padded-site flag.
    // Item w + grid is fetched while the tensor core runs stage 4 of item w, so the DRAM latency is off the serial chain.
    auto load_tile = [&](int w, float (&vv)[16], float (&xx)[16], float& qsc) {
        const int b = w / a.groups_per_tree, grp = w - b * a.groups_per_tree;
        const int c = grp * s_tile + si;
        const bool valid = w < n_work && r < R && c < a.C;
        // all keys of a padded site get the same logit (-10000, axial_attention.py:220-224): softmax is uniform, i.e. q = 0
        qsc = (valid && a.mask && a.mask[(size_t)b * a.C + c]) ? 0.f : a.q_scale_log2e;
        if (valid) {
            const float* xq = a.x + (size_t)b * a.x_tree_stride + xs_off((size_t)c * R + r, cq * 4);
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                const float* cp = a.ctx + (((size_t)b * H + cq * 2 + hh) * a.C + c) * KD + (size_t)r * DH;
                const float4 f0 = ld4(cp), f1 = ld4(cp + 4);
                vv[hh * 8] = f0.x; vv[hh * 8 + 1] = f0.y; vv[hh * 8 + 2] = f0.z; vv[hh * 8 + 3] = f0.w;
                vv[hh * 8 + 4] = f1.x; vv[hh * 8 + 5] = f1.y; vv[hh * 8 + 6] = f1.z; vv[hh * 8 + 7] = f1.w;
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) { const float4 f = ld4(xq + k * 512); xx[4 * k] = f.x; xx[4 * k + 1] = f.y; xx[4 * k + 2] = f.z; xx[4 * k + 3] = f.w; }
        } else {
#pragma unroll
            for (int k = 0; k < 16; ++k) { vv[k] = 0.f; xx[k] = 0.f; }
        }
    };
    float xn[16], vn[16], qsn = 0.f;
    load_tile(blockIdx.x, vn, xn, qsn);
    uint32_t ph = 0;   // completions of `bar` so far
#ifdef NNJ_COL_TRACE
    int trace_it = -1;
#endif
    for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
#ifdef NNJ_COL_TRACE
        ++trace_it;
#endif
        COL_STAMP(0);
        const int b = w / a.groups_per_tree, grp = w - b * a.groups_per_tree;
        const int c = grp * s_tile + si;
        const bool valid = r < R && c < a.C;
        float* xp = a.x + (size_t)b * a.x_tree_stride + xs_off((size_t)c * R + r, cq * 4);
        float xr[16], v[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) { xr[k] = xn[k]; v[k] = vn[k]; }
        const float qs = qsn;
        // ---- stage 1: x += ctx_row . W_o^T + b_o
        a_store16(a_hi, a_lo, row, cq, v);
        ET_PUBLISH_A();
        COL_STAMP(1);
        if (warp == 0) {
            tc_fence_after();
            if (elect_one()) {
                umma_split_k64(t_o, smem_u32(a_hi), smem_u32(a_lo), smem_u32(w_ro), smem_u32(w_ro) + 8192, id64, 0u, a.one);
                umma_commit(bar);
            }
            __syncwarp();
        }
        mbar_wait(bar, ph & 1); ++ph;
        tc_fence_after();
        COL_STAMP(2);
        {
            uint32_t acc[16];
            tmem_ld16_nw(t_o + lane_off + cq * 16, acc);
            tmem_ld_wait();
#pragma unroll
            for (int k = 0; k < 16; ++k) xr[k] += __uint_as_float(acc[k]) + s_rob[cq * 16 + k];
        }
        // ---- stage 2: q|k|v = LN2(x) . W^T + b
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] = xr[k];
        tc_fence_before();
        ln_quarter(v, part, row, cq, s_g, s_b);
        a_store16(a_hi, a_lo, row, cq, v);
        ET_PUBLISH_A();
        COL_STAMP(3);
        if (warp == 0) {
            tc_fence_after();
            if (elect_one()) {
                umma_split_k64(t_qkv, smem_u32(a_hi), smem_u32(a_lo), smem_u32(w_qkv), smem_u32(w_qkv) + 24576, id192, 0u, a.one);
                umma_commit(bar);
            }
            __syncwarp();
        }
        mbar_wait(bar, ph & 1); ++ph;
        tc_fence_after();
        COL_STAMP(4);
        {   // q (scaled by dh^-0.5 log2 e, 0 on a padded site) | k | v + bias -> fp32 tiles (NT = 0) or bf16 hi / lo planes (NT > 0)
            uint32_t acc[16];
#pragma unroll
            for (int p = 0; p < 3; ++p) {
                tmem_ld16_nw(t_qkv + lane_off + p * 64 + cq * 16, acc);
                tmem_ld_wait();
                const float sc = p == 0 ? qs : 1.0f;
                if constexpr (NT > 0) {
                    float f[16];
#pragma unroll
                    for (int k = 0; k < 16; ++k) f[k] = (__uint_as_float(acc[k]) + s_qkvb[p * 64 + cq * 16 + k]) * sc;
                    a_store8(pl + (2 * p) * K2_PLANE, pl + (2 * p + 1) * K2_PLANE, row, cq * 2, &f[0]);
                    a_store8(pl + (2 * p) * K2_PLANE, pl + (2 * p + 1) * K2_PLANE, row, cq * 2 + 1, &f[8]);
                } else {
                    float* dst = qsm + p * 128 * CB_LDK + row * CB_LDK + cq * 16;
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        st4(dst + k * 4, make_float4((__uint_as_float(acc[4 * k]) + s_qkvb[p * 64 + cq * 16 + 4 * k]) * sc, (__uint_as_float(acc[4 * k + 1]) + s_qkvb[p * 64 + cq * 16 + 4 * k + 1]) * sc,
                                                     (__uint_as_float(acc[4 * k + 2]) + s_qkvb[p * 64 + cq * 16 + 4 * k + 2]) * sc, (__uint_as_float(acc[4 * k + 3]) + s_qkvb[p * 64 + cq * 16 + 4 * k + 3]) * sc));
                }
            }
        }
        tc_fence_before();
        __syncthreads();
        COL_STAMP(5);
        // ---- stage 3.  Rows >= R of a site block hold finite padding (LN of zeros); their results are never stored.
        if constexpr (NT > 0) {
            // warp = (site, head, 16-row block) items
            constexpr int MT = (NT + 1) / 2;
            for (int item = warp; item < s_tile * H * MT; item += K2_THREADS / 32) {
                const int mt = item % MT, uh = item / MT;
                col_attend_mma<NT>(pl, a_hi, a_lo, (uh >> 3) << rb_shift, mt, uh & 7, R, lane);
            }
        } else {
            // warp = (site, head) unit, lane = RPL query rows
            for (int unit = warp; unit < s_tile * H; unit += K2_THREADS / 32) {
                const int s_i = unit >> 3, h = unit & 7;
                const int base = (s_i << rb_shift) * CB_LDK + h * 8;
                float o[RPL][8];
                col_attend<RPL, RPL == 4 ? 2 : 5>(qsm + base, ks + base, vs + base, R, lane, o);
#pragma unroll
                for (int k = 0; k < RPL; ++k) a_store8(a_hi, a_lo, (s_i << rb_shift) + lane + 32 * k, h, o[k]);
            }
        }
        COL_STAMP(6);
        load_tile(w + gridDim.x, vn, xn, qsn);      // next work item's rows: in flight during stage 4
        // ---- stage 4: x += ctx_col . W_o^T + b_o
        ET_PUBLISH_A();
        COL_STAMP(7);
        if (warp == 0) {
            tc_fence_after();
            if (elect_one()) {
                umma_split_k64(t_o, smem_u32(a_hi), smem_u32(a_lo), smem_u32(w_co), smem_u32(w_co) + 8192, id64, 0u, a.one);
                umma_commit(bar);
            }
            __syncwarp();
        }
        mbar_wait(bar, ph & 1); ++ph;
        tc_fence_after();
        COL_STAMP(8);
        {
            uint32_t acc[16];
            tmem_ld16_nw(t_o + lane_off + cq * 16, acc);
            tmem_ld_wait();
            if (valid) {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    st4(xp + k * 512, make_float4(xr[4 * k] + __uint_as_float(acc[4 * k]) + s_cob[cq * 16 + 4 * k],
                                                xr[4 * k + 1] + __uint_as_float(acc[4 * k + 1]) + s_cob[cq * 16 + 4 * k + 1],
                                                xr[4 * k + 2] + __uint_as_float(acc[4 * k + 2]) + s_cob[cq * 16 + 4 * k + 2],
                                                xr[4 * k + 3] + __uint_as_float(acc[4 * k + 3]) + s_cob[cq * 16 + 4 * k + 3]));
            }
        }
        tc_fence_before();
        COL_STAMP(9);
    }
    __syncthreads();
    if (warp == 0) { tc_fence_after(); tmem_dealloc(tmem_base, 256); }
}
#ifdef NNJ_COL_TRACE
extern "C" int nnj_col_trace_read(long long* out) { return (int)cudaMemcpyFromSymbol(out, g_col_trace, sizeof(long long) * 32 * 16); }
#endif

// ------------------------------------------------------------------ site-major -> node-major (the NJ pool / public layout [B,R,C,64])
__global__ void __launch_bounds__(256) k_sm_to_nm(const float* __restrict__ xs, size_t xs_tree_stride, float* __restrict__ out, size_t out_tree_stride,
                                                  int R, int C) {
    const int b = blockIdx.y;
    const size_t n4 = (size_t)R * C * 16;
    const float* src = xs + (size_t)b * xs_tree_stride;
    float* dst = out + (size_t)b * out_tree_stride;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
        const size_t tok = i >> 4;
        const int c4 = (int)(i & 15);
        const int c = (int)(tok / R), r = (int)(tok - (size_t)c * R);
        st4(dst + ((size_t)r * C + c) * D + c4 * 4, ld4(src + xs_off(tok, c4)));
    }
}

// ------------------------------------------------------------------ launchers
static int enc_tc_attrs() {
    static DevOnce once;      // per device, not per process
    if (!once.need()) return 0;
    cudaError_t e = cudaFuncSetAttribute(k_enc_rowqkv_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, K1_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_enc_colblock_tc<1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_enc_colblock_tc<1, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_enc_colblock_tc<1, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_enc_colblock_tc<1, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_enc_colblock_tc<2, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_enc_colblock_tc<2, 6>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_enc_colblock_tc<2, 7>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_enc_colblock_tc<2, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_enc_colblock_tc<4, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_enc_ffn_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, K3_SMEM);
    if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    once.done();
    return 0;
}

int launch_enc_rowqkv_tc(const Model* m, int layer, const float* xs, size_t xs_tree_stride, int B, int R, int C, float q_scale, const uint8_t* mask,
                         void* qh, void* ql, void* kh, void* kl, void* vh, void* vl, cudaStream_t st) {
    if (int e = enc_tc_attrs()) return e;
    const LayerW& lw = m->layers[layer];
    const EncTcW& tw = m->enc_tc[layer];
    RowQkvArgs a;
    a.x = xs; a.x_tree_stride = xs_tree_stride; a.R = R; a.C = C; a.B = B; a.tiles_per_tree = (R * C + 127) / 128;
    a.w_img = tw.row_qkv; a.ln_g = lw.row.ln_g; a.ln_b = lw.row.ln_b; a.qkvb = tw.row_qkvb; a.q_scale = q_scale; a.mask = mask;
    a.qh = (__nv_bfloat16*)qh; a.ql = (__nv_bfloat16*)ql; a.kh = (__nv_bfloat16*)kh; a.kl = (__nv_bfloat16*)kl;
    a.vh = (__nv_bfloat16*)vh; a.vl = (__nv_bfloat16*)vl;
    a.one = m->cfg.precision == NNJ_PREC_BF16;
    const int work = B * a.tiles_per_tree;
    const int grid = work < 2 * sm_count() ? work : 2 * sm_count();
    prof_begin(KC_LN_QKV, st);
    k_enc_rowqkv_tc<<<grid, ET_THREADS, K1_SMEM, st>>>(a);
    LAUNCH_CHECK();
    return 0;
}

int launch_enc_colblock_tc(const Model* m, int layer, float* xs, size_t xs_tree_stride, const float* ctx, int B, int R, int C, const uint8_t* mask,
                           cudaStream_t st) {
    if (int e = enc_tc_attrs()) return e;
    if (R > 128) return set_error(NNJ_ERR_INVALID, "encode: the fused column block handles at most 128 taxa");
    const LayerW& lw = m->layers[layer];
    const EncTcW& tw = m->enc_tc[layer];
    ColBlkArgs a;
    a.rb_shift = R <= 32 ? 5 : (R <= 64 ? 6 : 7);
    const int s_tile = 128 >> a.rb_shift;
    a.x = xs; a.x_tree_stride = xs_tree_stride; a.R = R; a.C = C; a.B = B; a.groups_per_tree = (C + s_tile - 1) / s_tile;
    a.ctx = ctx; a.w_img = tw.row_o; a.rob = lw.row.ob; a.ln_g = lw.col.ln_g; a.ln_b = lw.col.ln_b; a.qkvb = tw.col_qkvb; a.cob = lw.col.ob;
    a.q_scale_log2e = (1.0f / sqrtf((float)DH)) * 1.4426950408889634f; a.mask = mask;
    a.one = m->cfg.precision == NNJ_PREC_BF16;
    const int work = B * a.groups_per_tree;
    const int grid = work < sm_count() ? work : sm_count();
    prof_begin(KC_COL_ATTN, st);
    switch (R <= 64 ? (R + 7) / 8 : 0) {     // key blocks of the tensor-path attention (R <= 64); CUDA-core attention above
        case 1: k_enc_colblock_tc<1, 1><<<grid, K2_THREADS, K2_SMEM, st>>>(a); break;
        case 2: k_enc_colblock_tc<1, 2><<<grid, K2_THREADS, K2_SMEM, st>>>(a); break;
        case 3: k_enc_colblock_tc<1, 3><<<grid, K2_THREADS, K2_SMEM, st>>>(a); break;
        case 4: k_enc_colblock_tc<1, 4><<<grid, K2_THREADS, K2_SMEM, st>>>(a); break;
        case 5: k_enc_colblock_tc<2, 5><<<grid, K2_THREADS, K2_SMEM, st>>>(a); break;
        case 6: k_enc_colblock_tc<2, 6><<<grid, K2_THREADS, K2_SMEM, st>>>(a); break;
        case 7: k_enc_colblock_tc<2, 7><<<grid, K2_THREADS, K2_SMEM, st>>>(a); break;
        case 8: k_enc_colblock_tc<2, 8><<<grid, K2_THREADS, K2_SMEM, st>>>(a); break;
        default: k_enc_colblock_tc<4, 0><<<grid, K2_THREADS, K2_SMEM, st>>>(a); break;
    }
    LAUNCH_CHECK();
    return 0;
}

int launch_enc_ffn_tc(const Model* m, int layer, float* xs, size_t xs_tree_stride, int B, int R, int C, cudaStream_t st) {
    if (int e = enc_tc_attrs()) return e;
    const LayerW& lw = m->layers[layer];
    const EncTcW& tw = m->enc_tc[layer];
    FfnTcArgs a;
    a.x = xs; a.x_tree_stride = xs_tree_stride; a.T = R * C; a.B = B; a.tiles_per_tree = (R * C + 127) / 128;
    a.w1 = tw.w1; a.w2 = tw.w2; a.ln_g = lw.ffn.ln_g; a.ln_b = lw.ffn.ln_b; a.b1 = lw.ffn.b1; a.b2 = lw.ffn.b2;
    a.one = m->cfg.precision == NNJ_PREC_BF16;
    const int work = B * a.tiles_per_tree;
    const int grid = work < sm_count() ? work : sm_count();
    prof_begin(KC_FFN, st);
    k_enc_ffn_tc<<<grid, K3_THREADS, K3_SMEM, st>>>(a);
    LAUNCH_CHECK();
    return 0;
}

int launch_sm_to_nm(const float* xs, size_t xs_tree_stride, float* out, size_t out_tree_stride, int B, int R, int C, cudaStream_t st) {
    prof_begin(KC_MISC, st);
    k_sm_to_nm<<<dim3(64, B), 256, 0, st>>>(xs, xs_tree_stride, out, out_tree_stride, R, C);
    LAUNCH_CHECK();
    return 0;
}

}  // namespace nnj
