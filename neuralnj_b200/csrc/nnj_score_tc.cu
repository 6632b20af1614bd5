// nnj_score_tc.cu — pair scoring on tcgen05 (precision bf16x3): the fused decode_gg kernel of the NJ loop.
//
// For every (pair, site) row the reference computes (model.py:90-99, 102-155)
//     x      = z*x_i + (1-z)*x_j                       (formed and stored as fp32 planes by k_alpha_v3)
//     x_glob = sum_r alpha[pair,r] * X[r,site,:]   \
//     g      = W_g x_glob + b_g = sum_r alpha[pair,r] * (W_g X[r,site,:]) + b_g   (sum_r alpha = 1)
//                                                       -> UMMA 1: [128 pairs x slots] . [slots x (64 | 64)]  (B MN-major, TMA)
//     w      = sigmoid(g);  x' = (1-w)*x + w*x_glob
//     score += w2 . GELU(W_s x' + b_s) + b2             -> UMMA 2: [128 x 64] . W_s^T
// G = W_g X is kept per node next to X in the node planes, which removes one GEMM and one operand round trip per row.
// One CTA = 128 pairs x 64 sites.  Sites alternate between two pipelines, each with its own TMEM accumulators
// ([x_glob | g]: 128 columns, s: 64), operand buffers and a group of 8 epilogue warps (4 TMEM lane quarters x 2 column
// halves); two control warps issue TMA + tcgen05.mma, so the tensor core works on one site while the CUDA cores run
// the sigmoid / blend / GELU epilogue of the other.  A tile of <= 64 pairs (the tail tile of step 0, e.g. 136 = 128 + 8 pairs at
// 17 taxa; later steps go to k_score_inc) has its pairs duplicated into rows 64..127 so that all four lane quarters - hence all
// 16 epilogue warps - have work.  Every product is split-bf16 (hi*hi + hi*lo + lo*hi, fp32 accumulate); operands produced on
// the fly are written by the epilogue threads straight into SWIZZLE_128B shared memory (validated by nnj_tc_selftest).  Node state
// for UMMA 1 comes from site-major bf16 planes [B][C][S][128] [X | W_g X], indexed by PHYSICAL slot, so alpha is scattered to slot
// order and dead / free slots simply get weight 0.
#include <cstdio>
#include <cstdlib>

#include "nnj_internal.h"
#include "nnj_tc.cuh"

namespace nnj {

constexpr int ST_THREADS = 576;            // 16 epilogue warps + 2 control warps
constexpr int ST_SITES = 64;               // sites per CTA
constexpr int ST_A0 = 0;                   // alpha operand   hi 16 KB | lo 16 KB
constexpr int ST_W = 32768;                // Ws_h, Ws_l: 2 x 8 KB
constexpr int ST_PIPE = 49152;             // per pipeline: [X|G]_h 16K | [X|G]_l 16K | A1_h 16K | A1_l 16K = 64 KB
constexpr int ST_PIPE_BYTES = 65536;
constexpr int ST_XT = ST_PIPE + 2 * ST_PIPE_BYTES;     // <= 64 pairs: per pipeline the site's x tile [64 pairs][64 ch] fp32 by TMA (2 x 8 KB halves)
constexpr int ST_MISC = ST_XT + 2 * 16384;             // biases (768 B) | part (4 KB) | barriers | tmem slot
constexpr int ST_SMEM = ST_MISC + 768 + 4096 + 256 + 1024;

struct ScoreTcArgs {
    const float4* xf;                      // x planes [B][pc][C][64] fp32 (written by k_alpha_v3)
    int pc;                                 // pairs capacity of the x planes
    const float* alpha; int RP;             // [B][PAIR_CHUNK][RP]
    int alpha_pairs;                        // PAIR_CHUNK stride of alpha / score_part
    const int32_t* slot_of; int slot_stride;
    const int32_t* pair_i; int pair_stride; int n0; int nc;
    int Rp, S, C;
    const uint4* wsh; const uint4* wsl;     // s_out.0 weight [64][64] as bf16 planes
    const float* bg; const float* bs; const float* w2; float b2;
    const uint8_t* mask;
    float* score_part; int nSG;
};

struct EpiCtx {
    uint64_t* pb; uint8_t* a1h; uint8_t* a1l; uint32_t t_d1; uint32_t t_s; uint32_t t_a1; const uint8_t* xt; uint64_t* x_full;
    const float* s_bias; int my_sites; int c_base; int p; int b;
};

// Epilogue of one warp over its sites.  NSUB 16-column sub-chunks per thread (2: one of two 32-column halves of a
// 128-pair tile; 1: one of four 16-column quarters when <= 64 pairs are duplicated into rows 64..127).
template <int NSUB>
__device__ __forceinline__ float score_epilogue(const ScoreTcArgs& a, const EpiCtx& e, int prow, int n, bool row_ok, int col0, bool dup) {
    const float* bgv = e.s_bias + col0;
    const float* bsv = e.s_bias + 64 + col0;
    const float* w2v = e.s_bias + 128 + col0;
    float score = 0.f;
    for (int i = 0; i < e.my_sites; ++i) {
        const uint32_t par = i & 1;
        const int c = e.c_base + 2 * i + e.p;
        const bool site_ok = !(a.mask && a.mask[(size_t)e.b * a.C + c]);      // loaded here, used after the GELU epilogue
        float4 x4[4 * NSUB];
        {
            // x tile of the site in shared memory (TMA, SWIZZLE_128B; 32-channel halves of [rows][128 B]): row prow, channels
            // [col0, col0 + 16 NSUB); rows without a pair were written as zeros / are zero-filled by the map
            mbar_wait(e.x_full, par);
            const uint8_t* xr = e.xt + (col0 >> 5) * (dup ? 8192 : 16384) + prow * 128;
#pragma unroll
            for (int j = 0; j < 4 * NSUB; ++j) x4[j] = *reinterpret_cast<const float4*>(xr + (((((col0 & 31) >> 2) + j) ^ (prow & 7)) << 4));
        }
        const float* xv = reinterpret_cast<const float*>(x4);
        // ---- gate: w = sigmoid(g + b_g), x' = (1-w) x + w x_glob  -> A1 operand of the s_out GEMM
        mbar_wait(e.pb + 1, par);
        tc_fence_after();
#pragma unroll
        for (int sub = 0; sub < NSUB; ++sub) {
            uint32_t g[16], xg[16];
            tmem_ld16_nw(e.t_d1 + 64 + col0 + sub * 16, g);
            tmem_ld16_nw(e.t_d1 + col0 + sub * 16, xg);
            tmem_ld_wait();
            float xp[16];
#pragma unroll
            for (int k = 0; k < 16; k += 2) {
                const float2 x2 = make_float2(xv[sub * 16 + k], xv[sub * 16 + k + 1]);
                const float2 w = sigmoid_fast2(fadd2(make_float2(__uint_as_float(g[k]), __uint_as_float(g[k + 1])), *reinterpret_cast<const float2*>(bgv + sub * 16 + k)));
                const float2 pp = ffma2(w, fsub2(make_float2(__uint_as_float(xg[k]), __uint_as_float(xg[k + 1])), x2), x2);   // (1-w) x + w x_glob
                xp[k] = pp.x; xp[k + 1] = pp.y;
            }
            if (dup) {
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    uint4 hh, ll;
                    split2(xp[8 * j + 0], xp[8 * j + 1], hh.x, ll.x);
                    split2(xp[8 * j + 2], xp[8 * j + 3], hh.y, ll.y);
                    split2(xp[8 * j + 4], xp[8 * j + 5], hh.z, ll.z);
                    split2(xp[8 * j + 6], xp[8 * j + 7], hh.w, ll.w);
                    const int off = prow * 128 + (((((col0 + sub * 16) >> 3) + j) ^ (prow & 7)) << 4);
                    *reinterpret_cast<uint4*>(e.a1h + off) = hh;
                    *reinterpret_cast<uint4*>(e.a1l + off) = ll;
                    *reinterpret_cast<uint4*>(e.a1h + off + 8192) = hh;      // rows 64..127 repeat the pairs
                    *reinterpret_cast<uint4*>(e.a1l + off + 8192) = ll;
                }
            } else {
                // a full tile keeps the A1 operand in tensor memory (row = this thread's TMEM lane, two bf16 per column)
                uint32_t hh[8], ll[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) split2(xp[2 * j], xp[2 * j + 1], hh[j], ll[j]);
                tmem_st8(e.t_a1 + ((col0 + sub * 16) >> 1), hh);
                tmem_st8(e.t_a1 + 32 + ((col0 + sub * 16) >> 1), ll);
            }
        }
        if (!dup) tmem_st_wait();
        fence_async_smem();
        tc_fence_before();
        __syncwarp();
        if ((threadIdx.x & 31) == 0) mbar_arrive(e.pb + 2);
        // ---- score: w2 . GELU(s + b_s) (+ b2 once per row), masked site sum
        mbar_wait(e.pb + 3, par);
        tc_fence_after();
        float2 acc = make_float2(0.f, 0.f);
#pragma unroll
        for (int sub = 0; sub < NSUB; ++sub) {
            uint32_t sv[16];
            tmem_ld16_nw(e.t_s + col0 + sub * 16, sv);
            tmem_ld_wait();
#pragma unroll
            for (int k = 0; k < 16; k += 2) {
                const float2 sb = fadd2(make_float2(__uint_as_float(sv[k]), __uint_as_float(sv[k + 1])), *reinterpret_cast<const float2*>(bsv + sub * 16 + k));
                acc = ffma2(gelu_fast2(sb), *reinterpret_cast<const float2*>(w2v + sub * 16 + k), acc);
            }
        }
        tc_fence_before();
        if (site_ok) score += (acc.x + acc.y) + (col0 == 0 ? a.b2 : 0.f);
    }
    return row_ok ? score : 0.f;
}

__global__ void __launch_bounds__(ST_THREADS, 1)
k_score_tc(const __grid_constant__ CUtensorMap mapXh, const __grid_constant__ CUtensorMap mapXl, const __grid_constant__ CUtensorMap mapXf,
           const ScoreTcArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* sm = smem_align1024(smem_raw);
    float* s_bias = reinterpret_cast<float*>(sm + ST_MISC);            // bg[64] | bs[64] | w2[64]
    float* s_part = s_bias + 192;                                       // [2 pipelines][4 column slots][128]
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_part + 1024);        // per pipeline: bx_full, d1_done, a1_ready, s_done; then x_full[2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 10);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b = blockIdx.z, pt = blockIdx.y, sg = blockIdx.x;
    const int rows_here = min(128, a.nc - pt * 128);
    const bool dup = rows_here <= 64;                                   // pairs duplicated into rows 64..127: all 16 warps stay busy
    const int act_warps = dup ? (rows_here > 32 ? 8 : 4) : 2 * ((rows_here + 31) >> 5);   // per pipeline
    const int c_base = sg * ST_SITES;
    const int n_sites = min(ST_SITES, a.C - c_base);

    // ---- one-time setup
    if (tid == 0) {
        for (int p = 0; p < 2; ++p) {
            uint64_t* pb = bars + p * 4;
            mbar_init(pb + 0, 1); mbar_init(pb + 1, 1); mbar_init(pb + 2, act_warps); mbar_init(pb + 3, 1); mbar_init(bars + 8 + p, 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 16) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    for (int i = tid; i < 2048; i += ST_THREADS) reinterpret_cast<uint4*>(sm + ST_A0)[i] = make_uint4(0u, 0u, 0u, 0u);
    for (int i = tid; i < 1024; i += ST_THREADS) {                      // W_s -> swizzled K-major tiles (hi, lo)
        const int plane = i >> 9, rem = i & 511, row = rem >> 3, j = rem & 7;
        const uint4* src = plane == 0 ? a.wsh : a.wsl;
        *reinterpret_cast<uint4*>(sm + ST_W + plane * 8192 + row * 128 + ((j ^ (row & 7)) << 4)) = __ldg(src + rem);
    }
    for (int i = tid; i < 1024; i += ST_THREADS) s_part[i] = 0.f;
    if (tid < 64) { s_bias[tid] = a.bg[tid]; s_bias[64 + tid] = a.bs[tid]; s_bias[128 + tid] = a.w2[tid]; }
    __syncthreads();
    {   // alpha scattered to physical-slot order: A0[row][slot] (K-major, 64 slots = one 128 B swizzle row)
        const int32_t* so = a.slot_of + (size_t)b * a.slot_stride;
        for (int idx = tid; idx < rows_here * a.Rp; idx += ST_THREADS) {
            const int row = idx / a.Rp, r = idx - row * a.Rp;
            const float v = a.alpha[((size_t)b * a.alpha_pairs + pt * 128 + row) * a.RP + r];
            const int slot = so[r];
            const __nv_bfloat16 h = __float2bfloat16_rn(v), l = NNJ_LO_BF16(__float2bfloat16_rn(v - __bfloat162float(h)));
            const int off = row * 128 + (((slot >> 3) ^ (row & 7)) << 4) + (slot & 7) * 2;
            *reinterpret_cast<__nv_bfloat16*>(sm + ST_A0 + off) = h;
            *reinterpret_cast<__nv_bfloat16*>(sm + ST_A0 + 16384 + off) = l;
            if (dup) {
                *reinterpret_cast<__nv_bfloat16*>(sm + ST_A0 + off + 8192) = h;
                *reinterpret_cast<__nv_bfloat16*>(sm + ST_A0 + 16384 + off + 8192) = l;
            }
        }
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp >= 16) {
        // ================= control warp of pipeline p: TMA + MMA issue (warp-uniform, one elected lane per action) =================
        const int p = warp - 16;
        uint64_t* pb = bars + p * 4;
        uint8_t* pipe = sm + ST_PIPE + p * ST_PIPE_BYTES;
        const uint32_t a0h = smem_u32(sm + ST_A0), a0l = a0h + 16384;
        const uint32_t wsh = smem_u32(sm + ST_W), wsl = wsh + 8192;
        const uint32_t bxh = smem_u32(pipe), bxl = bxh + 16384, a1h = bxh + 32768, a1l = bxh + 49152;
        const uint32_t t_d1 = tmem_base + p * 256, t_s = t_d1 + 128, t_a1 = t_d1 + 192;   // [x_glob | g] 128 | s 64 | A1 hi 32 | A1 lo 32
        const uint32_t id_s = umma_idesc_bf16(128, 64), id_d1 = umma_idesc_bf16(128, 128) | (1u << 16);
        const int ksteps = (a.S + 15) >> 4;
        const int my_sites = (n_sites - p + 1) >> 1;
        uint8_t* xt = dup ? sm + ST_XT + p * 16384 : pipe + 32768;   // a full tile has its A1 operand in TMEM: the x tile takes that space
        auto load_x = [&](int c) {      // one elected lane
            if (dup) {
                mbar_expect_tx(bars + 8 + p, 16384);
                tma_load_4d(xt, &mapXf, bars + 8 + p, 0, c, pt * 128, b);
                tma_load_4d(xt + 8192, &mapXf, bars + 8 + p, 32, c, pt * 128, b);
            } else {
                mbar_expect_tx(bars + 8 + p, 32768);
                tma_load_4d(xt, &mapXf, bars + 8 + p, 0, c, pt * 128, b);
                tma_load_4d(xt + 8192, &mapXf, bars + 8 + p, 0, c, pt * 128 + 64, b);
                tma_load_4d(xt + 16384, &mapXf, bars + 8 + p, 32, c, pt * 128, b);
                tma_load_4d(xt + 24576, &mapXf, bars + 8 + p, 32, c, pt * 128 + 64, b);
            }
        };
        if (my_sites > 0 && elect_one()) load_x(c_base + p);
        if (my_sites > 0 && elect_one()) {
            const int c = c_base + p;
            mbar_expect_tx(pb + 0, 32768);
            tma_load_3d(pipe, &mapXh, pb + 0, 0, 0, b * a.C + c);
            tma_load_3d(pipe + 8192, &mapXh, pb + 0, 64, 0, b * a.C + c);
            tma_load_3d(pipe + 16384, &mapXl, pb + 0, 0, 0, b * a.C + c);
            tma_load_3d(pipe + 24576, &mapXl, pb + 0, 64, 0, b * a.C + c);
        }
        __syncwarp();
        for (int i = 0; i < my_sites; ++i) {
            const uint32_t par = i & 1;
            mbar_wait(pb + 0, par);
            tc_fence_after();
            if (elect_one()) {      // [x_glob | g] = alpha . [X | W_g X]   (B MN-major: 16 slots = 2048 B per k-step, column blocks 8 KB apart)
                for (int k = 0; k < ksteps; ++k) {
                    umma_bf16(t_d1, umma_desc_k128(a0l + k * 32), umma_desc_lbo(bxh + k * 2048, 8192), id_d1, k ? 1u : 0u);
                    umma_bf16(t_d1, umma_desc_k128(a0h + k * 32), umma_desc_lbo(bxl + k * 2048, 8192), id_d1, 1u);
                    umma_bf16(t_d1, umma_desc_k128(a0h + k * 32), umma_desc_lbo(bxh + k * 2048, 8192), id_d1, 1u);
                }
                umma_commit(pb + 1);
            }
            __syncwarp();
            if (i + 1 < my_sites) {     // prefetch the next node tile as soon as UMMA 1 has retired (hides the HBM/L2 latency)
                mbar_wait(pb + 1, par);
                if (elect_one()) {
                    const int c = c_base + 2 * (i + 1) + p;
                    mbar_expect_tx(pb + 0, 32768);
                    tma_load_3d(pipe, &mapXh, pb + 0, 0, 0, b * a.C + c);
                    tma_load_3d(pipe + 8192, &mapXh, pb + 0, 64, 0, b * a.C + c);
                    tma_load_3d(pipe + 16384, &mapXl, pb + 0, 0, 0, b * a.C + c);
                    tma_load_3d(pipe + 24576, &mapXl, pb + 0, 64, 0, b * a.C + c);
                }
                __syncwarp();
            }
            mbar_wait(pb + 2, par);     // epilogue has consumed [x_glob | g] and the x tile, and written x' into the A1 operand
            tc_fence_after();
            if (i + 1 < my_sites && elect_one()) load_x(c_base + 2 * (i + 1) + p);   // next x tile of this pipeline
            if (elect_one()) {
                if (dup) {
                    for (int k = 0; k < 4; ++k) {   // s = x' . W_s^T
                        umma_bf16(t_s, umma_desc_k128(a1l + k * 32), umma_desc_k128(wsh + k * 32), id_s, k ? 1u : 0u);
                        umma_bf16(t_s, umma_desc_k128(a1h + k * 32), umma_desc_k128(wsl + k * 32), id_s, 1u);
                        umma_bf16(t_s, umma_desc_k128(a1h + k * 32), umma_desc_k128(wsh + k * 32), id_s, 1u);
                    }
                } else {
                    for (int k = 0; k < 4; ++k) {   // the same with x' read from tensor memory
                        umma_bf16_ta(t_s, t_a1 + 32 + k * 8, umma_desc_k128(wsh + k * 32), id_s, k ? 1u : 0u);
                        umma_bf16_ta(t_s, t_a1 + k * 8, umma_desc_k128(wsl + k * 32), id_s, 1u);
                        umma_bf16_ta(t_s, t_a1 + k * 8, umma_desc_k128(wsh + k * 32), id_s, 1u);
                    }
                }
                umma_commit(pb + 3);
            }
            __syncwarp();
        }
    } else {
        // ================= epilogue warps: pipeline p = warp / 8, TMEM lane quarter q, column half hf =================
        const int p = warp >> 3, q = warp & 3, hf = (warp >> 2) & 1;
        const bool active = dup ? ((q & 1) * 32 < rows_here) : (q * 32 < rows_here);
        if (active) {
            uint8_t* pipe = sm + ST_PIPE + p * ST_PIPE_BYTES;
            EpiCtx e;
            e.pb = bars + p * 4; e.a1h = pipe + 32768; e.a1l = pipe + 49152; e.xt = dup ? sm + ST_XT + p * 16384 : pipe + 32768; e.x_full = bars + 8 + p;
            e.t_d1 = tmem_base + ((uint32_t)(q * 32) << 16) + p * 256; e.t_s = e.t_d1 + 128; e.t_a1 = e.t_d1 + 192;
            e.s_bias = s_bias; e.my_sites = (n_sites - p + 1) >> 1; e.c_base = c_base; e.p = p; e.b = b;
            const int prow = dup ? ((q & 1) * 32 + lane) : (q * 32 + lane);
            const int n = pt * 128 + prow;
            const bool row_ok = n < a.nc && a.pair_i[(size_t)b * a.pair_stride + a.n0 + n] >= 0;
            if (dup) {
                const int cq = (q >> 1) * 2 + hf;
                s_part[(p * 4 + cq) * 128 + prow] = score_epilogue<1>(a, e, prow, n, row_ok, cq * 16, true);
            } else {
                s_part[(p * 4 + hf) * 128 + prow] = score_epilogue<2>(a, e, prow, n, row_ok, hf * 32, false);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (tid < rows_here) {
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) s += s_part[k * 128 + tid];
        a.score_part[((size_t)b * a.alpha_pairs + pt * 128 + tid) * a.nSG + sg] = s;
    }
    if (warp == 16) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
    }
}

// ------------------------------------------------------------------ host side

int make_tmap_nodes(CUtensorMap* map, const void* base, int S, int BC, int box_rows, int n_live) {
    const cuuint64_t gdim[3] = {128, (cuuint64_t)(n_live > 0 ? n_live : S), (cuuint64_t)BC};   // slots >= n_live are dead: zero-filled, never loaded
    const cuuint64_t gstr[2] = {256, (cuuint64_t)S * 256};
    const cuuint32_t box[3] = {64, (cuuint32_t)box_rows, 1};
    return encode_tmap(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, gdim, gstr, box, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                       "the node planes");
}

int make_tmap_xtile(CUtensorMap* map, const float* base, int pc, int nrows, int C, int B, int box_rows) {
    const cuuint64_t gdim[4] = {64, (cuuint64_t)C, (cuuint64_t)nrows, (cuuint64_t)B};
    const cuuint64_t gstr[3] = {256, (cuuint64_t)C * 256, (cuuint64_t)pc * C * 256};
    const cuuint32_t box[4] = {32, 1, (cuuint32_t)box_rows, 1};
    return encode_tmap(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, base, gdim, gstr, box, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                       "the x tiles");
}

int launch_score_tc(const Model* m, const PairChunk& c, int* n_part, cudaStream_t st) {
    static DevOnce once;      // per device, not per process
    if (int e = smem_opt_in(once, k_score_tc, ST_SMEM)) return e;
    if (c.S > 64) return set_error(NNJ_ERR_INVALID, "score_tc: at most 63 taxa on the tensor-core pair-score path");
    *n_part = (c.C + ST_SITES - 1) / ST_SITES;
    CUtensorMap mh, ml, mx;
    if (int e = make_tmap_xtile(&mx, c.xf, c.pc, c.nc, c.C, c.B)) return e;
    if (int e = make_tmap_nodes(&mh, c.nodes_h, c.S, c.B * c.C)) return e;
    if (int e = make_tmap_nodes(&ml, c.nodes_l, c.S, c.B * c.C)) return e;
    ScoreTcArgs a;
    a.xf = (const float4*)c.xf; a.pc = c.pc;
    a.alpha = c.alpha; a.RP = c.RP; a.alpha_pairs = c.alpha_pairs;
    a.slot_of = c.slot_of; a.slot_stride = c.slot_stride; a.pair_i = c.pair_i; a.pair_stride = c.pair_stride; a.n0 = c.n0; a.nc = c.nc;
    a.Rp = c.Rp; a.S = c.S; a.C = c.C;
    a.wsh = (const uint4*)m->nj_bf.wsh; a.wsl = (const uint4*)m->nj_bf.wsl;
    a.bg = m->nj.bg; a.bs = m->nj.bs; a.w2 = m->nj.w2; a.b2 = m->nj.b2;
    a.mask = c.mask; a.score_part = c.score_part; a.nSG = c.nSB;
    prof_begin(KC_SCORE, st);
    k_score_tc<<<dim3((c.C + ST_SITES - 1) / ST_SITES, (c.nc + 127) / 128, c.B), ST_THREADS, ST_SMEM, st>>>(mh, ml, mx, a);
    LAUNCH_CHECK();
    return 0;
}

}  // namespace nnj
