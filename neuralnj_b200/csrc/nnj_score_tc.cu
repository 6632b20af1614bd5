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

// ------------------------------------------------------------------ incremental steps: <= 64 pairs per tree
// Every NJ step after the first scores only the pairs of the new node (<= R-1 <= 63 rows), and the 48 of them dominate the loop.
// k_score_inc is the pair-score kernel for that regime, persistent over work items (tree, 128-site group):
//   * the 128-row tile is split by site parity like k_alpha_v3: lanes 0..63 = the pairs at site 2k, lanes 64..127 = the same
//     pairs at site 2k+1.  UMMA 1 runs once per site into its own accumulator ([x_glob | g] of site 2k in D1a rows 0..63,
//     of site 2k+1 in D1b rows 64..127; the other halves are ignored); UMMA 2 (x' . W_s^T) runs ONCE for both sites, its A
//     operand x' written by the epilogue threads straight into tensor memory (no shared-memory staging, no row duplication);
//   * a producer warp streams the node tiles ([X | W_g X] bf16 hi/lo) and the x tiles of the sites through a ring sized from
//     the slot / pair counts (4 sites at 51 slots), running ahead across work items, so the kernel can follow HBM;
//   * the issue warp queues UMMA 1 of the next site pair right behind UMMA 2 of the current one, so the tensor core works on
//     the next [x_glob | g] while the 16 epilogue warps run the GELU / site-sum epilogue.
// The alpha operand (A of UMMA 1) is rebuilt per work item from alpha[b] scattered to physical-slot order.
// With <= 32 pairs (narrow mode, see the epilogue warps) lanes 32..63 / 96..127 repeat the pairs and share their channels.
constexpr int SI_THREADS = 608;            // 16 epilogue warps + issue warp + node-tile producer + x-tile producer
constexpr int SI_SITES = 128;               // sites per work item (the pipeline drains at every work-item boundary)
constexpr int SI_A0 = 0;                   // staging of alpha by physical slot, fp32 [64 pairs][68] (the operand itself lives in tensor memory)
constexpr int SI_A0_LD = 68;
constexpr int SI_XCH = 9216;               // narrow mode (<= 32 pairs): x' word exchange between the two warps of a (half, column group), 16 KB behind the 32-row alpha staging
constexpr int SI_W = 32768;                // W_s hi 8 KB | lo 8 KB
constexpr int SI_RING = 49152;
constexpr int SI_MAXST = 6;
constexpr int SI_MISC_BYTES = 768 + 2048 + 512;   // biases | score partials [4][128] | barriers (4 x 6 + 7), tmem slot
constexpr int SI_SMEM_MAX = 232448;
constexpr uint32_t SI_TM_D1 = 0, SI_TM_S = 256, SI_TM_A1 = 320, SI_TM_A0 = 448;   // TMEM: D1a 128 | D1b 128 | s 64 | x'[0] hi/lo 64 | x'[1] hi/lo 64 | alpha hi/lo 64
// The x' operand of UMMA 2 is double-buffered by item parity and s is single: the gate epilogue of item k+1 then never waits for UMMA 2 of
// item k (with one x' buffer it did, and the ~2700 clk from "gate done" over "both halves ready -> UMMA 2 issued -> retired" to the next
// gate exceeded the ~1500 clk GELU epilogue that was meant to fill it: 1250 idle clk of a 4170 clk item period, profiles/r01_score_inc_experiments.txt).
// UMMA 2 of item k now waits for the GELU epilogue of item k-1 to have drained s (s_free) and runs while the warps work on gate k+1.

// Timing experiments (clock64 timeline of CTA 0, partial-math modes that give WRONG scores) exist only in builds made with
// -DNNJ_DEBUG_TOOLS; the default library reads none of NNJ_SCORE_TRACE / NNJ_SCORE_DBG / NNJ_SCORE_PF.
#ifdef NNJ_DEBUG_TOOLS
#define SI_TRACE(tag, item) do { if (a.trace && blockIdx.x == 0 && lane == 0 && (item) < 600) a.trace[(tag) * 600 + (item)] = clock64(); } while (0)
#define SI_DBG(a) ((a).dbg)
#else
#define SI_TRACE(tag, item) do { } while (0)
#define SI_DBG(a) 0
#endif

struct ScoreIncArgs {
    const float* alpha; int RP; int alpha_pairs;
    const int32_t* slot_of; int slot_stride;
    const int32_t* pair_i; int pair_stride; int n0; int nc;
    int Rp, S, C, B, groups;
#ifdef NNJ_DEBUG_TOOLS
    long long* trace;                        // NNJ_SCORE_TRACE: clock64 stamps of CTA 0 (tag, item, clock) triples, else null
    int dbg;                                 // timing experiments only (NNJ_SCORE_DBG): 2 = no gate math, 4 = no GELU math
#endif
    int narrow;                              // nc <= 32: lanes 32..63 of a half repeat the pairs; the two warps of a (half, column group) split its 16 channels
    int node_rows, x_rows, nst;              // ring geometry: node blocks [node_rows][128 B] x 4, x halves [x_rows][128 B] x 2
    const uint4* wsh; const uint4* wsl;
    const float* bg; const float* bs; const float* w2; float b2;
    const uint8_t* mask;
    float* score_part; int nSG;
};

__global__ void __launch_bounds__(SI_THREADS, 1)
k_score_inc(const __grid_constant__ CUtensorMap mapXh, const __grid_constant__ CUtensorMap mapXl, const __grid_constant__ CUtensorMap mapXf,
            const ScoreIncArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* sm = smem_align1024(smem_raw);
    const int NB = a.node_rows * 128, XB = a.x_rows * 128;      // bytes of one node column block / one x half
    const int STG = 4 * NB + 2 * XB, NST = a.nst;               // per site: node blocks X_h | G_h | X_l | G_l, x halves ch 0-31 | ch 32-63
    // Ring layout: [NST][4 node blocks] | 1 KB of zeros | [NST][2 x halves].  UMMA 1 reads 16 slot rows per k-step, up to 64, from
    // blocks of node_rows (>= slots, multiple of 8) rows: what lies behind a block must be finite bf16 (0 x NaN would poison
    // the accumulator) - the next node block, or the zero pad behind the last one; never the fp32 x tiles.
    uint8_t* ring = sm + SI_RING;
    uint8_t* xring = ring + NST * 4 * NB + 1024;
    float* s_bias = reinterpret_cast<float*>(ring + NST * STG + 1024);
    float* s_part = s_bias + 192;                                          // [4 column groups][128 rows]
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_part + 512);
    // the node tiles (freed by UMMA 1) and the x tiles (freed by the gate epilogue) run as two rings with their own barriers, so a
    // node stage is refilled as soon as its UMMA 1 has retired, one item earlier than the x tile of the same site
    uint64_t *full = bars, *stage_free = bars + SI_MAXST, *x_full = bars + 2 * SI_MAXST, *x_free = bars + 3 * SI_MAXST,
             *a0_ready = bars + 4 * SI_MAXST, *d1_done = a0_ready + 1, *a1_ready = d1_done + 2, *s_done = a1_ready + 2, *s_free = s_done + 1;   // d1_done[2] a1_ready[2] s_done s_free
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_done + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_work = a.B * a.groups;

    if (tid == 0) {
        for (int i = 0; i < NST; ++i) { mbar_init(full + i, 1); mbar_init(stage_free + i, 1); mbar_init(x_full + i, 1); mbar_init(x_free + i, 8); }
        mbar_init(a0_ready, 16); mbar_init(d1_done, 1); mbar_init(d1_done + 1, 1); mbar_init(a1_ready, 8); mbar_init(a1_ready + 1, 8);
        mbar_init(s_done, 1); mbar_init(s_free, 16);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 16) tmem_alloc(tmem_slot, 512);
    // the ring (and the pad behind it) starts as zeros: slot rows past the tile read by UMMA 1 must be finite
    for (int i = tid; i < (NST * STG + 1024) >> 4; i += SI_THREADS) reinterpret_cast<uint4*>(ring)[i] = make_uint4(0u, 0u, 0u, 0u);
    for (int i = tid; i < 1024; i += SI_THREADS) {                      // W_s -> swizzled K-major tiles (hi, lo)
        const int plane = i >> 9, rem = i & 511, row = rem >> 3, j = rem & 7;
        const uint4* src = plane == 0 ? a.wsh : a.wsl;
        *reinterpret_cast<uint4*>(sm + SI_W + plane * 8192 + row * 128 + ((j ^ (row & 7)) << 4)) = __ldg(src + rem);
    }
    if (tid < 64) { s_bias[tid] = a.bg[tid]; s_bias[64 + tid] = a.bs[tid]; s_bias[128 + tid] = a.w2[tid]; }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp >= 17) {
        // ================= producer warps: 17 streams the node tiles, 18 the x tiles, one site per ring stage =================
        const bool nodes = warp == 17;
        uint64_t* fullb = nodes ? full : x_full;
        uint64_t* freeb = nodes ? stage_free : x_free;
        int st = 0; uint32_t ph = 0; int gs = 0;
        for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
            const int b = w / a.groups, sg = w - b * a.groups;
            const int c_base = sg * SI_SITES, n_sites = min(SI_SITES, a.C - c_base);
            for (int s = 0; s < n_sites; ++s, ++gs) {
                if (gs >= NST) mbar_wait(freeb + st, ph ^ 1u);
                SI_TRACE(nodes ? 1 : 2, gs);
                if (elect_one()) {
                    const int c = c_base + s;
                    if (nodes) {
                        uint8_t* stg = ring + st * 4 * NB;
                        mbar_expect_tx(full + st, 4 * NB);
                        tma_load_3d(stg, &mapXh, full + st, 0, 0, b * a.C + c);
                        tma_load_3d(stg + NB, &mapXh, full + st, 64, 0, b * a.C + c);
                        tma_load_3d(stg + 2 * NB, &mapXl, full + st, 0, 0, b * a.C + c);
                        tma_load_3d(stg + 3 * NB, &mapXl, full + st, 64, 0, b * a.C + c);
                    } else {
                        uint8_t* xt = xring + st * 2 * XB;
                        mbar_expect_tx(x_full + st, 2 * XB);
                        tma_load_4d(xt, &mapXf, x_full + st, 0, c, 0, b);
                        tma_load_4d(xt + XB, &mapXf, x_full + st, 32, c, 0, b);
                    }
                }
                __syncwarp();
                if (++st == NST) { st = 0; ph ^= 1u; }
            }
        }
        (void)fullb;
    } else if (warp == 16) {
        // ================= issue warp =================
        const uint32_t wsh = smem_u32(sm + SI_W), wsl = wsh + 8192;
        const uint32_t id_s = umma_idesc_bf16(128, 64), id_d1 = umma_idesc_bf16(128, 128) | (1u << 16);
        const int ksteps = (a.S + 15) >> 4;
        int st = 0; uint32_t ph = 0;
        uint32_t gi = 0, wi = 0;        // items / work items so far (phases of a1_ready, a0_ready)
        for (int w = blockIdx.x; w < n_work; w += gridDim.x, ++wi) {
            const int sg = w % a.groups;
            const int n_sites = min(SI_SITES, a.C - sg * SI_SITES);
            const int n_items = (n_sites + 1) >> 1;
            mbar_wait(a0_ready, wi & 1u);
            // The two sites of an item are two half-pipelines: while the 8 epilogue warps of one half run the gate epilogue on their
            // accumulator (D1a / D1b), the tensor core refills the other one.  Issue order: U1a(0) U1b(0), then per item k:
            //   [half A done with D1a(k)] U1a(k+1)   [half B done with D1b(k)] U1b(k+1)   [GELU epilogue of item k-1 done] U2(k)
            // (sites stay in ring order A(k) B(k) A(k+1) ...).  [x_glob | g] = alpha . [X | W_g X]: alpha from TENSOR MEMORY (a 128 x 128
            // x 16 UMMA costs ~75 clk with A in TMEM against ~107 clk from shared memory), B MN-major from the node ring.
            auto issue_u1 = [&](int h) {
                mbar_wait(full + st, ph);
                tc_fence_after();
                if (elect_one()) {
                    // 16 slots = 2048 B per k-step, column blocks NB apart; descriptor low words advance by plain adds
                    const uint32_t bh = umma_desc_lo(smem_u32(ring + st * 4 * NB), NB), bl = umma_desc_lo(smem_u32(ring + st * 4 * NB + 2 * NB), NB);
                    const uint32_t ta0 = tmem_base + SI_TM_A0;
                    const uint32_t td = tmem_base + SI_TM_D1 + h * 128;
                    umma_ts<false>(td, ta0 + 32, bh, id_d1);
                    umma_ts<true>(td, ta0, bl, id_d1);
                    umma_ts<true>(td, ta0, bh, id_d1);
#pragma unroll
                    for (int kk = 1; kk < 4; ++kk) {
                        if (kk < ksteps) {
                            umma_ts<true>(td, ta0 + 32 + kk * 8, bh + kk * 128, id_d1);
                            umma_ts<true>(td, ta0 + kk * 8, bl + kk * 128, id_d1);
                            umma_ts<true>(td, ta0 + kk * 8, bh + kk * 128, id_d1);
                        }
                    }
                    umma_commit(stage_free + st);
                    umma_commit(d1_done + h);
                }
                __syncwarp();
                if (++st == NST) { st = 0; ph ^= 1u; }
            };
            issue_u1(0);
            if (n_sites > 1) issue_u1(1);
            for (int k = 0; k < n_items; ++k, ++gi) {
                mbar_wait(a1_ready, gi & 1u);           // half A has read D1a and written its x' rows
                SI_TRACE(4, (int)gi);
                if (2 * (k + 1) < n_sites) issue_u1(0);
                mbar_wait(a1_ready + 1, gi & 1u);       // half B likewise (it arrives with zeros when the item has no second site)
                if (2 * (k + 1) + 1 < n_sites) issue_u1(1);     // both D1 accumulators are refilled before UMMA 2 waits for the GELU epilogue
                if (gi >= 1) mbar_wait(s_free, (gi - 1) & 1u);   // all 16 epilogue warps have read s of the previous item
                SI_TRACE(5, (int)gi);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t ta = tmem_base + SI_TM_A1 + (gi & 1u) * 64, ts = tmem_base + SI_TM_S;
                    const uint32_t wh = umma_desc_lo(wsh), wl = umma_desc_lo(wsl);
                    umma_ts<false>(ts, ta + 32, wh, id_s);          // s = x' . W_s^T for both sites at once; small terms first
                    umma_ts<true>(ts, ta, wl, id_s);
                    umma_ts<true>(ts, ta, wh, id_s);
#pragma unroll
                    for (int kk = 1; kk < 4; ++kk) {
                        umma_ts<true>(ts, ta + 32 + kk * 8, wh + kk * 2, id_s);
                        umma_ts<true>(ts, ta + kk * 8, wl + kk * 2, id_s);
                        umma_ts<true>(ts, ta + kk * 8, wh + kk * 2, id_s);
                    }
                    umma_commit(s_done);
                }
                __syncwarp();
                SI_TRACE(6, (int)gi);
            }
        }
    } else {
        // ================= epilogue warps: TMEM lane quarter q (lanes < 64: site 2k, else site 2k+1), 16 columns cg =================
        const int q = warp & 3, cg = warp >> 2, h = q >> 1;
        // narrow mode (<= 32 pairs): rows 32..63 of a half would idle, and with them two of the four SM sub-partitions.  Instead they
        // repeat rows 0..31 (same alpha rows, same x rows), and the two warps (q even / odd) of a (half, column group) each take 8 of the
        // group's 16 channels in both epilogues; the packed x' words are swapped through shared memory so that both lanes of a pair
        // carry the complete x' row into UMMA 2.
        const bool narrow = a.narrow != 0;
        const int sub = q & 1;
        const int prow = narrow ? lane : (q & 1) * 32 + lane;       // pair row
        const bool warp_rows = narrow || (q & 1) * 32 < a.nc;       // this warp's rows hold listed pairs
        uint4* xch = reinterpret_cast<uint4*>(sm + SI_XCH) + (h * 4 + cg) * 128;      // [sub][hi | lo][32 lanes]
        const int xch_bar = 2 + h * 4 + cg;                         // named barrier of the warp pair
        const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
        const float* bgv = s_bias + cg * 16;
        const float* bsv = s_bias + 64 + cg * 16;
        const float* w2v = s_bias + 128 + cg * 16;
        int st = 0; uint32_t ph = 0;
        uint32_t gi = 0, c_d1 = 0;      // items so far; UMMA-1 completions of this half so far (phase of d1_done[h])
        for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
            const int b = w / a.groups, sg = w - b * a.groups;
            const int c_base = sg * SI_SITES, n_sites = min(SI_SITES, a.C - c_base);
            const int n_items = (n_sites + 1) >> 1;
            // ---- alpha operand of this tree: alpha[b][pair][r] scattered to physical-slot order through a shared-memory table, then
            //      split into bf16 hi / lo and stored to tensor memory by the row's own threads (lanes 64.. repeat the pairs)
            {
                float* tab = reinterpret_cast<float*>(sm + SI_A0);
                for (int i = tid; i < (narrow ? 32 : 64) * SI_A0_LD / 4; i += 512) reinterpret_cast<float4*>(tab)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
                asm volatile("bar.sync 1, 512;" ::: "memory");
                const int32_t* so = a.slot_of + (size_t)b * a.slot_stride;
                for (int idx = tid; idx < a.nc * a.Rp; idx += 512) {
                    const int row = idx / a.Rp, r = idx - row * a.Rp;
                    tab[row * SI_A0_LD + so[r]] = a.alpha[((size_t)b * a.alpha_pairs + row) * a.RP + r];
                }
                asm volatile("bar.sync 1, 512;" ::: "memory");
                uint32_t hh[8], ll[8];
                const float* tr = tab + prow * SI_A0_LD + cg * 16;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float4 v = *reinterpret_cast<const float4*>(tr + 4 * e);
                    split2(v.x, v.y, hh[2 * e], ll[2 * e]);
                    split2(v.z, v.w, hh[2 * e + 1], ll[2 * e + 1]);
                }
                tmem_st8(lane_base + SI_TM_A0 + cg * 8, hh);
                tmem_st8(lane_base + SI_TM_A0 + 32 + cg * 8, ll);
                tmem_st_wait();
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(a0_ready);
            const bool row_ok = prow < a.nc && a.pair_i[(size_t)b * a.pair_stride + a.n0 + prow] >= 0;
            float score = 0.f;
            // w2 . GELU(s + b_s) (+ b2 once per row), masked site sum, for item `it` (global count) whose site of this thread is `site`
            auto ep2 = [&](uint32_t it, int site) {
                const bool unmasked = site < n_sites && !(a.mask && a.mask[(size_t)b * a.C + c_base + site]);   // loaded before the wait
                mbar_wait(s_done, it & 1u);
                tc_fence_after();
                if (narrow && !(SI_DBG(a) & 4)) {
                    uint32_t sv[8];
                    tmem_ld8_nw(lane_base + SI_TM_S + cg * 16 + sub * 8, sv);
                    tmem_ld_wait();
                    float2 acc = make_float2(0.f, 0.f);
#pragma unroll
                    for (int e = 0; e < 8; e += 2) {
                        const float2 sb = fadd2(make_float2(__uint_as_float(sv[e]), __uint_as_float(sv[e + 1])), *reinterpret_cast<const float2*>(bsv + sub * 8 + e));
                        acc = ffma2(gelu_fast2(sb), *reinterpret_cast<const float2*>(w2v + sub * 8 + e), acc);
                    }
                    if (unmasked) score += (acc.x + acc.y) + ((cg | sub) == 0 ? a.b2 : 0.f);
                } else if (warp_rows && !(SI_DBG(a) & 4)) {
                    uint32_t sv[16];
                    tmem_ld16_nw(lane_base + SI_TM_S + cg * 16, sv);
                    tmem_ld_wait();
                    float2 acc = make_float2(0.f, 0.f);          // packed fp32x2 math: channel pairs (e, e+1) share every FMA-pipe instruction
#pragma unroll
                    for (int e = 0; e < 16; e += 2) {
                        const float2 sb = fadd2(make_float2(__uint_as_float(sv[e]), __uint_as_float(sv[e + 1])), *reinterpret_cast<const float2*>(bsv + e));
                        acc = ffma2(gelu_fast2(sb), *reinterpret_cast<const float2*>(w2v + e), acc);
                    }
                    if (unmasked) score += (acc.x + acc.y) + (cg == 0 ? a.b2 : 0.f);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(s_free);      // s may be overwritten by UMMA 2 of the next item
                if (warp == 0 || warp == 2) SI_TRACE(14 + 5 * warp, (int)it);
            };
            for (int k = 0; k < n_items; ++k, ++gi) {
                // The halves run decoupled (ping-pong), so a warp may wait only on the x stages its own half releases: the ring depth is
                // even and every work item starts on an even ring position, hence even stages always hold the first site of an item
                // (half A) and odd stages the second (half B), and a warp sees every phase of the stages it looks at.
                int st1 = st; uint32_t ph1 = ph;
                if (++st1 == NST) { st1 = 0; ph1 ^= 1u; }
                const bool two = 2 * k + 1 < n_sites;
                const int site = 2 * k + h;
                const bool site_ok = site < n_sites;
                const int my_st = h ? st1 : st;
                if (site_ok) mbar_wait(x_full + my_st, h ? ph1 : ph);
                if (++st == NST) { st = 0; ph ^= 1u; }
                if (two) { if (++st == NST) { st = 0; ph ^= 1u; } }
                // ---- gate: w = sigmoid(g + b_g), x' = (1-w) x + w x_glob  -> A operand of the s_out GEMM (tensor memory)
                float4 x4[4];
                if (site_ok && prow < a.x_rows) {
                    const uint8_t* xr = xring + my_st * 2 * XB + (cg >> 1) * XB + prow * 128;
                    if (narrow) {              // this warp's 8 channels only
#pragma unroll
                        for (int j = 0; j < 2; ++j) x4[j] = *reinterpret_cast<const float4*>(xr + ((((cg & 1) * 4 + sub * 2 + j) ^ (prow & 7)) << 4));
                    } else {
#pragma unroll
                        for (int j = 0; j < 4; ++j) x4[j] = *reinterpret_cast<const float4*>(xr + ((((cg & 1) * 4 + j) ^ (prow & 7)) << 4));
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) x4[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                }
                const float* xv = reinterpret_cast<const float*>(x4);
                if (warp == 0 || warp == 2) SI_TRACE(10 + 5 * warp, (int)gi);
                if (site_ok) { mbar_wait(d1_done + h, c_d1 & 1u); ++c_d1; }      // this half's [x_glob | g]
                if (warp == 0 || warp == 2) SI_TRACE(11 + 5 * warp, (int)gi);
                // x'[gi & 1] was last read by UMMA 2 of item gi-2, whose completion this warp saw in that item's GELU epilogue
                if (warp == 0 || warp == 2) SI_TRACE(12 + 5 * warp, (int)gi);
                tc_fence_after();
                const uint32_t t_xp = lane_base + SI_TM_A1 + (gi & 1u) * 64;
                if (!warp_rows || (SI_DBG(a) & 2)) {          // no listed pair in this warp's 32 rows: x' = 0 (keeps UMMA 2's operand finite), nothing to score
                    uint32_t z[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) z[e] = 0u;
                    if (gi < 2 || k < 2) {
                        tmem_st8(t_xp + cg * 8, z);
                        tmem_st8(t_xp + 32 + cg * 8, z);
                        tmem_st_wait();
                    }
                } else if (narrow && site_ok) {
                    uint32_t g[8], xg[8];
                    tmem_ld8_nw(lane_base + SI_TM_D1 + h * 128 + 64 + cg * 16 + sub * 8, g);
                    tmem_ld8_nw(lane_base + SI_TM_D1 + h * 128 + cg * 16 + sub * 8, xg);
                    tmem_ld_wait();
                    uint4 oh, ol;
                    {
                        uint32_t hw[4], lw[4];
#pragma unroll
                        for (int e = 0; e < 8; e += 2) {
                            const float2 x2 = make_float2(xv[e], xv[e + 1]);
                            const float2 w = sigmoid_fast2(fadd2(make_float2(__uint_as_float(g[e]), __uint_as_float(g[e + 1])), *reinterpret_cast<const float2*>(bgv + sub * 8 + e)));
                            const float2 pp = ffma2(w, fsub2(make_float2(__uint_as_float(xg[e]), __uint_as_float(xg[e + 1])), x2), x2);
                            split2(pp.x, pp.y, hw[e >> 1], lw[e >> 1]);
                        }
                        oh = make_uint4(hw[0], hw[1], hw[2], hw[3]); ol = make_uint4(lw[0], lw[1], lw[2], lw[3]);
                    }
                    // swap the packed words with the partner warp (same half, same column group, other 8 channels).  The first barrier
                    // orders this write behind the partner's read of the previous item, the second publishes it.
                    asm volatile("bar.sync %0, 64;" ::"r"(xch_bar) : "memory");
                    xch[(sub * 2) * 32 + lane] = oh;
                    xch[(sub * 2 + 1) * 32 + lane] = ol;
                    asm volatile("bar.sync %0, 64;" ::"r"(xch_bar) : "memory");
                    const uint4 ph_ = xch[((sub ^ 1) * 2) * 32 + lane], pl_ = xch[((sub ^ 1) * 2 + 1) * 32 + lane];
                    tmem_st4(t_xp + cg * 8 + sub * 4, oh.x, oh.y, oh.z, oh.w);
                    tmem_st4(t_xp + cg * 8 + (sub ^ 1) * 4, ph_.x, ph_.y, ph_.z, ph_.w);
                    tmem_st4(t_xp + 32 + cg * 8 + sub * 4, ol.x, ol.y, ol.z, ol.w);
                    tmem_st4(t_xp + 32 + cg * 8 + (sub ^ 1) * 4, pl_.x, pl_.y, pl_.z, pl_.w);
                    tmem_st_wait();
                } else {
                    uint32_t g[16], xg[16];
                    tmem_ld16_nw(lane_base + SI_TM_D1 + h * 128 + 64 + cg * 16, g);
                    tmem_ld16_nw(lane_base + SI_TM_D1 + h * 128 + cg * 16, xg);
                    tmem_ld_wait();
                    uint32_t hh[8], ll[8];
                    if (site_ok) {                   // packed fp32x2 math: channel pairs (e, e+1) share every FMA-pipe instruction
#pragma unroll
                        for (int e = 0; e < 16; e += 2) {
                            const float2 x2 = make_float2(xv[e], xv[e + 1]);
                            const float2 w = sigmoid_fast2(fadd2(make_float2(__uint_as_float(g[e]), __uint_as_float(g[e + 1])), *reinterpret_cast<const float2*>(bgv + e)));
                            const float2 pp = ffma2(w, fsub2(make_float2(__uint_as_float(xg[e]), __uint_as_float(xg[e + 1])), x2), x2);       // (1-w) x + w x_glob
                            split2(pp.x, pp.y, hh[e >> 1], ll[e >> 1]);
                        }
                    } else {
#pragma unroll
                        for (int e = 0; e < 8; ++e) { hh[e] = 0u; ll[e] = 0u; }
                    }
                    tmem_st8(t_xp + cg * 8, hh);
                    tmem_st8(t_xp + 32 + cg * 8, ll);
                    tmem_st_wait();
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive(a1_ready + h);
                    if (site_ok) mbar_arrive(x_free + my_st);           // x tile consumed
                }
                if (warp == 0 || warp == 2) SI_TRACE(13 + 5 * warp, (int)gi);
                // ---- score of the PREVIOUS item (its s = x' W_s^T has had the whole gate epilogue to finish): the tensor core runs
                //      UMMA 2 of this item and UMMA 1 of the next while the GELU / site-sum epilogue of item k-1 executes
                if (k > 0) ep2(gi - 1, 2 * (k - 1) + h);
            }
            ep2(gi - 1, 2 * (n_items - 1) + h);
            // ---- partial score of this site group: column groups, then the two site halves, in fixed order
            s_part[cg * 128 + q * 32 + lane] = row_ok ? score : 0.f;
            asm volatile("bar.sync 1, 512;" ::: "memory");
            if (tid < a.nc) {
                float sa = (s_part[tid] + s_part[128 + tid]) + (s_part[256 + tid] + s_part[384 + tid]);
                float sb = (s_part[64 + tid] + s_part[192 + tid]) + (s_part[320 + tid] + s_part[448 + tid]);
                if (narrow) {      // the other 8 channels of every column group live in rows 32..63 / 96..127
                    sa += (s_part[32 + tid] + s_part[160 + tid]) + (s_part[288 + tid] + s_part[416 + tid]);
                    sb += (s_part[96 + tid] + s_part[224 + tid]) + (s_part[352 + tid] + s_part[480 + tid]);
                }
                a.score_part[((size_t)b * a.alpha_pairs + tid) * a.nSG + sg] = sa + sb;
            }
            // s_part and the alpha operand are rewritten by the next work item only after this barrier and the next one
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 16) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
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

// <= 64 pairs per tree: the persistent site-parity kernel
int launch_score_inc(const Model* m, const PairChunk& c, int* n_part, cudaStream_t st) {
    static DevOnce once;      // per device, not per process
    if (int e = smem_opt_in(once, k_score_inc, SI_SMEM_MAX)) return e;
    if (c.S > 64 || c.nc > 64) return set_error(NNJ_ERR_INVALID, "score_inc: at most 64 pairs over 63 taxa");
    const int n_sm = sm_count();
    ScoreIncArgs a;
#ifdef NNJ_DEBUG_TOOLS
    a.trace = nullptr;
    static long long* trace_buf = nullptr; static int trace_state = -1;
    if (trace_state < 0) { const char* ev = getenv("NNJ_SCORE_TRACE"); trace_state = ev ? atoi(ev) : 0; }
    if (trace_state > 0 && c.nc == trace_state) { if (!trace_buf) cudaMalloc(&trace_buf, 32 * 600 * 8); cudaMemsetAsync(trace_buf, 0, 32 * 600 * 8, st); a.trace = trace_buf; }
    { static int dbg = -1; if (dbg < 0) { const char* ev = getenv("NNJ_SCORE_DBG"); dbg = ev ? atoi(ev) : 0; } a.dbg = dbg; }
#endif
    a.narrow = c.nc <= 32 ? 1 : 0;
    // the live nodes occupy physical slots [0, Rp) (k_select keeps them compact): only those rows are streamed / contracted
    a.node_rows = (c.Rp + 7) & ~7; a.x_rows = (c.nc + 7) & ~7;
    const int stage = 4 * a.node_rows * 128 + 2 * a.x_rows * 128;
    a.nst = (SI_SMEM_MAX - 1024 - SI_RING - 1024 - SI_MISC_BYTES) / stage;
    if (a.nst > SI_MAXST) a.nst = SI_MAXST;
    a.nst &= ~1;                      // even: the two half-pipelines own the even / odd ring stages (see the kernel)
    if (a.nst < 2) return set_error(NNJ_ERR_INVALID, "score_inc: ring does not fit");
    if (c.C & 7) return set_error(NNJ_ERR_INVALID, "score_inc: the tensor-core NJ kernels need a site count that is a multiple of 8 (nj_use_tc routes other shapes to the fp32 kernels)");
    CUtensorMap mh, ml, mx;
    if (int e = make_tmap_xtile(&mx, c.xf, c.pc, c.nc, c.C, c.B, a.x_rows)) return e;
    if (int e = make_tmap_nodes(&mh, c.nodes_h, c.S, c.B * c.C, a.node_rows, c.Rp)) return e;
    if (int e = make_tmap_nodes(&ml, c.nodes_l, c.S, c.B * c.C, a.node_rows, c.Rp)) return e;
    a.alpha = c.alpha; a.RP = c.RP; a.alpha_pairs = c.alpha_pairs;
    a.slot_of = c.slot_of; a.slot_stride = c.slot_stride; a.pair_i = c.pair_i; a.pair_stride = c.pair_stride; a.n0 = c.n0; a.nc = c.nc;
    a.Rp = c.Rp; a.S = c.Rp; a.C = c.C; a.B = c.B; a.groups = (c.C + SI_SITES - 1) / SI_SITES;   // a.S: slots contracted by UMMA 1
    *n_part = a.groups;
    if (a.groups > c.nSB) return set_error(NNJ_ERR_INVALID, "score_inc: partial buffer too small");
    a.wsh = (const uint4*)m->nj_bf.wsh; a.wsl = (const uint4*)m->nj_bf.wsl;
    a.bg = m->nj.bg; a.bs = m->nj.bs; a.w2 = m->nj.w2; a.b2 = m->nj.b2;
    a.mask = c.mask; a.score_part = c.score_part; a.nSG = c.nSB;
    const int n_work = c.B * a.groups;
    const size_t smem = 1024 + SI_RING + (size_t)a.nst * stage + 1024 + SI_MISC_BYTES;
    prof_begin(KC_SCORE, st);
    k_score_inc<<<n_work < n_sm ? n_work : n_sm, SI_THREADS, smem, st>>>(mh, ml, mx, a);
    LAUNCH_CHECK();
#ifdef NNJ_DEBUG_TOOLS
    if (a.trace) {
        cudaStreamSynchronize(st);
        std::vector<long long> h(32 * 600);
        cudaMemcpy(h.data(), trace_buf, h.size() * 8, cudaMemcpyDeviceToHost);
        FILE* f = fopen("gpurun_out/score_trace.txt", "w");
        if (f) { for (int t = 0; t < 32; ++t) for (int i = 0; i < 600; ++i) if (h[t * 600 + i]) fprintf(f, "%d %d %lld\n", t, i, h[t * 600 + i]); fclose(f); }
        trace_state = 0;
    }
#endif
    return 0;
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
