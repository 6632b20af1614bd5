// nnj_score_big.cu — tcgen05 pair scoring for node sets of 65 .. 256 slots (BASELINE config 4: 200 taxa x 4096 sites; the
// reference's own taxa100 test sets).  Same arithmetic as k_score_tc (model.py:90-99, 148-153):
//     [x_glob | g] = alpha[pair, :] . [X | W_g X][:, site, :]        UMMA 1, K = slots, blocked by 64 slots
//     x'           = x + sigmoid(g + b_g) (x_glob - x)               gate epilogue (x from the fp32 x planes)
//     s            = x' W_s^T                                        UMMA 2 (A from tensor memory)
//     score       += w2 . GELU(s + b_s) + b2 over unmasked sites     GELU epilogue
// What changes above 64 slots is where the operands live.  The alpha operand of a 128-pair tile ([128 x slots] bf16 hi / lo) is
// built ONCE per CTA and kept in TENSOR MEMORY (256 columns = 256 slots hi + lo), so shared memory is free for a ring of
// 64-slot node blocks ([X | W_g X] hi / lo, 32 KB each, TMA, SWIZZLE_128B, MN-major B operand): UMMA 1 of a site walks its
// ceil(slots / 64) blocks, accumulating in one [128 x 128] fp32 accumulator.  TMEM: alpha 256 | [x_glob | g] 128 | s 64 | x' 64 = 512.
// One pipeline per CTA (the accumulators are single): UMMA 1 of site s+1 is queued right behind UMMA 2 of site s, so the tensor
// core contracts the next site's nodes (the long pole at 200 slots: 48 UMMAs of 128 x 128 x 16) while the 8 epilogue warps run
// the GELU epilogue of site s; the gate epilogue of site s+1 then finds its accumulator ready.
// Work item = (tree, 128-pair tile, 64-site group); partial scores per site group are reduced in fixed order by k_score_reduce.
#include "nnj_internal.h"
#include "nnj_tc.cuh"

namespace nnj {

constexpr int SB_THREADS = 320;            // 8 epilogue warps + issue warp + producer warp
constexpr int SB_SITES = 64;               // sites per CTA
constexpr int SB_NSTG = 4;                 // node-block ring depth
constexpr int SB_BLK = 32768;              // one node block: X_h 8K | G_h 8K | X_l 8K | G_l 8K   (64 slots x 128 B each)
constexpr int SB_RING = 0;
constexpr int SB_XT = SB_NSTG * SB_BLK;    // 2 x tiles of 32 KB: [ch 0-31: rows 0-63 | rows 64-127 | ch 32-63: rows 0-63 | rows 64-127]
constexpr int SB_W = SB_XT + 2 * 32768;    // W_s hi 8 KB | lo 8 KB
constexpr int SB_MISC = SB_W + 16384;      // biases 768 B | partials [2][128] 1 KB | slot table 1 KB | barriers | tmem slot
constexpr int SB_SMEM = SB_MISC + 768 + 1024 + 1024 + 256 + 1024;
constexpr uint32_t SB_TM_A0 = 0, SB_TM_D1 = 256, SB_TM_S = 384, SB_TM_A1 = 448;
constexpr int SB_TAB_LD = 260;             // fp32 pitch of the alpha staging table [128][256 + 4] (aliases the ring during set-up)

struct ScoreBigArgs {
    const float* alpha; int RP; int alpha_pairs;
    const int32_t* slot_of; int slot_stride;
    const int32_t* pair_i; int pair_stride; int n0; int nc;
    int Rp, C, KB;                          // live nodes (= live physical slots), sites, 64-slot blocks
    const uint4* wsh; const uint4* wsl;
    const float* bg; const float* bs; const float* w2; float b2;
    const uint8_t* mask;
    float* score_part; int nSG;
};

__global__ void __launch_bounds__(SB_THREADS, 1)
k_score_big(const __grid_constant__ CUtensorMap mapXh, const __grid_constant__ CUtensorMap mapXl, const __grid_constant__ CUtensorMap mapXf,
            const ScoreBigArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* sm = smem_align1024(smem_raw);
    float* s_bias = reinterpret_cast<float*>(sm + SB_MISC);             // bg[64] | bs[64] | w2[64]
    float* s_part = s_bias + 192;                                        // [2 column halves][128 rows]
    int* s_slot = reinterpret_cast<int*>(s_part + 256);                  // logical node -> physical slot [256]
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_slot + 256);
    uint64_t *full = bars, *stage_free = bars + SB_NSTG, *x_full = bars + 2 * SB_NSTG, *x_free = x_full + 2, *d1_done = x_free + 2,
             *a1_ready = d1_done + 1, *s_done = a1_ready + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_done + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b = blockIdx.z, pt = blockIdx.y, sg = blockIdx.x;
    const int rows_here = min(128, a.nc - pt * 128);
    const int c_base = sg * SB_SITES;
    const int n_sites = min(SB_SITES, a.C - c_base);
    const int KB = a.KB;

    if (tid == 0) {
        for (int i = 0; i < SB_NSTG; ++i) { mbar_init(full + i, 1); mbar_init(stage_free + i, 1); }
        mbar_init(x_full, 1); mbar_init(x_full + 1, 1); mbar_init(x_free, 8); mbar_init(x_free + 1, 8);
        mbar_init(d1_done, 1); mbar_init(a1_ready, 8); mbar_init(s_done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 8) tmem_alloc(tmem_slot, 512);
    for (int i = tid; i < 1024; i += SB_THREADS) {                      // W_s -> swizzled K-major tiles (hi, lo)
        const int plane = i >> 9, rem = i & 511, row = rem >> 3, j = rem & 7;
        const uint4* src = plane == 0 ? a.wsh : a.wsl;
        *reinterpret_cast<uint4*>(sm + SB_W + plane * 8192 + row * 128 + ((j ^ (row & 7)) << 4)) = __ldg(src + rem);
    }
    if (tid < 64) { s_bias[tid] = a.bg[tid]; s_bias[64 + tid] = a.bs[tid]; s_bias[128 + tid] = a.w2[tid]; }
    for (int r = tid; r < 256; r += SB_THREADS) s_slot[r] = r < a.Rp ? a.slot_of[(size_t)b * a.slot_stride + r] : 0;
    // ---- alpha of this pair tile, scattered to physical-slot order in a shared-memory table (it aliases the ring: nothing streams yet)
    float* tab = reinterpret_cast<float*>(sm);
    for (int i = tid; i < 128 * SB_TAB_LD / 4; i += SB_THREADS) reinterpret_cast<float4*>(tab)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    for (int idx = tid; idx < rows_here * a.Rp; idx += SB_THREADS) {
        const int row = idx / a.Rp, r = idx - row * a.Rp;
        tab[row * SB_TAB_LD + s_slot[r]] = a.alpha[((size_t)b * a.alpha_pairs + pt * 128 + row) * a.RP + r];
    }
    __syncthreads();
    if (warp < 8) {
        // thread (row, hf) stores half of its row's slots, 16 slots (8 packed words per plane) per tcgen05.st
        const int q = warp & 3, hf = warp >> 2, row = q * 32 + lane;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
        const int groups = KB * 4;                                      // 16-slot groups in the operand
        for (int gidx = hf; gidx < groups; gidx += 2) {
            const float* tr = tab + row * SB_TAB_LD + gidx * 16;
            uint32_t hh[8], ll[8];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float4 v = *reinterpret_cast<const float4*>(tr + 4 * e);
                split2(v.x, v.y, hh[2 * e], ll[2 * e]);
                split2(v.z, v.w, hh[2 * e + 1], ll[2 * e + 1]);
            }
            tmem_st8(lane_base + SB_TM_A0 + gidx * 8, hh);
            tmem_st8(lane_base + SB_TM_A0 + 128 + gidx * 8, ll);
        }
        tmem_st_wait();
    }
    fence_async_smem();         // generic-proxy accesses of the table are ordered before the TMA (async-proxy) writes that reuse its bytes
    tc_fence_before();
    __syncthreads();            // the table is dead: the ring may be filled
    tc_fence_after();

    if (warp == 9) {
        // ================= producer: node blocks of site s (ring), then the site's x tile =================
        int st = 0; uint32_t ph = 0; int gs = 0;
        for (int s = 0; s < n_sites; ++s) {
            const int c = c_base + s;
            for (int kb = 0; kb < KB; ++kb, ++gs) {
                if (gs >= SB_NSTG) mbar_wait(stage_free + st, ph ^ 1u);
                if (elect_one()) {
                    uint8_t* stg = sm + SB_RING + st * SB_BLK;
                    mbar_expect_tx(full + st, SB_BLK);
                    tma_load_3d(stg, &mapXh, full + st, 0, kb * 64, b * a.C + c);
                    tma_load_3d(stg + 8192, &mapXh, full + st, 64, kb * 64, b * a.C + c);
                    tma_load_3d(stg + 16384, &mapXl, full + st, 0, kb * 64, b * a.C + c);
                    tma_load_3d(stg + 24576, &mapXl, full + st, 64, kb * 64, b * a.C + c);
                }
                __syncwarp();
                if (++st == SB_NSTG) { st = 0; ph ^= 1u; }
            }
            const int xb = s & 1;
            if (s >= 2) mbar_wait(x_free + xb, ((s >> 1) - 1) & 1u);
            if (elect_one()) {
                uint8_t* xt = sm + SB_XT + xb * 32768;
                mbar_expect_tx(x_full + xb, 32768);
                tma_load_4d(xt, &mapXf, x_full + xb, 0, c, pt * 128, b);
                tma_load_4d(xt + 8192, &mapXf, x_full + xb, 0, c, pt * 128 + 64, b);
                tma_load_4d(xt + 16384, &mapXf, x_full + xb, 32, c, pt * 128, b);
                tma_load_4d(xt + 24576, &mapXf, x_full + xb, 32, c, pt * 128 + 64, b);
            }
            __syncwarp();
        }
    } else if (warp == 8) {
        // ================= issue warp =================
        const uint32_t wsh = smem_u32(sm + SB_W), wsl = wsh + 8192;
        const uint32_t id_s = umma_idesc_bf16(128, 64), id_d1 = umma_idesc_bf16(128, 128) | (1u << 16);
        const uint32_t td = tmem_base + SB_TM_D1, ts = tmem_base + SB_TM_S, ta0 = tmem_base + SB_TM_A0, ta1 = tmem_base + SB_TM_A1;
        int st = 0; uint32_t ph = 0;
        auto issue_u1 = [&]() {          // [x_glob | g] of the next site: ceil(slots / 64) node blocks into one accumulator
            for (int kb = 0; kb < KB; ++kb) {
                mbar_wait(full + st, ph);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t bh = umma_desc_lo(smem_u32(sm + SB_RING + st * SB_BLK), 8192), bl = umma_desc_lo(smem_u32(sm + SB_RING + st * SB_BLK + 16384), 8192);
                    const uint32_t ah = ta0 + kb * 32, al = ta0 + 128 + kb * 32;
                    if (kb == 0) umma_ts<false>(td, al, bh, id_d1); else umma_ts<true>(td, al, bh, id_d1);      // small terms first
                    umma_ts<true>(td, ah, bl, id_d1);
                    umma_ts<true>(td, ah, bh, id_d1);
#pragma unroll
                    for (int kk = 1; kk < 4; ++kk) {      // 16 slots = 2048 B per k-step
                        umma_ts<true>(td, al + kk * 8, bh + kk * 128, id_d1);
                        umma_ts<true>(td, ah + kk * 8, bl + kk * 128, id_d1);
                        umma_ts<true>(td, ah + kk * 8, bh + kk * 128, id_d1);
                    }
                    umma_commit(stage_free + st);
                    if (kb == KB - 1) umma_commit(d1_done);
                }
                __syncwarp();
                if (++st == SB_NSTG) { st = 0; ph ^= 1u; }
            }
        };
        if (n_sites > 0) issue_u1();
        for (int s = 0; s < n_sites; ++s) {
            mbar_wait(a1_ready, s & 1u);        // the gate epilogue has read [x_glob | g] and written x'
            tc_fence_after();
            if (elect_one()) {
                const uint32_t wh = umma_desc_lo(wsh), wl = umma_desc_lo(wsl);
                umma_ts<false>(ts, ta1 + 32, wh, id_s);       // s = x' . W_s^T; small terms first
                umma_ts<true>(ts, ta1, wl, id_s);
                umma_ts<true>(ts, ta1, wh, id_s);
#pragma unroll
                for (int kk = 1; kk < 4; ++kk) {
                    umma_ts<true>(ts, ta1 + 32 + kk * 8, wh + kk * 2, id_s);
                    umma_ts<true>(ts, ta1 + kk * 8, wl + kk * 2, id_s);
                    umma_ts<true>(ts, ta1 + kk * 8, wh + kk * 2, id_s);
                }
                umma_commit(s_done);
            }
            __syncwarp();
            if (s + 1 < n_sites) issue_u1();    // runs on the tensor core while the warps do the GELU epilogue of site s
        }
    } else {
        // ================= epilogue warps: TMEM lane quarter q, column half hf (32 channels) =================
        const int q = warp & 3, hf = warp >> 2, prow = q * 32 + lane, col0 = hf * 32;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
        const int n = pt * 128 + prow;
        const bool row_ok = n < a.nc && a.pair_i[(size_t)b * a.pair_stride + a.n0 + n] >= 0;
        const float* bgv = s_bias + col0;
        const float* bsv = s_bias + 64 + col0;
        const float* w2v = s_bias + 128 + col0;
        float score = 0.f;
        for (int s = 0; s < n_sites; ++s) {
            const uint32_t par = s & 1u;
            const int c = c_base + s, xb = s & 1;
            const bool site_ok = !(a.mask && a.mask[(size_t)b * a.C + c]);      // loaded here, used after the GELU epilogue
            float4 x4[8];
            {
                mbar_wait(x_full + xb, (s >> 1) & 1u);
                const uint8_t* xr = sm + SB_XT + xb * 32768 + hf * 16384 + prow * 128;
#pragma unroll
                for (int j = 0; j < 8; ++j) x4[j] = *reinterpret_cast<const float4*>(xr + ((j ^ (prow & 7)) << 4));
            }
            const float* xv = reinterpret_cast<const float*>(x4);
            __syncwarp();
            if (lane == 0) mbar_arrive(x_free + xb);      // the x tile is in registers
            // ---- gate: w = sigmoid(g + b_g), x' = (1-w) x + w x_glob  -> A operand of the s_out GEMM (tensor memory)
            mbar_wait(d1_done, par);
            tc_fence_after();
#pragma unroll
            for (int sub = 0; sub < 2; ++sub) {
                uint32_t g[16], xg[16];
                tmem_ld16_nw(lane_base + SB_TM_D1 + 64 + col0 + sub * 16, g);
                tmem_ld16_nw(lane_base + SB_TM_D1 + col0 + sub * 16, xg);
                tmem_ld_wait();
                uint32_t hh[8], ll[8];
#pragma unroll
                for (int k = 0; k < 16; k += 2) {
                    const float2 x2 = make_float2(xv[sub * 16 + k], xv[sub * 16 + k + 1]);
                    const float2 w = sigmoid_fast2(fadd2(make_float2(__uint_as_float(g[k]), __uint_as_float(g[k + 1])), *reinterpret_cast<const float2*>(bgv + sub * 16 + k)));
                    const float2 pp = ffma2(w, fsub2(make_float2(__uint_as_float(xg[k]), __uint_as_float(xg[k + 1])), x2), x2);   // (1-w) x + w x_glob
                    split2(pp.x, pp.y, hh[k >> 1], ll[k >> 1]);
                }
                tmem_st8(lane_base + SB_TM_A1 + ((col0 + sub * 16) >> 1), hh);
                tmem_st8(lane_base + SB_TM_A1 + 32 + ((col0 + sub * 16) >> 1), ll);
            }
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(a1_ready);
            // ---- score: w2 . GELU(s + b_s) (+ b2 once per row), masked site sum
            mbar_wait(s_done, par);
            tc_fence_after();
            float2 acc = make_float2(0.f, 0.f);
#pragma unroll
            for (int sub = 0; sub < 2; ++sub) {
                uint32_t sv[16];
                tmem_ld16_nw(lane_base + SB_TM_S + col0 + sub * 16, sv);
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
        s_part[hf * 128 + prow] = row_ok ? score : 0.f;
    }
    tc_fence_before();
    __syncthreads();
    if (tid < rows_here) a.score_part[((size_t)b * a.alpha_pairs + pt * 128 + tid) * a.nSG + sg] = s_part[tid] + s_part[128 + tid];
    if (warp == 8) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
}

// ------------------------------------------------------------------ pair blend -> x planes (fp32 + bf16 hi / lo)
// x = z x_i + (1 - z) x_j, z = sigmoid(Y_i - Y_j + b_h) (model.py:105-108) for the listed pairs, written as the fp32 x planes the score
// kernel reads and as K-major bf16 hi / lo planes [pair][site * 64 + d]: the A operand of the alpha-logit GEMM.  One thread = one
// site x 4 channels; a block walks 64 sites x BP_PAIRS consecutive pairs.  Consecutive pairs share a node (step 0 lists the pairs
// i-major; every later step pairs ONE node with all others), so a node row that is still in registers from the previous pair is
// not fetched again: ~2 node rows per pair instead of 4, the rest of the re-reads come from L2.
constexpr int BP_PAIRS = 8;
__global__ void __launch_bounds__(256) k_blend_planes(const float* __restrict__ X, const float* __restrict__ Y, size_t tree_stride, int C,
                                                      const int32_t* __restrict__ slot_of, int slot_stride, const int32_t* __restrict__ pair_i,
                                                      const int32_t* __restrict__ pair_j, int pair_stride, int n0, int nc,
                                                      const float* __restrict__ bh, float* __restrict__ xf, uint2* __restrict__ xh,
                                                      uint2* __restrict__ xl, int pc) {
    __shared__ int s_pi[BP_PAIRS], s_pj[BP_PAIRS];
    const int b = blockIdx.z, nb0 = blockIdx.y * BP_PAIRS;
    const int c4 = threadIdx.x & 15, sl = threadIdx.x >> 4;
    if (threadIdx.x < BP_PAIRS) {
        const int n = nb0 + threadIdx.x;
        int pi = -1, pj = -1;
        if (n < nc) {
            const size_t po = (size_t)b * pair_stride + n0 + n;
            const int li = pair_i[po], lj = pair_j[po];
            if (li >= 0) { pi = slot_of[(size_t)b * slot_stride + li]; pj = slot_of[(size_t)b * slot_stride + lj]; }
        }
        s_pi[threadIdx.x] = pi; s_pj[threadIdx.x] = pj;
    }
    __syncthreads();
    const float4 b4 = __ldg(reinterpret_cast<const float4*>(bh) + c4);
    const size_t tb = (size_t)b * tree_stride;
#pragma unroll 1
    for (int it = 0; it < 4; ++it) {
        const int c = blockIdx.x * 64 + it * 16 + sl;
        if (c >= C) break;
        int ci = -1, cj = -1;                              // physical slots whose rows are in registers
        float4 xi = make_float4(0.f, 0.f, 0.f, 0.f), xj = xi, yi = xi, yj = xi;
#pragma unroll
        for (int k = 0; k < BP_PAIRS; ++k) {
            const int n = nb0 + k;
            if (n >= nc) break;
            const int pi = s_pi[k], pj = s_pj[k];
            float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
            if (pi >= 0) {
                if (pi != ci) {
                    if (pi == cj) { xi = xj; yi = yj; }
                    else { const size_t oi = tb + ((size_t)pi * C + c) * D + c4 * 4; xi = ld4(X + oi); yi = ld4(Y + oi); }
                    ci = pi;
                }
                if (pj != cj) {
                    const size_t oj = tb + ((size_t)pj * C + c) * D + c4 * 4;
                    xj = ld4(X + oj); yj = ld4(Y + oj);
                    cj = pj;
                }
                const float2 z0 = sigmoid_fast2(fadd2(fsub2(make_float2(yi.x, yi.y), make_float2(yj.x, yj.y)), make_float2(b4.x, b4.y)));
                const float2 z1 = sigmoid_fast2(fadd2(fsub2(make_float2(yi.z, yi.w), make_float2(yj.z, yj.w)), make_float2(b4.z, b4.w)));
                const float2 v0 = ffma2(z0, fsub2(make_float2(xi.x, xi.y), make_float2(xj.x, xj.y)), make_float2(xj.x, xj.y));
                const float2 v1 = ffma2(z1, fsub2(make_float2(xi.z, xi.w), make_float2(xj.z, xj.w)), make_float2(xj.z, xj.w));
                o = make_float4(v0.x, v0.y, v1.x, v1.y);
            }
            const size_t e = (((size_t)b * pc + n) * C + c) * 16 + c4;                // float4 / uint2 index
            reinterpret_cast<float4*>(xf)[e] = o;
            uint2 hh, ll;
            split2(o.x, o.y, hh.x, ll.x);
            split2(o.z, o.w, hh.y, ll.y);
            xh[e] = hh; xl[e] = ll;
        }
    }
}

// ------------------------------------------------------------------ host side
int launch_blend_planes(const Model* m, const PairChunk& c, cudaStream_t st) {
    prof_begin(KC_BLEND, st);
    k_blend_planes<<<dim3((c.C + 63) / 64, (c.nc + BP_PAIRS - 1) / BP_PAIRS, c.B), 256, 0, st>>>(c.X, c.Y, c.tree_stride, c.C, c.slot_of, c.slot_stride,
                                                                                            c.pair_i, c.pair_j, c.pair_stride, c.n0, c.nc, m->nj.bh,
                                                                                            c.xf, (uint2*)c.xh, (uint2*)c.xl, c.pc);
    LAUNCH_CHECK();
    return 0;
}

int launch_score_big(const Model* m, const PairChunk& c, int* n_part, cudaStream_t st) {
    static DevOnce once;      // per device, not per process
    if (int e = smem_opt_in(once, k_score_big, SB_SMEM)) return e;
    if (c.Rp > 256 || c.S > 256) return set_error(NNJ_ERR_INVALID, "score_big: at most 256 node slots");
    if (c.C & 7) return set_error(NNJ_ERR_INVALID, "score_big: site count must be a multiple of 8");
    CUtensorMap mh, ml, mx;      // node planes: 64 slots of one site per box, slots >= Rp dead (zero-filled); x tiles: 64 pairs, pairs >= nc read as 0
    if (int e = make_tmap_nodes(&mh, c.nodes_h, c.S, c.B * c.C, 64, c.Rp)) return e;
    if (int e = make_tmap_nodes(&ml, c.nodes_l, c.S, c.B * c.C, 64, c.Rp)) return e;
    if (int e = make_tmap_xtile(&mx, c.xf, c.pc, c.nc, c.C, c.B)) return e;
    ScoreBigArgs a;
    a.alpha = c.alpha; a.RP = c.RP; a.alpha_pairs = c.alpha_pairs;
    a.slot_of = c.slot_of; a.slot_stride = c.slot_stride; a.pair_i = c.pair_i; a.pair_stride = c.pair_stride; a.n0 = c.n0; a.nc = c.nc;
    a.Rp = c.Rp; a.C = c.C; a.KB = (c.Rp + 63) / 64;
    a.wsh = (const uint4*)m->nj_bf.wsh; a.wsl = (const uint4*)m->nj_bf.wsl;
    a.bg = m->nj.bg; a.bs = m->nj.bs; a.w2 = m->nj.w2; a.b2 = m->nj.b2;
    a.mask = c.mask; a.score_part = c.score_part; a.nSG = c.nSB;
    *n_part = (c.C + SB_SITES - 1) / SB_SITES;
    if (*n_part > c.nSB) return set_error(NNJ_ERR_INVALID, "score_big: partial buffer too small");
    prof_begin(KC_SCORE, st);
    k_score_big<<<dim3(*n_part, (c.nc + 127) / 128, c.B), SB_THREADS, SB_SMEM, st>>>(mh, ml, mx, a);
    LAUNCH_CHECK();
    return 0;
}

}  // namespace nnj
