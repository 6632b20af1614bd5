// nnj_score_small.cu — pair scoring for the LATE steps of the NJ loop (<= 16 pairs over <= 16 live nodes per tree).
//
// Same arithmetic as k_score_inc (model.py:90-99, 148-153), per (pair p, site c):
//     [x_glob | g] = alpha[p, :] . [X | W_g X][:, c, :]                 GEMM 1, K = live slots
//     x'           = x + sigmoid(g + b_g) (x_glob - x)                  gate
//     s            = x' W_s^T                                           GEMM 2, K = 64
//     score[p]    += w2 . GELU(s + b_s) + b2 over unmasked sites
// The round-2 k_score_inc put pairs on TMEM lanes: a work item cost the same ~2 950 clocks whether a tree has 32 live pairs or 2
// (profiles/r02_ncu_launches: 715 us per launch of 128 trees at n = 2, 770 us at n = 32), because a tcgen05 tile is 128 rows and
// every epilogue instruction is a full warp.  With 16 rows the natural tile is the 16 x 8 x 16 register-fragment instruction
// (mma.sync, 8 clocks per sub-partition, scratch/hmma_bench.cu): one warp owns one site at a time, the alpha operand of the tree
// lives in its registers as A fragments for all sites, the site's node rows come through ldmatrix.trans as B fragments, the C
// fragments of GEMM 1 turn into the A fragments of GEMM 2 without leaving the registers (same trick as the column attention), and
// the GELU / w2 epilogue runs on the C fragments of GEMM 2.  Every product is the 3-term bf16 split, accumulated in fp32.
// 144 tensor instructions per site instead of a fixed ~1 500 clocks.
// CTA = (tree, 128-site group), 16 warps x 8 sites; a warp streams its sites through a private buffer with cp.async.
// Partial scores per site group go to the same buffer k_score_inc fills (fixed-order reduction: bit-reproducible).
#include "nnj_internal.h"
#include "nnj_tc.cuh"

namespace nnj {

constexpr int SS_SITES = 128;                 // sites per CTA = one partial of the score reduction (as in k_score_inc)
constexpr int SS_WPITCH = 144;                // W_s rows: 64 bf16 + 16 B pad (B-fragment loads of 8 rows hit 32 different banks)

struct ScoreSmallArgs {
    const float* xf; int pc;                  // x planes fp32 [B][pc][C][64]
    const __nv_bfloat16* nodes_h; const __nv_bfloat16* nodes_l; int S;   // site-major node planes [B*C][S][128] = [X | W_g X]
    const float* alpha; int RP; int alpha_pairs;
    const int32_t* slot_of; int slot_stride;
    const int32_t* pair_i; int pair_stride; int n0; int nc;
    int Rp, C;
    const uint4* wsh; const uint4* wsl;
    const float* bg; const float* bs; const float* w2; float b2;
    const uint8_t* mask;
    float* score_part; int nSG;
};

// T = 1 16-row / 16-slot tile (<= 16 pairs and slots); SS_WARPS warps with one private tile buffer each.
// Measured (128 trees, DESIGN 4.6): a 32-row form (17-32 pairs) is bound by its 384 tensor instructions per site (8 clocks each and
// sub-partition: 770 clocks per site and SM) and loses to k_score_inc's narrow mode (860 vs 770 us per launch); the 16-row tile with
// 8 warps ran at 43 % of the legacy tensor pipe (two warps per sub-partition cannot cover the 20-clock dependent instruction chains
// and the gate math between the two GEMMs; an 8-warp double-buffered variant measured 355 vs 340 us), hence 16 warps with one buffer each.
// HALF: at most 8 listed pairs - rows 8..15 of the tile are padding and their gate / GELU math is compiled out.
template <int T, int SS_WARPS, bool HALF>
__global__ void __launch_bounds__(SS_WARPS * 32, 1) k_score_small(const ScoreSmallArgs a) {
    constexpr int ROWS = 16 * T;
    constexpr int NODE_B = ROWS * 256;                  // one node plane of a site: [slot][128 ch] bf16, 16-byte chunk c stored at c ^ (slot & 7)
    constexpr int X_B = ROWS * 256;                     // x tile of a site: [pair][64 ch] fp32, chunk c stored at c ^ (pair & 7)
    constexpr int BUF = 2 * NODE_B + X_B;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* sm = smem_align1024(smem_raw);
    uint8_t* wsm = sm;                                  // W_s hi | lo, [64 out][SS_WPITCH]
    float* tab = reinterpret_cast<float*>(sm + 2 * 64 * SS_WPITCH);          // alpha by physical slot [ROWS][ROWS + 1]; later the warps' partial scores
    float* s_bias = tab + 32 * 33;                      // b_g | b_s | w2
    uint8_t* bufs = reinterpret_cast<uint8_t*>(s_bias + 192);
    bufs += (1024 - (smem_u32(bufs) & 1023)) & 1023;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const int sg = blockIdx.x, b = blockIdx.y;
    const int c_base = sg * SS_SITES, n_sites = min(SS_SITES, a.C - c_base);

    // ---- per-CTA set-up: W_s, biases, alpha of this tree scattered to physical-slot order, zeroed tile buffers (rows past the
    //      live ones are never loaded and must read as zeros)
    for (int i = tid; i < 1024; i += SS_WARPS * 32) {
        const int plane = i >> 9, rem = i & 511, row = rem >> 3, j = rem & 7;
        *reinterpret_cast<uint4*>(wsm + plane * 64 * SS_WPITCH + row * SS_WPITCH + j * 16) = __ldg((plane ? a.wsl : a.wsh) + rem);
    }
    if (tid < 64) { s_bias[tid] = a.bg[tid]; s_bias[64 + tid] = a.bs[tid]; s_bias[128 + tid] = a.w2[tid]; }
    for (int i = tid; i < 32 * 33; i += SS_WARPS * 32) tab[i] = 0.f;
    for (int i = tid; i < (SS_WARPS * BUF) >> 4; i += SS_WARPS * 32) reinterpret_cast<uint4*>(bufs)[i] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    {
        const int32_t* so = a.slot_of + (size_t)b * a.slot_stride;
        for (int idx = tid; idx < a.nc * a.Rp; idx += SS_WARPS * 32) {
            const int row = idx / a.Rp, r = idx - row * a.Rp;
            tab[row * 33 + so[r]] = a.alpha[((size_t)b * a.alpha_pairs + row) * a.RP + r];
        }
    }
    __syncthreads();
    // alpha as A fragments (hi, lo) of every (row tile m, slot step k): a0 = [g][2t], a1 = [g+8][2t], a2 = [g][8+2t], a3 = [g+8][8+2t]
    uint32_t ah[T][T][4], al[T][T][4];
#pragma unroll
    for (int m = 0; m < T; ++m)
#pragma unroll
        for (int k = 0; k < T; ++k) {
            const float* p0 = tab + (16 * m + g) * 33 + 16 * k + 2 * t;
            const float* p1 = p0 + 8 * 33;
            split2(p0[0], p0[1], ah[m][k][0], al[m][k][0]);
            split2(p1[0], p1[1], ah[m][k][1], al[m][k][1]);
            split2(p0[8], p0[9], ah[m][k][2], al[m][k][2]);
            split2(p1[8], p1[9], ah[m][k][3], al[m][k][3]);
        }
    __syncthreads();                                     // tab is reused for the partial scores below

    uint8_t* mybuf = bufs + warp * BUF;
    const uint32_t mybuf_u = smem_u32(mybuf);
    const uint32_t wsm_u = smem_u32(wsm);
    const size_t node_site_stride = (size_t)a.S * 128;  // bf16 elements per site in a node plane
    // this warp's sites: warp, warp + SS_WARPS, ...
    auto issue = [&](int site) {
        const int c = c_base + site;
        const uint32_t dst = mybuf_u;
        const uint8_t* nh = reinterpret_cast<const uint8_t*>(a.nodes_h + ((size_t)b * a.C + c) * node_site_stride);
        const uint8_t* nl = reinterpret_cast<const uint8_t*>(a.nodes_l + ((size_t)b * a.C + c) * node_site_stride);
        {   // live node rows (contiguous in both planes): lane = (slot parity, 16-byte chunk), two slots per pass
            const int ch = lane & 15;
            const uint8_t* ph = nh + lane * 16;
            const uint8_t* pl = nl + lane * 16;
            for (int slot = lane >> 4; slot < a.Rp; slot += 2, ph += 512, pl += 512) {
                const uint32_t off = dst + slot * 256 + ((ch ^ (slot & 7)) << 4);
                cp_async16(off, ph);
                cp_async16(off + NODE_B, pl);
            }
            // x rows of the listed pairs at this site (one 256-byte row per pair, C rows apart)
            const float* px = a.xf + (((size_t)b * a.pc + (lane >> 4)) * a.C + c) * 64 + ch * 4;
            const size_t xstride = (size_t)2 * a.C * 64;
            for (int row = lane >> 4; row < a.nc; row += 2, px += xstride)
                cp_async16(dst + 2 * NODE_B + row * 256 + ((ch ^ (row & 7)) << 4), px);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    float part[T][2];
#pragma unroll
    for (int m = 0; m < T; ++m) { part[m][0] = 0.f; part[m][1] = 0.f; }
    int n_unmasked = 0;
    for (int site = warp; site < n_sites; site += SS_WARPS) {
        issue(site);
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncwarp();
        const bool unmasked = !(a.mask && a.mask[(size_t)b * a.C + c_base + site]);
        const uint8_t* xt = mybuf + 2 * NODE_B;
        float sacc[T][8][4];
#pragma unroll
        for (int m = 0; m < T; ++m)
#pragma unroll
            for (int f = 0; f < 8; ++f) { sacc[m][f][0] = 0.f; sacc[m][f][1] = 0.f; sacc[m][f][2] = 0.f; sacc[m][f][3] = 0.f; }
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {                 // 16 channels of x' at a time = one K step of GEMM 2
            uint32_t xh[T][4], xl[T][4];                 // x' as A fragments: [row g | row g+8] of channel block 2kk, then of block 2kk + 1
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int j = 2 * kk + e;                // channel block: channels 8j .. 8j+7 of X (n-tile j) and of W_g X (n-tile 8 + j)
                float xg[T][4], gg[T][4];
#pragma unroll
                for (int m = 0; m < T; ++m) { xg[m][0] = xg[m][1] = xg[m][2] = xg[m][3] = 0.f; gg[m][0] = gg[m][1] = gg[m][2] = gg[m][3] = 0.f; }
#pragma unroll
                for (int k = 0; k < T; ++k) {
                    // four 8 x 8 matrices: slots 16k + 0..7 / 8..15 of chunk j (x_glob), the same of chunk 8 + j (g); lane l supplies row l & 7 of matrix l >> 3
                    const int slot = 16 * k + ((lane >> 3) & 1) * 8 + (lane & 7);
                    const uint32_t ad = mybuf_u + slot * 256 + ((((lane >> 4) * 8 + j) ^ (lane & 7)) << 4);
                    uint32_t bh[4], bl[4];
                    ldsm_x4_t(bh, ad);
                    ldsm_x4_t(bl, ad + NODE_B);
#pragma unroll
                    for (int m = 0; m < T; ++m) {
                        mma_m16n8k16(xg[m], al[m][k], bh[0], bh[1]);      // small terms first
                        mma_m16n8k16(xg[m], ah[m][k], bl[0], bl[1]);
                        mma_m16n8k16(xg[m], ah[m][k], bh[0], bh[1]);
                        mma_m16n8k16(gg[m], al[m][k], bh[2], bh[3]);
                        mma_m16n8k16(gg[m], ah[m][k], bl[2], bl[3]);
                        mma_m16n8k16(gg[m], ah[m][k], bh[2], bh[3]);
                    }
                }
                // gate on this thread's elements: rows 16m + g and 16m + g + 8, channels 8j + 2t, 8j + 2t + 1
                const int ch = 8 * j + 2 * t;
                const float2 bgv = *reinterpret_cast<const float2*>(s_bias + ch);
#pragma unroll
                for (int m = 0; m < T; ++m) {
#pragma unroll
                    for (int hrow = 0; hrow < 2; ++hrow) {
                        const int row = 16 * m + g + 8 * hrow;
                        if (HALF && hrow == 1) { xh[m][2 * e + hrow] = 0u; xl[m][2 * e + hrow] = 0u; continue; }
                        const float2 x2 = *reinterpret_cast<const float2*>(xt + row * 256 + (((ch >> 2) ^ (row & 7)) << 4) + (ch & 3) * 4);
                        const float2 w = sigmoid_fast2(fadd2(make_float2(gg[m][2 * hrow], gg[m][2 * hrow + 1]), bgv));
                        const float2 pp = ffma2(w, fsub2(make_float2(xg[m][2 * hrow], xg[m][2 * hrow + 1]), x2), x2);       // (1-w) x + w x_glob
                        split2(pp.x, pp.y, xh[m][2 * e + hrow], xl[m][2 * e + hrow]);
                    }
                }
            }
            // GEMM 2, K step kk: s[row][out] += x'[row][16kk ..] . W_s[out][16kk ..]
#pragma unroll
            for (int f = 0; f < 8; ++f) {
                const uint32_t wa = wsm_u + (8 * f + g) * SS_WPITCH + (16 * kk + 2 * t) * 2;
                uint32_t wh0, wh1, wl0, wl1;
                asm volatile("ld.shared.b32 %0, [%1];" : "=r"(wh0) : "r"(wa));
                asm volatile("ld.shared.b32 %0, [%1];" : "=r"(wh1) : "r"(wa + 16));
                asm volatile("ld.shared.b32 %0, [%1];" : "=r"(wl0) : "r"(wa + 64 * SS_WPITCH));
                asm volatile("ld.shared.b32 %0, [%1];" : "=r"(wl1) : "r"(wa + 64 * SS_WPITCH + 16));
#pragma unroll
                for (int m = 0; m < T; ++m) {
                    mma_m16n8k16(sacc[m][f], xl[m], wh0, wh1);
                    mma_m16n8k16(sacc[m][f], xh[m], wl0, wl1);
                    mma_m16n8k16(sacc[m][f], xh[m], wh0, wh1);
                }
            }
        }
        // ---- w2 . GELU(s + b_s) on the C fragments: rows g / g+8, outputs 8f + 2t, 8f + 2t + 1
        if (unmasked) {
            ++n_unmasked;
#pragma unroll
            for (int m = 0; m < T; ++m) {
                float2 acc0 = make_float2(0.f, 0.f), acc1 = make_float2(0.f, 0.f);
#pragma unroll
                for (int f = 0; f < 8; ++f) {
                    const float2 bsv = *reinterpret_cast<const float2*>(s_bias + 64 + 8 * f + 2 * t), w2v = *reinterpret_cast<const float2*>(s_bias + 128 + 8 * f + 2 * t);
                    acc0 = ffma2(gelu_fast2(fadd2(make_float2(sacc[m][f][0], sacc[m][f][1]), bsv)), w2v, acc0);
                    if (!HALF) acc1 = ffma2(gelu_fast2(fadd2(make_float2(sacc[m][f][2], sacc[m][f][3]), bsv)), w2v, acc1);
                }
                part[m][0] += acc0.x + acc0.y;
                part[m][1] += acc1.x + acc1.y;
            }
        }
        __syncwarp();                                    // everybody done with this buffer before the next site's loads land in it
    }
    // ---- partial score of this site group: quad sum, then the warps in fixed order
#pragma unroll
    for (int m = 0; m < T; ++m)
#pragma unroll
        for (int hrow = 0; hrow < 2; ++hrow) {
            float v = part[m][hrow];
            v += __shfl_xor_sync(0xffffffffu, v, 1);
            v += __shfl_xor_sync(0xffffffffu, v, 2);
            if (t == 0) tab[warp * 32 + 16 * m + g + 8 * hrow] = v + a.b2 * (float)n_unmasked;
        }
    __syncthreads();
    if (tid < a.nc) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < SS_WARPS; ++w) s += tab[w * 32 + tid];
        const bool row_ok = a.pair_i[(size_t)b * a.pair_stride + a.n0 + tid] >= 0;
        a.score_part[((size_t)b * a.alpha_pairs + tid) * a.nSG + sg] = row_ok ? s : 0.f;
    }
}

template <bool HALF>
static int launch_small_t(const ScoreSmallArgs& a, int groups, int B, cudaStream_t st) {
    constexpr size_t smem = 1024 + 2 * 64 * SS_WPITCH + (32 * 33 + 192) * 4 + 1024 + (size_t)16 * (3 * 16 * 256);
    static DevOnce once;      // per device, not per process
    if (int e = smem_opt_in(once, k_score_small<1, 16, HALF>, smem)) return e;
    prof_begin(KC_SCORE, st);
    k_score_small<1, 16, HALF><<<dim3(groups, B), 16 * 32, smem, st>>>(a);
    LAUNCH_CHECK();
    return 0;
}

int launch_score_small(const Model* m, const PairChunk& c, int* n_part, cudaStream_t st) {
    if (c.nc > 16 || c.Rp > 16 || c.nc < 1) return set_error(NNJ_ERR_INVALID, "score_small: at most 16 pairs over 16 live nodes");
    ScoreSmallArgs a;
    a.xf = c.xf; a.pc = c.pc; a.nodes_h = (const __nv_bfloat16*)c.nodes_h; a.nodes_l = (const __nv_bfloat16*)c.nodes_l; a.S = c.S;
    a.alpha = c.alpha; a.RP = c.RP; a.alpha_pairs = c.alpha_pairs; a.slot_of = c.slot_of; a.slot_stride = c.slot_stride;
    a.pair_i = c.pair_i; a.pair_stride = c.pair_stride; a.n0 = c.n0; a.nc = c.nc; a.Rp = c.Rp; a.C = c.C;
    a.wsh = (const uint4*)m->nj_bf.wsh; a.wsl = (const uint4*)m->nj_bf.wsl;
    a.bg = m->nj.bg; a.bs = m->nj.bs; a.w2 = m->nj.w2; a.b2 = m->nj.b2;
    a.mask = c.mask; a.score_part = c.score_part; a.nSG = c.nSB;
    const int groups = (c.C + SS_SITES - 1) / SS_SITES;
    *n_part = groups;
    if (groups > c.nSB) return set_error(NNJ_ERR_INVALID, "score_small: partial buffer too small");
    return c.nc <= 8 ? launch_small_t<true>(a, groups, c.B, st) : launch_small_t<false>(a, groups, c.B, st);
}

}  // namespace nnj
