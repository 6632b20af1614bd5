// nnj_score_inc.cu — pair scoring for the incremental NJ steps (<= 64 pairs per tree, <= 64 slots) on tcgen05, channels on the TMEM lanes.
//
// Per (pair p, site c), as in k_score_tc (model.py:90-99, 148-153):
//     [x_glob | g] = alpha[p, :] . [X | W_g X][:, c, :]            UMMA 1
//     x'           = x + sigmoid(g + b_g) (x_glob - x)            gate epilogue
//     s            = W_s x'                                       UMMA 2
//     score[p]    += w2 . GELU(s + b_s) + b2 over unmasked sites  GELU / site-sum epilogue
// A step after the first scores at most 63 pairs, so a tile with pairs on the 128 TMEM lanes leaves most lanes idle and gives each thread
// one row and no independent work.  Here both products are transposed so that the lanes are CHANNELS and the columns are pairs:
//   * UMMA 1: [x_glob | g]^T = [X | W_g X]^T . alpha^T with M = 128 = two sites stacked (rows 0..63: the channels of site 2k, rows 64..127
//     those of site 2k+1), K = slots, N = pairs padded to 16 (NP).  A is the node tile as TMA streamed it (site-major [slot][128 ch] bf16,
//     SWIZZLE_128B), read MN-major: the two sites' 64-channel blocks are NB bytes apart (the LBO).  The X half goes to accumulator columns
//     [0, NP), the W_g X half to [64, 64 + NP), so one thread holds x_glob[c] and g[c] of the same channel and site for all its pairs.
//     B = alpha^T (K-major, [NP pairs][64 slots]) is the same for every site of a tree: built once per work item in shared memory.
//   * gate: thread (site half, channel c) owns NP / 4 independent pair columns.  x comes from the x planes as a [NP pairs][64 ch] fp32 TMA
//     box per site (thread c reads n * 256 + 4c: conflict-free); x' (bf16 hi / lo) is written IN PLACE of that box as the K-major
//     B operand of UMMA 2 ([NP pairs][64 ch] hi plane, then the lo plane: the same 256 bytes per pair).
//   * UMMA 2: s = W_s x' with M = 128 output rows (site 2k | site 2k+1) against a block-diagonal [[W_s, 0], [0, W_s]] A operand that lives
//     in tensor memory (K = 128: the x' boxes of both sites), so s[o] of a site lands on the lane that computed x'[o] of it.
//   * GELU / site sum: thread o accumulates w2[o] GELU(s + b_s[o]) over the unmasked sites of its half, one register per pair; at the end
//     of a work item the 128 lanes are reduced in fixed order (warp butterfly, then the four lane quarters) into score_part.
// Persistent over work items (tree, 128-site group).  Warps: 16 epilogue warps (TMEM lane quarter q = warp % 4, pair-column quarter
// warp / 4), one issue warp, two producer warps streaming the node and x tiles through rings of item stages (two sites each).
// Every product is the 3-term bf16 split (hi*hi + hi*lo + lo*hi, small terms first), fp32 accumulation.
#include "nnj_internal.h"
#include "nnj_tc.cuh"

namespace nnj {

constexpr int SI_THREADS = 608;             // 16 epilogue warps + issue warp + node-tile producer + x-tile producer
constexpr int SI_SITES = 128;                // sites per work item (one partial of the score reduction)
constexpr int SI_ALPHA = 0;                  // alpha^T operand: hi [NP][128 B] at 0, lo at 8 KB
constexpr int SI_RINGS = 16384;              // x ring, then node ring, then 1 KB of zeros, then the misc block
constexpr int SI_MISC_BYTES = 2048;          // score reduction [4][64] | unmasked-site count | barriers | tmem slot
constexpr int SI_MAXST = 4;
constexpr int SI_SMEM_MAX = 232448;
constexpr uint32_t SI_TM_D1 = 0, SI_TM_S = 256, SI_TM_W = 384;   // TMEM: D1[2] x 128 ([x_glob | g]) | s[2] x 64 | W_s block-diagonal hi 64 | lo 64

struct ScoreIncArgs {
    const float* alpha; int RP; int alpha_pairs;
    const int32_t* slot_of; int slot_stride;
    const int32_t* pair_i; int pair_stride; int n0; int nc;
    int Rp, C, B, groups;
    int node_rows, nns, nxs;                 // node blocks [node_rows][128 B]; node / x ring depths in items
    const uint4* wsh; const uint4* wsl;
    const float* bg; const float* bs; const float* w2; float b2;
    const uint8_t* mask;
    float* score_part; int nSG;
};

// NPW consecutive accumulator columns of this warp's lanes, in x16 / x8 / x4 pieces (no wait)
template <int NPW>
__device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, uint32_t (&v)[NPW]) {
    int j = 0;
    if constexpr (NPW >= 16) { tmem_ld16_nw(taddr, *reinterpret_cast<uint32_t(*)[16]>(v)); j = 16; }
    if constexpr (NPW % 16 >= 8) { tmem_ld8_nw(taddr + j, *reinterpret_cast<uint32_t(*)[8]>(v + j)); j += 8; }
    if constexpr (NPW % 8 == 4) tmem_ld4_nw(taddr + j, *reinterpret_cast<uint32_t(*)[4]>(v + j));
}

template <int NP>
__global__ void __launch_bounds__(SI_THREADS, 1)
k_score_inc(const __grid_constant__ CUtensorMap mapXh, const __grid_constant__ CUtensorMap mapXl, const __grid_constant__ CUtensorMap mapXf,
            const ScoreIncArgs a) {
    constexpr int NPW = NP / 4;               // pair columns per epilogue thread
    constexpr int XSB = NP * 256;             // one site's x box = its x' hi | lo planes
    extern __shared__ uint8_t smem_raw[];
    uint8_t* sm = smem_align1024(smem_raw);
    const int NB = a.node_rows * 128;         // one node column block
    const int NSB = 8 * NB;                   // node item stage: X_h s0 | X_h s1 | G_h s0 | G_h s1 | X_l s0 | X_l s1 | G_l s0 | G_l s1
    uint8_t* xring = sm + SI_RINGS;
    uint8_t* nring = xring + a.nxs * 2 * XSB;
    // UMMA 1 reads 16 slot rows per k-step from blocks of node_rows (>= Rp, multiple of 8) rows: what lies behind a block must be finite
    // bf16 (0 x NaN would poison the accumulator): the next block, or the zero pad behind the ring
    float* s_red = reinterpret_cast<float*>(nring + a.nns * NSB + 1024);   // [4 lane quarters][64 pairs]
    int* s_cnt = reinterpret_cast<int*>(s_red + 256);
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_red + 272);
    uint64_t *n_full = bars, *n_free = bars + SI_MAXST, *x_full = bars + 2 * SI_MAXST, *x_free = bars + 3 * SI_MAXST;
    uint64_t *a0_ready = bars + 4 * SI_MAXST, *d1_done = a0_ready + 1, *a1_ready = d1_done + 2, *s_done = a1_ready + 2;   // [2] each, by item parity
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_done + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_work = a.B * a.groups;

    if (tid == 0) {
        for (int i = 0; i < SI_MAXST; ++i) { mbar_init(n_full + i, 1); mbar_init(n_free + i, 1); mbar_init(x_full + i, 1); mbar_init(x_free + i, 1); }
        mbar_init(a0_ready, 16);
        for (int i = 0; i < 2; ++i) { mbar_init(d1_done + i, 1); mbar_init(a1_ready + i, 16); mbar_init(s_done + i, 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 16) tmem_alloc(tmem_slot, 512);
    for (int i = tid; i < (a.nns * NSB + 1024) >> 4; i += SI_THREADS) reinterpret_cast<uint4*>(nring)[i] = make_uint4(0u, 0u, 0u, 0u);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp >= 17) {
        // ================= producers: warp 17 streams the node tiles, warp 18 the x boxes, one item (two sites) per ring stage =================
        const bool nodes = warp == 17;
        const int nst_max = nodes ? a.nns : a.nxs;
        int st = 0; uint32_t ph = 0, gi = 0;
        for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
            const int b = w / a.groups, sg = w - b * a.groups;
            const int c_base = sg * SI_SITES, n_items = min(SI_SITES, a.C - c_base) >> 1;
            for (int k = 0; k < n_items; ++k, ++gi) {
                if ((int)gi >= nst_max) mbar_wait((nodes ? n_free : x_free) + st, ph ^ 1u);
                if (elect_one()) {
                    const int c = c_base + 2 * k;
                    if (nodes) {
                        uint8_t* stg = nring + st * NSB;
                        mbar_expect_tx(n_full + st, NSB);
                        for (int s = 0; s < 2; ++s) {
                            const int row = b * a.C + c + s;
                            tma_load_3d(stg + s * NB, &mapXh, n_full + st, 0, 0, row);
                            tma_load_3d(stg + (2 + s) * NB, &mapXh, n_full + st, 64, 0, row);
                            tma_load_3d(stg + (4 + s) * NB, &mapXl, n_full + st, 0, 0, row);
                            tma_load_3d(stg + (6 + s) * NB, &mapXl, n_full + st, 64, 0, row);
                        }
                    } else {
                        uint8_t* xs = xring + st * 2 * XSB;
                        mbar_expect_tx(x_full + st, 2 * XSB);
                        tma_load_4d(xs, &mapXf, x_full + st, 0, c, 0, b);
                        tma_load_4d(xs + XSB, &mapXf, x_full + st, 0, c + 1, 0, b);
                    }
                }
                __syncwarp();
                if (++st == nst_max) { st = 0; ph ^= 1u; }
            }
        }
    } else if (warp == 16) {
        // ================= issue warp =================
        // per work item: U1(0) U1(1), then for every item k: [gate epilogue of k done] U2(k), U1(k+2).  D1 and s are double-buffered by item
        // parity; the gate epilogue of item k runs after the GELU epilogue of item k-2 in every warp, so its a1_ready arrival also frees s[k & 1].
        const uint32_t id1 = umma_idesc_bf16(128, NP) | (1u << 15);     // A (node tile) MN-major, B (alpha^T) K-major
        const uint32_t id2 = umma_idesc_bf16(128, NP);                   // A (W_s, tensor memory) . B (x', K-major)
        const uint32_t al_h = umma_desc_lo(smem_u32(sm + SI_ALPHA)), al_l = umma_desc_lo(smem_u32(sm + SI_ALPHA + 8192));
        const int ksteps = (a.Rp + 15) >> 4;
        int nst = 0, xst = 0; uint32_t nph = 0, gi = 0, wi = 0;
        auto issue_u1 = [&](uint32_t g) {
            mbar_wait(n_full + nst, nph);
            tc_fence_after();
            if (elect_one()) {
                const uint32_t base = smem_u32(nring + nst * NSB);
                const uint32_t td = tmem_base + SI_TM_D1 + (g & 1u) * 128;
#pragma unroll
                for (int half = 0; half < 2; ++half) {       // X -> columns [0, NP), W_g X -> [64, 64 + NP)
                    const uint32_t ah = umma_desc_lo(base + half * 2 * NB, NB), alo = umma_desc_lo(base + (4 + half * 2) * NB, NB);
                    const uint32_t d = td + half * 64;
                    umma_ss<false>(d, alo, al_h, id1);
                    umma_ss<true>(d, ah, al_l, id1);
                    umma_ss<true>(d, ah, al_h, id1);
#pragma unroll
                    for (int kk = 1; kk < 4; ++kk) {
                        if (kk < ksteps) {   // 16 slot rows = 2048 B of the MN-major A per k-step; 32 B along the K-major alpha rows
                            umma_ss<true>(d, alo + kk * 128, al_h + kk * 2, id1);
                            umma_ss<true>(d, ah + kk * 128, al_l + kk * 2, id1);
                            umma_ss<true>(d, ah + kk * 128, al_h + kk * 2, id1);
                        }
                    }
                }
                umma_commit(n_free + nst);
                umma_commit(d1_done + (g & 1u));
            }
            __syncwarp();
            if (++nst == a.nns) { nst = 0; nph ^= 1u; }
        };
        for (int w = blockIdx.x; w < n_work; w += gridDim.x, ++wi) {
            const int sg = w % a.groups;
            const int n_items = min(SI_SITES, a.C - sg * SI_SITES) >> 1;     // >= 4: C is a multiple of 8
            mbar_wait(a0_ready, wi & 1u);
            issue_u1(gi);
            issue_u1(gi + 1);
            for (int k = 0; k < n_items; ++k, ++gi) {
                mbar_wait(a1_ready + (gi & 1u), (gi >> 1) & 1u);
                tc_fence_after();
                if (elect_one()) {      // s = [[W_s, 0], [0, W_s]] . [x'(2k) ; x'(2k+1)]: K-steps 0..3 read site 2k's x' box, 4..7 site 2k+1's
                    const uint32_t ts = tmem_base + SI_TM_S + (gi & 1u) * 64, tw = tmem_base + SI_TM_W;
                    const uint32_t xb = smem_u32(xring + xst * 2 * XSB);
#pragma unroll
                    for (int kk = 0; kk < 8; ++kk) {
                        const uint32_t bh = umma_desc_lo(xb + (kk >> 2) * XSB + (kk & 3) * 32), bl = bh + (NP * 128 >> 4);
                        if (kk == 0) umma_ts<false>(ts, tw + 64 + kk * 8, bh, id2); else umma_ts<true>(ts, tw + 64 + kk * 8, bh, id2);
                        umma_ts<true>(ts, tw + kk * 8, bl, id2);
                        umma_ts<true>(ts, tw + kk * 8, bh, id2);
                    }
                    umma_commit(x_free + xst);
                    umma_commit(s_done + (gi & 1u));
                }
                __syncwarp();
                if (++xst == a.nxs) xst = 0;
                if (k + 2 < n_items) issue_u1(gi + 2);
            }
        }
    } else {
        // ================= epilogue warps: lanes 32q .. 32q + 31 = (site half h, channel c); pair columns [cg NPW, cg NPW + NPW) =================
        const int q = warp & 3, cg = warp >> 2, h = q >> 1, c = (q & 1) * 32 + lane;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
        const int n0 = cg * NPW;
        {   // block-diagonal W_s into tensor memory (A of UMMA 2): row (h, o), K = (site half, input channel); this warp's 32 K of both planes
            const int hk = cg >> 1;
            uint32_t wh[16], wl[16];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint4 vh = hk == h ? __ldg(a.wsh + c * 8 + (cg & 1) * 4 + j) : make_uint4(0u, 0u, 0u, 0u);
                const uint4 vl = hk == h ? __ldg(a.wsl + c * 8 + (cg & 1) * 4 + j) : make_uint4(0u, 0u, 0u, 0u);
                wh[4 * j] = vh.x; wh[4 * j + 1] = vh.y; wh[4 * j + 2] = vh.z; wh[4 * j + 3] = vh.w;
                wl[4 * j] = vl.x; wl[4 * j + 1] = vl.y; wl[4 * j + 2] = vl.z; wl[4 * j + 3] = vl.w;
            }
            tmem_st16(lane_base + SI_TM_W + cg * 16, wh);
            tmem_st16(lane_base + SI_TM_W + 64 + cg * 16, wl);
            tmem_st_wait();
        }
        const float bgc = a.bg[c], bsc = a.bs[c], w2c = a.w2[c];
        uint8_t* ah = sm + SI_ALPHA;
        int xst = 0; uint32_t xph = 0, gi = 0;
        for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
            const int b = w / a.groups, sg = w - b * a.groups;
            const int c_base = sg * SI_SITES, n_sites = min(SI_SITES, a.C - c_base), n_items = n_sites >> 1;
            // ---- alpha^T of this tree (B of UMMA 1): rows = pairs, alpha scattered to physical-slot order, bf16 hi / lo, zeros elsewhere.
            //      All UMMA 1 of the previous work item have retired: every warp waited for each of them in its gate epilogue.
            for (int i = tid; i < NP * 16; i += 512) {
                const int off = (i >= NP * 8 ? 8192 - NP * 128 : 0) + i * 16;
                *reinterpret_cast<uint4*>(ah + off) = make_uint4(0u, 0u, 0u, 0u);
            }
            asm volatile("bar.sync 1, 512;" ::: "memory");
            {
                const int32_t* so = a.slot_of + (size_t)b * a.slot_stride;
                for (int idx = tid; idx < a.nc * a.Rp; idx += 512) {
                    const int row = idx / a.Rp, r = idx - row * a.Rp;
                    const float v = a.alpha[((size_t)b * a.alpha_pairs + row) * a.RP + r];
                    const int slot = so[r];
                    const __nv_bfloat16 hv = __float2bfloat16_rn(v), lv = NNJ_LO_BF16(__float2bfloat16_rn(v - __bfloat162float(hv)));
                    const int off = row * 128 + (((slot >> 3) ^ (row & 7)) << 4) + (slot & 7) * 2;
                    *reinterpret_cast<__nv_bfloat16*>(ah + off) = hv;
                    *reinterpret_cast<__nv_bfloat16*>(ah + 8192 + off) = lv;
                }
            }
            fence_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(a0_ready);

            float acc[NPW];
#pragma unroll
            for (int j = 0; j < NPW; ++j) acc[j] = 0.f;
            // w2[o] GELU(s + b_s[o]) of item g (site `site` of this half) into the per-pair accumulators
            auto gelu_epi = [&](uint32_t g, int site) {
                const bool unmasked = !(a.mask && a.mask[(size_t)b * a.C + c_base + site]);
                mbar_wait(s_done + (g & 1u), (g >> 1) & 1u);
                tc_fence_after();
                uint32_t sv[NPW];
                tmem_ld_cols<NPW>(lane_base + SI_TM_S + (g & 1u) * 64 + n0, sv);
                tmem_ld_wait();
                if (unmasked) {
#pragma unroll
                    for (int j = 0; j < NPW; j += 2) {
                        const float2 sb = fadd2(make_float2(__uint_as_float(sv[j]), __uint_as_float(sv[j + 1])), splat2(bsc));
                        const float2 r = ffma2(gelu_fast2(sb), splat2(w2c), make_float2(acc[j], acc[j + 1]));
                        acc[j] = r.x; acc[j + 1] = r.y;
                    }
                }
                tc_fence_before();
            };
            for (int k = 0; k < n_items; ++k, ++gi) {
                // ---- gate: x' = x + sigmoid(g + b_g) (x_glob - x), written over this site's x box as the hi / lo planes of UMMA 2's B
                uint8_t* xs = xring + xst * 2 * XSB + h * XSB;
                mbar_wait(x_full + xst, xph);
                float xv[NPW];
#pragma unroll
                for (int j = 0; j < NPW; ++j) xv[j] = *reinterpret_cast<const float*>(xs + (n0 + j) * 256 + 4 * c);
                mbar_wait(d1_done + (gi & 1u), (gi >> 1) & 1u);
                tc_fence_after();
                uint32_t xg[NPW], gg[NPW];
                const uint32_t td = lane_base + SI_TM_D1 + (gi & 1u) * 128 + n0;
                tmem_ld_cols<NPW>(td, xg);
                tmem_ld_cols<NPW>(td + 64, gg);
                tmem_ld_wait();
                // every x of this site has been read (the 8 warps of the half) before any x' overwrites the box
                asm volatile("bar.sync %0, 256;" ::"r"(2 + h) : "memory");
#pragma unroll
                for (int j = 0; j < NPW; j += 2) {
                    const float2 x2 = make_float2(xv[j], xv[j + 1]);
                    const float2 wv = sigmoid_fast2(fadd2(make_float2(__uint_as_float(gg[j]), __uint_as_float(gg[j + 1])), splat2(bgc)));
                    const float2 pp = ffma2(wv, fsub2(make_float2(__uint_as_float(xg[j]), __uint_as_float(xg[j + 1])), x2), x2);
                    uint32_t hw, lw;
                    split2(pp.x, pp.y, hw, lw);
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int n = n0 + j + e;
                        const int off = n * 128 + ((((c >> 3) ^ (n & 7))) << 4) + (c & 7) * 2;
                        *reinterpret_cast<uint16_t*>(xs + off) = (uint16_t)(e ? hw >> 16 : hw & 0xffffu);
                        *reinterpret_cast<uint16_t*>(xs + NP * 128 + off) = (uint16_t)(e ? lw >> 16 : lw & 0xffffu);
                    }
                }
                fence_async_smem();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(a1_ready + (gi & 1u));
                if (++xst == a.nxs) { xst = 0; xph ^= 1u; }
                // ---- GELU / site sum of the previous item: the tensor core runs UMMA 2 of this item meanwhile
                if (k > 0) gelu_epi(gi - 1, 2 * (k - 1) + h);
            }
            gelu_epi(gi - 1, 2 * (n_items - 1) + h);
            // ---- partial score of this site group: lanes by a fixed butterfly, then the four lane quarters in fixed order
#pragma unroll
            for (int j = 0; j < NPW; ++j) {
                float v = acc[j];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                if (lane == 0) s_red[q * 64 + n0 + j] = v;
            }
            if (warp == 0) {       // b2 is added once per unmasked site
                int cnt = 0;
                for (int s0 = 0; s0 < n_sites; s0 += 32)
                    cnt += __popc(__ballot_sync(0xffffffffu, s0 + lane < n_sites && !(a.mask && a.mask[(size_t)b * a.C + c_base + s0 + lane])));
                if (lane == 0) *s_cnt = cnt;
            }
            asm volatile("bar.sync 1, 512;" ::: "memory");
            if (tid < a.nc) {
                const float s = ((s_red[tid] + s_red[64 + tid]) + (s_red[128 + tid] + s_red[192 + tid])) + a.b2 * (float)*s_cnt;
                const bool row_ok = a.pair_i[(size_t)b * a.pair_stride + a.n0 + tid] >= 0;
                a.score_part[((size_t)b * a.alpha_pairs + tid) * a.nSG + sg] = row_ok ? s : 0.f;
            }
            // s_red, s_cnt and the alpha operand are rewritten by the next work item only after its first bar.sync 1
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 16) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
}

// ------------------------------------------------------------------ host side

// x boxes of the chunk's pairs at one site: [box_rows pairs][64 ch] fp32, rows past nrows read as zeros (no swizzle: thread c reads word c)
static int make_tmap_xbox(CUtensorMap* map, const float* base, int pc, int nrows, int C, int B, int box_rows) {
    const cuuint64_t gdim[4] = {64, (cuuint64_t)C, (cuuint64_t)nrows, (cuuint64_t)B};
    const cuuint64_t gstr[3] = {256, (cuuint64_t)C * 256, (cuuint64_t)pc * C * 256};
    const cuuint32_t box[4] = {64, 1, (cuuint32_t)box_rows, 1};
    return encode_tmap(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, base, gdim, gstr, box, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                       "the x boxes");
}

template <int NP>
static int launch_inc_t(const ScoreIncArgs& a, const CUtensorMap& mh, const CUtensorMap& ml, const CUtensorMap& mx, size_t smem, cudaStream_t st) {
    static DevOnce once;      // per device, not per process
    if (int e = smem_opt_in(once, k_score_inc<NP>, SI_SMEM_MAX)) return e;
    const int n_work = a.B * a.groups, n_sm = sm_count();
    prof_begin(KC_SCORE, st);
    k_score_inc<NP><<<n_work < n_sm ? n_work : n_sm, SI_THREADS, smem, st>>>(mh, ml, mx, a);
    LAUNCH_CHECK();
    return 0;
}

// <= 64 pairs over <= 64 live nodes: the persistent channel-lane kernel
int launch_score_inc(const Model* m, const PairChunk& c, int* n_part, cudaStream_t st) {
    if (c.S > 64 || c.nc > 64 || c.nc < 1) return set_error(NNJ_ERR_INVALID, "score_inc: at most 64 pairs over 63 taxa");
    if (c.C & 7) return set_error(NNJ_ERR_INVALID, "score_inc: the tensor-core NJ kernels need a site count that is a multiple of 8 (nj_use_tc routes other shapes to the fp32 kernels)");
    const int np = (c.nc + 15) & ~15;
    ScoreIncArgs a;
    // the live nodes occupy physical slots [0, Rp) (k_select keeps them compact): only those rows are streamed / contracted
    a.node_rows = (c.Rp + 7) & ~7;
    const int nsb = 8 * a.node_rows * 128, xsb = 2 * np * 256;
    const int avail = SI_SMEM_MAX - 1024 - SI_RINGS - 1024 - SI_MISC_BYTES;
    a.nxs = 2;
    a.nns = (avail - a.nxs * xsb) / nsb;
    if (a.nns > SI_MAXST) a.nns = SI_MAXST;
    if (a.nns < 2) return set_error(NNJ_ERR_INVALID, "score_inc: ring does not fit");
    a.nxs = (avail - a.nns * nsb) / xsb;
    if (a.nxs > SI_MAXST) a.nxs = SI_MAXST;
    CUtensorMap mh, ml, mx;
    if (int e = make_tmap_xbox(&mx, c.xf, c.pc, c.nc, c.C, c.B, np)) return e;
    if (int e = make_tmap_nodes(&mh, c.nodes_h, c.S, c.B * c.C, a.node_rows, c.Rp)) return e;
    if (int e = make_tmap_nodes(&ml, c.nodes_l, c.S, c.B * c.C, a.node_rows, c.Rp)) return e;
    a.alpha = c.alpha; a.RP = c.RP; a.alpha_pairs = c.alpha_pairs;
    a.slot_of = c.slot_of; a.slot_stride = c.slot_stride; a.pair_i = c.pair_i; a.pair_stride = c.pair_stride; a.n0 = c.n0; a.nc = c.nc;
    a.Rp = c.Rp; a.C = c.C; a.B = c.B; a.groups = (c.C + SI_SITES - 1) / SI_SITES;
    *n_part = a.groups;
    if (a.groups > c.nSB) return set_error(NNJ_ERR_INVALID, "score_inc: partial buffer too small");
    a.wsh = (const uint4*)m->nj_bf.wsh; a.wsl = (const uint4*)m->nj_bf.wsl;
    a.bg = m->nj.bg; a.bs = m->nj.bs; a.w2 = m->nj.w2; a.b2 = m->nj.b2;
    a.mask = c.mask; a.score_part = c.score_part; a.nSG = c.nSB;
    const size_t smem = 1024 + SI_RINGS + (size_t)a.nxs * xsb + (size_t)a.nns * nsb + 1024 + SI_MISC_BYTES;
    switch (np) {
    case 16: return launch_inc_t<16>(a, mh, ml, mx, smem, st);
    case 32: return launch_inc_t<32>(a, mh, ml, mx, smem, st);
    case 48: return launch_inc_t<48>(a, mh, ml, mx, smem, st);
    default: return launch_inc_t<64>(a, mh, ml, mx, smem, st);
    }
}

}  // namespace nnj
