// nnj_alpha_tc.cu — pair blend + global-attention logits of the NJ loop on tcgen05 (precision bf16x3).
//
// For every listed pair n = (i, j) of a tree and every site c the reference forms (model.py:105-118)
//     z = sigmoid(W_h (x_i - x_j) + b_h) = sigmoid(Y_i - Y_j + b_h),      x = z x_i + (1 - z) x_j
//     alpha[n, r] = sum_{c,d} (W_q x + b_q)[c,d] K_r[c,d] = sum_{c,d} x[c,d] K'_r[c,d] + kappa_r        (K' = W_q^T K)
// One work item = one tree x 128 sites x up to 4 tiles of 128 pairs (persistent CTAs).  Per site a producer warp streams the site's node tile
// (X, Y fp32 [slots x 64], K' bf16 hi/lo [slots x 64]) into a shared-memory ring by TMA (SWIZZLE_128B, so that
// lanes reading different slots hit different banks); the ring is 3..12 deep by the slot count; 16 blend warps form x for one pair row x 16 channels per thread,
// write it (fp32, staged per warp and sent by TMA store) to the x planes the pair-score kernel reads later, and store its bf16 hi/lo split straight into TENSOR
// MEMORY (tcgen05.st: row = TMEM lane, two bf16 per column) as the A operand; an issue warp runs
//     acc[tile][pair, slot] += x[pair, site, :] . K'[slot, site, :]        (tcgen05.mma, A from TMEM, 3-product split)
// with a double-buffered A operand, so the tensor core works on one (site, tile) while the CUDA cores blend the next.
// Shared memory carries only the node ring: the A operand never touches it.
// With <= 64 pairs (every step after the first) rows 64..127 would idle, so the tile is split by site parity instead:
// lanes 0..63 hold the pairs at site 2k, lanes 64..127 the same pairs at site 2k+1, and two UMMA groups (K' of site 2k ->
// accumulator 0, K' of site 2k+1 -> accumulator 1) leave the even-site sums in rows 0..63 of accumulator 0 and the
// odd-site sums in rows 64..127 of accumulator 1 (the other halves are ignored).
// With <= 32 pairs the split is 4-way: lane quarter q holds the pairs at site 4k+q, four UMMA groups, four accumulators.  A warp's
// TMEM lane quarter and its SM sub-partition are both warp % 4, so this is what puts real rows on all four schedulers.
// The accumulators are written once per work item as partials of this site group; k_alpha_softmax reduces them in fixed order.
#include "nnj_internal.h"
#include "nnj_tc.cuh"

namespace nnj {

constexpr int AV_BLEND_WARPS = 16;
constexpr int AV_THREADS = (AV_BLEND_WARPS + 2) * 32;   // + UMMA issue warp + TMA producer warp
constexpr int AV_SITES = 128;                           // sites per work item (accumulators are read out and the roles resynchronise at every boundary)
constexpr int AV_MAXST = 12;                            // node-ring depth (runtime, 3..12 by the slot count)
constexpr int AV_MAXT = 4;                              // pair tiles per work item
constexpr int AV_XS_BYTES = AV_BLEND_WARPS * 2048;      // x staging for the TMA stores: 16 warps x [32 rows][64 B] (SWIZZLE_64B)
constexpr int AV_TAB_BYTES = 2 * 2 * AV_MAXT * 128 * 4; // pair tables: 2 buffers x (slot_i, slot_j) x 512 rows
constexpr int AV_MISC_BYTES = AV_TAB_BYTES + 256 + 512; // + b_h + barriers / tmem slot
constexpr int AV_SMEM_MAX = 232448;
constexpr uint32_t AV_TM_A = 256;                       // TMEM columns: acc tiles [0,256) | A buffers 2 x (hi 32 | lo 32)

struct AlphaV3Args {
    const int32_t* slot_of; int slot_stride;
    const int32_t* pair_i; const int32_t* pair_j; int pair_stride; int n0; int nc;
    int C, B, groups;                          // work item = (tree, 64-site group)
    const float* bh;
    float* alpha_part; int alpha_pairs; int nSG; int RP;
    int dup;                                   // nc <= 64: tile split by site parity, two partials per site group
    int ways;                                  // sites per 128-lane tile: 1, 2 (dup, nc <= 64) or 4 (nc <= 32: lane quarter q = site 4k+q)
    int tile_bytes, nst;                       // ring geometry: [round8(live slots)][128 B] tiles, 6 per stage, nst stages
    int nmma;                                  // UMMA N = round16(live slots)
};

struct RingPos {                               // position in the node ring / its phase bit
    int st; uint32_t ph;
    __device__ __forceinline__ void next(int nst) { if (++st == nst) { st = 0; ph ^= 1u; } }
};

// Persistent: grid = min(work items, SMs); every role walks the same static list of work items (w = blockIdx.x, += gridDim.x)
// and the node ring, its barriers and the A-operand buffers keep running across items, so the next item's node tiles are
// already in flight while the partials of the current one are written out.
__global__ void __launch_bounds__(AV_THREADS, 1)
k_alpha_v3(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapY, const __grid_constant__ CUtensorMap mapKh,
           const __grid_constant__ CUtensorMap mapKl, const __grid_constant__ CUtensorMap mapXo, const AlphaV3Args a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* sm = smem_align1024(smem_raw);
    const int T = a.tile_bytes, STG = 6 * T, NST = a.nst;      // stage: X ch 0-31 | X ch 32-63 | Y | Y | K'_hi | K'_lo
    uint8_t* xs_base = sm + NST * STG;
    int* s_tab = reinterpret_cast<int*>(xs_base + AV_XS_BYTES);    // [buf][slot_i 512 | slot_j 512]  (physical slots, -1: no pair)
    float* s_bh = reinterpret_cast<float*>(s_tab + 2 * 2 * AV_MAXT * 128);
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_bh + 64);
    uint64_t *full = bars, *stage_free = bars + AV_MAXST, *a_ready = bars + 2 * AV_MAXST, *a_free = a_ready + 2, *done = a_free + 2,
             *tab_full = done + 1, *tab_free = tab_full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tab_free + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int rows_cta = a.nc;
    const int NT = (rows_cta + 127) >> 7;
    const bool dup = a.dup != 0;                                          // site-parity split of a half-empty tile
    const int WAYS = a.ways;                                              // 2 or 4 sites per item when dup
    const bool quad = WAYS == 4;
    const int n_work = a.B * a.groups;

    if (tid == 0) {
        for (int i = 0; i < NST; ++i) { mbar_init(full + i, 1); mbar_init(stage_free + i, AV_BLEND_WARPS / WAYS + 1); }
        mbar_init(a_ready, AV_BLEND_WARPS); mbar_init(a_ready + 1, AV_BLEND_WARPS);
        mbar_init(a_free, 1); mbar_init(a_free + 1, 1);
        mbar_init(done, 1);
        mbar_init(tab_full, 1); mbar_init(tab_full + 1, 1);
        mbar_init(tab_free, AV_BLEND_WARPS); mbar_init(tab_free + 1, AV_BLEND_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == AV_BLEND_WARPS) tmem_alloc(tmem_slot, 512);
    if (tid < 64) s_bh[tid] = a.bh[tid];
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == AV_BLEND_WARPS + 1) {
        // ================= producer warp: pair table of the work item, then the node tiles of its sites =================
        RingPos rp{0, 0u};
        int gs = 0, wi = 0;
        for (int w = blockIdx.x; w < n_work; w += gridDim.x, ++wi) {
            const int b = w / a.groups, sg = w - b * a.groups;
            const int c_base = sg * AV_SITES, n_sites = min(AV_SITES, a.C - c_base);
            {
                const int tb = wi & 1;
                if (wi >= 2) mbar_wait(tab_free + tb, ((wi >> 1) - 1) & 1);
                int* tpi = s_tab + tb * (2 * AV_MAXT * 128);
                int* tpj = tpi + AV_MAXT * 128;
                const int32_t* so = a.slot_of + (size_t)b * a.slot_stride;
                for (int r = lane; r < NT * 128; r += 32) {
                    int pi = -1, pj = -1;
                    if (r < rows_cta) {
                        const size_t o = (size_t)b * a.pair_stride + a.n0 + r;
                        const int li = a.pair_i[o], lj = a.pair_j[o];
                        if (li >= 0) { pi = so[li]; pj = so[lj]; }
                    }
                    tpi[r] = pi; tpj[r] = pj;
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(tab_full + tb);
            }
            for (int s = 0; s < n_sites; ++s, ++gs) {
                if (gs >= NST) mbar_wait(stage_free + rp.st, rp.ph ^ 1u);
                if (elect_one()) {
                    uint8_t* stg = sm + rp.st * STG;
                    const int c = c_base + s;
                    mbar_expect_tx(full + rp.st, STG);
                    tma_load_4d(stg, &mapX, full + rp.st, 0, c, 0, b);
                    tma_load_4d(stg + T, &mapX, full + rp.st, 32, c, 0, b);
                    tma_load_4d(stg + 2 * T, &mapY, full + rp.st, 0, c, 0, b);
                    tma_load_4d(stg + 3 * T, &mapY, full + rp.st, 32, c, 0, b);
                    tma_load_4d(stg + 4 * T, &mapKh, full + rp.st, 0, c, 0, b);
                    tma_load_4d(stg + 5 * T, &mapKl, full + rp.st, 0, c, 0, b);
                }
                __syncwarp();
                rp.next(NST);
            }
        }
    } else if (warp == AV_BLEND_WARPS) {
        // ================= issue warp: acc (+)= A (tensor memory) . K'^T =================
        const uint32_t idesc = umma_idesc_bf16(128, a.nmma);
        RingPos rp{0, 0u};
        int gk = 0;
        for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
            const int b = w / a.groups, sg = w - b * a.groups;
            const int n_sites = min(AV_SITES, a.C - sg * AV_SITES);
            if (!dup) {
                for (int s = 0; s < n_sites; ++s) {
                    mbar_wait(full + rp.st, rp.ph);
                    const uint32_t kh = smem_u32(sm + rp.st * STG + 4 * T), kl = kh + T;
                    for (int t = 0; t < NT; ++t, ++gk) {
                        const int buf = gk & 1;
                        mbar_wait(a_ready + buf, (gk >> 1) & 1);
                        tc_fence_after();
                        if (elect_one()) {
                            const uint32_t ta = tmem_base + AV_TM_A + buf * 64, td = tmem_base + t * 64;
#pragma unroll
                            for (int kk = 0; kk < 4; ++kk) {
                                umma_bf16_ta(td, ta + 32 + kk * 8, umma_desc_k128(kh + kk * 32), idesc, (s | kk) ? 1u : 0u);   // small terms first
                                umma_bf16_ta(td, ta + kk * 8, umma_desc_k128(kl + kk * 32), idesc, 1u);
                                umma_bf16_ta(td, ta + kk * 8, umma_desc_k128(kh + kk * 32), idesc, 1u);
                            }
                            umma_commit(a_free + buf);
                            if (t == NT - 1) umma_commit(stage_free + rp.st);
                        }
                        __syncwarp();
                    }
                    rp.next(NST);
                }
            } else {
                const int n_items = (n_sites + WAYS - 1) / WAYS;
                for (int k = 0; k < n_items; ++k, ++gk) {
                    const int buf = gk & 1;
                    mbar_wait(a_ready + buf, (gk >> 1) & 1);
                    for (int h = 0; h < WAYS; ++h) {
                        if (WAYS * k + h >= n_sites) break;
                        mbar_wait(full + rp.st, rp.ph);
                        tc_fence_after();
                        if (elect_one()) {
                            const uint32_t kh = smem_u32(sm + rp.st * STG + 4 * T), kl = kh + T;
                            const uint32_t ta = tmem_base + AV_TM_A + buf * 64, td = tmem_base + h * 64;
#pragma unroll
                            for (int kk = 0; kk < 4; ++kk) {
                                umma_bf16_ta(td, ta + 32 + kk * 8, umma_desc_k128(kh + kk * 32), idesc, (k | kk) ? 1u : 0u);
                                umma_bf16_ta(td, ta + kk * 8, umma_desc_k128(kl + kk * 32), idesc, 1u);
                                umma_bf16_ta(td, ta + kk * 8, umma_desc_k128(kh + kk * 32), idesc, 1u);
                            }
                            umma_commit(stage_free + rp.st);
                        }
                        __syncwarp();
                        rp.next(NST);
                    }
                    if (elect_one()) umma_commit(a_free + buf);
                    __syncwarp();
                }
            }
            if (elect_one()) umma_commit(done);
            __syncwarp();
        }
    } else {
        // ================= blend warps: TMEM lane quarter q, channels [16 cg, 16 cg + 16) =================
        const int q = warp & 3, cg = warp >> 2;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
        const int half_off = (cg >> 1) * T, j0 = (cg & 1) * 4;
        uint8_t* xs = xs_base + warp * 2048 + lane * 64;   // this thread's row of the warp's store box
        float bh[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) bh[e] = s_bh[cg * 16 + e];
        RingPos rp{0, 0u};          // ring position of the first site of the current item
        int gk = 0, wi = 0;
        for (int w = blockIdx.x; w < n_work; w += gridDim.x, ++wi) {
            const int b = w / a.groups, sg = w - b * a.groups;
            const int c_base = sg * AV_SITES, n_sites = min(AV_SITES, a.C - c_base);
            const int n_items = dup ? (n_sites + WAYS - 1) / WAYS : n_sites * NT;
            const int* tpi = s_tab + (wi & 1) * (2 * AV_MAXT * 128);
            const int* tpj = tpi + AV_MAXT * 128;
            mbar_wait(tab_full + (wi & 1), (wi >> 1) & 1);
            int t = 0, s = 0;                 // non-dup: tile / site of the item
            for (int k = 0; k < n_items; ++k, ++gk) {
                const int buf = gk & 1;
                int row, site, st;
                bool site_ok = true, last_use;
                if (dup) {
                    // every warp observes every phase of every ring stage (both sites of the item, in order): a warp that skipped
                    // the other parity's phases could otherwise pass a later wait on a stale phase bit
                    const int h = quad ? q : q >> 1;
                    st = rp.st;
                    for (int i = 0; i < WAYS; ++i) {
                        if (WAYS * k + i >= n_sites) break;
                        mbar_wait(full + rp.st, rp.ph);
                        if (i == h) st = rp.st;
                        rp.next(NST);
                    }
                    site = WAYS * k + h; site_ok = site < n_sites;
                    row = quad ? lane : (q & 1) * 32 + lane; last_use = true;
                } else {
                    mbar_wait(full + rp.st, rp.ph);
                    site = s; st = rp.st; row = t * 128 + q * 32 + lane; last_use = (t == NT - 1);
                    if (++t == NT) { t = 0; ++s; rp.next(NST); }
                }
                const int pi = tpi[row], pj = tpj[row];
                if (gk >= 2) { mbar_wait(a_free + buf, ((gk >> 1) - 1) & 1); tc_fence_after(); }
                uint32_t hh[8], ll[8];
                if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the previous store has read the staging buffer
                __syncwarp();
                if (site_ok && pi >= 0) {
                    const uint8_t* xb = sm + st * STG + half_off;
                    const uint8_t* xi_r = xb + pi * 128;
                    const uint8_t* xj_r = xb + pj * 128;
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int ci = ((j0 + e) ^ (pi & 7)) << 4, cj = ((j0 + e) ^ (pj & 7)) << 4;
                        const float4 xa = *reinterpret_cast<const float4*>(xi_r + ci), xc = *reinterpret_cast<const float4*>(xj_r + cj);
                        const float4 ya = *reinterpret_cast<const float4*>(xi_r + 2 * T + ci), yc = *reinterpret_cast<const float4*>(xj_r + 2 * T + cj);
                        // z x_i + (1-z) x_j in packed fp32x2 math (channel pairs share every FMA-pipe instruction; same operations and
                        // order as the scalar form)
                        const float2 z0 = sigmoid_fast2(fadd2(fsub2(make_float2(ya.x, ya.y), make_float2(yc.x, yc.y)), make_float2(bh[4 * e + 0], bh[4 * e + 1])));
                        const float2 z1 = sigmoid_fast2(fadd2(fsub2(make_float2(ya.z, ya.w), make_float2(yc.z, yc.w)), make_float2(bh[4 * e + 2], bh[4 * e + 3])));
                        const float2 v0 = ffma2(z0, fsub2(make_float2(xa.x, xa.y), make_float2(xc.x, xc.y)), make_float2(xc.x, xc.y));
                        const float2 v1 = ffma2(z1, fsub2(make_float2(xa.z, xa.w), make_float2(xc.z, xc.w)), make_float2(xc.z, xc.w));
                        const float4 v = make_float4(v0.x, v0.y, v1.x, v1.y);
                        split2(v.x, v.y, hh[2 * e], ll[2 * e]);
                        split2(v.z, v.w, hh[2 * e + 1], ll[2 * e + 1]);
                        *reinterpret_cast<float4*>(xs + ((e ^ ((lane >> 1) & 3)) << 4)) = v;
                    }
                } else {
#pragma unroll
                    for (int e = 0; e < 8; ++e) { hh[e] = 0u; ll[e] = 0u; }
#pragma unroll
                    for (int e = 0; e < 4; ++e) *reinterpret_cast<float4*>(xs + (e << 4)) = make_float4(0.f, 0.f, 0.f, 0.f);
                }
                fence_async_smem();
                tmem_st8(lane_base + AV_TM_A + buf * 64 + cg * 8, hh);
                tmem_st8(lane_base + AV_TM_A + buf * 64 + 32 + cg * 8, ll);
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if (site_ok && row < rows_cta) {   // x rows of this warp -> x planes [b][pair][site][16 channels]; the map clips rows >= nc
                        tma_store_4d(&mapXo, xs, cg * 16, c_base + site, row, b);
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    mbar_arrive(a_ready + buf);
                    if (site_ok && last_use) mbar_arrive(stage_free + st);   // this warp's last read of the stage
                }
            }
            // ---- partial alpha of this site group: TMEM -> alpha_part[pair][partial][slot]
            mbar_wait(done, wi & 1);
            tc_fence_after();
            if (cg * 16 < a.RP) {
                if (!dup) {
                    for (int tt = 0; tt < NT; ++tt) {
                        uint32_t acc[16];
                        tmem_ld16_nw(lane_base + tt * 64 + cg * 16, acc);
                        tmem_ld_wait();
                        const int row = tt * 128 + q * 32 + lane;
                        if (row < rows_cta) {
                            float* o = a.alpha_part + (((size_t)b * a.alpha_pairs + row) * a.nSG + sg) * a.RP + cg * 16;
#pragma unroll
                            for (int e = 0; e < 4; ++e)
                                if (cg * 16 + 4 * e < a.RP)
                                    st4(o + 4 * e, make_float4(__uint_as_float(acc[4 * e]), __uint_as_float(acc[4 * e + 1]), __uint_as_float(acc[4 * e + 2]), __uint_as_float(acc[4 * e + 3])));
                        }
                    }
                } else {
                    const int h = quad ? q : q >> 1, row = quad ? lane : (q & 1) * 32 + lane;
                    uint32_t acc[16];
                    tmem_ld16_nw(lane_base + h * 64 + cg * 16, acc);
                    tmem_ld_wait();
                    const bool have = h < n_sites;             // the odd-site accumulator is never written when the group has one site
                    if (row < rows_cta) {
                        float* o = a.alpha_part + (((size_t)b * a.alpha_pairs + row) * a.nSG + WAYS * sg + h) * a.RP + cg * 16;
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            if (cg * 16 + 4 * e < a.RP)
                                st4(o + 4 * e, have ? make_float4(__uint_as_float(acc[4 * e]), __uint_as_float(acc[4 * e + 1]), __uint_as_float(acc[4 * e + 2]), __uint_as_float(acc[4 * e + 3]))
                                                    : make_float4(0.f, 0.f, 0.f, 0.f));
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tab_free + (wi & 1));
        }
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    if (warp == AV_BLEND_WARPS) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
}

// ------------------------------------------------------------------ host side
// fp32 node pool [B][S][C][64] (tree stride given) as a 4-D tensor (d, site, slot, tree); box = 32 channels of all slots at one site
static int make_tmap_pool_f32(CUtensorMap* map, const float* base, size_t tree_stride, int S, int C, int B, int box_rows) {
    const cuuint64_t gdim[4] = {64, (cuuint64_t)C, (cuuint64_t)S, (cuuint64_t)B};
    const cuuint64_t gstr[3] = {256, (cuuint64_t)C * 256, (cuuint64_t)tree_stride * 4};
    const cuuint32_t box[4] = {32, 1, (cuuint32_t)box_rows, 1};
    return encode_tmap(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, base, gdim, gstr, box, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                       "the fp32 node pool");
}

// x planes [B][pc][C][64] fp32 as a 4-D tensor (d, site, pair, tree); store box = 16 channels of 32 pairs at one site (SWIZZLE_64B)
static int make_tmap_xplanes(CUtensorMap* map, float* base, int pc, int nrows, int C, int B) {
    const cuuint64_t gdim[4] = {64, (cuuint64_t)C, (cuuint64_t)nrows, (cuuint64_t)B};   // rows past the pair list are clipped by the map
    const cuuint64_t gstr[3] = {256, (cuuint64_t)C * 256, (cuuint64_t)pc * C * 256};
    const cuuint32_t box[4] = {16, 1, 32, 1};
    return encode_tmap(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, base, gdim, gstr, box, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                       "the x planes");
}

// K' planes [B][S][C][64] bf16 as a 4-D tensor (d, site, slot, tree); box = all slots of one site: [64 slots][64 d]
static int make_tmap_kprime(CUtensorMap* map, const void* base, int S, int n_live, int C, int B, int box_rows) {
    const cuuint64_t gdim[4] = {64, (cuuint64_t)C, (cuuint64_t)n_live, (cuuint64_t)B};   // slots >= n_live are dead: never loaded (zero-filled)
    const cuuint64_t gstr[3] = {128, (cuuint64_t)C * 128, (cuuint64_t)S * C * 128};
    const cuuint32_t box[4] = {64, 1, (cuuint32_t)box_rows, 1};
    return encode_tmap(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, base, gdim, gstr, box, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                       "the K' planes");
}

// writes the x planes of pairs [n0, n0+nc) and alpha_part[b][n][partial][slot]; returns the number of partials per pair in *n_part
int launch_alpha_v3(const Model* m, const PairChunk& c, int* n_part, cudaStream_t st) {
    static DevOnce once;      // per device, not per process
    if (int e = smem_opt_in(once, k_alpha_v3, AV_SMEM_MAX)) return e;
    const int n_sm = sm_count();
    if (c.S > 64) return set_error(NNJ_ERR_INVALID, "alpha_v3: at most 63 taxa on the tensor-core path");
    if (c.nc > AV_MAXT * 128 || c.nc > c.pc) return set_error(NNJ_ERR_INVALID, "alpha_v3: at most 512 pairs per launch");
    const int groups = (c.C + AV_SITES - 1) / AV_SITES;
    const bool dup = c.nc <= 64;
    const int ways = !dup ? 1 : (c.nc <= 32 && 4 * groups <= c.nAP) ? 4 : 2;
    *n_part = ways * groups;
    if (*n_part > c.nAP) return set_error(NNJ_ERR_INVALID, "alpha_v3: partial buffer too small");
    // the live nodes occupy physical slots [0, Rp) (k_select keeps them compact): only those rows are streamed
    const int rows8 = (c.Rp + 7) & ~7;
    AlphaV3Args a;
    a.tile_bytes = rows8 * 128;
    a.nmma = (rows8 + 15) & ~15;
    a.nst = (AV_SMEM_MAX - 1024 - AV_XS_BYTES - AV_MISC_BYTES) / (6 * a.tile_bytes);
    if (a.nst > AV_MAXST) a.nst = AV_MAXST;
    CUtensorMap mx, my, mh, ml, mo;
    if (int e = make_tmap_xplanes(&mo, c.xf, c.pc, c.nc, c.C, c.B)) return e;
    if (int e = make_tmap_pool_f32(&mx, c.X, c.tree_stride, c.Rp, c.C, c.B, rows8)) return e;
    if (int e = make_tmap_pool_f32(&my, c.Y, c.tree_stride, c.Rp, c.C, c.B, rows8)) return e;
    if (int e = make_tmap_kprime(&mh, c.kp_h, c.S, c.Rp, c.C, c.B, rows8)) return e;
    if (int e = make_tmap_kprime(&ml, c.kp_l, c.S, c.Rp, c.C, c.B, rows8)) return e;
    a.slot_of = c.slot_of; a.slot_stride = c.slot_stride;
    a.pair_i = c.pair_i; a.pair_j = c.pair_j; a.pair_stride = c.pair_stride; a.n0 = c.n0; a.nc = c.nc; a.C = c.C; a.B = c.B; a.groups = groups;
    a.bh = m->nj.bh;
    a.dup = dup ? 1 : 0; a.ways = ways;
    a.alpha_part = c.alpha_part; a.alpha_pairs = c.alpha_pairs; a.nSG = c.nAP; a.RP = c.RP;
    const int n_work = c.B * groups;
    const size_t smem = 1024 + (size_t)a.nst * 6 * a.tile_bytes + AV_XS_BYTES + AV_MISC_BYTES;
    prof_begin(KC_ALPHA, st);
    k_alpha_v3<<<n_work < n_sm ? n_work : n_sm, AV_THREADS, smem, st>>>(mx, my, mh, ml, mo, a);
    LAUNCH_CHECK();
    return 0;
}

}  // namespace nnj
