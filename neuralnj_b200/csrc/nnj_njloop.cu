// nnj_njloop.cu — learned neighbour-joining loop (fp32 CUDA-core path).
//
// Restates PhyloATTN.decode_zxr / decode_gg / aggregate (model.py:90-209), the select step
// (finetune_rl_search.py:140-160), the stale-score cache map (utils.py:213-251) and the
// tensor half of PhyInferEnv.step (environment.py:760-835) as device kernels over a node
// pool.  Exact algebraic restructuring (rounding-level differences only):
//   h = W_h(x_i - x_j) + b_h            = Y_i - Y_j + b_h,       Y  = W_h X        per node
//   alpha = sum_{c,d} (W_q x + b_q).K   = sum x.K' + kappa,      K' = W_q^T K, kappa = sum_c b_q.K,  K = W_k X + b_k
// so the per-pair work is: gate/blend (elementwise), alpha (pairs x nodes contraction over all
// sites), x_glob = alpha.V, the W_g gate and the s_out MLP.  Node tensors live in pools
// [B][S][C][64] addressed through a per-tree logical->physical slot table; a merge writes the
// new node into a free slot ("slot i <- new, slot j removed" becomes a table update).
// All cross-CTA reductions go through partial buffers summed in a fixed order: results are
// run-to-run deterministic.
#include "nnj_internal.h"
#include "nnj_tc.cuh"

namespace nnj {

constexpr int SB_SITES = 32;   // sites per alpha partial / score partial
constexpr int PAIR_CHUNK = 2048;

struct Pool {
    const float* X; const float* Y; const float* K;  // [B][S][C][64]
    const float* kap;                                 // [B][S][nCT] partial sums of b_q . K
    size_t tree_stride;                               // S*C*64
    int S, nCT;
};

// ------------------------------------------------------------------ [128 x 64] x [64 x 64] on the legacy tensor path
// The five 64 x 64 products of the merge step (gate, Y, K, K', G) and the four of the node-derive step are the part of those kernels
// that does not shrink with the number of live nodes.  In the tensor-core precision mode they run on mma.sync.m16n8k16 bf16 register
// fragments - A split into hi / lo on the fly from the fp32 tile in shared memory, B from the fragment-packed weights (NjFrag),
// hi*hi + hi*lo + lo*hi with fp32 accumulation like every other contraction of that mode.  Warp w owns tile rows 16w .. 16w+15.
__device__ __forceinline__ void load_wfrag(float* __restrict__ Ws, const uint4* __restrict__ Wf) {
#pragma unroll
    for (int it = 0; it < 4; ++it) {
        const int idx = it * NTHREADS + threadIdx.x;
        reinterpret_cast<uint4*>(Ws)[idx] = __ldg(Wf + idx);
    }
}
// c[nt][0..1] += row g, columns nt*8 + 2t, +1;  c[nt][2..3]: row g + 8   (g = lane / 4, t = lane % 4)
__device__ __forceinline__ void warp_mma64(float (&c)[8][4], const float* __restrict__ As, const float* __restrict__ Ws) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
    const float* ap = As + (warp * 16 + g) * LDA + 2 * t;
    const uint4* wf = reinterpret_cast<const uint4*>(Ws) + lane;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
        const float2 v0 = *reinterpret_cast<const float2*>(ap + ks * 16), v1 = *reinterpret_cast<const float2*>(ap + 8 * LDA + ks * 16);
        const float2 v2 = *reinterpret_cast<const float2*>(ap + ks * 16 + 8), v3 = *reinterpret_cast<const float2*>(ap + 8 * LDA + ks * 16 + 8);
        uint32_t ah[4], al[4];
        split2(v0.x, v0.y, ah[0], al[0]); split2(v1.x, v1.y, ah[1], al[1]);
        split2(v2.x, v2.y, ah[2], al[2]); split2(v3.x, v3.y, ah[3], al[3]);
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const uint4 wv = wf[(ks * 8 + nt) * 32];
            mma_m16n8k16(c[nt], al, wv.x, wv.y);       // lo * hi
            mma_m16n8k16(c[nt], ah, wv.z, wv.w);       // hi * lo
            mma_m16n8k16(c[nt], ah, wv.x, wv.y);       // hi * hi
        }
    }
}
__device__ __forceinline__ void frag_set_bias(float (&c)[8][4], const float* __restrict__ bias) {
    const int t = threadIdx.x & 3;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
        const float2 b = bias ? __ldg(reinterpret_cast<const float2*>(bias + nt * 8 + 2 * t)) : make_float2(0.f, 0.f);
        c[nt][0] = b.x; c[nt][1] = b.y; c[nt][2] = b.x; c[nt][3] = b.y;
    }
}
// Regroup a fragment into runs of four columns (16-byte stores, the pair packing of the bf16 planes): the two lanes of a column pair swap
// one n-tile of each tile pair p = (2p, 2p+1).  Even t ends up with columns 2t .. 2t+3 of tile 2p, odd t with columns 2t-2 .. 2t+1 of tile
// 2p+1; q[p][h] is the run of row g + 8h and starts at column frag_col4(p).
__device__ __forceinline__ void frag_to_quads(const float (&c)[8][4], float4 (&q)[4][2]) {
    const bool odd = threadIdx.x & 1;
#pragma unroll
    for (int p = 0; p < 4; ++p) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const float a0 = c[2 * p][2 * h], a1 = c[2 * p][2 * h + 1], b0 = c[2 * p + 1][2 * h], b1 = c[2 * p + 1][2 * h + 1];
            const float r0 = __shfl_xor_sync(0xffffffffu, odd ? a0 : b0, 1), r1 = __shfl_xor_sync(0xffffffffu, odd ? a1 : b1, 1);
            q[p][h] = odd ? make_float4(r0, r1, b0, b1) : make_float4(a0, a1, r0, r1);
        }
    }
}
__device__ __forceinline__ int frag_col4(int p) { const int t = threadIdx.x & 3; return (2 * p + (t & 1)) * 8 + (t >> 1) * 4; }

// ------------------------------------------------------------------ per-node derived tensors
// xs: [128][LDA] tile of node rows (x).  Produces Y, K' (global) and the kappa partial of the tile.
template <bool TC>
__device__ __forceinline__ void derive_tile(float* xs, float* tmp, float* Ws, const NjW& w, const NjFrag& wf, float* __restrict__ Yout,
                                            float* __restrict__ Kout, float* __restrict__ kap_out, int row0, int C,
                                            float* red, uint2* __restrict__ Kh = nullptr, uint2* __restrict__ Kl = nullptr,
                                            uint2* __restrict__ Nh = nullptr, uint2* __restrict__ Nl = nullptr, int S = 0, int slot = 0) {
    if constexpr (TC) {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
        const int rr[2] = {warp * 16 + g, warp * 16 + g + 8};      // tile rows of the two fragment halves
        float c[8][4];
        float4 q[4][2];
        // Y = x W_h^T
        load_wfrag(Ws, wf.h);
        __syncthreads();
        frag_set_bias(c, nullptr);
        warp_mma64(c, xs, Ws);
        frag_to_quads(c, q);
#pragma unroll
        for (int p = 0; p < 4; ++p)
#pragma unroll
            for (int h = 0; h < 2; ++h)
                if (row0 + rr[h] < C) st4(Yout + (size_t)(row0 + rr[h]) * D + frag_col4(p), q[p][h]);
        __syncthreads();
        // K = x W_k^T + b_k, kappa partial = sum over the tile's rows of b_q . K
        load_wfrag(Ws, wf.k);
        __syncthreads();
        frag_set_bias(c, w.bk);
        warp_mma64(c, xs, Ws);
        {
            float p0 = 0.f, p1 = 0.f;
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                const float2 bq = __ldg(reinterpret_cast<const float2*>(w.bq + nt * 8 + 2 * t));
                p0 = fmaf(c[nt][0], bq.x, p0); p0 = fmaf(c[nt][1], bq.y, p0);
                p1 = fmaf(c[nt][2], bq.x, p1); p1 = fmaf(c[nt][3], bq.y, p1);
            }
            p0 += __shfl_xor_sync(0xffffffffu, p0, 1); p0 += __shfl_xor_sync(0xffffffffu, p0, 2);
            p1 += __shfl_xor_sync(0xffffffffu, p1, 1); p1 += __shfl_xor_sync(0xffffffffu, p1, 2);
            if (t == 0) {
                red[rr[0]] = (row0 + rr[0] < C) ? p0 : 0.f;
                red[rr[1]] = (row0 + rr[1] < C) ? p1 : 0.f;
            }
        }
        frag_to_quads(c, q);
#pragma unroll
        for (int p = 0; p < 4; ++p)
#pragma unroll
            for (int h = 0; h < 2; ++h) st4(tmp + rr[h] * LDA + frag_col4(p), q[p][h]);
        __syncthreads();
        if (threadIdx.x < 32) {
            float s = (red[threadIdx.x] + red[threadIdx.x + 32]) + (red[threadIdx.x + 64] + red[threadIdx.x + 96]);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (threadIdx.x == 0) *kap_out = s;
        }
        // K' = K W_q
        load_wfrag(Ws, wf.q);
        __syncthreads();
        frag_set_bias(c, nullptr);
        warp_mma64(c, tmp, Ws);
        frag_to_quads(c, q);
#pragma unroll
        for (int p = 0; p < 4; ++p)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int cc = row0 + rr[h];
                if (cc < C) {
                    const int c4 = frag_col4(p);
                    st4(Kout + (size_t)cc * D + c4, q[p][h]);
                    if (Kh) {
                        uint2 oh, ol;
                        split2(q[p][h].x, q[p][h].y, oh.x, ol.x);
                        split2(q[p][h].z, q[p][h].w, oh.y, ol.y);
                        Kh[(size_t)cc * 16 + c4 / 4] = oh;
                        Kl[(size_t)cc * 16 + c4 / 4] = ol;
                    }
                }
            }
        if (Nh) {
            // site-major node planes [C][S][128] = [X | G], G = x W_g^T (no bias)
            __syncthreads();
            load_wfrag(Ws, wf.g);
            __syncthreads();
            frag_set_bias(c, nullptr);
            warp_mma64(c, xs, Ws);
            frag_to_quads(c, q);
#pragma unroll
            for (int p = 0; p < 4; ++p)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int cc = row0 + rr[h];
                    if (cc < C) {
                        const int c4 = frag_col4(p);
                        const float4 xv = ld4(xs + rr[h] * LDA + c4);
                        const size_t o = ((size_t)cc * S + slot) * 32 + c4 / 4;
                        uint2 oh, ol;
                        split2(xv.x, xv.y, oh.x, ol.x);
                        split2(xv.z, xv.w, oh.y, ol.y);
                        Nh[o] = oh; Nl[o] = ol;
                        split2(q[p][h].x, q[p][h].y, oh.x, ol.x);
                        split2(q[p][h].z, q[p][h].w, oh.y, ol.y);
                        Nh[o + 16] = oh; Nl[o + 16] = ol;
                    }
                }
        }
        return;
    }
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    float acc[8][4];
    // Y = x W_h^T   (bias b_h is added when the pair gate is formed)
    load_w64(Ws, w.wht);
    __syncthreads();
    acc_set_bias(acc, nullptr, tx);
    tile_mma64(acc, xs, Ws, ty, tx);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        int c = row0 + ty * 8 + i;
        if (c < C) st4(Yout + (size_t)c * D + tx * 4, make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]));
    }
    __syncthreads();
    // K = x W_k^T + b_k
    load_w64(Ws, w.wkt);
    __syncthreads();
    acc_set_bias(acc, w.bk, tx);
    tile_mma64(acc, xs, Ws, ty, tx);
    acc_store_smem(acc, tmp, ty, tx);
    {
        float4 bq = __ldg(reinterpret_cast<const float4*>(w.bq) + tx);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float p = acc[i][0] * bq.x;
            p = fmaf(acc[i][1], bq.y, p); p = fmaf(acc[i][2], bq.z, p); p = fmaf(acc[i][3], bq.w, p);
            p = reduce16(p);
            int c = row0 + ty * 8 + i;
            if (tx == 0) red[ty * 8 + i] = (c < C) ? p : 0.f;
        }
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        float s = (red[threadIdx.x] + red[threadIdx.x + 32]) + (red[threadIdx.x + 64] + red[threadIdx.x + 96]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (threadIdx.x == 0) *kap_out = s;
    }
    // K' = K W_q   (Ws[k=d][col=e] = Wq[d][e], i.e. the untransposed torch weight)
    load_w64(Ws, w.wq);
    __syncthreads();
    acc_set_bias(acc, nullptr, tx);
    tile_mma64(acc, tmp, Ws, ty, tx);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        int c = row0 + ty * 8 + i;
        if (c < C) {
            st4(Kout + (size_t)c * D + tx * 4, make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]));
            if (Kh) {   // bf16 hi/lo planes of K' (B operand of the tensor-core alpha GEMM)
                uint2 oh, ol;
                split2(acc[i][0], acc[i][1], oh.x, ol.x);
                split2(acc[i][2], acc[i][3], oh.y, ol.y);
                Kh[(size_t)c * 16 + tx] = oh;
                Kl[(size_t)c * 16 + tx] = ol;
            }
        }
    }
    if (Nh) {
        // site-major node planes [C][S][128] = [X | G], G = x W_g^T (no bias): the B operand of the fused pair-score UMMA
        __syncthreads();
        load_w64(Ws, w.wgt);
        __syncthreads();
        acc_set_bias(acc, nullptr, tx);
        tile_mma64(acc, xs, Ws, ty, tx);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            int c = row0 + ty * 8 + i;
            if (c < C) {
                const float4 xv = ld4(xs + (ty * 8 + i) * LDA + tx * 4);
                const size_t o = ((size_t)c * S + slot) * 32 + tx;
                uint2 oh, ol;
                split2(xv.x, xv.y, oh.x, ol.x);
                split2(xv.z, xv.w, oh.y, ol.y);
                Nh[o] = oh; Nl[o] = ol;
                split2(acc[i][0], acc[i][1], oh.x, ol.x);
                split2(acc[i][2], acc[i][3], oh.y, ol.y);
                Nh[o + 16] = oh; Nl[o + 16] = ol;
            }
        }
    }
}

// grid (nCT, n_nodes, B): derive Y/K'/kappa for physical slots node_list[b][k] (or slot k when null)
template <bool TC>
__global__ void __launch_bounds__(NTHREADS) k_node_derive(const float* __restrict__ X, float* __restrict__ Y, float* __restrict__ K,
                                                          float* __restrict__ kap, size_t tree_stride, int S, int C, int nCT,
                                                          const int32_t* __restrict__ node_list, int list_stride, NjW w, NjFrag wf,
                                                          uint2* __restrict__ Kh, uint2* __restrict__ Kl, uint2* __restrict__ Nh,
                                                          uint2* __restrict__ Nl) {
    extern __shared__ __align__(16) float smem[];
    float* xs = smem;
    float* tmp = xs + TILE_ROWS * LDA;
    float* Ws = tmp + TILE_ROWS * LDA;
    float* red = Ws + 4096;
    const int b = blockIdx.z, ct = blockIdx.x;
    const int slot = node_list ? node_list[(size_t)b * list_stride + blockIdx.y] : (int)blockIdx.y;
    const size_t base = (size_t)b * tree_stride + (size_t)slot * C * D;
    const int row0 = ct * TILE_ROWS;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        int idx = it * NTHREADS + threadIdx.x;
        int row = idx >> 4, c4 = idx & 15;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row0 + row < C) v = ld4(X + base + (size_t)(row0 + row) * D + c4 * 4);
        st4(xs + row * LDA + c4 * 4, v);
    }
    __syncthreads();
    derive_tile<TC>(xs, tmp, Ws, w, wf, Y + base, K + base, kap + ((size_t)b * S + slot) * nCT + ct, row0, C, red,
                Kh ? Kh + base / 4 : nullptr, Kl ? Kl + base / 4 : nullptr, Nh ? Nh + (size_t)b * C * S * 32 : nullptr,
                Nl ? Nl + (size_t)b * C * S * 32 : nullptr, S, slot);
}

// ------------------------------------------------------------------ pair blend helper
// x = z*x_i + (1-z)*x_j,  z = sigmoid(Y_i - Y_j + b_h)     (model.py:105-108)
__device__ __forceinline__ float4 blend4(float4 xi, float4 xj, float4 yi, float4 yj, float4 bh) {
    float4 o;
    float z;
    z = sigmoidf_(yi.x - yj.x + bh.x); o.x = fmaf(z, xi.x, (1.0f - z) * xj.x);
    z = sigmoidf_(yi.y - yj.y + bh.y); o.y = fmaf(z, xi.y, (1.0f - z) * xj.y);
    z = sigmoidf_(yi.z - yj.z + bh.z); o.z = fmaf(z, xi.z, (1.0f - z) * xj.z);
    z = sigmoidf_(yi.w - yj.w + bh.w); o.w = fmaf(z, xi.w, (1.0f - z) * xj.w);
    return o;
}

// ------------------------------------------------------------------ alpha partials: pairs x nodes over a block of sites
// grid (nSB, pair_tiles * node_tiles, B).  alpha_part[b][n][sb][r] = sum_{c in block, d} x[n,c,d] K'[r,c,d]
__global__ void __launch_bounds__(NTHREADS) k_alpha(Pool pool, const int32_t* __restrict__ slot_of, int slot_stride, int Rp, int C,
                                                    const int32_t* __restrict__ pair_i, const int32_t* __restrict__ pair_j,
                                                    int pair_stride, int n0, int nc, int node_tiles, const float* __restrict__ bh,
                                                    float* __restrict__ alpha_part, int nSB, int RP) {
    __shared__ __align__(16) float As[64][LDA];   // [d][pair]
    __shared__ __align__(16) float Bs[64][LDA];   // [d][node]
    __shared__ int s_pi[64], s_pj[64], s_nd[64];
    const int b = blockIdx.z, sb = blockIdx.x;
    const int pt = blockIdx.y / node_tiles, nt = blockIdx.y - pt * node_tiles;
    const int tid = threadIdx.x;
    const int32_t* so = slot_of + (size_t)b * slot_stride;
    if (tid < 64) {
        int n = pt * 64 + tid;
        int pi = -1, pj = -1;
        if (n < nc) {
            int li = pair_i[(size_t)b * pair_stride + n0 + n], lj = pair_j[(size_t)b * pair_stride + n0 + n];
            if (li >= 0) { pi = so[li]; pj = so[lj]; }
        }
        s_pi[tid] = pi; s_pj[tid] = pj;
        int r = nt * 64 + tid;
        s_nd[tid] = r < Rp ? so[r] : -1;
    }
    __syncthreads();
    const int lp = tid & 63, dq = tid >> 6;      // loader: pair/node lp, d range dq*16..+15
    const int tx = tid & 15, ty = tid >> 4;      // compute: pairs ty*4..+3, nodes tx*4..+3
    const size_t tb = (size_t)b * pool.tree_stride;
    const int pi = s_pi[lp], pj = s_pj[lp], nd = s_nd[lp];
    float4 bh4[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) bh4[e] = __ldg(reinterpret_cast<const float4*>(bh) + dq * 4 + e);
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    const int c_end = min(C, (sb + 1) * SB_SITES);
    for (int c = sb * SB_SITES; c < c_end; ++c) {
        float4 xa[4], kb[4];
        if (pi >= 0) {
            const size_t oi = tb + ((size_t)pi * C + c) * D + dq * 16, oj = tb + ((size_t)pj * C + c) * D + dq * 16;
#pragma unroll
            for (int e = 0; e < 4; ++e)
                xa[e] = blend4(ld4(pool.X + oi + e * 4), ld4(pool.X + oj + e * 4), ld4(pool.Y + oi + e * 4), ld4(pool.Y + oj + e * 4), bh4[e]);
        } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) xa[e] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (nd >= 0) {
            const size_t on = tb + ((size_t)nd * C + c) * D + dq * 16;
#pragma unroll
            for (int e = 0; e < 4; ++e) kb[e] = ld4(pool.K + on + e * 4);
        } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) kb[e] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        __syncthreads();   // previous site's tiles fully consumed
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            int d = dq * 16 + e * 4;
            As[d][lp] = xa[e].x; As[d + 1][lp] = xa[e].y; As[d + 2][lp] = xa[e].z; As[d + 3][lp] = xa[e].w;
            Bs[d][lp] = kb[e].x; Bs[d + 1][lp] = kb[e].y; Bs[d + 2][lp] = kb[e].z; Bs[d + 3][lp] = kb[e].w;
        }
        __syncthreads();
#pragma unroll 16
        for (int d = 0; d < 64; ++d) {
            float4 a = ld4(&As[d][ty * 4]), k4 = ld4(&Bs[d][tx * 4]);
            acc[0][0] = fmaf(a.x, k4.x, acc[0][0]); acc[0][1] = fmaf(a.x, k4.y, acc[0][1]); acc[0][2] = fmaf(a.x, k4.z, acc[0][2]); acc[0][3] = fmaf(a.x, k4.w, acc[0][3]);
            acc[1][0] = fmaf(a.y, k4.x, acc[1][0]); acc[1][1] = fmaf(a.y, k4.y, acc[1][1]); acc[1][2] = fmaf(a.y, k4.z, acc[1][2]); acc[1][3] = fmaf(a.y, k4.w, acc[1][3]);
            acc[2][0] = fmaf(a.z, k4.x, acc[2][0]); acc[2][1] = fmaf(a.z, k4.y, acc[2][1]); acc[2][2] = fmaf(a.z, k4.z, acc[2][2]); acc[2][3] = fmaf(a.z, k4.w, acc[2][3]);
            acc[3][0] = fmaf(a.w, k4.x, acc[3][0]); acc[3][1] = fmaf(a.w, k4.y, acc[3][1]); acc[3][2] = fmaf(a.w, k4.z, acc[3][2]); acc[3][3] = fmaf(a.w, k4.w, acc[3][3]);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int n = pt * 64 + ty * 4 + i;
        if (n >= nc) continue;
        float* o = alpha_part + (((size_t)b * PAIR_CHUNK + n) * nSB + sb) * RP;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int r = nt * 64 + tx * 4 + j;
            if (r < Rp) o[r] = acc[i][j];
        }
    }
}

// single pair per tree (the merge pair): grid (nSB, B).  Writes alpha_part[b][0][sb][r].
__global__ void __launch_bounds__(NTHREADS) k_alpha1(Pool pool, const int32_t* __restrict__ slot_of, int slot_stride, int Rp, int C,
                                                     const int32_t* __restrict__ merge_ij, int ij_stride, const float* __restrict__ bh,
                                                     float* __restrict__ alpha_part, int nSB, int RP) {
    __shared__ __align__(16) float xs[SB_SITES * D];
    const int b = blockIdx.y, sb = blockIdx.x, tid = threadIdx.x;
    const int32_t* so = slot_of + (size_t)b * slot_stride;
    const int li = merge_ij[(size_t)b * ij_stride], lj = merge_ij[(size_t)b * ij_stride + 1];
    const int pi = so[li], pj = so[lj];
    const size_t tb = (size_t)b * pool.tree_stride;
    const int c0 = sb * SB_SITES;
    {
        int s = tid >> 3, d8 = (tid & 7) * 8;
        int c = c0 + s;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
            if (c < C) {
                size_t oi = tb + ((size_t)pi * C + c) * D + d8 + e * 4, oj = tb + ((size_t)pj * C + c) * D + d8 + e * 4;
                o = blend4(ld4(pool.X + oi), ld4(pool.X + oj), ld4(pool.Y + oi), ld4(pool.Y + oj),
                           __ldg(reinterpret_cast<const float4*>(bh + d8 + e * 4)));
            }
            st4(xs + s * D + d8 + e * 4, o);
        }
    }
    __syncthreads();
    const int warp = tid >> 5, lane = tid & 31;
    const int nsite = min(SB_SITES, C - c0);
    for (int r = warp; r < Rp; r += 8) {
        const float* kp = pool.K + tb + ((size_t)so[r] * C + c0) * D;
        float s = 0.f;
        for (int m = 0; m < 16; ++m) {
            int f4 = lane + 32 * m;               // float4 index within the [32 sites][64] block
            if ((f4 >> 4) < nsite) {
                float4 kv = ld4(kp + f4 * 4), xv = ld4(xs + f4 * 4);
                s = fmaf(kv.x, xv.x, s); s = fmaf(kv.y, xv.y, s); s = fmaf(kv.z, xv.z, s); s = fmaf(kv.w, xv.w, s);
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) alpha_part[(((size_t)b * PAIR_CHUNK) * nSB + sb) * RP + r] = s;
    }
}

// one warp per (tree, pair): reduce partials, add kappa, scale, mask i/j, softmax over nodes  (model.py:118-146)
__global__ void __launch_bounds__(NTHREADS) k_alpha_softmax(const float* __restrict__ alpha_part, const float* __restrict__ kap,
                                                            const int32_t* __restrict__ slot_of, int slot_stride, int S, int nCT,
                                                            int Rp, const int32_t* __restrict__ pair_i, const int32_t* __restrict__ pair_j,
                                                            int pair_stride, int n0, int nc, int nSB, int RP, float inv_scale,
                                                            float* __restrict__ alpha, int by_slot, int n_part) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = blockIdx.x * 8 + warp, b = blockIdx.y;
    if (n >= nc) return;
    const int li = pair_i[(size_t)b * pair_stride + n0 + n], lj = pair_j[(size_t)b * pair_stride + n0 + n];
    float* out = alpha + ((size_t)b * PAIR_CHUNK + n) * RP;
    if (li < 0) {
        for (int r = lane; r < Rp; r += 32) out[r] = 0.f;
        return;
    }
    const float* ap = alpha_part + ((size_t)b * PAIR_CHUNK + n) * nSB * RP;
    const int32_t* so = slot_of + (size_t)b * slot_stride;
    float m = -INFINITY;
    for (int r = lane; r < Rp; r += 32) {
        float s = 0.f;
        const int col = by_slot ? so[r] : r;   // tensor-core alpha partials are indexed by physical slot
        for (int k = 0; k < n_part; ++k) s += ap[(size_t)k * RP + col];   // n_part <= nSB partials, fixed order
        const float* kp = kap + ((size_t)b * S + so[r]) * nCT;
        float kk = 0.f;
        for (int k = 0; k < nCT; ++k) kk += kp[k];
        s = (s + kk) * inv_scale;
        if (r == li || r == lj) s = -INFINITY;
        out[r] = s;
        m = fmaxf(m, s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float l = 0.f;
    for (int r = lane; r < Rp; r += 32) {
        float e = expf(out[r] - m);
        out[r] = e;
        l += e;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
    const float inv = 1.0f / l;
    for (int r = lane; r < Rp; r += 32) out[r] *= inv;
}

// The same for up to 256 nodes with many partials (large-slot path: <= 64 K splits of the alpha GEMM, indexed by physical slot): one CTA
// per (tree, pair), thread r = node r, so the partial rows are read coalesced and the dependent-load chain of a lane is the number of
// partials, not partials x nodes / 32.  Fixed summation order: deterministic.
__global__ void __launch_bounds__(NTHREADS) k_alpha_softmax_wide(const float* __restrict__ alpha_part, const float* __restrict__ kap,
                                                                 const int32_t* __restrict__ slot_of, int slot_stride, int S, int nCT, int Rp,
                                                                 const int32_t* __restrict__ pair_i, const int32_t* __restrict__ pair_j,
                                                                 int pair_stride, int n0, int nc, int nSB, int RP, float inv_scale,
                                                                 float* __restrict__ alpha, int n_part) {
    __shared__ float s_red[NTHREADS / 32];
    const int n = blockIdx.x, b = blockIdx.y, r = threadIdx.x, warp = r >> 5, lane = r & 31;
    const int li = pair_i[(size_t)b * pair_stride + n0 + n], lj = pair_j[(size_t)b * pair_stride + n0 + n];
    float* out = alpha + ((size_t)b * PAIR_CHUNK + n) * RP;
    if (li < 0) {
        if (r < Rp) out[r] = 0.f;
        return;
    }
    float v = -INFINITY;
    if (r < Rp) {
        const int col = slot_of[(size_t)b * slot_stride + r];
        const float* ap = alpha_part + ((size_t)b * PAIR_CHUNK + n) * nSB * RP + col;
        float s = 0.f;
        for (int k = 0; k < n_part; ++k) s += ap[(size_t)k * RP];
        const float* kp = kap + ((size_t)b * S + col) * nCT;
        float kk = 0.f;
        for (int k = 0; k < nCT; ++k) kk += kp[k];
        v = (r == li || r == lj) ? -INFINITY : (s + kk) * inv_scale;
    }
    float m = v;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) s_red[warp] = m;
    __syncthreads();
    m = s_red[0];
#pragma unroll
    for (int w = 1; w < NTHREADS / 32; ++w) m = fmaxf(m, s_red[w]);
    __syncthreads();
    const float e = r < Rp ? expf(v - m) : 0.f;
    float l = e;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
    if (lane == 0) s_red[warp] = l;
    __syncthreads();
    l = 0.f;
#pragma unroll
    for (int w = 0; w < NTHREADS / 32; ++w) l += s_red[w];
    if (r < Rp) out[r] = e * (1.0f / l);
}

// ------------------------------------------------------------------ pair scores
// grid (nSG, ceil(nc/32), B).  CTA tile = 32 pairs x 4 sites per iteration, 8 iterations (32 sites).
// rows of the [128][64] tile: row = site_local*32 + pair_local.
template <bool GLOB>
__global__ void __launch_bounds__(NTHREADS) k_score(Pool pool, const int32_t* __restrict__ slot_of, int slot_stride, int Rp, int C,
                                                    const int32_t* __restrict__ pair_i, const int32_t* __restrict__ pair_j,
                                                    int pair_stride, int n0, int nc, const float* __restrict__ alpha, int RP,
                                                    NjW w, const uint8_t* __restrict__ mask, float* __restrict__ score_part, int nSG) {
    extern __shared__ __align__(16) float smem[];
    float* Wg = smem;                          // [64][64]
    float* Wsd = Wg + 4096;                    // [64][64]
    float* xs = Wsd + 4096;                    // [128][LDA]
    float* xg = xs + TILE_ROWS * LDA;          // [128][LDA]; also the V chunk [32 nodes][4 sites][64]
    float* tot = xg + TILE_ROWS * LDA;         // [16][8]
    int* s_pi = reinterpret_cast<int*>(tot + 128);   // [32]
    int* s_pj = s_pi + 32;                     // [32]
    int* s_slot = s_pj + 32;                   // [Rp]
    float* al = reinterpret_cast<float*>(s_slot + ((Rp + 3) & ~3));   // [Rp][32]
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int b = blockIdx.z, ptile = blockIdx.y, sg = blockIdx.x;
    const int32_t* so = slot_of + (size_t)b * slot_stride;
    const size_t tb = (size_t)b * pool.tree_stride;
    if (GLOB) load_w64(Wg, w.wgt);
    load_w64(Wsd, w.wst);
    if (tid < 32) {
        int n = ptile * 32 + tid, pi = -1, pj = -1;
        if (n < nc) {
            int li = pair_i[(size_t)b * pair_stride + n0 + n], lj = pair_j[(size_t)b * pair_stride + n0 + n];
            if (li >= 0) { pi = so[li]; pj = so[lj]; }
        }
        s_pi[tid] = pi; s_pj[tid] = pj;
    }
    if (GLOB) {
        for (int r = tid; r < Rp; r += NTHREADS) s_slot[r] = so[r];
        for (int idx = tid; idx < Rp * 32; idx += NTHREADS) {
            int p = idx / Rp, r = idx - p * Rp;
            int n = ptile * 32 + p;
            al[r * 32 + p] = (n < nc) ? alpha[((size_t)b * PAIR_CHUNK + n) * RP + r] : 0.f;
        }
    }
    __syncthreads();
    const float4 w2 = __ldg(reinterpret_cast<const float4*>(w.w2) + tx);
    float sc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) sc[i] = 0.f;
    const int sl = ty >> 2, pg = (ty & 3) * 8;
    for (int it = 0; it < SB_SITES / 4; ++it) {
        const int s0 = sg * SB_SITES + it * 4;
        if (s0 >= C) break;
        // (a) blended pair rows
        {
            int row = tid >> 1, half = tid & 1;
            int rs = row >> 5, rp = row & 31;
            int c = s0 + rs;
            int pi = s_pi[rp], pj = s_pj[rp];
            float* dst = xs + row * LDA + half * 32;
            if (pi >= 0 && c < C) {
                size_t oi = tb + ((size_t)pi * C + c) * D + half * 32, oj = tb + ((size_t)pj * C + c) * D + half * 32;
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    st4(dst + e * 4, blend4(ld4(pool.X + oi + e * 4), ld4(pool.X + oj + e * 4), ld4(pool.Y + oi + e * 4),
                                            ld4(pool.Y + oj + e * 4), __ldg(reinterpret_cast<const float4*>(w.bh) + half * 8 + e)));
            } else {
#pragma unroll
                for (int e = 0; e < 8; ++e) st4(dst + e * 4, make_float4(0.f, 0.f, 0.f, 0.f));
            }
        }
        float acc[8][4];
        if (GLOB) {
            // (b) x_glob = sum_r alpha[pair][r] * V[r][site]     (model.py:148)
#pragma unroll
            for (int i = 0; i < 8; ++i) { acc[i][0] = 0.f; acc[i][1] = 0.f; acc[i][2] = 0.f; acc[i][3] = 0.f; }
            for (int r0 = 0; r0 < Rp; r0 += 32) {
                __syncthreads();
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    int idx = k * NTHREADS + tid;
                    int node = idx >> 6, rem = idx & 63, site = rem >> 4, c4 = rem & 15;
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (r0 + node < Rp && s0 + site < C)
                        v = ld4(pool.X + tb + ((size_t)s_slot[r0 + node] * C + s0 + site) * D + c4 * 4);
                    st4(xg + (node * 4 + site) * D + c4 * 4, v);
                }
                __syncthreads();
                const int nn = min(32, Rp - r0);
                for (int node = 0; node < nn; ++node) {
                    float4 v = ld4(xg + (node * 4 + sl) * D + tx * 4);
                    float4 a0 = ld4(al + (r0 + node) * 32 + pg), a1 = ld4(al + (r0 + node) * 32 + pg + 4);
                    float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        acc[i][0] = fmaf(a[i], v.x, acc[i][0]); acc[i][1] = fmaf(a[i], v.y, acc[i][1]);
                        acc[i][2] = fmaf(a[i], v.z, acc[i][2]); acc[i][3] = fmaf(a[i], v.w, acc[i][3]);
                    }
                }
            }
            __syncthreads();
            // (c) x_glob tile -> smem
            acc_store_smem(acc, xg, ty, tx);
            __syncthreads();
            // (d) w = sigmoid(W_g x_glob + b_g);  x' = (1-w) x + w x_glob    (model.py:150-153)
            float g[8][4];
            acc_set_bias(g, w.bg, tx);
            tile_mma64(g, xg, Wg, ty, tx);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float* xp = xs + (ty * 8 + i) * LDA + tx * 4;
                float4 xv = ld4(xp);
                float wv;
                wv = sigmoidf_(g[i][0]); xv.x = fmaf(wv, acc[i][0], (1.0f - wv) * xv.x);
                wv = sigmoidf_(g[i][1]); xv.y = fmaf(wv, acc[i][1], (1.0f - wv) * xv.y);
                wv = sigmoidf_(g[i][2]); xv.z = fmaf(wv, acc[i][2], (1.0f - wv) * xv.z);
                wv = sigmoidf_(g[i][3]); xv.w = fmaf(wv, acc[i][3], (1.0f - wv) * xv.w);
                st4(xp, xv);
            }
        }
        __syncthreads();
        // (e) score = w2 . GELU(W_s x' + b_s) + b2, masked site sum        (model.py:95-97)
        acc_set_bias(acc, w.bs, tx);
        tile_mma64(acc, xs, Wsd, ty, tx);
        {
            int c = s0 + sl;
            float valid = (c < C && !(mask && mask[(size_t)b * C + c])) ? 1.0f : 0.0f;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float p = gelu_erf(acc[i][0]) * w2.x;
                p = fmaf(gelu_erf(acc[i][1]), w2.y, p); p = fmaf(gelu_erf(acc[i][2]), w2.z, p); p = fmaf(gelu_erf(acc[i][3]), w2.w, p);
                p = reduce16(p);
                sc[i] += (p + w.b2) * valid;
            }
        }
        __syncthreads();
    }
    if (tx == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) tot[ty * 8 + i] = sc[i];
    }
    __syncthreads();
    if (tid < 32) {
        int n = ptile * 32 + tid;
        if (n < nc) {
            int g8 = tid >> 3, i = tid & 7;
            float s = 0.f;
#pragma unroll
            for (int s4 = 0; s4 < 4; ++s4) s += tot[(s4 * 4 + g8) * 8 + i];
            score_part[((size_t)b * PAIR_CHUNK + n) * nSG + sg] = (s_pi[tid] >= 0) ? s : 0.f;
        }
    }
}

__global__ void k_score_reduce(const float* __restrict__ score_part, int nSG, int count, int nc, float* __restrict__ scores, int score_stride, int n0) {
    int n = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
    if (n >= nc) return;
    const float* p = score_part + ((size_t)b * PAIR_CHUNK + n) * nSG;
    float s = 0.f;
    for (int k = 0; k < count; ++k) s += p[k];
    scores[(size_t)b * score_stride + n0 + n] = s;
}

// ------------------------------------------------------------------ merged-node embedding (+ derived tensors)
// grid (nCT, B).  Rows = 128 sites of the merge pair.  out_x: where x' goes ([B] stride out_stride);
// when `derive` the Y/K'/kappa of the new node are produced as well (physical slot new_slot[b]).
template <bool GLOB, bool TC>
__global__ void __launch_bounds__(NTHREADS) k_merge(Pool pool, float* __restrict__ Xw, float* __restrict__ Yw, float* __restrict__ Kw,
                                                    float* __restrict__ kapw, const int32_t* __restrict__ slot_of, int slot_stride,
                                                    int Rp, int C, const int32_t* __restrict__ merge_ij, int ij_stride,
                                                    const float* __restrict__ alpha, int RP, NjW w, NjFrag wf, float* __restrict__ out_x,
                                                    size_t out_stride, const int32_t* __restrict__ new_slot, int derive,
                                                    uint2* __restrict__ nodes_h, uint2* __restrict__ nodes_l, uint2* __restrict__ kp_h,
                                                    uint2* __restrict__ kp_l, const int32_t* __restrict__ move_dst) {
    extern __shared__ __align__(16) float smem[];
    float* xs = smem;
    float* xg = xs + TILE_ROWS * LDA;
    float* Ws = xg + TILE_ROWS * LDA;
    float* red = Ws + 4096;          // [128]
    float* al = red + 128;           // [Rp]
    int* s_slot = reinterpret_cast<int*>(al + ((Rp + 3) & ~3));
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int b = blockIdx.y, ct = blockIdx.x, row0 = ct * TILE_ROWS;
    const int32_t* so = slot_of + (size_t)b * slot_stride;
    const size_t tb = (size_t)b * pool.tree_stride;
    const int li = merge_ij[(size_t)b * ij_stride], lj = merge_ij[(size_t)b * ij_stride + 1];
    const int pi = so[li], pj = so[lj];
    if (GLOB) {
        if constexpr (TC) load_wfrag(Ws, wf.g); else load_w64(Ws, w.wgt);
        for (int r = tid; r < Rp; r += NTHREADS) { s_slot[r] = so[r]; al[r] = alpha[(size_t)b * PAIR_CHUNK * RP + r]; }
    }
    {
        int row = tid >> 1, half = tid & 1;
        int c = row0 + row;
        float* dst = xs + row * LDA + half * 32;
        if (c < C) {
            size_t oi = tb + ((size_t)pi * C + c) * D + half * 32, oj = tb + ((size_t)pj * C + c) * D + half * 32;
            // loads first, in two batches of 16 (the shared-memory stores below may alias them for the compiler: without the explicit
            // batches every 16-byte group waited for its own DRAM round trip)
#pragma unroll
            for (int e0 = 0; e0 < 8; e0 += 4) {
                float4 xi[4], xj[4], yi[4], yj[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    xi[e] = ld4(pool.X + oi + (e0 + e) * 4); xj[e] = ld4(pool.X + oj + (e0 + e) * 4);
                    yi[e] = ld4(pool.Y + oi + (e0 + e) * 4); yj[e] = ld4(pool.Y + oj + (e0 + e) * 4);
                }
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    st4(dst + (e0 + e) * 4, blend4(xi[e], xj[e], yi[e], yj[e], __ldg(reinterpret_cast<const float4*>(w.bh) + half * 8 + e0 + e)));
            }
        } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) st4(dst + e * 4, make_float4(0.f, 0.f, 0.f, 0.f));
        }
    }
    __syncthreads();
    float* xo = out_x + (size_t)b * out_stride;
    if (GLOB) {
        float acc[8][4];
#pragma unroll
        for (int i = 0; i < 8; ++i) { acc[i][0] = 0.f; acc[i][1] = 0.f; acc[i][2] = 0.f; acc[i][3] = 0.f; }
        // alpha is exactly 0 at r = li, lj (softmax of -inf), so those nodes add nothing and the loop needs no branch; two nodes per
        // iteration keep 16 independent 16-byte loads in flight per thread (rows past C: clamped to the last row, weight 0 below)
        const int rclamp = C - 1 - row0 - ty * 8;           // last valid row offset of this thread's 8 rows (may be negative: tile past C)
        auto node_ptr = [&](int r) { return pool.X + tb + ((size_t)s_slot[r] * C + row0 + ty * 8) * D + tx * 4; };
        int r = 0;
        if (rclamp >= 7) {
            for (; r + 1 < Rp; r += 2) {
                const float a0 = al[r], a1 = al[r + 1];
                const float* v0p = node_ptr(r);
                const float* v1p = node_ptr(r + 1);
                float4 v0[8], v1[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) { v0[i] = ld4(v0p + (size_t)i * D); v1[i] = ld4(v1p + (size_t)i * D); }
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    acc[i][0] = fmaf(a0, v0[i].x, acc[i][0]); acc[i][1] = fmaf(a0, v0[i].y, acc[i][1]);
                    acc[i][2] = fmaf(a0, v0[i].z, acc[i][2]); acc[i][3] = fmaf(a0, v0[i].w, acc[i][3]);
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    acc[i][0] = fmaf(a1, v1[i].x, acc[i][0]); acc[i][1] = fmaf(a1, v1[i].y, acc[i][1]);
                    acc[i][2] = fmaf(a1, v1[i].z, acc[i][2]); acc[i][3] = fmaf(a1, v1[i].w, acc[i][3]);
                }
            }
        }
        for (; r < Rp; ++r) {
            const float a = al[r];
            const float* vp = node_ptr(r);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                if (i <= rclamp) {
                    float4 v = ld4(vp + (size_t)i * D);
                    acc[i][0] = fmaf(a, v.x, acc[i][0]); acc[i][1] = fmaf(a, v.y, acc[i][1]);
                    acc[i][2] = fmaf(a, v.z, acc[i][2]); acc[i][3] = fmaf(a, v.w, acc[i][3]);
                }
            }
        }
        acc_store_smem(acc, xg, ty, tx);
        __syncthreads();
        if constexpr (TC) {
            // gate on register fragments: every element of the tile is owned by exactly one thread in both layouts
            const int lane = tid & 31, warp = tid >> 5;
            const int rr[2] = {warp * 16 + (lane >> 2), warp * 16 + (lane >> 2) + 8};
            float c[8][4];
            float4 q[4][2];
            frag_set_bias(c, w.bg);
            warp_mma64(c, xg, Ws);
            frag_to_quads(c, q);
#pragma unroll
            for (int p = 0; p < 4; ++p)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    float* xp = xs + rr[h] * LDA + frag_col4(p);
                    const float4 gl = ld4(xg + rr[h] * LDA + frag_col4(p));
                    float4 xv = ld4(xp);
                    float wv;
                    wv = sigmoidf_(q[p][h].x); xv.x = fmaf(wv, gl.x, (1.0f - wv) * xv.x);
                    wv = sigmoidf_(q[p][h].y); xv.y = fmaf(wv, gl.y, (1.0f - wv) * xv.y);
                    wv = sigmoidf_(q[p][h].z); xv.z = fmaf(wv, gl.z, (1.0f - wv) * xv.z);
                    wv = sigmoidf_(q[p][h].w); xv.w = fmaf(wv, gl.w, (1.0f - wv) * xv.w);
                    st4(xp, xv);
                }
            __syncthreads();
        } else {
        float g[8][4];
        acc_set_bias(g, w.bg, tx);
        tile_mma64(g, xg, Ws, ty, tx);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float* xp = xs + (ty * 8 + i) * LDA + tx * 4;
            float4 xv = ld4(xp);
            float wv;
            wv = sigmoidf_(g[i][0]); xv.x = fmaf(wv, acc[i][0], (1.0f - wv) * xv.x);
            wv = sigmoidf_(g[i][1]); xv.y = fmaf(wv, acc[i][1], (1.0f - wv) * xv.y);
            wv = sigmoidf_(g[i][2]); xv.z = fmaf(wv, acc[i][2], (1.0f - wv) * xv.z);
            wv = sigmoidf_(g[i][3]); xv.w = fmaf(wv, acc[i][3], (1.0f - wv) * xv.w);
            st4(xp, xv);
        }
        __syncthreads();
        }
    }
    if (derive) {
        const int ns = new_slot[b];
        const size_t nb = tb + (size_t)ns * C * D;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            int c = row0 + ty * 8 + i;
            if (c < C) {
                const float4 v = ld4(xs + (ty * 8 + i) * LDA + tx * 4);
                st4(Xw + nb + (size_t)c * D + tx * 4, v);
            }
        }
        derive_tile<TC>(xs, xg, Ws, w, wf, Yw + nb, Kw + nb, kapw + ((size_t)b * pool.S + ns) * pool.nCT + ct, row0, C, red,
                    kp_h ? kp_h + nb / 4 : nullptr, kp_l ? kp_l + nb / 4 : nullptr, nodes_h ? nodes_h + (size_t)b * C * pool.S * 32 : nullptr,
                    nodes_l ? nodes_l + (size_t)b * C * pool.S * 32 : nullptr, pool.S, ns);
        // ---- compaction: this tile's rows of the last live node (slot Rp-1) -> the freed slot move_dst[b] (k_select).  Everything this
        //      CTA read from the destination slot (the pair's x, Y) was consumed above; other CTAs own other sites.
        const int dst = move_dst ? move_dst[b] : -1;
        if (dst >= 0) {
            const int src = Rp - 1;
            const int rows = min(TILE_ROWS, C - row0);
            const size_t so_ = tb + ((size_t)src * C + row0) * D, do_ = tb + ((size_t)dst * C + row0) * D;
            // Source and destination slots never overlap, but they live in the same arrays, so the compiler keeps every load behind
            // the previous store: a plain copy loop makes one DRAM round trip per 16 bytes and thread.  Each plane is therefore copied
            // as "all loads of this thread, then all stores" (TILE_ROWS * 16 / NTHREADS = 8 uint4 per thread and plane).
            auto copy8 = [&](const uint4* __restrict__ sp, uint4* __restrict__ dp, int n16) {
                uint4 v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) { const int k = tid + u * NTHREADS; if (k < n16) v[u] = sp[k]; }
#pragma unroll
                for (int u = 0; u < 8; ++u) { const int k = tid + u * NTHREADS; if (k < n16) dp[k] = v[u]; }
            };
            copy8(reinterpret_cast<const uint4*>(Xw + so_), reinterpret_cast<uint4*>(Xw + do_), rows * 16);
            copy8(reinterpret_cast<const uint4*>(Yw + so_), reinterpret_cast<uint4*>(Yw + do_), rows * 16);
            copy8(reinterpret_cast<const uint4*>(Kw + so_), reinterpret_cast<uint4*>(Kw + do_), rows * 16);
            if (kp_h) {
                copy8(reinterpret_cast<const uint4*>(kp_h) + so_ / 8, reinterpret_cast<uint4*>(kp_h) + do_ / 8, rows * 8);
                copy8(reinterpret_cast<const uint4*>(kp_l) + so_ / 8, reinterpret_cast<uint4*>(kp_l) + do_ / 8, rows * 8);
            }
            if (nodes_h) {     // site-major planes [C][S][128 bf16]: one 256-byte row per (site, slot)
                uint4* nh = reinterpret_cast<uint4*>(nodes_h) + (size_t)b * C * pool.S * 16;
                uint4* nl = reinterpret_cast<uint4*>(nodes_l) + (size_t)b * C * pool.S * 16;
                uint4 vh[8], vl[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int k = tid + u * NTHREADS;
                    if (k < rows * 16) { const size_t os = (((size_t)row0 + (k >> 4)) * pool.S + src) * 16 + (k & 15); vh[u] = nh[os]; vl[u] = nl[os]; }
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int k = tid + u * NTHREADS;
                    if (k < rows * 16) { const size_t od = (((size_t)row0 + (k >> 4)) * pool.S + dst) * 16 + (k & 15); nh[od] = vh[u]; nl[od] = vl[u]; }
                }
            }
            if (tid == 0) kapw[((size_t)b * pool.S + dst) * pool.nCT + ct] = kapw[((size_t)b * pool.S + src) * pool.nCT + ct];
        }
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            int c = row0 + ty * 8 + i;
            if (c < C) st4(xo + (size_t)c * D + tx * 4, ld4(xs + (ty * 8 + i) * LDA + tx * 4));
        }
    }
}

// ------------------------------------------------------------------ small index / select kernels
__global__ void k_fill_pairs_full(int32_t* __restrict__ pair_i, int32_t* __restrict__ pair_j, int stride, int n, int B) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    int P = n * (n - 1) / 2;
    if (p >= P) return;
    int i, j;
    pair_from_index(p, n, i, j);
    for (int b = blockIdx.y; b < B; b += gridDim.y) { pair_i[(size_t)b * stride + p] = i; pair_j[(size_t)b * stride + p] = j; }
}

__global__ void k_fill_slots(int32_t* __restrict__ slot_of, int stride, int n, int32_t* __restrict__ free_slot) {
    int b = blockIdx.x;
    for (int r = threadIdx.x; r < n; r += blockDim.x) slot_of[(size_t)b * stride + r] = r;
    if (free_slot && threadIdx.x == 0) free_slot[b] = n;
}

// pairs (a, r) for r = 0..n-1 of the current node list, a = prev_ij[b][0]; the self pair is flagged -1  (model.py:186-197)
__global__ void k_fill_pairs_incr(int32_t* __restrict__ pair_i, int32_t* __restrict__ pair_j, int stride, int n,
                                  const int32_t* __restrict__ prev_ij, int ij_stride) {
    int b = blockIdx.x;
    int a = prev_ij[(size_t)b * ij_stride];
    for (int r = threadIdx.x; r < n; r += blockDim.x) {
        int lo = min(a, r), hi = max(a, r);
        pair_i[(size_t)b * stride + r] = (r == a) ? -1 : lo;
        pair_j[(size_t)b * stride + r] = (r == a) ? -1 : hi;
    }
}

// logits of the n-node list from [logits_prev | new_scores]  (utils.py:213-251 in closed form)
__device__ __forceinline__ float cached_logit(int p, int n, int a, int bb, const float* __restrict__ prev, const float* __restrict__ nw) {
    int ii, jj;
    pair_from_index(p, n, ii, jj);
    if (ii == a) return nw[jj];
    if (jj == a) return nw[ii];
    return prev[pair_index(ii + (ii >= bb ? 1 : 0), jj + (jj >= bb ? 1 : 0), n + 1)];
}

__global__ void k_assemble_logits(const float* __restrict__ logits_prev, int prev_stride, const float* __restrict__ new_scores,
                                  int new_stride, const int32_t* __restrict__ prev_ij, int ij_stride, int n, float* __restrict__ out,
                                  int out_stride) {
    int b = blockIdx.y;
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n * (n - 1) / 2) return;
    int a = prev_ij[(size_t)b * ij_stride], bb = prev_ij[(size_t)b * ij_stride + 1];
    out[(size_t)b * out_stride + p] = cached_logit(p, n, a, bb, logits_prev + (size_t)b * prev_stride, new_scores + (size_t)b * new_stride);
}

// One CTA per tree: assemble this step's logits, select (argmax / Gumbel-max, lowest index wins ties),
// record the merge, the selected log-probability, the next slot table and the next step's pair list.
__global__ void __launch_bounds__(NTHREADS) k_select(int t, int n, int R, const float* __restrict__ logits_prev, const float* __restrict__ new_scores,
                                                     int new_stride, float* __restrict__ logits_cur, int logit_stride,
                                                     const float* __restrict__ gumbel, int32_t* __restrict__ merges,
                                                     float* __restrict__ selected_logp, float* __restrict__ logits_trace,
                                                     size_t trace_stride, size_t trace_off, const int32_t* __restrict__ slot_cur,
                                                     int32_t* __restrict__ slot_next, int slot_stride, int32_t* __restrict__ free_slot,
                                                     int32_t* __restrict__ new_slot, int32_t* __restrict__ pair_i,
                                                     int32_t* __restrict__ pair_j, int pair_stride, int forced) {
    __shared__ float s_val[NTHREADS];
    __shared__ int s_idx[NTHREADS];
    __shared__ float s_red[NTHREADS];
    const int b = blockIdx.x, tid = threadIdx.x;
    const int P = n * (n - 1) / 2, P0 = R * (R - 1) / 2;
    float* cur = logits_cur + (size_t)b * logit_stride;
    if (t > 0) {
        const int32_t* pm = merges + ((size_t)b * (R - 1) + (t - 1)) * 2;
        const int a = pm[0], bb = pm[1];
        const float* prev = logits_prev + (size_t)b * logit_stride;
        const float* nw = new_scores + (size_t)b * new_stride;
        for (int p = tid; p < P; p += NTHREADS) cur[p] = cached_logit(p, n, a, bb, prev, nw);
        __syncthreads();
    }
    const float* gb = gumbel ? gumbel + ((size_t)b * (R - 1) + t) * P0 : nullptr;
    float best = -INFINITY, mx = -INFINITY;
    int bi = 0x7fffffff;
    for (int p = tid; p < P; p += NTHREADS) {
        float v = cur[p];
        if (logits_trace) logits_trace[(size_t)b * trace_stride + trace_off + p] = v;
        mx = fmaxf(mx, v);
        float s = gb ? v + gb[p] : v;
        if (s > best || (s == best && p < bi) || bi == 0x7fffffff) { best = s; bi = p; }
    }
    s_val[tid] = best; s_idx[tid] = bi; s_red[tid] = mx;
    __syncthreads();
    for (int o = NTHREADS / 2; o > 0; o >>= 1) {
        if (tid < o) {
            float v2 = s_val[tid + o]; int i2 = s_idx[tid + o];
            if (i2 != 0x7fffffff && (s_idx[tid] == 0x7fffffff || v2 > s_val[tid] || (v2 == s_val[tid] && i2 < s_idx[tid]))) { s_val[tid] = v2; s_idx[tid] = i2; }
            s_red[tid] = fmaxf(s_red[tid], s_red[tid + o]);
        }
        __syncthreads();
    }
    int act = s_idx[0];
    if (forced) {     // teacher forcing (train.py:116-119): merges[b][t] holds the action on entry; anything that is not a pair i < j < n falls back to the argmax
        const int fi = merges[((size_t)b * (R - 1) + t) * 2], fj = merges[((size_t)b * (R - 1) + t) * 2 + 1];
        if (fi >= 0 && fi < fj && fj < n) act = pair_index(fi, fj, n);
    }
    const float gmax = s_red[0];
    __syncthreads();
    float se = 0.f;
    for (int p = tid; p < P; p += NTHREADS) se += expf(cur[p] - gmax);
    s_red[tid] = se;
    __syncthreads();
    for (int o = NTHREADS / 2; o > 0; o >>= 1) {
        if (tid < o) s_red[tid] += s_red[tid + o];
        __syncthreads();
    }
    int i, j;
    pair_from_index(act, n, i, j);
    if (tid == 0) {
        merges[((size_t)b * (R - 1) + t) * 2] = i;
        merges[((size_t)b * (R - 1) + t) * 2 + 1] = j;
        if (selected_logp) selected_logp[(size_t)b * (R - 1) + t] = (cur[act] - gmax) - logf(s_red[0]);
    }
    if (n > 2) {
        // Physical slots stay COMPACT: the n live nodes occupy slots [0, n).  The merged node is written in place into the lower of
        // the pair's two slots, and the node in the last live slot (n-1) moves into the higher one (k_merge does both), so every
        // kernel that streams "all nodes of a site" reads n slots, not the R+1 the pool was allocated with.
        const int32_t* sc = slot_cur + (size_t)b * slot_stride;
        int32_t* sn = slot_next + (size_t)b * slot_stride;
        const int pi_phys = sc[i], pj_phys = sc[j];
        const int lo = min(pi_phys, pj_phys), hi = max(pi_phys, pj_phys), last = n - 1;
        __syncthreads();
        for (int r = tid; r < n - 1; r += NTHREADS) {
            int src = r + (r >= j ? 1 : 0);
            int p = (r == i) ? lo : sc[src];
            if (r != i && p == last) p = hi;           // the moved node (never i or j: then hi == last and nothing moves)
            sn[r] = p;
            pair_i[(size_t)b * pair_stride + r] = (r == i) ? -1 : min(i, r);
            pair_j[(size_t)b * pair_stride + r] = (r == i) ? -1 : max(i, r);
        }
        if (tid == 0) { new_slot[b] = lo; free_slot[b] = (hi != last) ? hi : -1; }   // free_slot: destination of the moved node, -1: none
    }
}

// state_out[b][r] = r == i ? new : state_in[b][r + (r >= j)]      (environment.py:764-768, 833-835)
__global__ void k_reindex_copy(const float* __restrict__ in, const float* __restrict__ newx, float* __restrict__ out, int Rp, size_t CD,
                               const int32_t* __restrict__ ij) {
    const int b = blockIdx.z, r = blockIdx.y;
    const int i = ij[b * 2], j = ij[b * 2 + 1];
    const float* src = (r == i) ? newx + (size_t)b * CD : in + ((size_t)b * Rp + r + (r >= j ? 1 : 0)) * CD;
    float* dst = out + ((size_t)b * (Rp - 1) + r) * CD;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < CD / 4; k += (size_t)gridDim.x * blockDim.x)
        st4(dst + k * 4, ld4(src + k * 4));
}

// ------------------------------------------------------------------ host side
struct NjBuffers {
    float *Y, *K, *kap, *alpha_part, *alpha, *score_part, *new_scores, *logits[2], *newx;
    int32_t *slot[2], *free_slot, *new_slot, *pair_i, *pair_j;
    float* X;         // pool X when owned by the workspace (rollout), else null
    float* xf;                // tensor-core path: x planes of the current pair chunk [B][pc][C][64] fp32
    void *xh, *xl;            // large-slot tensor-core path: the same rows as K-major bf16 hi / lo planes (A operand of the alpha-logit GEMM)
    void *nodes_h, *nodes_l;  // tensor-core path: site-major node planes [B][C][S][128] bf16 = [X | W_g X]
    void *kp_h, *kp_l;        // tensor-core path: K' planes [B][S][C][64] bf16 (B operand of the alpha GEMM)
    bool tc;                  // nj_use_tc: tensor-core NJ kernels, the merge / node-derive products on mma.sync
    bool big;                 // tc and 65 .. 256 slots: the large-slot pair-score path (nj_path)
    int pc;                   // pairs per launch on the tensor-core path (capacity of the x planes)
    int S, nCT, nSB, nAP, RP, pair_stride, P0;   // nSB: 32-site groups (fp32 kernels); nAP: alpha partials allocated per pair (stride)
    size_t total;
};

constexpr int TC_PAIRS = 256;   // pairs per launch on the tensor-core pair-score path

// The tensor-core NJ kernels take at most 256 physical slots (the fused kernels up to 64, the large-slot path 65 .. 256; nj_path) and -
// like the tensor-core encoder (use_tc in nnj_encoder.cu) - need C % 8 == 0: their TMA boxes and the two-sites-per-item ring assume
// 16-byte rows and an even site count.  Every other shape runs the fp32 CUDA-core kernels of this file, whatever the precision mode.
static bool nj_use_tc(const Model* m, int S, int C) { return m->cfg.precision != NNJ_PREC_FP32 && S <= 256 && (C % 8) == 0; }
constexpr int BIG_PAIRS = 512;  // pairs per launch of the large-slot path (4 pair tiles share one pass over the K' planes in the alpha GEMM)

// carve the NJ workspace; X_in_ws: the node pool X lives in the workspace too (rollout)
static NjBuffers nj_layout(char* base, int B, int S, int R, int C, bool X_in_ws, bool need_newx, bool tc) {
    NjBuffers nb{};
    nb.S = S; nb.nCT = (C + TILE_ROWS - 1) / TILE_ROWS; nb.nSB = (C + SB_SITES - 1) / SB_SITES;
    const bool big = tc && S > 64;
    const int tc_parts = tc ? (big ? 64 : 4 * ((C + 63) / 64)) : 0;          // tensor-core alpha: up to four partials per 64-site group; large-slot path: <= 64 K splits
    nb.nAP = nb.nSB > tc_parts ? nb.nSB : tc_parts;
    nb.RP = (S + 3) & ~3;     // >= S: tensor-core alpha partials are indexed by physical slot
    nb.P0 = R * (R - 1) / 2;
    nb.pair_stride = nb.P0 > R ? nb.P0 : R;
    WsCarver c(base);
    const size_t pool = (size_t)B * S * C * D;
    nb.X = X_in_ws ? c.take<float>(pool) : nullptr;
    nb.Y = c.take<float>(pool);
    nb.K = c.take<float>(pool);
    nb.kap = c.take<float>((size_t)B * S * nb.nCT);
    nb.alpha_part = c.take<float>((size_t)B * PAIR_CHUNK * nb.nAP * nb.RP);
    nb.alpha = c.take<float>((size_t)B * PAIR_CHUNK * nb.RP);
    nb.score_part = c.take<float>((size_t)B * PAIR_CHUNK * nb.nSB);
    nb.new_scores = c.take<float>((size_t)B * nb.pair_stride);
    nb.logits[0] = c.take<float>((size_t)B * nb.P0);
    nb.logits[1] = c.take<float>((size_t)B * nb.P0);
    nb.newx = need_newx ? c.take<float>((size_t)B * C * D) : nullptr;
    nb.slot[0] = c.take<int32_t>((size_t)B * S);
    nb.slot[1] = c.take<int32_t>((size_t)B * S);
    nb.free_slot = c.take<int32_t>(B);
    nb.new_slot = c.take<int32_t>(B);
    nb.pair_i = c.take<int32_t>((size_t)B * nb.pair_stride);
    nb.pair_j = c.take<int32_t>((size_t)B * nb.pair_stride);
    nb.tc = tc; nb.big = big; nb.pc = big ? BIG_PAIRS : TC_PAIRS;
    if (tc) {                 // bf16 planes as 16-bit words
        const size_t xp = (size_t)B * nb.pc * C * D, np = (size_t)B * C * S * D;
        nb.xf = c.take<float>(xp); nb.nodes_h = c.take<uint16_t>(2 * np); nb.nodes_l = c.take<uint16_t>(2 * np); nb.kp_h = c.take<uint16_t>(np);
        nb.kp_l = c.take<uint16_t>(np);
        if (big) { nb.xh = c.take<uint16_t>(xp); nb.xl = c.take<uint16_t>(xp); }
    }
    nb.total = c.off + 256;
    return nb;
}

static size_t smem_score(int Rp) { return (2 * 4096 + 2 * TILE_ROWS * LDA + 128 + 64 + ((Rp + 3) & ~3) + (size_t)Rp * 32) * sizeof(float); }
static size_t smem_merge(int Rp) { return (2 * TILE_ROWS * LDA + 4096 + 128 + 2 * ((Rp + 3) & ~3) + 8) * sizeof(float); }
static const size_t smem_derive = (2 * TILE_ROWS * LDA + 4096 + 128) * sizeof(float);

static int set_attrs() {
    static DevOnce once;      // per device, not per process
    if (!once.need()) return 0;
    const int big = 220 * 1024;
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(k_score<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    if ((e = cudaFuncSetAttribute(k_score<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    if ((e = cudaFuncSetAttribute(k_merge<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    if ((e = cudaFuncSetAttribute(k_merge<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    if ((e = cudaFuncSetAttribute(k_merge<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    if ((e = cudaFuncSetAttribute(k_merge<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    if ((e = cudaFuncSetAttribute(k_node_derive<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_derive)) != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    if ((e = cudaFuncSetAttribute(k_node_derive<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_derive)) != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    once.done();
    return 0;
}

static int check_dims(int Rp, int C) {
    if (Rp < 2) return set_error(NNJ_ERR_INVALID, "need at least 2 nodes");
    if (C < 1) return set_error(NNJ_ERR_INVALID, "need at least 1 site");
    if (smem_score(Rp) > 220 * 1024) return set_error(NNJ_ERR_INVALID, "too many nodes for the pair-score kernel (max ~1000)");
    return 0;
}

// Kernels of the pair-score step for a chunk of nc pairs over Rp live nodes.  The rules are checked in order; S is the physical slot
// count of the workspace (R + 1 in the rollout, Rp in the step-wise API), so a rollout keeps the path S gives it down to its last step.
//   rule                    alpha                                                         pair score
//   Rp <= 2                 (none: no global attention, model.py:111)                     k_score<false>
//   !nj_use_tc(m, S, C)     k_alpha + k_alpha_softmax                                     k_score<true>
//   S > 64 (nj_layout: big) k_blend_planes + split-K k_tc_gemm + k_alpha_softmax_wide     k_score_big
//   nc <= 16 and Rp <= 16   k_alpha_small + k_alpha_softmax                               k_score_small
//   nc <= 64                k_alpha_v3 (2- or 4-way site split) + k_alpha_softmax         k_score_inc
//   otherwise               k_alpha_v3 + k_alpha_softmax                                  k_score_tc
// The first three rules do not depend on nc, so they also fix the pairs per launch: PAIR_CHUNK on the fp32 kernels, nb.pc (BIG_PAIRS on
// the large-slot path, TC_PAIRS otherwise) on the tensor-core ones.
enum class NjPath { NoGlobal, Fp32, Big, Small, Inc, Tc };
static NjPath nj_path(const NjBuffers& nb, int Rp, int nc) {
    if (Rp <= 2) return NjPath::NoGlobal;
    if (!nb.tc) return NjPath::Fp32;
    if (nb.big) return NjPath::Big;
    if (nc <= 16 && Rp <= 16) return NjPath::Small;
    if (nc <= 64) return NjPath::Inc;
    return NjPath::Tc;
}

// scores of N listed pairs per tree against Rp nodes; pool tensors must be derived already.
static int score_pairs(const Model* m, const Pool& pool, const NjBuffers& nb, const int32_t* slot, int Rp, int C, int N,
                       const uint8_t* mask, int B, float* scores, int score_stride, cudaStream_t st) {
    const NjPath first = nj_path(nb, Rp, N);
    const int step = (first == NjPath::NoGlobal || first == NjPath::Fp32) ? PAIR_CHUNK : nb.pc;
    const float inv_scale = 1.0f / sqrtf((float)D * (float)C);   // model.py:118 (patch_num == C)
    PairChunk c;
    c.B = B; c.Rp = Rp; c.S = nb.S; c.C = C;
    c.slot_of = slot; c.slot_stride = nb.S;
    c.pair_i = nb.pair_i; c.pair_j = nb.pair_j; c.pair_stride = nb.pair_stride;
    c.mask = mask;
    c.X = pool.X; c.Y = pool.Y; c.tree_stride = pool.tree_stride;
    c.kp_h = nb.kp_h; c.kp_l = nb.kp_l; c.nodes_h = nb.nodes_h; c.nodes_l = nb.nodes_l;
    c.xf = nb.xf; c.pc = nb.pc; c.xh = nb.xh; c.xl = nb.xl;
    c.alpha_part = nb.alpha_part; c.nAP = nb.nAP;
    c.alpha = nb.alpha; c.RP = nb.RP; c.alpha_pairs = PAIR_CHUNK;
    c.score_part = nb.score_part; c.nSB = nb.nSB;
    for (int n0 = 0; n0 < N; n0 += step) {
        const int nc = (N - n0 < step) ? (N - n0) : step;
        c.n0 = n0; c.nc = nc;
        int n_part = nb.nSB;    // score partials per pair, summed by k_score_reduce
        const NjPath path = nj_path(nb, Rp, nc);
        switch (path) {
        case NjPath::NoGlobal:
            prof_begin(KC_SCORE, st);
            k_score<false><<<dim3(nb.nSB, (nc + 31) / 32, B), NTHREADS, smem_score(Rp), st>>>(pool, slot, nb.S, Rp, C, nb.pair_i, nb.pair_j,
                                                                                             nb.pair_stride, n0, nc, nb.alpha, nb.RP, m->nj, mask,
                                                                                             nb.score_part, nb.nSB);
            LAUNCH_CHECK();
            break;
        case NjPath::Fp32: {
            const int node_tiles = (Rp + 63) / 64, pair_tiles = (nc + 63) / 64;
            prof_begin(KC_ALPHA, st);
            k_alpha<<<dim3(nb.nSB, pair_tiles * node_tiles, B), NTHREADS, 0, st>>>(pool, slot, nb.S, Rp, C, nb.pair_i, nb.pair_j, nb.pair_stride,
                                                                                   n0, nc, node_tiles, m->nj.bh, nb.alpha_part, nb.nAP, nb.RP);
            LAUNCH_CHECK();
            prof_begin(KC_ALPHA_SOFTMAX, st);
            k_alpha_softmax<<<dim3((nc + 7) / 8, B), NTHREADS, 0, st>>>(nb.alpha_part, pool.kap, slot, nb.S, nb.S, nb.nCT, Rp, nb.pair_i,
                                                                        nb.pair_j, nb.pair_stride, n0, nc, nb.nAP, nb.RP, inv_scale, nb.alpha, 0, nb.nSB);
            LAUNCH_CHECK();
            prof_begin(KC_SCORE, st);
            k_score<true><<<dim3(nb.nSB, (nc + 31) / 32, B), NTHREADS, smem_score(Rp), st>>>(pool, slot, nb.S, Rp, C, nb.pair_i, nb.pair_j,
                                                                                            nb.pair_stride, n0, nc, nb.alpha, nb.RP, m->nj, mask,
                                                                                            nb.score_part, nb.nSB);
            LAUNCH_CHECK();
            break;
        }
        case NjPath::Big: {
            // pair blend -> x planes (fp32 + bf16 hi / lo), alpha logits as a split-K tcgen05 GEMM [pairs x C*64] . [slots x C*64]^T over the
            // K' planes (one 64-element K chunk = one site; partials per split, indexed by physical slot), softmax, then the K-blocked fused
            // score kernel
            if (int e = launch_blend_planes(m, c, st)) return e;
            const int bn = Rp <= 64 ? 64 : (Rp <= 128 ? 128 : 256);
            // K splits: a function of the site count only (NOT of the batch or the pair count), so that a tree's logits do not depend on
            // what else is in the batch: >= 32 sites per split, <= 64 partials per pair
            const int cps = (C + 63) / 64 > 32 ? (C + 63) / 64 : 32;
            const int nsplit = (C + cps - 1) / cps;
            if (nsplit > nb.nAP) return set_error(NNJ_ERR_INVALID, "large-slot alpha: partial buffer too small");
            const size_t K = (size_t)C * D;
            if (int e = launch_tc_gemm_ex(KC_ALPHA, nb.xh, nb.xl, nb.kp_h, nb.kp_l, nb.alpha_part, B, nc, Rp, (int)K, K, (size_t)nb.pc * K, K, (size_t)nb.S * K,
                                          nb.nAP * nb.RP, (size_t)PAIR_CHUNK * nb.nAP * nb.RP, bn, nsplit, cps, (size_t)nb.RP, st)) return e;
            prof_begin(KC_ALPHA_SOFTMAX, st);
            k_alpha_softmax_wide<<<dim3(nc, B), NTHREADS, 0, st>>>(nb.alpha_part, pool.kap, slot, nb.S, nb.S, nb.nCT, Rp, nb.pair_i,
                                                                   nb.pair_j, nb.pair_stride, n0, nc, nb.nAP, nb.RP, inv_scale, nb.alpha, nsplit);
            LAUNCH_CHECK();
            if (int e = launch_score_big(m, c, &n_part, st)) return e;
            break;
        }
        case NjPath::Small: case NjPath::Inc: case NjPath::Tc: {
            // blend + alpha partials in one kernel (fp32 x planes written on the way, partials per site group, indexed by physical slot)
            // -> softmax -> fused score kernel
            int a_part = 0;
            if (int e = (path == NjPath::Small ? launch_alpha_small : launch_alpha_v3)(m, c, &a_part, st)) return e;
            prof_begin(KC_ALPHA_SOFTMAX, st);
            k_alpha_softmax<<<dim3((nc + 7) / 8, B), NTHREADS, 0, st>>>(nb.alpha_part, pool.kap, slot, nb.S, nb.S, nb.nCT, Rp, nb.pair_i,
                                                                        nb.pair_j, nb.pair_stride, n0, nc, nb.nAP, nb.RP, inv_scale, nb.alpha, 1, a_part);
            LAUNCH_CHECK();
            if (int e = (path == NjPath::Small ? launch_score_small : path == NjPath::Inc ? launch_score_inc : launch_score_tc)(m, c, &n_part, st))
                return e;
            break;
        }
        }
        prof_begin(KC_MISC, st);
        k_score_reduce<<<dim3((nc + 127) / 128, B), 128, 0, st>>>(nb.score_part, nb.nSB, n_part, nc, scores, score_stride, n0);
        LAUNCH_CHECK();
    }
    return 0;
}

// merged-node embedding for pair ij[b] against Rp nodes
static int merge_pair(const Model* m, const Pool& pool, const NjBuffers& nb, float* Xw, const int32_t* slot, int Rp, int C,
                      const int32_t* ij, int ij_stride, int B, float* out_x, size_t out_stride, bool derive, cudaStream_t st) {
    const float inv_scale = 1.0f / sqrtf((float)D * (float)C);
    auto launch_merge = [&](bool glob) {
        uint2* nh = (derive && nb.tc) ? (uint2*)nb.nodes_h : nullptr; uint2* nl = (derive && nb.tc) ? (uint2*)nb.nodes_l : nullptr;
        uint2* kh = (derive && nb.tc) ? (uint2*)nb.kp_h : nullptr;    uint2* kl = (derive && nb.tc) ? (uint2*)nb.kp_l : nullptr;
        const int32_t* mv = derive ? nb.free_slot : nullptr;
        const dim3 grid(nb.nCT, B);
        const size_t sm = smem_merge(Rp);
#define NNJ_MERGE_ARGS pool, Xw, nb.Y, nb.K, nb.kap, slot, nb.S, Rp, C, ij, ij_stride, nb.alpha, nb.RP, m->nj, m->nj_frag, out_x, out_stride, nb.new_slot, derive ? 1 : 0, nh, nl, kh, kl, mv
        // second template argument: the 64 x 64 products on mma.sync (tensor-core precision modes)
        if (glob) { if (nb.tc) k_merge<true, true><<<grid, NTHREADS, sm, st>>>(NNJ_MERGE_ARGS); else k_merge<true, false><<<grid, NTHREADS, sm, st>>>(NNJ_MERGE_ARGS); }
        else      { if (nb.tc) k_merge<false, true><<<grid, NTHREADS, sm, st>>>(NNJ_MERGE_ARGS); else k_merge<false, false><<<grid, NTHREADS, sm, st>>>(NNJ_MERGE_ARGS); }
#undef NNJ_MERGE_ARGS
    };
    if (Rp > 2) {
        prof_begin(KC_MERGE, st);     // the merge pair's own attention logits: counted with the merge
        k_alpha1<<<dim3(nb.nSB, B), NTHREADS, 0, st>>>(pool, slot, nb.S, Rp, C, ij, ij_stride, m->nj.bh, nb.alpha_part, nb.nAP, nb.RP);
        LAUNCH_CHECK();
        // pair list for the softmax kernel: reuse it with one pair per tree = ij itself
        prof_begin(KC_ALPHA_SOFTMAX, st);
        k_alpha_softmax<<<dim3(1, B), NTHREADS, 0, st>>>(nb.alpha_part, pool.kap, slot, nb.S, nb.S, nb.nCT, Rp, ij, ij + 1, ij_stride, 0, 1,
                                                         nb.nAP, nb.RP, inv_scale, nb.alpha, 0, nb.nSB);
        LAUNCH_CHECK();
        prof_begin(KC_MERGE, st);
        launch_merge(true);
        LAUNCH_CHECK();
    } else {
        prof_begin(KC_MERGE, st);
        launch_merge(false);
        LAUNCH_CHECK();
    }
    return 0;
}

// Y, K, kappa (and on the tensor-core path the K' and node planes) of `nodes` nodes in slots [0, nodes) of S
static int derive_all(const Model* m, const float* X, const NjBuffers& nb, int B, int S, int nodes, int C, cudaStream_t st) {
    prof_begin(KC_DERIVE, st);
    if (nb.tc && nodes < S) {   // the spare slots' rows are read (with weight 0) by the pair-score UMMA: they must be finite
        const size_t npb = (size_t)B * C * S * 2 * D * 2;
        cudaError_t e1 = cudaMemsetAsync(nb.nodes_h, 0, npb, st), e2 = cudaMemsetAsync(nb.nodes_l, 0, npb, st);
        if (e1 != cudaSuccess || e2 != cudaSuccess) return set_cuda_error(e1 != cudaSuccess ? e1 : e2, __FILE__, __LINE__);
    }
    if (nb.tc)
        k_node_derive<true><<<dim3(nb.nCT, nodes, B), NTHREADS, smem_derive, st>>>(X, nb.Y, nb.K, nb.kap, (size_t)S * C * D, S, C, nb.nCT, nullptr, 0, m->nj, m->nj_frag,
                                                                                   (uint2*)nb.kp_h, (uint2*)nb.kp_l, (uint2*)nb.nodes_h, (uint2*)nb.nodes_l);
    else
        k_node_derive<false><<<dim3(nb.nCT, nodes, B), NTHREADS, smem_derive, st>>>(X, nb.Y, nb.K, nb.kap, (size_t)S * C * D, S, C, nb.nCT, nullptr, 0, m->nj, m->nj_frag,
                                                                                    nullptr, nullptr, nullptr, nullptr);
    LAUNCH_CHECK();
    return 0;
}

size_t nj_scores_ws_bytes(const Model* m, int B, int Rp, int C, int N) {
    (void)N;
    return nj_layout(nullptr, B, Rp, Rp, C, false, true, nj_use_tc(m, Rp, C)).total;
}

static Pool make_pool(const float* X, const NjBuffers& nb, int S, int C) {
    Pool p;
    p.X = X; p.Y = nb.Y; p.K = nb.K; p.kap = nb.kap;
    p.tree_stride = (size_t)S * C * D; p.S = S; p.nCT = nb.nCT;
    return p;
}

int run_pair_scores(Model* m, const float* state, const uint8_t* mask, int B, int Rp, int C, const int32_t* pi, const int32_t* pj, int N,
                    bool full, float* scores, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (int e = check_dims(Rp, C)) return e;
    if (int e = set_attrs()) return e;
    NjBuffers nb = nj_layout(ws_align(ws), B, Rp, Rp, C, false, true, nj_use_tc(m, Rp, C));
    if (ws_bytes < nb.total) return set_error(NNJ_ERR_WORKSPACE, "pair scores: workspace too small");
    if (full) N = Rp * (Rp - 1) / 2;
    if (N > nb.pair_stride) return set_error(NNJ_ERR_INVALID, "pair scores: more pairs than R(R-1)/2");
    prof_begin(KC_MISC, st);
    k_fill_slots<<<B, 128, 0, st>>>(nb.slot[0], nb.S, Rp, nullptr);
    LAUNCH_CHECK();
    if (full) {
        prof_begin(KC_MISC, st);
        k_fill_pairs_full<<<dim3((N + 127) / 128, B < 64 ? B : 64), 128, 0, st>>>(nb.pair_i, nb.pair_j, nb.pair_stride, Rp, B);
        LAUNCH_CHECK();
    } else {
        cudaError_t e1 = cudaMemcpy2DAsync(nb.pair_i, nb.pair_stride * sizeof(int32_t), pi, N * sizeof(int32_t), N * sizeof(int32_t), B, cudaMemcpyDeviceToDevice, st);
        cudaError_t e2 = cudaMemcpy2DAsync(nb.pair_j, nb.pair_stride * sizeof(int32_t), pj, N * sizeof(int32_t), N * sizeof(int32_t), B, cudaMemcpyDeviceToDevice, st);
        if (e1 != cudaSuccess || e2 != cudaSuccess) return set_cuda_error(e1 != cudaSuccess ? e1 : e2, __FILE__, __LINE__);
    }
    if (int e = derive_all(m, state, nb, B, Rp, Rp, C, st)) return e;
    Pool pool = make_pool(state, nb, Rp, C);
    return score_pairs(m, pool, nb, nb.slot[0], Rp, C, N, mask, B, scores, N, st);
}

int run_pair_scores_incr(Model* m, const float* state, const uint8_t* mask, int B, int Rp, int C, const int32_t* prev_ij,
                         const float* logits_prev, float* logits_out, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (int e = check_dims(Rp, C)) return e;
    if (int e = set_attrs()) return e;
    NjBuffers nb = nj_layout(ws_align(ws), B, Rp, Rp, C, false, true, nj_use_tc(m, Rp, C));
    if (ws_bytes < nb.total) return set_error(NNJ_ERR_WORKSPACE, "pair scores: workspace too small");
    prof_begin(KC_MISC, st);
    k_fill_slots<<<B, 128, 0, st>>>(nb.slot[0], nb.S, Rp, nullptr);
    LAUNCH_CHECK();
    prof_begin(KC_MISC, st);
    k_fill_pairs_incr<<<B, 128, 0, st>>>(nb.pair_i, nb.pair_j, nb.pair_stride, Rp, prev_ij, 2);
    LAUNCH_CHECK();
    if (int e = derive_all(m, state, nb, B, Rp, Rp, C, st)) return e;
    Pool pool = make_pool(state, nb, Rp, C);
    if (int e = score_pairs(m, pool, nb, nb.slot[0], Rp, C, Rp, mask, B, nb.new_scores, nb.pair_stride, st)) return e;
    const int P = Rp * (Rp - 1) / 2;
    prof_begin(KC_MISC, st);
    k_assemble_logits<<<dim3((P + 127) / 128, B), 128, 0, st>>>(logits_prev, (Rp + 1) * Rp / 2, nb.new_scores, nb.pair_stride, prev_ij, 2, Rp,
                                                                logits_out, P);
    LAUNCH_CHECK();
    return 0;
}

int run_aggregate(Model* m, const float* state, int B, int Rp, int C, const int32_t* ij, float* out, size_t out_tree_stride, void* ws,
                  size_t ws_bytes, cudaStream_t st) {
    if (int e = check_dims(Rp, C)) return e;
    if (int e = set_attrs()) return e;
    NjBuffers nb = nj_layout(ws_align(ws), B, Rp, Rp, C, false, true, nj_use_tc(m, Rp, C));
    if (ws_bytes < nb.total) return set_error(NNJ_ERR_WORKSPACE, "aggregate: workspace too small");
    prof_begin(KC_MISC, st);
    k_fill_slots<<<B, 128, 0, st>>>(nb.slot[0], nb.S, Rp, nullptr);
    LAUNCH_CHECK();
    if (int e = derive_all(m, state, nb, B, Rp, Rp, C, st)) return e;
    Pool pool = make_pool(state, nb, Rp, C);
    return merge_pair(m, pool, nb, nullptr, nb.slot[0], Rp, C, ij, 2, B, out, out_tree_stride, false, st);
}

int run_merge(Model* m, const float* state_in, int B, int Rp, int C, const int32_t* ij, float* state_out, void* ws, size_t ws_bytes,
              cudaStream_t st) {
    NjBuffers nb = nj_layout(ws_align(ws), B, Rp, Rp, C, false, true, nj_use_tc(m, Rp, C));
    if (int e = run_aggregate(m, state_in, B, Rp, C, ij, nb.newx, (size_t)C * D, ws, ws_bytes, st)) return e;
    prof_begin(KC_MISC, st);
    k_reindex_copy<<<dim3(8, Rp - 1, B), 256, 0, st>>>(state_in, nb.newx, state_out, Rp, (size_t)C * D, ij);
    LAUNCH_CHECK();
    return 0;
}

// ---- fused rollout
int nj_rollout_chunk(const Model* m, int B, int R, int C) {
    size_t per = nj_layout(nullptr, 1, R + 1, R, C, true, false, nj_use_tc(m, R + 1, C)).total + encoder_ws_bytes(m, 1, R, C);
    // defaults: 48 GB of the 180 GB HBM3e, at most 128 trees per chunk; NNJ_WS_GB / NNJ_CHUNK_MAX override them (tuning runs)
    static int ws_gb = 0, ch_max = 0;
    if (!ws_gb) { const char* e = getenv("NNJ_WS_GB"); ws_gb = e && atoi(e) > 0 ? atoi(e) : 48; }
    if (!ch_max) { const char* e = getenv("NNJ_CHUNK_MAX"); ch_max = e && atoi(e) > 0 ? atoi(e) : 128; }
    size_t budget = (size_t)ws_gb << 30;
    int ch = (int)(budget / per);
    if (ch < 1) ch = 1;
    if (ch > ch_max) ch = ch_max;
    if (ch > B) ch = B;
    const int n = (B + ch - 1) / ch;      // equal-sized chunks: no small tail launch
    return (B + n - 1) / n;
}

size_t nj_rollout_ws_bytes(const Model* m, int B, int R, int C) {
    int ch = nj_rollout_chunk(m, B, R, C);
    return nj_layout(nullptr, ch, R + 1, R, C, true, false, nj_use_tc(m, R + 1, C)).total + encoder_ws_bytes(m, ch, R, C) + 512;
}

int run_rollout(Model* m, const int8_t* data, const float* state0, const uint8_t* mask, int B, int R, int L, int select_mode,
                const float* gumbel, int32_t* merges, float* logits_trace, float* selected_logp, void* ws, size_t ws_bytes,
                cudaStream_t st) {
    const int C = L;
    if (R < 2) return set_error(NNJ_ERR_INVALID, "rollout: need at least 2 taxa");
    if (int e = check_dims(R, C)) return e;
    if (int e = set_attrs()) return e;
    if (select_mode == NNJ_SELECT_GUMBEL && !gumbel) return set_error(NNJ_ERR_INVALID, "rollout: gumbel noise required for NNJ_SELECT_GUMBEL");
    if (select_mode != NNJ_SELECT_GUMBEL) gumbel = nullptr;
    if (select_mode < NNJ_SELECT_ARGMAX || select_mode > NNJ_SELECT_FORCED) return set_error(NNJ_ERR_INVALID, "rollout: unknown select mode");
    if (ws_bytes < nj_rollout_ws_bytes(m, B, R, C)) return set_error(NNJ_ERR_WORKSPACE, "rollout: workspace too small");
    const int chunk = nj_rollout_chunk(m, B, R, C);
    const int S = R + 1;
    char* base = ws_align(ws);
    NjBuffers nb = nj_layout(base, chunk, S, R, C, true, false, nj_use_tc(m, S, C));
    void* enc_ws = base + nb.total;
    const size_t enc_bytes = encoder_ws_bytes(m, chunk, R, C);
    const size_t tree_stride = (size_t)S * C * D;
    const int P0 = nb.P0;
    size_t trace_stride = 0;
    for (int n = R; n >= 2; --n) trace_stride += (size_t)n * (n - 1) / 2;
    for (int b0 = 0; b0 < B; b0 += chunk) {
        const int nbt = (B - b0 < chunk) ? (B - b0) : chunk;
        const uint8_t* mk = mask ? mask + (size_t)b0 * C : nullptr;
        if (state0) {
            cudaError_t e = cudaMemcpy2DAsync(nb.X, tree_stride * sizeof(float), state0 + (size_t)b0 * R * C * D, (size_t)R * C * D * sizeof(float),
                                              (size_t)R * C * D * sizeof(float), nbt, cudaMemcpyDeviceToDevice, st);
            if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
        } else {
            if (int e = run_encoder(m, data + (size_t)b0 * R * L * 4, mk, nbt, R, L, nb.X, tree_stride, enc_ws, enc_bytes, st)) return e;
        }
        prof_begin(KC_MISC, st);
        k_fill_slots<<<nbt, 128, 0, st>>>(nb.slot[0], S, R, nb.free_slot);
        LAUNCH_CHECK();
        prof_begin(KC_MISC, st);
        k_fill_pairs_full<<<dim3((P0 + 127) / 128, nbt < 64 ? nbt : 64), 128, 0, st>>>(nb.pair_i, nb.pair_j, nb.pair_stride, R, nbt);
        LAUNCH_CHECK();
        if (int e = derive_all(m, nb.X, nb, nbt, S, R, C, st)) return e;
        Pool pool = make_pool(nb.X, nb, S, C);
        int32_t* mg = merges + (size_t)b0 * (R - 1) * 2;
        float* slp = selected_logp ? selected_logp + (size_t)b0 * (R - 1) : nullptr;
        float* ltr = logits_trace ? logits_trace + (size_t)b0 * trace_stride : nullptr;
        const float* gmb = gumbel ? gumbel + (size_t)b0 * (R - 1) * P0 : nullptr;
        size_t trace_off = 0;
        int cur = 0;
        for (int t = 0; t < R - 1; ++t) {
            const int n = R - t;
            const int32_t* slot = nb.slot[t & 1];
            if (t == 0) {
                if (int e = score_pairs(m, pool, nb, slot, n, C, P0, mk, nbt, nb.logits[0], P0, st)) return e;
            } else {
                // The last step has a single candidate pair: its score cannot change the merge, and log_softmax of one logit is 0.  It is
                // evaluated only when the caller records the logits (one fp32 launch, 1.4 ms per 128 trees); otherwise the score buffer is
                // set to a defined 0 so that logits_cur never holds a stale value.
                if (n == 2 && !ltr) {
                    cudaError_t e0 = cudaMemsetAsync(nb.new_scores, 0, (size_t)nbt * nb.pair_stride * sizeof(float), st);
                    if (e0 != cudaSuccess) return set_cuda_error(e0, __FILE__, __LINE__);
                } else if (int e = score_pairs(m, pool, nb, slot, n, C, n, mk, nbt, nb.new_scores, nb.pair_stride, st)) return e;
                cur ^= 1;
            }
            prof_begin(KC_SELECT, st);
            k_select<<<nbt, NTHREADS, 0, st>>>(t, n, R, nb.logits[cur ^ 1], nb.new_scores, nb.pair_stride, nb.logits[cur], P0, gmb, mg, slp, ltr,
                                               trace_stride, trace_off, slot, nb.slot[(t + 1) & 1], S, nb.free_slot, nb.new_slot, nb.pair_i,
                                               nb.pair_j, nb.pair_stride, select_mode == NNJ_SELECT_FORCED);
            LAUNCH_CHECK();
            trace_off += (size_t)n * (n - 1) / 2;
            if (n == 2) break;
            if (int e = merge_pair(m, pool, nb, nb.X, slot, n, C, mg + (size_t)t * 2, (R - 1) * 2, nbt, nullptr, 0, true, st)) return e;
        }
    }
    return 0;
}

}  // namespace nnj
