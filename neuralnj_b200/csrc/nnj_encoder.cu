// nnj_encoder.cu — MSA axial encoder (fp32 CUDA-core path).
//
// Restates PhyloATTN.encode_zxr (model.py:67-88): embed -> L x [row attention, column
// attention, feed-forward], each in a pre-LN residual block (msa_modules.py:62-125).
// Activations stay [B,R,C,64] fp32 (tree stride configurable so the NJ node pool can be
// written in place).  Kernels:
//   k_embed          model.py:39-43,77      16-entry LUT of Linear(4->64)+GELU+Linear(64->64)
//   k_ln_qkv         LN + q/k/v projections (axial_attention.py:75-82, 211-214)
//   k_gemm           tied row-attention logits / PV as batched GEMMs (axial_attention.py:97,114)
//   k_softmax_rows   softmax over key columns with the -10000 pad fill (:99-103,135)
//   k_col_attn       per-site attention over taxa (:216-234)
//   k_out_proj       out_proj + residual add (:116,236; msa_modules.py:120)
//   k_ffn            LN + fc1 + GELU + fc2 + residual (msa_modules.py:144-151)
#include <cuda_bf16.h>

#include "nnj_internal.h"
#include "nnj_tc.cuh"

namespace nnj {

// ------------------------------------------------------------------ token addressing
// NATURAL order: t = r*C + c.   CMAJOR order: t = c*R + r (rows of one site are adjacent,
// which makes the head-major q/k/v/ctx layout [B,H,C,R,8] contiguous per head).
template <bool CMAJOR>
__device__ __forceinline__ void tok_rc(int t, int R, int C, int& r, int& c) {
    if (CMAJOR) { c = t / R; r = t - c * R; } else { r = t / C; c = t - r * C; }
}

// element offset of the 16-byte column chunk c4 of token (taxon r, site c) in the residual stream: node-major [R][C][64], or (xsm)
// the site-major tile-planar stream of the tensor-core encoder (xs_off in nnj_internal.h)
__device__ __forceinline__ size_t x_off(int r, int c, int R, int C, int xsm, int c4) {
    return xsm ? xs_off((size_t)c * R + r, c4) : ((size_t)r * C + c) * D + c4 * 4;
}

template <bool CMAJOR>
__device__ __forceinline__ void load_x_tile(float* __restrict__ xs, const float* __restrict__ xb, int tile, int R, int C, int xsm = 0) {
    const int T = R * C;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        int idx = it * NTHREADS + threadIdx.x;
        int row = xsm ? (idx & 127) : (idx >> 4), c4 = xsm ? (idx >> 7) : (idx & 15);   // lanes follow the contiguous direction of the stream
        int t = tile * TILE_ROWS + row;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (t < T) {
            int r, c;
            tok_rc<CMAJOR>(t, R, C, r, c);
            v = ld4(xb + x_off(r, c, R, C, xsm, c4));
        }
        st4(xs + row * LDA + c4 * 4, v);
    }
}

// ------------------------------------------------------------------ embed
__global__ void __launch_bounds__(NTHREADS) k_embed(const int8_t* __restrict__ data, float* __restrict__ x, size_t x_tree_stride,
                                                    int R, int L, EmbedW w, int xsm) {
    __shared__ float hbuf[16][64];
    __shared__ float lut[16][64];
    const int tid = threadIdx.x;
    for (int idx = tid; idx < 1024; idx += NTHREADS) {
        int p = idx >> 6, o = idx & 63;
        float s = 0.f;
#pragma unroll
        for (int e = 0; e < 4; ++e) s = fmaf((p >> e) & 1 ? 1.0f : 0.0f, __ldg(w.w1 + o * 4 + e), s);
        hbuf[p][o] = gelu_erf(s + __ldg(w.b1 + o));
    }
    __syncthreads();
    for (int idx = tid; idx < 1024; idx += NTHREADS) {
        int p = idx >> 6, o = idx & 63;
        float s = 0.f;
        for (int k = 0; k < 64; ++k) s = fmaf(hbuf[p][k], __ldg(w.w2t + k * 64 + o), s);
        lut[p][o] = s + __ldg(w.b2 + o);
    }
    __syncthreads();
    const int b = blockIdx.y;
    const int T = R * L;
    const int8_t* db = data + (size_t)b * T * 4;
    float* xb = x + (size_t)b * x_tree_stride;
    const int t0 = blockIdx.x * 1024;
    for (int it = 0; it < 64; ++it) {
        int idx = it * NTHREADS + tid;
        int t = t0 + (idx >> 4), c4 = idx & 15;
        int r, c;
        if (xsm) {      // tile-planar site-major stream: lanes follow its tokens (site * R + taxon), one column chunk per pass
            t = t0 + (idx & 1023); c4 = idx >> 10;
            if (t >= T) continue;
            c = t / R; r = t - c * R;
        } else {
            if (t >= T) break;
            r = t / L; c = t - r * L;
        }
        char4 v = *reinterpret_cast<const char4*>(db + ((size_t)r * L + c) * 4);
        float4 o;
        if (((v.x | v.y | v.z | v.w) & ~1) == 0) {
            int p = v.x | (v.y << 1) | (v.z << 2) | (v.w << 3);
            o = ld4(&lut[p][c4 * 4]);
        } else {  // non one-hot input: evaluate the two Linear layers directly
            float in[4] = {(float)v.x, (float)v.y, (float)v.z, (float)v.w};
            float acc[4] = {__ldg(w.b2 + c4 * 4), __ldg(w.b2 + c4 * 4 + 1), __ldg(w.b2 + c4 * 4 + 2), __ldg(w.b2 + c4 * 4 + 3)};
            for (int k = 0; k < 64; ++k) {
                float s = 0.f;
                for (int e = 0; e < 4; ++e) s = fmaf(in[e], __ldg(w.w1 + k * 4 + e), s);
                float hk = gelu_erf(s + __ldg(w.b1 + k));
                for (int j = 0; j < 4; ++j) acc[j] = fmaf(hk, __ldg(w.w2t + k * 64 + c4 * 4 + j), acc[j]);
            }
            o = make_float4(acc[0], acc[1], acc[2], acc[3]);
        }
        st4(xb + x_off(r, c, R, L, xsm, c4), o);
    }
}

// ------------------------------------------------------------------ LN + QKV
// ROW=true : CMAJOR tiles, outputs head-major [B,H,C,R,8]; q scaled by dh^-0.5/sqrt(R) and zeroed at padded sites.
// ROW=false: NATURAL tiles, outputs [B,R,C,64]; q scaled by dh^-0.5.
template <bool ROW>
__global__ void __launch_bounds__(NTHREADS) k_ln_qkv(const float* __restrict__ x, size_t x_tree_stride, int R, int C,
                                                     AttnW w, float q_scale, const uint8_t* __restrict__ mask,
                                                     float* __restrict__ q, float* __restrict__ k, float* __restrict__ v, int xsm) {
    extern __shared__ __align__(16) float smem[];
    float* xs = smem;
    float* Ws = smem + TILE_ROWS * LDA;
    const int b = blockIdx.y, tile = blockIdx.x;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int T = R * C;
    load_x_tile<ROW>(xs, x + (size_t)b * x_tree_stride, tile, R, C, xsm);
    __syncthreads();
    tile_layernorm(xs, w.ln_g, w.ln_b);
    __syncthreads();
    const float* wt[3] = {w.qt, w.kt, w.vt};
    const float* bs[3] = {w.qb, w.kb, w.vb};
    float* outp[3] = {q, k, v};
#pragma unroll
    for (int p = 0; p < 3; ++p) {
        load_w64(Ws, wt[p]);
        __syncthreads();
        float acc[8][4];
        acc_set_bias(acc, bs[p], tx);
        tile_mma64(acc, xs, Ws, ty, tx);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            int t = tile * TILE_ROWS + ty * 8 + i;
            if (t < T) {
                int r, c;
                tok_rc<ROW>(t, R, C, r, c);
                float4 o = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
                if (p == 0) {
                    float s = q_scale;
                    if (ROW && mask && mask[(size_t)b * C + c]) s = 0.f;   // axial_attention.py:82
                    o.x *= s; o.y *= s; o.z *= s; o.w *= s;
                }
                size_t off;
                if (ROW) off = ((((size_t)b * H + (tx >> 1)) * C + c) * R + r) * DH + (tx & 1) * 4;
                else off = (((size_t)b * R + r) * C + c) * D + tx * 4;
                st4(outp[p] + off, o);
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------ out_proj + residual
template <bool ROW>
__global__ void __launch_bounds__(NTHREADS) k_out_proj(float* __restrict__ x, size_t x_tree_stride, int R, int C,
                                                       const float* __restrict__ ctx, const float* __restrict__ wt,
                                                       const float* __restrict__ bias, int xsm) {
    extern __shared__ __align__(16) float smem[];
    float* as = smem;
    float* Ws = smem + TILE_ROWS * LDA;
    const int b = blockIdx.y, tile = blockIdx.x;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int T = R * C;
    load_w64(Ws, wt);
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        int idx = it * NTHREADS + threadIdx.x;
        int row = idx >> 4, c4 = idx & 15;
        int t = tile * TILE_ROWS + row;
        float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
        if (t < T) {
            int r, c;
            tok_rc<ROW>(t, R, C, r, c);
            size_t off;
            if (ROW) off = ((((size_t)b * H + (c4 >> 1)) * C + c) * R + r) * DH + (c4 & 1) * 4;
            else off = (((size_t)b * R + r) * C + c) * D + c4 * 4;
            val = ld4(ctx + off);
        }
        st4(as + row * LDA + c4 * 4, val);
    }
    __syncthreads();
    float acc[8][4];
    acc_set_bias(acc, bias, tx);
    tile_mma64(acc, as, Ws, ty, tx);
    float* xb = x + (size_t)b * x_tree_stride;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        int t = tile * TILE_ROWS + ty * 8 + i;
        if (t < T) {
            int r, c;
            tok_rc<ROW>(t, R, C, r, c);
            float* p = xb + x_off(r, c, R, C, xsm, tx);
            float4 o = ld4(p);
            o.x += acc[i][0]; o.y += acc[i][1]; o.z += acc[i][2]; o.w += acc[i][3];
            st4(p, o);
        }
    }
}

// ------------------------------------------------------------------ feed-forward
__global__ void __launch_bounds__(NTHREADS) k_ffn(float* __restrict__ x, size_t x_tree_stride, int R, int C, FfnW w, int xsm) {
    extern __shared__ __align__(16) float smem[];
    float* xs = smem;
    float* hs = xs + TILE_ROWS * LDA;
    float* W1 = hs + TILE_ROWS * LDA;
    float* W2 = W1 + 4096;
    const int b = blockIdx.y, tile = blockIdx.x;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int T = R * C;
    float* xb = x + (size_t)b * x_tree_stride;
    if (xsm) load_x_tile<true>(xs, xb, tile, R, C, 1);   // per-token work: any token order will do, take the stream's own
    else load_x_tile<false>(xs, xb, tile, R, C);
    __syncthreads();
    tile_layernorm(xs, w.ln_g, w.ln_b);
    float out[8][4];
    acc_set_bias(out, w.b2, tx);
    for (int ch = 0; ch < 4; ++ch) {
        __syncthreads();  // xs normalised (ch==0) / previous chunk done with hs, W1, W2
        load_w64(W1, w.w1t + ch * 4096);
        load_w64(W2, w.w2t + ch * 4096);
        __syncthreads();
        float acc[8][4];
        acc_set_bias(acc, w.b1 + ch * 64, tx);
        tile_mma64(acc, xs, W1, ty, tx);
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = gelu_erf(acc[i][j]);
        acc_store_smem(acc, hs, ty, tx);
        __syncthreads();
        tile_mma64(out, hs, W2, ty, tx);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        int t = tile * TILE_ROWS + ty * 8 + i;
        if (t < T) {
            float* p = xb + (xsm ? xs_off((size_t)t, tx) : (size_t)t * D + tx * 4);
            float4 o = ld4(p);
            o.x += out[i][0]; o.y += out[i][1]; o.z += out[i][2]; o.w += out[i][3];
            st4(p, o);
        }
    }
}

// ------------------------------------------------------------------ column attention
// One CTA per (site c, tree b); warp h = head h; lane i = query taxon (strided by 32).
__global__ void __launch_bounds__(NTHREADS) k_col_attn(const float* __restrict__ q, const float* __restrict__ k,
                                                       const float* __restrict__ v, float* __restrict__ ctx, int R, int C,
                                                       const uint8_t* __restrict__ mask) {
    extern __shared__ __align__(16) float smem[];
    float* ks = smem;
    float* vs = smem + (size_t)R * D;
    const int c = blockIdx.x, b = blockIdx.y;
    const size_t base = ((size_t)b * R * C + c) * D;
    const size_t rstride = (size_t)C * D;
    for (int idx = threadIdx.x; idx < R * 16; idx += NTHREADS) {
        int r = idx >> 4, c4 = idx & 15;
        st4(ks + r * D + c4 * 4, ld4(k + base + r * rstride + c4 * 4));
        st4(vs + r * D + c4 * 4, ld4(v + base + r * rstride + c4 * 4));
    }
    __syncthreads();
    const int h = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool padded = mask && mask[(size_t)b * C + c];
    for (int i = lane; i < R; i += 32) {
        float4 q0 = ld4(q + base + i * rstride + h * DH), q1 = ld4(q + base + i * rstride + h * DH + 4);
        float m = -INFINITY;
        for (int j = 0; j < R; ++j) {
            float4 k0 = ld4(ks + j * D + h * DH), k1 = ld4(ks + j * D + h * DH + 4);
            float s = q0.x * k0.x;
            s = fmaf(q0.y, k0.y, s); s = fmaf(q0.z, k0.z, s); s = fmaf(q0.w, k0.w, s);
            s = fmaf(q1.x, k1.x, s); s = fmaf(q1.y, k1.y, s); s = fmaf(q1.z, k1.z, s); s = fmaf(q1.w, k1.w, s);
            if (padded) s = -10000.0f;   // axial_attention.py:220-224
            m = fmaxf(m, s);
        }
        float l = 0.f, o[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int j = 0; j < R; ++j) {
            float4 k0 = ld4(ks + j * D + h * DH), k1 = ld4(ks + j * D + h * DH + 4);
            float s = q0.x * k0.x;
            s = fmaf(q0.y, k0.y, s); s = fmaf(q0.z, k0.z, s); s = fmaf(q0.w, k0.w, s);
            s = fmaf(q1.x, k1.x, s); s = fmaf(q1.y, k1.y, s); s = fmaf(q1.z, k1.z, s); s = fmaf(q1.w, k1.w, s);
            if (padded) s = -10000.0f;
            float p = expf(s - m);
            l += p;
            float4 v0 = ld4(vs + j * D + h * DH), v1 = ld4(vs + j * D + h * DH + 4);
            o[0] = fmaf(p, v0.x, o[0]); o[1] = fmaf(p, v0.y, o[1]); o[2] = fmaf(p, v0.z, o[2]); o[3] = fmaf(p, v0.w, o[3]);
            o[4] = fmaf(p, v1.x, o[4]); o[5] = fmaf(p, v1.y, o[5]); o[6] = fmaf(p, v1.z, o[6]); o[7] = fmaf(p, v1.w, o[7]);
        }
        float inv = 1.0f / l;
        float* op = ctx + base + i * rstride + h * DH;
        st4(op, make_float4(o[0] * inv, o[1] * inv, o[2] * inv, o[3] * inv));
        st4(op + 4, make_float4(o[4] * inv, o[5] * inv, o[6] * inv, o[7] * inv));
    }
}

// ------------------------------------------------------------------ batched fp32 GEMM (row attention)
// C[z] = A[z] (MxK, K contiguous) * B[z]   with B given as [N][K] (BT) or [K][N] (!BT).
template <bool BT>
__global__ void __launch_bounds__(NTHREADS) k_gemm(const float* __restrict__ A, const float* __restrict__ Bm, float* __restrict__ Cm,
                                                   int M, int N, int K, size_t sA, size_t sB, size_t sC, int lda, int ldb, int ldc) {
    constexpr int KT = 8, LD = 132;
    __shared__ __align__(16) float As[2][KT][LD];
    __shared__ __align__(16) float Bs[2][KT][LD];
    const int z = blockIdx.z;
    A += z * sA; Bm += z * sB; Cm += z * sC;
    const int m0 = blockIdx.y * 128, n0 = blockIdx.x * 128;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    // loader coordinates
    const int lrow = tid >> 1, lk = (tid & 1) * 4;          // K-contiguous operands: 128 rows x 8 k
    const int bk = tid >> 5, bn = (tid & 31) * 4;           // N-contiguous B: 8 k x 128 n
    float4 ra, rb;
    // 16-byte loads need rows that start on a 16-byte boundary: a site count that is not a multiple of 4 (the logits S have
    // row pitch C) falls back to scalar loads
    const bool va = (lda & 3) == 0 && (sA & 3) == 0, vb = (ldb & 3) == 0 && (sB & 3) == 0;
    auto gload = [&](int k0) {
        ra = make_float4(0.f, 0.f, 0.f, 0.f);
        rb = ra;
        int m = m0 + lrow, kk = k0 + lk;
        if (m < M) {
            const float* p = A + (size_t)m * lda + kk;
            if (kk + 3 < K && va) ra = ld4(p);
            else { if (kk < K) ra.x = p[0]; if (kk + 1 < K) ra.y = p[1]; if (kk + 2 < K) ra.z = p[2]; if (kk + 3 < K) ra.w = p[3]; }
        }
        if (BT) {
            int n = n0 + lrow;
            if (n < N) {
                const float* p = Bm + (size_t)n * ldb + kk;
                if (kk + 3 < K && vb) rb = ld4(p);
                else { if (kk < K) rb.x = p[0]; if (kk + 1 < K) rb.y = p[1]; if (kk + 2 < K) rb.z = p[2]; if (kk + 3 < K) rb.w = p[3]; }
            }
        } else {
            int k = k0 + bk, n = n0 + bn;
            if (k < K) {
                const float* p = Bm + (size_t)k * ldb + n;
                if (n + 3 < N && vb) rb = ld4(p);
                else { if (n < N) rb.x = p[0]; if (n + 1 < N) rb.y = p[1]; if (n + 2 < N) rb.z = p[2]; if (n + 3 < N) rb.w = p[3]; }
            }
        }
    };
    auto sstore = [&](int buf) {
        As[buf][lk][lrow] = ra.x; As[buf][lk + 1][lrow] = ra.y; As[buf][lk + 2][lrow] = ra.z; As[buf][lk + 3][lrow] = ra.w;
        if (BT) { Bs[buf][lk][lrow] = rb.x; Bs[buf][lk + 1][lrow] = rb.y; Bs[buf][lk + 2][lrow] = rb.z; Bs[buf][lk + 3][lrow] = rb.w; }
        else st4(&Bs[buf][bk][bn], rb);
    };
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    gload(0);
    sstore(0);
    __syncthreads();
    const int nk = (K + KT - 1) / KT;
    for (int kt = 0; kt < nk; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < nk) gload((kt + 1) * KT);
#pragma unroll
        for (int k = 0; k < KT; ++k) {
            float4 a0 = ld4(&As[buf][k][ty * 4]), a1 = ld4(&As[buf][k][64 + ty * 4]);
            float4 b0 = ld4(&Bs[buf][k][tx * 4]), b1 = ld4(&Bs[buf][k][64 + tx * 4]);
            float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
        }
        if (kt + 1 < nk) sstore(buf ^ 1);
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        int m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
        if (m >= M) continue;
#pragma unroll
        for (int jh = 0; jh < 2; ++jh) {
            int n = n0 + jh * 64 + tx * 4;
            float* p = Cm + (size_t)m * ldc + n;
            if (n + 3 < N && (ldc & 3) == 0 && (sC & 3) == 0) st4(p, make_float4(acc[i][jh * 4], acc[i][jh * 4 + 1], acc[i][jh * 4 + 2], acc[i][jh * 4 + 3]));
            else for (int j = 0; j < 4; ++j) if (n + j < N) p[j] = acc[i][jh * 4 + j];
        }
    }
}

// softmax over the last axis of S [B*H, C, C] with the pad fill; one warp per row.
__global__ void __launch_bounds__(NTHREADS) k_softmax_rows(float* __restrict__ S, int C, int rows_per_z, const uint8_t* __restrict__ mask) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * 8 + warp;
    if (row >= rows_per_z) return;
    const int z = blockIdx.y;
    const int b = z / H;
    float* p = S + ((size_t)z * rows_per_z + row) * C;
    const uint8_t* mk = mask ? mask + (size_t)b * C : nullptr;
    float m = -INFINITY;
    for (int j = lane; j < C; j += 32) {
        float s = (mk && mk[j]) ? -10000.0f : p[j];
        m = fmaxf(m, s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float l = 0.f;
    for (int j = lane; j < C; j += 32) {
        float s = (mk && mk[j]) ? -10000.0f : p[j];
        float e = expf(s - m);
        p[j] = e;
        l += e;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
    float inv = 1.0f / l;
    for (int j = lane; j < C; j += 32) p[j] *= inv;
}


// ------------------------------------------------------------------ tensor-core row attention (precision bf16x3)
__device__ __forceinline__ void split_bf16(float v, __nv_bfloat16& hi, __nv_bfloat16& lo) {
    hi = __float2bfloat16_rn(v);
    lo = NNJ_LO_BF16(__float2bfloat16_rn(v - __bfloat162float(hi)));
}

// softmax over key sites of S [Z, C, C] (fp32) -> probabilities as bf16 hi/lo planes; one warp per row; C even.
__global__ void __launch_bounds__(NTHREADS) k_softmax_rows_split(const float* __restrict__ S, __nv_bfloat16* __restrict__ Ph,
                                                                 __nv_bfloat16* __restrict__ Pl, int C, const uint8_t* __restrict__ mask) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * 8 + warp;
    if (row >= C) return;
    const int z = blockIdx.y, b = z / H;
    const size_t base = ((size_t)z * C + row) * C;
    const float2* p = reinterpret_cast<const float2*>(S + base);
    const uint8_t* mk = mask ? mask + (size_t)b * C : nullptr;
    const int C2 = C >> 1;
    float m = -INFINITY;
    for (int j = lane; j < C2; j += 32) {
        float2 v = p[j];
        if (mk) { if (mk[2 * j]) v.x = -10000.0f; if (mk[2 * j + 1]) v.y = -10000.0f; }
        m = fmaxf(m, fmaxf(v.x, v.y));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float l = 0.f;
    for (int j = lane; j < C2; j += 32) {
        float2 v = p[j];
        if (mk) { if (mk[2 * j]) v.x = -10000.0f; if (mk[2 * j + 1]) v.y = -10000.0f; }
        l += expf(v.x - m) + expf(v.y - m);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
    const float inv = 1.0f / l;
    __nv_bfloat162* oh = reinterpret_cast<__nv_bfloat162*>(Ph + base);
    __nv_bfloat162* ol = reinterpret_cast<__nv_bfloat162*>(Pl + base);
    for (int j = lane; j < C2; j += 32) {
        float2 v = p[j];
        if (mk) { if (mk[2 * j]) v.x = -10000.0f; if (mk[2 * j + 1]) v.y = -10000.0f; }
        float e0 = expf(v.x - m) * inv, e1 = expf(v.y - m) * inv;
        __nv_bfloat162 hh, ll;
        split_bf16(e0, hh.x, ll.x);
        split_bf16(e1, hh.y, ll.y);
        oh[j] = hh; ol[j] = ll;
    }
}

// The same for rows of at most 256 NCH sites (C % 8 == 0): the row stays in registers (one read of S instead of three), 32-byte loads and
// 16-byte stores per lane, MUFU ex2 on log2-scaled logits (2^-22 relative, far below the bf16 hi/lo split of P).
template <int NCH>
__global__ void __launch_bounds__(NTHREADS) k_softmax_rows_split_reg(const float* __restrict__ S, __nv_bfloat16* __restrict__ Ph,
                                                                     __nv_bfloat16* __restrict__ Pl, int C, const uint8_t* __restrict__ mask) {
    // Pl == nullptr (NNJ_PREC_BF16): P leaves as one bf16 plane
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * 8 + warp;
    if (row >= C) return;
    const int z = blockIdx.y, b = z / H;
    const size_t base = ((size_t)z * C + row) * C;
    const uint8_t* mk = mask ? mask + (size_t)b * C : nullptr;
    float v[NCH][8];
    float m = -INFINITY;
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
        const int j = c * 256 + lane * 8;
        if (j < C) {
            const float4 a0 = __ldcs(reinterpret_cast<const float4*>(S + base + j)), a1 = __ldcs(reinterpret_cast<const float4*>(S + base + j + 4));
            v[c][0] = a0.x; v[c][1] = a0.y; v[c][2] = a0.z; v[c][3] = a0.w; v[c][4] = a1.x; v[c][5] = a1.y; v[c][6] = a1.z; v[c][7] = a1.w;
            if (mk) {
                const uint2 mm = *reinterpret_cast<const uint2*>(mk + j);
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    if (((e < 4 ? mm.x : mm.y) >> (8 * (e & 3))) & 0xffu) v[c][e] = -10000.0f;      // axial_attention.py:81-82
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) m = fmaxf(m, v[c][e]);
        } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) v[c][e] = -INFINITY;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    const float ms = -m * 1.4426950408889634f;
    float l = 0.f;
#pragma unroll
    for (int c = 0; c < NCH; ++c)
#pragma unroll
        for (int e = 0; e < 8; ++e) { v[c][e] = ex2_approx(fmaf(v[c][e], 1.4426950408889634f, ms)); l += v[c][e]; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
    const float inv = 1.0f / l;
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
        const int j = c * 256 + lane * 8;
        if (j < C) {
            uint4 hh, ll;
            split2(v[c][0] * inv, v[c][1] * inv, hh.x, ll.x);
            split2(v[c][2] * inv, v[c][3] * inv, hh.y, ll.y);
            split2(v[c][4] * inv, v[c][5] * inv, hh.z, ll.z);
            split2(v[c][6] * inv, v[c][7] * inv, hh.w, ll.w);
            *reinterpret_cast<uint4*>(Ph + base + j) = hh;
            if (Pl) *reinterpret_cast<uint4*>(Pl + base + j) = ll;
        }
    }
}

// ------------------------------------------------------------------ host-side driver
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// The tensor-core path works on the site-major residual stream: LN1 + row q|k|v, the row GEMMs and the feed-forward block run on
// tcgen05 (nnj_encoder_tc.cu, nnj_tc.cu), and so does the fused column block up to 128 taxa; above that the CUDA-core column
// stages below run on the same stream.
static bool use_tc(const Model* m, int C) { return m->cfg.precision != NNJ_PREC_FP32 && (C % 8) == 0; }

// per-tree workspace floats for the encoder
static size_t enc_tree_floats(const Model* m, int R, int C) {
    size_t act = (size_t)R * C * D;
    size_t s = (size_t)H * C * C;         // row-attention logits; also holds the column-attention context
    size_t p = use_tc(m, C) ? s : 0;      // probabilities as bf16 hi/lo planes (tensor-core path)
    size_t xs = use_tc(m, C) ? xs_tree_floats(R * C) : 0;   // site-major residual stream (tile-planar, whole 128-token tiles)
    return 3 * act + (s > act ? s : act) + p + xs; // q (row ctx), k, v, S [, P] [, xs]
}

int encoder_chunk(const Model* m, int B, int R, int C) {
    size_t per = enc_tree_floats(m, R, C) * sizeof(float);
    size_t budget = (size_t)16 << 30;
    int ch = (int)(budget / per);
    if (ch < 1) ch = 1;
    if (ch > B) ch = B;
    const int n = (B + ch - 1) / ch;     // equal-sized chunks: no small tail launch
    return (B + n - 1) / n;
}

size_t encoder_ws_bytes(const Model* m, int B, int R, int C) {
    return align_up(enc_tree_floats(m, R, C) * sizeof(float) * encoder_chunk(m, B, R, C), 256) + 256;
}

int run_encoder(Model* m, const int8_t* data, const uint8_t* mask, int B, int R, int L, float* x, size_t x_tree_stride,
                void* ws, size_t ws_bytes, cudaStream_t st) {
    const int C = L;  // patch_size == 1
    if (ws_bytes < encoder_ws_bytes(m, B, R, C)) return set_error(NNJ_ERR_WORKSPACE, "encode: workspace too small");
    const int chunk = encoder_chunk(m, B, R, C);
    const size_t act = (size_t)R * C * D;
    float* wsf = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 255) / 256 * 256);
    float* q = wsf;
    float* k = q + act * chunk;
    float* v = k + act * chunk;
    float* S = v + act * chunk;   // region of chunk * max(H*C*C, act) floats
    const bool tc = use_tc(m, C);
    const bool col_tc = tc && R <= 128;       // the fused column block (k_enc_colblock_tc) holds at most 128 taxa
    const int xsm = tc ? 1 : 0;
    const size_t s_floats = (size_t)H * C * C > act ? (size_t)H * C * C : act;
    __nv_bfloat16* P = reinterpret_cast<__nv_bfloat16*>(S + s_floats * chunk);   // [2 planes][chunk*H][C][C] (tensor-core path only)
    float* xs_ws = S + s_floats * chunk + (tc ? (size_t)H * C * C * chunk : 0);  // site-major residual stream [chunk][tiles of 128 tokens t = c R + r][16 chunks][128][4]
    const int T = R * C;
    const int tiles = (T + TILE_ROWS - 1) / TILE_ROWS;
    const size_t smem_qkv = (TILE_ROWS * LDA + 4096) * sizeof(float);
    const size_t smem_ffn = (2 * TILE_ROWS * LDA + 2 * 4096) * sizeof(float);
    const size_t smem_col = (size_t)2 * R * D * sizeof(float);
    static DevOnce attr_once;      // per device, not per process
    if (attr_once.need()) {
        cudaFuncSetAttribute(k_ffn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ffn);
        cudaFuncSetAttribute(k_ln_qkv<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_qkv);
        cudaFuncSetAttribute(k_ln_qkv<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_qkv);
        cudaFuncSetAttribute(k_out_proj<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_qkv);
        cudaFuncSetAttribute(k_out_proj<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_qkv);
        cudaFuncSetAttribute(k_col_attn, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        attr_once.done();
    }
    if (!col_tc && smem_col > 200 * 1024) return set_error(NNJ_ERR_INVALID, "encode: too many taxa for the column-attention kernel (max 400)");
    if (R == 1) return set_error(NNJ_ERR_INVALID, "encode: R == 1 is not supported");
    const float row_scale = (1.0f / sqrtf((float)DH)) / sqrtf((float)R);   // align_scaling, axial_attention.py:31-33
    const float col_scale = 1.0f / sqrtf((float)DH);
    for (int b0 = 0; b0 < B; b0 += chunk) {
        const int nb = (B - b0 < chunk) ? (B - b0) : chunk;
        float* xout = x + (size_t)b0 * x_tree_stride;
        float* xb = xsm ? xs_ws : xout;                       // the residual stream the layers work on
        const size_t xstr = xsm ? xs_tree_floats(R * C) : x_tree_stride;
        const int8_t* db = data + (size_t)b0 * R * L * 4;
        const uint8_t* mb = mask ? mask + (size_t)b0 * C : nullptr;
        prof_begin(KC_EMBED, st);
        k_embed<<<dim3((T + 1023) / 1024, nb), NTHREADS, 0, st>>>(db, xb, xstr, R, L, m->embed, xsm);
        LAUNCH_CHECK();
        for (int l = 0; l < m->num_layers; ++l) {
            const LayerW& lw = m->layers[l];
            // --- tied row attention
            if (tc) {
                const size_t pl = act * chunk;                 // elements per bf16 plane of q / k / v
                __nv_bfloat16 *qh = reinterpret_cast<__nv_bfloat16*>(q), *ql = qh + pl;
                __nv_bfloat16 *kh = reinterpret_cast<__nv_bfloat16*>(k), *kl = kh + pl;
                __nv_bfloat16 *vh = reinterpret_cast<__nv_bfloat16*>(v), *vl = vh + pl;
                const size_t pp = (size_t)chunk * H * C * C;   // elements per plane of P
                const int KD = R * DH;
                // V as [B,H,C,R*8]: the MN-major B operand of ctx = P V
                if (int e = launch_enc_rowqkv_tc(m, l, xb, xstr, nb, R, C, row_scale, mb, qh, ql, kh, kl, vh, vl, st)) return e;
                const int products = m->cfg.precision == NNJ_PREC_BF16 ? 1 : 3;
                __nv_bfloat16* Plo = products == 1 ? nullptr : P + pp;      // one-product mode: the register softmax writes the hi plane only
                float* rowsum = nullptr;
                if (row_qk_softmax_ok(C, products)) {      // softmax in the Q K^T epilogue: S never leaves the chip
                    rowsum = S;                             // [nb * H][C]: the logits buffer is free in this form
                    if (int e = launch_row_qk_softmax(KC_ROW_QK, qh, ql, kh, kl, P, P + pp, rowsum, mb, H, nb * H, C, KD, st)) return e;
                } else {
                    if (int e = launch_tc_gemm(KC_ROW_QK, qh, ql, kh, kl, S, nb * H, C, C, KD, KD, (size_t)C * KD, KD, (size_t)C * KD, C, (size_t)C * C, st, products)) return e;
                    prof_begin(KC_ROW_SOFTMAX, st);
                    if (C <= 512) k_softmax_rows_split_reg<2><<<dim3((C + 7) / 8, nb * H), NTHREADS, 0, st>>>(S, P, Plo, C, mb);
                    else if (C <= 1024) k_softmax_rows_split_reg<4><<<dim3((C + 7) / 8, nb * H), NTHREADS, 0, st>>>(S, P, Plo, C, mb);
                    else k_softmax_rows_split<<<dim3((C + 7) / 8, nb * H), NTHREADS, 0, st>>>(S, P, P + pp, C, mb);
                    LAUNCH_CHECK();
                }
                if (int e = launch_tc_gemm_bmn(KC_ROW_PV, P, P + pp, vh, vl, q /*ctx fp32 [B,H,C,R*8]*/, nb * H, C, KD, C, C, (size_t)C * C, KD,
                                               (size_t)C * KD, KD, (size_t)C * KD, st, products, rowsum)) return e;
            } else {
                prof_begin(KC_LN_QKV, st);
                k_ln_qkv<true><<<dim3(tiles, nb), NTHREADS, smem_qkv, st>>>(xb, xstr, R, C, lw.row, row_scale, mb, q, k, v, xsm);
                LAUNCH_CHECK();
                prof_begin(KC_ROW_QK, st);
                k_gemm<true><<<dim3((C + 127) / 128, (C + 127) / 128, nb * H), NTHREADS, 0, st>>>(
                    q, k, S, C, C, R * DH, (size_t)C * R * DH, (size_t)C * R * DH, (size_t)C * C, R * DH, R * DH, C);
                LAUNCH_CHECK();
                prof_begin(KC_ROW_SOFTMAX, st);
                k_softmax_rows<<<dim3((C + 7) / 8, nb * H), NTHREADS, 0, st>>>(S, C, C, mb);
                LAUNCH_CHECK();
                prof_begin(KC_ROW_PV, st);
                k_gemm<false><<<dim3((R * DH + 127) / 128, (C + 127) / 128, nb * H), NTHREADS, 0, st>>>(
                    S, v, q /*ctx*/, C, R * DH, C, (size_t)C * C, (size_t)C * R * DH, (size_t)C * R * DH, C, R * DH, R * DH);
                LAUNCH_CHECK();
            }
            if (col_tc) {
                // --- row out_proj + residual, LN2, column attention, column out_proj + residual: one kernel
                if (int e = launch_enc_colblock_tc(m, l, xb, xstr, q, nb, R, C, mb, st)) return e;
            } else {
                prof_begin(KC_OUT_PROJ, st);
                k_out_proj<true><<<dim3(tiles, nb), NTHREADS, smem_qkv, st>>>(xb, xstr, R, C, q, lw.row.ot, lw.row.ob, xsm);
                LAUNCH_CHECK();
                // --- column attention
                prof_begin(KC_LN_QKV, st);
                k_ln_qkv<false><<<dim3(tiles, nb), NTHREADS, smem_qkv, st>>>(xb, xstr, R, C, lw.col, col_scale, mb, q, k, v, xsm);
                LAUNCH_CHECK();
                prof_begin(KC_COL_ATTN, st);
                k_col_attn<<<dim3(C, nb), NTHREADS, smem_col, st>>>(q, k, v, S /*ctx [B,R,C,64]*/, R, C, mb);
                LAUNCH_CHECK();
                prof_begin(KC_OUT_PROJ, st);
                k_out_proj<false><<<dim3(tiles, nb), NTHREADS, smem_qkv, st>>>(xb, xstr, R, C, S, lw.col.ot, lw.col.ob, xsm);
                LAUNCH_CHECK();
            }
            // --- feed forward (per token: the memory order of the stream does not matter)
            if (tc) {
                if (int e = launch_enc_ffn_tc(m, l, xb, xstr, nb, R, C, st)) return e;
            } else {
                prof_begin(KC_FFN, st);
                k_ffn<<<dim3(tiles, nb), NTHREADS, smem_ffn, st>>>(xb, xstr, R, C, lw.ffn, xsm);
                LAUNCH_CHECK();
            }
        }
        if (xsm) {
            if (int e = launch_sm_to_nm(xb, xstr, xout, x_tree_stride, nb, R, C, st)) return e;
        }
    }
    return NNJ_OK;
}

}  // namespace nnj
