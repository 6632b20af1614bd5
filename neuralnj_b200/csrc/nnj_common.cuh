// nnj_common.cuh — shared device helpers for the NeuralNJ hot-path kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

namespace nnj {

constexpr int D = 64;          // embedding width (cfgs.model.embed_dim)
constexpr int H = 8;           // heads
constexpr int DH = 8;          // head dim
constexpr int FF = 256;        // feed-forward width (4*D, model.py:28)
constexpr int TILE_ROWS = 128; // rows of a token tile
constexpr int LDA = 68;        // smem row pitch (floats) of a [128][64] tile: 16B aligned, conflict-free
constexpr int NTHREADS = 256;  // 16 x 16 thread grid: 8 rows x 4 cols per thread

extern thread_local long long g_launches;   // kernels launched by this library on this host thread

__device__ __forceinline__ float gelu_erf(float x) {            // torch.nn.GELU() (exact erf form)
    return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

// ---- fast forms used by the tensor-core (bf16x3) kernels: MUFU ex2 / rcp (2^-22 relative), far below the ~2^-17 operand split
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float sigmoid_fast(float x) { return rcp_approx(1.0f + ex2_approx(-1.4426950408889634f * x)); }
// GELU(x) = x * Phi(x), Phi(-|x|) = 0.5 erfc(|x|/sqrt 2) = poly6(u) exp(-x^2/2), u = 1/(1 + p|x|): coefficients fitted here
// (scratch/phi_fit.py), |gelu_fast - gelu_erf| < 1e-7 absolute over the whole fp32 range (erff itself carries ~1e-7).
__device__ __forceinline__ float gelu_fast(float x) {
    const float z = fabsf(x);
    const float u = rcp_approx(fmaf(2.760034502e-01f, z, 1.0f));
    float p = -1.134462506e-01f;
    p = fmaf(p, u, 4.407724440e-01f);
    p = fmaf(p, u, -3.137964904e-01f);
    p = fmaf(p, u, 3.221081495e-01f);
    p = fmaf(p, u, 4.673849419e-02f);
    p = fmaf(p, u, 1.176236272e-01f);
    const float h = p * u * ex2_approx(z * z * -0.72134752044448170f);
    return x * (x >= 0.f ? 1.0f - h : h);
}

// ---- packed fp32x2 arithmetic (FFMA2 / FMUL2 / FADD2 on sm_100): one issue slot for two lanes of work, each lane rounded exactly
//      like the scalar instruction (the packed forms below are bit-identical to their scalar counterparts)
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
        "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return d;
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmul.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tadd.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
__device__ __forceinline__ float2 fsub2(float2 a, float2 b) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tsub.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
__device__ __forceinline__ float2 splat2(float v) { return make_float2(v, v); }
// sigmoid_fast / gelu_fast on two values.  The score / blend epilogues are bound by the MUFU pipe (16 results per clock and SM: a
// warp instruction holds a quadrant's unit for 8 clocks, four MUFU per pair-site-channel), so the two reciprocals of a value pair
// share ONE MUFU: r = rcp(a b), 1/a = b r, 1/b = a r (two extra FMA-pipe multiplies).  Both results carry the 2^-22 of rcp.approx plus
// one rounding - the same grade as the scalar forms, not bit-identical to them.  NNJ_RCP_PAIR=0 restores one rcp per value.
#ifndef NNJ_RCP_PAIR
#define NNJ_RCP_PAIR 1
#endif
__device__ __forceinline__ float2 rcp_pair(float2 d) {
#if NNJ_RCP_PAIR
    const float r = rcp_approx(d.x * d.y);
    return fmul2(make_float2(d.y, d.x), splat2(r));
#else
    return make_float2(rcp_approx(d.x), rcp_approx(d.y));
#endif
}
__device__ __forceinline__ float2 sigmoid_fast2(float2 x) {
    float2 t = fmul2(splat2(-1.4426950408889634f), x);
#if NNJ_RCP_PAIR
    t.x = fminf(t.x, 60.0f); t.y = fminf(t.y, 60.0f);      // (1 + 2^60)^2 stays finite; sigmoid < 2^-60 reads as 2^-60
#endif
    const float2 d = fadd2(splat2(1.0f), make_float2(ex2_approx(t.x), ex2_approx(t.y)));
    return rcp_pair(d);
}
__device__ __forceinline__ float2 gelu_fast2(float2 x) {
    const float2 z = make_float2(fabsf(x.x), fabsf(x.y));
    const float2 d = ffma2(splat2(2.760034502e-01f), z, splat2(1.0f));
    const float2 u = rcp_pair(d);
    float2 p = splat2(-1.134462506e-01f);
    p = ffma2(p, u, splat2(4.407724440e-01f));
    p = ffma2(p, u, splat2(-3.137964904e-01f));
    p = ffma2(p, u, splat2(3.221081495e-01f));
    p = ffma2(p, u, splat2(4.673849419e-02f));
    p = ffma2(p, u, splat2(1.176236272e-01f));
    const float2 t = fmul2(fmul2(z, z), splat2(-0.72134752044448170f));
    const float2 h = fmul2(fmul2(p, u), make_float2(ex2_approx(t.x), ex2_approx(t.y)));
    const float2 g = fsub2(splat2(1.0f), h);
    return fmul2(x, make_float2(x.x >= 0.f ? g.x : h.x, x.y >= 0.f ? g.y : h.y));
}

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ float f4c(const float4& v, int k) { return k == 0 ? v.x : (k == 1 ? v.y : (k == 2 ? v.z : v.w)); }

// Copy a [64 k][64 col] fp32 weight (already transposed on the host) into shared memory.
__device__ __forceinline__ void load_w64(float* __restrict__ Ws, const float* __restrict__ Wg) {
#pragma unroll
    for (int it = 0; it < 4; ++it) {
        int idx = it * NTHREADS + threadIdx.x;
        st4(Ws + idx * 4, __ldg(reinterpret_cast<const float4*>(Wg) + idx));
    }
}

// acc[8][4] += As[rows ty*8..+7][0..63] * Ws[0..63][cols tx*4..+3]
// As: smem row-major, pitch LDA.  Ws: smem [k][64].  k ascends -> deterministic sums.
__device__ __forceinline__ void tile_mma64(float (&acc)[8][4], const float* __restrict__ As,
                                           const float* __restrict__ Ws, int ty, int tx) {
    const float* ap = As + ty * 8 * LDA;
    const float* wp = Ws + tx * 4;
#pragma unroll 2
    for (int k = 0; k < 64; k += 4) {
        float4 a[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) a[i] = ld4(ap + i * LDA + k);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            float4 w = ld4(wp + (k + kk) * 64);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float av = f4c(a[i], kk);
                acc[i][0] = fmaf(av, w.x, acc[i][0]);
                acc[i][1] = fmaf(av, w.y, acc[i][1]);
                acc[i][2] = fmaf(av, w.z, acc[i][2]);
                acc[i][3] = fmaf(av, w.w, acc[i][3]);
            }
        }
    }
}

__device__ __forceinline__ void acc_set_bias(float (&acc)[8][4], const float* __restrict__ bias, int tx) {
    float4 b = bias ? __ldg(reinterpret_cast<const float4*>(bias) + tx) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int i = 0; i < 8; ++i) { acc[i][0] = b.x; acc[i][1] = b.y; acc[i][2] = b.z; acc[i][3] = b.w; }
}

__device__ __forceinline__ void acc_store_smem(const float (&acc)[8][4], float* __restrict__ As, int ty, int tx) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
        st4(As + (ty * 8 + i) * LDA + tx * 4, make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]));
}

// In-place LayerNorm(64) of a [128][LDA] smem tile; 2 threads per row (torch LayerNorm, eps 1e-5, biased var).
__device__ __forceinline__ void tile_layernorm(float* __restrict__ As, const float* __restrict__ gamma,
                                               const float* __restrict__ beta) {
    int row = threadIdx.x >> 1, half = threadIdx.x & 1;
    float* p = As + row * LDA + half * 32;
    float v[32];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 32; k += 4) {
        float4 t = ld4(p + k);
        v[k] = t.x; v[k + 1] = t.y; v[k + 2] = t.z; v[k + 3] = t.w;
        s += (t.x + t.y) + (t.z + t.w);
    }
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    float mean = s * (1.0f / 64.0f);
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < 32; ++k) { float d = v[k] - mean; q = fmaf(d, d, q); }
    q += __shfl_xor_sync(0xffffffffu, q, 1);
    float rstd = 1.0f / sqrtf(q * (1.0f / 64.0f) + 1e-5f);
#pragma unroll
    for (int k = 0; k < 32; k += 4) {
        float4 g = __ldg(reinterpret_cast<const float4*>(gamma + half * 32 + k));
        float4 b = __ldg(reinterpret_cast<const float4*>(beta + half * 32 + k));
        st4(p + k, make_float4((v[k] - mean) * rstd * g.x + b.x, (v[k + 1] - mean) * rstd * g.y + b.y,
                               (v[k + 2] - mean) * rstd * g.z + b.z, (v[k + 3] - mean) * rstd * g.w + b.w));
    }
}

// Sum over the 16 lanes that share `ty` (consecutive lanes of a warp).
__device__ __forceinline__ float reduce16(float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    return v;
}

// Philox4x32-10 (Salmon et al., SC 2011; the constants of Random123), word 0 of the output block: the resampling draws of the bootstrap
// (nnj_support.cu) and of the RELL replicates (nnj_llh_nni.cu).
__device__ __forceinline__ uint32_t philox_x0(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int round = 0; round < 10; ++round) {
        const uint32_t lo0 = 0xD2511F53u * c0, hi0 = __umulhi(0xD2511F53u, c0);
        const uint32_t lo1 = 0xCD9E8D57u * c2, hi1 = __umulhi(0xCD9E8D57u, c2);
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return c0;
}

// position of pair (i<j) among combinations(range(n), 2)  (environment.py:458)
__host__ __device__ __forceinline__ int pair_index(int i, int j, int n) { return i * n - i * (i + 1) / 2 + (j - i - 1); }

// inverse of pair_index
__device__ __forceinline__ void pair_from_index(int p, int n, int& i, int& j) {
    float fn = 2.0f * n - 1.0f;
    int ii = (int)floorf((fn - sqrtf(fmaxf(fn * fn - 8.0f * (float)p, 0.f))) * 0.5f);
    if (ii < 0) ii = 0;
    if (ii > n - 2) ii = n - 2;
    while (ii > 0 && pair_index(ii, ii + 1, n) > p) --ii;
    while (ii < n - 2 && pair_index(ii + 1, ii + 2, n) <= p) ++ii;
    i = ii;
    j = p - pair_index(ii, ii + 1, n) + ii + 1;
}

}  // namespace nnj
