// nnj_llh.cuh — device helpers of the tree likelihood shared by k_llh (nnj_llh.cu), the NNI quartet kernel (nnj_llh_nni.cu) and the
// RELL draws of branch support and the topology test (nnj_llh_nni.cu, nnj_llh_topo.cu).
// Everything is fp64; CLVs are [4 rate classes][4 states] per (node, pattern), scaled by 2^256 as described in nnj_llh.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "nnj_common.cuh"

namespace nnj {

constexpr int LLH_THREADS = 512;
constexpr int LLH_MODEL = 64;      // doubles per tree of the packed model; its slots below (likelihood.py SubstModel.pack writes the same layout)
constexpr int MDL_LAM = 0;         // 4 eigenvalues of the normalised rate matrix
constexpr int MDL_U = 4;           // U [4][4] and U^-1 [4][4]: Q = U diag(lam) U^-1
constexpr int MDL_UINV = 20;
constexpr int MDL_FREQ = 36;       // 4 base frequencies
constexpr int MDL_RATE = 40;       // 4 gamma class rates
constexpr int MDL_PINV = 44, MDL_ALPHA = 45;
constexpr int MDL_FLAGS = 46;      // free parameters: 1 GTR rates, 2 alpha (+G), 4 p_inv (+I); slot 47 is padding
constexpr int MDL_GTR = 48;        // 6 GTR exchangeabilities AC AG AT CG CT GT; slots 54..63 are padding
constexpr double BRLEN_MIN = 1e-6, BRLEN_MAX = 100.0;    // every length, in evaluation and optimisation, is clamped to this range
constexpr int SCALE_EXP = 256;
constexpr double SCALE_BELOW = 0x1p-256, SCALE_UP = 0x1p256, SCALE_LN = 256.0 * 0.69314718055994530942;

__host__ __device__ __forceinline__ double clampd(double v, double lo, double hi) { return v < lo ? lo : (v > hi ? hi : v); }

// P(t)[k][a][b] = sum_j U[a][j] exp(lam_j r_k t) Uinv[j][b] for two branch lengths at once (threads 0..127), then a barrier
__device__ __forceinline__ void pmat2(double* Pm, const double* mdl, double t0, double t1) {
    const int i = threadIdx.x;
    if (i < 128) {
        const int w = i >> 6, k = (i >> 4) & 3, a = (i >> 2) & 3, b = i & 3;
        const double t = w ? t1 : t0;
        double s = 0.0;
#pragma unroll
        for (int j = 0; j < 4; ++j) s += mdl[MDL_U + a * 4 + j] * exp(mdl[MDL_LAM + j] * mdl[MDL_RATE + k] * t) * mdl[MDL_UINV + j * 4 + b];
        Pm[i] = s;
    }
    __syncthreads();
}
// the same for one branch length (threads 0..63), then a barrier
__device__ __forceinline__ void pmat1(double* Pm, const double* mdl, double t) {
    const int i = threadIdx.x;
    if (i < 64) {
        const int k = (i >> 4) & 3, a = (i >> 2) & 3, b = i & 3;
        double s = 0.0;
#pragma unroll
        for (int j = 0; j < 4; ++j) s += mdl[MDL_U + a * 4 + j] * exp(mdl[MDL_LAM + j] * mdl[MDL_RATE + k] * t) * mdl[MDL_UINV + j * 4 + b];
        Pm[i] = s;
    }
    __syncthreads();
}

// subtree vector of node v at pattern s: the tip's state mask for a leaf (v < R), else D[v] (Dt = [R-1][L][16] of one tree)
__device__ __forceinline__ void clv_load(int R, int L, const double* Dt, const uint8_t* tips, int v, int s, double (&x)[16]) {
    if (v < R) {
        const int m = tips[(size_t)v * L + s];
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int c = 0; c < 4; ++c) x[k * 4 + c] = (double)((m >> c) & 1);
    } else {
        const double2* p = reinterpret_cast<const double2*>(Dt + ((size_t)(v - R) * L + s) * 16);
#pragma unroll
        for (int i = 0; i < 8; ++i) { const double2 d = p[i]; x[2 * i] = d.x; x[2 * i + 1] = d.y; }
    }
}
__device__ __forceinline__ int cnt_load(int R, int L, const int32_t* Dnt, int v, int s) { return v < R ? 0 : Dnt[(size_t)(v - R) * L + s]; }
__device__ __forceinline__ void vec_load(const double* p, double (&x)[16]) {
    const double2* q = reinterpret_cast<const double2*>(p);
#pragma unroll
    for (int i = 0; i < 8; ++i) { const double2 d = q[i]; x[2 * i] = d.x; x[2 * i + 1] = d.y; }
}
__device__ __forceinline__ void vec_store(double* p, const double (&x)[16]) {
    double2* q = reinterpret_cast<double2*>(p);
#pragma unroll
    for (int i = 0; i < 8; ++i) q[i] = make_double2(x[2 * i], x[2 * i + 1]);
}
// y[k][a] = sum_b P[k][a][b] x[k][b]
__device__ __forceinline__ void pm_apply(const double* P, const double (&x)[16], double (&y)[16]) {
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            double s = 0.0;
#pragma unroll
            for (int b = 0; b < 4; ++b) s = fma(P[k * 16 + c * 4 + b], x[k * 4 + b], s);
            y[k * 4 + c] = s;
        }
}
// the scaled combine: px = px * py, multiplied by 2^256 (exact) when all 16 entries are below 2^-256; returns 1 then, else 0
__device__ __forceinline__ int mul_scaled(double (&px)[16], const double (&py)[16]) {
    double mx = 0.0;
#pragma unroll
    for (int i = 0; i < 16; ++i) { px[i] *= py[i]; mx = fmax(mx, px[i]); }
    if (mx < SCALE_BELOW) {
#pragma unroll
        for (int i = 0; i < 16; ++i) px[i] *= SCALE_UP;
        return 1;
    }
    return 0;
}

// block-wide sums of two values in a fixed order; every thread returns with the totals.  red: 2 * 32 + 2 doubles.
__device__ __forceinline__ void block_sum2(double& v0, double& v1, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { v0 += __shfl_xor_sync(0xffffffffu, v0, o); v1 += __shfl_xor_sync(0xffffffffu, v1, o); }
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { red[warp] = v0; red[32 + warp] = v1; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double s0 = 0.0, s1 = 0.0;
        for (int w = 0; w < LLH_THREADS / 32; ++w) { s0 += red[w]; s1 += red[32 + w]; }
        red[64] = s0; red[65] = s1;
    }
    __syncthreads();
    v0 = red[64]; v1 = red[65];
    __syncthreads();
}

// one pattern's row of the Newton sumtable of a branch: S[k][j] = (sum_c pi_c u[k][c] Umat[c][j]) (sum_c Uinv[j][c] d[k][c]),
// u the vector at the far end, d the vector below the branch
__device__ __forceinline__ void sumtable_row(const double* mdl, const double (&u)[16], const double (&d)[16], double (&sv)[16]) {
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double A = 0.0, Bm = 0.0;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                A = fma(mdl[MDL_FREQ + c] * u[k * 4 + c], mdl[MDL_U + c * 4 + j], A);
                Bm = fma(mdl[MDL_UINV + j * 4 + c], d[k * 4 + c], Bm);
            }
            sv[k * 4 + j] = A * Bm;
        }
}

// log-likelihood of one pattern at a branch: p = P(t) x on one side, y the other side, n the scale count of the pair.  The site
// likelihood is the mixture wk l + p_inv inv with l = sum_k sum_c pi_c p[k][c] y[k][c]; with n > 0 the 2^(256 n) scaling is undone
// (exact: wherever n = 0 the arithmetic is the unscaled one)
__device__ __forceinline__ double site_loglik(const double* mdl, const double (&p)[16], const double (&y)[16], int n, double wk, double pinv, double inv) {
    double l = 0.0;
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int c = 0; c < 4; ++c) l = fma(mdl[MDL_FREQ + c] * p[k * 4 + c], y[k * 4 + c], l);
    if (n == 0) return log(wk * l + pinv * inv);
    if (pinv * inv == 0.0) return log(wk * l) - n * SCALE_LN;
    return log(ldexp(wk * l, -SCALE_EXP * n) + pinv * inv);
}

// safeguarded Newton-Raphson on one branch from tv, over the sumtable St [L][16] and its scale counts Snt [L] (the block's own
// patterns s = tid, tid + LLH_THREADS, ...); ek: 48 doubles of shared scratch, red: block_sum2's.  Every thread returns the new length.
__device__ __forceinline__ double newton_brlen(const double* St, const int32_t* Snt, const double* mdl, double* ek, double* red, const double* wts,
                                               const double* invt, double pinv, double wk, int L, double tv) {
    const int tid = threadIdx.x;
    double lo = BRLEN_MIN, hi = BRLEN_MAX;
    for (int it = 0; it < 32; ++it) {
        if (tid < 16) {
            const double rate = mdl[MDL_LAM + (tid & 3)] * mdl[MDL_RATE + (tid >> 2)];
            ek[tid] = exp(rate * tv); ek[16 + tid] = rate; ek[32 + tid] = rate * rate;
        }
        __syncthreads();
        double f1 = 0.0, f2 = 0.0;
        for (int s = tid; s < L; s += LLH_THREADS) {
            double sv[16];
            vec_load(St + (size_t)s * 16, sv);
            double l0 = 0.0, l1 = 0.0, l2 = 0.0;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const double se = sv[i] * ek[i];
                l0 += se; l1 = fma(se, ek[16 + i], l1); l2 = fma(se, ek[32 + i], l2);
            }
            // a scaled pattern: its invariant term scaled up to match (inf where that overflows: then g = 0, and no 0 * inf)
            const int n = Snt[s];
            const double L0 = n == 0 ? wk * l0 + pinv * invt[s] : wk * l0 + (invt[s] > 0.0 ? ldexp(pinv * invt[s], SCALE_EXP * n) : 0.0);
            const double g = wk * l1 / L0;
            f1 = fma(wts[s], g, f1);
            f2 = fma(wts[s], wk * l2 / L0 - g * g, f2);
        }
        block_sum2(f1, f2, red);
        if (f1 > 0.0) lo = tv; else hi = tv;
        double tn = f2 < 0.0 ? tv - f1 / f2 : (f1 > 0.0 ? tv * 4.0 : tv * 0.25);
        if (!(tn > lo && tn < hi)) tn = 0.5 * (lo + hi);
        const bool done = fabs(tn - tv) < 1e-9 + 1e-7 * tv;
        tv = tn;
        if (done) break;
    }
    return tv;
}

// RELL replicate counts, shared by branch support (nnj_llh_nni.cu) and the topology test (nnj_llh_topo.cu).  cum [B][L+1] holds each
// tree's cumulative pattern weights, n_b = cum[L] its site count.  Replicate rep0 + r makes `draws` draws (0: n_b of its tree); draw i
// is the site u = (x0 * n_b) >> 32, x0 = word 0 of Philox4x32-10 with counter (i, r lo, r hi, w3) and key (seed lo, seed hi), and
// cnt[b][p][r] += 1 for the pattern p with cum[p] <= u < cum[p + 1].  Grid: x over draws, y over (tree, replicate).
constexpr int RELL_THREADS = 256;
static __global__ void __launch_bounds__(RELL_THREADS) k_rell_counts(const uint32_t* __restrict__ cum, int B, int L, uint64_t seed, int64_t rep0, int nr,
                                                                     uint32_t draws, uint32_t w3, int32_t* __restrict__ cnt) {
    const uint32_t i = blockIdx.x * RELL_THREADS + threadIdx.x;
    for (int y = blockIdx.y; y < B * nr; y += gridDim.y) {
        const int b = y / nr, rl = y - b * nr;
        const uint32_t* cb = cum + (size_t)b * (L + 1);
        const uint32_t n = cb[L];
        if (i >= (draws ? draws : n)) continue;
        const uint64_t r = (uint64_t)rep0 + (uint64_t)rl;
        const uint32_t x0 = philox_x0(i, (uint32_t)r, (uint32_t)(r >> 32), w3, (uint32_t)seed, (uint32_t)(seed >> 32));
        const uint32_t u = (uint32_t)(((uint64_t)x0 * (uint64_t)n) >> 32);
        int lo = 0, hi = L;                                   // cb[lo] <= u < cb[hi]
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(cb + mid) <= u) lo = mid; else hi = mid;
        }
        atomicAdd(cnt + ((size_t)b * L + lo) * nr + rl, 1);
    }
}

}  // namespace nnj
