// Balanced-ELU margin ranking loss of the reference's pre-training step (train.py:448-545), evaluated on the device over the
// logits trace a teacher-forced rollout leaves behind (nnj_rollout with NNJ_SELECT_FORCED).  SURVEY.md section 8 row f3, the
// forward half: the backward pass and the optimiser stay with the reference (DESIGN.md section 8).
//
// Per step t (n = R - t live nodes, P = n(n-1)/2 candidate pairs) and tree b the reference forms
//     S = scores of the pairs in the step's action set (the label tree's cherries among the live nodes)
//     U = scores of the other pairs, the K largest of them kept, K = min(W, max(int(W * ratio), 8)),  W = widest complement of the batch
//     loss_t = sum_b sum_{s in S} sum_{u in top-K(U)} elu(-(s - margin - u)) / sum_b |S| * |top-K(U)|
// and the step's "precision" counts s > u over the same pairs; the loss is the mean of loss_t over the R-2 steps that have more than
// one candidate.  One CTA per (step, tree): the step's scores are split into S and U in shared memory in pair order, U is sorted by a
// bitonic network, and the |S| x K terms are summed in a fixed order (thread-strided partial sums in fp64, then a tree) so the result
// does not depend on the launch.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>

#include "nnj_common.cuh"
#include "nnj_internal.h"

namespace nnj {

namespace {

constexpr int RL_THREADS = 256;

__host__ __device__ inline size_t trace_offset(int R, int t) {     // sum_{s<t} (R-s)(R-s-1)/2
    size_t o = 0;
    for (int s = 0; s < t; ++s) o += (size_t)(R - s) * (R - s - 1) / 2;
    return o;
}

// set_count[b][t] = |S|;  widest[t] = max_b (P - |S|): the width the reference pads every tree's complement to (utils.py:198-209)
__global__ void __launch_bounds__(RL_THREADS) k_rank_count(const uint8_t* __restrict__ in_set, size_t trace_stride, int R, int T,
                                                           int32_t* __restrict__ set_count, int32_t* __restrict__ widest) {
    __shared__ int s_cnt[RL_THREADS];
    const int t = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
    const int n = R - t, P = n * (n - 1) / 2;
    const uint8_t* f = in_set + (size_t)b * trace_stride + trace_offset(R, t);
    int c = 0;
    for (int p = tid; p < P; p += RL_THREADS) c += f[p] != 0;
    s_cnt[tid] = c;
    __syncthreads();
    for (int o = RL_THREADS / 2; o > 0; o >>= 1) {
        if (tid < o) s_cnt[tid] += s_cnt[tid + o];
        __syncthreads();
    }
    if (tid == 0) {
        set_count[(size_t)b * T + t] = s_cnt[0];
        atomicMax(&widest[t], P - s_cnt[0]);          // a maximum: independent of the order of arrival
    }
}

// part[b][t] = { sum of elu terms, number of (s, u) pairs, number of pairs with s > u }
__global__ void __launch_bounds__(RL_THREADS) k_rank_loss(const float* __restrict__ logits, const uint8_t* __restrict__ in_set, size_t trace_stride,
                                                          int R, int T, float margin, double ratio, const int32_t* __restrict__ set_count,
                                                          const int32_t* __restrict__ widest, double* __restrict__ part, int u_cap) {
    extern __shared__ float sm[];
    float* u = sm;                    // [u_cap] complement scores, sorted descending
    float* sv = sm + u_cap;           // [R] action-set scores in pair order
    __shared__ int s_scan[RL_THREADS + 1];
    __shared__ double s_acc[RL_THREADS];
    __shared__ double s_prec[RL_THREADS];
    const int t = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
    const int n = R - t, P = n * (n - 1) / 2;
    const size_t off = (size_t)b * trace_stride + trace_offset(R, t);
    const float* lg = logits + off;
    const uint8_t* f = in_set + off;

    const int W = widest[t];
    const int K = min(W, max((int)((double)W * ratio), 8));
    const int ns = set_count[(size_t)b * T + t];
    const int U = P - ns;

    // ordered split: thread i owns the contiguous pair range [i*chunk, (i+1)*chunk)
    const int chunk = (P + RL_THREADS - 1) / RL_THREADS;
    const int p0 = min(tid * chunk, P), p1 = min(p0 + chunk, P);
    int c = 0;
    for (int p = p0; p < p1; ++p) c += f[p] != 0;
    __syncthreads();
    s_scan[tid + 1] = c;
    if (tid == 0) s_scan[0] = 0;
    __syncthreads();
    if (tid == 0) for (int i = 1; i <= RL_THREADS; ++i) s_scan[i] += s_scan[i - 1];
    __syncthreads();
    int is = s_scan[tid], iu = p0 - is;
    for (int p = p0; p < p1; ++p) {
        const float v = lg[p];
        if (f[p]) { if (is < R) sv[is] = v; ++is; }
        else u[iu++] = v;
    }
    int cap = 1;
    while (cap < U) cap <<= 1;
    for (int k = U + tid; k < cap; k += RL_THREADS) u[k] = -INFINITY;
    __syncthreads();
    // bitonic sort of u[0, cap), descending
    for (int size = 2; size <= cap; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int k = tid; k < cap / 2; k += RL_THREADS) {
                const int lo = 2 * k - (k & (stride - 1));
                const int hi = lo + stride;
                const bool desc = ((lo & size) == 0);
                const float a = u[lo], c2 = u[hi];
                if (desc ? (a < c2) : (a > c2)) { u[lo] = c2; u[hi] = a; }
            }
            __syncthreads();
        }
    }
    const int Kv = min(K, U);          // padded entries of the reference's top-K are masked out again (train.py:500-507)
    double acc = 0.0, prec = 0.0;
    const bool too_many = ns > R;      // an action set larger than the node count is not a set of cherries: poison the result
    const int total = too_many ? 0 : ns * Kv;
    for (int idx = tid; idx < total; idx += RL_THREADS) {
        const int s = idx / Kv, k = idx - s * Kv;
        const float d = (sv[s] - margin) - u[k];          // scores_diff, train.py:504
        const float x = -d;
        acc += (double)(x > 0.f ? x : expm1f(x));          // F.elu
        prec += (sv[s] > u[k]) ? 1.0 : 0.0;
    }
    s_acc[tid] = acc; s_prec[tid] = prec;
    __syncthreads();
    for (int o = RL_THREADS / 2; o > 0; o >>= 1) {
        if (tid < o) { s_acc[tid] += s_acc[tid + o]; s_prec[tid] += s_prec[tid + o]; }
        __syncthreads();
    }
    if (tid == 0) {
        double* o = part + ((size_t)b * T + t) * 3;
        o[0] = too_many ? NAN : s_acc[0];
        o[1] = (double)ns * (double)Kv;
        o[2] = s_prec[0];
    }
}

// out[0] = loss (mean over steps of sum_b terms / sum_b pairs), out[1] = precision, out[2 + t] = loss of step t
__global__ void __launch_bounds__(RL_THREADS) k_rank_final(const double* __restrict__ part, int B, int T, float* __restrict__ out) {
    __shared__ double s_loss[RL_THREADS], s_cnt[RL_THREADS], s_prec[RL_THREADS];
    const int tid = threadIdx.x;
    double lsum = 0.0, csum = 0.0, psum = 0.0;
    for (int t = tid; t < T; t += RL_THREADS) {
        double a = 0.0, c = 0.0, p = 0.0;
        for (int b = 0; b < B; ++b) {
            const double* o = part + ((size_t)b * T + t) * 3;
            a += o[0]; c += o[1]; p += o[2];
        }
        const double lt = a / c;
        out[2 + t] = (float)lt;
        lsum += lt; csum += c; psum += p;
    }
    s_loss[tid] = lsum; s_cnt[tid] = csum; s_prec[tid] = psum;
    __syncthreads();
    for (int o = RL_THREADS / 2; o > 0; o >>= 1) {
        if (tid < o) { s_loss[tid] += s_loss[tid + o]; s_cnt[tid] += s_cnt[tid + o]; s_prec[tid] += s_prec[tid + o]; }
        __syncthreads();
    }
    if (tid == 0) { out[0] = (float)(s_loss[0] / T); out[1] = (float)(s_prec[0] / s_cnt[0]); }
}

struct RankLossBuffers { int32_t* set_count; double* part; int32_t* widest; size_t total; };
RankLossBuffers rank_loss_layout(char* base, int B, int R) {
    const size_t T = (size_t)R - 2;
    WsCarver c(base);
    RankLossBuffers w;
    w.set_count = c.take<int32_t>((size_t)B * T);
    w.part = c.take<double>((size_t)B * T * 3);
    w.widest = c.take<int32_t>(T);
    w.total = c.off + 256;
    return w;
}

}  // namespace

size_t rank_loss_ws_bytes(int B, int R) { return rank_loss_layout(nullptr, B, R).total; }

int run_rank_loss(const float* logits_trace, const uint8_t* in_set, int B, int R, float margin, double ratio, float* out, void* ws, size_t ws_bytes,
                  cudaStream_t st) {
    if (R < 3 || R > 256) return set_error(NNJ_ERR_INVALID, "rank_loss: 3 <= taxa <= 256");
    if (B < 1 || B > 65535) return set_error(NNJ_ERR_INVALID, "rank_loss: 1 <= trees <= 65535 per call");
    if (!(ratio > 0.0) || !(ratio <= 1.0)) return set_error(NNJ_ERR_INVALID, "rank_loss: ratio must be in (0, 1]");
    if (ws_bytes < rank_loss_ws_bytes(B, R)) return set_error(NNJ_ERR_WORKSPACE, "rank_loss: workspace too small (nnj_rank_loss_workspace_bytes)");
    const int T = R - 2;
    const RankLossBuffers w = rank_loss_layout(ws_align(ws), B, R);
    int32_t *set_count = w.set_count, *widest = w.widest;
    double* part = w.part;
    {
        cudaError_t e = cudaMemsetAsync(widest, 0, (size_t)T * sizeof(int32_t), st);
        if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    }
    const size_t trace_stride = trace_offset(R, R - 1);
    int u_cap = 1;
    while (u_cap < R * (R - 1) / 2) u_cap <<= 1;
    const size_t smem = ((size_t)u_cap + R) * sizeof(float);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(k_rank_loss, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    }
    const dim3 grid(T, B);
    prof_begin(KC_MISC, st);
    k_rank_count<<<grid, RL_THREADS, 0, st>>>(in_set, trace_stride, R, T, set_count, widest);
    ++g_launches; prof_end(st);
    prof_begin(KC_MISC, st);
    k_rank_loss<<<grid, RL_THREADS, smem, st>>>(logits_trace, in_set, trace_stride, R, T, margin, ratio, set_count, widest, part, u_cap);
    ++g_launches; prof_end(st);
    prof_begin(KC_MISC, st);
    k_rank_final<<<1, RL_THREADS, 0, st>>>(part, B, T, out);
    ++g_launches; prof_end(st);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    return NNJ_OK;
}

}  // namespace nnj
