// nnj_llh_topo.cu — tree topology tests over K candidate trees of one alignment: RELL bootstrap proportions, KH, SH, expected likelihood
// weights and the multiscale winner counts of the AU test (IQ-TREE -z trees -zb N -au, CONSEL).  DESIGN.md section 13 gives the
// definitions; oracle/topotest_oracle.py restates them in numpy.
//
// 1. llh_prepare (nnj_llh.cu) over the K trees, the alignment broadcast to each: per-pattern log-likelihoods l[k][p] at the given
//    lengths and models.  k_topo_llh: L_k = sum_p w[p] l[k][p].
// 2. Per scale s = 0..9 (n_s = floor((5 + s) / 10 * n + 0.5) draws per replicate, Philox counter word 3 = s + 1), in chunks of
//    replicates: k_rell_counts (nnj_llh.cuh) -> counts c[p][j]; k_topo_totals -> T[j][k] = sum_p c[p][j] l[k][p]; k_topo_stats ->
//    winner counts, and at scale 5 the ELW terms q[j][k]; k_topo_sums (scale 5) -> running sums over j of T and q, per tree in j order.
// 3. Scale 5 again, the counts and totals regenerated, now against the means: KH and SH counts.
// Every sum has a fixed order and every count is an integer: results are bit-reproducible and do not depend on the chunk size.
#include "nnj_internal.h"
#include "nnj_llh.cuh"

namespace nnj {

namespace {

constexpr int TOPO_SCALES = 10, TOPO_REF = 5;       // scales r_s = (5 + s) / 10; s = 5 is r = 1
constexpr int TOPO_CHUNK = 4096;                    // replicates per pass (counts [L][chunk] int32, T and q [chunk][K] fp64 in the workspace)
constexpr int TOT_TILE = 64, TOT_PB = 16, TOT_THREADS = 256;   // k_topo_totals: 64 replicates x 64 trees per CTA, 16 patterns per staged block
constexpr int STATS_THREADS = 256, STATS_REPS = 64;  // k_topo_stats: one warp per replicate, 64 replicates per CTA

// the alignment once per tree: llh_prepare reads tips [B][R][L] and weights [B][L]
__global__ void k_topo_broadcast(const uint8_t* __restrict__ tips, const double* __restrict__ w, int K, size_t RL, int L, uint8_t* __restrict__ tips_k,
                                 double* __restrict__ w_k) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)K * RL; i += stride) tips_k[i] = tips[i % RL];
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)K * L; i += stride) w_k[i] = w[i % L];
}

// one thread per tree: L_k = sum_p w[p] l[k][p] in pattern order, each product rounded, then each add
__global__ void k_topo_llh(const double* __restrict__ site, const double* __restrict__ w, int K, int P, double* __restrict__ llh) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    const double* l = site + (size_t)k * P;
    double acc = 0.0;
    for (int p = 0; p < P; ++p) acc = __dadd_rn(acc, __dmul_rn(w[p], l[p]));
    llh[k] = acc;
}

// T[j][k] = sum_p c[p][j] l[k][p] for a 64 x 64 tile of (replicate, tree); thread (tx, ty) holds replicates ty + 16 a and trees tx + 16 b.
// Blocks of 16 patterns of both operands are staged in shared memory (the counts converted to double once there; patterns past P and
// rows past nr / K read as 0, whose products add exactly nothing).  Every output is one sequential sum in pattern order, a rounded multiply
// then a rounded add: the tile decides which thread holds a sum, never the order of its terms.  fp64 CUDA cores: an FMA, or an fp64
// mma, would round once per term and break the bitwise agreement of the integer counts with their CPU restatement.
__global__ void __launch_bounds__(TOT_THREADS) k_topo_totals(const int32_t* __restrict__ cnt, const double* __restrict__ site, int K, int P, int nr,
                                                             double* __restrict__ T) {
    __shared__ double cs[TOT_PB][TOT_TILE];
    __shared__ double ls[TOT_PB][TOT_TILE + 1];      // +1: the transposing stores of a warp spread over the banks
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int k0 = blockIdx.x * TOT_TILE, j0 = blockIdx.y * TOT_TILE;
    double acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
    for (int p0 = 0; p0 < P; p0 += TOT_PB) {
#pragma unroll
        for (int e = tid; e < TOT_PB * TOT_TILE; e += TOT_THREADS) {
            const int pc = e / TOT_TILE, jj = e % TOT_TILE;        // counts: a warp reads consecutive replicates of one pattern
            const int p = p0 + pc, j = j0 + jj;
            cs[pc][jj] = (p < P && j < nr) ? (double)__ldg(cnt + (size_t)p * nr + j) : 0.0;
            const int kk = e / TOT_PB, pl = e % TOT_PB;            // l: a warp reads 16 consecutive patterns of two trees
            const int k = k0 + kk, q = p0 + pl;
            ls[pl][kk] = (k < K && q < P) ? __ldg(site + (size_t)k * P + q) : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int pp = 0; pp < TOT_PB; ++pp) {
            double c[4], l[4];
#pragma unroll
            for (int a = 0; a < 4; ++a) { c[a] = cs[pp][ty + 16 * a]; l[a] = ls[pp][tx + 16 * a]; }
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) acc[a][b] = __dadd_rn(acc[a][b], __dmul_rn(c[a], l[b]));
        }
        __syncthreads();
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int j = j0 + ty + 16 * a;
        if (j >= nr) continue;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int k = k0 + tx + 16 * b;
            if (k < K) T[(size_t)j * K + k] = acc[a][b];
        }
    }
}

__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

struct StatsArgs {
    const double* T;                 // [nr][K] totals of the chunk
    int K, nr;
    int pass;                        // 1: winners (and at scale 5 the ELW terms), 2: KH and SH (scale 5)
    double* q;                       // [nr][K] ELW terms q[j][k] (pass 1 at scale 5), else null
    const double *tsum, *llh;        // pass 2: sum_j T[j][k] over all N replicates of scale 5, L_k
    int kstar; double n_boot;
    int32_t *out0, *out1;            // pass 1: win[s] [K]; pass 2: kh [K], sh [K]
};

// one warp per replicate of the chunk; integer counts gathered per CTA in shared memory, then one atomic per tree and CTA
__global__ void __launch_bounds__(STATS_THREADS) k_topo_stats(const StatsArgs a) {
    extern __shared__ int32_t cntr[];                      // [2][K]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, K = a.K;
    for (int k = tid; k < 2 * K; k += STATS_THREADS) cntr[k] = 0;
    __syncthreads();
    for (int jl = warp; jl < STATS_REPS; jl += STATS_THREADS / 32) {
        const int j = blockIdx.x * STATS_REPS + jl;
        if (j >= a.nr) break;
        const double* t = a.T + (size_t)j * K;
        if (a.pass == 1) {
            double mx = -INFINITY;
            for (int k = lane; k < K; k += 32) mx = fmax(mx, t[k]);
            mx = warp_max(mx);
            for (int k = lane; k < K; k += 32)
                if (t[k] >= mx) atomicAdd(cntr + k, 1);    // every tied tree wins
            if (a.q) {
                // q_k = e_k / sum_k' e_k', e_k = exp(T[j][k] - max), the sum in k order
                double* q = a.q + (size_t)j * K;
                for (int k = lane; k < K; k += 32) q[k] = exp(t[k] - mx);
                __syncwarp();
                double s = 0.0;
                if (lane == 0)
                    for (int k = 0; k < K; ++k) s = __dadd_rn(s, q[k]);
                s = __shfl_sync(0xffffffffu, s, 0);
                for (int k = lane; k < K; k += 32) q[k] = q[k] / s;
            }
        } else {
            // centred values a_k = T[j][k] - m_k, m_k = tsum[k] / N; KH against k*, SH against the largest centred value
            const double as = t[a.kstar] - a.tsum[a.kstar] / a.n_boot, ls = a.llh[a.kstar];
            double amax = -INFINITY;
            for (int k = lane; k < K; k += 32) amax = fmax(amax, t[k] - a.tsum[k] / a.n_boot);
            amax = warp_max(amax);
            for (int k = lane; k < K; k += 32) {
                const double ak = t[k] - a.tsum[k] / a.n_boot, d = ls - a.llh[k];
                if (as - ak >= d) atomicAdd(cntr + k, 1);
                if (amax - ak >= d) atomicAdd(cntr + K + k, 1);
            }
        }
    }
    __syncthreads();
    for (int k = tid; k < K; k += STATS_THREADS) {
        if (cntr[k]) atomicAdd(a.out0 + k, cntr[k]);
        if (a.pass == 2 && cntr[K + k]) atomicAdd(a.out1 + k, cntr[K + k]);
    }
}

// one thread per tree: the chunk's T[j][k] and q[j][k] added in j order to the running sums of scale 5
__global__ void k_topo_sums(const double* __restrict__ T, const double* __restrict__ q, int K, int nr, double* __restrict__ tsum, double* __restrict__ qsum) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    double st = tsum[k], sq = qsum[k];
#pragma unroll 16
    for (int j = 0; j < nr; ++j) {                         // unrolled: the loads of 16 rows are in flight ahead of the adds
        st = __dadd_rn(st, T[(size_t)j * K + k]);
        sq = __dadd_rn(sq, q[(size_t)j * K + k]);
    }
    tsum[k] = st;
    qsum[k] = sq;
}

struct TopoBuffers {
    uint8_t* tips; double* w;           // the alignment once per tree
    double* site;                       // l [K][L] when the caller passes no site_dev
    double *llh, *tsum, *qsum;          // [K]
    uint32_t* cum;                      // [L + 1]
    int32_t* cnt;                       // [L][chunk]
    double *T, *q;                      // [chunk][K]
    int32_t *win, *kh, *sh;             // [10][K], [K], [K]
    size_t total;
};
static int topo_chunk(int n_boot) { return n_boot < TOPO_CHUNK ? n_boot : TOPO_CHUNK; }
static TopoBuffers topo_layout(char* base, int K, int R, int L, int n_boot) {
    const size_t chunk = (size_t)topo_chunk(n_boot);
    WsCarver c(base);
    TopoBuffers w;
    w.tips = c.take<uint8_t>((size_t)K * R * L); w.w = c.take<double>((size_t)K * L); w.site = c.take<double>((size_t)K * L);
    w.llh = c.take<double>(K); w.tsum = c.take<double>(K); w.qsum = c.take<double>(K);
    w.cum = c.take<uint32_t>((size_t)L + 1); w.cnt = c.take<int32_t>((size_t)L * chunk);
    w.T = c.take<double>(chunk * K); w.q = c.take<double>(chunk * K);
    w.win = c.take<int32_t>((size_t)TOPO_SCALES * K); w.kh = c.take<int32_t>(K); w.sh = c.take<int32_t>(K);
    w.total = c.off + 256;
    return w;
}

// n_s = floor(r_s n + 0.5), r_s = (5 + s) / 10 in fp64; at least 1 for n >= 1
static uint32_t topo_scale_draws(uint32_t n, int s) {
    volatile double x = (double)(5 + s) / 10.0 * (double)n;     // volatile: the product is rounded on its own, as the oracle rounds it
    return (uint32_t)floor(x + 0.5);
}

}  // namespace

size_t llh_topo_ws_bytes(int K, int R, int L, int n_boot) { return llh_ws_bytes(K, R, L) + topo_layout(nullptr, K, R, L, n_boot).total; }

int run_llh_topo(const uint8_t* tips, const double* weights, const int32_t* children_h, const double* brlen_h, const double* model_h, int K, int R,
                 int L, uint64_t seed, int n_boot, double* llh_h, int32_t* win_h, int32_t* kh_h, int32_t* sh_h, double* elw_h, double* site_dev,
                 void* ws, size_t ws_bytes, cudaStream_t st) {
    const size_t base = llh_ws_bytes(K, R, L);
    if (ws_bytes < base + topo_layout(nullptr, K, R, L, n_boot).total)
        return set_error(NNJ_ERR_WORKSPACE, "llh_topology_test: workspace too small (nnj_llh_topotest_workspace_bytes)");
    for (int k = 0; k < K; ++k)
        if (llh_check_tree(children_h + (size_t)k * (R - 1) * 2, R)) return set_error(NNJ_ERR_INVALID, "llh_topology_test: children is not a binary tree in join order");
    // ---- integral weights: a replicate draws sites, and a pattern of weight w is w sites
    std::vector<double> w(L);
    cudaError_t e = cudaMemcpyAsync(w.data(), weights, (size_t)L * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    std::vector<uint32_t> cum(L + 1, 0);
    uint64_t acc = 0;
    for (int p = 0; p < L; ++p) {
        if (!(w[p] >= 0.0 && w[p] <= 2147483647.0) || w[p] != floor(w[p])) return set_error(NNJ_ERR_INVALID, "llh_topology_test: pattern weights must be non-negative integers");
        acc += (uint64_t)w[p];
        if (acc > 2147483647ull) return set_error(NNJ_ERR_INVALID, "llh_topology_test: more than 2^31 - 1 sites");
        cum[p + 1] = (uint32_t)acc;
    }
    if (acc == 0) return set_error(NNJ_ERR_INVALID, "llh_topology_test: every pattern weight is 0");
    const uint32_t n = (uint32_t)acc;
    const TopoBuffers tw = topo_layout(ws_align(static_cast<char*>(ws) + base), K, R, L, n_boot);
    double* site = site_dev ? site_dev : tw.site;
    // ---- 1. per-pattern log-likelihoods of the K trees and L_k
    prof_begin(KC_LLH, st);
    k_topo_broadcast<<<2 * sm_count(), 256, 0, st>>>(tips, weights, K, (size_t)R * L, L, tw.tips, tw.w);
    LAUNCH_CHECK();
    std::vector<double> llh_tree(K), llh(K);
    const LlhTrees in{tw.tips, tw.w, children_h, const_cast<double*>(brlen_h), const_cast<double*>(model_h), K, R, L};
    const LlhPrepared pre = llh_prepare(in, site, llh_tree.data(), ws, base, st);
    if (pre.rc) return pre.rc;
    prof_begin(KC_LLH, st);
    k_topo_llh<<<(K + 127) / 128, 128, 0, st>>>(site, weights, K, L, tw.llh);
    LAUNCH_CHECK();
    e = cudaMemcpyAsync(llh.data(), tw.llh, (size_t)K * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(tw.cum, cum.data(), cum.size() * 4, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(tw.tsum, 0, (size_t)K * 8, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(tw.qsum, 0, (size_t)K * 8, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(tw.win, 0, (size_t)TOPO_SCALES * K * 4, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(tw.kh, 0, (size_t)K * 4, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(tw.sh, 0, (size_t)K * 4, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    int kstar = 0;                                         // the largest L_k, the lowest index on a tie
    for (int k = 1; k < K; ++k)
        if (llh[k] > llh[kstar]) kstar = k;
    // ---- 2. every scale, then 3. scale 5 again for KH and SH
    const int chunk = topo_chunk(n_boot);
    const size_t stats_smem = (size_t)2 * K * sizeof(int32_t);
    for (int step = 0; step <= TOPO_SCALES; ++step) {
        const int s = step < TOPO_SCALES ? step : TOPO_REF, pass = step < TOPO_SCALES ? 1 : 2;
        const uint32_t draws = topo_scale_draws(n, s);
        for (int j0 = 0; j0 < n_boot; j0 += chunk) {
            const int nr = n_boot - j0 < chunk ? n_boot - j0 : chunk;
            e = cudaMemsetAsync(tw.cnt, 0, (size_t)L * nr * 4, st);
            if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
            const dim3 grid((draws + RELL_THREADS - 1) / RELL_THREADS, nr < 65535 ? nr : 65535);
            prof_begin(KC_LLH, st);
            k_rell_counts<<<grid, RELL_THREADS, 0, st>>>(tw.cum, 1, L, seed, j0, nr, draws, (uint32_t)(s + 1), tw.cnt);
            LAUNCH_CHECK();
            prof_begin(KC_LLH, st);
            k_topo_totals<<<dim3((K + TOT_TILE - 1) / TOT_TILE, (nr + TOT_TILE - 1) / TOT_TILE), TOT_THREADS, 0, st>>>(tw.cnt, site, K, L, nr, tw.T);
            LAUNCH_CHECK();
            StatsArgs a;
            a.T = tw.T; a.K = K; a.nr = nr; a.pass = pass;
            a.q = (pass == 1 && s == TOPO_REF) ? tw.q : nullptr;
            a.tsum = tw.tsum; a.llh = tw.llh; a.kstar = kstar; a.n_boot = (double)n_boot;
            a.out0 = pass == 1 ? tw.win + (size_t)s * K : tw.kh; a.out1 = tw.sh;
            prof_begin(KC_LLH, st);
            k_topo_stats<<<(nr + STATS_REPS - 1) / STATS_REPS, STATS_THREADS, stats_smem, st>>>(a);
            LAUNCH_CHECK();
            if (a.q) {
                prof_begin(KC_LLH, st);
                k_topo_sums<<<(K + 127) / 128, 128, 0, st>>>(tw.T, tw.q, K, nr, tw.tsum, tw.qsum);
                LAUNCH_CHECK();
            }
        }
    }
    // ---- results
    std::vector<double> qsum(K);
    e = cudaMemcpyAsync(win_h, tw.win, (size_t)TOPO_SCALES * K * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(kh_h, tw.kh, (size_t)K * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(sh_h, tw.sh, (size_t)K * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(qsum.data(), tw.qsum, (size_t)K * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    for (int k = 0; k < K; ++k) {
        llh_h[k] = llh[k];
        elw_h[k] = qsum[k] / (double)n_boot;
    }
    return NNJ_OK;
}

}  // namespace nnj
