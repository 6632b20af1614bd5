// Bootstrap branch support (FBP / TBE) of NJ trees: column resampling of one alignment and transfer distances of reference splits
// to replicate trees given as merge lists.  DESIGN.md section 11 gives the definitions; oracle/support_oracle.py restates both
// kernels in numpy / Python and the GPU tests hold them to bit-identical results.
//
// k_boot_columns: replicate r of an alignment with l_eff real columns (the prefix; padded columns form the suffix) takes, for
// output column c < l_eff, input column (x0 * l_eff) >> 32 where x0 is word 0 of Philox4x32-10 with counter (c, r_lo, r_hi, 0)
// and key (seed_lo, seed_hi).  Columns c >= l_eff are copied unchanged.  A replicate depends only on (seed, r, l_eff), so the
// chunking of replicates over calls or ranks cannot change a result.
//
// k_split_dist: one CTA per replicate tree.  Warp 0 replays the merge list (slot i <- new node, slot j removed) into the R-1 clade
// bitsets of the tree, indexed by join, in shared memory; then one warp per reference split A computes
//     delta = min(p - 1, min over the tree's non-root clades c of min(|A ^ c|, R - |A ^ c|)),   p = size of A's lighter side,
// lanes over clades, popcount of the XOR, warp minimum.  R <= 512 keeps a split in 8 words of registers per lane.
#include <cuda_runtime.h>

#include <cstdint>

#include "nnj_common.cuh"
#include "nnj_internal.h"

namespace nnj {

namespace {

constexpr int BOOT_THREADS = 256;
constexpr int SPLIT_THREADS = 256;
constexpr int SPLIT_MAX_WORDS = 8;                   // R <= 512
constexpr int SPLIT_MAX_TAXA = 64 * SPLIT_MAX_WORDS;

// out[b][t][c] (4-byte one-hot words) = data[t][src(rep0 + b, c)][:]; one thread per (replicate, column), writes coalesced along c
__global__ void __launch_bounds__(BOOT_THREADS) k_boot_columns(const uint32_t* __restrict__ data, int R, int L, int l_eff, uint64_t seed,
                                                              int64_t rep0, int B, uint32_t* __restrict__ out) {
    const int c = blockIdx.x * BOOT_THREADS + threadIdx.x;
    if (c >= L) return;
    for (int b = blockIdx.y; b < B; b += gridDim.y) {
        const uint64_t r = (uint64_t)rep0 + (uint64_t)b;
        int src = c;
        if (c < l_eff) {
            const uint32_t x0 = philox_x0((uint32_t)c, (uint32_t)r, (uint32_t)(r >> 32), 0u, (uint32_t)seed, (uint32_t)(seed >> 32));
            src = (int)(((uint64_t)x0 * (uint64_t)l_eff) >> 32);
        }
        uint32_t* dst = out + (size_t)b * R * L + c;
        for (int t = 0; t < R; ++t) dst[(size_t)t * L] = __ldg(data + (size_t)t * L + src);
    }
}

// dist[b][s]: transfer distance of reference split s to tree b; the whole row is -1 when the merge list of b is not valid
__global__ void __launch_bounds__(SPLIT_THREADS) k_split_dist(const int32_t* __restrict__ merges, int R, const uint64_t* __restrict__ splits,
                                                             int S, int32_t* __restrict__ dist) {
    extern __shared__ unsigned long long smem_u64[];
    const int W = (R + 63) >> 6;
    uint64_t* clade = reinterpret_cast<uint64_t*>(smem_u64);          // [R-1][W], join k = node R + k
    int* slot = reinterpret_cast<int*>(clade + (size_t)(R - 1) * W);  // [R] live node of each slot
    __shared__ int s_bad;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int32_t* mg = merges + (size_t)b * (R - 1) * 2;

    if (warp == 0) {
        for (int s = lane; s < R; s += 32) slot[s] = s;
        int bad = 0;
        __syncwarp();
        for (int t = 0; t < R - 1; ++t) {
            const int n = R - t;
            const int i = mg[2 * t], j = mg[2 * t + 1];
            if (!(0 <= i && i < j && j < n)) { bad = 1; break; }
            const int a = slot[i], c = slot[j];
            __syncwarp();                  // every lane has read the two slots before any lane rewrites them
            for (int w = lane; w < W; w += 32) {
                const uint64_t va = a < R ? ((a >> 6) == w ? 1ull << (a & 63) : 0ull) : clade[(size_t)(a - R) * W + w];
                const uint64_t vc = c < R ? ((c >> 6) == w ? 1ull << (c & 63) : 0ull) : clade[(size_t)(c - R) * W + w];
                clade[(size_t)t * W + w] = va | vc;
            }
            // slot j removed: slots j+1 .. n-1 move down one, 32 at a time (each chunk reads before it writes)
            for (int s0 = j; s0 < n - 1; s0 += 32) {
                const int s = s0 + lane;
                const int v = s < n - 1 ? slot[s + 1] : 0;
                __syncwarp();
                if (s < n - 1) slot[s] = v;
                __syncwarp();
            }
            if (lane == 0) slot[i] = R + t;
            __syncwarp();
        }
        if (lane == 0) s_bad = bad;
    }
    __syncthreads();
    int32_t* row = dist + (size_t)b * S;
    if (s_bad) {
        for (int s = tid; s < S; s += SPLIT_THREADS) row[s] = -1;
        return;
    }
    const uint64_t last = (R & 63) ? (1ull << (R & 63)) - 1ull : ~0ull;   // bits of the last word that are taxa
    const int n_clades = R - 2;                                          // join R-2 is the root: all leaves, never closer than p
    for (int s = warp; s < S; s += SPLIT_THREADS / 32) {
        uint64_t A[SPLIT_MAX_WORDS];
        int pa = 0;
#pragma unroll
        for (int w = 0; w < SPLIT_MAX_WORDS; ++w) {
            A[w] = w < W ? splits[(size_t)s * W + w] & (w == W - 1 ? last : ~0ull) : 0ull;
            pa += __popcll(A[w]);
        }
        const int p = min(pa, R - pa);
        int best = max(p - 1, 0);
        for (int k = lane; k < n_clades; k += 32) {
            const uint64_t* ck = clade + (size_t)k * W;
            int d = 0;
#pragma unroll
            for (int w = 0; w < SPLIT_MAX_WORDS; ++w)
                if (w < W) d += __popcll(A[w] ^ ck[w]);
            best = min(best, min(d, R - d));
        }
        best = __reduce_min_sync(0xffffffffu, best);
        if (lane == 0) row[s] = best;
    }
}

size_t split_smem_bytes(int R) { return (size_t)(R - 1) * ((R + 63) / 64) * sizeof(uint64_t) + (size_t)R * sizeof(int); }

DevOnce g_split_smem_once;

}  // namespace

int run_bootstrap_columns(const int8_t* data, int R, int L, int l_eff, uint64_t seed, int64_t rep0, int B, int8_t* out, cudaStream_t st) {
    const dim3 grid((L + BOOT_THREADS - 1) / BOOT_THREADS, B < 65535 ? B : 65535);
    prof_begin(KC_MISC, st);
    k_boot_columns<<<grid, BOOT_THREADS, 0, st>>>(reinterpret_cast<const uint32_t*>(data), R, L, l_eff, seed, rep0, B,
                                                  reinterpret_cast<uint32_t*>(out));
    ++g_launches; prof_end(st);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    return NNJ_OK;
}

int run_split_distances(const int32_t* merges, int B, int R, const uint64_t* splits, int S, int32_t* dist, cudaStream_t st) {
    if (R < 4 || R > SPLIT_MAX_TAXA) return set_error(NNJ_ERR_INVALID, "split_distances: 4 <= taxa <= 512");
    if (S == 0) return NNJ_OK;
    if (g_split_smem_once.need()) {      // opt-in sized for the largest supported tree (idempotent per device)
        cudaError_t e = cudaFuncSetAttribute(k_split_dist, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)split_smem_bytes(SPLIT_MAX_TAXA));
        if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
        g_split_smem_once.done();
    }
    prof_begin(KC_MISC, st);
    k_split_dist<<<B, SPLIT_THREADS, split_smem_bytes(R), st>>>(merges, R, splits, S, dist);
    ++g_launches; prof_end(st);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    return NNJ_OK;
}

}  // namespace nnj
