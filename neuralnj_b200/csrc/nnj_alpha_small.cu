// nnj_alpha_small.cu — pair blend + global-attention logits for the LATE steps of the NJ loop (<= 16 pairs, <= 16 live nodes).
//
// Same arithmetic as k_alpha_v3 (model.py:105-118):
//     z = sigmoid(Y_i - Y_j + b_h),   x = z x_i + (1 - z) x_j                         per listed pair and site
//     acc[pair, slot] += sum_d x[pair, site, d] K'[slot, site, d]                     summed over the sites of a 128-site group
// k_alpha_v3 is built around 128-row tcgen05 tiles and costs 430-530 us per launch of 128 trees however few pairs are alive
// (profiles/r02_ncu_launches); the contraction itself is tiny at this size (16 x 16 x 64 per site), the work is the blend.  Here a
// warp owns one site at a time: the site's node rows (X, Y fp32, K' bf16 hi / lo) arrive in a private buffer by cp.async, every
// thread blends exactly the elements of the 16 x 16 register-fragment A operand it holds (and writes them to the x planes the
// pair-score kernel reads), K' rows are the B fragments (4-byte loads), and the [pairs x slots] accumulator stays in the warp's
// registers across all its sites (3-term bf16 split, fp32 accumulate).  The warps' accumulators are summed in fixed order into the
// ONE partial of the site group (bit-reproducible), indexed by physical slot like k_alpha_v3's.
// CTA = (tree, 128-site group), 16 warps; T = 1 row tile of 16 pairs over 16 slots.
#include "nnj_internal.h"
#include "nnj_tc.cuh"

namespace nnj {

constexpr int AS_SITES = 128;

struct AlphaSmallArgs {
    const float* X; const float* Y; size_t tree_stride;          // fp32 node pools [B][S][C][64]
    const __nv_bfloat16* kph; const __nv_bfloat16* kpl; int S;   // K' planes [B][S][C][64]
    const int32_t* slot_of; int slot_stride;
    const int32_t* pair_i; const int32_t* pair_j; int pair_stride; int n0; int nc;
    int Rp, C;
    const float* bh;
    float* xf; int pc;                                            // x planes fp32 [B][pc][C][64]
    float* alpha_part; int alpha_pairs; int nSG; int RP;
};

template <int T, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, 1) k_alpha_small(const AlphaSmallArgs a) {
    constexpr int ROWS = 16 * T;
    constexpr int XB = ROWS * 256, KB = ROWS * 128;     // X / Y tile [slot][64 fp32] (16-byte chunk c at c ^ (slot & 7)); K' plane [slot][64 bf16] (same swizzle, 8 chunks)
    constexpr int BUF = 2 * XB + 2 * KB;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* sm = smem_align1024(smem_raw);
    float* s_bh = reinterpret_cast<float*>(sm);
    int* s_pi = reinterpret_cast<int*>(s_bh + 64);      // physical slots of the listed pairs (-1: none)
    int* s_pj = s_pi + 32;
    uint8_t* bufs = sm + 1024;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const int sg = blockIdx.x, b = blockIdx.y;
    const int c_base = sg * AS_SITES, n_sites = min(AS_SITES, a.C - c_base);
    if (tid < 64) s_bh[tid] = a.bh[tid];
    if (tid < 32) {
        int pi = -1, pj = -1;
        if (tid < a.nc) {
            const int li = a.pair_i[(size_t)b * a.pair_stride + a.n0 + tid], lj = a.pair_j[(size_t)b * a.pair_stride + a.n0 + tid];
            if (li >= 0) { pi = a.slot_of[(size_t)b * a.slot_stride + li]; pj = a.slot_of[(size_t)b * a.slot_stride + lj]; }
        }
        s_pi[tid] = pi; s_pj[tid] = pj;
    }
    // rows past the live slots are never loaded: K' rows there must read as zeros (they meet real x rows in the contraction)
    for (int i = tid; i < (WARPS * BUF) >> 4; i += WARPS * 32) reinterpret_cast<uint4*>(bufs)[i] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    // Per row of this thread: byte offset of its pair's two node rows in the X tile and the swizzle term of its channel chunks.  Channel
    // d = 16kk + 8e + 2t lives in 16-byte chunk 4kk + 2e + (t >> 1) (an even constant + one bit), stored at chunk ^ (slot & 7):
    // offset = slot * 256 + 8 (t & 1) + ((4kk + 2e) << 4 ^ u), u = ((t >> 1) ^ (slot & 7)) << 4  - one LOP and one add per load.
    int bi[T][2], bj[T][2], ui[T][2], uj[T][2];
#pragma unroll
    for (int m = 0; m < T; ++m)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int si = s_pi[16 * m + g + 8 * h], sj = s_pj[16 * m + g + 8 * h];
            bi[m][h] = si < 0 ? -1 : si * 256 + 8 * (t & 1); bj[m][h] = sj * 256 + 8 * (t & 1);
            ui[m][h] = ((t >> 1) ^ (si & 7)) << 4; uj[m][h] = ((t >> 1) ^ (sj & 7)) << 4;
        }

    uint8_t* mybuf = bufs + warp * BUF;
    const uint32_t mybuf_u = smem_u32(mybuf);
    const size_t tb = (size_t)b * a.tree_stride;
    float acc[T][2 * T][4];
#pragma unroll
    for (int m = 0; m < T; ++m)
#pragma unroll
        for (int j = 0; j < 2 * T; ++j) { acc[m][j][0] = 0.f; acc[m][j][1] = 0.f; acc[m][j][2] = 0.f; acc[m][j][3] = 0.f; }

    const int ld_slot0 = lane >> 4, ld_ch = lane & 15;
    const size_t ld_stride_x = (size_t)2 * a.C * 64, ld_stride_k = (size_t)4 * a.C * 64;
    for (int site = warp; site < n_sites; site += WARPS) {
        const int c = c_base + site;
        {   // X, Y rows of the live slots at this site: lane = (slot parity, 16-byte chunk), two slots per pass; pointers advance by constant strides
            const float* px = a.X + tb + ((size_t)ld_slot0 * a.C + c) * 64 + ld_ch * 4;
            const float* py = a.Y + tb + ((size_t)ld_slot0 * a.C + c) * 64 + ld_ch * 4;
            for (int slot = ld_slot0; slot < a.Rp; slot += 2, px += ld_stride_x, py += ld_stride_x) {
                const uint32_t off = mybuf_u + slot * 256 + ((ld_ch ^ (slot & 7)) << 4);
                cp_async16(off, px);
                cp_async16(off + XB, py);
            }
            // K' rows (hi, lo): lane = (slot mod 4, chunk), four slots per pass
            const __nv_bfloat16* ph = a.kph + (((size_t)b * a.S + (lane >> 3)) * a.C + c) * 64 + (lane & 7) * 8;
            const __nv_bfloat16* pl = a.kpl + (((size_t)b * a.S + (lane >> 3)) * a.C + c) * 64 + (lane & 7) * 8;
            for (int slot = lane >> 3; slot < a.Rp; slot += 4, ph += ld_stride_k, pl += ld_stride_k) {
                const uint32_t off = mybuf_u + 2 * XB + slot * 128 + (((lane & 7) ^ (slot & 7)) << 4);
                cp_async16(off, ph);
                cp_async16(off + KB, pl);
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncwarp();
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            uint32_t xh[T][4], xl[T][4];                 // x of this K step as A fragments: a0 [g][16kk+2t], a1 [g+8][same], a2 [g][16kk+8+2t], a3 [g+8][same]
#pragma unroll
            for (int m = 0; m < T; ++m)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int d = 16 * kk + 8 * e + 2 * t;
                    const float2 bh2 = *reinterpret_cast<const float2*>(s_bh + d);
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        float2 v = make_float2(0.f, 0.f);
                        if (bi[m][h] >= 0) {
                            const uint32_t oi = bi[m][h] + (((4 * kk + 2 * e) << 4) ^ ui[m][h]), oj = bj[m][h] + (((4 * kk + 2 * e) << 4) ^ uj[m][h]);
                            const float2 xi = *reinterpret_cast<const float2*>(mybuf + oi), xj = *reinterpret_cast<const float2*>(mybuf + oj);
                            const float2 yi = *reinterpret_cast<const float2*>(mybuf + XB + oi), yj = *reinterpret_cast<const float2*>(mybuf + XB + oj);
                            const float2 z = sigmoid_fast2(fadd2(fsub2(yi, yj), bh2));
                            v = ffma2(z, fsub2(xi, xj), xj);                        // z x_i + (1 - z) x_j, same operations as k_alpha_v3
                        }
                        split2(v.x, v.y, xh[m][2 * e + h], xl[m][2 * e + h]);
                        const int row = 16 * m + g + 8 * h;
                        if (row < a.nc) *reinterpret_cast<float2*>(a.xf + (((size_t)b * a.pc + row) * a.C + c) * 64 + d) = v;
                    }
                }
#pragma unroll
            for (int j = 0; j < 2 * T; ++j) {            // slots 8j .. 8j+7
                const uint8_t* kr = mybuf + 2 * XB + (8 * j + g) * 128 + 4 * t;
                const uint32_t kh0 = *reinterpret_cast<const uint32_t*>(kr + (((2 * kk) ^ g) << 4)), kh1 = *reinterpret_cast<const uint32_t*>(kr + (((2 * kk + 1) ^ g) << 4));
                const uint32_t kl0 = *reinterpret_cast<const uint32_t*>(kr + KB + (((2 * kk) ^ g) << 4)), kl1 = *reinterpret_cast<const uint32_t*>(kr + KB + (((2 * kk + 1) ^ g) << 4));
#pragma unroll
                for (int m = 0; m < T; ++m) {
                    mma_m16n8k16(acc[m][j], xl[m], kh0, kh1);      // small terms first
                    mma_m16n8k16(acc[m][j], xh[m], kl0, kl1);
                    mma_m16n8k16(acc[m][j], xh[m], kh0, kh1);
                }
            }
        }
        __syncwarp();                                    // all lanes done with the buffer before the next site's loads land in it
    }
    // ---- the site group's partial: every warp parks its accumulator tile in its own buffer, then a fixed-order sum over the warps
    __syncthreads();
    float* mine = reinterpret_cast<float*>(mybuf);
#pragma unroll
    for (int m = 0; m < T; ++m)
#pragma unroll
        for (int j = 0; j < 2 * T; ++j)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                float* o = mine + (16 * m + g + 8 * h) * ROWS + 8 * j + 2 * t;
                o[0] = acc[m][j][2 * h]; o[1] = acc[m][j][2 * h + 1];
            }
    __syncthreads();
    for (int idx = tid; idx < a.nc * ROWS; idx += WARPS * 32) {
        const int row = idx / ROWS, slot = idx - row * ROWS;
        if (slot >= a.RP) continue;
        float s = 0.f;
        for (int w = 0; w < WARPS; ++w) s += reinterpret_cast<const float*>(bufs + w * BUF)[row * ROWS + slot];
        a.alpha_part[(((size_t)b * a.alpha_pairs + row) * a.nSG + sg) * a.RP + slot] = s;
    }
}

int launch_alpha_small(const Model* m, const PairChunk& c, int* n_part, cudaStream_t st) {
    if (c.nc > 16 || c.Rp > 16 || c.nc < 1 || c.nc > c.pc) return set_error(NNJ_ERR_INVALID, "alpha_small: at most 16 pairs over 16 live nodes");
    const int groups = (c.C + AS_SITES - 1) / AS_SITES;
    *n_part = groups;
    if (groups > c.nAP) return set_error(NNJ_ERR_INVALID, "alpha_small: partial buffer too small");
    AlphaSmallArgs a;
    a.X = c.X; a.Y = c.Y; a.tree_stride = c.tree_stride; a.kph = (const __nv_bfloat16*)c.kp_h; a.kpl = (const __nv_bfloat16*)c.kp_l; a.S = c.S;
    a.slot_of = c.slot_of; a.slot_stride = c.slot_stride; a.pair_i = c.pair_i; a.pair_j = c.pair_j; a.pair_stride = c.pair_stride; a.n0 = c.n0;
    a.nc = c.nc; a.Rp = c.Rp; a.C = c.C; a.bh = m->nj.bh; a.xf = c.xf; a.pc = c.pc;
    a.alpha_part = c.alpha_part; a.alpha_pairs = c.alpha_pairs; a.nSG = c.nAP; a.RP = c.RP;
    constexpr size_t smem = 1024 + 1024 + 16 * (16 * 768);      // alignment | biases, pair slots | 16 warps x one site buffer (X, Y, K' hi / lo)
    static DevOnce once;      // per device, not per process
    if (int e = smem_opt_in(once, k_alpha_small<1, 16>, smem)) return e;
    prof_begin(KC_ALPHA, st);
    k_alpha_small<1, 16><<<dim3(groups, c.B), 16 * 32, smem, st>>>(a);
    LAUNCH_CHECK();
    return 0;
}

}  // namespace nnj
