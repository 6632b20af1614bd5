// nnj_tc.cuh — inline-PTX helpers for tcgen05 / TMEM / TMA / mbarrier and for mma.sync / ldmatrix / cp.async on sm_100a (shared by the
// tensor-core kernels).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdint.h>
#ifdef NNJ_MBAR_DEBUG
#include <cstdio>
#endif

#ifndef NNJ_LO_WORD
#define NNJ_LO_WORD(x) (x)     // see nnj_internal.h (experiment builds zero the low parts)
#endif

namespace nnj {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// 1024-byte aligned start inside the dynamic shared-memory window.  Pure pointer arithmetic on the __shared__ array (no integer
// round trip), so the compiler keeps the shared address space and emits LDS / STS instead of generic LD / ST.
__device__ __forceinline__ uint8_t* smem_align1024(uint8_t* raw) { return raw + ((1024u - (smem_u32(raw) & 1023u)) & 1023u); }

// D[16 x 8] += A[16 x 16] . B[16 x 8] on register fragments (bf16 operands, fp32 accumulate).  Lane (g = lane >> 2, t = lane & 3):
// a0 = A[g][2t, 2t+1], a1 = A[g+8][2t, 2t+1], a2 = A[g][8+2t, 9+2t], a3 = A[g+8][8+2t, 9+2t]; b0 = B[2t, 2t+1][g], b1 = B[8+2t, 9+2t][g];
// d0 d1 = D[g][2t, 2t+1], d2 d3 = D[g+8][2t, 2t+1].  Measured on B200 (scratch/hmma_bench.cu): one m16n8k16 and one m16n8k8 both hold a
// sub-partition's legacy tensor pipe for 8 clocks (20 clocks latency), so the K = 16 form is used throughout.
__device__ __forceinline__ void mma_m16n8k16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// four 8 x 8 b16 matrices (rows of 16 B, lane l supplies the address of row l & 7 of matrix l >> 3), transposed on the way in:
// lane (g, t) receives M[2t, 2t+1][g] of every matrix = a B fragment half for a row-major [k][n] operand
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
// 16-byte global -> shared copy, bypassing L1 (cp.async.cg); completes at the next commit_group / wait_group
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Blocking wait.  try_wait itself suspends the warp for a hardware-chosen time slice before it reports failure, so the loop below
// turns over slowly; the time-out check reads the clock only once per 64 turns (a clock64 per turn showed up as 3 % of all
// executed instructions - CS2R - in the score kernel, issue slots taken from the warps that had work).
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    long long t0 = 0;
    uint32_t turns = 0;
    while (!mbar_try_wait(bar, parity)) {
        if ((++turns & 63u) == 0u) {
            const long long now = clock64();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 40000000000LL) {   // ~20 s at 1.9 GHz (instrumented profiler passes run 100x slower): protocol error, fail loudly instead of hanging
#ifdef NNJ_MBAR_DEBUG
                printf("mbar timeout: block (%d,%d,%d) thread %d bar smem+%u parity %u\n", blockIdx.x, blockIdx.y, blockIdx.z, threadIdx.x,
                       smem_u32(bar), parity);
#endif
                __trap();
            }
        }
    }
}

__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}

__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

// TMA prefetch of a tile into L2 (no shared memory, no barrier): hides the HBM latency of a later tma_load of the same box
__device__ __forceinline__ void tma_prefetch_3d(const CUtensorMap* map, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];"
                 ::"l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_prefetch_4d(const CUtensorMap* map, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.prefetch.tensor.4d.L2.global.tile [%0, {%1, %2, %3, %4}];"
                 ::"l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
// [0,14) start>>4, [16,30) LBO>>4 (unused for swizzled K-major), [32,46) SBO>>4 = 1024 B (8 rows x 128 B),
// [46,48) version = 1 (sm_100), [61,64) layout = 2 (SWIZZLE_128B).
__device__ __forceinline__ uint64_t umma_desc_k128(uint32_t smem_addr) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFF) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

// Same, with a leading-dimension byte offset: MN-major operands wider than one 128-byte swizzle row place their
// 64-element column blocks LBO bytes apart (canonical layout ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units).
__device__ __forceinline__ uint64_t umma_desc_lbo(uint32_t smem_addr, uint32_t lbo_bytes) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) |
           (2ull << 61);
}

// One lane of a converged warp (warp-uniform control flow keeps descriptors in uniform registers).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}

// Instruction descriptor (cute::UMMA::InstrDescriptor): D fp32, A/B bf16, both K-major, M x N.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// A operand read from tensor memory (128 lanes x K/2 32-bit columns, two bf16 per column), B from shared memory.
__device__ __forceinline__ void umma_bf16_ta(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// ---- cheap-issue forms.  One thread issues every UMMA of a CTA, and with 128 x 64..128 x 16 instructions and the 3-product
// split the tensor core finishes one in 32-64 clk: building two 64-bit descriptors per instruction (shifts, masks, ors) made the
// ISSUING THREAD the bottleneck (~125 clk per UMMA measured).  Here the descriptors are split into a constant high word and a
// low word (start address >> 4 | LBO >> 4 << 16) that advances by a plain 32-bit add per k-step; `ACC` is a template constant.
__device__ __forceinline__ uint32_t umma_desc_lo(uint32_t smem_addr, uint32_t lbo_bytes = 0) { return ((smem_addr >> 4) & 0x3FFFu) | (((lbo_bytes >> 4) & 0x3FFFu) << 16); }
constexpr uint32_t UMMA_DESC_HI = (uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29);     // SBO 1024 B, version 1, SWIZZLE_128B
template <bool ACC>
__device__ __forceinline__ void umma_ss(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "mov.b64 da, {%1, %5};\n\tmov.b64 db, {%2, %5};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(idesc), "n"(ACC ? 1 : 0), "r"(UMMA_DESC_HI)
        : "memory");
}
template <bool ACC>
__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint32_t b_lo, uint32_t idesc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 db;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "mov.b64 db, {%2, %5};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "r"(b_lo), "r"(idesc), "n"(ACC ? 1 : 0), "r"(UMMA_DESC_HI)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// ---- CTA-pair forms (cta_group::2: the two CTAs of a cluster on one TPC execute one 256-row UMMA; each holds its 128 rows of A, half of
//      B's N range and its 128 rows of the accumulator).  Only the rank-0 CTA issues MMAs and commits.
template <bool ACC>
__device__ __forceinline__ void umma_ss2(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "mov.b64 da, {%1, %5};\n\tmov.b64 db, {%2, %5};\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(idesc), "n"(ACC ? 1 : 0), "r"(UMMA_DESC_HI)
        : "memory");
}
// arrive on the barrier at this shared-memory offset in every CTA of `mask` once all MMAs issued so far have retired
__device__ __forceinline__ void umma_commit2_mc(uint64_t* bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(mask) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same shared-memory location in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load into THIS CTA's shared memory whose bytes are counted on a barrier of the pair's leader (shared::cluster address)
__device__ __forceinline__ void tma_load_3d_2sm(void* smem_dst, const CUtensorMap* map, uint32_t bar_cluster_addr, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* slot, uint32_t cols) {      // one warp of EACH CTA of the pair, same slot offset
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t base, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols));
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}


// generic-proxy shared-memory writes -> visible to the async proxy (tensor core / TMA)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// two floats -> bf16x2 word (element 0 = a in the low half), round to nearest even: one cvt.rn.bf16x2.f32
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
}
// pack (hi, lo) bf16 split of two floats: returns hi pair / lo pair as bf16x2 words (element 0 in the low half)
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
    hi = pack_bf16x2(a, b);
    const float2 r = fsub2(make_float2(a, b), make_float2(__uint_as_float(hi << 16), __uint_as_float(hi & 0xffff0000u)));   // one FADD2
    lo = NNJ_LO_WORD(pack_bf16x2(r.x, r.y));
}
__device__ __forceinline__ float bf_lo(uint32_t w) { return __uint_as_float(w << 16); }          // element 0 of a bf16x2 word
__device__ __forceinline__ float bf_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }  // element 1

// ---- TMEM allocation (one warp, converged) and wider loads
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols));
}
// tcgen05.ld without the trailing wait: issue several, then tmem_ld_wait() once
__device__ __forceinline__ void tmem_ld32_nw(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16_nw(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
          "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_ld8_nw(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld4_nw(uint32_t taddr, uint32_t (&v)[4]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(taddr));
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, uint32_t v0, uint32_t v1, uint32_t v2, uint32_t v3) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(v0), "r"(v1), "r"(v2), "r"(v3) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- operand staging by threads: K-major SWIZZLE_128B tiles [rows][64 bf16] (128 B per row, 16-byte chunk j stored at j ^ (row & 7))
// 8 consecutive K elements (chunk j) of one row, split into the hi / lo planes.
__device__ __forceinline__ void a_store8(uint8_t* hi, uint8_t* lo, int row, int j, const float* v) {
    uint4 hh, ll;
    split2(v[0], v[1], hh.x, ll.x);
    split2(v[2], v[3], hh.y, ll.y);
    split2(v[4], v[5], hh.z, ll.z);
    split2(v[6], v[7], hh.w, ll.w);
    const int off = row * 128 + ((j ^ (row & 7)) << 4);
    *reinterpret_cast<uint4*>(hi + off) = hh;
    *reinterpret_cast<uint4*>(lo + off) = ll;
}

// D[128 x N] (+)= A[128 x 64] * W[N x 64]^T with the 3-product bf16 split; all four operands are K-major SWIZZLE_128B tiles
// (A planes 16 KB, W planes N*128 B).  Call from ONE elected lane.  first_acc = 0 starts a fresh accumulator.
// Descriptor low words advance by 2 (32 B >> 4) per 16-element k-step (cheap-issue forms above).
__device__ __forceinline__ void umma_split_k64(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, uint32_t w_hi, uint32_t w_lo, uint32_t idesc,
                                               uint32_t first_acc, int one = 0) {
    const uint32_t dah = umma_desc_lo(a_hi), dal = umma_desc_lo(a_lo), dwh = umma_desc_lo(w_hi), dwl = umma_desc_lo(w_lo);
    if (one) {      // NNJ_PREC_BF16: plain bf16 operands, hi * hi only
        if (first_acc) umma_ss<true>(tmem_d, dah, dwh, idesc); else umma_ss<false>(tmem_d, dah, dwh, idesc);
#pragma unroll
        for (int k = 1; k < 4; ++k) umma_ss<true>(tmem_d, dah + 2 * k, dwh + 2 * k, idesc);
        return;
    }
    if (first_acc) umma_ss<true>(tmem_d, dal, dwh, idesc); else umma_ss<false>(tmem_d, dal, dwh, idesc);   // small terms first
    umma_ss<true>(tmem_d, dah, dwl, idesc);
    umma_ss<true>(tmem_d, dah, dwh, idesc);
#pragma unroll
    for (int k = 1; k < 4; ++k) {
        umma_ss<true>(tmem_d, dal + 2 * k, dwh + 2 * k, idesc);
        umma_ss<true>(tmem_d, dah + 2 * k, dwl + 2 * k, idesc);
        umma_ss<true>(tmem_d, dah + 2 * k, dwh + 2 * k, idesc);
    }
}

}  // namespace nnj
