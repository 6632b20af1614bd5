// nnj_internal.h — host-side structures shared by the libnnj translation units.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include <atomic>
#include <mutex>
#include <vector>
#include <string>
#include <vector>

#include "../../include/nnj.h"
#include "nnj_common.cuh"

// Experiment builds only (-DNNJ_ONE_PRODUCT, scratch/one_product_report.py): every low part of the bf16 split is forced to zero, i.e. the
// kernels compute with plain bf16 operands - the NUMERICS of a one-product mode (DESIGN.md 9.4), not its speed.  Never set in the product build.
#ifdef NNJ_ONE_PRODUCT
#define NNJ_LO_BF16(x) __float2bfloat16_rn(0.0f)
#define NNJ_LO_WORD(x) 0u
#else
#define NNJ_LO_BF16(x) (x)
#define NNJ_LO_WORD(x) (x)
#endif

namespace nnj {

// Site-major residual stream of the tensor-core encoder ("xs"): tokens t = site * R + taxon in tiles of 128; inside a tile the 64
// channels are split into 16-byte column chunks and every chunk is a plane of its own, [tile][chunk 0..15][token 0..127][4 floats].
// The encoder kernels own TMEM lane = token row and a few column chunks per thread, so a warp instruction that moves one chunk of
// 32 consecutive rows touches 512 contiguous bytes (4 lines); with a row-major [token][64] stream the same instruction touched
// 32 lines of 256-byte rows, 16 bytes each, and the loads / stores of a tile queued on the L1 tag stage.
__host__ __device__ __forceinline__ size_t xs_off(size_t t, int chunk) { return (t >> 7) * 8192 + (size_t)chunk * 512 + (t & 127) * 4; }
__host__ __device__ __forceinline__ size_t xs_tree_floats(size_t tokens) { return ((tokens + 127) >> 7) * 8192; }

// "t" suffix: transposed to [in k][out col] so a CTA can copy it straight into shared memory.
struct EmbedW { const float *w1, *b1, *w2t, *b2; };                 // model.py:39-43
struct AttnW { const float *ln_g, *ln_b, *qt, *kt, *vt, *ot, *qb, *kb, *vb, *ob; };
struct FfnW { const float *ln_g, *ln_b, *w1t, *b1, *w2t, *b2; };   // w1t/w2t: 4 chunks of [64][64]
struct LayerW { AttnW row, col; FfnW ffn; };
struct NjW {                                                        // model.py:46-59
    const float *wht, *bh;      // h_linear_last
    const float *wgt, *bg;      // g_linear_last
    const float *wq, *bq;       // g_attn_q, NOT transposed: K' = K * Wq folds the query projection into the keys
    const float *wkt, *bk;      // g_attn_k
    const float *wst, *bs;      // s_out.0
    const float *w2;            // s_out.2 weight [64]
    float b2;                   // s_out.2 bias
};

struct NjBf { const void *wgh, *wgl, *wsh, *wsl; };
// The four [64 k][64 n] weights of the merge / node-derive products as mma.sync B fragments (bf16 hi / lo):
// entry [(k16 * 8 + n8) * 32 + lane] = { hi(b0 b1), hi(b2 b3), lo(b0 b1), lo(b2 b3) } of m16n8k16, 16 KB per weight.
struct NjFrag { const uint4 *h, *k, *q, *g; };                       // h_linear_last^T, g_attn_k^T, g_attn_q, g_linear_last^T
// Encoder weights for the tcgen05 kernels: ready-to-copy shared-memory images (bf16 hi plane, then lo plane; every [N][64]
// block K-major SWIZZLE_128B), one set per layer, plus the stacked q|k|v biases.
struct EncTcW {
    const uint4 *row_qkv, *row_o, *col_qkv, *col_o;   // 48 KB, 16 KB, 48 KB, 16 KB
    const uint4 *w1, *w2;                              // fc1 [256][64]: 64 KB; fc2 [64][256]: 4 K-chunks of [64][64] per plane, 64 KB
    const float *row_qkvb, *col_qkvb;                  // [192]
};   // g_linear_last / s_out.0 weights [out][in] as bf16 hi/lo planes

struct Model {
    nnj_config cfg;
    int device;
    int num_layers;
    float* blob;                 // one device allocation holding every tensor
    EmbedW embed;
    std::vector<LayerW> layers;
    NjW nj;
    NjBf nj_bf;
    NjFrag nj_frag;
    void* blob_bf;               // device allocation behind nj_bf
    std::vector<EncTcW> enc_tc;  // per layer
    void* blob_enc;              // device allocation behind enc_tc
    void* host_ws; size_t host_ws_bytes;   // grow-only device workspace of nnj_rollout_host
    // nnj_rollout_host: its own non-blocking streams (H2D staging of chunk i+1 overlaps the rollout of chunk i) and a lock,
    // because the workspace above is owned by the model (one host call at a time per model; use one model per thread otherwise)
    cudaStream_t host_compute, host_copy;
    std::vector<cudaEvent_t> host_events;
    std::mutex host_lock;
};

// kernel classes for the optional per-class CUDA-event profiler (nnj_profile_*)
enum KClass { KC_EMBED = 0, KC_LN_QKV, KC_ROW_QK, KC_ROW_SOFTMAX, KC_ROW_PV, KC_OUT_PROJ, KC_COL_ATTN, KC_FFN, KC_DERIVE,
              KC_ALPHA, KC_ALPHA_SOFTMAX, KC_SCORE, KC_SELECT, KC_MERGE, KC_MISC, KC_BLEND, KC_LLH, KC_COUNT };
void prof_begin(int cls, cudaStream_t st);   // no-op unless profiling is enabled
void prof_end(cudaStream_t st);

int set_error(int code, const char* msg);
int set_cuda_error(cudaError_t e, const char* file, int line);

// Tail of every kernel launch inside a function returning an NNJ error code, with the stream in `st`: count the launch, close the
// profiler window prof_begin opened, and return the launch error, if any.
#define LAUNCH_CHECK()                                                         \
    do {                                                                       \
        ++g_launches;                                                          \
        prof_end(st);                                                          \
        cudaError_t e_ = cudaGetLastError();                                   \
        if (e_ != cudaSuccess) return set_cuda_error(e_, __FILE__, __LINE__);  \
    } while (0)

// ---- per-device state.  cudaFuncSetAttribute and the SM count belong to a DEVICE, not to the process: a second model on another
// GPU of the same process must raise the shared-memory limits there too.  `DevOnce` is a bit mask of initialised devices (the
// initialisers are idempotent, so two threads racing on the same device both succeed).
int current_device();
int sm_count();                                   // multiprocessors of the current device (cached per device)
struct DevOnce {
    std::atomic<unsigned long long> mask{0};
    bool need() const { return !((mask.load(std::memory_order_acquire) >> (current_device() & 63)) & 1ull); }
    void done() { mask.fetch_or(1ull << (current_device() & 63), std::memory_order_release); }
};
// Raise `kernel`'s dynamic shared-memory limit to `bytes` on the current device, once per device: `once` is the call site's own
// static DevOnce.
template <typename Kernel>
int smem_opt_in(DevOnce& once, Kernel* kernel, size_t bytes) {
    if (!once.need()) return 0;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    once.done();
    return 0;
}
// Workspace layout: regions taken one after another, each rounded up to 256 bytes.  The same lines size a workspace (null base: the
// pointers are null, `off` ends as the bytes the regions need) and carve it (base from ws_align), so the two cannot drift apart.
inline char* ws_align(void* ws) { return reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255); }
struct WsCarver {
    char* base; size_t off = 0;
    explicit WsCarver(char* b = nullptr) : base(b) {}
    template <typename T> T* take(size_t count) {
        T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
        off += (count * sizeof(T) + 255) & ~(size_t)255;
        return p;
    }
};
// RAII: make the model's device current for the duration of an entry point, restore the caller's device afterwards
struct DeviceGuard {
    int prev = -1; bool switched = false; cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int dev) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != dev) { err = cudaSetDevice(dev); switched = (err == cudaSuccess); }
    }
    ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};

// encoder (nnj_encoder.cu)
size_t encoder_ws_bytes(const Model* m, int B, int R, int C);
int run_encoder(Model* m, const int8_t* data, const uint8_t* mask, int B, int R, int L, float* x, size_t x_tree_stride,
                void* ws, size_t ws_bytes, cudaStream_t st);

// learned neighbour-joining loop (nnj_njloop.cu)
struct NjBuffers;
size_t nj_scores_ws_bytes(const Model* m, int B, int Rp, int C, int N);
size_t nj_rollout_ws_bytes(const Model* m, int B, int R, int C);
int nj_rollout_chunk(const Model* m, int B, int R, int C);
int run_pair_scores(Model* m, const float* state, const uint8_t* mask, int B, int Rp, int C, const int32_t* pi,
                    const int32_t* pj, int N, bool full, float* scores, void* ws, size_t ws_bytes, cudaStream_t st);
int run_pair_scores_incr(Model* m, const float* state, const uint8_t* mask, int B, int Rp, int C, const int32_t* prev_ij,
                         const float* logits_prev, float* logits_out, void* ws, size_t ws_bytes, cudaStream_t st);
int run_aggregate(Model* m, const float* state, int B, int Rp, int C, const int32_t* ij, float* out, size_t out_tree_stride,
                  void* ws, size_t ws_bytes, cudaStream_t st);
int run_merge(Model* m, const float* state_in, int B, int Rp, int C, const int32_t* ij, float* state_out, void* ws,
              size_t ws_bytes, cudaStream_t st);
int run_rollout(Model* m, const int8_t* data, const float* state0, const uint8_t* mask, int B, int R, int L, int select_mode,
                const float* gumbel, int32_t* merges, float* logits_trace, float* selected_logp, void* ws, size_t ws_bytes,
                cudaStream_t st);

// One launch of the NJ pair-score step: pairs [n0, n0 + nc) of the pair lists of B trees, against the Rp live nodes that occupy physical
// slots [0, Rp) of S, over C sites.  score_pairs (nnj_njloop.cu) fills it from its workspace; nj_path there picks the launchers below.
struct PairChunk {
    int B, Rp, S, C, n0, nc;
    const int32_t* slot_of; int slot_stride;                  // logical node -> physical slot, per tree
    const int32_t *pair_i, *pair_j; int pair_stride;          // pair lists by logical node (pair_i < 0: no pair)
    const uint8_t* mask;                                      // [B][C], nonzero = masked site; or null
    const float *X, *Y; size_t tree_stride;                   // fp32 node pools [B][S][C][64]
    const void *kp_h, *kp_l;                                  // K' planes [B][S][C][64] bf16 hi / lo
    const void *nodes_h, *nodes_l;                            // node planes [B][C][S][128] bf16 hi / lo = [X | W_g X]
    float* xf; int pc;                                        // x planes of the chunk [B][pc][C][64] fp32, pc pairs per tree
    void *xh, *xl;                                            // large-slot path: the x planes as K-major bf16 hi / lo
    float* alpha_part; int nAP;                               // alpha partials [B][alpha_pairs][nAP][RP], by physical slot
    float* alpha; int RP; int alpha_pairs;                    // softmaxed alpha [B][alpha_pairs][RP]
    float* score_part; int nSB;                               // score partials [B][alpha_pairs][nSB]
};
// Tensor-core pair-score launchers.  The alpha launchers write the chunk's x planes and alpha_part, the score launchers score_part;
// *n_part: the partials per pair they wrote.  A chunk outside a launcher's range is refused with NNJ_ERR_INVALID.
int launch_alpha_v3(const Model* m, const PairChunk& c, int* n_part, cudaStream_t st);        // nnj_alpha_tc.cu
int launch_alpha_small(const Model* m, const PairChunk& c, int* n_part, cudaStream_t st);     // nnj_alpha_small.cu
int launch_score_tc(const Model* m, const PairChunk& c, int* n_part, cudaStream_t st);        // nnj_score_tc.cu
int launch_score_inc(const Model* m, const PairChunk& c, int* n_part, cudaStream_t st);       // nnj_score_inc.cu
int launch_score_small(const Model* m, const PairChunk& c, int* n_part, cudaStream_t st);     // nnj_score_small.cu
int launch_score_big(const Model* m, const PairChunk& c, int* n_part, cudaStream_t st);       // nnj_score_big.cu
int launch_blend_planes(const Model* m, const PairChunk& c, cudaStream_t st);                 // nnj_score_big.cu: x planes, fp32 and bf16

// tcgen05 split-bf16 GEMM (nnj_tc.cu)
// products: 3 = hi*hi + hi*lo + lo*hi (NNJ_PREC_BF16X3), 1 = hi*hi only (NNJ_PREC_BF16: plain bf16 operands, the lo planes are not read)
int launch_tc_gemm(int cls, const void* Ah, const void* Al, const void* Bh, const void* Bl, float* Cm, int Z, int M, int N, int K, size_t lda,
                   size_t sA, size_t ldb, size_t sB, int ldc, size_t sC, cudaStream_t st, int products = 3);
int launch_tc_gemm_ex(int cls, const void* Ah, const void* Al, const void* Bh, const void* Bl, float* Cm, int Z, int M, int N, int K, size_t lda,
                      size_t sA, size_t ldb, size_t sB, int ldc, size_t sC, int bn, int nsplit, int chunks_per_split, size_t split_stride,
                      cudaStream_t st, int products = 3);
int launch_tc_gemm_bmn(int cls, const void* Ah, const void* Al, const void* Bh, const void* Bl, float* Cm, int Z, int M, int N, int K, size_t lda,
                       size_t sA, size_t ldb, size_t sB, int ldc, size_t sC, cudaStream_t st, int products = 3, const float* row_div = nullptr);
// TMA tensor maps (nnj_tc.cu).  encode_tmap: cuTensorMapEncodeTiled through the runtime's driver entry point, element strides 1, no
// interleave, no out-of-bounds fill; dims / strides / box as that call takes them.  Returns 0, or NNJ_ERR_CUDA with a message naming `what`.
int encode_tmap(CUtensorMap* map, CUtensorMapDataType dtype, int rank, const void* base, const cuuint64_t* dims, const cuuint64_t* strides,
                const cuuint32_t* box, CUtensorMapSwizzle swizzle, CUtensorMapL2promotion l2, const char* what);
// node planes [B*C][S][128] bf16 ([X | W_g X] per slot), box 64 channels x box_rows slots of one site; slots >= n_live (when > 0) read as 0
// (nnj_score_tc.cu)
int make_tmap_nodes(CUtensorMap* map, const void* base, int S, int BC, int box_rows = 64, int n_live = -1);
// x planes [B][pc][C][64] fp32 as (d, site, pair, tree), box 32 channels x box_rows pairs at one site; pairs >= nrows read as 0 (nnj_score_tc.cu)
int make_tmap_xtile(CUtensorMap* map, const float* base, int pc, int nrows, int C, int B, int box_rows = 64);
// S = Q K^T of the tied row attention with the softmax in the epilogue: unnormalised exp(s - max) as bf16 hi / lo planes + the row sums, which the
// P V launch takes as `row_div` (k_tc_gemm2s, CTA pairs; site count a multiple of 256)
bool row_qk_softmax_ok(int C, int products);
int launch_row_qk_softmax(int cls, const void* Qh, const void* Ql, const void* Kh, const void* Kl, void* Ph, void* Pl, float* rowsum, const uint8_t* mask,
                          int heads, int Z, int C, int K, cudaStream_t st);
// tcgen05 encoder kernels over the site-major residual stream (nnj_encoder_tc.cu)
int launch_enc_rowqkv_tc(const Model* m, int layer, const float* xs, size_t xs_tree_stride, int B, int R, int C, float q_scale, const uint8_t* mask,
                         void* qh, void* ql, void* kh, void* kl, void* vh, void* vl, cudaStream_t st);
int launch_enc_colblock_tc(const Model* m, int layer, float* xs, size_t xs_tree_stride, const float* ctx, int B, int R, int C, const uint8_t* mask,
                           cudaStream_t st);
int launch_enc_ffn_tc(const Model* m, int layer, float* xs, size_t xs_tree_stride, int B, int R, int C, cudaStream_t st);
int launch_sm_to_nm(const float* xs, size_t xs_tree_stride, float* out, size_t out_tree_stride, int B, int R, int C, cudaStream_t st);
int run_tc_unit(const float* A, const float* B, float* Dm, int bn, cudaStream_t st);
int run_gemm_split_bf16(const float* A, const float* B, float* Cm, int Z, int M, int N, int K, void* ws, size_t ws_bytes, cudaStream_t st);

// tree likelihood / branch-length optimisation (nnj_llh.cu)
// The inputs of every likelihood entry point: tips [B][R][L] (4-bit state masks) and pattern weights [B][L] on the device; children
// [B][R-1][2] in join order, brlen [B][2R-2] and the packed model [B][LLH_MODEL] on the host.  The modes that optimise branch
// lengths write them back to brlen, LlhMode::All the optimised model to model.
struct LlhTrees {
    const uint8_t* tips; const double* weights;
    const int32_t* children; double* brlen; double* model;
    int B, R, L;
};
// Eval: log L at the given lengths; Brlen: branch-length sweeps; All: branch lengths and model parameters; Prepare: llh_prepare
enum class LlhMode : int { Eval = 0, Brlen = 1, All = 2, Prepare = 3 };
struct LlhOptions {
    int max_passes; double eps;        // branch-length sweeps until one gains < eps (Brlen, All)
    double lh_eps; int max_rounds;     // rounds of (model parameters, sweeps) until one gains < lh_eps (All)
};
size_t llh_ws_bytes(int B, int R, int L);
int llh_check_tree(const int32_t* ch, int R);     // 0 when children is a binary tree in join order
// modes Eval, Brlen, All; llh_before / llh_after [B] (host) may be null
int run_llh(const LlhTrees& in, LlhMode mode, const LlhOptions& opt, double* llh_before, double* llh_after, void* ws, size_t ws_bytes, cudaStream_t st);
// First step of branch support, for trees the caller has checked: the subtree vectors D and, for every branch, the vector U of the
// rest of the tree, at the given lengths; the per-pattern log-likelihoods to site_dev [B][L] (device) and log L to llh_h [B] (host).
// rc is 0 or an error code; the vectors and their scale counts stay in ws.
struct LlhPrepared { int rc; const double *D, *U, *inv; const int32_t *Dn, *Un; };
LlhPrepared llh_prepare(const LlhTrees& in, double* site_dev, double* llh_h, void* ws, size_t ws_bytes, cudaStream_t st);
// likelihood branch support (nnj_llh_nni.cu): NNI quartets of every internal branch, RELL replicates
size_t llh_support_ws_bytes(int B, int R, int L, int n_rell);
int run_llh_support(const LlhTrees& in, uint64_t seed, int64_t rep0, int n_rell, int32_t* branch_node_h, double* llh_h, double* nni_brlen_h,
                    int32_t* sh_h, int32_t* lbp_h, double* site_dev, void* ws, size_t ws_bytes, cudaStream_t st);
// tree topology test over K trees of one alignment (nnj_llh_topo.cu): tips [R][L] and weights [L] on the device, the trees on the host
size_t llh_topo_ws_bytes(int K, int R, int L, int n_boot);
int run_llh_topo(const uint8_t* tips, const double* weights, const int32_t* children_h, const double* brlen_h, const double* model_h, int K, int R,
                 int L, uint64_t seed, int n_boot, double* llh_h, int32_t* win_h, int32_t* kh_h, int32_t* sh_h, double* elw_h, double* site_dev,
                 void* ws, size_t ws_bytes, cudaStream_t st);
int gamma_rates(double alpha, int ncat, double* out);

// pre-training loss over a teacher-forced rollout's logits trace (nnj_rankloss.cu)
size_t rank_loss_ws_bytes(int B, int R);
int run_rank_loss(const float* logits_trace, const uint8_t* in_set, int B, int R, float margin, double ratio, float* out, void* ws, size_t ws_bytes,
                  cudaStream_t st);

// bootstrap support: column resampling and transfer distances of reference splits to NJ trees (nnj_support.cu)
int run_bootstrap_columns(const int8_t* data, int R, int L, int l_eff, uint64_t seed, int64_t rep0, int B, int8_t* out, cudaStream_t st);
int run_split_distances(const int32_t* merges, int B, int R, const uint64_t* splits, int S, int32_t* dist, cudaStream_t st);

}  // namespace nnj
