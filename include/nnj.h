/* nnj.h — C ABI of libnnj: the B200-native NeuralNJ inference hot path.
 *
 * The reference (DingShizhe/NeuralNJ) has no FFI: its boundary for this path is
 * a set of Python call signatures (SURVEY.md section 8b).  Each entry point
 * below names the reference interface it replaces (file:line relative to the
 * reference checkout).  Plain pointers and sizes only; no torch / C++ types.
 *
 * Conventions
 *   - every function returns 0 on success, a negative nnj_status otherwise, and
 *     never aborts; nnj_last_error() returns a thread-local message.
 *   - "dev" pointers are CUDA device pointers on the device the model was
 *     created on; "host" pointers are ordinary (ideally pinned) host memory.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default
 *     stream).  All device-pointer entry points are asynchronous on it.
 *   - tensors are dense row-major; D = 64 embedding width, C = L / patch.
 *   - the caller owns every buffer, including the workspace.
 */
#ifndef NNJ_H_
#define NNJ_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NNJ_ABI_VERSION 1

typedef enum nnj_status {
    NNJ_OK = 0,
    NNJ_ERR_INVALID = -1,     /* bad argument / unsupported shape or config        */
    NNJ_ERR_CUDA = -2,        /* a CUDA runtime call failed (message has details)  */
    NNJ_ERR_WORKSPACE = -3,   /* workspace too small                               */
    NNJ_ERR_NOMEM = -4
} nnj_status;

/* Model hyper-parameters: cfgs.model.* of the reference (utils.py:44-51, YAML :24-30). */
typedef struct nnj_config {
    int32_t embed_dim;    /* must be 64                                   */
    int32_t num_heads;    /* must be 8                                    */
    int32_t num_layers;   /* >= 1 (6 in the shipped configs)              */
    int32_t vocab_size;   /* must be 4                                    */
    int32_t patch_size;   /* must be 1                                    */
    int32_t precision;    /* nnj_precision                                */
} nnj_config;

typedef enum nnj_precision {
    NNJ_PREC_FP32 = 0,        /* fp32 CUDA-core arithmetic everywhere                       */
    NNJ_PREC_BF16X3 = 1,      /* dense contractions on tcgen05: split-bf16 (hi*hi+hi*lo+lo*hi), fp32 accumulate */
    NNJ_PREC_BF16 = 2         /* "bf16 encoder": the encoder's contractions (row q|k|v, Q K^T, P V, out projections, column q|k|v, FFN) take
                                 plain bf16 operands - one tcgen05 product, fp32 accumulate, the lo planes neither written nor read; residual
                                 stream, LayerNorm, softmax statistics stay fp32 and the NJ loop keeps the split form.  Scores stay within
                                 1e-2 relative of the fp32 reference; Argmax topologies are NOT guaranteed to match it (DESIGN.md 5). */
} nnj_precision;

typedef enum nnj_select_mode {
    NNJ_SELECT_ARGMAX = 0,    /* torch.argmax(logits)            finetune_rl_search.py:145 */
    NNJ_SELECT_GUMBEL = 1,    /* argmax(logits + gumbel noise) == Categorical(logits).sample()  :147 */
    NNJ_SELECT_FORCED = 2     /* teacher forcing, train.py:116-119 (supervise_rollout): the merge-list buffer holds the actions (i < j in the
                               * current node list) ON ENTRY; an entry that is not such a pair falls back to the argmax, and the buffer holds the
                               * actions actually taken on return */
} nnj_select_mode;

typedef struct nnj_model nnj_model;   /* opaque: device copy of the state_dict tensors */

const char* nnj_last_error(void);
int nnj_abi_version(void);

/* Replaces PhyloATTN.__init__ + load_state_dict + .to(device) (model.py:12-60,
 * finetune_rl_search.py:482-484).  `tensors` are n_tensors host pointers to
 * fp32 arrays in the reference's state_dict order (172 for 6 layers: 26 per layer + 16):
 * per layer row{k,v,q,out}.{weight,bias}, row LN, col{k,v,q,out}, col LN,
 * fc1, fc2, ffn LN; then embed.0, embed.2, h_linear_last, g_linear_last,
 * g_attn_q, g_attn_k, s_out.0, s_out.2.  `numels` gives each array's length
 * and is checked against the config. */
int nnj_model_create(nnj_model** out, const nnj_config* cfg, const float* const* tensors,
                     const int64_t* numels, int n_tensors, int device);
void nnj_model_destroy(nnj_model* m);

/* Bytes of device workspace needed by the entry points below for a batch of
 * B alignments of R taxa x L sites (what: 0 = encode, 1 = pair scoring /
 * aggregate, 2 = fused rollout). */
int64_t nnj_workspace_bytes(const nnj_model* m, int what, int B, int R, int L);

/* PhyloATTN.encode_zxr(batch_input, batch_seq_mask) (model.py:67-88).
 * data int8 [B,R,L,4]; seq_mask uint8 [B,L] (1 = padded column); out fp32 [B,R,C,64]. */
int nnj_encode(nnj_model* m, const int8_t* data_dev, const uint8_t* seq_mask_dev, int B, int R, int L,
               float* out_dev, void* ws_dev, int64_t ws_bytes, void* stream);

/* decode_zxr step 0 + decode_gg (model.py:168-181, :90-99): scores of all
 * P = R'(R'-1)/2 pairs in itertools.combinations order.  state fp32 [B,R',C,64];
 * logits fp32 [B,P]. */
int nnj_pair_scores_full(nnj_model* m, const float* state_dev, const uint8_t* seq_mask_dev, int B, int Rp, int C,
                         float* logits_dev, void* ws_dev, int64_t ws_bytes, void* stream);

/* decode_gg on an explicit pair list (model.py:184-197): scores of N pairs
 * (pair_i[b,n], pair_j[b,n]) per tree against the node set `state`.
 * pair_i/pair_j int32 [B,N]; scores fp32 [B,N]. */
int nnj_pair_scores_list(nnj_model* m, const float* state_dev, const uint8_t* seq_mask_dev, int B, int Rp, int C,
                         const int32_t* pair_i_dev, const int32_t* pair_j_dev, int N,
                         float* scores_dev, void* ws_dev, int64_t ws_bytes, void* stream);

/* decode_zxr step t>=1 (model.py:184-201) with the cache index map of
 * utils.get_score_indices_to_prev (utils.py:213-251) evaluated in closed form
 * on the device.  prev_ij int32 [B,2] = pair merged to obtain `state` (R' nodes);
 * logits_prev fp32 [B, (R'+1)R'/2]; logits_out fp32 [B, R'(R'-1)/2]. */
int nnj_pair_scores_incr(nnj_model* m, const float* state_dev, const uint8_t* seq_mask_dev, int B, int Rp, int C,
                         const int32_t* prev_ij_dev, const float* logits_prev_dev, float* logits_out_dev,
                         void* ws_dev, int64_t ws_bytes, void* stream);

/* PhyloATTN.aggregate(x_i, x_j, (ii, jj), batchwise_ij_indices=True)
 * (model.py:102-155, called from environment.py:829): merged-node embedding of
 * pair ij[b] computed against the pre-merge node set.  ij int32 [B,2];
 * out fp32 [B,C,64]. */
int nnj_aggregate(nnj_model* m, const float* state_dev, int B, int Rp, int C, const int32_t* ij_dev,
                  float* out_dev, void* ws_dev, int64_t ws_bytes, void* stream);

/* PhyInferEnv.step tensor half (environment.py:760-835): slot i <- aggregate(i,j),
 * slot j removed, order kept.  state_in [B,R',C,64] -> state_out [B,R'-1,C,64]. */
int nnj_merge(nnj_model* m, const float* state_in_dev, int B, int Rp, int C, const int32_t* ij_dev,
              float* state_out_dev, void* ws_dev, int64_t ws_bytes, void* stream);

/* Fused reinforce_rollout(eval=True) device loop (finetune_rl_search.py:107-175):
 * encode, then R-1 x (score -> select -> merge) without leaving the device.
 * gumbel fp32 [B,R-1,P0] (P0 = R(R-1)/2) or NULL for argmax.
 * merges int32 [B,R-1,2]; optional traces: logits_trace fp32 [B, sum_t P_t]
 * (steps concatenated, P_t = (R-t)(R-t-1)/2), selected_logp fp32 [B,R-1]
 * (log_softmax(logits)[action], the last entry belongs to the final 2-node step). */
int nnj_rollout(nnj_model* m, const int8_t* data_dev, const uint8_t* seq_mask_dev, int B, int R, int L,
                int select_mode, const float* gumbel_dev, int32_t* merges_dev,
                float* logits_trace_dev, float* selected_logp_dev,
                void* ws_dev, int64_t ws_bytes, void* stream);

/* Same, but starting from a supplied encoder output (state fp32 [B,R,C,64]) —
 * used by Search mode to share one encoder pass across sampled rollouts. */
int nnj_rollout_from_state(nnj_model* m, const float* state_dev, const uint8_t* seq_mask_dev, int B, int R, int C,
                           int select_mode, const float* gumbel_dev, int32_t* merges_dev,
                           float* logits_trace_dev, float* selected_logp_dev,
                           void* ws_dev, int64_t ws_bytes, void* stream);

/* End-to-end convenience with HOST buffers: copies data/mask to the device,
 * runs nnj_rollout in chunks sized to the free device memory, copies the merge
 * lists back and synchronises.  data_host int8 [B,R,L,4]; merges_host int32 [B,R-1,2]. */
int nnj_rollout_host(nnj_model* m, const int8_t* data_host, const uint8_t* seq_mask_host, int B, int R, int L,
                     int select_mode, const float* gumbel_host, int32_t* merges_host, float* selected_logp_host);

/* ---- Tree likelihood (SURVEY.md 8 f2): what Search / branch_optimize=True use to score a topology.
 * Replaces the reference's native binding raxmlpy.compute_llh / raxmlpy.optimize_brlen
 * (RAxMLpy/raxmlpy/core.py:6-12 -> RAxMLpy/cpp/raxmlpy.cpp:1790-1805, 1854-1872; call sites environment.py:365-379, 625-670).
 * Model GTR+I+G4 (raxmlpy's model string "GTR+I+G"); one CTA per tree, fp64.  3 <= R <= 4096 taxa (others: NNJ_ERR_INVALID).
 * Every branch length, and the root branch brlen[c1] + brlen[c2] as a whole, is clamped to [1e-6, 100] in evaluation and
 * optimisation alike, so zero or negative input lengths score as 1e-6.  Conditional likelihood vectors are rescaled per
 * (node, pattern) by 2^256 when all their entries fall below 2^-256, with an int32 count per (node, pattern) in the workspace:
 * no site underflows fp64 at any R in range, and where no vector is rescaled the results are those of unscaled pruning, bit for bit.
 *   tips_dev      uint8 [B,R,L]   4-bit state masks per taxon and alignment pattern (bit a = state a possible; gap / N = 15)
 *   weights_dev   double [B,L]    pattern multiplicities (1 for uncompressed columns)
 *   children_host int32 [B,R-1,2] topology in join order: leaves 0..R-1, inner node R+k = (children[k][0], children[k][1]),
 *                                 the last join is the root (the NJ merge list replayed, neuralnj_b200/likelihood.py)
 *   brlen_host    double [B,2R-2] length of the branch above node v; the two root branches are one branch of the unrooted tree
 *   model_host    double [B,64]   eigenvalues 4 | eigenvectors U 16 | U^-1 16 | base frequencies 4 | class rates 4 | p_inv | alpha |
 *                                 flags (1: GTR rates free, 2: +G, 4: +I) | pad | GTR rates AC AG AT CG CT GT | pad 10
 * nnj_llh_eval returns log L per tree; nnj_llh_optimize_brlen maximises it over the branch lengths (Newton-Raphson per branch,
 * depth-first sweeps until a sweep gains less than eps or max_passes), updates brlen_host (root branch split evenly) and returns
 * log L before / after.  nnj_llh_optimize_all also searches the free model parameters named by `flags` inside the kernel (golden
 * section per parameter, eigen-system and class rates rebuilt on the device; rounds of parameters + branch sweeps until a round
 * gains < lh_eps - the loop shape of raxmlpy.cpp:1721-1746 with lh_epsilon = lh_eps) and returns the optimised model in model_host.
 * All three synchronise `stream` (their results are host values). */
int64_t nnj_llh_workspace_bytes(int B, int R, int L);
int nnj_llh_eval(const uint8_t* tips_dev, const double* weights_dev, const int32_t* children_host, const double* brlen_host,
                 const double* model_host, int B, int R, int L, double* llh_host, void* ws_dev, int64_t ws_bytes, void* stream);
int nnj_llh_optimize_brlen(const uint8_t* tips_dev, const double* weights_dev, const int32_t* children_host, double* brlen_host,
                           const double* model_host, int B, int R, int L, int max_passes, double eps,
                           double* llh_before_host, double* llh_after_host, void* ws_dev, int64_t ws_bytes, void* stream);
int nnj_llh_optimize_all(const uint8_t* tips_dev, const double* weights_dev, const int32_t* children_host, double* brlen_host,
                         double* model_host, int B, int R, int L, int max_passes, double eps, double lh_eps, int max_rounds,
                         double* llh_before_host, double* llh_after_host, void* ws_dev, int64_t ws_bytes, void* stream);
/* Likelihood branch support of a fixed tree (IQ-TREE -alrt / -abayes, PhyML aLRT; DESIGN.md 12): for each of the R-3 internal
 * branches (in increasing v: the branch above inner node v, the root branch once at the first root child and only when both root
 * children are inner) the two NNI alternatives of its quartet, each with its central and four outer lengths optimised by rounds of
 * Newton (model fixed; a round optimises central, A, B, C, D; rounds stop after one gains < 1e-3, or after 8), and RELL replicates
 * rep0 .. rep0+n_rell-1 of the per-pattern log-likelihoods.  Inputs as nnj_llh_eval; 3 <= R <= 4096 (R = 3: no branches, nothing
 * written).  The pattern weights must be non-negative integers (their sum n is the site count the replicates draw from).
 * Draw i of replicate r is the site u = (x0 * n) >> 32, x0 = word 0 of Philox4x32-10 with counter (i, r & 0xffffffff, r >> 32, 0)
 * and key (seed & 0xffffffff, seed >> 32) (the rule of nnj_bootstrap_columns); pattern p takes the sites cum[p] <= u < cum[p+1].
 *   branch_node_host int32  [B,R-3]      v of each internal branch
 *   llh_host         double [B,R-3,3]    L0 (the tree), L1 (AC|BD), L2 (AD|BC)
 *   nni_brlen_host   double [B,R-3,2,5]  optimised central, A, B, C, D lengths of each alternative
 *   sh_count_host    int32  [B,R-3]      replicates with delta > (largest - second largest of Lk* - Lk) + 0.05 (SH-aLRT = 100 count / n_rell)
 *   lbp_count_host   int32  [B,R-3]      replicates with L0* >= max(L1*, L2*) (local bootstrap probability)
 *   site_llh_dev     double [B,R-3,3,L]  per-pattern log-likelihoods l0, l1, l2 (device; may be NULL)
 * In the RELL statistics Lk = sum_p w[p] lk[p], Lk* = sum_p c_r[p] lk[p] (pattern order, a multiply then an add) and delta = L0 - max(L1, L2)
 * from those sums.  A replicate depends only on (seed, r, n): counts over disjoint rep0 ranges add.  Bad weights, an invalid tree:
 * NNJ_ERR_INVALID; a workspace smaller than nnj_llh_support_workspace_bytes(B, R, L, n_rell): NNJ_ERR_WORKSPACE.  Synchronises `stream`. */
int64_t nnj_llh_support_workspace_bytes(int B, int R, int L, int n_rell);
int nnj_llh_branch_support(const uint8_t* tips_dev, const double* weights_dev, const int32_t* children_host, const double* brlen_host,
                           const double* model_host, int B, int R, int L, uint64_t seed, int64_t rep0, int n_rell,
                           int32_t* branch_node_host, double* llh_host, double* nni_brlen_host, int32_t* sh_count_host,
                           int32_t* lbp_count_host, double* site_llh_dev, void* ws_dev, int64_t ws_bytes, void* stream);
/* Tree topology test over K candidate trees of one alignment (IQ-TREE -z trees -zb n_boot -au, CONSEL; DESIGN.md 13).  Each tree is
 * scored at its own lengths and model (fit them first, e.g. with nnj_llh_optimize_all): l_k[p] is its per-pattern log-likelihood and
 * L_k = sum_p w[p] l_k[p] (pattern order, a multiply then an add); k* is the largest L_k, the lowest index on a tie.  Scales
 * s = 0..9, r_s = (5 + s) / 10, draw n_s = floor(r_s n + 0.5) sites per replicate (n = sum of the weights); draw i of replicate j
 * is the site u = (x0 * n) >> 32, x0 = word 0 of Philox4x32-10 with counter (i, j & 0xffffffff, j >> 32, s + 1) and key
 * (seed & 0xffffffff, seed >> 32); pattern p takes the sites cum[p] <= u < cum[p+1].  T_s[j][k] = sum_p c_{s,j}[p] l_k[p] in pattern
 * order, a multiply then an add.  2 <= K <= 1024, 4 <= R <= 4096, 1 <= n_boot <= 10^6 (others: NNJ_ERR_INVALID).
 *   tips_dev       uint8  [R,L]      the one alignment's state masks, shared by every tree
 *   weights_dev    double [L]        pattern weights: non-negative integers, 0 < n < 2^31
 *   children_host  int32  [K,R-1,2]  the trees in join order; brlen_host double [K,2R-2], model_host double [K,64] as nnj_llh_eval
 *   llh_host       double [K]        L_k
 *   win_host       int32  [10,K]     win[s][k]: replicates of scale s whose largest T_s[j][.] is tree k's (every tied tree counts)
 *   kh_host        int32  [K]        replicates with a_{j,k*} - a_{j,k} >= L_k* - L_k, a_{j,k} = T_5[j][k] - m_k, m_k = (sum_j T_5[j][k]) / n_boot
 *   sh_host        int32  [K]        replicates with max_k' a_{j,k'} - a_{j,k} >= L_k* - L_k
 *   elw_host       double [K]        (sum_j q_{j,k}) / n_boot, q_{j,k} = e_k / sum_k' e_k' (k order), e_k = exp(T_5[j][k] - max_k' T_5[j][k'])
 *   site_llh_dev   double [K,L]      l_k[p] (device; may be NULL)
 * The sums over j run in replicate order.  Bad weights, an invalid tree: NNJ_ERR_INVALID; a workspace smaller than
 * nnj_llh_topotest_workspace_bytes(K, R, L, n_boot): NNJ_ERR_WORKSPACE.  Synchronises `stream`. */
int64_t nnj_llh_topotest_workspace_bytes(int K, int R, int L, int n_boot);
int nnj_llh_topology_test(const uint8_t* tips_dev, const double* weights_dev, const int32_t* children_host, const double* brlen_host,
                          const double* model_host, int K, int R, int L, uint64_t seed, int n_boot,
                          double* llh_host, int32_t* win_host, int32_t* kh_host, int32_t* sh_host, double* elw_host,
                          double* site_llh_dev, void* ws_dev, int64_t ws_bytes, void* stream);
/* Mean rates of the ncat equal-probability classes of Gamma(alpha, alpha) (Yang 1994): rates_host double [ncat]. */
int nnj_gamma_rates(double alpha, int ncat, double* rates_host);

/* ---- Pre-training loss, forward (SURVEY.md 8 f3; train.py:448-545, BALANCED_ELU_LOSS) over the logits trace of a teacher-forced rollout
 * (nnj_rollout with NNJ_SELECT_FORCED and a logits_trace buffer).  The backward pass is not part of this library.
 *   logits_trace_dev fp32  [B, trace_len]  step t at offset sum_{s<t} P_s, P_s = (R-s)(R-s-1)/2, trace_len = sum over all R-1 steps
 *   in_set_dev       uint8 [B, trace_len]  same layout: 1 = the pair is in the step's action set (train.py:30-39), 0 = complement
 *   margin 0.5 (train.py:478); ratio = max(1 - 3/80 * epoch / 2, 1/4) * cfgs.ratio_factor (train.py:495): per step the K = min(W, max(int(W*ratio), 8))
 *   largest complement scores enter the loss, W = the batch's widest complement of that step.
 *   out_dev          fp32  [R]  out[0] = loss (mean over the R-2 steps with more than one candidate), out[1] = precision (fraction of
 *                               (set, top-K complement) pairs ranked correctly), out[2+t] = loss of step t.
 * R <= 256; an action set holds at most R pairs (a tree has at most n/2 cherries) - a larger one yields NaN. */
int64_t nnj_rank_loss_workspace_bytes(int B, int R);
int nnj_rank_loss(const float* logits_trace_dev, const uint8_t* in_set_dev, int B, int R, float margin, double ratio,
                  float* out_dev, void* ws_dev, int64_t ws_bytes, void* stream);

/* ---- Bootstrap branch support (RAxML-NG --bootstrap / --support --bs-metric fbp,tbe; DESIGN.md 11).  No model handle or workspace:
 * both run on the current device, asynchronously on `stream`.
 * Replicate r of an alignment with l_eff real columns (the prefix; padded columns are the suffix): output column c < l_eff is input
 * column (x0 * l_eff) >> 32 (64-bit product), x0 = word 0 of Philox4x32-10 with counter (c, r & 0xffffffff, r >> 32, 0) and key
 * (seed & 0xffffffff, seed >> 32); columns c >= l_eff are copied unchanged.  A replicate depends only on (seed, r, l_eff).
 * Bootstrap replicates rep0 .. rep0+B-1 of one alignment: data int8 [R,L,4] -> out int8 [B,R,L,4] (both 4-byte aligned). */
int nnj_bootstrap_columns(const int8_t* data_dev, int R, int L, int l_eff, uint64_t seed, int64_t rep0, int B,
                          int8_t* out_dev, void* stream);
/* Transfer distance of S reference splits (leaf bitsets uint64 [S, ceil(R/64)], either side; bit t of word t/64 = taxon t) to each of
 * B NJ trees (merges int32 [B,R-1,2], the slot rule of nnj_rollout): dist int32 [B,S],
 *   dist = min(p-1, min over the tree's R-2 non-root clades c of min(|A ^ c|, R - |A ^ c|)),  p = size of the split's lighter side;
 * a row of -1 = that merge list is not valid (an entry (i, j) of step t that is not 0 <= i < j < R-t).  4 <= R <= 512, S >= 0.
 * The 512 is this primitive's own limit: it takes merge lists from any source.  Replicate trees from nnj_rollout stop at 400 taxa,
 * the limit of the encoder's column attention, so a whole bootstrap does too. */
int nnj_split_distances(const int32_t* merges_dev, int B, int R, const uint64_t* splits_dev, int S, int32_t* dist_dev, void* stream);

/* Building block of the tensor-core path (precision NNJ_PREC_BF16X3), exposed for unit tests and reuse:
 * C[z] = A[z] * B[z]^T with fp32 A [Z,M,K], B [Z,N,K], C [Z,M,N]; operands are split into bf16 hi/lo planes and
 * multiplied on tcgen05 as hi*hi + hi*lo + lo*hi with fp32 accumulation in TMEM.  K must be a multiple of 8;
 * ws needs 4*(Z*M*K + Z*N*K) + 2048 bytes.  Replaces the einsum contractions of axial_attention.py:97,114. */
int nnj_gemm_split_bf16(const float* A_dev, const float* B_dev, float* C_dev, int Z, int M, int N, int K,
                        void* ws_dev, int64_t ws_bytes, void* stream);

/* Hardware self-test of the operand forms used inside the fused tensor-core kernels: D [128,N] = A [128,64] * B [64,N]
 * (N = 64 or 128) with A written K-major / B written MN-major into SWIZZLE_128B shared memory by threads (no TMA),
 * split-bf16; N = 128 exercises the leading-byte-offset form of the MN-major descriptor. */
int nnj_tc_selftest(const float* A_dev, const float* B_dev, float* D_dev, int N, void* stream);

/* Optional per-kernel-class timing with CUDA events recorded on the launching stream (used by bench.py for the
 * roofline numbers).  enable(1) clears and starts recording on the calling thread, enable(0) stops.
 * read() synchronises the device and returns summed milliseconds / launch counts per class. */
int nnj_profile_enable(int on);
int nnj_profile_classes(void);
const char* nnj_profile_name(int cls);
int nnj_profile_read(int n, double* ms, int64_t* launches);

/* Number of kernel launches issued by this library on the calling thread since the last reset. */
int64_t nnj_launch_count(int reset);

#ifdef __cplusplus
}
#endif
#endif /* NNJ_H_ */
