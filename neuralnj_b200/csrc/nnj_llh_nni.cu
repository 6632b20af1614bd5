// nnj_llh_nni.cu — likelihood branch support of a fixed tree: the two NNI alternatives of every internal branch, each with its
// five quartet lengths optimised, and RELL replicates of the per-pattern log-likelihoods for SH-aLRT and the local bootstrap
// probability.  DESIGN.md section 12 gives the definitions; oracle/alrt_oracle.py restates them in numpy.
//
// 1. llh_prepare (nnj_llh.cu), k_llh with one CTA per tree: subtree vectors D, the U pass of the build_ops schedule (its UP and
//    SWAPROOT rows) and the per-pattern log-likelihoods l0 at the given lengths.
// 2. k_llh_nni, one CTA per (tree, internal branch, alternative), threads over patterns.  The quartet around the branch above v has
//    the outer vectors A = D[a], B = D[b] (children of v), C = D[s] (sibling of v) and D = U[p] (parent of v), or for the root
//    branch the two children of the other root child.  Alternative 1 pairs (A, C | B, D), alternative 2 (A, D | B, C).  Rounds of
//    Newton on the central branch and on A, B, C, D (the vector opposite a branch rebuilt from the current lengths, per pattern in
//    registers, into the CTA's own sumtable) stop after the first round that gains < 1e-3, or after 8.  D and U are read-only.
// 3. k_rell_counts: one thread per (tree, replicate, draw) adds 1 to the count of the drawn pattern, c[b][p][r]; k_rell: one thread
//    per (tree, branch, replicate) forms the three resampled sums in pattern order and adds integer SH and LBP counts per branch.
// All reductions have a fixed order: results are bit-reproducible.
#include "nnj_internal.h"
#include "nnj_llh.cuh"

namespace nnj {

namespace {

constexpr int NNI_MAX_ROUNDS = 8;
constexpr double NNI_EPS = 1e-3;
constexpr double SH_TOL = 0.05;
constexpr int RELL_CHUNK = 256;          // replicates per pass of the two RELL kernels (the counts c[b][p][r] live in the workspace)

struct NniArgs {
    const uint8_t* tips;        // [B][R][L]
    const double* weights;      // [B][L]
    const double* model;        // [B][LLH_MODEL]
    const double *D, *U, *inv;  // llh_prepare results: [B][R-1][L][16], [B][2R-2][L][16], [B][L]
    const int32_t *Dn, *Un;
    const int32_t* qnode;       // [B][nb][4] A, B, C, D: node id of a subtree vector (tip or D), or -(p + 1) for U[p]
    const double* qlen;         // [B][nb][5] central, A, B, C, D at the tree's (clamped) lengths
    double* S; int32_t* Sn;     // [B][nb][2][L][16], [B][nb][2][L]: each CTA's sumtable
    const double* site0;        // [B][L] l0
    double* site;               // [B][nb][3][L] l0, l1, l2
    double* llh;                // [B][nb][2] L1, L2
    double* len;                // [B][nb][2][5] optimised central, A, B, C, D
    int R, L, nb;
};

__global__ void __launch_bounds__(LLH_THREADS) k_llh_nni(const NniArgs a) {
    __shared__ double mdl[LLH_MODEL], Pm[5 * 64], red[66], ek[48], tq[5];
    const int item = blockIdx.x, alt = item & 1, bi = item >> 1, b = bi / a.nb;
    const int tid = threadIdx.x, R = a.R, L = a.L;
    const uint8_t* tips = a.tips + (size_t)b * R * L;
    const double* wts = a.weights + (size_t)b * L;
    const double* invt = a.inv + (size_t)b * L;
    const double* Dt = a.D + (size_t)b * (R - 1) * L * 16;
    const int32_t* Dnt = a.Dn + (size_t)b * (R - 1) * L;
    const double* Ut = a.U + (size_t)b * (2 * R - 2) * L * 16;
    const int32_t* Unt = a.Un + (size_t)b * (2 * R - 2) * L;
    double* St = a.S + (size_t)item * L * 16;
    int32_t* Snt = a.Sn + (size_t)item * L;
    double* site = a.site + ((size_t)bi * 3 + 1 + alt) * L;
    int q[5];                   // q[e] = source of the vector of quartet edge e = 1..4 (A, B, C, D)
#pragma unroll
    for (int e = 1; e < 5; ++e) q[e] = a.qnode[(size_t)bi * 4 + e - 1];
    if (tid < LLH_MODEL) mdl[tid] = a.model[(size_t)b * LLH_MODEL + tid];
    if (tid < 5) tq[tid] = a.qlen[(size_t)bi * 5 + tid];
    __syncthreads();
    const double pinv = mdl[MDL_PINV], wk = (1.0 - pinv) * 0.25;
    for (int e = 0; e < 5; ++e) pmat1(Pm + 64 * e, mdl, tq[e]);
    // the two sides of the central branch: X = (edge 1, x2), Y = (edge 2, y2); alternative 1 is AC|BD, alternative 2 AD|BC
    const int x2 = alt ? 4 : 3, y2 = alt ? 3 : 4;
    auto load = [&](int e, int s, double (&x)[16]) -> int {
        const int v = q[e];
        if (v >= 0) { clv_load(R, L, Dt, tips, v, s, x); return cnt_load(R, L, Dnt, v, s); }
        vec_load(Ut + ((size_t)(-v - 1) * L + s) * 16, x);
        return Unt[(size_t)(-v - 1) * L + s];
    };
    // (P(t_e) vec_e) * (P(t_f) vec_f), scaled; returns its count
    auto half = [&](int e, int f, int s, double (&out)[16]) -> int {
        double x[16], y[16];
        int n = load(e, s, x) + load(f, s, y);
        pm_apply(Pm + 64 * e, x, out);
        pm_apply(Pm + 64 * f, y, x);
        return n + mul_scaled(out, x);
    };
    // log L of the alternative at the current lengths, at the central branch; writes the sites
    auto evaluate = [&]() {
        double acc = 0.0, dummy = 0.0;
        for (int s = tid; s < L; s += LLH_THREADS) {
            double X[16], Y[16], p1[16];
            const int n = half(1, x2, s, X) + half(2, y2, s, Y);
            pm_apply(Pm, X, p1);
            const double st = site_loglik(mdl, p1, Y, n, wk, pinv, invt[s]);
            site[s] = st;
            acc += wts[s] * st;
        }
        block_sum2(acc, dummy, red);
        return acc;
    };
    // Newton on quartet edge e from its current length; the vector opposite it is rebuilt per pattern from the current lengths
    auto newton_edge = [&](int e) {
        for (int s = tid; s < L; s += LLH_THREADS) {
            double u[16], d[16], sv[16];
            int n;
            if (e == 0) {
                n = half(2, y2, s, u) + half(1, x2, s, d);
            } else {
                // e's partner f on its side, and the pair (g, h) across the central branch
                const bool xs = e == 1 || e == x2;
                const int f = e == 1 ? x2 : (e == x2 ? 1 : (e == 2 ? y2 : 2));
                const int g = xs ? 2 : 1, h = xs ? y2 : x2;
                double o[16];
                n = half(g, h, s, o);
                pm_apply(Pm, o, d);                   // d: P(t_central) o, for the moment
                n += load(f, s, o);
                pm_apply(Pm + 64 * f, o, u);
                n += mul_scaled(u, d);
                n += load(e, s, d);
            }
            sumtable_row(mdl, u, d, sv);
            vec_store(St + (size_t)s * 16, sv);
            Snt[s] = n;
        }
        const double tv = newton_brlen(St, Snt, mdl, ek, red, wts, invt, pinv, wk, L, tq[e]);
        if (tid == 0) tq[e] = tv;
        __syncthreads();
        pmat1(Pm + 64 * e, mdl, tv);
    };
    double ll = evaluate();
    for (int round = 0; round < NNI_MAX_ROUNDS; ++round) {
        for (int e = 0; e < 5; ++e) newton_edge(e);
        const double nl = evaluate();
        const double gain = nl - ll;
        ll = nl;
        if (gain < NNI_EPS) break;
    }
    if (tid == 0) a.llh[(size_t)bi * 2 + alt] = ll;
    if (tid < 5) a.len[((size_t)bi * 2 + alt) * 5 + tid] = tq[tid];
    if (alt == 0) {
        double* s0 = a.site + (size_t)bi * 3 * L;
        for (int s = tid; s < L; s += LLH_THREADS) s0[s] = a.site0[(size_t)b * L + s];
    }
}

// one thread per (tree, branch, replicate): Lk* = sum_p c[p] lk[p] and Lk = sum_p w[p] lk[p] in pattern order, multiply then add
__global__ void __launch_bounds__(RELL_THREADS) k_rell(const int32_t* __restrict__ cnt, const double* __restrict__ weights, const double* __restrict__ site,
                                                       int B, int nb, int L, int nr, int32_t* __restrict__ sh, int32_t* __restrict__ lbp) {
    const size_t idx = (size_t)blockIdx.x * RELL_THREADS + threadIdx.x;
    if (idx >= (size_t)B * nb * nr) return;
    const int rl = (int)(idx % nr);
    const size_t bi = idx / nr;
    const int b = (int)(bi / nb);
    const double* l0 = site + bi * 3 * L;
    const double* l1 = l0 + L;
    const double* l2 = l1 + L;
    const double* w = weights + (size_t)b * L;
    const int32_t* c = cnt + (size_t)b * L * nr + rl;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, w0 = 0.0, w1 = 0.0, w2 = 0.0;
    for (int p = 0; p < L; ++p) {
        const double cp = (double)c[(size_t)p * nr], wp = w[p], a0 = l0[p], a1 = l1[p], a2 = l2[p];
        s0 = __dadd_rn(s0, __dmul_rn(cp, a0)); s1 = __dadd_rn(s1, __dmul_rn(cp, a1)); s2 = __dadd_rn(s2, __dmul_rn(cp, a2));
        w0 = __dadd_rn(w0, __dmul_rn(wp, a0)); w1 = __dadd_rn(w1, __dmul_rn(wp, a1)); w2 = __dadd_rn(w2, __dmul_rn(wp, a2));
    }
    const double delta = w0 - fmax(w1, w2);
    const double c0 = s0 - w0, c1 = s1 - w1, c2 = s2 - w2;
    const double m1 = fmax(c0, fmax(c1, c2)), m2 = fmax(fmin(c0, c1), fmin(fmax(c0, c1), c2));     // largest, second largest
    if (delta > (m1 - m2) + SH_TOL) atomicAdd(sh + bi, 1);
    if (s0 >= fmax(s1, s2)) atomicAdd(lbp + bi, 1);
}

struct SupBuffers {
    double* S; int32_t* Sn;             // each CTA's sumtable
    double *site, *site0;               // per-pattern log-likelihoods (when the caller passes no site_dev) and l0
    int32_t* qnode; double *qlen, *model, *llh, *len;
    uint32_t* cum; int32_t *cnt, *sh, *lbp;
    size_t total;
};
static SupBuffers sup_layout(char* base, int B, int R, int L, int n_rell) {
    const size_t nb = R > 3 ? (size_t)(R - 3) : 0, items = (size_t)B * nb * 2;
    const size_t chunk = n_rell < RELL_CHUNK ? (size_t)(n_rell > 0 ? n_rell : 1) : RELL_CHUNK;
    WsCarver c(base);
    SupBuffers w;
    w.S = c.take<double>(items * L * 16); w.Sn = c.take<int32_t>(items * L);
    w.site = c.take<double>((size_t)B * nb * 3 * L); w.site0 = c.take<double>((size_t)B * L);
    w.qnode = c.take<int32_t>((size_t)B * nb * 4); w.qlen = c.take<double>((size_t)B * nb * 5); w.model = c.take<double>((size_t)B * LLH_MODEL);
    w.llh = c.take<double>(items); w.len = c.take<double>(items * 5);
    w.cum = c.take<uint32_t>((size_t)B * (L + 1)); w.cnt = c.take<int32_t>((size_t)B * L * chunk);
    w.sh = c.take<int32_t>((size_t)B * nb); w.lbp = c.take<int32_t>((size_t)B * nb);
    w.total = c.off + 256;
    return w;
}

}  // namespace

size_t llh_support_ws_bytes(int B, int R, int L, int n_rell) { return llh_ws_bytes(B, R, L) + sup_layout(nullptr, B, R, L, n_rell).total; }

int run_llh_support(const LlhTrees& in, uint64_t seed, int64_t rep0, int n_rell, int32_t* branch_node_h, double* llh_h, double* nni_brlen_h,
                    int32_t* sh_h, int32_t* lbp_h, double* site_dev, void* ws, size_t ws_bytes, cudaStream_t st) {
    const int B = in.B, R = in.R, L = in.L, nb = R - 3;
    const int32_t* children_h = in.children;
    const size_t base = llh_ws_bytes(B, R, L);
    if (ws_bytes < base + sup_layout(nullptr, B, R, L, n_rell).total) return set_error(NNJ_ERR_WORKSPACE, "llh_branch_support: workspace too small (nnj_llh_support_workspace_bytes)");
    // ---- host checks: trees, integral weights (the RELL draws pick sites, and a pattern of weight w is w sites)
    for (int b = 0; b < B; ++b)
        if (llh_check_tree(children_h + (size_t)b * (R - 1) * 2, R)) return set_error(NNJ_ERR_INVALID, "llh_branch_support: children is not a binary tree in join order");
    std::vector<double> w((size_t)B * L);
    cudaError_t e = cudaMemcpyAsync(w.data(), in.weights, w.size() * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    std::vector<uint32_t> cum((size_t)B * (L + 1));
    uint32_t nmax = 0;
    for (int b = 0; b < B; ++b) {
        uint64_t acc = 0;
        cum[(size_t)b * (L + 1)] = 0;
        for (int p = 0; p < L; ++p) {
            const double x = w[(size_t)b * L + p];
            if (!(x >= 0.0 && x <= 2147483647.0) || x != floor(x)) return set_error(NNJ_ERR_INVALID, "llh_branch_support: pattern weights must be non-negative integers");
            acc += (uint64_t)x;
            if (acc > 2147483647ull) return set_error(NNJ_ERR_INVALID, "llh_branch_support: more than 2^31 - 1 sites");
            cum[(size_t)b * (L + 1) + p + 1] = (uint32_t)acc;
        }
        if (acc == 0 && n_rell > 0) return set_error(NNJ_ERR_INVALID, "llh_branch_support: every pattern weight is 0");
        nmax = acc > nmax ? (uint32_t)acc : nmax;
    }
    if (nb <= 0) return NNJ_OK;
    // ---- quartets of the internal branches, in increasing v (DESIGN.md 12), at the lengths k_llh uses
    std::vector<int32_t> qnode((size_t)B * nb * 4);
    std::vector<double> qlen((size_t)B * nb * 5);
    for (int b = 0; b < B; ++b) {
        const int32_t* ch = children_h + (size_t)b * (R - 1) * 2;
        std::vector<int> parent(2 * R - 1, -1);
        for (int k = 0; k < R - 1; ++k) { parent[ch[2 * k]] = R + k; parent[ch[2 * k + 1]] = R + k; }
        std::vector<double> t(2 * R - 2);
        for (int v = 0; v < 2 * R - 2; ++v) t[v] = clampd(in.brlen[(size_t)b * (2 * R - 2) + v], BRLEN_MIN, BRLEN_MAX);
        const int root = 2 * R - 2, c1 = ch[2 * (R - 2)], c2 = ch[2 * (R - 2) + 1];
        t[c1] = t[c2] = clampd(t[c1] + t[c2], BRLEN_MIN, BRLEN_MAX);
        int i = 0;
        for (int v = R; v < root; ++v) {
            const int p = parent[v];
            if (p == root && !(v == c1 && c2 >= R)) continue;
            const size_t bi = (size_t)b * nb + i++;
            const int a = ch[2 * (v - R)], bb = ch[2 * (v - R) + 1];
            int c, d, cd, dd;                // C, D and the nodes whose lengths they carry
            if (p == root) { c = ch[2 * (c2 - R)]; d = ch[2 * (c2 - R) + 1]; cd = c; dd = d; }
            else {
                c = ch[2 * (p - R)] == v ? ch[2 * (p - R) + 1] : ch[2 * (p - R)];
                cd = c; dd = p; d = -(p + 1);
            }
            branch_node_h[bi] = v;
            qnode[bi * 4 + 0] = a; qnode[bi * 4 + 1] = bb; qnode[bi * 4 + 2] = c; qnode[bi * 4 + 3] = d;
            qlen[bi * 5 + 0] = t[v]; qlen[bi * 5 + 1] = t[a]; qlen[bi * 5 + 2] = t[bb]; qlen[bi * 5 + 3] = t[cd]; qlen[bi * 5 + 4] = t[dd];
        }
        if (i != nb) return set_error(NNJ_ERR_INVALID, "llh_branch_support: internal error (branch count)");
    }
    const SupBuffers sw = sup_layout(ws_align(static_cast<char*>(ws) + base), B, R, L, n_rell);
    // ---- 1. subtree vectors, the U pass and l0
    std::vector<double> l0_tree(B);
    const LlhPrepared pre = llh_prepare(in, sw.site0, l0_tree.data(), ws, base, st);
    if (pre.rc) return pre.rc;
    // ---- 2. the NNI quartets
    e = cudaMemcpyAsync(sw.qnode, qnode.data(), qnode.size() * 4, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(sw.qlen, qlen.data(), qlen.size() * 8, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(sw.model, in.model, (size_t)B * LLH_MODEL * 8, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(sw.cum, cum.data(), cum.size() * 4, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(sw.sh, 0, (size_t)B * nb * 4, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(sw.lbp, 0, (size_t)B * nb * 4, st);
    if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    NniArgs a;
    a.tips = in.tips; a.weights = in.weights; a.model = sw.model;
    a.D = pre.D; a.U = pre.U; a.inv = pre.inv; a.Dn = pre.Dn; a.Un = pre.Un;
    a.qnode = sw.qnode; a.qlen = sw.qlen; a.S = sw.S; a.Sn = sw.Sn; a.site0 = sw.site0; a.site = site_dev ? site_dev : sw.site;
    a.llh = sw.llh; a.len = sw.len; a.R = R; a.L = L; a.nb = nb;
    prof_begin(KC_LLH, st);
    k_llh_nni<<<B * nb * 2, LLH_THREADS, 0, st>>>(a);
    ++g_launches; prof_end(st);
    e = cudaGetLastError();
    if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    // ---- 3. RELL, in chunks of replicates
    for (int r0 = 0; r0 < n_rell; r0 += RELL_CHUNK) {
        const int nr = n_rell - r0 < RELL_CHUNK ? n_rell - r0 : RELL_CHUNK;
        e = cudaMemsetAsync(sw.cnt, 0, (size_t)B * L * nr * 4, st);
        if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
        const dim3 grid((nmax + RELL_THREADS - 1) / RELL_THREADS, B * nr < 65535 ? B * nr : 65535);
        prof_begin(KC_LLH, st);
        k_rell_counts<<<grid, RELL_THREADS, 0, st>>>(sw.cum, B, L, seed, rep0 + r0, nr, 0u, 0u, sw.cnt);
        ++g_launches; prof_end(st);
        const size_t threads = (size_t)B * nb * nr;
        prof_begin(KC_LLH, st);
        k_rell<<<(unsigned)((threads + RELL_THREADS - 1) / RELL_THREADS), RELL_THREADS, 0, st>>>(sw.cnt, in.weights, a.site, B, nb, L, nr, sw.sh, sw.lbp);
        ++g_launches; prof_end(st);
        e = cudaGetLastError();
        if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    }
    // ---- results
    std::vector<double> l12((size_t)B * nb * 2);
    e = cudaMemcpyAsync(l12.data(), sw.llh, l12.size() * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(nni_brlen_h, sw.len, (size_t)B * nb * 10 * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(sh_h, sw.sh, (size_t)B * nb * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(lbp_h, sw.lbp, (size_t)B * nb * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    for (size_t bi = 0; bi < (size_t)B * nb; ++bi) {
        llh_h[bi * 3] = l0_tree[bi / nb];
        llh_h[bi * 3 + 1] = l12[bi * 2];
        llh_h[bi * 3 + 2] = l12[bi * 2 + 1];
    }
    return NNJ_OK;
}

}  // namespace nnj
