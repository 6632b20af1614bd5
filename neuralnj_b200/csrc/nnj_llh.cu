// nnj_llh.cu — tree log-likelihood under GTR+I+G4 and its maximisation over branch lengths (SURVEY.md 8 f2).
//
// Replaces, for Search / branch_optimize scoring, the reference's native binding raxmlpy.compute_llh / optimize_brlen
// (RAxMLpy/cpp/raxmlpy.cpp:1749-1872 -> raxml-ng TreeInfo::loglh / optimize_branches; call sites environment.py:365-379,625-670,
// finetune_rl_search.py:401-411).  raxml-ng / libpll are git-cloned by the reference's setup.py and are not available: the
// algorithm is the published one (Felsenstein pruning; Yang's discrete gamma, class means; invariant-site mixture; Newton-Raphson
// per branch on the eigen-space sumtable, branches swept depth-first with the conditional likelihood vectors refreshed on the way),
// restated on the CPU in oracle/llh_oracle.py - parity against raxml-ng itself is UNPINNED (DESIGN.md).
//
// One CTA per tree, threads over alignment patterns, everything in fp64 (log-likelihoods of ~1e4 with gains of ~1e-3 per pass).
// Conditional likelihood vectors (CLVs) [node][pattern][4 rate classes][4 states] live in the caller's workspace: D[v] = subtree
// below v, U[v] = everything else, seen from the parent end of the branch above v.  A thread owns its patterns through the whole
// traversal, so the only block-wide steps are the 4 x 4 transition matrices of an operation (64 threads, then a barrier) and
// the reductions of the Newton iteration (fixed order: results are bit-reproducible).
// Node numbering: leaves 0..R-1, inner node R+k = k-th join (children[k]), root = the last; brlen[v] = branch above v.
// Scaling: site likelihoods of a few hundred taxa and more underflow fp64.  When all 16 entries of a freshly combined
// (node, pattern) vector are below 2^-256 the vector is multiplied by 2^256 and an int32 count of that (node, pattern) goes
// up by one; counts add along the tree like the vectors (D(v) = D(a) + D(b) + own, U(c) = U(parent) + D(sibling) + own) and
// copies carry theirs.  The root takes log(wk l) - 256 n ln 2, or log(ldexp(wk l, -256 n) + p_inv inv) where there is an
// invariant term; Newton scales the invariant term up by 2^(256 n) instead.  Powers of two are exact, so wherever n = 0 the
// arithmetic is the unscaled one, bit for bit.  The CPU restatement (oracle/llh_oracle.py) applies the same rule.
#include "nnj_internal.h"
#include "nnj_llh.cuh"

namespace nnj {

constexpr double RATE_LO = 1e-3, RATE_HI = 1e3, ALPHA_LO = 0.02, ALPHA_HI = 100.0, PINV_HI = 0.99, GOLD = 0.3819660112501051;   // as in oracle/llh_oracle.py
constexpr int GOLDEN_ITERS = 24;          // golden-section steps per model parameter and round (LlhMode::All)
enum { OP_OPT = 0, OP_UP = 1, OP_DOWN = 2, OP_SWAPROOT = 3 };

struct LlhArgs {
    const uint8_t* tips;        // [B][R][L] 4-bit state masks
    const double* weights;      // [B][L] pattern multiplicities
    const int32_t* children;    // [B][R-1][2]
    const int32_t* ops;         // [B][n_ops][4] (Brlen, All: the build_ops schedule; Prepare: its UP and SWAPROOT rows)
    double* brlen;              // [B][2R-2] in / out
    const double* model;        // [B][LLH_MODEL]
    double *D, *U, *S, *inv;    // workspace: [B][R-1][L][16], [B][2R-2][L][16], [B][L][16], [B][L]
    int32_t *Dn, *Un, *Sn;      // scale counts of D, U and the Newton sumtable: [B][R-1][L], [B][2R-2][L], [B][L]
    double* llh;                // [B][2]: before, after
    double* site;               // [B][L] per-pattern log-likelihood at the given lengths (Prepare), else null
    int B, R, L, n_ops, max_passes;
    LlhMode mode;
    double eps;
    double lh_eps; int max_rounds, golden_iters;  // All: rounds of (free parameters one at a time, branch sweeps) until a round gains < lh_eps
    double* model_out;                            // [B][LLH_MODEL] optimised model (All)
};

// ---- discrete gamma (Yang 1994), on the host (gamma_rates) and, for LlhMode::All, on the device (rebuild_model)
// regularised lower incomplete gamma P(a, x): series / continued fraction (Lentz)
__host__ __device__ double gammp(double a, double x) {
    if (x <= 0.0) return 0.0;
    const double gln = lgamma(a);
    if (x < a + 1.0) {
        double ap = a, sum = 1.0 / a, del = sum;
        for (int n = 0; n < 2000; ++n) { ap += 1.0; del *= x / ap; sum += del; if (fabs(del) < fabs(sum) * 1e-17) break; }
        return sum * exp(-x + a * log(x) - gln);
    }
    double b = x + 1.0 - a, c = 1e300, d = 1.0 / b, h = d;
    for (int i = 1; i < 2000; ++i) {
        const double an = -i * (i - a);
        b += 2.0;
        d = an * d + b; if (fabs(d) < 1e-300) d = 1e-300;
        c = b + an / c; if (fabs(c) < 1e-300) c = 1e-300;
        d = 1.0 / d;
        const double del = d * c;
        h *= del;
        if (fabs(del - 1.0) < 1e-17) break;
    }
    return 1.0 - exp(-x + a * log(x) - gln) * h;
}
// class boundary: the quantile x of Gamma(alpha, 1) at q (Newton on P(alpha, x), monotone with a known density, kept inside a
// bracket: a bisection step whenever Newton leaves it), then P(alpha + 1, x), the share of the mean below x
__host__ __device__ double gamma_class_cdf(double alpha, double q) {
    const double gln = lgamma(alpha);
    double lo = 0.0, hi = alpha + 1.0;
    while (gammp(alpha, hi) < q) hi *= 2.0;
    double x = 0.5 * (lo + hi);
    for (int it = 0; it < 200; ++it) {
        const double f = gammp(alpha, x) - q;
        if (f < 0.0) lo = x; else hi = x;
        const double pdf = exp((alpha - 1.0) * log(x) - x - gln);
        double xn = pdf > 0.0 ? x - f / pdf : 0.5 * (lo + hi);
        if (!(xn > lo && xn < hi)) xn = 0.5 * (lo + hi);
        const bool done = fabs(xn - x) <= 1e-15 * x || hi - lo <= 1e-300;
        x = xn;
        if (done) break;
    }
    return gammp(alpha + 1.0, x);
}

// ---- model parameters on the device (LlhMode::All): one thread rebuilds the eigen-system and the class rates of its tree
// mdl: raw parameters (GTR rates, freqs, alpha) -> eigenvalues, U, U^-1, class rates.
// Threads 0 (eigen-system: cyclic Jacobi on the symmetrised rate matrix) and 1..3 (class boundaries) work, then a barrier.
__device__ void rebuild_model(double* mdl, double* scratch /* 4 doubles */, bool eigen, bool gamma) {
    const int tid = threadIdx.x;
    if (tid == 0 && eigen) {
        const double* pi = mdl + MDL_FREQ;
        const double* g = mdl + MDL_GTR;
        double r[4][4] = {{0, g[0], g[1], g[2]}, {g[0], 0, g[3], g[4]}, {g[1], g[3], 0, g[5]}, {g[2], g[4], g[5], 0}};
        double Q[4][4], S[4][4], V[4][4];
        double norm = 0.0;
        for (int a = 0; a < 4; ++a) {
            double d = 0.0;
            for (int c = 0; c < 4; ++c) { Q[a][c] = r[a][c] * pi[c]; if (c != a) d += Q[a][c]; }
            Q[a][a] = -d;
            norm += pi[a] * d;
        }
        for (int a = 0; a < 4; ++a)
            for (int c = 0; c < 4; ++c) { S[a][c] = sqrt(pi[a]) * Q[a][c] / (norm * sqrt(pi[c])); V[a][c] = a == c ? 1.0 : 0.0; }
        for (int a = 0; a < 4; ++a)
            for (int c = a + 1; c < 4; ++c) { const double m = 0.5 * (S[a][c] + S[c][a]); S[a][c] = m; S[c][a] = m; }
        double diag2 = 0.0;
        for (int p = 0; p < 4; ++p) diag2 += S[p][p] * S[p][p];
        for (int sweep = 0; sweep < 16; ++sweep) {           // quadratic convergence: 5-6 sweeps reach the rounding level of a 4 x 4 matrix
            double off = 0.0;
            for (int p = 0; p < 4; ++p) for (int q = p + 1; q < 4; ++q) off += S[p][q] * S[p][q];
            if (off < 1e-31 * diag2) break;
            for (int p = 0; p < 4; ++p)
                for (int q = p + 1; q < 4; ++q) {
                    if (fabs(S[p][q]) < 1e-300) continue;
                    const double theta = (S[q][q] - S[p][p]) / (2.0 * S[p][q]);
                    const double tt = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                    const double cs = 1.0 / sqrt(tt * tt + 1.0), sn = tt * cs;
                    for (int k = 0; k < 4; ++k) { const double skp = S[k][p], skq = S[k][q]; S[k][p] = cs * skp - sn * skq; S[k][q] = sn * skp + cs * skq; }
                    for (int k = 0; k < 4; ++k) { const double spk = S[p][k], sqk = S[q][k]; S[p][k] = cs * spk - sn * sqk; S[q][k] = sn * spk + cs * sqk; }
                    for (int k = 0; k < 4; ++k) { const double vkp = V[k][p], vkq = V[k][q]; V[k][p] = cs * vkp - sn * vkq; V[k][q] = sn * vkp + cs * vkq; }
                }
        }
        for (int j = 0; j < 4; ++j) mdl[MDL_LAM + j] = S[j][j];
        for (int a = 0; a < 4; ++a)
            for (int j = 0; j < 4; ++j) { mdl[MDL_U + a * 4 + j] = V[a][j] / sqrt(pi[a]); mdl[MDL_UINV + j * 4 + a] = V[a][j] * sqrt(pi[a]); }
    }
    if (gamma && tid >= 1 && tid <= 3) scratch[tid] = gamma_class_cdf(mdl[MDL_ALPHA], (double)tid * 0.25);   // boundaries of classes 0..2
    __syncthreads();
    if (gamma && tid == 0) {
        scratch[0] = 0.0;
        const double c4 = 1.0;
        double* rate = mdl + MDL_RATE;
        rate[0] = 4.0 * (scratch[1] - 0.0); rate[1] = 4.0 * (scratch[2] - scratch[1]); rate[2] = 4.0 * (scratch[3] - scratch[2]); rate[3] = 4.0 * (c4 - scratch[3]);
    }
    __syncthreads();
}

__global__ void __launch_bounds__(LLH_THREADS) k_llh(const LlhArgs a) {
    extern __shared__ double sm_d[];
    double* mdl = sm_d;                 // [48]
    double* Pm = mdl + LLH_MODEL;       // [2][4][16]
    double* red = Pm + 128;             // [66]
    double* ek = red + 66;              // [3][16]: exp(rate t), rate, rate^2 of the Newton iteration
    double* t = ek + 48;                // [2R-2]
    const int b = blockIdx.x, tid = threadIdx.x, R = a.R, L = a.L;
    const uint8_t* tips = a.tips + (size_t)b * R * L;
    const double* wts = a.weights + (size_t)b * L;
    const int32_t* ch = a.children + (size_t)b * (R - 1) * 2;
    double* Dt = a.D + (size_t)b * (R - 1) * L * 16;
    double* Ut = a.U + (size_t)b * (2 * R - 2) * L * 16;
    double* St = a.S + (size_t)b * L * 16;
    double* invt = a.inv + (size_t)b * L;
    int32_t* Dnt = a.Dn + (size_t)b * (R - 1) * L;
    int32_t* Unt = a.Un + (size_t)b * (2 * R - 2) * L;
    int32_t* Snt = a.Sn + (size_t)b * L;
    if (tid < LLH_MODEL) mdl[tid] = a.model[(size_t)b * LLH_MODEL + tid];
    for (int v = tid; v < 2 * R - 2; v += LLH_THREADS) t[v] = clampd(a.brlen[(size_t)b * (2 * R - 2) + v], BRLEN_MIN, BRLEN_MAX);
    __syncthreads();
    const int c1 = ch[(R - 2) * 2], c2 = ch[(R - 2) * 2 + 1];
    if (tid == 0) { const double t0 = clampd(t[c1] + t[c2], BRLEN_MIN, BRLEN_MAX); t[c1] = t0; t[c2] = t0; }   // the root branch, stored at both ends
    __syncthreads();
    double pinv = mdl[MDL_PINV], wk = (1.0 - pinv) * 0.25;      // re-read after every change of the model (All)
    // invariant-site term: pi_x where every tip of the pattern is compatible with exactly one state x
    for (int s = tid; s < L; s += LLH_THREADS) {
        int m = 15;
        for (int v = 0; v < R; ++v) m &= tips[(size_t)v * L + s];
        invt[s] = (m != 0 && (m & (m - 1)) == 0) ? mdl[MDL_FREQ + (31 - __clz(m))] : 0.0;      // times p_inv where it is used
    }
    // ---- subtree vectors, children before parents (join order); the virtual root itself is never needed
    // dst = (P(t_x) X) * (P(t_y) D[y]) with X = D[x], or U[x] when xsrc_U is given; scaled as described at the top
    auto combine = [&](int x, int y, double* dst_base /* [L][16] */, int32_t* dst_n /* [L] */, const double* xsrc_U, const int32_t* xsrc_Un) {
        pmat2(Pm, mdl, t[x], t[y]);
        for (int s = tid; s < L; s += LLH_THREADS) {
            double vx[16], vy[16], px[16], py[16];
            if (xsrc_U) vec_load(xsrc_U + (size_t)s * 16, vx); else clv_load(R, L, Dt, tips, x, s, vx);
            clv_load(R, L, Dt, tips, y, s, vy);
            int n = (xsrc_U ? xsrc_Un[s] : cnt_load(R, L, Dnt, x, s)) + cnt_load(R, L, Dnt, y, s);
            pm_apply(Pm, vx, px);
            pm_apply(Pm + 64, vy, py);
            n += mul_scaled(px, py);
            vec_store(dst_base + (size_t)s * 16, px);
            dst_n[s] = n;
        }
        __syncthreads();      // Pm is rewritten by the next operation
    };
    auto down_pass = [&]() {
        for (int k = 0; k < R - 2; ++k) combine(ch[2 * k], ch[2 * k + 1], Dt + (size_t)k * L * 16, Dnt + (size_t)k * L, nullptr, nullptr);
    };
    down_pass();
    auto root_loglik = [&]() {
        pmat2(Pm, mdl, t[c1], 0.0);
        double acc = 0.0, dummy = 0.0;
        for (int s = tid; s < L; s += LLH_THREADS) {
            double v1[16], v2[16], p1[16];
            clv_load(R, L, Dt, tips, c1, s, v1);
            clv_load(R, L, Dt, tips, c2, s, v2);
            pm_apply(Pm, v1, p1);
            const int n = cnt_load(R, L, Dnt, c1, s) + cnt_load(R, L, Dnt, c2, s);
            const double site = site_loglik(mdl, p1, v2, n, wk, pinv, invt[s]);
            acc += wts[s] * site;
            if (a.site) a.site[(size_t)b * L + s] = site;
        }
        block_sum2(acc, dummy, red);
        return acc;
    };
    double ll = root_loglik();
    const double ll0 = ll;
    const int32_t* ops = a.ops + (size_t)b * a.n_ops * 4;
    // branch-length sweeps from the current subtree vectors (which must match t[] and the model) until a sweep gains < eps
    auto sweeps = [&]() {
        for (int pass = 0; pass < a.max_passes; ++pass) {
            // U[c1] = D[c2]
            for (int s = tid; s < L; s += LLH_THREADS) {
                double v2[16];
                clv_load(R, L, Dt, tips, c2, s, v2);
                vec_store(Ut + ((size_t)c1 * L + s) * 16, v2);
                Unt[(size_t)c1 * L + s] = cnt_load(R, L, Dnt, c2, s);
            }
            for (int oi = 0; oi < a.n_ops; ++oi) {
                const int op = ops[oi * 4], v = ops[oi * 4 + 1], x = ops[oi * 4 + 2], y = ops[oi * 4 + 3];
                if (op == OP_UP) {
                    combine(x, y, Ut + (size_t)v * L * 16, Unt + (size_t)v * L, Ut + (size_t)x * L * 16, Unt + (size_t)x * L);
                } else if (op == OP_DOWN) {
                    combine(x, y, Dt + (size_t)(v - R) * L * 16, Dnt + (size_t)(v - R) * L, nullptr, nullptr);
                } else if (op == OP_SWAPROOT) {
                    for (int s = tid; s < L; s += LLH_THREADS) {
                        double v1[16];
                        clv_load(R, L, Dt, tips, x, s, v1);
                        vec_store(Ut + ((size_t)v * L + s) * 16, v1);
                        Unt[(size_t)v * L + s] = cnt_load(R, L, Dnt, x, s);
                    }
                } else {
                    // ---- Newton-Raphson on the branch above v.  Sumtable S[s][k][j] = (sum_a pi_a U[a] Umat[a][j]) (sum_b Uinv[j][b] D[b])
                    for (int s = tid; s < L; s += LLH_THREADS) {
                        double u[16], d[16], sv[16];
                        vec_load(Ut + ((size_t)v * L + s) * 16, u);
                        clv_load(R, L, Dt, tips, v, s, d);
                        sumtable_row(mdl, u, d, sv);
                        vec_store(St + (size_t)s * 16, sv);
                        Snt[s] = Unt[(size_t)v * L + s] + cnt_load(R, L, Dnt, v, s);
                    }
                    const double tv = newton_brlen(St, Snt, mdl, ek, red, wts, invt, pinv, wk, L, t[v]);
                    if (tid == 0) { t[v] = tv; if (v == c1) t[c2] = tv; }
                    __syncthreads();
                }
            }
            const double nl = root_loglik();
            const double gain = nl - ll;
            ll = nl;
            if (gain < a.eps) break;
        }
    };
    if (a.mode == LlhMode::Prepare) {
        sweeps();             // one pass over the UP / SWAPROOT rows (llh_prepare) fills U[v] for every v at the given lengths
    } else if (a.mode != LlhMode::Eval) {
        sweeps();
        if (a.mode == LlhMode::All) {
            // ---- model parameters: rounds of (every free parameter by golden section, all else fixed; branch sweeps) until a round
            //      gains < lh_eps - the loop of oracle/llh_oracle.py optimize_all, one tree per CTA, no host round trips
            const int flags = (int)mdl[MDL_FLAGS];
            auto objective = [&](int prm, double x) {            // set parameter prm to x (log scale for rates / alpha), rebuild, evaluate
                if (tid == 0) {
                    if (prm < 5) mdl[MDL_GTR + prm] = exp(x); else if (prm == 5) mdl[MDL_ALPHA] = exp(x); else mdl[MDL_PINV] = x;
                }
                __syncthreads();
                rebuild_model(mdl, ek, prm < 5, prm == 5);
                pinv = mdl[MDL_PINV]; wk = (1.0 - pinv) * 0.25;
                down_pass();
                return root_loglik();
            };
            for (int round = 0; round < a.max_rounds; ++round) {
                const double start = ll;
                for (int prm = 0; prm < 7; ++prm) {
                    if (prm < 5 ? !(flags & 1) : (prm == 5 ? !(flags & 2) : !(flags & 4))) continue;
                    double lo = prm < 5 ? log(RATE_LO) : (prm == 5 ? log(ALPHA_LO) : 0.0), hi = prm < 5 ? log(RATE_HI) : (prm == 5 ? log(ALPHA_HI) : PINV_HI);
                    double x1 = lo + GOLD * (hi - lo), x2 = hi - GOLD * (hi - lo);
                    double f1 = objective(prm, x1), f2 = objective(prm, x2);
                    for (int it = 0; it < a.golden_iters; ++it) {
                        if (f1 < f2) { lo = x1; x1 = x2; f1 = f2; x2 = hi - GOLD * (hi - lo); f2 = objective(prm, x2); }
                        else { hi = x2; x2 = x1; f2 = f1; x1 = lo + GOLD * (hi - lo); f1 = objective(prm, x1); }
                    }
                    ll = objective(prm, f1 > f2 ? x1 : x2);
                }
                sweeps();
                if (ll - start < a.lh_eps) break;
            }
            if (tid < LLH_MODEL) a.model_out[(size_t)b * LLH_MODEL + tid] = mdl[tid];
        }
        __syncthreads();
        if (tid == 0) { const double h = 0.5 * t[c1]; t[c1] = h; t[c2] = h; }     // the rooted form splits the root branch evenly
        __syncthreads();
        for (int v = tid; v < 2 * R - 2; v += LLH_THREADS) a.brlen[(size_t)b * (2 * R - 2) + v] = t[v];
    }
    if (tid == 0) { a.llh[2 * b] = ll0; a.llh[2 * b + 1] = ll; }
}

// ---- host side
struct LlhBuffers {
    double *D, *U, *S, *inv;
    int32_t *Dn, *Un, *Sn;
    int32_t *ch, *ops; double *br, *md, *ll;     // staged host arrays: children, schedule, brlen, model, llh (before, after)
    size_t total;
};
static LlhBuffers llh_layout(char* base, int B, int R, int L, int n_ops) {
    WsCarver c(base);
    LlhBuffers w;
    const size_t inner = (size_t)B * (R - 1), edges = (size_t)B * (2 * R - 2);
    w.D = c.take<double>(inner * L * 16);
    w.U = c.take<double>(edges * L * 16);
    w.S = c.take<double>((size_t)B * L * 16);
    w.inv = c.take<double>((size_t)B * L);
    w.Dn = c.take<int32_t>(inner * L);
    w.Un = c.take<int32_t>(edges * L);
    w.Sn = c.take<int32_t>((size_t)B * L);
    w.ch = c.take<int32_t>(inner * 2);
    w.ops = c.take<int32_t>((size_t)B * n_ops * 4);
    w.br = c.take<double>(edges);
    w.md = c.take<double>((size_t)B * LLH_MODEL);
    w.ll = c.take<double>((size_t)B * 2);
    w.total = c.off + 256;
    return w;
}

// build_ops emits 5R - 8 rows for every binary tree: OPT for each of the 2R - 3 branches, two UP rows and one DOWN row for each of the
// R - 2 inner nodes below the root, and SWAPROOT.  5R rows bound every mode's schedule.
size_t llh_ws_bytes(int B, int R, int L) { return llh_layout(nullptr, B, R, L, 5 * R).total; }

// depth-first schedule of oracle/llh_oracle.py build_ops (same order: the two implementations visit the branches identically)
static void build_ops(const int32_t* ch, int R, std::vector<int32_t>& ops) {
    struct Item { int what, v, x, y; };   // 0 enter(optimise = x), 1 up, 2 down
    auto is_inner = [&](int v) { return v >= R; };
    std::vector<Item> st;
    auto run = [&](int v0, int optimise) {
        st.push_back({0, v0, optimise, 0});
        while (!st.empty()) {
            const Item it = st.back(); st.pop_back();
            if (it.what == 0) {
                if (it.x) { ops.insert(ops.end(), {OP_OPT, it.v, 0, 0}); }
                if (is_inner(it.v)) {
                    const int a = ch[2 * (it.v - R)], b = ch[2 * (it.v - R) + 1];
                    st.push_back({2, it.v, a, b});
                    st.push_back({0, b, 1, 0});
                    st.push_back({1, b, it.v, a});
                    st.push_back({0, a, 1, 0});
                    st.push_back({1, a, it.v, b});
                }
            } else if (it.what == 1) {
                ops.insert(ops.end(), {OP_UP, it.v, it.x, it.y});
            } else {
                ops.insert(ops.end(), {OP_DOWN, it.v, it.x, it.y});
            }
        }
    };
    const int c1 = ch[2 * (R - 2)], c2 = ch[2 * (R - 2) + 1];
    run(c1, 1);
    ops.insert(ops.end(), {OP_SWAPROOT, c2, c1, 0});
    run(c2, 0);
}

// the build_ops schedules of the B trees, one after another -> rows per tree, or an error code (< 0)
static int schedule(const LlhTrees& in, std::vector<int32_t>& all) {
    int n_ops = 0;
    for (int b = 0; b < in.B; ++b) {
        const size_t start = all.size();
        build_ops(in.children + (size_t)b * (in.R - 1) * 2, in.R, all);
        const int n = (int)((all.size() - start) / 4);
        if (b == 0) n_ops = n;
        if (n != n_ops) return set_error(NNJ_ERR_INVALID, "llh: internal error (schedule length differs between trees)");
    }
    return n_ops;
}

int llh_check_tree(const int32_t* ch, int R) {
    std::vector<char> used(2 * R - 1, 0);
    for (int k = 0; k < R - 1; ++k)
        for (int e = 0; e < 2; ++e) {
            const int c = ch[2 * k + e];
            if (c < 0 || c >= R + k || used[c]) return -1;      // children are created before their parent, every node has one parent
            used[c] = 1;
        }
    return 0;
}

// one k_llh launch over B checked trees with the schedule ops (n_ops rows per tree); llh_before / llh_after / site_dev may be null.
// w: where the workspace holds the buffers.
static int launch_llh(const LlhTrees& in, LlhMode mode, const LlhOptions& opt, const std::vector<int32_t>& ops, int n_ops, double* llh_before,
                      double* llh_after, double* site_dev, void* ws, size_t ws_bytes, cudaStream_t st, LlhBuffers& w) {
    const int B = in.B, R = in.R, L = in.L;
    if (ws_bytes < llh_layout(nullptr, B, R, L, n_ops).total) return set_error(NNJ_ERR_WORKSPACE, "llh: workspace too small (nnj_llh_workspace_bytes)");
    w = llh_layout(ws_align(ws), B, R, L, n_ops);
    cudaError_t e = cudaMemcpyAsync(w.ch, in.children, (size_t)B * (R - 1) * 2 * 4, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && n_ops) e = cudaMemcpyAsync(w.ops, ops.data(), (size_t)B * n_ops * 4 * 4, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(w.br, in.brlen, (size_t)B * (2 * R - 2) * 8, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(w.md, in.model, (size_t)B * LLH_MODEL * 8, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    LlhArgs a;
    a.tips = in.tips; a.weights = in.weights; a.children = w.ch; a.ops = w.ops; a.brlen = w.br; a.model = w.md;
    a.D = w.D; a.U = w.U; a.S = w.S; a.inv = w.inv; a.Dn = w.Dn; a.Un = w.Un; a.Sn = w.Sn;
    a.llh = w.ll; a.site = site_dev;
    a.B = B; a.R = R; a.L = L; a.n_ops = n_ops; a.max_passes = opt.max_passes; a.mode = mode; a.eps = opt.eps;
    a.lh_eps = opt.lh_eps; a.max_rounds = opt.max_rounds; a.golden_iters = GOLDEN_ITERS; a.model_out = w.md;
    const size_t smem = (LLH_MODEL + 128 + 66 + 48 + 2 * (size_t)R) * sizeof(double);      // 67 968 bytes at R = 4096
    if (smem > 48 * 1024) {       // above the default limit the kernel must opt in (from R = 2920 on)
        e = cudaFuncSetAttribute(k_llh, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    }
    prof_begin(KC_LLH, st);
    k_llh<<<B, LLH_THREADS, smem, st>>>(a);
    ++g_launches;
    prof_end(st);
    std::vector<double> ll((size_t)B * 2);
    const bool brlen_out = mode == LlhMode::Brlen || mode == LlhMode::All;
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(ll.data(), w.ll, ll.size() * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && brlen_out) e = cudaMemcpyAsync(in.brlen, w.br, (size_t)B * (2 * R - 2) * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && mode == LlhMode::All) e = cudaMemcpyAsync(in.model, w.md, (size_t)B * LLH_MODEL * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);       // the small results are host values: the call returns them
    if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    for (int b = 0; b < B; ++b) {
        if (llh_before) llh_before[b] = ll[2 * b];
        if (llh_after) llh_after[b] = ll[2 * b + 1];
    }
    return 0;
}

int run_llh(const LlhTrees& in, LlhMode mode, const LlhOptions& opt, double* llh_before, double* llh_after, void* ws, size_t ws_bytes, cudaStream_t st) {
    for (int b = 0; b < in.B; ++b)
        if (llh_check_tree(in.children + (size_t)b * (in.R - 1) * 2, in.R)) return set_error(NNJ_ERR_INVALID, "llh: children is not a binary tree in join order");
    std::vector<int32_t> ops;
    const int n_ops = mode == LlhMode::Eval ? 0 : schedule(in, ops);
    if (n_ops < 0) return n_ops;
    LlhBuffers w;
    return launch_llh(in, mode, opt, ops, n_ops, llh_before, llh_after, nullptr, ws, ws_bytes, st, w);
}

LlhPrepared llh_prepare(const LlhTrees& in, double* site_dev, double* llh_h, void* ws, size_t ws_bytes, cudaStream_t st) {
    std::vector<int32_t> ops, u_pass;
    const int n = schedule(in, ops);
    if (n < 0) return {n, nullptr, nullptr, nullptr, nullptr, nullptr};
    // the U pass alone: UP and SWAPROOT rows (2R - 3 per tree), no Newton, no refreshed subtree vectors; one pass fills U[v] for every v
    for (size_t i = 0; i < ops.size(); i += 4)
        if (ops[i] == OP_UP || ops[i] == OP_SWAPROOT) u_pass.insert(u_pass.end(), ops.begin() + i, ops.begin() + i + 4);
    const LlhOptions one_pass{1, 0.0, 0.0, 0};
    LlhBuffers w{};
    const int rc = launch_llh(in, LlhMode::Prepare, one_pass, u_pass, (int)(u_pass.size() / 4 / in.B), nullptr, llh_h, site_dev, ws, ws_bytes, st, w);
    return {rc, w.D, w.U, w.inv, w.Dn, w.Un};
}

int gamma_rates(double alpha, int ncat, double* out) {
    if (!(alpha > 0.0) || ncat < 1 || ncat > 64) return set_error(NNJ_ERR_INVALID, "gamma_rates: alpha must be > 0 and 1 <= ncat <= 64");
    std::vector<double> cdf(ncat + 1, 0.0);
    cdf[ncat] = 1.0;
    for (int i = 1; i < ncat; ++i) cdf[i] = gamma_class_cdf(alpha, (double)i / ncat);
    for (int i = 0; i < ncat; ++i) out[i] = ncat * (cdf[i + 1] - cdf[i]);
    return 0;
}

}  // namespace nnj
