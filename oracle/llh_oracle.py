"""CPU restatement (TEST INFRASTRUCTURE ONLY) of the tree-likelihood scorer behind the reference's
`raxmlpy.optimize_brlen / compute_llh` (RAxMLpy/cpp/raxmlpy.cpp:1749-1872; call sites environment.py:365-379,
625-670; finetune_rl_search.py:401-411): log-likelihood of an alignment on a fixed topology under GTR+I+G4 and its
maximisation over branch lengths (Newton-Raphson per branch) and model parameters.

PARITY UNPINNED against the reference: the arithmetic lives in raxml-ng / pll-modules / libpll-2, which
RAxMLpy/setup.py:20,37 git-clones at install time (no pinned version, not under /root/reference, no network here),
and RAxMLpy/test/*.py only print.  What pins this file instead (tests/test_llh_oracle.py):
  * Felsenstein pruning vs brute-force enumeration of every internal-state assignment (small trees);
  * the discrete-gamma mean rates vs the published table value (Yang 1994: alpha 0.5, 4 categories ->
    0.0334, 0.2519, 0.8203, 2.8944);
  * JC69 two-taxon closed form: d = -3/4 ln(1 - 4p/3) maximises the likelihood;
  * the optimiser never decreases the likelihood, and a numerical gradient at its fixed point vanishes;
  * for trees whose site likelihoods underflow fp64 (a few hundred taxa and up), `loglik_logspace`: pruning on
    log-CLVs with logsumexp and transition matrices from scipy.linalg.expm - no eigen form and no rescaling.
The published algorithm restated: Felsenstein (1981) pruning; Yang (1994) discrete gamma, mean of each quantile
class; invariant-site mixture L = (1-p) L_gamma + p * pi_x for columns whose tips share one state x; per-branch
Newton-Raphson on the eigen-space "sumtable" with the other branches fixed, swept in depth-first order with the
conditional likelihood vectors refreshed on the way (the scheme of libpll's pllmod_algo_opt_brlen_treeinfo);
branch lengths in [1e-6, 100], default 0.1 (raxml-ng's RAXML_BRLEN_MIN / MAX / DEFAULT): evaluation and optimisation
both clamp every length, and the root branch brlen[c1] + brlen[c2], into that range.

Scaling (the rule of csrc/nnj_llh.cu, applied everywhere a CLV is formed): when all 16 entries of a (node, pattern)
vector are below 2^-256, the vector is multiplied by 2^256 and the pattern's integer count of that node goes up by one.
Counts add along the tree: D(v) = D(a) + D(b) + own, U(c) = U(parent) + D(sibling) + own, and copies keep theirs.  A
site likelihood is ldexp(wk * l, -256 n) + p_inv * inv; its log is taken as log(wk * l) - 256 n ln 2 when p_inv * inv
is 0.  Powers of two are exact: where nothing is scaled, every result is bit-identical to unscaled pruning.

Tree encoding shared with the CUDA path: leaves 0..R-1, inner node R+k = k-th join, children[k] = (left, right);
the last inner node is the (virtual) root.  brlen[v] = length of the edge above node v (v < 2R-2); the two root
edges form ONE branch of the unrooted tree (length brlen[c1] + brlen[c2]).
"""
from __future__ import annotations

import itertools

import numpy as np
from scipy import special

BRLEN_MIN, BRLEN_MAX, BRLEN_DEFAULT = 1e-6, 100.0, 0.1
SCALE_EXP = 256                        # a CLV whose entries are all below 2^-SCALE_EXP is multiplied by 2^SCALE_EXP
SCALE_THRESHOLD = 2.0 ** -SCALE_EXP
LN2 = float(np.log(2.0))
NCAT = 4
OP_OPT, OP_UP, OP_DOWN, OP_SWAPROOT = 0, 1, 2, 3


# ------------------------------------------------------------------ model
def gamma_rates(alpha: float, ncat: int = NCAT) -> np.ndarray:
    """Mean rate of each of the ncat equal-probability classes of Gamma(shape alpha, rate alpha) (Yang 1994, eq. 10)."""
    q = special.gammaincinv(alpha, np.arange(1, ncat) / ncat)            # class boundaries (in units of rate * x)
    cdf = np.concatenate([[0.0], special.gammainc(alpha + 1.0, q), [1.0]])
    return ncat * np.diff(cdf)


def gtr_eigen(rates6, freqs):
    """Eigen-decomposition of the normalised GTR rate matrix.  rates6 = (AC, AG, AT, CG, CT, GT).
    Returns lam [4], U [4,4], Uinv [4,4] with P(t) = U diag(exp(lam t)) Uinv."""
    pi = np.asarray(freqs, dtype=np.float64)
    r = np.zeros((4, 4))
    for (a, b), v in zip(itertools.combinations(range(4), 2), rates6):
        r[a, b] = r[b, a] = v
    Q = r * pi[None, :]
    np.fill_diagonal(Q, 0.0)
    np.fill_diagonal(Q, -Q.sum(1))
    Q /= -(pi * np.diag(Q)).sum()                                         # one expected substitution per unit time
    sq = np.sqrt(pi)
    S = (sq[:, None] * Q) / sq[None, :]
    lam, V = np.linalg.eigh(0.5 * (S + S.T))
    return lam, V / sq[:, None], V.T * sq[None, :]


def empirical_freqs(tips: np.ndarray) -> np.ndarray:
    """Base frequencies from the alignment (uint8 4-bit masks [R, L]); an ambiguous character spreads its count
    evenly over its states, fully undetermined ones (gap / N) are skipped."""
    cnt = np.zeros(4)
    for m in range(1, 15):
        n = int((tips == m).sum())
        bits = [(m >> a) & 1 for a in range(4)]
        cnt += n * np.array(bits) / sum(bits)
    return cnt / cnt.sum()


def compress_patterns(tips: np.ndarray):
    """Unique alignment columns and their multiplicities (raxmlpy.cpp:1646-1657 compresses patterns too)."""
    cols, inv, w = np.unique(tips, axis=1, return_inverse=True, return_counts=True)
    return np.ascontiguousarray(cols), w.astype(np.float64)


def masks_from_onehot(data) -> np.ndarray:
    """int8 one-hot [R, L, 4] (gap = 1111) -> uint8 state masks [R, L] (bit a = state a possible)."""
    d = np.asarray(data).astype(np.uint8)
    m = d[..., 0] | (d[..., 1] << 1) | (d[..., 2] << 2) | (d[..., 3] << 3)
    m[m == 0] = 15
    return m


class Model:
    def __init__(self, rates6=(1, 1, 1, 1, 1, 1), freqs=(0.25,) * 4, alpha=1.0, pinv=0.0, ncat=NCAT, gamma=True):
        self.rates6 = np.asarray(rates6, dtype=np.float64)
        self.freqs = np.asarray(freqs, dtype=np.float64)
        self.alpha, self.pinv, self.ncat, self.gamma = float(alpha), float(pinv), ncat, gamma
        self.refresh()

    def refresh(self):
        self.lam, self.U, self.Uinv = gtr_eigen(self.rates6, self.freqs)
        self.cat = gamma_rates(self.alpha, self.ncat) if self.gamma else np.ones(self.ncat)

    def pmats(self, t: float) -> np.ndarray:                              # [ncat, 4, 4]
        e = np.exp(self.lam[None, :] * self.cat[:, None] * t)
        return np.einsum("aj,kj,jb->kab", self.U, e, self.Uinv)

    def packed(self) -> np.ndarray:
        """The 48 doubles the CUDA kernels take per tree: lam 4 | U 16 | Uinv 16 | freqs 4 | cat rates 4 | pinv | pad 3."""
        return np.concatenate([self.lam, self.U.ravel(), self.Uinv.ravel(), self.freqs, self.cat, [self.pinv, 0, 0, 0]])


# ------------------------------------------------------------------ likelihood
def tip_clv(col: np.ndarray, ncat: int) -> np.ndarray:                    # masks [L] -> [L, ncat, 4]
    bits = ((col[:, None] >> np.arange(4)[None, :]) & 1).astype(np.float64)
    return np.repeat(bits[:, None, :], ncat, axis=1)


def invariant_term(tips: np.ndarray, freqs: np.ndarray) -> np.ndarray:
    """pi_x for columns whose tips are all compatible with exactly one state x, else 0."""
    m = np.bitwise_and.reduce(tips, axis=0)
    single = (m & (m - 1)) == 0
    idx = np.log2(np.maximum(m, 1)).astype(int)
    return np.where(single & (m > 0), freqs[np.minimum(idx, 3)], 0.0)


def _scale(x: np.ndarray, n: np.ndarray, scaling: bool):
    """The kernel's rule on one freshly combined CLV x [L, ncat, 4] with the summed counts n [L] of its inputs."""
    if scaling:
        small = (x < SCALE_THRESHOLD).all(axis=(1, 2))
        if small.any():
            x[small] = np.ldexp(x[small], SCALE_EXP)
            n = n + small
    return x, n


def _combine(Px, x, nx, Py, y, ny, scaling: bool):
    z = np.einsum("kxy,sky->skx", Px, x) * np.einsum("kxy,sky->skx", Py, y)
    return _scale(z, nx + ny, scaling)


def down_clvs(children, brlen, tips, model: Model, scaling: bool = True):
    """Subtree CLVs of every node -> (D [2R-1] of [L, ncat, 4], counts [2R-1] of int [L])."""
    R, L = tips.shape
    D = [tip_clv(tips[v], model.ncat) for v in range(R)]
    N = [np.zeros(L, dtype=np.int64) for _ in range(R)]
    for a, b in children:
        d, n = _combine(model.pmats(brlen[a]), D[a], N[a], model.pmats(brlen[b]), D[b], N[b], scaling)
        D.append(d)
        N.append(n)
    return D, N


def clamp_lengths(children, brlen) -> np.ndarray:
    """The lengths every computation uses: each clamped to [BRLEN_MIN, BRLEN_MAX], and the root branch (the two root
    edges, one branch of the unrooted tree) clamped as a whole and stored at both ends."""
    t = np.clip(np.array(brlen, dtype=np.float64), BRLEN_MIN, BRLEN_MAX)
    c1, c2 = (int(v) for v in children[-1])
    t[c1] = t[c2] = min(max(t[c1] + t[c2], BRLEN_MIN), BRLEN_MAX)
    return t


def log_sites(lw: np.ndarray, n: np.ndarray, iv: np.ndarray) -> np.ndarray:
    """log(ldexp(lw, -256 n) + iv) per pattern; log(lw) - 256 n ln 2 where iv (= p_inv * inv) is 0 and n > 0."""
    with np.errstate(divide="ignore"):
        out = np.log(np.ldexp(lw, -SCALE_EXP * n) + iv)
        sc = (n > 0) & (iv == 0)
        if sc.any():
            out[sc] = np.log(lw[sc]) - n[sc] * (SCALE_EXP * LN2)
    return out


def root_terms(children, brlen, tips, model: Model, scaling: bool = True):
    """-> (wk * l, n, p_inv * inv) per pattern: the site likelihood is ldexp(wk * l, -256 n) + p_inv * inv.  The root branch
    is one branch of length t[c1] (clamp_lengths), between D[c1] and D[c2]."""
    children = np.asarray(children)
    t = clamp_lengths(children, brlen)
    c1, c2 = (int(v) for v in children[-1])
    D, N = down_clvs(children[:-1], t, tips, model, scaling)
    x = np.einsum("kxy,sky->skx", model.pmats(t[c1]), D[c1]) * D[c2]
    lw = (1.0 - model.pinv) * (np.einsum("ska,a->s", x, model.freqs) / model.ncat)
    return lw, N[c1] + N[c2], model.pinv * invariant_term(tips, model.freqs)


def site_likelihoods(children, brlen, tips, model: Model, scaling: bool = False) -> np.ndarray:
    """Plain site likelihoods.  Unscaled (the default) they underflow to subnormals or 0 on large trees - which is what
    tests use this for; scaled, the result is exact up to the final ldexp, which may underflow the same way."""
    lw, n, iv = root_terms(children, brlen, tips, model, scaling)
    return np.ldexp(lw, -SCALE_EXP * n) + iv


def site_logliks(children, brlen, tips, model: Model, scaling: bool = True) -> np.ndarray:
    return log_sites(*root_terms(children, brlen, tips, model, scaling))


def loglik(children, brlen, tips, weights, model: Model, scaling: bool = True) -> float:
    return float((weights * site_logliks(children, brlen, tips, model, scaling)).sum())


def loglik_logspace(children, brlen, tips, weights, model: Model) -> float:
    """Independent reference for trees of any size: pruning on log-CLVs (scipy.special.logsumexp), transition matrices
    scipy.linalg.expm(Q r_k t) of the normalised GTR matrix built here again - neither the eigen form nor any rescaling.
    Slow; it exists to pin the scaled pruning above."""
    from scipy import linalg
    children = np.asarray(children)
    R = tips.shape[0]
    t = clamp_lengths(children, brlen)
    c1, c2 = (int(v) for v in children[-1])
    pi = np.asarray(model.freqs, dtype=np.float64)
    Q = np.zeros((4, 4))
    for (a, b), v in zip(itertools.combinations(range(4), 2), model.rates6):
        Q[a, b], Q[b, a] = v * pi[b], v * pi[a]
    Q -= np.diag(Q.sum(1))
    Q /= -(pi * np.diag(Q)).sum()
    cat = model.cat

    def logp(tv):                                                         # [ncat, 4, 4]
        with np.errstate(divide="ignore"):
            return np.log(np.stack([linalg.expm(Q * r * tv) for r in cat]))

    def move(lp, x):                                                      # log sum_y P[k, a, y] exp(x[s, k, y])
        return special.logsumexp(lp[None, :, :, :] + x[:, :, None, :], axis=3)

    with np.errstate(divide="ignore"):
        logD = [np.log(tip_clv(tips[v], model.ncat)) for v in range(R)]
    for a, b in children[:-1]:
        logD.append(move(logp(t[a]), logD[a]) + move(logp(t[b]), logD[b]))
    x = move(logp(t[c1]), logD[c1]) + logD[c2]                              # [L, ncat, 4]
    with np.errstate(divide="ignore"):
        lg = special.logsumexp(x + np.log(pi)[None, None, :], axis=(1, 2)) - np.log(model.ncat)
        iv = np.log(model.pinv * invariant_term(tips, pi))
        site = np.logaddexp(np.log1p(-model.pinv) + lg, iv)
    return float((weights * site).sum())


def loglik_bruteforce(children, brlen, tips, weights, model: Model) -> float:
    """Sum over every assignment of states to the inner nodes - exponential, for trees with <= 6 inner nodes."""
    R, L = tips.shape
    n_inner = len(children)
    parent_edge = {}
    for k, (a, b) in enumerate(children):
        parent_edge[a] = R + k
        parent_edge[b] = R + k
    P = {v: model.pmats(brlen[v]) for v in parent_edge}
    site = np.zeros(L)
    for k in range(model.ncat):
        for states in itertools.product(range(4), repeat=n_inner):
            pr = np.full(L, model.freqs[states[-1]])
            for v, p in parent_edge.items():
                sp = states[p - R]
                if v >= R:
                    pr = pr * P[v][k][sp, states[v - R]]
                else:
                    bits = ((tips[v][:, None] >> np.arange(4)[None, :]) & 1).astype(np.float64)
                    pr = pr * (bits @ P[v][k][sp, :])
            site += pr / model.ncat
    site = (1.0 - model.pinv) * site + model.pinv * invariant_term(tips, model.freqs)
    return float((weights * np.log(site)).sum())


# ------------------------------------------------------------------ branch-length optimiser
def build_ops(children, R: int):
    """The depth-first schedule executed by both this file and the CUDA kernel, as rows (op, v, x, y):
       OPT v         Newton-Raphson on the branch above v (outer vector U[v], subtree vector D[v])
       UP c, v, s    U[c] = (P(t_v) U[v]) * (P(t_s) D[s])     c, s children of v
       DOWN v, a, b  D[v] = (P(t_a) D[a]) * (P(t_b) D[b])     refresh after both subtrees changed
       SWAPROOT c2, c1   U[c2] = D[c1]: cross the root branch (c1, c2 = the root's children; t[c2] is tied to t[c1])
    The root branch is optimised once (at c1); U[c1] = D[c2] is set before the first op."""
    ops = []
    kids = {R + k: (int(a), int(b)) for k, (a, b) in enumerate(children)}

    def process(v, optimise=True):
        stack = [("enter", v, optimise)]
        while stack:
            what, v, flag = stack.pop()
            if what == "enter":
                if flag:
                    ops.append((OP_OPT, v, 0, 0))
                if v in kids:
                    a, b = kids[v]
                    stack.append(("down", v, 0))
                    stack.append(("enter", b, True))
                    stack.append(("up", (b, v, a), 0))
                    stack.append(("enter", a, True))
                    stack.append(("up", (a, v, b), 0))
            elif what == "up":
                c, p, s = v
                ops.append((OP_UP, c, p, s))
            else:
                a, b = kids[v]
                ops.append((OP_DOWN, v, a, b))

    root = R + len(children) - 1
    c1, c2 = kids[root]
    process(c1, True)
    ops.append((OP_SWAPROOT, c2, c1, 0))
    process(c2, False)
    return np.asarray(ops, dtype=np.int32).reshape(-1, 4)


def _newton(S, lam, cat, wk, inv, weights, t0):
    """Safeguarded Newton-Raphson on f(t) = sum_s w_s log L_s(t), L_s = sum_kj S[s,k,j] exp(lam_j r_k t) * wk + inv_s.
    Same arithmetic and control flow as the Newton loop in csrc/nnj_llh.cu; S is scaled by 2^(-256 n_s), inv_s by the
    caller to match."""
    rate = lam[None, :] * cat[:, None]                                    # [k, j]
    t, lo, hi = min(max(t0, BRLEN_MIN), BRLEN_MAX), BRLEN_MIN, BRLEN_MAX
    for _ in range(32):
        e = np.exp(rate * t)
        L0 = wk * np.einsum("skj,kj->s", S, e) + inv
        L1 = wk * np.einsum("skj,kj->s", S, e * rate)
        L2 = wk * np.einsum("skj,kj->s", S, e * rate * rate)
        g = L1 / L0
        f1 = float((weights * g).sum())
        f2 = float((weights * (L2 / L0 - g * g)).sum())
        if f1 > 0:
            lo = t
        else:
            hi = t
        if f2 < 0:
            tn = t - f1 / f2
        else:
            tn = t * 4.0 if f1 > 0 else t * 0.25
        if not (lo < tn < hi):
            tn = 0.5 * (lo + hi)
        done = abs(tn - t) < 1e-9 + 1e-7 * t
        t = tn
        if done:
            break
    return t


def optimize_branches(children, brlen, tips, weights, model: Model, max_passes=32, eps=1e-3, scaling: bool = True):
    """Returns (brlen_opt, loglik_before, loglik_after).  A pass = one sweep of build_ops; passes stop when the
    log-likelihood gain of a pass is below eps."""
    children = np.asarray(children)
    R = tips.shape[0]
    t = clamp_lengths(children, brlen)                                    # the root branch is stored at both ends
    c1, c2 = (int(v) for v in children[-1])
    ops = build_ops(children, R)
    inv = model.pinv * invariant_term(tips, model.freqs)
    wk = (1.0 - model.pinv) / model.ncat

    def root_loglik(D, N):
        x = np.einsum("kxy,sky->skx", model.pmats(t[c1]), D[c1]) * D[c2]
        return float((weights * log_sites(wk * np.einsum("ska,a->s", x, model.freqs), N[c1] + N[c2], inv)).sum())

    tt = t.copy()
    tt[c2] = 0.0
    D, N = down_clvs(children, tt, tips, model, scaling)
    U, NU = [None] * (2 * R - 1), [None] * (2 * R - 1)
    ll0 = ll = root_loglik(D, N)
    for _ in range(max_passes):
        U[c1], NU[c1] = D[c2], N[c2]
        for op, v, x, y in ops:
            if op == OP_OPT:
                A = np.einsum("ska,a,aj->skj", U[v], model.freqs, model.U)
                Bm = np.einsum("jb,skb->skj", model.Uinv, D[v])
                n = NU[v] + N[v]
                with np.errstate(over="ignore"):                          # 2^(256 n) p_inv pi_x may be inf: then g = 0, exactly enough
                    invs = np.where((inv > 0) & (n > 0), np.ldexp(inv, SCALE_EXP * n), inv)
                t[v] = _newton(A * Bm, model.lam, model.cat, wk, invs, weights, t[v])
                if v == c1:
                    t[c2] = t[c1]
            elif op == OP_UP:
                U[v], NU[v] = _combine(model.pmats(t[x]), U[x], NU[x], model.pmats(t[y]), D[y], N[y], scaling)
            elif op == OP_DOWN:
                D[v], N[v] = _combine(model.pmats(t[x]), D[x], N[x], model.pmats(t[y]), D[y], N[y], scaling)
            else:
                U[v], NU[v] = D[x], N[x]
        new = root_loglik(D, N)
        gain, ll = new - ll, new
        if gain < eps:
            break
    out = t.copy()
    out[c1] = out[c2] = 0.5 * t[c1]                                       # the rooted form splits the root branch evenly
    return out, ll0, ll


# ------------------------------------------------------------------ model-parameter optimiser (coordinate golden section)
GOLD = 0.3819660112501051
RATE_LO, RATE_HI, ALPHA_LO, ALPHA_HI, PINV_HI = 1e-3, 1e3, 0.02, 100.0, 0.99


def golden_max(f, lo, hi, iters=24):
    a, b = lo, hi
    x1, x2 = a + GOLD * (b - a), b - GOLD * (b - a)
    f1, f2 = f(x1), f(x2)
    for _ in range(iters):
        if f1 < f2:
            a, x1, f1 = x1, x2, f2
            x2 = b - GOLD * (b - a)
            f2 = f(x2)
        else:
            b, x2, f2 = x2, x1, f1
            x1 = a + GOLD * (b - a)
            f1 = f(x1)
    return (x1, f1) if f1 > f2 else (x2, f2)


def optimize_all(children, brlen, tips, weights, model: Model, lh_eps=1.0, max_rounds=10, scaling: bool = True):
    """Branch lengths, then rounds of (5 free GTR rates, alpha, pinv, branch lengths) until a round gains < lh_eps
    (raxmlpy.cpp:1721-1746 `optimize_model(treeinfo, 1.0)` has this loop shape; its inner optimisers differ)."""
    t, ll0, ll = optimize_branches(children, brlen, tips, weights, model, scaling=scaling)
    for _ in range(max_rounds):
        start = ll

        def with_param(setter):
            def f(x):
                setter(x)
                model.refresh()
                return loglik(children, t, tips, weights, model, scaling)
            return f

        for i in range(5):
            def set_rate(x, i=i):
                model.rates6[i] = np.exp(x)
            x, _ = golden_max(with_param(set_rate), np.log(RATE_LO), np.log(RATE_HI))
            set_rate(x)
        def set_alpha(x):
            model.alpha = float(np.exp(x))
        x, _ = golden_max(with_param(set_alpha), np.log(ALPHA_LO), np.log(ALPHA_HI))
        set_alpha(x)
        def set_pinv(x):
            model.pinv = float(x)
        x, _ = golden_max(with_param(set_pinv), 0.0, PINV_HI)
        set_pinv(x)
        model.refresh()
        t, _, ll = optimize_branches(children, t, tips, weights, model, scaling=scaling)
        if ll - start < lh_eps:
            break
    return t, ll0, ll


# ------------------------------------------------------------------ helpers for tests
def random_tree(R: int, rng: np.random.Generator):
    """Random join order -> (children [R-1, 2], brlen [2R-2])."""
    cur = list(range(R))
    children = []
    for k in range(R - 1):
        i, j = sorted(rng.choice(len(cur), size=2, replace=False))
        children.append((cur[i], cur[j]))
        cur[i] = R + k
        del cur[j]
    return np.asarray(children, dtype=np.int32), rng.uniform(0.02, 0.4, size=2 * R - 2)


def simulate(children, brlen, R: int, L: int, model: Model, rng: np.random.Generator, gap_frac=0.0) -> np.ndarray:
    """Evolve L sites down the tree under the model -> uint8 masks [R, L]."""
    n = R + len(children)
    states = np.zeros((n, L), dtype=np.int64)
    cat = rng.integers(0, model.ncat, size=L)
    states[n - 1] = rng.choice(4, size=L, p=model.freqs)
    for k in range(len(children) - 1, -1, -1):
        for c in children[k]:
            P = model.pmats(brlen[c])[cat, states[R + k], :]               # [L, 4]
            P = np.maximum(P, 0)
            P /= P.sum(1, keepdims=True)
            u = rng.random(L)
            states[c] = (u[:, None] > np.cumsum(P, axis=1)).sum(1).clip(0, 3)
    tips = (1 << states[:R]).astype(np.uint8)
    if gap_frac:
        tips[rng.random(tips.shape) < gap_frac] = 15
    return tips
