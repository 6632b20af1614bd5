"""CPU oracle (test infrastructure) of likelihood branch support (DESIGN.md 12; csrc/nnj_llh_nni.cu): the NNI alternatives of
every internal branch with their five quartet lengths optimised, RELL replicates, SH-aLRT and the local bootstrap probability.
numpy fp64 on top of llh_oracle (the same CLVs, scaling rule and Newton iteration) and support_oracle's Philox.

    u_vectors(children, brlen, tips, model)                  D, U and their scale counts at the clamped lengths (down pass + U pass)
    quartet_sites(children, brlen, tips, model, v, k, lens)  per-pattern log-likelihoods of configuration k at the five lengths
    nni_optimize(children, brlen, tips, weights, model, v, k)  (L_k, the five optimised lengths, l_k)
    branch_support(children, brlen, tips, weights, model, n_rell, seed, rep0)  everything nnj_llh_branch_support returns
    rell_counts(weights, seed, reps)                         [n, L] integer counts c_r[p]
    rell_stats(site, weights, counts)                        SH and LBP counts per branch, sums in pattern order (np.cumsum)
"""
from __future__ import annotations

import numpy as np

import llh_oracle as O
from support_oracle import philox4x32_10

NNI_MAX_ROUNDS, NNI_EPS, SH_TOL = 8, 1e-3, 0.05
_MASK32 = np.uint64(0xFFFFFFFF)


def internal_branches(children):
    children = np.asarray(children)
    R = len(children) + 1
    c1, c2 = (int(c) for c in children[-1])
    return [v for v in range(R, 2 * R - 2) if v not in (c1, c2) or (v == c1 and c2 >= R)]


def u_vectors(children, brlen, tips, model: O.Model):
    """-> t (clamped lengths, root branch at both ends), D, N (subtree CLVs and counts of every node), U, NU (CLV of the rest of
    the tree seen from the parent end of the branch above each node: U[c1] = D[c2], U[c2] = D[c1])."""
    children = np.asarray(children)
    R = tips.shape[0]
    t = O.clamp_lengths(children, brlen)
    c1, c2 = (int(v) for v in children[-1])
    D, N = O.down_clvs(children[:-1], t, tips, model)
    U, NU = [None] * (2 * R - 1), [None] * (2 * R - 1)
    U[c1], NU[c1] = D[c2], N[c2]
    for op, v, x, y in O.build_ops(children, R):
        if op == O.OP_UP:
            U[v], NU[v] = O._combine(model.pmats(t[x]), U[x], NU[x], model.pmats(t[y]), D[y], N[y], True)
        elif op == O.OP_SWAPROOT:
            U[v], NU[v] = D[x], N[x]
    return t, D, N, U, NU


def _quartet(children, v, t, D, N, U, NU):
    """-> vectors [A, B, C, D], counts, lengths [central, A, B, C, D] of the branch above v."""
    children = np.asarray(children)
    R = len(children) + 1
    c1, c2 = (int(x) for x in children[-1])
    a, b = (int(x) for x in children[v - R])
    if v == c1:
        c, d = (int(x) for x in children[c2 - R])
        return [D[a], D[b], D[c], D[d]], [N[a], N[b], N[c], N[d]], [t[v], t[a], t[b], t[c], t[d]]
    p = next(R + k for k, pair in enumerate(children.tolist()) if v in pair)
    pa, pb = (int(x) for x in children[p - R])
    c = pb if pa == v else pa
    return [D[a], D[b], D[c], U[p]], [N[a], N[b], N[c], NU[p]], [t[v], t[a], t[b], t[c], t[p]]


class _Quartet:
    """Configuration k of one quartet: X = (A, x2) and Y = (B, y2) across the central branch; edges 0 central, 1..4 = A..D."""

    def __init__(self, vecs, cnts, lens, k, tips, model: O.Model):
        self.vec, self.cnt, self.t, self.m = [None] + vecs, [None] + cnts, list(lens), model
        (self.x1, self.x2), (self.y1, self.y2) = {0: ((1, 2), (3, 4)), 1: ((1, 3), (2, 4)), 2: ((1, 4), (2, 3))}[k]
        self.inv = model.pinv * O.invariant_term(tips, model.freqs)
        self.wk = (1.0 - model.pinv) / model.ncat

    def half(self, e, f):
        return O._combine(self.m.pmats(self.t[e]), self.vec[e], self.cnt[e], self.m.pmats(self.t[f]), self.vec[f], self.cnt[f], True)

    def sites(self):
        X, nX = self.half(self.x1, self.x2)
        Y, nY = self.half(self.y1, self.y2)
        x = np.einsum("kxy,sky->skx", self.m.pmats(self.t[0]), X) * Y
        return O.log_sites(self.wk * np.einsum("ska,a->s", x, self.m.freqs), nX + nY, self.inv)

    def newton(self, e, weights):
        m = self.m
        if e == 0:
            u, nu = self.half(self.y1, self.y2)
            d, nd = self.half(self.x1, self.x2)
        else:
            side_x = e in (self.x1, self.x2)
            pair = (self.x1, self.x2) if side_x else (self.y1, self.y2)
            f = pair[1] if e == pair[0] else pair[0]
            o, no = self.half(*((self.y1, self.y2) if side_x else (self.x1, self.x2)))
            u, nu = O._combine(m.pmats(self.t[f]), self.vec[f], self.cnt[f], m.pmats(self.t[0]), o, no, True)
            d, nd = self.vec[e], self.cnt[e]
        A = np.einsum("ska,a,aj->skj", u, m.freqs, m.U)
        Bm = np.einsum("jb,skb->skj", m.Uinv, d)
        n = nu + nd
        with np.errstate(over="ignore"):
            invs = np.where((self.inv > 0) & (n > 0), np.ldexp(self.inv, O.SCALE_EXP * n), self.inv)
        self.t[e] = O._newton(A * Bm, m.lam, m.cat, self.wk, invs, weights, self.t[e])


def quartet_sites(children, brlen, tips, model: O.Model, v: int, k: int, lens=None):
    """Per-pattern log-likelihoods of configuration k (0 the tree, 1 AC|BD, 2 AD|BC) of the branch above v, with the outer vectors
    of the tree at `brlen` and the five quartet lengths `lens` (default: the tree's)."""
    t, D, N, U, NU = u_vectors(children, brlen, tips, model)
    vecs, cnts, l0 = _quartet(children, v, t, D, N, U, NU)
    q = _Quartet(vecs, cnts, l0 if lens is None else lens, k, tips, model)
    return q.sites()


def _optimize(q: _Quartet, weights):
    ll = float((weights * q.sites()).sum())
    for _ in range(NNI_MAX_ROUNDS):
        for e in range(5):
            q.newton(e, weights)
        site = q.sites()
        nl = float((weights * site).sum())
        gain, ll = nl - ll, nl
        if gain < NNI_EPS:
            break
    return ll, np.array(q.t), q.sites()


def nni_optimize(children, brlen, tips, weights, model: O.Model, v: int, k: int):
    """-> (L_k, lengths [5], l_k [L]) of alternative k of the branch above v after the round rule of DESIGN 12."""
    t, D, N, U, NU = u_vectors(children, brlen, tips, model)
    vecs, cnts, lens = _quartet(children, v, t, D, N, U, NU)
    return _optimize(_Quartet(vecs, cnts, lens, k, tips, model), weights)


def rell_counts(weights, seed: int, reps) -> np.ndarray:
    """[len(reps), L] int64: how often replicate r draws pattern p; draw i is site (x0 * n) >> 32, x0 = Philox word 0 of counter
    (i, r lo, r hi, 0), key (seed lo, seed hi); pattern p owns the sites cum[p] <= u < cum[p+1]."""
    w = np.asarray(weights, dtype=np.float64)
    assert (w >= 0).all() and (w == np.floor(w)).all()
    cum = np.concatenate([[0], np.cumsum(w.astype(np.int64))])
    n = int(cum[-1])
    i = np.arange(n, dtype=np.uint64)
    out = np.zeros((len(reps), len(w)), dtype=np.int64)
    for j, r in enumerate(reps):
        r = np.uint64(r)
        x0 = philox4x32_10((i, np.full_like(i, r & _MASK32), np.full_like(i, r >> np.uint64(32)), np.zeros_like(i)),
                           (seed & 0xFFFFFFFF, seed >> 32))[0]
        u = ((x0 * np.uint64(n)) >> np.uint64(32)).astype(np.int64)
        out[j] = np.bincount(np.searchsorted(cum, u, side="right") - 1, minlength=len(w))
    return out


def _seqsum(x):
    """Sum along the last axis in order, one add at a time (np.cumsum accumulates sequentially)."""
    return np.cumsum(x, axis=-1)[..., -1]


def rell_stats(site, weights, counts):
    """site [nb, 3, L] (l0, l1, l2), weights [L], counts [N, L] -> (sh [nb], lbp [nb]) integer counts.  Lk = sum w lk, Lk* = sum c lk,
    products rounded, then added in pattern order; delta = L0 - max(L1, L2); SH: delta > (largest - second largest of Lk* - Lk) + 0.05;
    LBP: L0* >= max(L1*, L2*)."""
    site = np.asarray(site, dtype=np.float64)
    w = np.asarray(weights, dtype=np.float64)
    c = np.asarray(counts).astype(np.float64)
    nb = site.shape[0]
    sh, lbp = np.zeros(nb, dtype=np.int64), np.zeros(nb, dtype=np.int64)
    for i in range(nb):
        Lw = _seqsum(w[None, :] * site[i])                         # [3]
        Ls = _seqsum(c[:, None, :] * site[i][None])                 # [N, 3]
        delta = Lw[0] - max(Lw[1], Lw[2])
        cs = np.sort(Ls - Lw[None, :], axis=1)
        sh[i] = int((delta > (cs[:, 2] - cs[:, 1]) + SH_TOL).sum())
        lbp[i] = int((Ls[:, 0] >= np.maximum(Ls[:, 1], Ls[:, 2])).sum())
    return sh, lbp


def branch_support(children, brlen, tips, weights, model: O.Model, n_rell: int, seed: int, rep0: int = 0):
    """Everything nnj_llh_branch_support computes for one tree, plus the sites: dict(branch_node, llh [nb, 3], nni_brlen [nb, 2, 5],
    sh_count, lbp_count [nb], site [nb, 3, L])."""
    w = np.asarray(weights, dtype=np.float64)
    t, D, N, U, NU = u_vectors(children, brlen, tips, model)
    c1, c2 = (int(x) for x in np.asarray(children)[-1])
    l0 = O.log_sites(*O.root_terms(children, brlen, tips, model))
    L0 = float((w * l0).sum())
    nodes = internal_branches(children)
    llh, lens, site = np.zeros((len(nodes), 3)), np.zeros((len(nodes), 2, 5)), np.zeros((len(nodes), 3, tips.shape[1]))
    for i, v in enumerate(nodes):
        llh[i, 0], site[i, 0] = L0, l0
        vecs, cnts, ql = _quartet(children, v, t, D, N, U, NU)
        for k in (1, 2):
            llh[i, k], lens[i, k - 1], site[i, k] = _optimize(_Quartet(vecs, cnts, ql, k, tips, model), w)
    counts = rell_counts(w, seed, np.arange(rep0, rep0 + n_rell, dtype=np.uint64))
    sh, lbp = rell_stats(site, w, counts) if len(nodes) else (np.zeros(0, np.int64), np.zeros(0, np.int64))
    return dict(branch_node=np.asarray(nodes, dtype=np.int32), llh=llh, nni_brlen=lens, sh_count=sh, lbp_count=lbp, site=site)
