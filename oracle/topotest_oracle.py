"""CPU oracle (test infrastructure) of the tree topology test (DESIGN.md 13; csrc/nnj_llh_topo.cu): multiscale RELL counts, replicate
totals, winner counts, KH, SH, expected likelihood weights and the AU fit.  numpy fp64 on top of support_oracle's Philox and
alrt_oracle's sequential sum; scipy's normal distribution for the AU fit (the library uses Python's statistics.NormalDist).

    scale_draws(n, s)                                n_s = floor((5 + s) / 10 * n + 0.5)
    multiscale_counts(weights, seed, s, reps)        [len(reps), L] counts of replicates `reps` of scale s (Philox word 3 = s + 1)
    totals(site, counts)                             T [N, K] = sum_p c[j, p] l[k, p], pattern order, products rounded then added
    observed(site, weights)                          L [K]
    stats(T_scales, L)                               win [10, K], kh [K], sh [K], elw [K] from the totals of the 10 scales
    au_fit(win_s, n_s, n, N)                         p-AU, the weighted least-squares fit by its closed-form 2 x 2 normal equations
    topology_test(site, weights, n_boot, seed)       everything nnj_llh_topology_test returns, from per-pattern log-likelihoods
"""
from __future__ import annotations

import math

import numpy as np
from scipy import special

from alrt_oracle import _MASK32, _seqsum
from support_oracle import philox4x32_10

SCALES, REF = 10, 5


def scale_draws(n: int, s: int) -> int:
    return int(math.floor((5 + s) / 10 * n + 0.5))


def multiscale_counts(weights, seed: int, s: int, reps, draws=None, word3=None) -> np.ndarray:
    """[len(reps), L] int64: replicate j of scale s makes n_s draws; draw i is site (x0 * n) >> 32, x0 = Philox word 0 of counter
    (i, j lo, j hi, s + 1), key (seed lo, seed hi); pattern p owns the sites cum[p] <= u < cum[p+1].  `draws` / `word3` override
    n_s / s + 1 (draws = n, word3 = 0 is the aLRT stream of alrt_oracle.rell_counts)."""
    w = np.asarray(weights, dtype=np.float64)
    assert (w >= 0).all() and (w == np.floor(w)).all()
    cum = np.concatenate([[0], np.cumsum(w.astype(np.int64))])
    n = int(cum[-1])
    m = scale_draws(n, s) if draws is None else int(draws)
    w3 = s + 1 if word3 is None else int(word3)
    reps = np.asarray(reps, dtype=np.uint64)
    P = len(w)
    out = np.zeros((len(reps), P), dtype=np.int64)
    step = max(1, (1 << 20) // max(m, 1))                   # replicates per vectorised block
    for j0 in range(0, len(reps), step):
        r = np.repeat(reps[j0:j0 + step], m)
        i = np.tile(np.arange(m, dtype=np.uint64), len(r) // max(m, 1))
        x0 = philox4x32_10((i, r & _MASK32, r >> np.uint64(32), np.full_like(i, w3)), (seed & 0xFFFFFFFF, seed >> 32))[0]
        u = ((x0 * np.uint64(n)) >> np.uint64(32)).astype(np.int64)
        row = np.repeat(np.arange(len(r) // max(m, 1)), m)
        p = np.searchsorted(cum, u, side="right") - 1
        out[j0:j0 + step] = np.bincount(row * P + p, minlength=(len(r) // max(m, 1)) * P).reshape(-1, P)
    return out


def totals(site, counts, block: int = 256) -> np.ndarray:
    """site [K, P], counts [N, P] -> T [N, K]: each product rounded, then added in pattern order (blocks of replicates bound memory)."""
    site = np.asarray(site, dtype=np.float64)
    c = np.asarray(counts).astype(np.float64)
    out = np.zeros((c.shape[0], site.shape[0]))
    for j0 in range(0, c.shape[0], block):
        out[j0:j0 + block] = _seqsum(c[j0:j0 + block, None, :] * site[None])
    return out


def observed(site, weights) -> np.ndarray:
    return _seqsum(np.asarray(weights, dtype=np.float64)[None, :] * np.asarray(site, dtype=np.float64))


def stats(T, L):
    """T [10, N, K] replicate totals of every scale, L [K] -> (win [10, K], kh [K], sh [K], elw [K]) as DESIGN.md 13 defines them."""
    T = np.asarray(T, dtype=np.float64)
    L = np.asarray(L, dtype=np.float64)
    N = T.shape[1]
    win = np.stack([(Ts >= Ts.max(1, keepdims=True)).sum(0) for Ts in T]).astype(np.int64)
    T5 = T[REF]
    m = _seqsum(T5.T) / N                                   # sums over j, in j order
    a = T5 - m[None, :]
    ks = int(np.argmax(L))                                  # the lowest index on a tie
    d = L[ks] - L
    kh = (a[:, ks:ks + 1] - a >= d[None, :]).sum(0).astype(np.int64)
    sh = (a.max(1, keepdims=True) - a >= d[None, :]).sum(0).astype(np.int64)
    e = np.exp(T5 - T5.max(1, keepdims=True))
    q = e / _seqsum(e)[:, None]                             # the sum over trees in k order
    elw = _seqsum(q.T) / N
    return win, kh, sh, elw


def au_fit(win_s, n_s, n: int, N: int) -> float:
    """p-AU of one tree from its winner counts at the 10 scales: z_s = Phi^-1(1 - bp_s), weights N phi(z)^2 / (bp (1 - bp)), z ~ v sqrt(r)
    + c / sqrt(r) without an intercept, p = 1 - Phi(v - c); with fewer than two scales where 0 < win < N, bp at scale 5."""
    win_s = np.asarray(win_s, dtype=np.float64)
    r = np.asarray(n_s, dtype=np.float64) / n
    use = (win_s > 0) & (win_s < N)
    if use.sum() < 2:
        return float(win_s[REF] / N)
    bp, r = win_s[use] / N, r[use]
    z = special.ndtri(1.0 - bp)
    W = N * (np.exp(-0.5 * z * z) / math.sqrt(2 * math.pi)) ** 2 / (bp * (1.0 - bp))
    x1, x2 = np.sqrt(r), 1.0 / np.sqrt(r)
    a11, a12, a22 = (W * x1 * x1).sum(), (W * x1 * x2).sum(), (W * x2 * x2).sum()
    b1, b2 = (W * x1 * z).sum(), (W * x2 * z).sum()
    det = a11 * a22 - a12 * a12
    v = (a22 * b1 - a12 * b2) / det
    c = (a11 * b2 - a12 * b1) / det
    return float(special.ndtr(-(v - c)))


def topology_test(site, weights, n_boot: int, seed: int):
    """From per-pattern log-likelihoods site [K, P]: dict(llh, win [10, K], kh, sh, elw, p_au [K])."""
    w = np.asarray(weights, dtype=np.float64)
    n = int(w.sum())
    L = observed(site, w)
    reps = np.arange(n_boot, dtype=np.uint64)
    T = np.stack([totals(site, multiscale_counts(w, seed, s, reps)) for s in range(SCALES)])
    win, kh, sh, elw = stats(T, L)
    n_s = [scale_draws(n, s) for s in range(SCALES)]
    p_au = np.array([au_fit(win[:, k], n_s, n, n_boot) for k in range(site.shape[0])])
    return dict(llh=L, win=win, kh=kh, sh=sh, elw=elw, p_au=p_au)
