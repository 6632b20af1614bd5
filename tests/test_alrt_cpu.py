"""CPU tests of likelihood branch support (DESIGN.md 12): the internal-branch list, the NNI alternative trees, the quartet oracle
(oracle/alrt_oracle.py) against whole-tree likelihoods, the RELL draws and the statistics on worked cases."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import alrt_oracle as A  # noqa: E402
import llh_oracle as O  # noqa: E402
from support_oracle import philox4x32_10  # noqa: E402

from neuralnj_b200 import likelihood as LH  # noqa: E402
from neuralnj_b200.treeutil import bipartitions  # noqa: E402

GEN = O.Model(rates6=(1.2, 3.1, 0.8, 1.1, 4.2, 1.0), freqs=(0.3, 0.2, 0.2, 0.3), alpha=0.7, pinv=0.15)


def caterpillar(R):
    ch = [(0, 1)] + [(R + k, k + 2) for k in range(R - 2)]
    return np.asarray(ch, dtype=np.int32)


def balanced(R):
    cur, ch = list(range(R)), []
    while len(cur) > 1:
        nxt = []
        for i in range(0, len(cur) - 1, 2):
            ch.append((cur[i], cur[i + 1]))
            nxt.append(R + len(ch) - 1)
        if len(cur) % 2:
            nxt.append(cur[-1])
        cur = nxt
    return np.asarray(ch, dtype=np.int32)


def trees(R, rng, n=6):
    out = [O.random_tree(R, rng)[0] for _ in range(n)] + [caterpillar(R), balanced(R)]
    return out


def newick(ch, R):
    return LH.tuples_to_newick(LH.tuples_with_lengths(ch, np.full(2 * R - 2, 0.1), [f"t{i}" for i in range(R)], unrooted=True))


def root_case(ch, R):
    c1, c2 = (int(c) for c in ch[-1])
    return "both inner" if c1 >= R and c2 >= R else "one leaf"


@pytest.mark.parametrize("R", [3, 4, 5, 6, 9, 16, 33, 64])
def test_internal_branches_count_and_root_cases(R):
    rng = np.random.default_rng(R)
    seen = set()
    for ch in trees(R, rng, 12):
        nodes = LH.internal_branches(ch)
        assert len(nodes) == max(R - 3, 0) and nodes == sorted(nodes) and nodes == A.internal_branches(ch)
        c1, c2 = (int(c) for c in ch[-1])
        assert c2 not in nodes and (c1 in nodes) == (c1 >= R and c2 >= R)
        seen.add(root_case(ch, R))
        # one branch per non-trivial split of the unrooted tree
        assert len(bipartitions(newick(ch, R))) == len(nodes)
    if R >= 5:
        assert seen == {"both inner", "one leaf"}


@pytest.mark.parametrize("R", [4, 5, 7, 12, 30])
def test_nni_tree_changes_one_bipartition(R):
    rng = np.random.default_rng(100 + R)
    for ch in trees(R, rng, 4):
        base = bipartitions(newick(ch, R))
        for v in LH.internal_branches(ch):
            alts = []
            for k in (0, 1, 2):
                alt = LH.nni_tree(ch, v, k)
                assert alt.shape == (R - 1, 2)
                used = alt.ravel().tolist()
                assert sorted(used) == list(range(2 * R - 2))
                assert all(c < R + j for j, pair in enumerate(alt.tolist()) for c in pair)     # join order
                bp = bipartitions(newick(alt, R))
                alts.append(bp)
                assert len(bp ^ base) == (0 if k == 0 else 2), (v, k)
            assert alts[1] != alts[2] and alts[0] != alts[1]


def _sim(R, L, seed, iid=False):
    rng = np.random.default_rng(seed)
    ch, bl = O.random_tree(R, rng)
    tips = (1 << rng.integers(0, 4, size=(R, L))).astype(np.uint8) if iid else O.simulate(ch, bl, R, L, GEN, rng, gap_frac=0.05)
    pats, w = O.compress_patterns(tips)
    return ch, bl, pats, w


@pytest.mark.parametrize("R", [4, 5, 8, 20])
def test_configuration0_reproduces_the_tree(R):
    for ch, bl, pats, w in [_sim(R, 150, R), _sim(R, 150, R + 1, iid=True)] + [(caterpillar(R), *_sim(R, 150, R + 2)[1:])]:
        ref = O.loglik(ch, bl, pats, w, GEN)
        for v in LH.internal_branches(ch):
            got = float((w * A.quartet_sites(ch, bl, pats, GEN, v, 0)).sum())
            assert abs(got - ref) <= 1e-12 * abs(ref), (R, v)


def _explicit(ch, v, k, lens, bl):
    """The alternative tree of the branch above v with the five quartet lengths set, or None where the rooted form cannot hold a
    root-branch length below 2e-6 (each root half is clamped to 1e-6 on its own)."""
    _, edges = LH.quartet(ch, v)
    c1, c2 = (int(c) for c in ch[-1])
    bq = np.array(bl, dtype=np.float64)
    for e, ln in zip(edges, lens):
        if e in (c1, c2):
            if ln < 2e-6:
                return None
            bq[c1] = bq[c2] = 0.5 * ln
        else:
            bq[e] = ln
    return LH.nni_tree(ch, v, k, bq)


@pytest.mark.parametrize("R,L", [(5, 120), (8, 200), (20, 200), (50, 150)])
def test_oracle_alternatives_match_explicit_trees(R, L):
    ch, bl, pats, w = _sim(R, L, 7 * R)
    nodes = LH.internal_branches(ch)
    compared = 0
    for v in nodes[:: max(1, len(nodes) // 6)]:
        for k in (1, 2):
            Lk, lens, site = A.nni_optimize(ch, bl, pats, w, GEN, v, k)
            assert np.isclose(Lk, float((w * site).sum()), rtol=1e-12, atol=0)
            ex = _explicit(ch, v, k, lens, bl)
            if ex is None:
                continue
            ref = O.site_logliks(*ex, pats, GEN)
            assert np.abs(ref - site).max() <= 1e-12 * np.abs(site).max(), (R, v, k)
            compared += 1
    assert compared >= 2


@pytest.mark.parametrize("R", [4, 5, 6])
def test_oracle_against_brute_force(R):
    ch, bl, pats, w = _sim(R, 60, 31 + R)
    for v in LH.internal_branches(ch):
        for k in (1, 2):
            Lk, lens, _ = A.nni_optimize(ch, bl, pats, w, GEN, v, k)
            ex = _explicit(ch, v, k, lens, bl)
            if ex is not None:
                ch2, bl2 = ex
                ref = O.loglik_bruteforce(ch2, bl2, pats, w, GEN)
                assert abs(ref - Lk) <= 1e-11 * abs(ref)


@pytest.mark.parametrize("R", [300, 1000])
def test_oracle_against_logspace_where_scaling_is_active(R):
    rng = np.random.default_rng(R)
    ch, bl = O.random_tree(R, rng)
    tips = (1 << rng.integers(0, 4, size=(R, 24))).astype(np.uint8)      # independent columns: far from any tree, sites underflow
    pats, w = O.compress_patterns(tips)
    assert O.root_terms(ch, bl, pats, GEN)[1].max() > 0          # some vectors are rescaled
    for v in LH.internal_branches(ch)[:: R // 3][:2]:
        Lk, lens, _ = A.nni_optimize(ch, bl, pats, w, GEN, v, 1)
        ex = _explicit(ch, v, 1, lens, bl)
        if ex is not None:
            ref = O.loglik_logspace(*ex, pats, w, GEN)
            assert abs(ref - Lk) <= 1e-10 * abs(ref)


def test_r4_alternatives_equal_whole_tree_optimisation():
    ch, bl, pats, w = _sim(4, 300, 5)
    (v,) = LH.internal_branches(ch)
    for k in (1, 2):
        Lk, _, _ = A.nni_optimize(ch, bl, pats, w, GEN, v, k)
        ch2, bl2 = LH.nni_tree(ch, v, k, bl)
        _, _, ref = O.optimize_branches(ch2, bl2, pats, w, GEN)
        assert abs(Lk - ref) < 2e-3


def test_statistics_worked_cases():
    rng = np.random.default_rng(0)
    L = 40
    w = rng.integers(1, 4, size=L).astype(np.float64)
    counts = A.rell_counts(w, 3, np.arange(200, dtype=np.uint64))
    l0 = -rng.uniform(1.0, 5.0, size=L)
    # l1 = l0: delta = 0, SH-aLRT 0, aBayes 1/3
    site = np.stack([l0, l0, l0])[None]
    sh, lbp = A.rell_stats(site, w, counts)
    assert sh[0] == 0 and lbp[0] == 200
    L0 = float((w * l0).sum())
    assert 1.0 / (1.0 + 2 * np.exp(L0 - L0)) == pytest.approx(1 / 3)
    # l0 dominant at every site: SH-aLRT = LBP = 100 %
    site = np.stack([l0, l0 - 0.5, l0 - 0.7])[None]
    sh, lbp = A.rell_stats(site, w, counts)
    assert sh[0] == 200 and lbp[0] == 200
    # an NNI better than the tree (delta < 0): SH-aLRT 0
    site = np.stack([l0 - 0.1, l0, l0 - 0.7])[None]
    sh, _ = A.rell_stats(site, w, counts)
    assert sh[0] == 0


def test_rell_draw_rule_and_chunk_additivity():
    w = np.array([3.0, 0.0, 2.0, 5.0, 0.0, 1.0])
    n, seed = 11, 0x1234_5678_9ABC
    c = A.rell_counts(w, seed, np.arange(10, dtype=np.uint64))
    assert (c.sum(1) == n).all() and (c[:, [1, 4]] == 0).all()
    # draw i of replicate r by hand
    cum = np.array([0, 3, 3, 5, 10, 10, 11])
    for r in (0, 7):
        x0 = philox4x32_10((np.arange(n, dtype=np.uint64), np.full(n, r, np.uint64), np.zeros(n, np.uint64), np.zeros(n, np.uint64)),
                           (seed & 0xFFFFFFFF, seed >> 32))[0]
        u = (x0.astype(np.uint64) * np.uint64(n)) >> np.uint64(32)
        p = [int(np.searchsorted(cum, int(x), side="right") - 1) for x in u]
        assert np.array_equal(np.bincount(p, minlength=6), c[r])
    # replicate r depends on (seed, r, n) only: chunks add up
    big = A.rell_counts(w, seed, np.arange(0, 30, dtype=np.uint64))
    parts = np.concatenate([A.rell_counts(w, seed, np.arange(a, b, dtype=np.uint64)) for a, b in ((0, 13), (13, 30))])
    assert np.array_equal(big, parts)
    site = -np.random.default_rng(1).uniform(0.5, 3.0, size=(2, 3, 6))
    tot = A.rell_stats(site, w, big)
    s1, s2 = A.rell_stats(site, w, big[:13]), A.rell_stats(site, w, big[13:])
    assert np.array_equal(tot[0], s1[0] + s2[0]) and np.array_equal(tot[1], s1[1] + s2[1])
    # large replicate indices use the high counter word
    hi = A.rell_counts(w, seed, np.array([2 ** 32 + 5], dtype=np.uint64))
    assert hi.sum() == n and not np.array_equal(hi[0], c[5])


def test_cli_rejects_alrt_with_search():
    from neuralnj_b200.rollout import main
    with pytest.raises(SystemExit, match="--alrt applies to --infer_opt Argmax"):
        main(["--infer_opt", "Search", "--alrt", "10"])
