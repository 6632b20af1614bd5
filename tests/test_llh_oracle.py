"""CPU tests of the likelihood oracle (oracle/llh_oracle.py) and of the host logic of neuralnj_b200/likelihood.py.
Parity against RAxML-NG is unpinned (the library is absent); these are the anchors named in the oracle's header."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import llh_oracle as O  # noqa: E402

from neuralnj_b200 import _lib, likelihood as LH  # noqa: E402
from neuralnj_b200.treeutil import rf_distance, treestr_to_tuples  # noqa: E402

YANG_1994 = [0.0334, 0.2519, 0.8203, 2.8944]        # discrete gamma, alpha = 0.5, 4 classes, class means (published table value)


def _model():
    return O.Model(rates6=(1.2, 3.1, 0.8, 1.1, 4.2, 1.0), freqs=(0.3, 0.2, 0.2, 0.3), alpha=0.7, pinv=0.15)


def test_discrete_gamma_known_answer():
    assert np.allclose(O.gamma_rates(0.5), YANG_1994, atol=5e-5)
    assert abs(O.gamma_rates(0.5).mean() - 1.0) < 1e-12
    buf = (C.c_double * 4)()
    L = _lib.lib()
    for alpha in (0.021, 0.5, 1.0, 3.7, 99.0):
        assert L.nnj_gamma_rates(alpha, 4, buf) == 0
        assert np.allclose(np.array(buf[:]), O.gamma_rates(alpha), rtol=1e-9, atol=1e-300)
    assert L.nnj_gamma_rates(-1.0, 4, buf) != 0


def test_transition_matrices_are_stochastic_and_reversible():
    m = _model()
    for t in (1e-6, 0.1, 2.0, 50.0):
        P = m.pmats(t)
        assert np.allclose(P.sum(2), 1.0, atol=1e-12) and (P > -1e-14).all()
        assert np.allclose(m.freqs[:, None] * P[1], (m.freqs[:, None] * P[1]).T, atol=1e-13)     # detailed balance
    assert np.allclose(m.pmats(80.0)[3], np.tile(m.freqs, (4, 1)), atol=1e-6)


@pytest.mark.parametrize("R,seed", [(3, 0), (4, 1), (5, 2), (6, 3)])
def test_pruning_equals_bruteforce(R, seed):
    rng = np.random.default_rng(seed)
    m = _model()
    ch, bl = O.random_tree(R, rng)
    tips = O.simulate(ch, bl, R, 25, m, rng, gap_frac=0.15)
    tips[0, :3] = 5            # an ambiguity code (A or G)
    w = rng.integers(1, 4, size=25).astype(float)
    brute = O.loglik_bruteforce(ch, bl, tips, w, m)
    for scaling in (True, False):
        assert abs(O.loglik(ch, bl, tips, w, m, scaling=scaling) - brute) < 1e-9
    assert abs(O.loglik_logspace(ch, bl, tips, w, m) - brute) < 1e-9


def _iid(R, L, rng):
    return (1 << rng.integers(0, 4, size=(R, L))).astype(np.uint8)


def _underflows(ch, bl, tips, m):
    """Patterns whose unscaled site likelihood is 0 or subnormal in fp64."""
    with np.errstate(all="ignore"):
        s = O.site_likelihoods(ch, bl, tips, m, scaling=False)
    return int((s < np.finfo(np.float64).tiny).sum())


@pytest.mark.parametrize("R,L", [(3, 40), (12, 200), (50, 300), (130, 300)])
def test_scaling_changes_nothing_where_it_does_not_trigger(R, L):
    rng = np.random.default_rng(R)
    m = _model()
    ch, bl = O.random_tree(R, rng)
    tips = O.simulate(ch, bl, R, L, m, rng, gap_frac=0.05)
    pat, w = O.compress_patterns(tips)
    assert not O.root_terms(ch, bl, pat, m)[1].any()
    a, b = O.loglik(ch, bl, pat, w, m), O.loglik(ch, bl, pat, w, m, scaling=False)
    assert a == b and abs(a - O.loglik_logspace(ch, bl, pat, w, m)) < 1e-12 * abs(a)


# Each case underflows fp64 without scaling (asserted), so it pins the scaled pruning against the log-space one.
SCALED_CASES = [(300, 300, "iid", 0.1, 50.0), (512, 300, "iid", 1.0, 0.5), (1000, 200, "sim", 1.0, None), (4096, 64, "sim", 1.0, None)]


@pytest.mark.parametrize("R,L,kind,scale,alpha", SCALED_CASES)
def test_scaled_pruning_matches_logspace(R, L, kind, scale, alpha):
    rng = np.random.default_rng(R)
    gen = _model()
    ch, bl = O.random_tree(R, rng)
    tips = O.simulate(ch, bl, R, L, gen, rng, gap_frac=0.05) if kind == "sim" else _iid(R, L, rng)
    pat, w = O.compress_patterns(tips)
    m = gen if alpha is None else O.Model(alpha=alpha)
    bl = bl * scale
    assert _underflows(ch, bl, pat, m) > 0
    with np.errstate(divide="ignore"):
        assert not np.isfinite(O.loglik(ch, bl, pat, w, m, scaling=False)) or _underflows(ch, bl, pat, m) > 0
    got = O.loglik(ch, bl, pat, w, m)
    assert np.isfinite(got) and O.root_terms(ch, bl, pat, m)[1].max() >= 1
    assert abs(got - O.loglik_logspace(ch, bl, pat, w, m)) < 1e-10 * abs(got)


def test_scaled_optimiser_equals_unscaled_where_nothing_scales():
    rng = np.random.default_rng(12)
    m = _model()
    ch, bl = O.random_tree(30, rng)
    tips = O.simulate(ch, bl, 30, 300, m, rng, gap_frac=0.05)
    pat, w = O.compress_patterns(tips)
    start = np.full(58, O.BRLEN_DEFAULT)
    t1, b1, a1 = O.optimize_branches(ch, start, pat, w, m)
    t2, b2, a2 = O.optimize_branches(ch, start, pat, w, m, scaling=False)
    assert abs(a1 - a2) < 1e-12 * abs(a2) and abs(b1 - b2) < 1e-12 * abs(b2) and np.allclose(t1, t2, rtol=1e-12, atol=0)


def test_scaled_optimiser_on_an_underflowing_tree():
    """300 iid taxa at 0.1x lengths: every site underflows unscaled at the start; the optimiser climbs, and the log-space
    pruning reproduces its reported maximum at the returned lengths."""
    R, L = 300, 60
    rng = np.random.default_rng(30)
    ch, bl = O.random_tree(R, rng)
    tips = _iid(R, L, rng)
    m = O.Model(alpha=50.0)
    start = bl * 0.1
    assert _underflows(ch, start, tips, m) == L
    t, before, after = O.optimize_branches(ch, start, tips, np.ones(L), m, max_passes=2)
    assert np.isfinite(before) and after > before
    assert abs(O.loglik_logspace(ch, start, tips, np.ones(L), m) - before) < 1e-10 * abs(before)
    assert abs(O.loglik_logspace(ch, t, tips, np.ones(L), m) - after) < 1e-10 * abs(after)


def test_lengths_are_clamped_in_evaluation():
    """Zero, negative and huge lengths score as the clamped lengths [BRLEN_MIN, BRLEN_MAX]; the root branch is clamped as one."""
    rng = np.random.default_rng(6)
    m = _model()
    ch, bl = O.random_tree(8, rng)
    tips = O.simulate(ch, bl, 8, 50, m, rng)
    w = np.ones(50)
    c1, c2 = ch[-1]
    odd = bl.copy()
    odd[[0, 3]] = 0.0
    odd[5] = -0.3
    odd[7] = 250.0
    odd[c1], odd[c2] = 70.0, 60.0
    ref = bl.copy()
    ref[[0, 3, 5]] = O.BRLEN_MIN
    ref[7] = O.BRLEN_MAX
    ref[c1], ref[c2] = O.BRLEN_MAX, 0.0
    got = O.loglik(ch, odd, tips, w, m)
    assert np.isfinite(got) and got == O.loglik(ch, ref, tips, w, m)
    assert abs(got - O.loglik_logspace(ch, odd, tips, w, m)) < 1e-10 * abs(got)
    # two different tips on zero-length branches: the true site likelihood at length 0 is 0; clamped it is tiny and positive
    ch3 = np.array([[0, 1], [3, 2]], dtype=np.int32)
    tips3 = np.array([[1], [2], [1]], dtype=np.uint8)
    s = O.site_likelihoods(ch3, np.array([0.0, 0.0, 0.1, 0.1]), tips3, O.Model(pinv=0.0))
    assert s[0] > 0 and abs(s[0] - O.site_likelihoods(ch3, np.array([1e-6, 1e-6, 0.1, 0.1]), tips3, O.Model(pinv=0.0))[0]) == 0


def test_jc69_two_taxon_closed_form():
    rng = np.random.default_rng(5)
    L, p = 2000, 0.21
    a = rng.integers(0, 4, size=L)
    b = a.copy()
    diff = rng.choice(L, size=int(p * L), replace=False)
    b[diff] = (a[diff] + rng.integers(1, 4, size=len(diff))) % 4
    tips = (1 << np.stack([a, b])).astype(np.uint8)
    m = O.Model(gamma=False)
    t, _, _ = O.optimize_branches(np.array([[0, 1]]), np.array([0.3, 0.3]), tips, np.ones(L), m)
    assert abs((t[0] + t[1]) - (-0.75 * np.log(1 - 4 * p / 3))) < 1e-6


def test_pattern_compression_preserves_the_likelihood():
    rng = np.random.default_rng(7)
    m = _model()
    ch, bl = O.random_tree(8, rng)
    tips = O.simulate(ch, bl, 8, 400, m, rng, gap_frac=0.05)
    pat, w = O.compress_patterns(tips)
    assert pat.shape[1] < 400 and w.sum() == 400
    assert abs(O.loglik(ch, bl, tips, np.ones(400), m) - O.loglik(ch, bl, pat, w, m)) < 1e-8
    p2, w2 = LH.compress_patterns(tips)
    assert np.array_equal(p2, pat) and np.array_equal(w2, w)


def test_branch_optimiser_is_monotone_and_stationary():
    rng = np.random.default_rng(11)
    m = _model()
    ch, bl = O.random_tree(10, rng)
    tips = O.simulate(ch, bl, 10, 300, m, rng, gap_frac=0.05)
    pat, w = O.compress_patterns(tips)
    start = np.full(18, O.BRLEN_DEFAULT)
    prev = O.loglik(ch, start, pat, w, m)
    t = start
    for passes in (1, 2, 4, 32):
        t, before, after = O.optimize_branches(ch, start, pat, w, m, max_passes=passes, eps=1e-9)
        assert after >= prev - 1e-9
        prev = after
    assert after > O.loglik(ch, bl, pat, w, m)                     # beats the generating lengths on the sample
    assert abs(O.loglik(ch, t, pat, w, m) - after) < 1e-8          # the returned (root-split) lengths give that likelihood
    for v in range(18):
        if t[v] <= 2 * O.BRLEN_MIN:
            continue
        up, dn = t.copy(), t.copy()
        up[v] += 1e-5
        dn[v] -= 1e-5
        assert abs(O.loglik(ch, up, pat, w, m) - O.loglik(ch, dn, pat, w, m)) / 2e-5 < 0.05


def test_schedule_visits_every_branch_once():
    rng = np.random.default_rng(3)
    for R in (3, 4, 9, 30):
        ch, _ = O.random_tree(R, rng)
        ops = O.build_ops(ch, R)
        opt = sorted(int(v) for op, v, _, _ in ops if op == O.OP_OPT)
        c2 = int(ch[-1][1])
        assert opt == sorted(set(range(2 * R - 2)) - {c2})         # 2R-3 branches of the unrooted tree
        assert len(ops) <= 5 * R


def test_tree_array_conversions_round_trip():
    rng = np.random.default_rng(4)
    R = 9
    labels = [f"taxon{i}" for i in range(R)]
    ch, bl = O.random_tree(R, rng)
    rooted = LH.tuples_to_newick(LH.tuples_with_lengths(ch, bl, labels, unrooted=False))
    unrooted = LH.tuples_to_newick(LH.tuples_with_lengths(ch, bl, labels, unrooted=True))
    assert rf_distance(rooted, unrooted) == 0
    for text in (rooted, unrooted):
        ch2, bl2 = LH.tree_arrays_from_tuples(treestr_to_tuples(text), labels)
        assert ch2.shape == (R - 1, 2)
        again = LH.tuples_to_newick(LH.tuples_with_lengths(ch2, bl2, labels, unrooted=True))
        assert rf_distance(again, rooted) == 0
        m = _model()
        tips = O.simulate(ch, bl, R, 60, m, rng)
        assert abs(O.loglik(ch, bl, tips, np.ones(60), m) - O.loglik(ch2, bl2, tips, np.ones(60), m)) < 1e-6      # lengths print with 8 decimals
    # NJ merge list -> children: slot i <- new node, slot j removed
    merges = np.array([[0, 1], [1, 2], [0, 1]])
    assert LH.children_from_merges(merges, 4).tolist() == [[0, 1], [2, 3], [4, 5]]
    with pytest.raises(ValueError):
        LH.tree_arrays_from_tuples(treestr_to_tuples("(a:1,(b:1,zz:1):1);"), ["a", "b", "c"])


def test_masks_and_frequencies():
    m = LH.sequences_to_masks(["ACGT-NRY", "acgu?xkm"])
    assert m.tolist() == [[1, 2, 4, 8, 15, 15, 5, 10], [1, 2, 4, 8, 15, 15, 12, 3]]
    onehot = np.array([[[1, 0, 0, 0], [1, 1, 1, 1], [0, 0, 0, 0], [0, 0, 0, 1]]], dtype=np.int8)
    assert LH.onehot_to_masks(onehot).tolist() == [[1, 15, 15, 8]]
    f = LH.empirical_freqs(LH.sequences_to_masks(["AAAC", "GGTT", "RR--"]))
    assert abs(f.sum() - 1) < 1e-12 and np.allclose(f, O.empirical_freqs(LH.sequences_to_masks(["AAAC", "GGTT", "RR--"])), atol=1e-3)
    sm = LH.SubstModel("GTR+I+G", f, 2)
    packed = sm.pack()
    ref = O.Model(freqs=f, alpha=1.0, pinv=0.0).packed()
    assert packed.shape == (2, 64) and packed[0, 46] == 7.0 and np.allclose(packed[0, 48:54], 1.0)
    # eigenvectors are defined up to sign / order within degenerate eigenvalues: compare what they generate
    lam, U, Ui = packed[0, :4], packed[0, 4:20].reshape(4, 4), packed[0, 20:36].reshape(4, 4)
    P = U @ np.diag(np.exp(lam * 0.3)) @ Ui
    assert np.allclose(P, ref[4:20].reshape(4, 4) @ np.diag(np.exp(ref[:4] * 0.3)) @ ref[20:36].reshape(4, 4), atol=1e-12)
    assert np.allclose(packed[0, 36:45], ref[36:45])
    with pytest.raises(ValueError):
        LH.SubstModel("WAG+G", f, 1)
