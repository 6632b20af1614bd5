"""CPU tests of the tree topology test (DESIGN.md 13): the multiscale RELL draw rule, the AU fit of the library against the oracle's
closed form (oracle/topotest_oracle.py), the replicate statistics on a worked case, the result table and the command-line checks."""
import math
import os
import sys

import numpy as np
import pytest
from scipy import special

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import alrt_oracle as A  # noqa: E402
import topotest_oracle as TO  # noqa: E402
from support_oracle import philox4x32_10  # noqa: E402

from neuralnj_b200 import support as SUP  # noqa: E402

W = np.array([3.0, 0.0, 2.0, 5.0, 0.0, 1.0, 4.0])
SEED = 0x1234_5678_9ABC


def test_scale_draws():
    for n in (1, 2, 7, 15, 1000, 1023, 2 ** 31 - 1):
        ns = SUP.scale_draws(n)
        assert ns == [TO.scale_draws(n, s) for s in range(10)]
        assert ns[5] == n and all(a <= b for a, b in zip(ns, ns[1:])) and ns[0] >= 1
    assert SUP.scale_draws(15) == [8, 9, 11, 12, 14, 15, 17, 18, 20, 21]


def test_multiscale_draw_rule():
    n = int(W.sum())
    cum = np.concatenate([[0], np.cumsum(W.astype(np.int64))])
    for s in (0, 5, 9):
        c = TO.multiscale_counts(W, SEED, s, np.arange(12, dtype=np.uint64))
        assert (c.sum(1) == TO.scale_draws(n, s)).all() and (c[:, [1, 4]] == 0).all()
        # replicate 7 by hand: counter (i, 7, 0, s + 1)
        m = TO.scale_draws(n, s)
        x0 = philox4x32_10((np.arange(m, dtype=np.uint64), np.full(m, 7, np.uint64), np.zeros(m, np.uint64), np.full(m, s + 1, np.uint64)),
                           (SEED & 0xFFFFFFFF, SEED >> 32))[0]
        u = (x0.astype(np.uint64) * np.uint64(n)) >> np.uint64(32)
        p = [int(np.searchsorted(cum, int(x), side="right") - 1) for x in u]
        assert np.array_equal(np.bincount(p, minlength=len(W)), c[7])
    # scale 5 draws n sites like the aLRT replicates, from another stream (counter word 3 = 6, not 0)
    reps = np.arange(20, dtype=np.uint64)
    c5 = TO.multiscale_counts(W, SEED, 5, reps)
    alrt = A.rell_counts(W, SEED, reps)
    assert not np.array_equal(c5, alrt)
    assert np.array_equal(TO.multiscale_counts(W, SEED, 5, reps, draws=n, word3=0), alrt)
    # replicate indices from 2^32 on use the high counter word
    hi = TO.multiscale_counts(W, SEED, 5, np.array([2 ** 32 + 3], dtype=np.uint64))
    assert hi.sum() == n and not np.array_equal(hi[0], c5[3])


def test_totals_are_sequential_sums():
    rng = np.random.default_rng(3)
    site = -rng.uniform(0.1, 9.0, size=(4, 7))
    c = TO.multiscale_counts(W, SEED, 2, np.arange(6, dtype=np.uint64))
    T = TO.totals(site, c, block=4)
    for j in range(6):
        for k in range(4):
            acc = 0.0
            for p in range(7):
                acc = acc + float(c[j, p]) * site[k, p]
            assert T[j, k] == acc
    assert np.array_equal(TO.observed(site, W), np.array([sum(W[p] * site[k, p] for p in range(7)) for k in range(4)]))


# three trees, five replicates at every scale; scale 5 has means -101, -101, -102 (exact) and a tie in replicate 4
T5 = np.array([[-100.0, -101.0, -102.0],
               [-101.0, -100.0, -104.0],
               [-100.0, -102.0, -101.0],
               [-103.0, -101.0, -100.0],
               [-101.0, -101.0, -103.0]])
LOBS = np.array([-100.0, -101.0, -103.0])


def _scales(T5):
    T = np.stack([T5 + 0.25 * s for s in range(10)])
    T[0] = T5[:, ::-1]                    # scale 0: other winners
    return T


def test_statistics_worked_case():
    win, kh, sh, elw = TO.stats(_scales(T5), LOBS)
    assert list(win[5]) == [3, 2, 1]      # replicate 4 ties trees 0 and 1: both win
    assert list(win[0]) == [1, 2, 3]
    # centred values a = T - m: [1,0,0], [0,1,-2], [1,-1,1], [-2,0,2], [0,0,-1]; L* - L = 0, 1, 3
    assert list(kh) == [5, 2, 0]
    assert list(sh) == [5, 3, 1]
    e = np.exp(T5 - T5.max(1, keepdims=True))
    want = np.array([sum(e[j, k] / sum(e[j]) for j in range(5)) / 5 for k in range(3)])
    np.testing.assert_allclose(elw, want, rtol=0, atol=1e-15)
    assert abs(elw.sum() - 1.0) < 1e-12
    assert (sh >= kh).all() and kh[0] == sh[0] == 5


def test_statistics_invariants_and_identical_trees():
    rng = np.random.default_rng(5)
    T = -1000.0 + rng.normal(0, 3.0, size=(10, 40, 6))
    T[:, :, 4] = T[:, :, 1]               # tree 4 is tree 1 again
    L = -1000.0 + rng.normal(0, 3.0, size=6)
    L[4] = L[1]
    win, kh, sh, elw = TO.stats(T, L)
    ks = int(np.argmax(L))
    assert (sh >= kh).all() and kh[ks] == sh[ks] == 40
    assert abs(elw.sum() - 1.0) < 1e-12
    assert (win[:, 4] == win[:, 1]).all() and kh[4] == kh[1] and sh[4] == sh[1] and elw[4] == elw[1]
    assert (win.sum(1) >= 40).all()


@pytest.mark.parametrize("v,c", [(0.5, 0.2), (-1.0, 0.3), (1.2, -0.4), (0.0, 0.0)])
def test_au_fit_recovers_exact_curves(v, c):
    n, N = 1000, 10000
    n_s = SUP.scale_draws(n)
    r = np.asarray(n_s) / n
    bp = special.ndtr(-(v * np.sqrt(r) + c / np.sqrt(r)))
    want = float(special.ndtr(-(v - c)))
    assert SUP.au_pvalue(bp * N, n_s, n, N) == pytest.approx(want, abs=1e-9)
    assert TO.au_fit(bp * N, n_s, n, N) == pytest.approx(want, abs=1e-9)


def test_au_fit_matches_oracle_on_counts():
    rng = np.random.default_rng(11)
    n, N = 777, 1000
    n_s = SUP.scale_draws(n)
    for _ in range(20):
        win = np.sort(rng.integers(1, N, size=10))[::-1]
        assert SUP.au_pvalue(win, n_s, n, N) == pytest.approx(TO.au_fit(win, n_s, n, N), abs=1e-9)


def test_au_fit_degenerate_rules():
    n, N = 500, 200
    n_s = SUP.scale_draws(n)
    for f in (SUP.au_pvalue, TO.au_fit):
        assert f([0] * 10, n_s, n, N) == 0.0
        assert f([N] * 10, n_s, n, N) == 1.0
        one = [N] * 5 + [70] + [N] * 4      # only scale 5 is usable: bp-RELL
        assert f(one, n_s, n, N) == pytest.approx(70 / N)
        one = [0] * 7 + [30] + [0] * 2      # only scale 7 is usable: bp-RELL (0)
        assert f(one, n_s, n, N) == 0.0


def test_table_rows_and_marks():
    llh = np.array([-10.0, -12.5])
    t = SUP.topology_table(llh, llh.max() - llh, [0.9, 0.1], [1.0, 0.04], [1.0, 0.2], [0.8, 0.2], [0.95, 0.01])
    lines = t.splitlines()
    assert lines[0].split() == ["Tree", "logL", "deltaL", "bp-RELL", "p-KH", "p-SH", "c-ELW", "p-AU"] and set(lines[1]) == {"-"}
    row = lines[3].split()
    assert row[:3] == ["2", "-12.5000", "2.5000"] and row[3:] == ["0.1000", "+", "0.0400", "-", "0.2000", "+", "0.2000", "+", "0.0100", "-"]


def test_cli_rejects_topotest_with_argmax_and_one_candidate():
    from neuralnj_b200.rollout import main
    with pytest.raises(SystemExit, match="--topotest applies to --infer_opt Search"):
        main(["--infer_opt", "Argmax", "--topotest", "100"])
    with pytest.raises(SystemExit, match="--topotest_top must be at least 2"):
        main(["--infer_opt", "Search", "--topotest", "100", "--topotest_top", "1"])
