"""GPU tests of the tree topology test (csrc/nnj_llh_topo.cu, DESIGN.md 13) against the numpy oracle oracle/topotest_oracle.py.

The per-pattern log-likelihoods match llh_oracle within 1e-12 relative.  Fed the kernel's own per-pattern log-likelihoods, the oracle
gives exactly the kernel's L_k and integer counts (win, KH, SH), and ELW within 1e-12: every sum runs in one fixed order on both sides."""
import os
import shutil
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import llh_oracle as O  # noqa: E402
import topotest_oracle as TO  # noqa: E402

from neuralnj_b200 import likelihood as LH  # noqa: E402
from neuralnj_b200 import support as SUP  # noqa: E402

pytestmark = pytest.mark.gpu
GOLD = os.path.join(ROOT, "tests", "golden")
GEN = dict(rates6=(1.2, 3.1, 0.8, 1.1, 4.2, 1.0), freqs=(0.3, 0.2, 0.2, 0.3), alpha=0.7, pinv=0.15)


def _children(nested, R):
    """Nested pairs of leaf indices -> children [R-1, 2] in join order."""
    out = []

    def visit(t):
        if isinstance(t, int):
            return t
        a, b = visit(t[0]), visit(t[1])
        out.append((a, b))
        return R + len(out) - 1
    visit(nested)
    return np.asarray(out, dtype=np.int32)


def all_unrooted_5():
    """The 15 unrooted binary topologies of 5 taxa: the 15 rooted trees of taxa 0..3, each joined with taxon 4 at the root."""
    def insert(t, leaf):
        yield (t, leaf)
        if not isinstance(t, int):
            for left in insert(t[0], leaf):
                yield (left, t[1])
            for right in insert(t[1], leaf):
                yield (t[0], right)
    trees = [(0, 1)]
    for leaf in (2, 3):
        trees = [u for t in trees for u in insert(t, leaf)]
    assert len(trees) == 15
    return np.stack([_children((t, 4), 5) for t in trees])


def _sm(K):
    sm = LH.SubstModel("GTR+I+G", np.asarray(GEN["freqs"]), K)
    sm.rates[:] = GEN["rates6"]
    sm.alpha[:] = GEN["alpha"]
    sm.pinv[:] = GEN["pinv"]
    return sm


def _om(sm, k):
    return O.Model(sm.rates[k], sm.freqs[k], sm.alpha[k], sm.pinv[k])


def _case(R, L, K, seed, pad=0):
    """A simulated alignment (compressed; `pad` zero-weight patterns appended) and K trees: the generating tree, then random ones."""
    rng = np.random.default_rng(1000 * R + K + seed)
    ch0, bl0 = O.random_tree(R, rng)
    tips = O.simulate(ch0, bl0, R, L, O.Model(**GEN), rng, gap_frac=0.05)
    pats, w = O.compress_patterns(tips)
    if pad:
        pats = np.concatenate([pats, np.full((R, pad), 15, np.uint8)], 1)
        w = np.concatenate([w, np.zeros(pad)])
    if R == 5 and K == 15:
        ch = all_unrooted_5()
        bl = np.stack([O.random_tree(5, rng)[1] for _ in range(K)])
    else:
        others = [O.random_tree(R, rng) for _ in range(K - 1)]
        ch = np.stack([ch0] + [c for c, _ in others])
        bl = np.stack([bl0] + [b for _, b in others])
    return pats, w, ch, bl


def _check_against_oracle(pats, w, ch, bl, N, seed, fit=True):
    K = ch.shape[0]
    eng = LH.TreeLikelihood(pats, w)
    sm = _sm(K)
    if fit:
        bl, _, _ = eng.optimize_all(ch, bl, sm)
    got = eng.topology_test(ch, bl, sm, N, seed, site_llh=True)
    site = got["site_llh"].cpu().numpy()
    for k in range(K):
        ref = O.site_logliks(ch[k], bl[k], pats, _om(sm, k))
        assert np.abs(site[k] - ref).max() <= 1e-12 * np.abs(ref).max(), k
    ref = TO.topology_test(site, w, N, seed)
    assert np.array_equal(got["llh"], ref["llh"])
    assert np.array_equal(got["win"], ref["win"]) and np.array_equal(got["kh"], ref["kh"]) and np.array_equal(got["sh"], ref["sh"])
    np.testing.assert_allclose(got["elw"], ref["elw"], rtol=0, atol=1e-12)
    assert (got["sh"] >= got["kh"]).all()
    ks = int(np.argmax(got["llh"]))
    assert got["kh"][ks] == got["sh"][ks] == N
    assert abs(got["elw"].sum() - 1.0) <= 1e-12
    return got


CASES = [  # R, sites, K, N, zero-weight padding patterns
    (5, 200, 15, 300, 0),
    (20, 256, 2, 300, 0),
    (20, 256, 15, 200, 3),
    (20, 256, 64, 200, 0),
    (50, 400, 2, 200, 0),
    (50, 400, 15, 200, 5),
    (50, 400, 64, 150, 0),
    (20, 120, 300, 100, 0),      # five tiles of 64 trees
]


@pytest.mark.parametrize("R,L,K,N,pad", CASES)
def test_kernel_matches_oracle(R, L, K, N, pad):
    pats, w, ch, bl = _case(R, L, K, 0, pad)
    _check_against_oracle(pats, w, ch, bl, N, seed=R + K)


def test_more_replicates_than_two_chunks():
    """8300 replicates per scale: three passes of 4096, the running sums of scale 5 carried across them."""
    pats, w, ch, bl = _case(5, 60, 15, 1)
    _check_against_oracle(pats, w, ch, bl, 8300, seed=9, fit=False)


def test_kernel_matches_oracle_with_scaling():
    """1000 taxa, 24 distinct sites: rescaled vectors, and 24 patterns, one and a half blocks of 16."""
    R, L = 1000, 24
    rng = np.random.default_rng(77)
    tips = (1 << rng.integers(0, 4, size=(R, L))).astype(np.uint8)
    pats, w = O.compress_patterns(tips)
    assert pats.shape[1] % 16
    trees = [O.random_tree(R, rng) for _ in range(3)]
    ch, bl = np.stack([t[0] for t in trees]), np.stack([t[1] for t in trees])
    assert O.root_terms(ch[0], bl[0], pats, O.Model(**GEN))[1].max() > 0          # vectors are rescaled in this case
    _check_against_oracle(pats, w, ch, bl, 200, seed=4, fit=False)


def test_invariants_on_a_known_tree():
    """50 x 1024 sites simulated on a known tree; candidates: that tree, 40 of its NNI neighbours, 22 random trees and the known tree
    once more."""
    R, L, N = 50, 1024, 1000
    rng = np.random.default_rng(2024)
    ch0, bl0 = O.random_tree(R, rng)
    tips = O.simulate(ch0, bl0, R, L, O.Model(**GEN), rng, gap_frac=0.05)
    pats, w = O.compress_patterns(tips)
    cand = [(ch0, bl0)]
    for v in LH.internal_branches(ch0)[:20]:
        cand += [LH.nni_tree(ch0, v, k, bl0) for k in (1, 2)]
    n_rand = 22
    cand += [O.random_tree(R, rng) for _ in range(n_rand)]
    cand.append((ch0, bl0))
    K = len(cand)
    assert K == 64
    ch, bl = np.stack([c for c, _ in cand]), np.stack([b for _, b in cand])
    eng = LH.TreeLikelihood(pats, w)
    sm = LH.SubstModel("GTR+I+G", LH.empirical_freqs(tips), K)
    bl, _, _ = eng.optimize_all(ch, bl, sm)
    a = eng.topology_test(ch, bl, sm, N, 5)
    b = eng.topology_test(ch, bl, sm, N, 5)
    for key in a:
        assert np.array_equal(a[key], b[key]), key
    win, kh, sh, elw, llh = a["win"], a["kh"], a["sh"], a["elw"], a["llh"]
    ks = int(np.argmax(llh))
    assert (sh >= kh).all() and kh[ks] == sh[ks] == N
    assert abs(elw.sum() - 1.0) <= 1e-12
    assert llh[0] == llh[K - 1] and (win[:, 0] == win[:, K - 1]).all() and kh[0] == kh[K - 1] and sh[0] == sh[K - 1]
    # a permutation of the trees permutes the counts
    perm = np.random.default_rng(3).permutation(K)
    sp = LH.SubstModel("GTR+I+G", LH.empirical_freqs(tips), K)
    sp.rates, sp.freqs, sp.alpha, sp.pinv = sm.rates[perm], sm.freqs[perm], sm.alpha[perm], sm.pinv[perm]
    p = eng.topology_test(ch[perm], bl[perm], sp, N, 5)
    assert np.array_equal(p["llh"], llh[perm]) and np.array_equal(p["win"], win[:, perm])
    assert np.array_equal(p["kh"], kh[perm]) and np.array_equal(p["sh"], sh[perm])
    np.testing.assert_allclose(p["elw"], elw[perm], rtol=0, atol=1e-12)
    # the data reject the random trees
    n = int(w.sum())
    n_s = SUP.scale_draws(n)
    rand = range(K - 1 - n_rand, K - 1)
    for k in rand:
        assert sh[k] / N < 0.05 and SUP.au_pvalue(win[:, k], n_s, n, N) < 0.05, k


def test_search_inference_writes_candidates_and_table(tmp_path, gpu_models):
    from neuralnj_b200 import Search_inference, inference_config
    src = tmp_path / "msas"
    src.mkdir()
    shutil.copyfile(os.path.join(GOLD, "msa", "t20x256_120.phy"), src / "t20x256_120.phy")
    cfgs = inference_config()
    cfgs.env.batch_size = 8
    cfgs.num_episodes = 2
    kw = dict(cfgs=cfgs, device=torch.device("cuda:0"), policy_network=gpu_models["bf16x3"], stop_step=2)
    torch.manual_seed(123)
    Search_inference(str(src), str(tmp_path / "plain"), None, **kw)
    torch.manual_seed(123)
    Search_inference(str(src), str(tmp_path / "tt"), None, topotest=200, topotest_top=6, topotest_seed=1, **kw)
    tre = (tmp_path / "plain" / "t20x256_120.tre").read_bytes()
    assert (tmp_path / "tt" / "t20x256_120.tre").read_bytes() == tre
    assert not (tmp_path / "plain" / "t20x256_120.trees").exists()
    trees = (tmp_path / "tt" / "t20x256_120.trees").read_text().splitlines()
    assert 2 <= len(trees) <= 6 and trees[0] == tre.decode()
    lines = (tmp_path / "tt" / "t20x256_120.topotest.txt").read_text().splitlines()
    assert lines[0].split()[:3] == ["Tree", "logL", "deltaL"] and len(lines) == 2 + len(trees)
    rows = [ln.split() for ln in lines[2:]]
    assert [int(r[0]) for r in rows] == list(range(1, len(trees) + 1))
    res = SUP.topology_test(str(src / "t20x256_120.phy"), trees, n_boot=200, seed=1)
    for r, k in zip(rows, range(len(trees))):
        assert float(r[1]) == pytest.approx(res["llh"][k], abs=1e-4) and float(r[7]) == pytest.approx(res["p_sh"][k], abs=1e-4)
    assert res["delta"].min() == 0.0 and (res["p_au"] >= 0).all() and (res["p_au"] <= 1).all() and res["win"].shape == (len(trees), 10)
    assert all(t.endswith(";") for t in res["tree"]) and res["n_boot"] == 200 and res["seed"] == 1


def test_input_errors():
    from neuralnj_b200._lib import NnjError
    pats, w, ch, bl = _case(20, 100, 3, 2)
    eng = LH.TreeLikelihood(pats, w)
    with pytest.raises(NnjError, match="non-negative integers"):
        LH.TreeLikelihood(pats, w + 0.5).topology_test(ch, bl, _sm(3), 10, 0)
    with pytest.raises(ValueError, match="at least two"):
        eng.topology_test(ch[:1], bl[:1], _sm(1), 10, 0)
    R = 4097
    rng = np.random.default_rng(0)
    big_ch, big_bl = O.random_tree(R, rng)
    big = (1 << rng.integers(0, 4, size=(R, 4))).astype(np.uint8)
    with pytest.raises(ValueError, match="4096"):
        LH.TreeLikelihood(big, np.ones(4)).topology_test(np.stack([big_ch] * 2), np.stack([big_bl] * 2), _sm(2), 10, 0)
    path = os.path.join(GOLD, "msa", "t20x256_120.phy")
    from neuralnj_b200 import load_pi_instance
    keys = [str(k) for k in load_pi_instance(path)["seq_keys"][0]]
    newick = LH.tuples_to_newick(LH.tuples_with_lengths(ch[0], bl[0], keys, unrooted=True))
    with pytest.raises(ValueError, match="at least two"):
        SUP.topology_test(path, [newick], n_boot=10)
    with pytest.raises(ValueError, match="not among the alignment labels"):
        SUP.topology_test(path, [newick, newick.replace(keys[3] + ":", "stranger:")], n_boot=10)
