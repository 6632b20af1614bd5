"""GPU tests of likelihood branch support (csrc/nnj_llh_nni.cu, DESIGN.md 12) against the numpy oracle oracle/alrt_oracle.py.

Log-likelihoods and sites within 1e-9 relative, NNI lengths rtol 1e-5 / atol 1e-8 (the tolerances of tests/test_gpu_llh.py) wherever
the likelihood depends on the length (`_assert_lengths`: behind a saturated branch it may not, to the last bit).  The RELL statistics are bit-identical when the oracle runs on the kernel's own site log-likelihoods; against the oracle's sites a
replicate may differ only where its oracle margin is below 1e-7 |L0|."""
import os
import shutil
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import alrt_oracle as A  # noqa: E402
import llh_oracle as O  # noqa: E402

from neuralnj_b200 import likelihood as LH  # noqa: E402

pytestmark = pytest.mark.gpu
GOLD = os.path.join(ROOT, "tests", "golden")
GEN = dict(rates6=(1.2, 3.1, 0.8, 1.1, 4.2, 1.0), freqs=(0.3, 0.2, 0.2, 0.3), alpha=0.7, pinv=0.15)


def caterpillar(R):
    return np.asarray([(0, 1)] + [(R + k, k + 2) for k in range(R - 2)], dtype=np.int32)


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


def _case(R, L, kind, shape, seed=0):
    rng = np.random.default_rng(7919 * R + seed)
    ch, bl = O.random_tree(R, rng)
    if shape == "caterpillar":
        ch = caterpillar(R)
    elif shape == "balanced":
        ch = balanced(R)
    if kind == "iid":
        tips = (1 << rng.integers(0, 4, size=(R, L))).astype(np.uint8)
    else:
        tips = O.simulate(ch, bl, R, L, O.Model(**GEN), rng, gap_frac=0.05)
    pats, w = O.compress_patterns(tips)
    return ch, bl, pats, w


def _sm(B=1):
    sm = LH.SubstModel("GTR+I+G", np.asarray(GEN["freqs"]), B)
    sm.rates[:] = GEN["rates6"]
    sm.alpha[:] = GEN["alpha"]
    sm.pinv[:] = GEN["pinv"]
    return sm


def _om(sm):
    return O.Model(sm.rates[0], sm.freqs[0], sm.alpha[0], sm.pinv[0])


def _assert_lengths(got, ref, ch, bl, pats, w, om, nodes, ref_llh):
    """NNI lengths [nb, 2, 5] within rtol 1e-5 / atol 1e-8.  A length may differ by more only where the likelihood does not depend on
    it: behind a saturated branch (P(100) is the stationary distribution) a length can be flat to the last bit, and Newton then stops
    wherever rounding in its sums leaves it.  Such a length, moved alone to the kernel's value, must leave the oracle's log L within
    1e-9 relative, and the kernel's five lengths together must reach the oracle's optimum."""
    bad = ~np.isclose(got, ref, rtol=1e-5, atol=1e-8)
    for i, j, e in np.argwhere(bad):
        v, L = nodes[i], ref_llh[i, j + 1]

        def f(lens):
            return float((w * A.quartet_sites(ch, bl, pats, om, v, j + 1, lens)).sum())
        moved = ref[i, j].copy()
        moved[e] = got[i, j, e]
        assert abs(f(moved) - L) <= 1e-9 * abs(L), (v, j + 1, e, got[i, j], ref[i, j])
        assert abs(f(got[i, j]) - L) <= 1e-9 * abs(L), (v, j + 1, got[i, j], ref[i, j])
    return int(bad.sum())


def _near_ties(site, w, counts, L0):
    """Replicates of each branch whose SH or LBP decision lies within 1e-7 |L0| of its threshold (oracle arithmetic)."""
    c = counts.astype(np.float64)
    out = np.zeros(site.shape[0], dtype=np.int64)
    tol = 1e-7 * abs(L0)
    for i in range(site.shape[0]):
        Lw = A._seqsum(w[None] * site[i])
        Ls = A._seqsum(c[:, None, :] * site[i][None])
        delta = Lw[0] - max(Lw[1], Lw[2])
        cs = np.sort(Ls - Lw[None], axis=1)
        m_sh = np.abs(delta - (cs[:, 2] - cs[:, 1]) - A.SH_TOL)
        m_lbp = np.abs(Ls[:, 0] - np.maximum(Ls[:, 1], Ls[:, 2]))
        out[i] = int(((m_sh < tol) | (m_lbp < tol)).sum())
    return out


CASES = [(4, 300, "sim", "random"), (5, 300, "iid", "random"), (8, 400, "sim", "caterpillar"), (8, 400, "sim", "balanced"),
         (50, 1024, "sim", "random"), (50, 1024, "iid", "caterpillar"), (130, 256, "sim", "balanced")]


@pytest.mark.parametrize("R,L,kind,shape", CASES)
def test_kernel_matches_oracle(R, L, kind, shape):
    ch, bl, pats, w = _case(R, L, kind, shape)
    sm = _sm()
    N, seed = 200, 11
    got = LH.TreeLikelihood(pats, w).nni_support(ch[None], bl[None], sm, N, seed, site_llh=True)
    ref = A.branch_support(ch, bl, pats, w, _om(sm), N, seed)
    assert np.array_equal(got["branch_node"][0], ref["branch_node"])
    np.testing.assert_allclose(got["llh"][0], ref["llh"], rtol=1e-9, atol=0)
    _assert_lengths(got["nni_brlen"][0], ref["nni_brlen"], ch, bl, pats, w, _om(sm), ref["branch_node"], ref["llh"])
    site = got["site_llh"][0].cpu().numpy()
    assert np.abs(site - ref["site"]).max() <= 1e-9 * np.abs(ref["site"]).max()
    d_got = got["llh"][0][:, 0] - got["llh"][0][:, 1:].max(1)
    d_ref = ref["llh"][:, 0] - ref["llh"][:, 1:].max(1)
    assert int((d_got < 0).sum()) == int((d_ref < 0).sum())
    # RELL: the oracle on the kernel's own sites is bit-identical; on its own sites only near-ties may differ
    counts = A.rell_counts(w, seed, np.arange(N, dtype=np.uint64))
    sh, lbp = A.rell_stats(site, w, counts)
    assert np.array_equal(got["sh_count"][0], sh) and np.array_equal(got["lbp_count"][0], lbp)
    ties = _near_ties(ref["site"], w, counts, ref["llh"][0, 0])
    assert (np.abs(got["sh_count"][0] - ref["sh_count"]) <= ties).all()
    assert (np.abs(got["lbp_count"][0] - ref["lbp_count"]) <= ties).all()


@pytest.mark.parametrize("R,L,shape", [(300, 48, "random"), (1000, 24, "caterpillar")])
def test_kernel_matches_oracle_with_scaling(R, L, shape):
    ch, bl, pats, w = _case(R, L, "iid", shape)
    sm = _sm()
    om = _om(sm)
    assert O.root_terms(ch, bl, pats, om)[1].max() > 0                   # vectors are rescaled in this case
    N, seed = 100, 5
    got = LH.TreeLikelihood(pats, w).nni_support(ch[None], bl[None], sm, N, seed, site_llh=True)
    nodes = A.internal_branches(ch)
    assert np.array_equal(got["branch_node"][0], nodes)
    site = got["site_llh"][0].cpu().numpy()
    for i in list(range(0, len(nodes), len(nodes) // 4)) + [len(nodes) - 1]:
        for k in (1, 2):
            Lk, lens, sk = A.nni_optimize(ch, bl, pats, w, om, nodes[i], k)
            assert got["llh"][0, i, k] == pytest.approx(Lk, rel=1e-9, abs=0)
            ref_llh = np.zeros((1, 3))
            ref_llh[0, k] = Lk
            sel = np.zeros((1, 2, 5))
            sel[0, k - 1] = lens
            g = sel.copy()
            g[0, k - 1] = got["nni_brlen"][0, i, k - 1]
            _assert_lengths(g, sel, ch, bl, pats, w, om, [nodes[i]], ref_llh)
            assert np.abs(site[i, k] - sk).max() <= 1e-9 * np.abs(sk).max()
    L0 = O.loglik(ch, bl, pats, w, om)
    np.testing.assert_allclose(got["llh"][0, :, 0], L0, rtol=1e-9, atol=0)
    sh, lbp = A.rell_stats(site, w, A.rell_counts(w, seed, np.arange(N, dtype=np.uint64)))
    assert np.array_equal(got["sh_count"][0], sh) and np.array_equal(got["lbp_count"][0], lbp)


def test_reproducible_batched_chunked_and_padding_neutral():
    B, R = 3, 20
    cases = [_case(R, 300, "sim", "random", seed=s) for s in range(B)]
    L = max(c[2].shape[1] for c in cases)
    tips = np.full((B, R, L), 15, dtype=np.uint8)
    w = np.zeros((B, L))
    for b, (_, _, p, wb) in enumerate(cases):
        tips[b, :, :p.shape[1]] = p
        w[b, :p.shape[1]] = wb
    ch = np.stack([c[0] for c in cases])
    bl = np.stack([c[1] for c in cases])
    sm = _sm(B)
    eng = LH.TreeLikelihood(tips, w)
    a = eng.nni_support(ch, bl, sm, 1000, 3)
    b_ = eng.nni_support(ch, bl, sm, 1000, 3)
    for k in a:
        assert np.array_equal(a[k], b_[k]), k
    # chunks of replicates add up
    p1 = eng.nni_support(ch, bl, sm, 400, 3, rep0=0)
    p2 = eng.nni_support(ch, bl, sm, 600, 3, rep0=400)
    assert np.array_equal(a["sh_count"], p1["sh_count"] + p2["sh_count"]) and np.array_equal(a["lbp_count"], p1["lbp_count"] + p2["lbp_count"])
    assert np.array_equal(a["llh"], p1["llh"]) and np.array_equal(a["nni_brlen"], p2["nni_brlen"])
    # every tree alone, on its own unpadded patterns: the same results, bit for bit
    for b, (c, l, p, wb) in enumerate(cases):
        one = LH.TreeLikelihood(p, wb).nni_support(c[None], l[None], _sm(), 1000, 3)
        for k in one:
            assert np.array_equal(one[k][0], a[k][b]), (b, k)


def test_edges_taxon_range_and_multifurcation():
    from neuralnj_b200._lib import NnjError
    ch, bl, pats, w = _case(3, 50, "sim", "random")
    r = LH.TreeLikelihood(pats, w).nni_support(ch[None], bl[None], _sm(), 100, 0)
    assert r["llh"].shape == (1, 0, 3) and r["sh_count"].shape == (1, 0)
    R = 4097
    rng = np.random.default_rng(0)
    ch, bl = O.random_tree(R, rng)
    tips = (1 << rng.integers(0, 4, size=(R, 4))).astype(np.uint8)
    with pytest.raises(NnjError):
        LH.TreeLikelihood(tips, np.ones(4)).nni_support(ch[None], bl[None], _sm(), 10, 0)
    ch6, bl6, pats6, w6 = _case(6, 50, "sim", "random")
    with pytest.raises(NnjError, match="non-negative integers"):
        LH.TreeLikelihood(pats6, w6 + 0.5).nni_support(ch6[None], bl6[None], _sm(), 10, 0)
    # a multifurcating Newick: its zero-length resolving branches score as 1e-6, every value stays finite
    labels = [f"t{i}" for i in range(8)]
    tree = "((t0:0.1,t1:0.2,t2:0.1,t3:0.3):0.1,(t4:0.1,t5:0.1,t6:0.2):0.2,t7:0.1);"
    chm, blm = LH.tree_arrays_from_tuples(LH.treestr_to_tuples(tree), labels)
    _, _, pats, w = _case(8, 200, "sim", "random")
    r = LH.TreeLikelihood(pats, w).nni_support(chm[None], blm[None], _sm(), 100, 0)
    assert np.isfinite(r["llh"]).all() and np.isfinite(r["nni_brlen"]).all()
    assert ((r["sh_count"] >= 0) & (r["sh_count"] <= 100)).all()


def test_likelihood_support_and_argmax_files(tmp_path, gpu_models):
    from neuralnj_b200 import Argmax_inference, inference_config, likelihood_support
    from neuralnj_b200 import support as SUP
    src = tmp_path / "msas"
    src.mkdir()
    names = ["ex50x1024_73", "ex50x1024_71"]
    for n in names:
        shutil.copyfile(os.path.join(GOLD, "msa", n + ".phy"), src / (n + ".phy"))
    model = gpu_models["bf16x3"]
    kw = dict(cfgs=inference_config(), device=torch.device("cuda:0"), files_per_call=1, policy_network=model)
    Argmax_inference(str(src), str(tmp_path / "plain"), None, **kw)
    Argmax_inference(str(src), str(tmp_path / "alrt"), None, alrt=100, alrt_seed=2, **kw)
    for n in names:
        tre = (tmp_path / "plain" / (n + ".tre")).read_text()
        assert (tmp_path / "alrt" / (n + ".tre")).read_text() == tre
        res = likelihood_support(str(src / (n + ".phy")), model, tree=tre, n_rell=100, seed=2)
        assert len(res["splits"]) == 47 and res["n_rell"] == 100
        for kind in ("alrt", "abayes"):
            labelled = (tmp_path / "alrt" / f"{n}.{kind}.tre").read_text()
            assert labelled == res["newick_" + kind]
            assert SUP.strip_support_labels(labelled) == res["tree"]
        assert ((res["sh_alrt"] >= 0) & (res["sh_alrt"] <= 100)).all() and ((res["lbp"] >= 0) & (res["lbp"] <= 100)).all()
        assert ((res["abayes"] >= 0) & (res["abayes"] <= 1)).all() and np.isfinite(res["alrt"]).all()
        assert (res["sh_alrt"][res["alrt"] < 0] == 0).all() and res["n_better_nni"] == int((res["alrt"] < 0).sum())
        assert res["llh_nni"].shape == (47, 2) and np.isfinite(res["llh"])
    # tree=None builds the same Argmax tree
    res0 = likelihood_support(str(src / "ex50x1024_73.phy"), model, n_rell=100, seed=2)
    res1 = likelihood_support(str(src / "ex50x1024_73.phy"), model, tree=(tmp_path / "plain" / "ex50x1024_73.tre").read_text(), n_rell=100, seed=2)
    assert res0["newick_alrt"] == res1["newick_alrt"]
