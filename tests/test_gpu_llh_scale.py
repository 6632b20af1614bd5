"""GPU tests of the tree likelihood (csrc/nnj_llh.cu) from 200 to 4096 taxa and at its numerical edges, against the scaled CPU
oracle (oracle/llh_oracle.py, itself pinned to the underflow-free log-space pruning in tests/test_llh_oracle.py).

Site likelihoods of a few hundred taxa underflow fp64; both sides rescale a CLV by 2^256 when all its entries fall below
2^-256.  Most cases here are chosen so that the unscaled formula gives 0 or a subnormal site, and the file counts them.
Tolerances are those of tests/test_gpu_llh.py: log L 1e-9 relative, optimised log L 1e-8, lengths rtol 1e-5 / atol 1e-8."""
import ctypes as C
import functools
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import llh_oracle as O  # noqa: E402

from neuralnj_b200 import _lib, likelihood as LH  # noqa: E402

pytestmark = pytest.mark.gpu
GOLD = os.path.join(ROOT, "tests", "golden")
GEN = dict(rates6=(1.2, 3.1, 0.8, 1.1, 4.2, 1.0), freqs=(0.3, 0.2, 0.2, 0.3), alpha=0.7, pinv=0.15)
RATES, FREQS = (0.7, 2.0, 1.3, 0.9, 3.0, 1.0), (0.22, 0.28, 0.31, 0.19)


@functools.lru_cache(maxsize=None)
def _data(R, L, kind, seed=0):
    """-> children, generating lengths, lengths to score, masks.  kind: "sim" (simulated, scored at the generating lengths),
    "short" (the same data at 0.1x lengths), "iid" (independent uniform columns at the generating lengths)."""
    rng = np.random.default_rng(1000 * R + seed)
    ch, bl = O.random_tree(R, rng)
    if kind == "iid":
        tips = (1 << rng.integers(0, 4, size=(R, L))).astype(np.uint8)
    else:
        tips = O.simulate(ch, bl, R, L, O.Model(**GEN), rng, gap_frac=0.05)
    return ch, bl, bl * (0.1 if kind == "short" else 1.0), tips


def _sm(B, rates, freqs, alpha, pinv, spec="GTR+I+G"):
    sm = LH.SubstModel(spec, np.asarray(freqs, dtype=np.float64), B)
    if sm.gtr:
        sm.rates[:] = rates
    sm.alpha[:] = alpha
    sm.pinv[:] = pinv
    return sm


def _om(sm, b=0):
    """The oracle model of row b of a SubstModel."""
    return O.Model(sm.rates[b], sm.freqs[b], sm.alpha[b], sm.pinv[b], gamma=sm.gamma)


def _underflows(ch, bl, tips, m):
    with np.errstate(all="ignore"):
        s = O.site_likelihoods(ch, bl, tips, m, scaling=False)
    return int((s < np.finfo(np.float64).tiny).sum())


def _close(got, ref, rel):
    return np.isfinite(got) and abs(got - ref) < rel * abs(ref)


def _check_opt(ch, start, pat, w, sm, eng=None, **kw):
    """GPU branch optimisation of one tree vs the oracle; the returned lengths reproduce the reported maximum."""
    eng = eng or LH.TreeLikelihood(pat, w)
    t_ref, b_ref, a_ref = O.optimize_branches(ch, start, pat, w, _om(sm), **kw)
    t, before, after = eng.optimize_branches(ch[None], start[None], sm, **kw)
    assert _close(before[0], b_ref, 1e-9) and _close(after[0], a_ref, 1e-8), (before[0], b_ref, after[0], a_ref)
    assert after[0] > before[0] and np.isfinite(t).all()
    assert np.allclose(t[0], t_ref, rtol=1e-5, atol=1e-8)
    assert _close(eng.loglik(ch[None], t, sm)[0], after[0], 1e-8)
    return t[0], after[0]


# ---------------------------------------------------------------- evaluation at scale
EVAL_R = [(200, 300), (300, 300), (400, 300), (512, 256), (1000, 160), (2920, 64), (4096, 64)]
KINDS = ["sim", "short", "iid"]
MODELS = [(0.5, 0.0), (1.7, 0.3)]                 # (alpha, p_inv) of tree 0 and tree 1


def _eval_case(R, L, kind):
    ch, _, bl, tips = _data(R, L, kind)
    pat, w = O.compress_patterns(tips)
    ch2, _ = O.random_tree(R, np.random.default_rng(R + 1))                 # a second topology, as Search scores
    chs, bls = np.stack([ch, ch2]), np.stack([bl, bl])
    sm = LH.SubstModel("GTR+I+G", np.asarray(FREQS), 2)
    sm.rates[:] = RATES
    sm.alpha[:] = [a for a, _ in MODELS]
    sm.pinv[:] = [p for _, p in MODELS]
    return chs, bls, pat, w, sm


def test_evaluation_cases_exercise_scaling():
    """The evaluation cases below keep testing scaling: every (case, tree) pair rescales some pattern, and 26 of the 42 have a
    site that the unscaled formula makes 0 or subnormal - all from 1000 taxa on, 5 of 6 at 512, 3 at 300-400, none at 200."""
    hit = set()
    for R, L in EVAL_R:
        for kind in KINDS:
            chs, bls, pat, w, sm = _eval_case(R, L, kind)
            for b in range(2):
                assert O.root_terms(chs[b], bls[b], pat, _om(sm, b))[1].max() >= 1, (R, kind, b)
                if _underflows(chs[b], bls[b], pat, _om(sm, b)):
                    hit.add((R, kind, b))
    assert len(hit) == 26, sorted(hit)
    assert {(R, kind, b) for R in (1000, 2920, 4096) for kind in KINDS for b in (0, 1)} <= hit


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("R,L", EVAL_R)
def test_evaluation_at_scale_matches_oracle(R, L, kind):
    chs, bls, pat, w, sm = _eval_case(R, L, kind)
    got = LH.TreeLikelihood(pat, w).loglik(chs, bls, sm)
    for b in range(2):
        ref = O.loglik(chs[b], bls[b], pat, w, _om(sm, b))
        assert _close(got[b], ref, 1e-9), (b, got[b], ref)


# ---------------------------------------------------------------- optimisation at scale
@pytest.mark.parametrize("start", ["short", "default"])
@pytest.mark.parametrize("R", [300, 400, 512])
def test_branch_optimisation_at_scale(R, start):
    """From 0.1x the generating lengths (scaled patterns at the start) and from BRLEN_DEFAULT everywhere."""
    ch, bl, _, tips = _data(R, 150, "sim")
    pat, w = O.compress_patterns(tips)
    sm = _sm(1, RATES, FREQS, 0.8, 0.1)
    st = bl * 0.1 if start == "short" else np.full(2 * R - 2, LH.BRLEN_DEFAULT)
    assert O.root_terms(ch, st, pat, _om(sm))[1].max() >= 1
    _check_opt(ch, st, pat, w, sm)


def test_optimize_all_at_300_taxa():
    R = 300
    ch, bl, _, tips = _data(R, 100, "sim", seed=1)
    pat, w = O.compress_patterns(tips)
    freqs = LH.empirical_freqs(tips)
    start = np.full(2 * R - 2, LH.BRLEN_DEFAULT)
    om = O.Model(freqs=freqs, alpha=1.0, pinv=0.0)
    t_ref, _, a_ref = O.optimize_all(ch, start, pat, w, om, max_rounds=3)
    sm = LH.SubstModel("GTR+I+G", freqs, 1)
    t, before, after = LH.TreeLikelihood(pat, w).optimize_all(ch[None], start[None], sm, max_rounds=3)
    assert np.isfinite(t).all() and after[0] > before[0] and _close(after[0], a_ref, 1e-5), (after[0], a_ref)
    assert np.allclose(sm.rates[0], om.rates6, rtol=2e-3) and abs(sm.alpha[0] - om.alpha) < 2e-3 * om.alpha and abs(sm.pinv[0] - om.pinv) < 2e-3


# ---------------------------------------------------------------- tree shapes
def _caterpillar(R):
    """(((0,1),2),3)...: the deepest spine, so the largest scale counts; the last join is (clade, leaf)."""
    return np.asarray([(0, 1)] + [(R + k, k + 2) for k in range(R - 2)], dtype=np.int32)


def _balanced(R):
    cur, ch = list(range(R)), []
    while len(cur) > 1:
        nxt = []
        for i in range(0, len(cur) - 1, 2):
            ch.append((cur[i], cur[i + 1]))
            nxt.append(R + len(ch) - 1)
        cur = nxt + ([cur[-1]] if len(cur) % 2 else [])
    return np.asarray(ch, dtype=np.int32)


@pytest.mark.parametrize("shape", ["caterpillar", "balanced"])
def test_tree_shapes_at_400_taxa(shape):
    R, L = 400, 120
    ch = _caterpillar(R) if shape == "caterpillar" else _balanced(R)
    rng = np.random.default_rng(7)
    bl = rng.uniform(0.02, 0.4, size=2 * R - 2)
    tips = O.simulate(ch, bl, R, L, O.Model(**GEN), rng, gap_frac=0.05)
    pat, w = O.compress_patterns(tips)
    sm = _sm(1, RATES, FREQS, 0.8, 0.1)
    assert O.root_terms(ch, bl, pat, _om(sm))[1].max() >= 2
    got = LH.TreeLikelihood(pat, w).loglik(ch[None], bl[None], sm)[0]
    assert _close(got, O.loglik(ch, bl, pat, w, _om(sm)), 1e-9)
    _check_opt(ch, np.full(2 * R - 2, LH.BRLEN_DEFAULT), pat, w, sm)


# ---------------------------------------------------------------- the root branch under optimisation
@pytest.mark.parametrize("children", [
    [(0, 1), (3, 2)],                  # R = 3, root children (inner, leaf)
    [(0, 1), (2, 3)],                  # R = 3, (leaf, inner)
    [(0, 1), (2, 3), (4, 5)],          # R = 4, (inner, inner)
    [(0, 1), (4, 2), (5, 3)],          # R = 4, (inner, leaf)
    [(0, 1), (4, 2), (3, 5)],          # R = 4, (leaf, inner)
])
def test_root_crossing_under_optimisation(children):
    """The optimiser crosses the root branch (SWAPROOT) in every configuration of the root's children.  Two leaf children
    would need R = 2, which the ABI refuses."""
    ch = np.asarray(children, dtype=np.int32)
    R = len(ch) + 1
    rng = np.random.default_rng(R * 10 + int(ch[-1][0]))
    bl = rng.uniform(0.05, 0.4, size=2 * R - 2)
    tips = O.simulate(ch, bl, R, 300, O.Model(**GEN), rng, gap_frac=0.05)
    pat, w = O.compress_patterns(tips)
    sm = _sm(1, RATES, FREQS, 0.8, 0.1)
    _check_opt(ch, np.full(2 * R - 2, LH.BRLEN_DEFAULT), pat, w, sm)


# ---------------------------------------------------------------- branch-length edges
@pytest.mark.parametrize("R", [50, 300])
def test_zero_negative_tiny_and_huge_lengths(R):
    """Lengths 0, negative, 1e-7 and 250 score as the clamped lengths [BRLEN_MIN, BRLEN_MAX] on both sides; so do zero root edges.
    Optimisation from such a start matches the oracle too."""
    ch, bl, _, tips = _data(R, 120, "sim", seed=2)
    pat, w = O.compress_patterns(tips)
    rng = np.random.default_rng(R)
    odd = bl.copy()
    idx = rng.permutation(2 * R - 2)
    odd[idx[:R // 5]] = 0.0
    odd[idx[R // 5:R // 4]] = -0.05
    odd[idx[R // 4:R // 3]] = 1e-7
    odd[idx[R // 3]] = 250.0
    c1, c2 = ch[-1]
    odd[c1] = odd[c2] = 0.0
    clamped = np.clip(odd, LH.BRLEN_MIN, LH.BRLEN_MAX)
    sm = _sm(2, RATES, FREQS, 0.6, 0.2)
    got = LH.TreeLikelihood(pat, w).loglik(np.stack([ch, ch]), np.stack([odd, clamped]), sm)
    ref = O.loglik(ch, odd, pat, w, _om(sm))
    assert _close(got[0], ref, 1e-9) and got[0] == got[1] and ref == O.loglik(ch, clamped, pat, w, _om(sm))
    if R == 50:
        _check_opt(ch, odd, pat, w, _sm(1, RATES, FREQS, 0.6, 0.2))


def test_conflicting_tips_on_zero_length_branches():
    """Two different tips joined by zero-length branches: at length 0 the site likelihood is 0 and rounding noise of P(0) made it
    ~1e-17 or negative; clamped to BRLEN_MIN it is tiny, positive and equal on both sides."""
    ch = np.asarray([(0, 1), (3, 2)], dtype=np.int32)
    tips = np.array([[1, 1, 2, 4], [2, 1, 2, 8], [1, 1, 4, 4]], dtype=np.uint8)
    w = np.ones(4)
    bl = np.array([0.0, 0.0, 0.1, 0.1])
    for spec, sm in (("JC", _sm(1, RATES, np.full(4, 0.25), 1.0, 0.0, "JC")), ("GTR+I+G", _sm(1, RATES, FREQS, 0.7, 0.15))):
        got = LH.TreeLikelihood(tips, w).loglik(ch[None], bl[None], sm)[0]
        ref = O.loglik(ch, bl, tips, w, _om(sm))
        assert _close(got, ref, 1e-9), (spec, got, ref)


def test_multifurcating_newick_through_compute_llh():
    """tree_arrays_from_tuples resolves a multifurcation below the root with 0.0 branches; user trees carry zeros and negative
    NJ lengths.  compute_llh must equal the oracle at the clamped lengths."""
    R, L = 9, 200
    rng = np.random.default_rng(17)
    labels = [f"t{i}" for i in range(R)]
    ch0, bl0 = O.random_tree(R, rng)
    tips = O.simulate(ch0, bl0, R, L, O.Model(**GEN), rng, gap_frac=0.0)
    seqs = ["".join("ACGT"[int(np.log2(m))] for m in row) for row in tips]
    msa = {"labels": labels, "sequences": seqs}
    newick = "((t0:0.1,t1:0.0,t2:-0.02):0.05,(t3:0.2,t4:0.1,t5:0.0,t6:0.3):0.0,(t7:0.15,t8:1e-7):0.1);"
    from neuralnj_b200.treeutil import treestr_to_tuples
    ch, bl = LH.tree_arrays_from_tuples(treestr_to_tuples(newick), labels)
    assert (bl == 0.0).sum() >= 3 and (bl < 0).any()
    for model, om in (("JC", O.Model(gamma=False)), ("GTR+I+G", O.Model(freqs=LH.empirical_freqs(tips), alpha=1.0, pinv=0.0))):
        got = LH.compute_llh(newick, msa, model=model, opt_model=False)
        ref = O.loglik(ch, bl, tips, np.ones(L), om)
        assert _close(got, ref, 1e-9), (model, got, ref)
    _, before, after = LH.optimize_brlen(newick, msa, model="GTR+I+G", opt_model=False)
    assert np.isfinite(before) and after > before


# ---------------------------------------------------------------- model edges with scaling active
R_EDGE = 300


def _edge_models():
    f_floor = LH.empirical_freqs(np.array([[1] * 2000 + [2] * 2000 + [4] * 2000], dtype=np.uint8))     # T at the 1e-4 floor
    return {
        "alpha_lo": _sm(1, RATES, FREQS, LH.ALPHA_LO, 0.1),
        "alpha_hi": _sm(1, RATES, FREQS, LH.ALPHA_HI, 0.1),
        "pinv_0": _sm(1, RATES, FREQS, 0.8, 0.0),
        "pinv_hi": _sm(1, RATES, FREQS, 0.8, LH.PINV_HI),
        "rate_extremes": _sm(1, (LH.RATE_LO, 2.0, LH.RATE_HI, 0.9, 3.0, 1.0), FREQS, 0.8, 0.1),
        "freq_floor": _sm(1, RATES, f_floor, 0.8, 0.1),
        "jc": _sm(1, RATES, np.full(4, 0.25), 1.0, 0.0, "JC"),
    }


@pytest.mark.parametrize("name", ["alpha_lo", "alpha_hi", "pinv_0", "pinv_hi", "rate_extremes", "freq_floor", "jc"])
def test_model_edges_with_scaling(name):
    sm = _edge_models()[name]
    if name == "freq_floor":
        assert abs(sm.freqs[0, 3] - 1e-4) < 1e-6
    ch, bl, _, tips = _data(R_EDGE, 120, "sim", seed=3)
    pat, w = O.compress_patterns(tips)
    st = bl * 0.1
    assert O.root_terms(ch, bl, pat, _om(sm))[1].max() >= 1 or O.root_terms(ch, st, pat, _om(sm))[1].max() >= 1
    eng = LH.TreeLikelihood(pat, w)
    got = eng.loglik(np.stack([ch, ch]), np.stack([bl, st]), _sm(2, sm.rates[0], sm.freqs[0], sm.alpha[0], sm.pinv[0], "GTR+I+G" if sm.gtr else "JC"))
    for b, lens in enumerate((bl, st)):
        assert _close(got[b], O.loglik(ch, lens, pat, w, _om(sm)), 1e-9), (b, got[b])
    _check_opt(ch, st, pat, w, sm, eng=eng)


def test_invariant_sites_meet_a_scaled_gamma_term():
    """+I on 400 taxa: constant columns with 30 % gaps on long branches, so that in the same pattern the invariant term is
    positive and the gamma term is scaled (Newton scales the invariant term up by 2^(256 n))."""
    R, L = 400, 120
    rng = np.random.default_rng(401)
    ch, bl = O.random_tree(R, rng)
    bl = bl * 5.0
    tips = O.simulate(ch, bl, R, L, O.Model(**GEN), rng)
    tips[:, :L // 2] = (1 << rng.integers(0, 4, size=L // 2))[None, :]
    tips[rng.random(tips.shape) < 0.3] = 15
    pat, w = O.compress_patterns(tips)
    sm = _sm(1, RATES, FREQS, LH.ALPHA_HI, 0.5)
    _, n, iv = O.root_terms(ch, bl, pat, _om(sm))
    assert ((n > 0) & (iv > 0)).sum() >= 20
    eng = LH.TreeLikelihood(pat, w)
    assert _close(eng.loglik(ch[None], bl[None], sm)[0], O.loglik(ch, bl, pat, w, _om(sm)), 1e-9)
    _check_opt(ch, bl, pat, w, sm, eng=eng)


# ---------------------------------------------------------------- the model the kernel rebuilds
class _KeepPacked(LH.SubstModel):
    def unpack(self, packed):
        self.packed_out = packed.copy()
        super().unpack(packed)


def _check_rebuilt(sm):
    """model_host[0:44] after nnj_llh_optimize_all (eigen-system and class rates rebuilt on the device) vs SubstModel.pack() of the
    returned parameters: P(t) to 1e-12, class rates to scipy within 1e-9."""
    out = sm.packed_out
    exp = LH.SubstModel.pack(sm)
    for b in range(sm.B):
        for t in (0.01, 0.3, 2.0):
            def P(p):
                return p[4:20].reshape(4, 4) @ np.diag(np.exp(p[:4] * t)) @ p[20:36].reshape(4, 4)
            assert np.abs(P(out[b]) - P(exp[b])).max() < 1e-12
        assert np.allclose(out[b, 36:40], exp[b, 36:40], rtol=0, atol=0)
        cat = O.gamma_rates(float(sm.alpha[b])) if sm.gamma else np.ones(4)
        assert np.allclose(out[b, 40:44], cat, rtol=1e-9, atol=1e-300), (sm.alpha[b], out[b, 40:44], cat)


def test_rebuilt_model_matches_host_pack():
    # alpha driven down: half the columns constant, half iid; alpha driven up: no rate variation in the generating model
    R, L = 16, 3000
    rng = np.random.default_rng(44)
    ch, bl = O.random_tree(R, rng)
    lo = (1 << rng.integers(0, 4, size=(R, L))).astype(np.uint8)
    lo[:, :L // 2] = (1 << rng.integers(0, 4, size=L // 2))[None, :]
    hi = O.simulate(ch, bl, R, L, O.Model(rates6=GEN["rates6"], freqs=GEN["freqs"], gamma=False), rng)
    sim = _data(40, 800, "sim", seed=4)[3]
    ch40 = _data(40, 800, "sim", seed=4)[0]
    alphas = []
    for c, tips in ((ch, lo), (ch, hi), (ch40, sim)):
        pat, w = O.compress_patterns(tips)
        Rn = tips.shape[0]
        sm = _KeepPacked("GTR+G" if tips is not sim else "GTR+I+G", LH.empirical_freqs(tips), 1)
        t, before, after = LH.TreeLikelihood(pat, w).optimize_all(c[None], np.full((1, 2 * Rn - 2), 0.1), sm)
        assert np.isfinite(after[0]) and after[0] > before[0]
        _check_rebuilt(sm)
        alphas.append(float(sm.alpha[0]))
    assert alphas[0] < 0.05 and alphas[1] > 20.0, alphas


# ---------------------------------------------------------------- zero-weight padding
def test_zero_weight_padding_is_bit_neutral():
    """PhyInferEnv._finish_scored pads the alignments of a batch with all-gap, weight-0 patterns to one pattern count: each tree's
    result must be bit-equal to its own unpadded B = 1 call, evaluated and optimised."""
    R = 300
    cases = [_data(R, L, "sim", seed=10 + i) for i, L in enumerate((60, 90, 120))]
    pats = [O.compress_patterns(c[3]) for c in cases]
    Lp = max(p.shape[1] for p, _ in pats)
    P = np.full((3, R, Lp), 15, dtype=np.uint8)
    W = np.zeros((3, Lp))
    for b, (p, w) in enumerate(pats):
        P[b, :, :p.shape[1]], W[b, :len(w)] = p, w
    ch = np.stack([c[0] for c in cases])
    bl = np.stack([c[1] * 0.1 for c in cases])
    sm = _sm(3, RATES, FREQS, 0.8, 0.1)
    sm.alpha[:] = (0.5, 0.8, 1.9)
    ev = LH.TreeLikelihood(P, W).loglik(ch, bl, sm)
    t, before, after = LH.TreeLikelihood(P, W).optimize_branches(ch, bl, sm)
    for b, (p, w) in enumerate(pats):
        one = _sm(1, RATES, FREQS, sm.alpha[b], 0.1)
        eng = LH.TreeLikelihood(p, w)
        assert ev[b] == eng.loglik(ch[b:b + 1], bl[b:b + 1], one)[0]
        t1, b1, a1 = eng.optimize_branches(ch[b:b + 1], bl[b:b + 1], one)
        assert before[b] == b1[0] and after[b] == a1[0] and np.array_equal(t[b], t1[0])


def test_rollout_scores_of_a_two_alignment_batch(golden):
    """reinforce_rollout(branch_optimize=True) on two different alignments in one batch: each score equals that alignment alone."""
    from neuralnj_b200 import PhyInferEnv, PhyloATTN, inference_config, reinforce_rollout
    cfgs = inference_config()
    g = golden("batch2_20x256")
    torch.manual_seed(0)
    model = PhyloATTN(cfgs, precision="fp32").to("cuda:0").eval()
    B, R, L = g.data.shape[:3]
    assert B == 2 and not torch.equal(g.data[0], g.data[1])

    def batch_of(sl):
        return {"data": g.data[sl], "seq_weights": (~g.mask[sl]).float(), "seqs": [["A" * L] * R for _ in range(sl.stop - sl.start)],
                "seq_keys": g.seq_keys[sl]}

    env = PhyInferEnv(cfgs, torch.device("cuda:0"))
    _, _, scores, _ = reinforce_rollout(batch_of(slice(0, 2)), model, env, cfgs, eval=True, argmax=True, branch_optimize=True)
    trees = [env.states[b].subtrees[0].utree_op_str for b in range(2)]
    for b in range(2):
        env1 = PhyInferEnv(cfgs, torch.device("cuda:0"))
        _, _, s1, _ = reinforce_rollout(batch_of(slice(b, b + 1)), model, env1, cfgs, eval=True, argmax=True, branch_optimize=True)
        assert env1.states[0].subtrees[0].utree_op_str == trees[b]
        assert np.isfinite(float(scores[b])) and float(scores[b]) == float(s1[0])


# ---------------------------------------------------------------- determinism, arguments, the Search scorer
def test_optimize_all_is_deterministic_at_400_taxa():
    R = 400
    ch, bl, _, tips = _data(R, 80, "sim", seed=5)
    pat, w = O.compress_patterns(tips)
    runs = []
    for _ in range(2):
        sm = LH.SubstModel("GTR+I+G", LH.empirical_freqs(tips), 2)
        t, before, after = LH.TreeLikelihood(pat, w).optimize_all(np.stack([ch, ch]), np.stack([bl * 0.1, bl]), sm, max_rounds=2)
        runs.append((t, before, after, sm.rates.copy(), sm.alpha.copy(), sm.pinv.copy()))
    assert np.isfinite(runs[0][2]).all()
    for x, y in zip(*runs):
        assert np.array_equal(x, y)


def test_4096_taxa_evaluate_and_one_sweep():
    R = 4096
    ch, bl, _, tips = _data(R, 64, "sim")
    pat, w = O.compress_patterns(tips)
    sm = _sm(1, RATES, FREQS, 0.8, 0.1)
    eng = LH.TreeLikelihood(pat, w)
    ev = eng.loglik(ch[None], bl[None], sm)[0]
    assert _close(ev, O.loglik(ch, bl, pat, w, _om(sm)), 1e-9)
    t, before, after = eng.optimize_branches(ch[None], bl[None], sm, max_passes=1)
    assert np.isfinite(t).all() and np.isfinite(after[0]) and after[0] >= before[0] and before[0] == ev
    assert _close(eng.loglik(ch[None], t, sm)[0], after[0], 1e-8)


def _raw_eval(R, children, L=8):
    """nnj_llh_eval straight through the C ABI (TreeLikelihood refuses R < 3 itself)."""
    tips = torch.ones(1, R, L, dtype=torch.uint8, device="cuda")
    w = torch.ones(1, L, dtype=torch.float64, device="cuda")
    ch = np.ascontiguousarray(children, dtype=np.int32)
    bl = np.full(2 * R - 2, 0.1)
    pk = np.ascontiguousarray(_sm(1, RATES, FREQS, 0.8, 0.1).pack())
    out = np.zeros(1)
    lib = _lib.lib()
    need = max(int(lib.nnj_llh_workspace_bytes(1, max(R, 3), L)), 1)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    vp = C.c_void_p
    rc = lib.nnj_llh_eval(vp(tips.data_ptr()), vp(w.data_ptr()), ch.ctypes.data_as(vp), bl.ctypes.data_as(vp), pk.ctypes.data_as(vp), 1, R, L,
                          out.ctypes.data_as(vp), vp(ws.data_ptr()), need, vp(torch.cuda.current_stream().cuda_stream))
    _lib.check(rc, "nnj_llh_eval")
    return out[0]


def test_taxon_range_and_tree_checks():
    with pytest.raises(_lib.NnjError):
        _raw_eval(2, [(0, 1)])
    with pytest.raises(ValueError):
        LH.TreeLikelihood(np.ones((2, 8), dtype=np.uint8))
    with pytest.raises(_lib.NnjError):
        _raw_eval(4097, _caterpillar(4097))
    with pytest.raises(_lib.NnjError):
        _raw_eval(5, [(0, 1), (0, 2), (5, 3), (6, 4)])           # leaf 0 twice
    with pytest.raises(_lib.NnjError):
        _raw_eval(5, [(0, 1), (6, 2), (5, 3), (7, 4)])           # node 6 used before its join creates it
    assert np.isfinite(_raw_eval(4096, _caterpillar(4096)))     # a clean call after the refusals


def test_score_topologies_at_rollout_size():
    """Search's scorer on a simulated 400-taxon alignment: 7 random topologies and the generating one; the generating one wins."""
    R = 400
    ch0, _, _, tips = _data(R, 200, "sim", seed=6)
    rng = np.random.default_rng(66)
    ch = np.stack([O.random_tree(R, rng)[0] for _ in range(7)] + [ch0])
    ll, brl = LH.score_topologies(tips, ch, [f"t{i}" for i in range(R)])
    assert np.isfinite(ll).all() and np.isfinite(brl).all() and int(np.argmax(ll)) == 7
