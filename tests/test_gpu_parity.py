"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle and the reference's golden records.

Both precision modes are held to the same bar (fp32 CUDA-core path; bf16x3 = split-bf16 on tcgen05 for the dense
contractions that have been moved to tensor cores).  Tolerances: logits are compared as max|delta| / max|logit| of the step <= 2e-5 (the oracle
itself moves by ~4e-7 against the reference and ~1e-6 with thread count, SURVEY.md F6); encoder output
<= 2e-4 absolute on values of order 1; merge lists and Newick strings must be identical.
"""
import math

import pytest
import torch

from conftest import ALL_CASES, SMALL_CASES

pytestmark = pytest.mark.gpu

LOGIT_TOL = 2e-5
# Round-2 breadth set: the split-bf16 error (2^-17 per operand, 2^-16 per product for the dropped lo*lo term) averages down over
# the 1024 sites of a logit only when the sites differ.  data_gen/.../G_l_1024_n_50_0_0_65.phy (branch length 0: fifty identical
# sequences, |logit| ~ 196) makes every site round the same way and measured 2.1e-5; the breadth tests therefore hold bf16x3 to
# 4e-5 (the north star's score tolerance is 1e-2) and every case's measured maximum is written to profiles/r02_parity.json.
LOGIT_TOL_BY_PREC = {"fp32": 2e-5, "bf16x3": 4e-5}
STATE_TOL = 2e-4
# A step whose reference top-1/top-2 gap is below TIE_TOL * max|logit| is tie-ambiguous (SURVEY.md H1): fp32 kernels are held to
# ~8 fp32 ulps; the split-bf16 tensor-core path carries ~16-bit operand mantissas (logit error ~5e-6) and uses the survey's 1e-5.
TIE_TOL = {"fp32": 1e-6, "bf16x3": 1e-5}


def _rel(a, b):
    return float((a - b).abs().max() / b.abs().max())


def _min_rel_gap(logits):
    gaps = []
    for lg in logits:
        if lg.shape[1] >= 2:
            top = lg.topk(2, dim=1).values
            gaps.append(float(((top[:, 0] - top[:, 1]) / lg.abs().max(1).values).min()))
    return min(gaps) if gaps else 1.0


def _assert_equivalent_trajectory(sd, data, mask, merges, trace, tie_tol, logit_tol=LOGIT_TOL, pair_chunk=0):
    """`merges` may leave the oracle's trajectory only at tie-ambiguous steps: replay it on the oracle
    (teacher-forced) and require every chosen action to be an oracle argmax within tie_tol, logits within LOGIT_TOL.
    Returns the largest relative logit error along the replayed trajectory."""
    import nnj_oracle as O
    ref = O.rollout(sd, data, mask, forced_merges=merges, pair_chunk=pair_chunk)
    off, worst = 0, 0.0
    for t, lg in enumerate(ref["logits"]):
        p = lg.shape[1]
        err = _rel(trace[:, off:off + p], lg)
        assert err < logit_tol, t
        worst = max(worst, err)
        chosen = lg.gather(1, ref["actions"][t].unsqueeze(1)).squeeze(1)
        slack = (lg.max(1).values - chosen) / lg.abs().max(1).values
        assert float(slack.max()) < tie_tol, f"step {t}: chosen pair is not an oracle argmax (slack {float(slack.max()):.2e})"
        off += p
    return worst


@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
@pytest.mark.parametrize("case", ["t20x256_10", "padded_20x256", "tiny_5x128", "t50x256_a"])
def test_encoder_matches_oracle(case, prec, golden, sd0, gpu_models):
    import nnj_oracle as O
    g = golden(case)
    want = O.encode(sd0, g.data, g.mask)
    got = gpu_models[prec].encode_zxr(g.data.cuda(), g.mask.cuda()).cpu()
    assert got.shape == want.shape
    assert float((got - want).abs().max()) < STATE_TOL
    # and the strided sample the reference itself produced
    assert float((got[:, ::7, ::37, :] - g.state_sample).abs().max()) < STATE_TOL


@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
def test_encoder_layers_match_oracle(prec, golden, sd0):
    """Layer-by-layer: truncate the model to l layers on both sides (both precision modes)."""
    import nnj_oracle as O
    from neuralnj_b200 import PhyloATTN, inference_config
    g = golden("t20x256_103")
    for nl in (1, 2):
        cfg = inference_config()
        cfg.model.num_enc_layers = nl
        torch.manual_seed(0)
        m = PhyloATTN(cfg, precision=prec).cuda().eval()
        sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
        want = O.encode(sd, g.data, g.mask)
        got = m.encode_zxr(g.data.cuda(), g.mask.cuda()).cpu()
        assert float((got - want).abs().max()) < 5e-5, nl


@pytest.mark.parametrize("case", ["t20x256_104", "padded_20x256", "tiny_3x64", "tiny_4x96"])
def test_pair_scores_full_matches_oracle(case, golden, sd0, gpu_model):
    import nnj_oracle as O
    g = golden(case)
    state = O.encode(sd0, g.data, g.mask)
    B, R, C, _ = state.shape
    ii, jj = torch.triu_indices(R, R, offset=1)
    valid = (~g.mask[:, None, :]).float()
    want = O.pair_scores(sd0, state, valid, ii.expand(B, -1), jj.expand(B, -1), C)
    gpu_model.patch_num = C
    got = gpu_model.decode_zxr(state.cuda(), g.mask.cuda(), (None, None, None))["logits"].cpu()
    assert _rel(got, want) < LOGIT_TOL
    assert _rel(got, g.logits[0]) < LOGIT_TOL     # the reference's own step-0 logits


def test_incremental_scores_and_merge_match_oracle(golden, sd0, gpu_model):
    """Step t>=1 through the drop-in API: aggregate/merge, cached-score map (both forms), along the golden trajectory."""
    import nnj_oracle as O
    g = golden("batch2_20x256")
    X = O.encode(sd0, g.data, g.mask)
    B, R, C, _ = X.shape
    Xg = X.cuda()
    mask = g.mask.cuda()
    gpu_model.patch_num = C
    logits_prev = gpu_model.decode_zxr(Xg, mask, (None, None, None))["logits"]
    ar = torch.arange(B)
    for t in range(6):
        ij = g.merges[:, t]
        n = X.shape[1]
        # oracle merge
        new = O.aggregate(sd0, X, X[ar, ij[:, 0]].unsqueeze(1), X[ar, ij[:, 1]].unsqueeze(1), ij[:, :1], ij[:, 1:], C)
        got_new = gpu_model.aggregate(None, None, (ij[:, 0].cuda(), ij[:, 1].cuda()), batchwise_ij_indices=True).cpu()
        assert float((got_new - new).abs().max()) < 5e-5
        rows = []
        for b in range(B):
            i, j = ij[b].tolist()
            xb = X[b].clone(); xb[i] = new[b, 0]
            rows.append(torch.cat([xb[:j], xb[j + 1:]]))
        X = torch.stack(rows)
        Xg = gpu_model.merge_state(Xg, ij.cuda())
        assert float((Xg.cpu() - X).abs().max()) < 5e-5
        # incremental scores: closed-form device map and the caller-supplied gather map must agree with the reference
        idx = torch.tensor([O.score_indices_to_prev(int(a), int(b), n - 1) for a, b in ij.tolist()])
        out_closed = gpu_model.decode_zxr(Xg, mask, (ij.int().cuda(), None, logits_prev))["logits"]
        out_gather = gpu_model.decode_zxr(Xg, mask, (ij.int().cuda(), idx.cuda(), logits_prev))["logits"]
        assert torch.equal(out_closed, out_gather)
        assert _rel(out_closed.cpu(), g.logits[t + 1]) < LOGIT_TOL
        logits_prev = out_closed


# Records that must pass by STRICT identity in both precisions (never through the tie-aware branch): the two shipped example
# alignments (config 1 runs ex50x1024_73; SURVEY puts ex50x1024_71's smallest gap at 8.0e-6, inside the bf16x3 tie tolerance).
STRICT_BY_NAME = {"ex50x1024_73", "ex50x1024_71"}


def _max_trace_err(trace, logits):
    off, worst = 0, 0.0
    for lg in logits:
        p = lg.shape[1]
        worst = max(worst, _rel(trace[:, off:off + p], lg))
        off += p
    return worst


@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
@pytest.mark.parametrize("case", ALL_CASES)
def test_rollout_matches_reference_golden(case, prec, golden, sd0, gpu_models, parity_report):
    """Fused device rollout vs the executed reference: identical merges / Newick (RF = 0), logits and log-probs close.
    Only a record whose own top-1/top-2 gap falls below TIE_TOL[prec] somewhere (t100x256_a: 9.9e-8 at step 67, under one
    fp32 ulp; for bf16x3 also t50x512_a: 1.3e-6 at step 44) is allowed the tie-aware comparison instead; which branch a
    record took is written to profiles/r02_parity.json, and the records in STRICT_BY_NAME may never take it."""
    from neuralnj_b200 import PhyInferEnv, inference_config, rf_distance
    g = golden(case)
    merges, slp, trace = gpu_models[prec].rollout_fused(g.data.cuda(), g.mask.cuda(), want_logits=True)
    merges, slp, trace = merges.cpu().long(), slp.cpu(), trace.cpu()
    gap = _min_rel_gap(g.logits)
    entry = {"precision": prec, "source": "reference golden (tests/golden)", "shape": list(g.data.shape[:3]), "min_rel_top2_gap": gap,
             "mode": "strict", "max_logit_rel_err": None}
    parity_report[f"{case}/{prec}"] = entry
    if not torch.equal(merges, g.merges) and gap < TIE_TOL[prec] and case not in STRICT_BY_NAME:
        entry["mode"] = "tie_aware"
        _assert_equivalent_trajectory(sd0, g.data, g.mask, merges, trace, TIE_TOL[prec])
        return
    assert torch.equal(merges, g.merges), f"first differing step: {int((merges != g.merges).any(-1).any(0).nonzero()[0])}"
    entry["max_logit_rel_err"] = _max_trace_err(trace, g.logits)
    assert entry["max_logit_rel_err"] < LOGIT_TOL
    R = g.data.shape[1]
    if R > 2:
        assert float((slp[:, :R - 2] - g.selected_log_ps).abs().max()) < 1e-3
    env = PhyInferEnv(inference_config(), torch.device("cpu"))
    env.init_states([["A"] * R] * g.data.shape[0], g.seq_keys, g.data)
    env.replay_merges(merges)
    for b, st in enumerate(env.states):
        assert st.subtrees[0].utree_op_str == g.newick[b]
        assert rf_distance(st.subtrees[0].utree_op_str, g.newick[b]) == 0


@pytest.mark.parametrize("case", ["t20x256_117", "padded_20x256", "tiny_4x96"])
def test_stepwise_dropin_equals_fused(case, golden, gpu_model):
    """The reference's own loop over encode_zxr / decode_zxr / env.step gives the fused rollout's result."""
    from neuralnj_b200 import PhyInferEnv, inference_config, reinforce_rollout
    g = golden(case)
    cfgs = inference_config()
    B, R = g.data.shape[:2]
    batch = {"data": g.data, "seq_weights": (~g.mask).float(), "seqs": [["A"] * R] * B, "seq_keys": g.seq_keys}
    outs = []
    for fused in (True, False):
        env = PhyInferEnv(cfgs, torch.device("cuda:0"))
        sel, log_ps, scores, best = reinforce_rollout(batch, gpu_model, env, cfgs, eval=True, argmax=True, fused=fused)
        outs.append((sel.cpu(), [l.cpu() for l in log_ps], best, [s.subtrees[0].utree_op_str for s in env.states]))
    assert outs[0][3] == outs[1][3] == g.newick
    assert outs[0][2] == outs[1][2]
    assert float((outs[0][0] - outs[1][0]).abs().max()) < 1e-4
    assert float((outs[0][0] - g.selected_log_ps).abs().max()) < 1e-3
    assert len(outs[0][1]) == len(outs[1][1]) == max(R - 2, 0)


@pytest.mark.parametrize("case,S,prec", [("t20x256_120", 3, "fp32"), ("ex50x1024_73", 2, "bf16x3")])
def test_gumbel_rollout_replays_on_oracle(case, S, prec, golden, sd0, gpu_models):
    """Sampling mode: with the same Gumbel noise the oracle picks the same trajectory (config 3 parity; the second case is
    config 3's own shape - the 50 x 1024 example alignment - on the tensor-core path.  Gumbel noise of order 1 on logits whose
    top gaps are ~1e-5: the perturbed argmax is far from any tie, so the trajectories must be identical)."""
    import nnj_oracle as O
    gpu_model = gpu_models[prec]
    g = golden(case)
    R = g.data.shape[1]
    gen = torch.Generator().manual_seed(5)
    data, mask = g.data.expand(S, -1, -1, -1).contiguous(), g.mask.expand(S, -1).contiguous()
    u = torch.rand(S, R - 1, R * (R - 1) // 2, generator=gen).clamp_(1e-20, 1 - 1e-7)
    gum = -torch.log(-torch.log(u))
    state = gpu_model.encode_zxr(data[:1].cuda(), mask[:1].cuda()).expand(S, -1, -1, -1).contiguous()
    merges, slp, _ = gpu_model.rollout_fused(batch_seq_mask=mask.cuda(), gumbel=gum.cuda(), state=state)
    ref = O.rollout(sd0, data, mask, gumbel=gum)
    assert torch.equal(merges.cpu().long(), ref["merges"])
    assert len({tuple(m.flatten().tolist()) for m in merges.cpu()}) > 1   # the samples differ from each other
    assert float((slp[:, :R - 2].cpu() - ref["selected_log_ps"]).abs().max()) < 1e-3


def test_full_size_properties(gpu_model):
    """Config-2 shape (50 x 1024): determinism, batch independence, valid merge lists, host-buffer entry point."""
    import nnj_oracle as O
    data = O.evolved_msa(6, 50, 1024, seed=21)
    mask = torch.zeros(6, 1024, dtype=torch.bool)
    m1, s1, _ = gpu_model.rollout_fused(data.cuda(), mask.cuda())
    m2, s2, _ = gpu_model.rollout_fused(data.cuda(), mask.cuda())
    assert torch.equal(m1, m2) and torch.equal(s1, s2)                      # bit-exact rerun
    m3, s3, _ = gpu_model.rollout_fused(data[2:4].cuda(), mask[2:4].cuda())
    assert torch.equal(m3, m1[2:4]) and torch.equal(s3, s1[2:4])            # trees in a batch are independent
    mh = gpu_model.rollout_host(data, mask)
    assert torch.equal(mh, m1.cpu())                                        # C-ABI host entry point
    m = m1.cpu()
    for t in range(49):
        n = 50 - t
        assert bool(((0 <= m[:, t, 0]) & (m[:, t, 0] < m[:, t, 1]) & (m[:, t, 1] < n)).all())
    assert bool(torch.isfinite(s1).all()) and bool((s1 <= 1e-6).all())


def test_oracle_parity_50x1024_synthetic(sd0, gpu_models):
    """One config-2 sized alignment with phylogenetic signal against the oracle run on the box's CPU, both precisions."""
    import nnj_oracle as O
    data = O.evolved_msa(1, 50, 1024, seed=33)
    mask = torch.zeros(1, 1024, dtype=torch.bool)
    ref = O.rollout(sd0, data, mask)
    for prec in ("fp32", "bf16x3"):
        merges, slp, trace = gpu_models[prec].rollout_fused(data.cuda(), mask.cuda(), want_logits=True)
        assert torch.equal(merges.cpu().long(), ref["merges"]), prec
        off = 0
        for lg in ref["logits"]:
            p = lg.shape[1]
            assert _rel(trace[:, off:off + p].cpu(), lg) < LOGIT_TOL, prec
            off += p


def test_error_paths(gpu_model):
    from neuralnj_b200 import NnjError, PhyloATTN, inference_config
    cfg = inference_config()
    cfg.model.embed_dim = 32
    with pytest.raises(NnjError):
        PhyloATTN(cfg).cuda().handle()
    with pytest.raises(NnjError):
        PhyloATTN(inference_config()).handle()          # CPU model: no fallback
    with pytest.raises(NnjError):
        PhyloATTN(inference_config(), precision="fp16").cuda().handle()   # unknown precision mode
    with pytest.raises(NnjError):
        gpu_model.rollout_fused(torch.zeros(1, 1, 8, 4, dtype=torch.int8).cuda(), torch.zeros(1, 8, dtype=torch.bool).cuda())
