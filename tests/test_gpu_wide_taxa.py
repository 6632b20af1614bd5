"""GPU: alignments of 129 to 400 taxa against the oracle run in fp64.

The kernels change with the taxon count R (the NJ pool has S = R + 1 slots):
* R > 128: the encoder runs the row attention on tcgen05 and the rest of the layer on the fp32 tile-planar kernels (k_out_proj,
  k_ln_qkv<false>, k_col_attn); C % 256 == 0 selects the CTA-pair row GEMMs (ceil(8R / 256) N tiles, ragged at 129, 333, 400) and the
  fused Q K^T softmax, C = 200 the single-CTA GEMMs, C = 250 (not a multiple of 8) the fp32 encoder.
* R <= 255: the bf16x3 NJ loop stays on the large-slot path (k_blend_planes, split-K alpha, k_alpha_softmax_wide, k_score_big with
  bn = 64 / 128 / 256 by live nodes).  R >= 256 (S > 256): both precisions run the fp32 NJ kernels (k_alpha, k_alpha_softmax,
  k_score<GLOB>, k_merge).
* R > 400: k_col_attn would need more than 200 KB of shared memory; the encoder refuses the shape, and so does bootstrap_support.

The reference is nnj_oracle with the seed-0 weights cast to fp64, so its own rounding is far below the tolerances.  Wide trees have
near-ties (top-1 / top-2 gaps of 1e-8 relative at 400 taxa), so a rollout passes either strictly (identical merges, logits within
LOGIT_TOL_BY_PREC) or, only where the oracle's own gap is below TIE_TOL, by the teacher-forced replay of test_gpu_parity.  Each oracle
run is cached for the module and shared by both precisions."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import support_oracle as SO
from conftest import ROOT
from test_gpu_parity import LOGIT_TOL_BY_PREC, STATE_TOL, TIE_TOL, _assert_equivalent_trajectory, _max_trace_err, _min_rel_gap, _rel

pytestmark = pytest.mark.gpu

PAIR_CHUNK = 128         # the oracle scores step 0 in chunks of pairs: [B, pairs, C, D] fp64 temporaries would not fit otherwise
PRECS = ["fp32", "bf16x3"]


@pytest.fixture(scope="module")
def sd64(sd0):
    import nnj_oracle as O
    return O.cast_state_dict(sd0, torch.float64)


@pytest.fixture(scope="module")
def oracle64():
    """fp64 oracle results by key ((kind, R, L, seed, mask) and what else selects the input): computed once, used by both precisions."""
    cache = {}

    def get(key, compute):
        if key not in cache:
            cache[key] = compute()
        return cache[key]
    return get


def _msa(B, R, L, seed, pad=0):
    """evolved_msa with the last `pad` columns of the last tree padded (mask True, no tokens)."""
    import nnj_oracle as O
    data = O.evolved_msa(B, R, L, seed=seed)
    mask = torch.zeros(B, L, dtype=torch.bool)
    if pad:
        mask[B - 1, L - pad:] = True
        data[B - 1, :, L - pad:] = 0
    return data, mask


def _rollout_ref(oracle64, sd64, data, mask, key, gumbel=None):
    import nnj_oracle as O

    def run():
        ref = O.rollout(sd64, data, mask, gumbel=gumbel, pair_chunk=PAIR_CHUNK)
        return {k: ref[k] for k in ("merges", "logits", "selected_log_ps", "state0")}
    return oracle64(key, run)


def _check_trajectory(tag, prec, data, mask, merges, slp, trace, ref, sd64, parity_report):
    """Strict (identical merges, logits and selected log-probabilities within the bounds of test_gpu_breadth._check_against_oracle) or,
    only where the oracle's own gap is below TIE_TOL[prec], tie-aware (teacher-forced replay on the fp64 oracle)."""
    gap = _min_rel_gap(ref["logits"])
    entry = {"precision": prec, "source": "fp64 oracle on the box's CPU", "shape": list(data.shape[:3]), "min_rel_top2_gap": gap,
             "mode": "strict", "max_logit_rel_err": None}
    parity_report[f"{tag}/{prec}"] = entry
    if not torch.equal(merges, ref["merges"]):
        step = int((merges != ref["merges"]).any(-1).any(0).nonzero()[0])
        assert gap < TIE_TOL[prec], f"merge lists differ at step {step} although no step is tie-ambiguous (min gap {gap:.2e})"
        entry["mode"] = "tie_aware"
        entry["max_logit_rel_err"] = _assert_equivalent_trajectory(sd64, data, mask, merges, trace, TIE_TOL[prec], LOGIT_TOL_BY_PREC[prec],
                                                                   pair_chunk=PAIR_CHUNK)
        return
    entry["max_logit_rel_err"] = _max_trace_err(trace, ref["logits"])
    assert entry["max_logit_rel_err"] < LOGIT_TOL_BY_PREC[prec]
    R = data.shape[1]
    scale = max(float(lg.abs().max()) for lg in ref["logits"])
    assert float((slp[:, :R - 2] - ref["selected_log_ps"]).abs().max()) < max(1e-3, 2 * LOGIT_TOL_BY_PREC[prec] * scale)


# ------------------------------------------------------------------ encoder
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("C", [256, 200, 250])
@pytest.mark.parametrize("R", [129, 200, 256, 333, 400])
def test_encoder_matches_fp64_oracle(R, C, prec, sd64, oracle64, gpu_models):
    """B = 2, the second tree with 24 padded columns."""
    import nnj_oracle as O
    data, mask = _msa(2, R, C, seed=R + C, pad=24)
    ref = oracle64(("encode", R, C, R + C, "pad24"), lambda: O.encode(sd64, data, mask))
    got = gpu_models[prec].encode_zxr(data.cuda(), mask.cuda()).cpu().double()
    assert got.shape == ref.shape
    err = float((got - ref).abs().max())
    assert err / float(ref.abs().max()) < 5e-5, err
    assert err < STATE_TOL


# ------------------------------------------------------------------ whole rollouts
# 129: first shape of the fp32 encoder tail; 255: the last large-slot shape (its rollout crosses every bn boundary); 256, 257: the
# first shapes on the fp32 NJ kernels in both precisions; 400: the widest shape the encoder takes; 200 x 248: tcgen05 with a ragged
# last site group; 150 x 250: the fp32 kernels throughout
ROLLOUT_CASES = [(129, 64), (255, 72), (256, 64), (257, 72), (320, 64), (400, 64), (200, 248), (150, 250)]


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("R,L", ROLLOUT_CASES)
def test_rollout_matches_fp64_oracle(R, L, prec, sd64, oracle64, gpu_models, parity_report):
    data, mask = _msa(1, R, L, seed=300 + R)
    ref = _rollout_ref(oracle64, sd64, data, mask, ("rollout", R, L, 300 + R, "none"))
    merges, slp, trace = gpu_models[prec].rollout_fused(data.cuda(), mask.cuda(), want_logits=True)
    _check_trajectory(f"wide_{R}x{L}", prec, data, mask, merges.cpu().long(), slp.cpu(), trace.cpu(), ref, sd64, parity_report)


# ------------------------------------------------------------------ step-wise API above 256 slots
def _pair_index(i, j, n):
    return i * n - i * (i + 1) // 2 + (j - i - 1)


@pytest.mark.parametrize("prec", PRECS)
def test_stepwise_api_equals_fused_above_256_slots(prec, sd64, gpu_models):
    """decode_zxr (full, then incremental: k_score<true/false>), aggregate (k_alpha1) and merge_state at R = 300 against the fused
    rollout, and the merged node against the fp64 oracle's aggregate of the same device state."""
    import nnj_oracle as O
    model = gpu_models[prec]
    R, L = 300, 64
    data, mask = _msa(2, R, L, seed=31)
    data, mask = data.cuda(), mask.cuda()
    merges, _, trace = model.rollout_fused(data, mask, want_logits=True)
    X = model.encode_zxr(data, mask)
    logits = model.decode_zxr(X, mask, (None, None, None))["logits"]
    off = 0
    for t in range(5):
        n = R - t
        p = logits.shape[1]
        assert p == n * (n - 1) // 2
        lg = logits.cpu()
        assert _rel(lg, trace[:, off:off + p].cpu()) < LOGIT_TOL_BY_PREC[prec], t
        off += p
        ij = merges[:, t].long()
        # the fused rollout's pair is an argmax of the step-wise logits (up to the tie tolerance: two kernels, two summation orders)
        chosen = lg.gather(1, torch.tensor([[_pair_index(i, j, n)] for i, j in ij.tolist()])).squeeze(1)
        slack = (lg.max(1).values - chosen) / lg.abs().max(1).values
        assert float(slack.max()) < TIE_TOL[prec], (t, float(slack.max()))
        new = model.aggregate(None, None, (ij[:, 0], ij[:, 1]), batchwise_ij_indices=True)
        Xd = X.cpu().double()
        ar = torch.arange(2)
        ijc = ij.cpu()
        want = O.aggregate(sd64, Xd, Xd[ar, ijc[:, 0]].unsqueeze(1), Xd[ar, ijc[:, 1]].unsqueeze(1), ijc[:, :1], ijc[:, 1:], L)
        assert float((new.cpu().double() - want).abs().max()) < 5e-5, t
        X = model.merge_state(X, ij)
        for b in range(2):
            i, j = ij[b].tolist()
            assert float((X[b, i].cpu().double() - want[b, 0]).abs().max()) < 5e-5, t
            keep = [r for r in range(n) if r not in (i, j)]           # slot i <- the new node, slot j removed, the rest copied
            assert torch.equal(X[b, [r - (r > j) for r in keep]].cpu(), Xd[b, keep].float()), t
        logits = model.decode_zxr(X, mask, (ij.int(), None, logits))["logits"]


# ------------------------------------------------------------------ determinism
_CHUNK_SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/oracle")
import nnj_oracle as O
from neuralnj_b200 import PhyloATTN, inference_config
torch.manual_seed(0)
m = PhyloATTN(inference_config(), precision="bf16x3").cuda().eval()
data = O.evolved_msa(3, 300, 64, seed=41)
mask = torch.zeros(3, 64, dtype=torch.bool)
merges, slp, trace = m.rollout_fused(data.cuda(), mask.cuda(), want_logits=True)
torch.save({"merges": merges.cpu(), "slp": slp.cpu(), "trace": trace.cpu()}, sys.argv[2])
"""


def test_wide_rollout_is_deterministic(gpu_models, tmp_path):
    """R = 300: a rerun, the B = 1 slices of a B = 3 batch and one tree per workspace chunk (NNJ_CHUNK_MAX=1, read once per process:
    a subprocess) all give the same bits."""
    R, L = 300, 64
    data, mask = _msa(3, R, L, seed=41)
    data, mask = data.cuda(), mask.cuda()
    for prec in PRECS:
        model = gpu_models[prec]
        full = [x.cpu() for x in model.rollout_fused(data, mask, want_logits=True)]
        again = [x.cpu() for x in model.rollout_fused(data, mask, want_logits=True)]
        assert all(torch.equal(a, b) for a, b in zip(full, again)), prec
        for b in range(3):
            one = [x.cpu() for x in model.rollout_fused(data[b:b + 1], mask[b:b + 1], want_logits=True)]
            assert all(torch.equal(a[b:b + 1], o) for a, o in zip(full, one)), (prec, b)
        if prec == "bf16x3":
            path = str(tmp_path / "chunk1.pt")
            subprocess.run([sys.executable, "-c", _CHUNK_SCRIPT, ROOT, path], check=True, env={**os.environ, "NNJ_CHUNK_MAX": "1"},
                           timeout=600)
            got = torch.load(path)
            assert torch.equal(got["merges"], full[0]) and torch.equal(got["slp"], full[1]) and torch.equal(got["trace"], full[2])


# ------------------------------------------------------------------ sampling
@pytest.mark.parametrize("prec", PRECS)
def test_gumbel_rollout_at_256_taxa_replays_on_fp64_oracle(prec, sd64, oracle64, gpu_models):
    """Two Gumbel-max samples from one shared encoder state: with the same noise the fp64 oracle picks the same trajectories."""
    R, L, S = 256, 64, 2
    data, mask = _msa(1, R, L, seed=57)
    gen = torch.Generator().manual_seed(6)
    u = torch.rand(S, R - 1, R * (R - 1) // 2, generator=gen).clamp_(1e-20, 1 - 1e-7)
    gum = -torch.log(-torch.log(u))
    model = gpu_models[prec]
    state = model.encode_zxr(data.cuda(), mask.cuda()).expand(S, -1, -1, -1).contiguous()
    merges, slp, _ = model.rollout_fused(batch_seq_mask=mask.expand(S, -1).contiguous().cuda(), gumbel=gum.cuda(), state=state)
    ref = _rollout_ref(oracle64, sd64, data.expand(S, -1, -1, -1).contiguous(), mask.expand(S, -1).contiguous(),
                       ("gumbel", R, L, 57, "none", 6), gumbel=gum)
    assert torch.equal(merges.cpu().long(), ref["merges"])
    assert len({tuple(m.flatten().tolist()) for m in merges.cpu()}) > 1
    assert float((slp[:, :R - 2].cpu() - ref["selected_log_ps"]).abs().max()) < 1e-3


# ------------------------------------------------------------------ the limit
def test_more_than_400_taxa_are_refused_cleanly(gpu_models):
    """401 taxa: k_col_attn would need more than 200 KB of shared memory, so encode_zxr and rollout_fused raise "max 400"; a 400-taxon
    rollout on the same model afterwards gives the bits it gave before (no CUDA error left behind)."""
    from neuralnj_b200 import NnjError
    L = 64
    data, mask = _msa(1, 401, L, seed=401)
    data, mask = data.cuda(), mask.cuda()
    for prec in PRECS:
        model = gpu_models[prec]
        before = [x.cpu() for x in model.rollout_fused(data[:, :400], mask, want_logits=True)]
        with pytest.raises(NnjError, match="max 400"):
            model.encode_zxr(data, mask)
        with pytest.raises(NnjError, match="max 400"):
            model.rollout_fused(data, mask)
        after = [x.cpu() for x in model.rollout_fused(data[:, :400], mask, want_logits=True)]
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip(before, after)), prec


# ------------------------------------------------------------------ bootstrap
@pytest.mark.parametrize("prec", PRECS)
def test_bootstrap_support_at_300_taxa(prec, sd64, oracle64, gpu_models, parity_report, monkeypatch):
    """8 replicates of a 300 x 64 alignment: the replicate columns are the restatement's, each replicate tree is the fp64 oracle's
    (strict or tie-aware), FBP and TBE are support_from_newicks on the device's own merge lists, chunks of 3 change nothing."""
    import nnj_oracle as O
    from neuralnj_b200 import support as SUP
    R, L, N, seed = 300, 64, 8, 12
    model = gpu_models[prec]
    data, mask = _msa(1, R, L, seed=R)
    keys = [f"taxon{i}" for i in range(R)]
    batch = {"data": data, "seq_weights": torch.ones(1, L), "seqs": [["A" * L] * R], "seq_keys": [keys]}
    res = SUP.bootstrap_support(batch, model, N, seed=seed)
    m0, _, _ = model.rollout_fused(data.cuda(), mask.cuda())
    assert res["tree"] == O.newick_from_merges(m0[0].cpu().tolist(), keys)
    assert len(res["splits"]) == R - 3
    reps = SUP.bootstrap_columns(data[0].cuda(), L, seed, 0, N)
    masks = mask.expand(N, -1).contiguous()
    merges, slp, trace = model.rollout_fused(reps, masks.cuda(), want_logits=True)
    merges, slp, trace, reps = merges.cpu().long(), slp.cpu(), trace.cpu(), reps.cpu()
    assert torch.equal(reps, SO.bootstrap_columns(data[0], L, seed, 0, N))
    ref = _rollout_ref(oracle64, sd64, reps, masks, ("bootstrap", R, L, R, "none", seed, N))
    for b in range(N):
        one = {"merges": ref["merges"][b:b + 1], "logits": [lg[b:b + 1] for lg in ref["logits"]],
               "selected_log_ps": ref["selected_log_ps"][b:b + 1]}
        _check_trajectory(f"wide_{R}x{L}_boot{b}", prec, reps[b:b + 1], masks[b:b + 1], merges[b:b + 1], slp[b:b + 1], trace[b:b + 1], one,
                          sd64, parity_report)
    want = SO.support_from_newicks(res["tree"], [O.newick_from_merges(m.tolist(), keys) for m in merges])
    assert set(res["splits"]) == set(want)
    for sp, f, t in zip(res["splits"], res["fbp"], res["tbe"]):
        assert (f, t) == want[sp]
    monkeypatch.setattr(SUP, "CHUNK", 3)
    other = SUP.bootstrap_support(batch, model, N, seed=seed)
    assert np.array_equal(other["fbp"], res["fbp"]) and np.array_equal(other["tbe"], res["tbe"])
    assert other["newick_fbp"] == res["newick_fbp"] and other["newick_tbe"] == res["newick_tbe"]
