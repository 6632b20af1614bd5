"""GPU: the incremental pair-score kernel (k_score_inc: channels on the TMEM lanes, pairs padded to 16, 32, 48 or 64 columns).

Every NJ step after the first scores the new node's pairs, at most 63 over at most 64 slots, on this kernel (the last steps, <= 16 pairs
over <= 16 nodes, on k_score_small).  A rollout from R taxa runs it at every pair count from R - 2 down to 17, so the shapes below put
each padding width and both sides of every routing threshold under test.  The whole trajectory is checked against the CPU oracle with
the bf16x3 bar of the breadth tests, 4e-5 of a step's max |logit|: with few sites the split-bf16 error does not average down (step 0,
on k_score_tc, measures 2.9e-5 at 63 taxa x 8 sites).  Site counts include one site pair per item (8), a partial 128-site group (120, 1032) and several groups."""
import pytest
import torch

from test_gpu_parity import LOGIT_TOL_BY_PREC, TIE_TOL, _assert_equivalent_trajectory, _min_rel_gap, _rel

pytestmark = pytest.mark.gpu


def _check_against_oracle(sd0, model, data, mask):
    import nnj_oracle as O
    ref = O.rollout(sd0, data, mask)
    merges, _, trace = model.rollout_fused(data.cuda(), mask.cuda(), want_logits=True)
    merges, trace = merges.cpu().long(), trace.cpu()
    if torch.equal(merges, ref["merges"]):
        off = 0
        for lg in ref["logits"]:
            p = lg.shape[1]
            assert _rel(trace[:, off:off + p], lg) < LOGIT_TOL_BY_PREC["bf16x3"], off
            off += p
    else:
        assert _min_rel_gap(ref["logits"]) < TIE_TOL["bf16x3"], "merge lists differ although no step is tie-ambiguous"
        _assert_equivalent_trajectory(sd0, data, mask, merges, trace, TIE_TOL["bf16x3"], LOGIT_TOL_BY_PREC["bf16x3"])


# (taxa, sites, alignments): 63 taxa = 61 .. 2 new pairs per step over up to 64 slots
@pytest.mark.parametrize("R,L,B", [(63, 8, 1), (50, 120, 3), (34, 1032, 1), (19, 1024, 3)])
def test_incremental_steps_match_oracle(R, L, B, sd0, gpu_models):
    import nnj_oracle as O
    data = O.evolved_msa(B, R, L, seed=500 + R)
    mask = torch.zeros(B, L, dtype=torch.bool)
    _check_against_oracle(sd0, gpu_models["bf16x3"], data, mask)


def test_incremental_steps_masked_sites(sd0, gpu_models):
    import nnj_oracle as O
    R, L = 40, 264
    data = O.evolved_msa(3, R, L, seed=41)
    mask = torch.zeros(3, L, dtype=torch.bool)
    mask[0, 200:] = True
    mask[1, 3::7] = True
    mask[2, 128:136] = True
    data[mask[:, None, :].expand(-1, R, -1)] = 0
    _check_against_oracle(sd0, gpu_models["bf16x3"], data, mask)


def test_tree_alone_equals_tree_in_batch(gpu_models):
    """A tree's scores do not depend on the other trees of its batch or chunk: bit-identical merges and logits, alone and at
    position 130 of a 131-tree batch (two workspace chunks)."""
    import nnj_oracle as O
    model = gpu_models["bf16x3"]
    R, L = 30, 136
    data = O.evolved_msa(131, R, L, seed=9)
    mask = torch.zeros(131, L, dtype=torch.bool)
    m_all, _, t_all = model.rollout_fused(data.cuda(), mask.cuda(), want_logits=True)
    for i in (0, 130):
        m_one, _, t_one = model.rollout_fused(data[i:i + 1].cuda(), mask[i:i + 1].cuda(), want_logits=True)
        assert torch.equal(m_one.cpu(), m_all[i:i + 1].cpu())
        assert torch.equal(t_one.cpu(), t_all[i:i + 1].cpu())
