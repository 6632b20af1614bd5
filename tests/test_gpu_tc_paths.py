"""GPU: the tensor-core (bf16x3) NJ-loop kernels across the tile shapes they special-case.

k_alpha_v3 / k_score_tc treat a launch of <= 64 pairs (every step after the first, and the tail launch of step 0 when
R(R-1)/2 mod 256 <= 64) differently from full 128-pair tiles: the alpha tile is split by site parity, the score tile
duplicates its pairs into rows 64..127.  The cases below put the step-0 pair count on both sides of those boundaries and
check the whole trajectory against the CPU oracle with the same bar as test_gpu_parity (logits <= 2e-5 of the step's
max |logit|; merges identical unless the oracle's own top-2 gap is below the bf16x3 tie tolerance)."""
import pytest
import torch

from test_gpu_parity import LOGIT_TOL, TIE_TOL, _assert_equivalent_trajectory, _min_rel_gap, _rel

pytestmark = pytest.mark.gpu


# taxa -> step-0 pairs: 12 -> 66 (one full tile), 17 -> 136 (128 + 8: second score tile duplicated), 24 -> 276 (second
# alpha launch of 20 pairs: parity split at step 0), 33 -> 528 (two launches + 16), 63 -> 1953 (largest tensor-core size); 40 x 256:
# the late steps (33-64 pairs: 2-way site split, <= 32: lane quarters, <= 16: register-fragment kernels) over two 128-site groups
@pytest.mark.parametrize("R,L", [(12, 128), (17, 192), (24, 128), (33, 64), (63, 72), (64, 64), (49, 136), (40, 256)])
def test_tile_shapes_match_oracle(R, L, sd0, gpu_models):
    import nnj_oracle as O
    data = O.evolved_msa(2, R, L, seed=100 + R)
    mask = torch.zeros(2, L, dtype=torch.bool)
    ref = O.rollout(sd0, data, mask)
    merges, slp, trace = gpu_models["bf16x3"].rollout_fused(data.cuda(), mask.cuda(), want_logits=True)
    merges, trace = merges.cpu().long(), trace.cpu()
    if torch.equal(merges, ref["merges"]):
        off = 0
        for lg in ref["logits"]:
            p = lg.shape[1]
            assert _rel(trace[:, off:off + p], lg) < LOGIT_TOL
            off += p
    else:
        assert _min_rel_gap(ref["logits"]) < TIE_TOL["bf16x3"], "merge lists differ although no step is tie-ambiguous"
        _assert_equivalent_trajectory(sd0, data, mask, merges, trace, TIE_TOL["bf16x3"])


def test_padded_sites_on_tensor_core_path(sd0, gpu_models):
    """Padded sites (mask True): alpha sums over them, the score does not (model.py:97,118)."""
    import nnj_oracle as O
    L = 128
    data = O.evolved_msa(2, 14, L, seed=7)
    mask = torch.zeros(2, L, dtype=torch.bool)
    mask[0, 100:] = True
    mask[1, 64:] = True
    data[mask[:, None, :].expand(-1, 14, -1)] = 0
    ref = O.rollout(sd0, data, mask)
    merges, _, trace = gpu_models["bf16x3"].rollout_fused(data.cuda(), mask.cuda(), want_logits=True)
    assert torch.equal(merges.cpu().long(), ref["merges"])
    off = 0
    for lg in ref["logits"]:
        p = lg.shape[1]
        assert _rel(trace[:, off:off + p].cpu(), lg) < LOGIT_TOL
        off += p


def test_batch_larger_than_one_chunk(gpu_models):
    """More alignments than one workspace chunk (128): chunks are equal-sized and results do not depend on the chunking."""
    import nnj_oracle as O
    model = gpu_models["bf16x3"]
    B = 150
    data = O.evolved_msa(B, 9, 64, seed=3)
    mask = torch.zeros(B, 64, dtype=torch.bool)
    m_all, s_all, _ = model.rollout_fused(data.cuda(), mask.cuda())
    m_a, s_a, _ = model.rollout_fused(data[:37].cuda(), mask[:37].cuda())
    m_b, s_b, _ = model.rollout_fused(data[140:].cuda(), mask[140:].cuda())
    assert torch.equal(m_all[:37], m_a) and torch.equal(s_all[:37], s_a)
    assert torch.equal(m_all[140:], m_b) and torch.equal(s_all[140:], s_b)
    mh = model.rollout_host(data, mask)
    assert torch.equal(mh, m_all.cpu())


def test_stepwise_api_equals_fused_on_tensor_core_path(golden, gpu_models):
    """decode_zxr / aggregate / merge_state (the reference's step-wise calls) against the fused rollout, bf16x3."""
    model = gpu_models["bf16x3"]
    g = golden("t20x256_117")
    data, mask = g.data.cuda(), g.mask.cuda()
    merges, _, trace = model.rollout_fused(data, mask, want_logits=True)
    X = model.encode_zxr(data, mask)
    logits = model.decode_zxr(X, mask, (None, None, None))["logits"]
    off = 0
    R = data.shape[1]
    for t in range(5):
        p = logits.shape[1]
        assert _rel(logits.cpu(), trace[:, off:off + p].cpu()) < LOGIT_TOL
        off += p
        ij = merges[:, t].long()
        assert torch.equal(logits.argmax(1).cpu(), torch.tensor([model_pair_index(int(i), int(j), R - t) for i, j in ij.tolist()]))
        X = model.merge_state(X, ij)
        logits = model.decode_zxr(X, mask, (ij.int(), None, logits))["logits"]


def model_pair_index(i, j, n):
    return i * n - i * (i + 1) // 2 + (j - i - 1)


def test_full_size_properties_tensor_core(gpu_models):
    """Config-2 shape (50 x 1024) on the tensor-core path: bit-exact rerun, batch independence, same result at any batch size."""
    import nnj_oracle as O
    model = gpu_models["bf16x3"]
    data = O.evolved_msa(5, 50, 1024, seed=22)
    mask = torch.zeros(5, 1024, dtype=torch.bool)
    m1, s1, t1 = model.rollout_fused(data.cuda(), mask.cuda(), want_logits=True)
    m2, s2, t2 = model.rollout_fused(data.cuda(), mask.cuda(), want_logits=True)
    assert torch.equal(m1, m2) and torch.equal(s1, s2) and torch.equal(t1, t2)
    m3, s3, t3 = model.rollout_fused(data[3:4].cuda(), mask[3:4].cuda(), want_logits=True)
    assert torch.equal(m3, m1[3:4]) and torch.equal(t3, t1[3:4])


def test_large_alignment_200x4096(gpu_models):
    """BASELINE config 4 (200 taxa x 4096 sites, Argmax): 201 node slots put the NJ loop on the large-slot tensor-core path (k_blend_planes,
    split-K alpha GEMM, k_score_big; DESIGN 4.4), the encoder stays on tcgen05.  The CPU oracle needs minutes at this size, so the check is by properties: valid merge lists, finite
    log-probabilities, bit-exact rerun, and batch independence (B = 2 against its own B = 1 halves)."""
    import nnj_oracle as O
    model = gpu_models["bf16x3"]
    R, L = 200, 4096
    data = O.synthetic_msa(2, R, L, seed=7)
    mask = torch.zeros(2, L, dtype=torch.bool)
    m2, s2, _ = model.rollout_fused(data.cuda(), mask.cuda())
    m1, s1, _ = model.rollout_fused(data[:1].cuda(), mask[:1].cuda())
    m1b, _, _ = model.rollout_fused(data[:1].cuda(), mask[:1].cuda())
    assert torch.equal(m1, m1b)
    assert torch.equal(m2[:1], m1) and torch.equal(s2[:1], s1)
    mm = m2.cpu()
    for t in range(R - 1):
        n = R - t
        assert bool(((0 <= mm[:, t, 0]) & (mm[:, t, 0] < mm[:, t, 1]) & (mm[:, t, 1] < n)).all())
    assert bool(torch.isfinite(s2).all())


# Row-attention GEMM dispatch (nnj_tc.cu): ctx = P V has N = 8 R columns and M = C rows.  C % 256 == 0 selects the CTA-pair kernels:
# N <= 256 (R <= 32) k_tc_gemm2<true> with one (ragged) N tile, 256 < N <= 512 the one-pass k_tc_gemm2w (second UMMA of 16 .. 256 columns:
# R = 33 -> 16, 45 -> 112, 50 -> 144, 64 -> 256), N > 512 k_tc_gemm2<true> with three N tiles; C = 384 (odd number of 128-row blocks) stays on
# the single-CTA kernel.  S = Q K^T (N = C) runs the K-major pair kernel whenever C % 256 == 0.
@pytest.mark.parametrize("R,C", [(32, 256), (33, 256), (45, 256), (64, 512), (70, 256), (50, 384)])
def test_row_gemm_variants_encoder_matches_oracle(R, C, sd0, gpu_models):
    import nnj_oracle as O
    data = O.evolved_msa(1, R, C, seed=R + C)
    mask = torch.zeros(1, C, dtype=torch.bool)
    mask[0, C - 24:] = True
    ref = O.encode(sd0, data, mask)
    got = gpu_models["bf16x3"].encode_zxr(data.cuda(), mask.cuda()).cpu()
    err = float((got - ref).abs().max() / ref.abs().max())
    assert err < 5e-5, err
