"""GPU parity breadth (round 2): the code paths and inputs the round-1 suite never compared with the oracle.

* all 128 files of data_gen/data/test/len1024/taxa50 (the configs[1] parity set of SURVEY 8d), reference-executed, as one batch.
* wide goldens - 16 files of the reference's data_gen/data/test/len1024/taxa50 and 4 of len1024/taxa100, executed by the
  unmodified reference (oracle/make_golden.py wide); inputs are read back from the .phy files through load_pi_instance.
* BASELINE config-4 code paths against the pair-chunked oracle: more than 1024 sites (three-pass row softmax
  k_softmax_rows_split), more than 63 taxa (the NJ loop's large-slot path), more than 128 taxa (the CUDA-core column block),
  and the 200 x 4096 shape itself (minutes of CPU oracle time: runs only with NNJ_RUN_SLOW=1).
* site counts that are not a multiple of 8 in a tensor-core precision mode (documented fall-back to the fp32 kernels).
* the benchmark's own input (config-2 generator, iid tokens) against the oracle.
* the reference-signature entry points: Argmax_inference / Search_inference write .tre files; Agmax_one_instance, RL_Search.
Every case records how it passed in profiles/r02_parity.json (conftest.parity_report)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLD
from test_gpu_parity import LOGIT_TOL_BY_PREC, TIE_TOL, _assert_equivalent_trajectory, _max_trace_err, _min_rel_gap, _rel

pytestmark = pytest.mark.gpu

WIDE_DIR = os.path.join(GOLD, "wide")


def _wide_names():
    idx = os.path.join(WIDE_DIR, "INDEX.txt")
    if not os.path.exists(idx):
        return []
    with open(idx) as f:
        return [ln.strip() for ln in f if ln.strip()]


@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
@pytest.mark.parametrize("name", _wide_names())
def test_wide_reference_goldens(name, prec, sd0, gpu_models, parity_report):
    """Reference-executed records of the 50 x 1024 / 100 x 1024 test sets: identical merge list and Newick (tie-aware only when the
    record's own gap is below the precision's tie tolerance), step-0 logits and selected log-probabilities close."""
    from neuralnj_b200 import PhyInferEnv, inference_config, load_pi_instance
    z = np.load(os.path.join(WIDE_DIR, name + ".npz"), allow_pickle=False)
    batch = load_pi_instance(os.path.join(WIDE_DIR, name + ".phy"))
    data, mask = batch["data"], batch["seq_weights"] == 0
    want = torch.from_numpy(z["merges"]).long()
    gap = float(np.min(z["step_top2_gap"][:-1] / z["step_max_abs_logit"][:-1]))
    merges, slp, trace = gpu_models[prec].rollout_fused(data.cuda(), mask.cuda(), want_logits=True)
    merges, slp, trace = merges.cpu().long(), slp.cpu(), trace.cpu()
    entry = {"precision": prec, "source": "reference golden (tests/golden/wide): " + str(z["source"]), "shape": list(data.shape[:3]),
             "min_rel_top2_gap": gap, "mode": "strict", "max_logit_rel_err": None}
    parity_report[f"{name}/{prec}"] = entry
    if not torch.equal(merges, want) and gap < TIE_TOL[prec]:
        entry["mode"] = "tie_aware"
        _assert_equivalent_trajectory(sd0, data, mask, merges, trace, TIE_TOL[prec], LOGIT_TOL_BY_PREC[prec])
        return
    assert torch.equal(merges, want), f"first differing step: {int((merges != want).any(-1).any(0).nonzero()[0])}"
    l0 = torch.from_numpy(z["logits0"])
    entry["max_logit_rel_err"] = _rel(trace[:, :l0.shape[1]], l0)
    assert entry["max_logit_rel_err"] < LOGIT_TOL_BY_PREC[prec]
    R = data.shape[1]
    assert float((slp[:, :R - 2] - torch.from_numpy(z["selected_log_ps"])).abs().max()) < 1e-3
    env = PhyInferEnv(inference_config(), torch.device("cpu"))
    env.init_states(batch["seqs"], batch["seq_keys"], data)
    env.replay_merges(merges)
    assert env.states[0].subtrees[0].utree_op_str == str(z["newick"][0])


ALL50_DIR = os.path.join(GOLD, "all50")


def _load_all50():
    """The 128-file record, stored as parts of 64 alignments (each file stays below 1 MB), concatenated in file order."""
    parts = [np.load(os.path.join(ALL50_DIR, f), allow_pickle=False)
             for f in sorted(os.listdir(ALL50_DIR)) if f.startswith("len1024_taxa50_part")]
    return {k: parts[0][k] if k == "shape" else np.concatenate([p[k] for p in parts]) for k in parts[0].files}


@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
def test_all_len1024_taxa50_files_match_reference(prec, sd0, gpu_models, parity_report):
    """SURVEY.md 8(d), configs[1] parity set: ALL 128 alignments of the reference's data_gen/data/test/len1024/taxa50, each executed by
    the unmodified reference (oracle/make_golden.py all50), run here as one batch of 128: merge list and Newick identical per file;
    a file whose own top-2 gap is below the precision's tie tolerance may pass by teacher-forced replay on the oracle instead."""
    from neuralnj_b200 import PhyInferEnv, inference_config
    z = _load_all50()
    assert z["merges"].shape[0] == 128
    R, L, V = (int(x) for x in z["shape"])
    N = z["data_bits"].shape[0]
    data = torch.from_numpy(np.unpackbits(z["data_bits"], axis=1)[:, :R * L * V].reshape(N, R, L, V).astype(np.int8))
    mask = torch.zeros(N, L, dtype=torch.bool)
    want = torch.from_numpy(z["merges"].astype(np.int64))
    merges, slp, trace = gpu_models[prec].rollout_fused(data.cuda(), mask.cuda(), want_logits=True)
    merges, slp, trace = merges.cpu().long(), slp.cpu(), trace.cpu()
    gaps = np.min(z["step_top2_gap"][:, :-1] / z["step_max_abs_logit"][:, :-1], axis=1)
    keys = [[str(k) for k in row] for row in z["seq_keys"]]
    env = PhyInferEnv(inference_config(), torch.device("cpu"))
    env.init_states([["A" * L] * R for _ in range(N)], keys, data)
    env.replay_merges(merges)
    tie_aware = []
    for b in range(N):
        name = str(z["source"][b])
        entry = {"precision": prec, "source": "reference golden (tests/golden/all50): " + name, "shape": [1, R, L],
                 "min_rel_top2_gap": float(gaps[b]), "mode": "strict", "max_logit_rel_err": None}
        parity_report[f"all50_{b:03d}/{prec}"] = entry
        if torch.equal(merges[b], want[b]):
            assert env.states[b].subtrees[0].utree_op_str == str(z["newick"][b]), name
            assert float((slp[b, :R - 2] - torch.from_numpy(z["selected_log_ps"][b])).abs().max()) < 2e-3, name
            continue
        assert gaps[b] < TIE_TOL[prec], f"{name}: merge list differs at step {int((merges[b] != want[b]).any(-1).nonzero()[0])} although no step is tie-ambiguous (min gap {gaps[b]:.2e})"
        entry["mode"] = "tie_aware"
        tie_aware.append(name)
        _assert_equivalent_trajectory(sd0, data[b:b + 1], mask[b:b + 1], merges[b:b + 1], trace[b:b + 1], TIE_TOL[prec], LOGIT_TOL_BY_PREC[prec])
    assert len(tie_aware) <= 16, tie_aware           # measured on B200: fp32 2 (the two exact-tie files), bf16x3 9 of the 62 files whose own gap is < 1e-5
    print(f"all50[{prec}]: {N - len(tie_aware)} of {N} files strict-identical, tie-aware: {tie_aware}")


def _check_against_oracle(tag, prec, data, mask, sd0, model, parity_report, pair_chunk=128):
    """Whole trajectory against the oracle run on this box's CPU (pair-chunked so that step 0 fits in memory)."""
    import nnj_oracle as O
    ref = O.rollout(sd0, data, mask, pair_chunk=pair_chunk)
    merges, slp, trace = model.rollout_fused(data.cuda(), mask.cuda(), want_logits=True)
    merges, trace = merges.cpu().long(), trace.cpu()
    gap = _min_rel_gap(ref["logits"])
    entry = {"precision": prec, "source": "oracle on the box's CPU", "shape": list(data.shape[:3]), "min_rel_top2_gap": gap, "mode": "strict",
             "max_logit_rel_err": None}
    parity_report[f"{tag}/{prec}"] = entry
    enc = model.encode_zxr(data.cuda(), mask.cuda()).cpu()
    assert float((enc - ref["state0"]).abs().max()) < 2e-4, "encoder output"
    if not torch.equal(merges, ref["merges"]):
        assert gap < TIE_TOL[prec], f"merge lists differ although no step is tie-ambiguous (min gap {gap:.2e})"
        entry["mode"] = "tie_aware"
        _assert_equivalent_trajectory(sd0, data, mask, merges, trace, TIE_TOL[prec], LOGIT_TOL_BY_PREC[prec])
        return
    entry["max_logit_rel_err"] = _max_trace_err(trace, ref["logits"])
    assert entry["max_logit_rel_err"] < LOGIT_TOL_BY_PREC[prec]
    R = data.shape[1]
    # log_softmax(logits)[action] moves by at most twice the absolute logit error, which is the relative tolerance times the logit scale
    # (200 x 4096: |logit| reaches the hundreds, a fixed 1e-3 would be tighter than the logit tolerance itself)
    scale = max(float(lg.abs().max()) for lg in ref["logits"])
    assert float((slp.cpu()[:, :R - 2] - ref["selected_log_ps"]).abs().max()) < max(1e-3, 2 * LOGIT_TOL_BY_PREC[prec] * scale)


# (taxa, sites, padded sites): 12 x 2048 -> rows longer than 1024 sites (k_softmax_rows_split) with a padded tail;
# 70 x 1280 -> more than 63 taxa (NJ large-slot path) and more than 1024 sites; 130 x 1104 -> more than 128 taxa (CUDA-core column
# block behind the tensor-core row attention / FFN)
@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
@pytest.mark.parametrize("R,L,pad", [(12, 2048, 300), (70, 1280, 0), (130, 1104, 0)])
def test_config4_code_paths_match_oracle(R, L, pad, prec, sd0, gpu_models, parity_report):
    import nnj_oracle as O
    data = O.evolved_msa(1, R, L, seed=200 + R)
    mask = torch.zeros(1, L, dtype=torch.bool)
    if pad:
        mask[0, L - pad:] = True
        data[mask[:, None, :].expand(-1, R, -1)] = 0
    _check_against_oracle(f"oracle_{R}x{L}" + ("_padded" if pad else ""), prec, data, mask, sd0, gpu_models[prec], parity_report)


@pytest.mark.skipif(os.environ.get("NNJ_RUN_SLOW") != "1", reason="200 x 4096 needs minutes of CPU oracle time: set NNJ_RUN_SLOW=1")
def test_config4_200x4096_matches_oracle(sd0, gpu_models, parity_report):
    import nnj_oracle as O
    data = O.evolved_msa(1, 200, 4096, seed=404)
    mask = torch.zeros(1, 4096, dtype=torch.bool)
    _check_against_oracle("oracle_200x4096", "bf16x3", data, mask, sd0, gpu_models["bf16x3"], parity_report, pair_chunk=64)


@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
@pytest.mark.parametrize("L", [250, 255, 248])
def test_site_counts_not_multiple_of_8(L, prec, sd0, gpu_models, parity_report):
    """A tensor-core precision mode with C % 8 != 0 (250, 255) runs the fp32 kernels - encoder AND NJ loop (nj_use_tc / use_tc);
    248 = 8 * 31 stays on tcgen05 with a ragged last site group.  load_pi_instance never pads, so real alignments hit this.
    (Round 2 found the fp32 row-attention GEMM reading 16-byte vectors from rows of pitch C: C % 4 != 0 faulted.)"""
    import nnj_oracle as O
    data = O.evolved_msa(2, 14, L, seed=50 + L)
    mask = torch.zeros(2, L, dtype=torch.bool)
    _check_against_oracle(f"oracle_14x{L}", prec, data, mask, sd0, gpu_models[prec], parity_report)


def test_bench_input_matches_oracle(sd0, gpu_models, parity_report):
    """The benchmark's own input (config-2 generator: iid tokens, seed 1234) on one alignment.  iid-random alignments give
    near-tie logits, so this case is expected to be the one that needs the tie-aware comparison most often."""
    import nnj_oracle as O
    data = O.synthetic_msa(1, 50, 1024, seed=1234)
    mask = torch.zeros(1, 1024, dtype=torch.bool)
    _check_against_oracle("bench_input_50x1024", "bf16x3", data, mask, sd0, gpu_models["bf16x3"], parity_report)


# ------------------------------------------------------------------ entry points with the reference's signatures
def _phy_dir(tmp_path, names):
    import shutil
    d = tmp_path / "msas"
    d.mkdir()
    for n in names:
        shutil.copyfile(os.path.join(GOLD, "msa", n + ".phy"), d / (n + ".phy"))
    return str(d)


def test_argmax_inference_writes_reference_trees(tmp_path, golden):
    """Argmax_inference (finetune_rl_search.py:478-509): one .tre per .phy, equal to the Newick the reference produced; the policy
    is built by _load_policy, i.e. in the default (bf16x3) precision."""
    from neuralnj_b200 import Argmax_inference, inference_config
    names = ["t20x256_10", "t20x256_117", "ex50x1024_73"]
    src = _phy_dir(tmp_path, names)
    cfgs = inference_config()
    torch.manual_seed(0)
    written = Argmax_inference(src, str(tmp_path / "out"), None, cfgs=cfgs)
    assert sorted(os.path.basename(w) for w in written) == sorted(n + ".tre" for n in names)
    for n in names:
        with open(tmp_path / "out" / (n + ".tre")) as f:
            assert f.read().strip() == golden(n).newick[0], n


def test_agmax_one_instance_result_dict(golden, gpu_models):
    from neuralnj_b200 import Agmax_one_instance, PhyInferEnv, inference_config
    cfgs = inference_config()
    cfgs.env.batch_size = 2                      # the reference expands the instance to cfgs.env.batch_size copies (:444)
    env = PhyInferEnv(cfgs, torch.device("cuda:0"))
    res = Agmax_one_instance(cfgs, os.path.join(GOLD, "msa", "t20x256_103.phy"), gpu_models["bf16x3"], env)
    assert res["best_tree_str"] == golden("t20x256_103").newick[0]
    assert res["score"] == -111111 and set(res) >= {"rf_distance", "rf_distance_raw", "raw_tree_score"}


def test_search_inference_and_rl_search(tmp_path, golden, gpu_models):
    """RL_Search / Search_inference (finetune_rl_search.py:338-427, 512-541): sampled rollouts from one shared encoder pass.
    Seeded -> reproducible; the returned tree is one of the sampled topologies, scored by the caller's scorer."""
    from neuralnj_b200 import PhyInferEnv, RL_Search, Search_inference, inference_config, rf_distance
    cfgs = inference_config()
    cfgs.env.batch_size = 4
    cfgs.num_episodes = 2
    path = os.path.join(GOLD, "msa", "t20x256_120.phy")
    model = gpu_models["bf16x3"]
    env = PhyInferEnv(cfgs, torch.device("cuda:0"))
    ref_tree = golden("t20x256_120").newick[0]
    calls = []

    def scorer(newick, keys, seqs):          # stands in for the RAxML-NG likelihood: closer to the Argmax tree is better
        calls.append(newick)
        return -float(rf_distance(newick, ref_tree))

    outs = []
    for _ in range(2):
        gen = torch.Generator(device="cuda:0").manual_seed(11)
        outs.append(RL_Search(cfgs, path, model, env, scorer=scorer, stop_step=4, generator=gen))
    assert outs[0]["the_best_tree"] == outs[1]["the_best_tree"] and outs[0]["the_best_score"] == outs[1]["the_best_score"]
    assert outs[0]["step_cur"] >= 4 and outs[0]["distinct_topologies"] >= 1
    assert outs[0]["the_best_tree"] in calls and outs[0]["the_best_score"] == max(-float(rf_distance(c, ref_tree)) for c in calls)
    src = _phy_dir(tmp_path, ["t20x256_120"])
    written = Search_inference(src, str(tmp_path / "out"), None, cfgs=cfgs, stop_step=2)
    with open(written[0]) as f:
        tree = f.read().strip()
    assert tree.endswith(";") and all(k in tree for k in golden("t20x256_120").seq_keys[0])


def test_cli_main_argmax(tmp_path, golden, monkeypatch):
    """`python -m neuralnj_b200.rollout --config_path cfg.yaml --infer_opt Argmax` (finetune_rl_search.py:583-621)."""
    import yaml
    from neuralnj_b200 import rollout
    src = _phy_dir(tmp_path, ["t20x256_104"])
    cfg = {"instance_path": src, "env": {"batch_size": 1, "sequence_type": "DNA_WITH_GAP"},
           "model": {"vocab_size": 4, "patch_size": 1, "embed_dim": 64, "num_enc_heads": 8, "num_enc_layers": 6}}
    with open(tmp_path / "cfg.yaml", "w") as f:
        yaml.safe_dump(cfg, f)
    monkeypatch.chdir(tmp_path)
    torch.manual_seed(0)
    written = rollout.main(["--config_path", str(tmp_path / "cfg.yaml"), "--infer_opt", "Argmax"])
    assert written[0].startswith("output/Argmax_dim64_patch1/msas/")
    with open(written[0]) as f:
        assert f.read().strip() == golden("t20x256_104").newick[0]


def test_sharded_rollout_single_process(gpu_models):
    """shard.sharded_rollout without a process group (world 1) equals the plain fused rollout; the 2-rank form is a gloo CPU test."""
    import nnj_oracle as O
    from neuralnj_b200.shard import sharded_rollout
    data = O.evolved_msa(5, 10, 64, seed=9).cuda()
    mask = torch.zeros(5, 64, dtype=torch.bool).cuda()
    m = gpu_models["bf16x3"]
    assert torch.equal(sharded_rollout(m, data, mask), m.rollout_fused(data, mask)[0])
