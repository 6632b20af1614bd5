"""GPU: bootstrap branch support - nnj_bootstrap_columns and nnj_split_distances against the numpy / Python restatements of
oracle/support_oracle.py (bit for bit), and bootstrap_support end to end against the oracle rollout of the same replicates."""
import os
import shutil

import numpy as np
import pytest
import torch

import support_oracle as SO
from conftest import GOLD
from test_gpu_parity import TIE_TOL, _assert_equivalent_trajectory

pytestmark = pytest.mark.gpu


def _case(golden, name):
    g = golden(name)
    data, mask = g.data[0], g.mask[0]
    l_eff = int((~mask).sum())
    assert not bool(mask[:l_eff].any())
    return data, mask, l_eff


@pytest.mark.parametrize("name", ["ex50x1024_73", "padded_20x256"])
@pytest.mark.parametrize("rep0", [0, 2 ** 32 + 5])
def test_bootstrap_columns_match_restatement(name, rep0, golden):
    from neuralnj_b200 import support as SUP
    data, _, l_eff = _case(golden, name)
    seed = 0x1234_5678_9ABC_DEF0
    got = SUP.bootstrap_columns(data.cuda(), l_eff, seed, rep0, 6)
    assert torch.equal(got.cpu(), SO.bootstrap_columns(data, l_eff, seed, rep0, 6))
    # drawn two at a time: the same replicates
    parts = torch.cat([SUP.bootstrap_columns(data.cuda(), l_eff, seed, rep0 + k, 2) for k in range(0, 6, 2)])
    assert torch.equal(parts, got)


def _random_merges(rng, B, R):
    return np.array([[sorted(rng.choice(R - t, 2, replace=False)) for t in range(R - 1)] for _ in range(B)], dtype=np.int32)


def _multifurcating(R):
    """Taxa in groups of three under one root, plus a clade joining the first two groups: a non-binary tree."""
    names = [f"t{i}" for i in range(R)]
    groups = ["(" + ",".join(names[k:k + 3]) + ")" if len(names[k:k + 3]) > 1 else names[k] for k in range(0, R, 3)]
    if len(groups) > 3:
        groups = ["(" + groups[0] + "," + groups[1] + ")"] + groups[2:]
    return "(" + ",".join(groups) + ");", names


@pytest.mark.parametrize("R", [4, 5, 20, 63, 64, 65, 128, 200, 256, 512])
def test_split_distances_match_oracle(R):
    from neuralnj_b200 import support as SUP
    rng = np.random.default_rng(R)
    B = 6
    merges = _random_merges(rng, B + 1, R)
    clades = SO.clades_from_merges(merges[B], R)
    from_tree = sorted({min(c, (1 << R) - 1 - c) for c in clades if 2 <= bin(c).count("1") <= R - 2})
    sp_tree = [frozenset(i for i in range(R) if c >> i & 1) for c in from_tree]
    nw, names = _multifurcating(R)
    sp_multi, _ = SUP.reference_splits(nw, names)
    splits = SUP.split_bitsets(sp_tree + sp_multi, R)
    assert splits.shape[0] >= 1
    mg = torch.from_numpy(merges[:B])
    got = SUP.split_distances(mg.cuda(), splits.cuda()).cpu()
    assert torch.equal(got, SO.split_distances(mg, splits))
    assert bool((got >= 0).all())
    # corrupted merge rows: that row, and only that row, is -1
    bad = merges[:B].copy()
    bad[1, min(2, R - 2)] = (3, 3)
    bad[2, R - 2] = (0, 2)
    bad[4, 0] = (-1, 1)
    got_bad = SUP.split_distances(torch.from_numpy(bad).cuda(), splits.cuda()).cpu()
    assert torch.equal(got_bad[[1, 2, 4]], torch.full((3, splits.shape[0]), -1, dtype=torch.int32))
    assert torch.equal(got_bad[[0, 3, 5]], got[[0, 3, 5]])
    # no reference split: an empty result
    assert SUP.split_distances(mg.cuda(), splits[:0].cuda()).shape == (B, 0)


def test_split_distances_rejects_more_than_512_taxa():
    import ctypes as C
    from neuralnj_b200 import NnjError, lib
    from neuralnj_b200 import support as SUP
    R = 513
    merges = torch.from_numpy(_random_merges(np.random.default_rng(0), 1, R)).cuda()
    splits = SUP.split_bitsets([frozenset(range(5))], R).cuda()
    with pytest.raises(NnjError):
        SUP.split_distances(merges, splits)
    out = torch.empty(1, 1, dtype=torch.int32, device="cuda")
    assert lib().nnj_split_distances(C.c_void_p(merges.data_ptr()), 1, R, C.c_void_p(splits.data_ptr()), 1, C.c_void_p(out.data_ptr()),
                                     None) == -1


@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
def test_bootstrap_support_end_to_end(prec, golden, sd0, gpu_models, monkeypatch):
    """16 replicates of t20x256_10: each replicate tree is the oracle's rollout of the restated replicate, the supports are the
    oracle's on the device's own merge lists, and chunks of 3 give what chunks of 128 give."""
    import nnj_oracle as O
    from neuralnj_b200 import support as SUP
    model = gpu_models[prec]
    path = os.path.join(GOLD, "msa", "t20x256_10.phy")
    g = golden("t20x256_10")
    res = SUP.bootstrap_support(path, model, 16, seed=9)
    assert res["tree"] == g.newick[0]
    data, mask, l_eff = _case(golden, "t20x256_10")
    reps = SUP.bootstrap_columns(data.cuda(), l_eff, 9, 0, 16)
    masks = mask[None].expand(16, -1).contiguous()
    merges, _, trace = model.rollout_fused(reps, masks.cuda(), want_logits=True)
    merges, trace, reps = merges.cpu(), trace.cpu(), reps.cpu()
    assert torch.equal(reps, SO.bootstrap_columns(data, l_eff, 9, 0, 16))
    ref = O.rollout(sd0, reps, masks)
    if prec == "fp32" or torch.equal(merges.long(), ref["merges"]):
        assert torch.equal(merges.long(), ref["merges"])
    else:
        _assert_equivalent_trajectory(sd0, reps, masks, merges.long(), trace, TIE_TOL[prec])
    keys = g.seq_keys[0]
    want = SO.support_from_newicks(res["tree"], [O.newick_from_merges(m.tolist(), keys) for m in merges])
    assert set(res["splits"]) == set(want)
    for sp, f, t in zip(res["splits"], res["fbp"], res["tbe"]):
        assert (f, t) == want[sp]
    monkeypatch.setattr(SUP, "CHUNK", 3)
    other = SUP.bootstrap_support(path, model, 16, seed=9)
    assert np.array_equal(other["fbp"], res["fbp"]) and np.array_equal(other["tbe"], res["tbe"])
    assert other["newick_fbp"] == res["newick_fbp"] and other["newick_tbe"] == res["newick_tbe"]


def _root_child_labels(newick):
    """Labels after the `)` of the root's children."""
    out, depth = [], 0
    for k, ch in enumerate(newick):
        if ch == "(":
            depth += 1
        elif ch == ")":
            depth -= 1
            if depth == 1:
                end = k + 1
                while newick[end] not in ":,);":
                    end += 1
                out.append(newick[k + 1:end])
    return out


def test_directory_bootstrap_on_the_example_alignments(tmp_path, gpu_models):
    """ex50x1024_73 and _71 with 256 replicates through Argmax_inference(files_per_call=128, bootstrap=256): the .tre files are
    those of a run without bootstrap, supports lie in range, the root children carry one label, the labels strip off again."""
    from neuralnj_b200 import Argmax_inference, inference_config
    from neuralnj_b200 import support as SUP
    src = tmp_path / "msas"
    src.mkdir()
    names = ["ex50x1024_73", "ex50x1024_71"]
    for n in names:
        shutil.copyfile(os.path.join(GOLD, "msa", n + ".phy"), src / (n + ".phy"))
    model = gpu_models["bf16x3"]
    kw = dict(cfgs=inference_config(), device=torch.device("cuda:0"), files_per_call=128, policy_network=model)
    Argmax_inference(str(src), str(tmp_path / "plain"), None, **kw)
    Argmax_inference(str(src), str(tmp_path / "boot"), None, bootstrap=256, bootstrap_seed=1, **kw)
    res = SUP.bootstrap_support(str(src / "ex50x1024_73.phy"), model, 256, seed=1)
    assert len(res["splits"]) == 47
    assert bool(((res["fbp"] >= 0) & (res["fbp"] <= 100)).all()) and bool(((res["tbe"] >= 0) & (res["tbe"] <= 1)).all())
    assert bool((res["tbe"] >= res["fbp"] / 100 - 1e-12).all())         # an exact match is a transfer distance of 0
    for n in names:
        tre = (tmp_path / "plain" / (n + ".tre")).read_text()
        assert (tmp_path / "boot" / (n + ".tre")).read_text() == tre
        for kind in ("fbp", "tbe"):
            labelled = (tmp_path / "boot" / f"{n}.{kind}.tre").read_text()
            assert SUP.strip_support_labels(labelled) == tre
            roots = _root_child_labels(labelled)
            assert len(roots) == 2 and roots[0] == roots[1] != ""      # both root children are internal in these two trees
    assert (tmp_path / "boot" / "ex50x1024_73.fbp.tre").read_text() == res["newick_fbp"]
    assert (tmp_path / "boot" / "ex50x1024_73.tbe.tre").read_text() == res["newick_tbe"]
