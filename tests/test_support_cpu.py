"""CPU: bootstrap branch support (neuralnj_b200.support) - the definitions restated by oracle/support_oracle.py, the Newick labels,
and the host driver `bootstrap_support` / `Argmax_inference(bootstrap=N)` with the device model and the two device primitives
replaced by CPU stand-ins (the oracle rollout and the numpy restatements; the product path has no such fallback)."""
import os
import shutil
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import support_oracle as SO
from conftest import GOLD
from test_entry_batched_cpu import OracleAgent

from neuralnj_b200 import support as SUP
from neuralnj_b200.treeutil import bipartitions

N_REP = 12


def test_philox_known_answers():
    """Random123's known-answer vectors of Philox4x32-10."""
    cases = [((0, 0, 0, 0), (0, 0), "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
             ((0xffffffff,) * 4, (0xffffffff,) * 2, "408f276d 41c83b0e a20bc7c6 6d5451fd"),
             ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), "d16cfe09 94fdcceb 5001e420 24126ea1")]
    for ctr, key, want in cases:
        assert " ".join("%08x" % int(w) for w in SO.philox4x32_10(ctr, key)) == want


def _golden_batch(name):
    z = np.load(os.path.join(GOLD, name + ".npz"))
    R, L = z["data"].shape[1:3]
    keys = [[str(k) for k in z["seq_keys"][0]]]
    return {"data": torch.from_numpy(z["data"][:1]), "seq_weights": (~torch.from_numpy(z["seq_mask"][:1])).float(),
            "seqs": [["A" * L] * R], "seq_keys": keys}, str(z["newick"][0])


def test_resampling_draws_real_columns_and_keeps_the_padding():
    batch, _ = _golden_batch("padded_20x256")
    data = batch["data"][0]
    assert int(batch["seq_weights"][0].sum()) == 200 and bool((batch["seq_weights"][0][:200] == 1).all())
    src = SO.source_columns(200, 7, np.arange(2 ** 32 - 2, 2 ** 32 + 3, dtype=np.uint64))
    assert src.min() >= 0 and src.max() < 200
    assert len({tuple(r) for r in src}) == len(src)                      # replicates differ, across the 2^32 boundary too
    reps = SO.bootstrap_columns(data, 200, 7, 2 ** 32 - 2, 5)
    assert torch.equal(reps[:, :, 200:], data[None, :, 200:].expand(5, -1, -1, -1))
    for b in range(5):
        assert torch.equal(reps[b, :, :200], data[:, torch.from_numpy(src[b])])
    # a replicate depends on (seed, index, l_eff) only: drawing it inside another range gives the same columns
    assert torch.equal(SO.bootstrap_columns(data, 200, 7, 2 ** 32, 1)[0], reps[2])
    assert not torch.equal(SO.bootstrap_columns(data, 200, 8, 2 ** 32, 1)[0], reps[2])


def _merges_of(joins, R):
    """Merge list (slot indices) of a sequence of joins given as node ids (leaves 0..R-1, join k = node R+k)."""
    slots, out = list(range(R)), []
    for k, (a, b) in enumerate(joins):
        i, j = sorted((slots.index(a), slots.index(b)))
        out.append((i, j))
        slots[i] = R + k
        del slots[j]
    return np.array(out, dtype=np.int32)


def test_transfer_distance_by_hand():
    """R = 6, reference split {0,1,2}; replicate (((0,1),3),(2,(4,5))): the nearest clade {0,1} is one move away."""
    R = 6
    mg = _merges_of([(0, 1), (4, 5), (6, 3), (2, 7), (8, 9)], R)
    A = torch.tensor([[0b000111]], dtype=torch.int64)
    assert SO.split_distances(torch.from_numpy(mg)[None], A).tolist() == [[1]]
    sup = SO.support_from_newicks("((t0, t1), t2, ((t3, t4), t5));", ["(((t0, t1), t3), (t2, (t4, t5)));"])
    assert sup[frozenset(["t0", "t1", "t2"])] == (0.0, 0.5)
    # a merge entry outside i < j < R - t poisons the whole row
    bad = mg.copy()
    bad[3] = (1, 1)
    assert SO.split_distances(torch.from_numpy(np.stack([mg, bad])), A).tolist() == [[1], [-1]]


def test_newick_labels_and_stripping():
    keys = ["a", "b", "c", "d", "e"]
    nw = "((a:0.1, b:0.2):0.3, (c:0.1, (d:0.1, e:0.1):0.2):0.3);"
    splits, labelled = SUP.reference_splits(nw, keys)
    # the root children {a,b} and {c,d,e} are one split, labelled twice; {d,e} is the other
    assert [sorted(keys[i] for i in s) for s in splits] == [["a", "b"], ["d", "e"]]
    got = SUP.label_newick(nw, labelled, ["75", "100"])
    assert got == "((a:0.1, b:0.2)75:0.3, (c:0.1, (d:0.1, e:0.1)100:0.2)75:0.3);"
    assert SUP.strip_support_labels(got) == nw
    tbe = SUP.label_newick(nw, labelled, ["0.500", "1.000"])
    assert SUP.strip_support_labels(tbe) == nw
    # a multifurcating user tree without lengths: the trivial clade {a} and the root carry nothing
    user = "(a,(b,c,d),e);"
    s2, l2 = SUP.reference_splits(user, keys)
    assert [sorted(keys[i] for i in s) for s in s2] == [["a", "e"]] and SUP.label_newick(user, l2, ["9"]) == "(a,(b,c,d)9,e);"
    with pytest.raises(ValueError):
        SUP.reference_splits("((a,b)90,(c,(d,e)));", keys)                 # already labelled
    with pytest.raises(ValueError):
        SUP.reference_splits("((a,b),(c,(d,x)));", keys)                   # unknown taxon


class CachedOracleAgent(OracleAgent):
    """The oracle stand-in, memoised per alignment: the same replicate rolled out twice (another chunk size) costs nothing.
    `batches` records the batch size of every call."""
    cache = {}

    def __init__(self):
        super().__init__()
        self.batches = []

    def rollout_fused(self, data, mask, gumbel=None, want_logits=False):
        self.batches.append(data.shape[0])
        if want_logits:                   # the tree-writing call of Argmax_inference: not cached
            return super().rollout_fused(data, mask, gumbel, want_logits)
        out = []
        for b in range(data.shape[0]):
            key = (data[b].numpy().tobytes(), mask[b].numpy().tobytes())
            if key not in self.cache:
                self.cache[key] = self.O.rollout(self.sd, data[b:b + 1], mask[b:b + 1])["merges"].to(torch.int32)
            out.append(self.cache[key])
        mg = torch.cat(out)
        return mg, torch.zeros(mg.shape[0], mg.shape[1]), None


@pytest.fixture
def cpu_primitives(monkeypatch):
    monkeypatch.setattr(SUP, "bootstrap_columns", SO.bootstrap_columns)
    monkeypatch.setattr(SUP, "split_distances", SO.split_distances)


@pytest.mark.parametrize("name", ["t20x256_10", "padded_20x256"])
def test_bootstrap_support_pipeline_matches_oracle(name, cpu_primitives, monkeypatch):
    import nnj_oracle as O
    batch, gold_newick = _golden_batch(name)
    msa = os.path.join(GOLD, "msa", name + ".phy") if os.path.exists(os.path.join(GOLD, "msa", name + ".phy")) else batch
    agent = CachedOracleAgent()
    res = SUP.bootstrap_support(msa, agent, N_REP, seed=3)
    assert res["tree"] == gold_newick and res["n_replicates"] == N_REP and res["seed"] == 3
    assert set(res["splits"]) == bipartitions(gold_newick)
    # the oracle: support recomputed with Python sets from the Newick strings of the same replicate trees
    keys = batch["seq_keys"][0]
    l_eff = int(batch["seq_weights"][0].sum())
    reps = SO.bootstrap_columns(batch["data"][0], l_eff, 3, 0, N_REP)
    mask = (batch["seq_weights"] == 0).expand(N_REP, -1)
    merges = agent.rollout_fused(reps, mask)[0]
    want = SO.support_from_newicks(gold_newick, [O.newick_from_merges(m.tolist(), keys) for m in merges])
    for sp, f, t in zip(res["splits"], res["fbp"], res["tbe"]):
        assert (f, t) == want[sp]
    assert SUP.strip_support_labels(res["newick_fbp"]) == gold_newick == SUP.strip_support_labels(res["newick_tbe"])
    # chunk size cannot change a result
    for chunk in (5, 128):
        monkeypatch.setattr(SUP, "CHUNK", chunk)
        agent.batches.clear()
        other = SUP.bootstrap_support(msa, agent, N_REP, seed=3)
        assert agent.batches[1:] == [min(chunk, N_REP - r0) for r0 in range(0, N_REP, chunk)]
        assert other["newick_fbp"] == res["newick_fbp"] and other["newick_tbe"] == res["newick_tbe"]
        assert np.array_equal(other["fbp"], res["fbp"]) and np.array_equal(other["tbe"], res["tbe"])


class FixedAgent(torch.nn.Module):
    """Returns the same merge list for every alignment."""

    def __init__(self, merges):
        super().__init__()
        self.merges = torch.as_tensor(merges, dtype=torch.int32)
        self.anchor = torch.nn.Parameter(torch.zeros(1))

    def rollout_fused(self, data, mask, gumbel=None, want_logits=False):
        B = data.shape[0]
        return self.merges[None].expand(B, -1, -1).clone(), torch.zeros(B, self.merges.shape[0]), None


def test_identical_replicates_give_full_support(cpu_primitives):
    batch, _ = _golden_batch("t20x256_10")
    R = batch["data"].shape[1]
    rng = np.random.default_rng(1)
    mg = np.array([sorted(rng.choice(R - t, 2, replace=False)) for t in range(R - 1)], dtype=np.int32)
    res = SUP.bootstrap_support(batch, FixedAgent(mg), 7)
    assert len(res["splits"]) == R - 3
    assert (res["fbp"] == 100.0).all() and (res["tbe"] == 1.0).all()
    _, labelled = SUP.reference_splits(res["tree"], batch["seq_keys"][0])
    assert res["newick_fbp"].count(")100:") == res["newick_tbe"].count(")1.000:") == len(labelled) >= R - 3
    # a user tree without non-trivial splits (a star) comes back unlabelled
    star = "(" + ", ".join(batch["seq_keys"][0]) + ");"
    assert SUP.bootstrap_support(batch, FixedAgent(mg), 7, tree=star)["newick_fbp"] == star


class CountingFixedAgent(FixedAgent):
    """FixedAgent that records the batch size of every rollout call."""

    def __init__(self, merges):
        super().__init__(merges)
        self.batches = []

    def rollout_fused(self, data, mask, gumbel=None, want_logits=False):
        self.batches.append(data.shape[0])
        return super().rollout_fused(data, mask, gumbel, want_logits)


def _random_batch(R, L, seed):
    rng = np.random.default_rng(seed)
    data = torch.from_numpy(np.eye(4, dtype=np.int8)[rng.integers(0, 4, (1, R, L))])
    keys = [f"t{i}" for i in range(R)]
    mg = np.array([sorted(rng.choice(R - t, 2, replace=False)) for t in range(R - 1)], dtype=np.int32)
    return {"data": data, "seq_weights": torch.ones(1, L), "seqs": [["A" * L] * R], "seq_keys": [keys]}, mg


def test_more_than_400_taxa_raise_before_any_rollout(cpu_primitives):
    """Every replicate is an Argmax rollout, and the encoder's column attention stops at 400 taxa: 401 taxa are refused before the
    first rollout (the reference tree's, or the first replicate's when a tree is given), 400 taxa are accepted."""
    batch, mg = _random_batch(401, 16, 0)
    agent = CountingFixedAgent(mg)
    with pytest.raises(ValueError, match="at most 400"):
        SUP.bootstrap_support(batch, agent, 3)
    tree = "(" + ", ".join(f"({a}, {b})" for a, b in zip(batch["seq_keys"][0][0:400:2], batch["seq_keys"][0][1:400:2])) + ", t400);"
    with pytest.raises(ValueError, match="at most 400"):
        SUP.bootstrap_support(batch, agent, 3, tree=tree)
    assert agent.batches == []
    batch, mg = _random_batch(400, 16, 1)
    agent = CountingFixedAgent(mg)
    res = SUP.bootstrap_support(batch, agent, 2)
    assert agent.batches == [1, 2] and len(res["splits"]) == 397
    assert (res["fbp"] == 100.0).all() and (res["tbe"] == 1.0).all()


def test_invalid_merges_and_padding_raise(cpu_primitives):
    from neuralnj_b200 import NnjError
    batch, _ = _golden_batch("t20x256_10")
    R = batch["data"].shape[1]
    mg = np.array([(0, 1)] * (R - 1), dtype=np.int32)
    mg[4] = (3, 3)
    tree = "(" + ", ".join(f"({a}, {b})" for a, b in zip(batch["seq_keys"][0][0::2], batch["seq_keys"][0][1::2])) + ");"
    with pytest.raises(NnjError, match="not valid"):
        SUP.bootstrap_support(batch, FixedAgent(mg), 3, tree=tree)
    holey = dict(batch, seq_weights=batch["seq_weights"].clone())
    holey["seq_weights"][0, 10] = 0
    with pytest.raises(NnjError, match="prefix"):
        SUP.bootstrap_support(holey, FixedAgent(mg), 3, tree=tree)


DIR_NAMES = ["t20x256_10", "t20x256_103", "t20x256_104"]
DIR_REPS = 4


def _phy_dir(path):
    os.makedirs(path)
    for n in DIR_NAMES:
        shutil.copyfile(os.path.join(GOLD, "msa", n + ".phy"), os.path.join(path, n + ".phy"))
    return path


def _read(path):
    with open(path) as f:
        return f.read()


def _worker(rank, world, port, src, out_dir, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import conftest  # noqa: F401  (puts oracle/ on sys.path in the spawned process)
    import support_oracle as SO2
    from neuralnj_b200 import Argmax_inference, inference_config
    from neuralnj_b200 import support as S2
    S2.bootstrap_columns, S2.split_distances = SO2.bootstrap_columns, SO2.split_distances
    S2.CHUNK = 4
    res = S2.bootstrap_support(os.path.join(src, "t20x256_10.phy"), OracleAgent(), 9, seed=11)
    agent = OracleAgent()
    Argmax_inference(src, out_dir, None, cfgs=inference_config(), device=torch.device("cpu"), files_per_call=8, policy_network=agent,
                     bootstrap=DIR_REPS, bootstrap_seed=5)
    q.put((rank, res["newick_fbp"], res["newick_tbe"], res["fbp"].tolist(), res["tbe"].tolist(), [c[0] for c in agent.calls]))
    dist.barrier()
    dist.destroy_process_group()


def test_two_ranks_equal_one(tmp_path, cpu_primitives):
    """Replicate sharding of one alignment (one all_reduce) and Argmax_inference(bootstrap=N) over a directory (file sharding, no
    replicate sharding) give under two gloo ranks what one process gives."""
    from neuralnj_b200 import Argmax_inference, inference_config
    src = _phy_dir(str(tmp_path / "msas"))
    one = SUP.bootstrap_support(os.path.join(src, "t20x256_10.phy"), CachedOracleAgent(), 9, seed=11)
    Argmax_inference(src, str(tmp_path / "out1"), None, cfgs=inference_config(), device=torch.device("cpu"), files_per_call=8,
                     policy_network=CachedOracleAgent(), bootstrap=DIR_REPS, bootstrap_seed=5)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, src, str(tmp_path / "out2"), q)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict((g[0], g[1:]) for g in (q.get(timeout=600) for _ in range(2)))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for r in range(2):
        assert got[r][:4] == (one["newick_fbp"], one["newick_tbe"], one["fbp"].tolist(), one["tbe"].tolist())
    # rank 0 owns two files, rank 1 one: one batched call for the trees, then one chunk of DIR_REPS replicates per file
    assert got[0][4] == [2, 4, 4] and got[1][4] == [1, 4]
    for n in DIR_NAMES:
        for ext in (".tre", ".fbp.tre", ".tbe.tre"):
            assert _read(tmp_path / "out2" / (n + ext)) == _read(tmp_path / "out1" / (n + ext)), n + ext
        tre = _read(tmp_path / "out1" / (n + ".tre"))
        assert SUP.strip_support_labels(_read(tmp_path / "out1" / (n + ".fbp.tre"))) == tre
        assert SUP.strip_support_labels(_read(tmp_path / "out1" / (n + ".tbe.tre"))) == tre
