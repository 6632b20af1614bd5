"""Generate tests/golden/ by executing the UNMODIFIED reference (build container only).

    python oracle/make_golden.py            # writes tests/golden/*.npz + tests/golden/msa/*.phy
    python oracle/make_golden.py supervise  # teacher-forced rollouts + pre-training loss (tests/golden/supervise/, see main_supervise)
    python oracle/make_golden.py all50      # all 128 files of data_gen/data/test/len1024/taxa50 in one record (tests/golden/all50/)
    python oracle/make_golden.py wide       # round 2: 16 files of data_gen/data/test/len1024/taxa50 + 4 of len1024/taxa100
                                            #          as "lite" records under tests/golden/wide/ (see main_wide)

The reference (/root/reference, read-only, absent on the GPU box) is imported
with the stub packages under oracle/ref_stubs/ standing in for its missing
third-party imports (raxmlpy native binding, fvcore, ete3, dendropy, Bio).
For every case it drives the reference's own `reinforce_rollout(eval=True,
argmax=True, branch_optimize=False)` (finetune_rl_search.py:78-189) with
`torch.manual_seed(0)` default-initialised weights (the shipped checkpoint is a
missing blob, SURVEY.md F1) and records what the reference computed:
the merge list, the logits of every step, selected_log_ps, the Newick string and
a strided sample of the encoder output.  It then checks oracle/nnj_oracle.py
against those records and prints the deviations.  Nothing from here is used at
run time by the product.
"""
import hashlib
import os
import shutil
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
REF = os.environ.get("NNJ_REFERENCE", "/root/reference")
GOLD = os.path.join(REPO, "tests", "golden")

sys.path.insert(0, os.path.join(HERE, "ref_stubs"))
sys.path.insert(0, REF)
sys.path.insert(0, HERE)

import nnj_oracle as O  # noqa: E402

CASES = [
    # (case name, path relative to the reference)
    ("ex50x1024_73", "examples/len1024taxa50/G_l_1024_n_50_0_0.03_73.phy"),
    ("ex50x1024_71", "examples/len1024taxa50/G_l_1024_n_50_0_0.02_71.phy"),
    ("t20x256_10", "data_gen/data/test/len256/taxa20/G_l_256_n_20_0_0.01_10.phy"),
    ("t20x256_103", "data_gen/data/test/len256/taxa20/G_l_256_n_20_0_0.01_103.phy"),
    ("t20x256_104", "data_gen/data/test/len256/taxa20/G_l_256_n_20_0_0.01_104.phy"),
    ("t20x256_117", "data_gen/data/test/len256/taxa20/G_l_256_n_20_0_0.01_117.phy"),
    ("t20x256_120", "data_gen/data/test/len256/taxa20/G_l_256_n_20_0_0.01_120.phy"),
]


def _pick(dirpath, k):
    fs = sorted(f for f in os.listdir(os.path.join(REF, dirpath)) if f.endswith(".phy"))
    return os.path.join(dirpath, fs[k])


def main():
    torch.set_num_threads(8)
    import utils as ref_utils
    import finetune_rl_search as ref_main
    from environment import PhyInferEnv
    from model import PhyloATTN
    from phydata import load_pi_instance

    torch.autograd.set_detect_anomaly(False)  # finetune_rl_search.py:33 turns it on globally; irrelevant under no_grad
    cfgs = ref_utils.empty_config()
    cfgs.merge_from_file(os.path.join(REF, "config/finetune_reinforce_search_example.yaml"))
    ref_main.cfgs = cfgs
    ref_main.device = torch.device("cpu")

    cases = list(CASES)
    cases.append(("t50x256_a", _pick("data_gen/data/test/len256/taxa50", 3)))
    cases.append(("t100x256_a", _pick("data_gen/data/test/len256/taxa100", 5)))
    cases.append(("t20x512_a", _pick("data_gen/data/test/len512/taxa20", 7)))
    cases.append(("t50x512_a", _pick("data_gen/data/test/len512/taxa50", 11)))

    os.makedirs(os.path.join(GOLD, "msa"), exist_ok=True)

    torch.manual_seed(0)
    model = PhyloATTN(cfgs).eval()
    sd_ref = {k: v.detach().clone() for k, v in model.state_dict().items()}
    sd = O.init_state_dict(0)
    assert list(sd.keys()) == list(sd_ref.keys()), "state_dict key order differs"
    for k in sd:
        assert torch.equal(sd[k], sd_ref[k]), f"seed-0 init differs at {k}"
    h = hashlib.sha256()
    for k in sd_ref:
        h.update(sd_ref[k].numpy().tobytes())
    with open(os.path.join(GOLD, "weights_seed0.sha256"), "w") as f:
        f.write(h.hexdigest() + "\n")
    np.savez_compressed(os.path.join(GOLD, "weights_seed0_sample.npz"),
                        **{k.replace(".", "__"): v.numpy().ravel()[:8] for k, v in sd_ref.items()})
    print("weights: oracle init == reference init, sha256", h.hexdigest()[:16])

    def run_reference(batch):
        """Drive the reference rollout, recording logits / actions through its own call sites."""
        env = PhyInferEnv(cfgs, torch.device("cpu"))
        rec = {"logits": [], "merges": [], "state0": None}
        orig_dec, orig_enc, orig_step = model.decode_zxr, model.encode_zxr, env.step

        def enc(*a, **k):
            out = orig_enc(*a, **k)
            rec["state0"] = out.detach().clone()
            return out

        def dec(*a, **k):
            out = orig_dec(*a, **k)
            rec["logits"].append(out["logits"].detach().clone())
            return out

        def step(actions, *a, **k):
            n = env.states[0].num_trees
            rec["merges"].append([list(map(int, env.tree_pairs_dict[n][int(x)])) for x in actions])
            return orig_step(actions, *a, **k)

        model.decode_zxr, model.encode_zxr, env.step = dec, enc, step
        try:
            t = time.time()
            sel, log_ps, scores, best = ref_main.reinforce_rollout(
                batch, model, env, cfgs, eval=True, argmax=True, branch_optimize=False)
            dt = time.time() - t
        finally:
            del model.decode_zxr, model.encode_zxr
        newicks = [s.subtrees[0].utree_op_str for s in env.states]
        return rec, sel, newicks, dt

    def save_case(name, batch, rec, sel, newicks, extra=None):
        B = batch["data"].shape[0]
        merges = np.array(rec["merges"], dtype=np.int32).transpose(1, 0, 2)  # [B,R-1,2]
        logits = [l.numpy() for l in rec["logits"]]
        offs = np.cumsum([0] + [l.shape[1] for l in logits]).astype(np.int64)
        st = rec["state0"]
        out = dict(
            data=batch["data"].numpy().astype(np.int8),
            seq_mask=(batch["seq_weights"] == 0).numpy(),
            merges=merges,
            logits=np.concatenate(logits, 1).astype(np.float32),
            logit_offsets=offs,
            selected_log_ps=sel.numpy().astype(np.float32),
            state_sample=st[:, ::7, ::37, :].numpy().astype(np.float32),
            state_abs_mean=np.array([float(st.abs().mean())], dtype=np.float64),
            newick=np.array(newicks),
            seq_keys=np.array(batch["seq_keys"]),
        )
        if extra:
            out.update(extra)
        np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)

    def check_oracle(name, batch, rec, sel, newicks):
        data = batch["data"]
        mask = batch["seq_weights"] == 0
        t = time.time()
        r = O.rollout(sd, data, mask)
        dt = time.time() - t
        gm = torch.tensor(np.array(rec["merges"]).transpose(1, 0, 2))
        same = bool(torch.equal(r["merges"], gm))
        dl = max(float((a - b).abs().max() / b.abs().max()) for a, b in zip(r["logits"], rec["logits"]))
        ds = float((r["state0"] - rec["state0"]).abs().max())
        nw = [O.newick_from_merges([tuple(m) for m in r["merges"][b].tolist()], batch["seq_keys"][b])
              for b in range(data.shape[0])]
        print(f"  oracle vs reference [{name}]: merges identical={same} max rel dlogit={dl:.2e} "
              f"max |dstate|={ds:.2e} newick identical={nw == list(newicks)} ({dt:.1f}s)")
        assert same and nw == list(newicks) and dl < 1e-5

    for name, rel in cases:
        src = os.path.join(REF, rel)
        dst = os.path.join(GOLD, "msa", name + ".phy")
        shutil.copyfile(src, dst)
        batch = load_pi_instance(src)
        # the oracle's own PHYLIP reader must agree with the reference loader
        d2, m2, keys2, _ = O.load_phy(dst)
        assert torch.equal(d2, batch["data"]) and keys2 == batch["seq_keys"][0], name
        rec, sel, newicks, dt = run_reference(batch)
        print(f"[{name}] reference rollout {dt:.1f}s  data {tuple(batch['data'].shape)}")
        save_case(name, batch, rec, sel, newicks)
        check_oracle(name, batch, rec, sel, newicks)

    # batch of two different MSAs of one shape (B>1 semantics), and a padded-column case
    b1 = load_pi_instance(os.path.join(REF, CASES[2][1]))
    b2 = load_pi_instance(os.path.join(REF, CASES[3][1]))
    both = {"data": torch.cat([b1["data"], b2["data"]]), "seq_weights": torch.cat([b1["seq_weights"], b2["seq_weights"]]),
            "seqs": b1["seqs"] + b2["seqs"], "seq_keys": b1["seq_keys"] + b2["seq_keys"]}
    rec, sel, newicks, dt = run_reference(both)
    print(f"[batch2_20x256] reference rollout {dt:.1f}s")
    save_case("batch2_20x256", both, rec, sel, newicks)
    check_oracle("batch2_20x256", both, rec, sel, newicks)

    pad = {k: (v.clone() if torch.is_tensor(v) else list(v)) for k, v in b1.items() if k in ("data", "seq_weights", "seqs", "seq_keys")}
    pad["data"][:, :, 200:, :] = 0          # '*' padding columns (phydata.py:45)
    pad["seq_weights"][:, 200:] = 0
    rec, sel, newicks, dt = run_reference(pad)
    print(f"[padded_20x256] reference rollout {dt:.1f}s")
    save_case("padded_20x256", pad, rec, sel, newicks)
    check_oracle("padded_20x256", pad, rec, sel, newicks)

    # tiny cases: 3, 4 and 5 taxa (R'>2 gate, last-step path), random tokens
    for R, L, seed in ((3, 64, 11), (4, 96, 12), (5, 128, 13)):
        data = O.evolved_msa(1, R, L, seed=seed)
        keys = [[f"taxon{i + 1}" for i in range(R)]]
        tiny = {"data": data, "seq_weights": torch.ones(1, L), "seqs": [["A" * L] * R], "seq_keys": keys}
        rec, sel, newicks, dt = run_reference(tiny)
        nm = f"tiny_{R}x{L}"
        save_case(nm, tiny, rec, sel, newicks)
        check_oracle(nm, tiny, rec, sel, newicks)

    # closed-form cache index map against the reference's table-driven one (utils.py:213-251)
    env = PhyInferEnv(cfgs, torch.device("cpu"))
    env.init_states([["A"] * 12], [[f"t{i}" for i in range(12)]], None)
    for n_new in range(2, 12):
        for (a, b) in env.tree_pairs_dict[n_new + 1]:
            ref_idx = ref_utils.get_score_indices_to_prev(torch.tensor([[a, b]]), env, n_new, 1)[0]
            assert [int(x) for x in ref_idx] == O.score_indices_to_prev(int(a), int(b), n_new)
    print("cache index map: closed form == reference for n<=12")


def main_wide():
    """Breadth set (VERDICT r1 item 1b): every 8th file of data_gen/data/test/len1024/taxa50 (16 files) and every 32nd of
    len1024/taxa100 (4 files), run through the unmodified reference.  To keep the fixtures small a "lite" record holds what
    topology parity needs - merge list, Newick, selected_log_ps, the step-0 logits, and per step the maximum |logit| and the
    top-1 / top-2 gap - while the input travels as the .phy file itself (read back through neuralnj_b200.load_pi_instance)."""
    torch.set_num_threads(8)
    import utils as ref_utils
    import finetune_rl_search as ref_main
    from environment import PhyInferEnv
    from model import PhyloATTN
    from phydata import load_pi_instance

    torch.autograd.set_detect_anomaly(False)
    cfgs = ref_utils.empty_config()
    cfgs.merge_from_file(os.path.join(REF, "config/finetune_reinforce_search_example.yaml"))
    ref_main.cfgs = cfgs
    ref_main.device = torch.device("cpu")
    torch.manual_seed(0)
    model = PhyloATTN(cfgs).eval()
    sd = O.init_state_dict(0)
    for k, v in model.state_dict().items():
        assert torch.equal(sd[k], v), k
    out_dir = os.path.join(GOLD, "wide")
    os.makedirs(out_dir, exist_ok=True)
    sets = [("w50", "data_gen/data/test/len1024/taxa50", 8), ("w100", "data_gen/data/test/len1024/taxa100", 32)]
    index = []
    for tag, d, stride in sets:
        files = sorted(f for f in os.listdir(os.path.join(REF, d)) if f.endswith(".phy"))[::stride]
        for k, fn in enumerate(files):
            name = f"{tag}_{k:02d}"
            src = os.path.join(REF, d, fn)
            shutil.copyfile(src, os.path.join(out_dir, name + ".phy"))
            batch = load_pi_instance(src)
            env = PhyInferEnv(cfgs, torch.device("cpu"))
            rec = {"logits": [], "merges": []}
            orig_dec, orig_step = model.decode_zxr, env.step

            def dec(*a, **kw):
                o = orig_dec(*a, **kw)
                rec["logits"].append(o["logits"].detach().clone())
                return o

            def step(actions, *a, **kw):
                n = env.states[0].num_trees
                rec["merges"].append([list(map(int, env.tree_pairs_dict[n][int(x)])) for x in actions])
                return orig_step(actions, *a, **kw)

            model.decode_zxr, env.step = dec, step
            try:
                t = time.time()
                sel, _, _, _ = ref_main.reinforce_rollout(batch, model, env, cfgs, eval=True, argmax=True, branch_optimize=False)
                dt = time.time() - t
            finally:
                del model.decode_zxr
            newick = env.states[0].subtrees[0].utree_op_str
            lmax, gap = [], []
            for lg in rec["logits"]:
                lmax.append(float(lg.abs().max()))
                gap.append(float(lg.topk(2, dim=1).values.diff(dim=1).abs().max()) if lg.shape[1] > 1 else float("inf"))
            np.savez_compressed(os.path.join(out_dir, name + ".npz"),
                                source=np.array(os.path.join(d, fn)),
                                merges=np.array(rec["merges"], dtype=np.int32).transpose(1, 0, 2),
                                newick=np.array([newick]), selected_log_ps=sel.numpy().astype(np.float32),
                                logits0=rec["logits"][0].numpy().astype(np.float32),
                                step_max_abs_logit=np.array(lmax, dtype=np.float32), step_top2_gap=np.array(gap, dtype=np.float32))
            rel_gap = min(g / m for g, m in zip(gap, lmax) if np.isfinite(g))
            print(f"[{name}] {fn}: reference rollout {dt:.1f}s, min relative top-2 gap {rel_gap:.2e}", flush=True)
            index.append(name)
    with open(os.path.join(out_dir, "INDEX.txt"), "w") as f:
        f.write("\n".join(index) + "\n")


def main_supervise():
    """Row f3, forward half (SURVEY.md 8): teacher-forced rollouts and the pre-training loss, executed by the unmodified reference.

    For each case: the label tree next to the alignment is read by the reference's own `phydata.load_tree_file` (on the Bio.Phylo
    stand-in of oracle/ref_stubs), a bottom-up trajectory and its per-step action sets come from `sample_trajectory_set_bottom_top`
    (phydata.py:779-834) under a recorded `random.seed`, `train.supervise_rollout(eval=True, pretrained=True)` (train.py:43-161)
    supplies the per-step logits, and the loss is computed by EXECUTING the reference's own statements (train.py, from
    "Policy_loss = 0" to "policy_loss = Policy_loss/len(logitss)", read from the source file at generation time - nothing of it is
    stored in this repository) for two epochs of the K-ratio schedule.  Records go to tests/golden/supervise/."""
    import random
    import textwrap
    torch.set_num_threads(8)
    import utils as ref_utils
    import phydata as ref_phy
    import train as ref_train
    from environment import PhyInferEnv
    from model import PhyloATTN
    import torch.nn.functional as F

    torch.autograd.set_detect_anomaly(False)
    cfgs = ref_utils.empty_config()
    cfgs.merge_from_file(os.path.join(REF, "config/pretrain_mix.yaml"))
    ref_train.device = torch.device("cpu")
    torch.manual_seed(0)
    model = PhyloATTN(cfgs).eval()
    sd = O.init_state_dict(0)
    for k, v in model.state_dict().items():
        assert torch.equal(sd[k], v), k

    src_lines = open(os.path.join(REF, "train.py")).read().split("\n")
    lo = next(i for i, l in enumerate(src_lines) if l.strip() == "Policy_loss = 0")
    hi = next(i for i, l in enumerate(src_lines) if l.strip() == "policy_loss = Policy_loss/len(logitss)")
    loss_src = textwrap.dedent("\n".join(src_lines[lo:hi + 1]))

    def reference_loss(ret, epoch):
        logitss, _, set_masks, sets, comp_masks, comps, _ = ret
        ns = dict(torch=torch, F=F, os=os, cfgs=cfgs, epoch=epoch, BALANCED_ELU_LOSS=cfgs.loss.BALANCED_ELU_LOSS,
                  ELU_LOSS=cfgs.loss.ELU_LOSS, logitss=[l.clone() for l in logitss], actions_set_masks=set_masks, actions_sets=sets,
                  actions_set_complement_masks=comp_masks, actions_sets_complement=comps)
        exec(loss_src, ns)
        return float(ns["policy_loss"]), float(ns["precision"])

    out_dir = os.path.join(GOLD, "supervise")
    os.makedirs(out_dir, exist_ok=True)
    t20 = "data_gen/data/test/len256/taxa20/"
    cases = [
        ("sup_20x256_b2", [t20 + "G_l_256_n_20_0_0.01_10", t20 + "G_l_256_n_20_0_0.01_103"], 5),
        ("sup_50x256", [_pick("data_gen/data/test/len256/taxa50", 3)[:-4]], 6),
        ("sup_50x1024", ["examples/len1024taxa50/G_l_1024_n_50_0_0.03_73"], 7),
    ]
    for name, stems, seed in cases:
        items = []
        random.seed(seed)
        for stem in stems:
            b = ref_phy.load_pi_instance(os.path.join(REF, stem + ".phy"))
            tree = ref_phy.load_tree_file(os.path.join(REF, stem + ".tre"), None, pos=5)
            acts, sets = ref_phy.sample_trajectory_set_bottom_top(tree, pos=5)
            items.append((b, tree, acts, sets, open(os.path.join(REF, stem + ".tre")).read().strip()))
        batch = {
            "data": torch.cat([it[0]["data"] for it in items]),
            "seq_weights": torch.cat([it[0]["seq_weights"] for it in items]),
            "seqs": [it[0]["seqs"][0] for it in items],
            "seq_keys": [it[0]["seq_keys"][0] for it in items],
            "trees": [it[1] for it in items],
            "actions": torch.from_numpy(np.array([[it[2]] for it in items], dtype=np.int32)),
            "actions_set": [[it[3]] for it in items],
        }
        env = PhyInferEnv(cfgs, torch.device("cpu"))
        t = time.time()
        ret = ref_train.supervise_rollout(batch, model, env, eval=True, pretrained=True)
        dt = time.time() - t
        logitss, sets_list, _, _, _, _, sel = ret
        losses = {ep: reference_loss(ret, ep) for ep in (0, 30)}
        B, R = batch["data"].shape[:2]
        flat_sets = []          # per tree and step: pair indices of the action set, -1 padded
        width = max(len(s) for st in sets_list for s in st)
        set_idx = -np.ones((B, len(sets_list), width), dtype=np.int32)
        for st, step_sets in enumerate(sets_list):
            for bb, s in enumerate(step_sets):
                set_idx[bb, st, :len(s)] = s
        lg = [l.numpy() for l in logitss]
        offs = np.cumsum([0] + [l.shape[1] for l in lg]).astype(np.int64)
        np.savez_compressed(os.path.join(out_dir, name + ".npz"),
                            data=batch["data"].numpy().astype(np.int8), seq_mask=(batch["seq_weights"] == 0).numpy(),
                            seq_keys=np.array(batch["seq_keys"]), label_newick=np.array([it[4] for it in items]),
                            random_seed=np.array([seed]), actions=batch["actions"][:, 0].numpy().astype(np.int32),
                            action_set_pair_index=set_idx, logits=np.concatenate(lg, 1).astype(np.float32), logit_offsets=offs,
                            selected_log_ps=sel.numpy().astype(np.float32),
                            loss_epochs=np.array(sorted(losses)), loss=np.array([losses[e][0] for e in sorted(losses)]),
                            precision=np.array([losses[e][1] for e in sorted(losses)]),
                            ratio_factor=np.array([cfgs.ratio_factor]), margin=np.array([0.5]))
        # the oracle along the same forced trajectory
        r = O.rollout(sd, batch["data"], batch["seq_weights"] == 0, forced_merges=batch["actions"][:, 0].long())
        dl = max(float((a - b).abs().max() / b.abs().max()) for a, b in zip(r["logits"], logitss))
        print(f"[{name}] reference supervise_rollout {dt:.1f}s, steps {len(logitss)}, loss {losses}, oracle max rel dlogit {dl:.2e}", flush=True)
        assert dl < 1e-5


def main_all50(taxa=50, threads=8):
    """The whole of data_gen/data/test/len1024/taxa50 (128 alignments - the set SURVEY.md 8(d) names for configs[1]) through the
    unmodified reference: merge list, Newick, selected_log_ps and per-step max |logit| / top-2 gap of every file, in ONE record
    (tests/golden/all50/len1024_taxa50_part*.npz, 64 alignments per part) together with the inputs as bit-packed one-hot tokens
    (25.6 KB per alignment).  `all100` does the same for len1024/taxa100 (tests/golden/all100/)."""
    torch.set_num_threads(threads)
    import utils as ref_utils
    import finetune_rl_search as ref_main
    from environment import PhyInferEnv
    from model import PhyloATTN
    from phydata import load_pi_instance

    torch.autograd.set_detect_anomaly(False)
    cfgs = ref_utils.empty_config()
    cfgs.merge_from_file(os.path.join(REF, "config/finetune_reinforce_search_example.yaml"))
    ref_main.cfgs = cfgs
    ref_main.device = torch.device("cpu")
    torch.manual_seed(0)
    model = PhyloATTN(cfgs).eval()
    sd = O.init_state_dict(0)
    for k, v in model.state_dict().items():
        assert torch.equal(sd[k], v), k
    d = f"data_gen/data/test/len1024/taxa{taxa}"
    files = sorted(f for f in os.listdir(os.path.join(REF, d)) if f.endswith(".phy"))
    rec = {k: [] for k in ("bits", "keys", "merges", "newick", "slp", "lmax", "gap", "src")}
    for k, fn in enumerate(files):
        batch = load_pi_instance(os.path.join(REF, d, fn))
        env = PhyInferEnv(cfgs, torch.device("cpu"))
        got = {"logits": [], "merges": []}
        orig_dec, orig_step = model.decode_zxr, env.step

        def dec(*a, **kw):
            o = orig_dec(*a, **kw)
            got["logits"].append(o["logits"].detach().clone())
            return o

        def step(actions, *a, **kw):
            n = env.states[0].num_trees
            got["merges"].append([list(map(int, env.tree_pairs_dict[n][int(x)])) for x in actions])
            return orig_step(actions, *a, **kw)

        model.decode_zxr, env.step = dec, step
        try:
            t = time.time()
            sel, _, _, _ = ref_main.reinforce_rollout(batch, model, env, cfgs, eval=True, argmax=True, branch_optimize=False)
            dt = time.time() - t
        finally:
            del model.decode_zxr
        data = batch["data"].numpy().astype(np.uint8)
        assert data.max() <= 1 and (batch["seq_weights"] != 0).all()
        rec["bits"].append(np.packbits(data.reshape(-1)))
        rec["keys"].append(batch["seq_keys"][0])
        rec["merges"].append(np.array(got["merges"], dtype=np.int8)[:, 0])
        rec["newick"].append(env.states[0].subtrees[0].utree_op_str)
        rec["slp"].append(sel.numpy().astype(np.float32)[0])
        rec["lmax"].append([float(lg.abs().max()) for lg in got["logits"]])
        rec["gap"].append([float(lg.topk(2, dim=1).values.diff(dim=1).abs().max()) if lg.shape[1] > 1 else np.inf for lg in got["logits"]])
        rec["src"].append(fn)
        rel = min(g / m for g, m in zip(rec["gap"][-1], rec["lmax"][-1]) if np.isfinite(g))
        print(f"[{k:3d}] {fn}: reference rollout {dt:.1f}s, min relative top-2 gap {rel:.2e}", flush=True)
    out_dir = os.path.join(GOLD, f"all{taxa}")
    os.makedirs(out_dir, exist_ok=True)
    for p, lo in enumerate(range(0, len(files), 64)):      # parts of 64 alignments keep every file below 1 MB
        s = slice(lo, lo + 64)
        np.savez_compressed(os.path.join(out_dir, f"len1024_taxa{taxa}_part{p}.npz"), shape=np.array([taxa, 1024, 4]),
                            data_bits=np.stack(rec["bits"][s]), seq_keys=np.array(rec["keys"][s]), merges=np.stack(rec["merges"][s]),
                            newick=np.array(rec["newick"][s]), selected_log_ps=np.stack(rec["slp"][s]),
                            step_max_abs_logit=np.array(rec["lmax"][s], dtype=np.float32),
                            step_top2_gap=np.array(rec["gap"][s], dtype=np.float32), source=np.array(rec["src"][s]))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "wide":
        main_wide()
    elif len(sys.argv) > 1 and sys.argv[1] == "all50":
        main_all50()
    elif len(sys.argv) > 1 and sys.argv[1] == "all100":
        main_all50(taxa=100, threads=int(os.environ.get("NNJ_GOLDEN_THREADS", "8")))
    elif len(sys.argv) > 1 and sys.argv[1] == "supervise":
        main_supervise()
    else:
        main()
