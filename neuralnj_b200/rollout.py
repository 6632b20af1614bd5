"""Rollout drivers and entry points with the reference's signatures (finetune_rl_search.py).

    reinforce_rollout(batch, agent, env, cfgs, ..., eval=True, argmax=...)      :78-189
    Agmax_one_instance(cfgs, MSA_file, policy_network, env, ...)                 :430-475
    Argmax_inference(test_file_path, write_dir, write_file_name, ...)            :478-509
    RL_Search(cfgs, MSA_file, policy_network, env, ...)                          :338-427
    Search_inference(test_file_path, write_dir, write_file_name)                 :512-541

Inference only (eval=True).  Two execution modes give the same results:
  * fused   — one `nnj_rollout` call does encode + all NJ steps on the device, then the merge list is
              replayed into `PhyInferEnv` so every host object ends up as in the reference;
  * stepwise — the reference's own loop (decode_zxr -> select -> env.step) over the drop-in methods.
Sampling (argmax=False) uses the Gumbel-max trick on the device; it draws from the same categorical
distribution as `Categorical(logits=logits).sample()` but not from the same RNG stream.
"""
from __future__ import annotations

import os
import time
from typing import Optional

import numpy as np
import torch

from .config import empty_config
from .environment import PhyInferEnv
from .model import PhyloATTN
from .phydata import load_pi_instance
from .support import _support, likelihood_support
from .treeutil import normalized_rf, rf_distance

EXPLORE_TEMPERTURE = lambda step: 1.0   # finetune_rl_search.py:39
STOP_STEP = 100                          # --stop_step default, finetune_rl_search.py:588
cfgs = None                              # module-level config like the reference's __main__ (set by main())


def _device_of(agent) -> torch.device:
    return next(agent.parameters()).device


def _step_slices(R: int):
    off, out = 0, []
    for n in range(R, 1, -1):
        p = n * (n - 1) // 2
        out.append((off, off + p))
        off += p
    return out


def sample_gumbel(shape, device, generator: Optional[torch.Generator] = None) -> torch.Tensor:
    u = torch.rand(shape, device=device, generator=generator).clamp_(1e-20, 1.0 - 1e-7)
    return -torch.log(-torch.log(u))


def reinforce_rollout(batch, agent, env, cfgs, replay_buffer=None, eval=False, argmax=False, get_all_tree=False,
                      branch_optimize=False, fused=True, generator: Optional[torch.Generator] = None):
    if not eval:
        raise NotImplementedError("reinforce_rollout(eval=False) is REINFORCE training (finetune_rl_search.py:192-335): "
                                  "outside the inference hot path")
    device = _device_of(agent)
    batch_seqs, batch_seq_keys, batch_array = batch["seqs"], batch["seq_keys"], batch["data"]
    batch_array = batch_array.to(device)
    batch_seq_mask = batch["seq_weights"].to(device) == 0
    env.init_states(batch_seqs, batch_seq_keys, batch_array)
    agent.eval()
    B, R = batch_array.shape[:2]

    if fused and hasattr(agent, "rollout_fused"):
        with torch.no_grad():
            gumbel = None if argmax else sample_gumbel((B, R - 1, R * (R - 1) // 2), device, generator)
            merges, slp, trace = agent.rollout_fused(batch_array, batch_seq_mask, gumbel=gumbel, want_logits=True)
            log_ps = [torch.log_softmax(trace[:, a:b] / EXPLORE_TEMPERTURE(t), dim=-1) for t, (a, b) in enumerate(_step_slices(R))][:-1]
            selected_log_ps = slp[:, :R - 2]
        env.replay_merges(merges, branch_optimize=branch_optimize)
    else:
        selected, log_ps = [], []
        actions_ij_prev = logits_prev = None
        step = 0
        with torch.no_grad():
            env.state_tensor = agent.encode_zxr(env.init_state_tensor, batch_seq_mask)
            while True:
                nb_seq = env.state_tensor.shape[1]
                ret = agent.decode_zxr(env.state_tensor, batch_seq_mask, (actions_ij_prev, None, logits_prev))
                logits = ret["logits"]
                log_p = torch.log_softmax(logits / EXPLORE_TEMPERTURE(step), dim=-1)
                if argmax:
                    actions = torch.argmax(logits, dim=-1)
                else:
                    actions = torch.argmax(logits / EXPLORE_TEMPERTURE(step) + sample_gumbel(logits.shape, device, generator), dim=-1)
                acts = actions.tolist()
                actions_ij_prev = torch.tensor([env.tree_pairs_dict[nb_seq][a] for a in acts], dtype=torch.int32, device=device)
                done = env.step(actions, [(None, None)] * B, branch_optimize=branch_optimize, agent=agent)
                if done:
                    break
                step += 1
                selected.append(torch.gather(log_p, 1, actions.unsqueeze(1)))
                log_ps.append(log_p)
                logits_prev = logits
        selected_log_ps = torch.cat(selected, dim=1) if selected else torch.zeros(B, 0, device=device)

    scores, best_rtree_tuple, best_tree_tuple, best_tree = env.evaluate_loglikelihood(get_all_tree=get_all_tree)
    return selected_log_ps, log_ps, scores, best_tree


def _expand(batch: dict, n: int) -> dict:
    out = {}
    for k, v in batch.items():
        one = v[0:1]
        out[k] = one * n if isinstance(one, list) else one.expand(n, *one.shape[1:])
    return out


def _tree_string(path: Optional[str]) -> Optional[str]:
    if not path:
        return None
    with open(path) as f:
        return f.readline().strip()


def Agmax_one_instance(cfgs, MSA_file, policy_network, env, c_best_tree_file=None, raw_tree_file=None, branch_optimize=False):
    batch = _expand(load_pi_instance(MSA_file), cfgs.env.batch_size)
    raw_tree_str, c_best_tree_str = _tree_string(raw_tree_file), _tree_string(c_best_tree_file)
    _, _, scores, best_tree = reinforce_rollout(batch, policy_network, env, cfgs, eval=True, argmax=True, branch_optimize=branch_optimize)
    out = dict(best_tree_str=best_tree, score=float(scores[0]), raw_tree_score=None, c_best_tree_score=None,
               rf_distance=None, rf_distance_raw=None, rf_distance_c_raw=None)
    # the reference scores the comparison trees with RAxML-NG (not available); topological distances need no likelihood
    if c_best_tree_str:
        out["rf_distance"] = normalized_rf(c_best_tree_str, best_tree)
    if raw_tree_str:
        out["rf_distance_raw"] = normalized_rf(raw_tree_str, best_tree)
    if raw_tree_str and c_best_tree_str:
        out["rf_distance_c_raw"] = normalized_rf(raw_tree_str, c_best_tree_str)
    return out


PRECISION = None                        # --precision of the CLI; None = cfgs.model.precision or the library default (bf16x3)


def _load_policy(cfgs, device, precision=None) -> PhyloATTN:
    net = PhyloATTN(cfgs, precision=precision or PRECISION).to(device)
    if cfgs.reload_checkpoint_path and os.path.exists(cfgs.reload_checkpoint_path):
        ckpt = torch.load(cfgs.reload_checkpoint_path, map_location="cpu")
        net.load_state_dict(ckpt["model_state_dict"])
        print(f"Reloaded checkpoint at epoch {ckpt.get('epoch')}, accumulated_steps {ckpt.get('accumulated_steps')}")
    elif cfgs.reload_checkpoint_path:
        print(f"checkpoint {cfgs.reload_checkpoint_path} not found: using default-initialised weights")
    return net.eval()


def _cfg(c):
    c = c if c is not None else cfgs
    if c is None:
        raise ValueError("no configuration: pass cfgs=... or set neuralnj_b200.rollout.cfgs")
    return c


def _stack_instances(instances) -> dict:
    """Batch dicts of `load_pi_instance` (one alignment each, equal taxa / site counts) -> one batch dict."""
    out = {}
    for k in instances[0]:
        vals = [inst[k] for inst in instances]
        out[k] = torch.cat(vals, dim=0) if torch.is_tensor(vals[0]) else [x for v in vals for x in v]
    return out


def _rank_share(items):
    """This rank's contiguous share of `items` when a process group is up (alignments are independent: no collective)."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return items
    from .shard import shard_bounds
    lo, hi = shard_bounds(len(items), dist.get_rank(), dist.get_world_size())
    return items[lo:hi]


def Argmax_inference(test_file_path, write_dir, write_file_name=None, branch_optimize=False, cfgs=None, device=None, precision=None,
                     files_per_call=1, policy_network=None, bootstrap=0, bootstrap_seed=0,
                     alrt=0, alrt_seed=0):
    """One `.tre` per `.phy` of a directory (finetune_rl_search.py:478-509).

    `files_per_call=1` is the reference's loop: one alignment per call (expanded to `cfgs.env.batch_size` copies, :444).
    `files_per_call=N` (not a reference argument) stacks up to N alignments of EQUAL taxa and site counts into one rollout call -
    what the batched kernels are built for (hundreds of trees/s instead of one 15 ms call per file); alignments of other shapes go
    into their own calls, nothing is padded, and the rollout of an alignment does not depend on its batch mates, so the trees
    are the ones the per-file loop writes.  Under an initialised process group every rank takes a contiguous share of the sorted
    file list and writes its own trees (no collective); the return value lists this rank's files.

    `bootstrap=N` (not a reference argument) also writes `<name>.fbp.tre` and `<name>.tbe.tre` beside each `<name>.tre`: the same tree
    with FBP / TBE support from N bootstrap replicates drawn with `bootstrap_seed` (`neuralnj_b200.support`).  A file's replicates
    run on the rank that owns the file.

    `alrt=N` (not a reference argument) also writes `<name>.alrt.tre` (SH-aLRT from N RELL replicates drawn with `alrt_seed`) and
    `<name>.abayes.tre` (aBayes): the tree with its branch lengths and model optimised (`neuralnj_b200.support.likelihood_support`)."""
    c = _cfg(cfgs)
    if device is None:                # one process per GPU under torchrun: the rank's own device
        import torch.distributed as dist
        ranked = dist.is_available() and dist.is_initialized() and "LOCAL_RANK" in os.environ
        device = torch.device("cuda", int(os.environ["LOCAL_RANK"])) if ranked else torch.device("cuda")
    env = PhyInferEnv(c, device)
    policy = policy_network if policy_network is not None else _load_policy(c, device, precision)
    os.makedirs(write_dir, exist_ok=True)
    files = _rank_share(sorted(f for f in os.listdir(test_file_path) if f.endswith(".phy")))
    written = []

    def write_support(file, msa, tree):
        runs = []                     # (labelled trees it writes, the support computation)
        if alrt > 0:
            runs.append((("alrt", "abayes"), lambda: likelihood_support(msa, policy, tree=tree, n_rell=alrt, seed=alrt_seed)))
        if bootstrap > 0:             # no replicate sharding: the file is this rank's
            runs.append((("fbp", "tbe"), lambda: _support(msa, policy, bootstrap, bootstrap_seed, tree, None)))
        for kinds, run in runs:
            res = run()
            for kind in kinds:
                with open(os.path.join(write_dir, f"{file[:-4]}.{kind}.tre"), "w") as f:
                    f.write(res["newick_" + kind])

    if files_per_call <= 1:
        for file in files:
            res = Agmax_one_instance(c, os.path.join(test_file_path, file), policy, env, branch_optimize=branch_optimize)
            dst = os.path.join(write_dir, file[:-4] + ".tre")
            with open(dst, "w") as f:
                f.write(res["best_tree_str"])
            written.append(dst)
            write_support(file, os.path.join(test_file_path, file), res["best_tree_str"])
        return written

    pending = {}                      # (taxa, sites) -> [(file, instance), ...]

    def run(items):
        batch = _stack_instances([inst for _, inst in items])
        _, _, _, trees = reinforce_rollout(batch, policy, env, c, eval=True, argmax=True, get_all_tree=True, branch_optimize=branch_optimize)
        for (file, inst), tree in zip(items, trees):
            with open(os.path.join(write_dir, file[:-4] + ".tre"), "w") as f:
                f.write(tree)
            write_support(file, inst, tree)

    for file in files:
        inst = load_pi_instance(os.path.join(test_file_path, file))
        shape = tuple(inst["data"].shape[1:3])
        pending.setdefault(shape, []).append((file, inst))
        if len(pending[shape]) == files_per_call:
            run(pending.pop(shape))
    for shape in sorted(pending):
        run(pending[shape])
    return [os.path.join(write_dir, file[:-4] + ".tre") for file in files]


def RL_Search(cfgs, MSA_file, policy_network, env, c_best_tree_file=None, raw_tree_file=None, scorer=None, stop_step=None,
              generator: Optional[torch.Generator] = None, topotest_top: int = 20):
    """NeuralNJ-MC: sampled rollouts, keep the best-scoring tree (finetune_rl_search.py:338-427).

    One encoder pass is shared by every sampled rollout (the reference re-encodes the same MSA each time, :112), the
    rollouts are sampled on the device (Gumbel-max), identical topologies are scored once, and the score is what the
    reference uses: the log-likelihood under GTR+I+G after branch-length / model optimisation (`optimize_brlen`,
    environment.py:365-379) - here on the GPU (`neuralnj_b200.likelihood.score_topologies`), all new topologies of an
    episode in one call.  `scorer` overrides it: a callable `scorer(newick, seq_keys, seqs) -> float`, or "logp" to rank by
    the policy's own trajectory log-probability (no likelihood at all).

    Beside the reference's keys the result holds `candidates` (not a reference key): the up to `topotest_top` distinct topologies
    with the highest scores as (score, Newick) pairs, best first, ties in the order first seen - the input of a tree topology test.
    """
    from . import likelihood as LH
    from .environment import EVOLUTION_MODEL
    stop = STOP_STEP if stop_step is None else stop_step
    device = _device_of(policy_network)
    batch = _expand(load_pi_instance(MSA_file), cfgs.env.batch_size)
    data = batch["data"].to(device)
    mask = batch["seq_weights"].to(device) == 0
    B, R = data.shape[:2]
    raw_tree_str = _tree_string(raw_tree_file)
    policy_network.eval()
    start = time.time()
    best_tree, best_score, t_best = None, -np.inf, None
    seen = {}
    masks = LH.onehot_to_masks(batch["data"][0]) if scorer is None else None
    keys = batch["seq_keys"][0]
    with torch.no_grad():
        state = policy_network.encode_zxr(data[:1], mask[:1]).expand(B, -1, -1, -1).contiguous()
        step_cur = 0
        for epoch in range(1, cfgs.num_epoch):
            for episode in range(cfgs.num_episodes):
                gumbel = sample_gumbel((B, R - 1, R * (R - 1) // 2), device, generator)
                merges, slp, _ = policy_network.rollout_fused(batch_seq_mask=mask, gumbel=gumbel, state=state)
                env.init_states(batch["seqs"], batch["seq_keys"], data)
                env.replay_merges(merges)
                traj_logp = slp[:, :R - 2].sum(1).tolist()
                fresh = {}
                for b, st in enumerate(env.states):
                    tr = st.subtrees[0].topo_repr
                    if tr not in seen and tr not in fresh:
                        fresh[tr] = b
                if fresh and scorer is None:
                    mg = merges.cpu().numpy()
                    ch = np.stack([LH.children_from_merges(mg[b], R) for b in fresh.values()])
                    ll, brl = LH.score_topologies(masks, ch, keys, model=EVOLUTION_MODEL, opt_model=True, device=device)
                    for k, tr in enumerate(fresh):
                        seen[tr] = (float(ll[k]), LH.tuples_to_newick(LH.tuples_with_lengths(ch[k], brl[k], keys, unrooted=True)))
                else:
                    for tr, b in fresh.items():
                        tree = env.states[b].subtrees[0]
                        sc = traj_logp[b] if scorer == "logp" else scorer(tree.utree_op_str, batch["seq_keys"][b], batch["seqs"][b])
                        seen[tr] = (float(sc), tree.utree_op_str)
                for st in env.states:
                    score, newick = seen[st.subtrees[0].topo_repr]
                    if best_tree is None or score > best_score:
                        best_tree, best_score, t_best = newick, score, time.time() - start
                step_cur = 1 + episode + (epoch - 1) * cfgs.num_episodes
            if step_cur >= stop:
                break
    rel_rf = normalized_rf(raw_tree_str, best_tree) if raw_tree_str else None
    values = list(seen.values())                                          # in the order first seen
    order = sorted(range(len(values)), key=lambda i: (-values[i][0], i))
    return dict(the_best_tree=best_tree, the_best_score=best_score, raw_tree_score=None, c_best_tree_score=None,
                time_when_best_score_max=t_best, relative_rf_distance=rel_rf, step_cur=step_cur, distinct_topologies=len(seen),
                candidates=[values[i] for i in order[:max(int(topotest_top), 0)]])


def Search_inference(test_file_path, write_dir, write_file_name=None, cfgs=None, device=None, scorer=None, stop_step=None, precision=None,
                     policy_network=None, topotest=0, topotest_top=20, topotest_seed=0):
    """One `.tre` per `.phy` of a directory: the best tree of RL_Search (finetune_rl_search.py:512-541).

    `topotest=N` (not a reference argument) also writes, for an alignment with at least two distinct candidate topologies,
    `<name>.trees` (the up to `topotest_top` best-scoring candidates, one Newick per line, best first) and `<name>.topotest.txt`
    (IQ-TREE's tree test table of those trees from N RELL replicates per scale drawn with `topotest_seed`,
    `neuralnj_b200.support.topology_test`).  The `.tre` is the same with and without it."""
    from .environment import EVOLUTION_MODEL
    from .support import topology_test
    c = _cfg(cfgs)
    device = device or torch.device("cuda")
    env = PhyInferEnv(c, device)
    policy = policy_network if policy_network is not None else _load_policy(c, device, precision)
    os.makedirs(write_dir, exist_ok=True)
    written = []
    for file in sorted(f for f in os.listdir(test_file_path) if f.endswith(".phy")):
        path = os.path.join(test_file_path, file)
        res = RL_Search(c, path, policy, env, scorer=scorer, stop_step=stop_step, topotest_top=topotest_top)
        dst = os.path.join(write_dir, file[:-4] + ".tre")
        with open(dst, "w") as f:
            f.write(res["the_best_tree"])
        written.append(dst)
        if topotest > 0 and len(res["candidates"]) >= 2:
            trees = [newick for _, newick in res["candidates"]]
            with open(os.path.join(write_dir, file[:-4] + ".trees"), "w") as f:
                f.write("".join(t + "\n" for t in trees))
            tt = topology_test(path, trees, n_boot=topotest, seed=topotest_seed, model=EVOLUTION_MODEL, device=device)
            with open(os.path.join(write_dir, file[:-4] + ".topotest.txt"), "w") as f:
                f.write(tt["table"])
        print(f"finish NerualNJ-MC for {file}")
    return written


def main(argv=None):
    """CLI with the reference's flags (finetune_rl_search.py:583-621)."""
    import argparse
    global cfgs, STOP_STEP, PRECISION
    ap = argparse.ArgumentParser(description="NeuralNJ inference (B200 path)")
    ap.add_argument("--config_path", type=str, default="")
    ap.add_argument("--infer_opt", type=str, default="Argmax", help='"Argmax" (NeuralNJ) or "Search" (NeuralNJ-MC)')
    ap.add_argument("--stop_step", type=int, default=100)
    ap.add_argument("--evolution_model", type=str, default="GTR+I+G")
    ap.add_argument("--branch_optimize", action="store_true")
    ap.add_argument("--precision", type=str, default=None, choices=["fp32", "bf16x3", "bf16"],
                    help="arithmetic of the CUDA path (not a reference flag); default bf16x3: tcgen05 split-bf16, topologies identical to fp32")
    ap.add_argument("--files_per_call", type=int, default=1,
                    help="Argmax: alignments of equal shape stacked into one rollout call (not a reference flag); 1 = the reference's per-file loop")
    ap.add_argument("--bootstrap", type=int, default=0,
                    help="Argmax: also write <name>.fbp.tre / <name>.tbe.tre with support from N bootstrap replicates (not a reference flag)")
    ap.add_argument("--bootstrap_seed", type=int, default=0, help="seed of the bootstrap replicates (not a reference flag)")
    ap.add_argument("--alrt", type=int, default=0,
                    help="Argmax: also write <name>.alrt.tre / <name>.abayes.tre with SH-aLRT from N RELL replicates and aBayes (not a reference flag)")
    ap.add_argument("--alrt_seed", type=int, default=0, help="seed of the RELL replicates (not a reference flag)")
    ap.add_argument("--topotest", type=int, default=0,
                    help="Search: also write <name>.trees / <name>.topotest.txt, a tree topology test (KH, SH, ELW, AU) of the best candidates "
                         "from N RELL replicates per scale (not a reference flag)")
    ap.add_argument("--topotest_top", type=int, default=20, help="Search: candidates the topology test compares, at least 2 (not a reference flag)")
    ap.add_argument("--topotest_seed", type=int, default=0, help="seed of the topology test's replicates (not a reference flag)")
    args = ap.parse_args(argv)
    if args.bootstrap and args.infer_opt != "Argmax":
        raise SystemExit("--bootstrap applies to --infer_opt Argmax")
    if args.alrt and args.infer_opt != "Argmax":
        raise SystemExit("--alrt applies to --infer_opt Argmax")
    if args.topotest and args.infer_opt != "Search":
        raise SystemExit("--topotest applies to --infer_opt Search (pass the Argmax tree and its alternatives to support.topology_test)")
    if args.topotest_top < 2:
        raise SystemExit("--topotest_top must be at least 2: a topology test compares trees")
    PRECISION = args.precision
    cfgs = empty_config()
    if args.config_path:
        cfgs.merge_from_file(args.config_path)
    STOP_STEP = args.stop_step
    name = os.path.basename(os.path.normpath(cfgs.instance_path))
    write_dir = f"output/{args.infer_opt}_dim{cfgs.model.embed_dim}_patch{cfgs.model.patch_size}/{name}"
    if args.infer_opt == "Argmax":
        return Argmax_inference(cfgs.instance_path, write_dir, None, branch_optimize=args.branch_optimize, files_per_call=args.files_per_call,
                                bootstrap=args.bootstrap, bootstrap_seed=args.bootstrap_seed, alrt=args.alrt, alrt_seed=args.alrt_seed)
    if args.infer_opt == "Search":
        return Search_inference(cfgs.instance_path, write_dir, None, topotest=args.topotest, topotest_top=args.topotest_top,
                                topotest_seed=args.topotest_seed)
    raise SystemExit(f'--infer_opt {args.infer_opt}: "Finetune" (NeuralNJ-RL) trains the policy and is outside this path')


if __name__ == "__main__":
    main()
