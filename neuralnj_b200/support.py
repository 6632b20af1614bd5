"""Bootstrap branch support of NJ trees: Felsenstein's bootstrap proportion (FBP) and the transfer bootstrap expectation (TBE,
Lemoine et al., Nature 2018) on the branches of one reference tree - what RAxML-NG computes with `--bootstrap` and
`--support --bs-metric fbp,tbe`.

    res = bootstrap_support("alignment.phy", policy_network, n_replicates=1000, seed=0)
    res["newick_fbp"], res["newick_tbe"], res["fbp"], res["tbe"], res["splits"]

The replicates are drawn on the device (`nnj_bootstrap_columns`), each one is an Argmax rollout (`rollout_fused`), and the
transfer distances of the reference splits to the replicate trees are computed on the device from the merge lists
(`nnj_split_distances`); per chunk of CHUNK replicates only the int64 totals [2, S] stay behind, and merge lists never reach the
host.  Definitions: DESIGN.md section 11.  A replicate depends only on (seed, replicate index, real column count), so the chunk
size and the number of ranks do not change any result.

`likelihood_support` puts aLRT, SH-aLRT, aBayes and the local bootstrap probability on the branches of one tree instead (DESIGN.md
section 12): no rollouts, the NNI alternatives of every branch and RELL replicates on the device, trees up to 4096 taxa.
"""
from __future__ import annotations

import ctypes as C
import os
import re
from typing import List, Optional, Tuple

import numpy as np
import torch

from ._lib import NnjError, check, lib
from .config import empty_config
from .environment import PhyInferEnv
from .phydata import load_pi_instance

CHUNK = 128            # replicates per device round trip (resample -> rollout -> split distances)
# Every replicate is an Argmax rollout, and the encoder's column attention holds the keys and values of one site column in shared
# memory (512 bytes a taxon, at most 200 KB): rollouts stop at 400 taxa.  nnj_split_distances alone goes to 512.
MAX_TAXA = 400


def _ptr(t: torch.Tensor):
    return C.c_void_p(t.data_ptr()) if t.numel() else C.c_void_p(0)


def _on_cuda(what: str, *tensors: torch.Tensor) -> torch.device:
    dev = tensors[0].device
    if dev.type != "cuda" or any(t.device != dev for t in tensors):
        raise NnjError(f"{what}: tensors must be on one CUDA device (there is no CPU fallback)")
    return dev


def bootstrap_columns(data: torch.Tensor, l_eff: int, seed: int, rep0: int, n: int) -> torch.Tensor:
    """Replicates rep0 .. rep0+n-1 of one alignment (nnj_bootstrap_columns): data int8 [R,L,4] on the device -> int8 [n,R,L,4]."""
    dev = _on_cuda("bootstrap_columns", data)
    data = data.to(torch.int8).contiguous()
    R, L = data.shape[:2]
    out = torch.empty(n, R, L, 4, dtype=torch.int8, device=dev)
    with torch.cuda.device(dev):
        check(lib().nnj_bootstrap_columns(_ptr(data), R, L, l_eff, seed, rep0, n, _ptr(out),
                                          C.c_void_p(torch.cuda.current_stream().cuda_stream)), "nnj_bootstrap_columns")
    return out


def split_distances(merges: torch.Tensor, splits: torch.Tensor) -> torch.Tensor:
    """Transfer distances (nnj_split_distances): merges int32 [B,R-1,2], splits int64 [S,ceil(R/64)] (uint64 bit patterns)
    -> int32 [B,S]; a row of -1 marks a merge list that is not valid."""
    dev = _on_cuda("split_distances", merges, splits)
    merges = merges.to(torch.int32).contiguous()
    splits = splits.to(torch.int64).contiguous()
    B, R, S = merges.shape[0], merges.shape[1] + 1, splits.shape[0]
    out = torch.empty(B, S, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        check(lib().nnj_split_distances(_ptr(merges), B, R, _ptr(splits), S, _ptr(out),
                                        C.c_void_p(torch.cuda.current_stream().cuda_stream)), "nnj_split_distances")
    return out


# ---------------------------------------------------------------------------------------------------------- Newick side

def internal_clades(newick: str, keys) -> List[Tuple[int, frozenset]]:
    """(offset just after the `)`, leaf indices below) of every internal node of `newick`, in text order; leaf names are `keys`."""
    index = {k: i for i, k in enumerate(keys)}
    stack, out, seen = [set()], [], []
    s, pos = newick, 0
    while pos < len(s):
        ch = s[pos]
        if ch == "(":
            stack.append(set())
            pos += 1
        elif ch == ")":
            if len(stack) < 2:
                raise ValueError(f"bad Newick near position {pos}")
            clade = stack.pop()
            stack[-1] |= clade
            pos += 1
            out.append((pos, frozenset(clade)))
            if pos < len(s) and s[pos] not in ":,);" and not s[pos].isspace():
                raise ValueError("the reference tree already carries internal node labels")
        elif ch == ":":
            while pos < len(s) and s[pos] not in ",);":
                pos += 1
        elif ch in ",;" or ch.isspace():
            pos += 1
        else:
            st = pos
            while pos < len(s) and s[pos] not in ":,();":
                pos += 1
            name = s[st:pos].strip()
            if name not in index:
                raise ValueError(f"taxon {name!r} of the tree is not in the alignment")
            seen.append(index[name])
            stack[-1].add(index[name])
    if len(stack) != 1 or sorted(seen) != list(range(len(keys))):
        raise ValueError("the tree must name every taxon of the alignment exactly once")
    return out


def light_side(clade: frozenset, keys) -> frozenset:
    """The side of the split a clade defines that names a split: the smaller one, on a tie the one whose sorted taxon names come first."""
    rest = frozenset(range(len(keys))) - clade
    return min(clade, rest, key=lambda t: (len(t), sorted(keys[i] for i in t)))


def reference_splits(newick: str, keys):
    """Non-trivial splits of `newick`: (light sides as leaf-index frozensets in order of first appearance, split index of each
    labelled node as (offset, split))."""
    R = len(keys)
    splits, where, labelled = [], {}, []
    for pos, clade in internal_clades(newick, keys):
        if not 2 <= len(clade) <= R - 2:
            continue
        light = light_side(clade, keys)
        if light not in where:                   # the two root children of a rooted binary tree are one split
            where[light] = len(splits)
            splits.append(light)
        labelled.append((pos, where[light]))
    return splits, labelled


def split_bitsets(splits, R: int) -> torch.Tensor:
    """Leaf-index sets -> the bitsets nnj_split_distances reads: int64 [S, ceil(R/64)] holding uint64 bit patterns."""
    bits = np.zeros((len(splits), (R + 63) // 64), dtype=np.uint64)
    for k, sp in enumerate(splits):
        for i in sp:
            bits[k, i // 64] |= np.uint64(1) << np.uint64(i % 64)
    return torch.from_numpy(bits.view(np.int64))


def label_newick(newick: str, labelled, labels) -> str:
    """Insert labels[split] after the `)` of every labelled node."""
    parts, last = [], 0
    for pos, k in labelled:
        parts += [newick[last:pos], labels[k]]
        last = pos
    return "".join(parts) + newick[last:]


def strip_support_labels(newick: str) -> str:
    """Inverse of the labelling: drop the text between each `)` and the next `:`, `,`, `)` or `;`."""
    return re.sub(r"\)[^:,;()\s]+", ")", newick)


# ---------------------------------------------------------------------------------------------------------- driver

def _process_group():
    import torch.distributed as dist
    return dist if dist.is_available() and dist.is_initialized() else None


def bootstrap_support(msa, policy_network, n_replicates: int, seed: int = 0, tree: Optional[str] = None) -> dict:
    """FBP and TBE support of the branches of one tree from `n_replicates` bootstrap replicates of the alignment `msa`.

    `msa` is a path (.phy / .fasta / .aln) or a `load_pi_instance` batch of one alignment of at most 400 taxa (MAX_TAXA).  `tree=None`
    puts support on the Argmax tree of the original alignment (the Newick string `Argmax_inference` writes); `tree="<newick>"` on a given tree instead (for
    example the best tree of `RL_Search`), whose taxon names must be the alignment's.  Replicates are drawn, inferred (Argmax
    rollouts of `policy_network`) and compared on the device.  Under an initialised process group every rank runs a contiguous
    share of the replicate indices and one all_reduce sums the totals: the result is that of a single process.

    Returns `tree` (unlabelled Newick), `splits` (light sides as frozensets of taxon names), `fbp` [S] (percent), `tbe` [S],
    `newick_fbp` / `newick_tbe` (labels after the `)` of each internal node with a non-trivial split), `n_replicates`, `seed`."""
    return _support(msa, policy_network, n_replicates, seed, tree, _process_group())


def _count_and_seed(n: int, what: str, seed: int) -> Tuple[int, int]:
    if int(n) < 1:
        raise ValueError(f"{what} must be >= 1")
    if not 0 <= int(seed) < 2 ** 64:
        raise ValueError("seed must be in [0, 2^64)")
    return int(n), int(seed)


def _one_alignment(msa, caller: str) -> dict:
    """A path (.phy / .fasta / .aln) or a `load_pi_instance` batch -> the batch, which must hold one alignment."""
    batch = load_pi_instance(os.fspath(msa)) if isinstance(msa, (str, os.PathLike)) else msa
    if batch["data"].shape[0] != 1:
        raise ValueError(f"{caller} takes one alignment")
    return batch


def _argmax_tree(policy_network, batch: dict, data: torch.Tensor, mask: torch.Tensor) -> str:
    """Unrooted Newick of the Argmax rollout of one alignment (data int8 [R, L, 4] and the padding mask [L] on the network's device),
    as `Argmax_inference` writes it."""
    with torch.no_grad():
        merges, _, _ = policy_network.rollout_fused(data[None], mask[None])
    env = PhyInferEnv(empty_config(), data.device)
    env.init_states(batch["seqs"], batch["seq_keys"], batch["data"])
    env.replay_merges(merges)
    return env.states[0].subtrees[0].utree_op_str


def _support(msa, policy_network, n_replicates: int, seed: int, tree: Optional[str], group) -> dict:
    N, seed = _count_and_seed(n_replicates, "n_replicates", seed)
    batch = _one_alignment(msa, "bootstrap_support")
    R, L = batch["data"].shape[1:3]
    if R > MAX_TAXA:
        raise ValueError(f"bootstrap_support: {R} taxa, at most {MAX_TAXA} are supported: every replicate is an Argmax rollout, and the "
                         f"encoder's column attention stops at {MAX_TAXA} taxa")
    keys = [str(k) for k in batch["seq_keys"][0]]
    padded = batch["seq_weights"][0] == 0
    l_eff = int((~padded).sum())
    if l_eff == 0 or bool(padded[:l_eff].any()):
        raise NnjError("bootstrap_support: the real columns of the alignment must be a non-empty prefix (padding is the suffix)")
    device = next(policy_network.parameters()).device
    data = batch["data"][0].to(device=device, dtype=torch.int8).contiguous()
    mask = padded.to(device)
    if tree is None:
        tree = _argmax_tree(policy_network, batch, data, mask)
    splits, labelled = reference_splits(tree, keys)
    S = len(splits)
    splits_dev = split_bitsets(splits, R).to(device)
    lo, hi = 0, N
    if group is not None:
        from .shard import shard_bounds
        lo, hi = shard_bounds(N, group.get_rank(), group.get_world_size())
    # totals[0, :S] = replicates with delta = 0, totals[1, :S] = sum of delta; totals[0, S] counts replicate trees whose merge list
    # was not valid, so that every rank learns of one after the single all_reduce
    totals = torch.zeros(2, S + 1, dtype=torch.int64, device=device)
    if S:
        with torch.no_grad():
            for r0 in range(lo, hi, CHUNK):
                n = min(CHUNK, hi - r0)
                reps = bootstrap_columns(data, l_eff, seed, r0, n)
                merges, _, _ = policy_network.rollout_fused(reps, mask.expand(n, L))
                d = split_distances(merges, splits_dev)
                totals[0, :S] += (d == 0).sum(0)
                totals[1, :S] += d.clamp(min=0).sum(0)
                totals[0, S] += (d < 0).any(1).sum()
    if group is not None:
        group.all_reduce(totals)
    tot = totals.cpu().numpy()
    if tot[0, S]:
        raise NnjError(f"bootstrap_support: {int(tot[0, S])} replicate merge lists are not valid")
    count, dsum = tot[0, :S], tot[1, :S]
    p = np.array([len(sp) for sp in splits], dtype=np.int64)
    fbp = 100.0 * count / N
    tbe = 1.0 - dsum / (N * (p - 1))
    fbp_labels = [str(int(100 * int(c) / N + 0.5)) for c in count]
    tbe_labels = [f"{v:.3f}" for v in tbe]
    return dict(tree=tree, splits=[frozenset(keys[i] for i in sp) for sp in splits], fbp=fbp, tbe=tbe,
                newick_fbp=label_newick(tree, labelled, fbp_labels), newick_tbe=label_newick(tree, labelled, tbe_labels),
                n_replicates=N, seed=seed)


# ---------------------------------------------------------------------------------------------------------- likelihood support

def likelihood_support(msa, policy_network=None, tree: Optional[str] = None, n_rell: int = 1000, seed: int = 0, model: str = "GTR+I+G") -> dict:
    """Likelihood branch support (DESIGN.md 12) of one tree: aLRT, SH-aLRT, aBayes and the local bootstrap probability (LBP) of
    every internal branch - what IQ-TREE reports with `-alrt 1000 -abayes`.

    `msa` is a path or a `load_pi_instance` batch of one alignment.  `tree=None` builds the Argmax tree of `policy_network` (at most
    400 taxa, the rollout's limit); a given Newick `tree` may have up to 4096 taxa.  The branch lengths and model parameters are
    optimised first (`TreeLikelihood.optimize_all`), then the two NNI alternatives of every internal branch are optimised and
    n_rell RELL replicates drawn with `seed` (`TreeLikelihood.nni_support`), all on the device.

    Returns `tree` (unrooted Newick with the optimised lengths), `splits` (light sides as frozensets of taxon names), per split
    `alrt` (2 delta), `sh_alrt` and `lbp` (percent), `abayes`, `llh_nni` [S, 2] (L1, L2), and `llh` (L0), `n_better_nni` (splits
    where an NNI has the higher likelihood, delta < 0), `newick_alrt` (SH-aLRT, %.1f) and `newick_abayes` (%.3f), `n_rell`, `seed`."""
    from . import likelihood as LH
    from .treeutil import treestr_to_tuples
    N, seed = _count_and_seed(n_rell, "n_rell", seed)
    batch = _one_alignment(msa, "likelihood_support")
    R = batch["data"].shape[1]
    if R > 4096:
        raise ValueError(f"likelihood_support: {R} taxa, the tree likelihood supports at most 4096")
    keys = [str(k) for k in batch["seq_keys"][0]]
    real = (batch["seq_weights"][0] != 0).cpu().numpy()
    if tree is None:
        if policy_network is None:
            raise ValueError("likelihood_support: tree=None needs a policy_network to build the Argmax tree")
        device = next(policy_network.parameters()).device
        data = batch["data"][0].to(device=device, dtype=torch.int8).contiguous()
        tree = _argmax_tree(policy_network, batch, data, torch.from_numpy(~real).to(device))
    else:
        device = next(policy_network.parameters()).device if policy_network is not None else torch.device("cuda")
    masks = LH.onehot_to_masks(batch["data"][0])[:, real]
    pats, w = LH.compress_patterns(masks)
    children, brlen = LH.tree_arrays_from_tuples(treestr_to_tuples(tree), keys)
    ch = children[None]
    eng = LH.TreeLikelihood(pats, w, device=device)
    sm = LH.SubstModel(model, LH.empirical_freqs(masks), 1)
    t, _, ll = eng.optimize_all(ch, brlen[None], sm)
    res = eng.nni_support(ch, t, sm, N, seed)
    out_tree = LH.tuples_to_newick(LH.tuples_with_lengths(children, t[0], keys, unrooted=True))
    splits, labelled = reference_splits(out_tree, keys)
    S = len(splits)
    where = {sp: k for k, sp in enumerate(splits)}
    order = np.zeros(S, dtype=np.int64)
    nodes = res["branch_node"][0]
    if len(nodes) != S:
        raise NnjError(f"likelihood_support: {len(nodes)} internal branches but {S} splits in the tree")
    branch = {v: i for i, v in enumerate(nodes.tolist())}
    below = [frozenset([i]) for i in range(R)] + [None] * (R - 1)      # leaves below each node; a child's set goes once joined
    for k, (a, b) in enumerate(children.tolist()):
        below[R + k], below[a], below[b] = below[a] | below[b], None, None
        if R + k in branch:
            order[where[light_side(below[R + k], keys)]] = branch[R + k]
    llh3 = res["llh"][0][order]
    delta = llh3[:, 0] - np.maximum(llh3[:, 1], llh3[:, 2])
    with np.errstate(over="ignore"):
        abayes = 1.0 / (1.0 + np.exp(llh3[:, 1] - llh3[:, 0]) + np.exp(llh3[:, 2] - llh3[:, 0]))
    sh = 100.0 * res["sh_count"][0][order] / N
    lbp = 100.0 * res["lbp_count"][0][order] / N
    return dict(tree=out_tree, splits=[frozenset(keys[i] for i in sp) for sp in splits], alrt=2.0 * delta, sh_alrt=sh, abayes=abayes, lbp=lbp,
                llh_nni=llh3[:, 1:].copy(), llh=float(ll[0]), n_better_nni=int((delta < 0).sum()),
                newick_alrt=label_newick(out_tree, labelled, [f"{x:.1f}" for x in sh]),
                newick_abayes=label_newick(out_tree, labelled, [f"{x:.3f}" for x in abayes]), n_rell=N, seed=seed)


# ---------------------------------------------------------------------------------------------------------- tree topology tests

TOPO_SCALES = 10       # multiscale bootstrap: r_s = (5 + s) / 10, s = 0..9; scale 5 (r = 1) is the RELL bootstrap of bp, KH, SH and ELW


def scale_draws(n: int) -> List[int]:
    """Sites drawn per replicate at each scale: n_s = floor(r_s n + 0.5), r_s = (5 + s) / 10 (the rule of nnj_llh_topology_test)."""
    return [int(np.floor((5 + s) / 10 * n + 0.5)) for s in range(TOPO_SCALES)]


def au_pvalue(win_s, n_s, n: int, N: int) -> float:
    """Approximately unbiased p-value of one tree (Shimodaira 2002, first-order fit as in CONSEL): win_s [10] replicates of each scale
    the tree wins, n_s [10] sites drawn at each scale, n the site count, N replicates per scale.  Over the scales with 0 < win_s < N,
    z_s = Phi^-1(1 - bp_s) is fitted as v sqrt(r_s) + c / sqrt(r_s), r_s = n_s / n, by least squares weighted with
    N phi(z_s)^2 / (bp_s (1 - bp_s)); p-AU = 1 - Phi(v - c).  With fewer than two such scales: bp at r = 1."""
    from statistics import NormalDist
    nd = NormalDist()
    win_s = np.asarray(win_s, dtype=np.float64)
    use = [s for s in range(len(win_s)) if 0 < win_s[s] < N]
    if len(use) < 2:
        return float(win_s[5] / N)
    bp = win_s[use] / N
    r = np.asarray(n_s, dtype=np.float64)[use] / n
    z = np.array([nd.inv_cdf(1.0 - b) for b in bp])
    sw = np.sqrt(N * np.array([nd.pdf(x) for x in z]) ** 2 / (bp * (1.0 - bp)))
    (v, c), *_ = np.linalg.lstsq(np.stack([np.sqrt(r), 1.0 / np.sqrt(r)], 1) * sw[:, None], z * sw, rcond=None)
    return 1.0 - nd.cdf(v - c)


def _mark(p: float) -> str:
    return "+" if p >= 0.05 else "-"


def topology_table(llh, delta, bp, p_kh, p_sh, elw, p_au) -> str:
    """IQ-TREE's tree test table: one row per tree in input order; + / - after a value marks value >= / < 0.05."""
    head = f"{'Tree':>4} {'logL':>14} {'deltaL':>10} {'bp-RELL':>9} {'p-KH':>8} {'p-SH':>8} {'c-ELW':>9} {'p-AU':>9}"
    rows = [head, "-" * len(head)]
    for k in range(len(llh)):
        rows.append(f"{k + 1:>4} {llh[k]:>14.4f} {delta[k]:>10.4f} {bp[k]:>7.4f} {_mark(bp[k])} {p_kh[k]:>6.4f} {_mark(p_kh[k])} "
                    f"{p_sh[k]:>6.4f} {_mark(p_sh[k])} {elw[k]:>7.4f} {_mark(elw[k])} {p_au[k]:>7.4f} {_mark(p_au[k])}")
    return "\n".join(rows) + "\n"


def topology_test(msa, trees: List[str], n_boot: int = 10000, seed: int = 0, model: str = "GTR+I+G", device=None) -> dict:
    """Tree topology test (DESIGN.md 13) of candidate trees of one alignment - what IQ-TREE reports with `-z trees -zb 10000 -au`:
    bp-RELL, p-KH, p-SH, c-ELW and p-AU of every tree, which trees the data reject at the 5% level and which they cannot.

    `msa` is a path or a `load_pi_instance` batch of one alignment, `trees` two or more Newick strings on its taxa (up to 4096).  Each
    tree's branch lengths (starting from the given ones) and model parameters are optimised (`TreeLikelihood.optimize_all`), then
    n_boot RELL replicates at each of 10 scales are drawn with `seed` and scored against every tree on the device
    (`TreeLikelihood.topology_test`); the AU fit runs on the host (`au_pvalue`).

    Returns, per tree in input order: `tree` (unrooted Newick with the fitted lengths), `llh`, `delta` (largest llh - llh), `bp`,
    `p_kh`, `p_sh`, `elw`, `p_au` and `win` [K, 10] (replicates each scale's winner); and `table` (IQ-TREE's columns), `n_boot`, `seed`."""
    from . import likelihood as LH
    from .treeutil import treestr_to_tuples
    N, seed = _count_and_seed(n_boot, "n_boot", seed)
    if N > 10 ** 6:
        raise ValueError("n_boot must be <= 10^6")
    if len(trees) < 2:
        raise ValueError("topology_test compares at least two trees")
    batch = _one_alignment(msa, "topology_test")
    R = batch["data"].shape[1]
    if R > 4096:
        raise ValueError(f"topology_test: {R} taxa, the tree likelihood supports at most 4096")
    keys = [str(k) for k in batch["seq_keys"][0]]
    real = (batch["seq_weights"][0] != 0).cpu().numpy()
    masks = LH.onehot_to_masks(batch["data"][0])[:, real]
    pats, w = LH.compress_patterns(masks)
    arrays = [LH.tree_arrays_from_tuples(treestr_to_tuples(t), keys) for t in trees]
    ch = np.stack([a[0] for a in arrays])
    K = len(trees)
    eng = LH.TreeLikelihood(pats, w, device=device)
    sm = LH.SubstModel(model, LH.empirical_freqs(masks), K)
    t, _, _ = eng.optimize_all(ch, np.stack([a[1] for a in arrays]), sm)
    res = eng.topology_test(ch, t, sm, N, seed)
    n = int(w.sum())
    n_s = scale_draws(n)
    llh = res["llh"]
    delta = llh.max() - llh
    bp, p_kh, p_sh, elw = res["win"][5] / N, res["kh"] / N, res["sh"] / N, res["elw"]
    p_au = np.array([au_pvalue(res["win"][:, k], n_s, n, N) for k in range(K)])
    return dict(tree=[LH.tuples_to_newick(LH.tuples_with_lengths(ch[k], t[k], keys, unrooted=True)) for k in range(K)], llh=llh, delta=delta,
                bp=bp, p_kh=p_kh, p_sh=p_sh, elw=elw, p_au=p_au, win=res["win"].T.copy(),
                table=topology_table(llh, delta, bp, p_kh, p_sh, elw, p_au), n_boot=N, seed=seed)

