"""CPU oracle of bootstrap branch support (test infrastructure): a numpy restatement of the two device primitives of
neuralnj_b200/csrc/nnj_support.cu and FBP / TBE recomputed with Python sets from replicate Newick strings.

    philox4x32_10(ctr, key)                      Philox4x32-10, vectorised over uint32 numpy arrays
    source_columns(l_eff, seed, reps)            [n, l_eff] input column of every output column of replicates `reps`
    bootstrap_columns(data, l_eff, seed, rep0, n)  nnj_bootstrap_columns: int8 [R,L,4] -> [n,R,L,4]
    split_distances(merges, splits)              nnj_split_distances with Python integers as bitsets
    support_from_newicks(ref, replicates)        FBP / TBE over treeutil.bipartitions of the replicate trees

`bootstrap_columns` and `split_distances` take and return torch tensors like the device primitives of
`neuralnj_b200.support`, so a test can put them in their place (the same pattern as the oracle stand-in agent of
tests/test_entry_batched_cpu.py)."""
from __future__ import annotations

import numpy as np
import torch

M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
_MASK32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr: 4 uint32 arrays (broadcastable), key: 2 uint32 values -> 4 uint64 arrays holding the uint32 output words."""
    c = [np.asarray(x, dtype=np.uint64) & _MASK32 for x in ctr]
    k = [np.uint64(int(x) & 0xFFFFFFFF) for x in key]
    for _ in range(10):
        p0 = np.uint64(M0) * c[0]              # < 2^64: both factors are below 2^32
        p1 = np.uint64(M1) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k[0], p1 & _MASK32, (p0 >> np.uint64(32)) ^ c[3] ^ k[1], p0 & _MASK32]
        k = [(k[0] + np.uint64(W0)) & _MASK32, (k[1] + np.uint64(W1)) & _MASK32]
    return c


def source_columns(l_eff: int, seed: int, reps) -> np.ndarray:
    """Input column of each of the l_eff real output columns of every replicate index in `reps` -> int64 [len(reps), l_eff]."""
    reps = np.asarray(reps, dtype=np.uint64)[:, None]
    cols = np.arange(l_eff, dtype=np.uint64)[None, :]
    x0 = philox4x32_10((cols, reps & _MASK32, reps >> np.uint64(32), np.zeros_like(cols)), (seed & 0xFFFFFFFF, seed >> 32))[0]
    return ((x0 * np.uint64(l_eff)) >> np.uint64(32)).astype(np.int64)


def bootstrap_columns(data: torch.Tensor, l_eff: int, seed: int, rep0: int, n: int) -> torch.Tensor:
    """Replicates rep0 .. rep0+n-1 of one alignment: data int8 [R,L,4] -> int8 [n,R,L,4]; padded columns (>= l_eff) copied."""
    src = source_columns(l_eff, seed, np.arange(rep0, rep0 + n, dtype=np.uint64))
    d = data.cpu().numpy()
    out = np.repeat(d[None], n, axis=0)
    for b in range(n):
        out[b, :, :l_eff] = d[:, src[b]]
    return torch.from_numpy(out).to(data.device)


def clades_from_merges(merges, R: int):
    """The R-2 non-root clades of an NJ merge list (slot i <- new node, slot j removed) as int bitsets; None if not valid."""
    slots = list(range(R))
    bits = [1 << t for t in range(R)]
    for t, (i, j) in enumerate(np.asarray(merges).tolist()):
        if not 0 <= i < j < R - t:
            return None
        bits.append(bits[slots[i]] | bits[slots[j]])
        slots[i] = R + t
        del slots[j]
    return bits[R:2 * R - 2]


def transfer_distance(A: int, clades, R: int) -> int:
    full = (1 << R) - 1
    A &= full
    pa = bin(A).count("1")
    best = max(min(pa, R - pa) - 1, 0)
    for c in clades:
        d = bin(A ^ c).count("1")
        best = min(best, d, R - d)
    return best


def split_distances(merges: torch.Tensor, splits: torch.Tensor) -> torch.Tensor:
    """nnj_split_distances: merges int32 [B,R-1,2], splits int64 [S,W] (uint64 bit patterns) -> int32 [B,S], -1 rows = invalid."""
    B, R = merges.shape[0], merges.shape[1] + 1
    sp = splits.cpu().numpy().view(np.uint64)
    As = [sum(int(w) << (64 * k) for k, w in enumerate(row)) for row in sp]
    out = np.full((B, len(As)), -1, dtype=np.int32)
    for b, mg in enumerate(merges.cpu().numpy()):
        cl = clades_from_merges(mg, R)
        if cl is not None:
            out[b] = [transfer_distance(A, cl, R) for A in As]
    return torch.from_numpy(out).to(merges.device)


def support_from_newicks(ref_newick: str, replicate_newicks):
    """{light side of each non-trivial split of ref_newick (treeutil.bipartitions): (fbp, tbe)} from replicate Newick strings."""
    from neuralnj_b200.treeutil import bipartitions, treestr_to_tuples

    def leaves(t):
        return [t] if isinstance(t, str) else [x for item in t if isinstance(item, (tuple, str)) for x in leaves(item)]

    taxa = frozenset(leaves(treestr_to_tuples(ref_newick)))
    R, N = len(taxa), len(replicate_newicks)
    rep_splits = [bipartitions(nw) for nw in replicate_newicks]
    out = {}
    for A in bipartitions(ref_newick):
        p = min(len(A), R - len(A))
        exact, total = 0, 0
        for bp in rep_splits:
            d = min([p - 1] + [min(len(A ^ c), R - len(A ^ c)) for c in bp])
            exact += d == 0
            total += d
        out[A] = (100.0 * exact / N, 1.0 - total / (N * (p - 1)))
    return out
