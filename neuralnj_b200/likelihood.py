"""Tree likelihood on the GPU: the scorer behind Search (NeuralNJ-MC) and `branch_optimize=True`.

Drop-in for the two functions the reference takes from its native RAxML-NG binding
(`RAxMLpy/raxmlpy/core.py:6-12` -> `RAxMLpy/cpp/raxmlpy.cpp:1790-1872`):

    optimize_brlen(tree_str, msa, is_root=False, iters=32, model="JC", opt_model=True) -> (utree_str, llh_before, llh_after)
    compute_llh(tree_str, msa, is_root=False, model="JC", opt_model=True)               -> llh

with `msa = {"labels": [...], "sequences": [...]}` (environment.py:365-379).  The likelihood and the Newton-Raphson branch
optimiser run in `csrc/nnj_llh.cu` (one CTA per tree, fp64) through the C ABI (`nnj_llh_eval`, `nnj_llh_optimize_brlen`);
this module holds what is host logic in any implementation: Newick <-> join-order arrays, alignment patterns, the model
parametrisation and the outer loop over model parameters.  There is no CPU fallback.

Model: GTR (or JC) + optional invariant sites (+I) + optional discrete gamma, 4 classes (+G), empirical base
frequencies.  Branch lengths are clamped to [BRLEN_MIN, BRLEN_MAX] = [1e-6, 100] everywhere, evaluation included, and so is
the root branch (the two root edges, one branch of the unrooted tree): zero or negative lengths, which Newick files and the
zero branches that resolve a multifurcation bring, score as 1e-6.  Per-pattern scaling of the conditional likelihood vectors
keeps trees of 3 to 4096 taxa free of fp64 underflow.  RAxML-NG itself is not available (the reference git-clones it at install time): parity with its numbers is
UNPINNED; tests pin this implementation against an independent CPU restatement and brute-force enumeration
(oracle/llh_oracle.py).  The optimiser is this repo's own (coordinate golden-section over 5 rates, alpha, p_inv between
branch-length sweeps, stopping when a round gains < 1 log-unit like `optimize_model(treeinfo, 1.0)`, raxmlpy.cpp:1721-1746) and
runs inside the kernel, one tree per CTA.
"""
from __future__ import annotations

import ctypes as C
import itertools
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from .treeutil import treestr_to_tuples

BRLEN_DEFAULT = 0.1                    # raxml-ng's RAXML_BRLEN_DEFAULT: trees without lengths start here
BRLEN_MIN, BRLEN_MAX = 1e-6, 100.0     # every length is clamped to this range, when evaluated as when optimised
PLACEHOLDER = 0.12345                  # environment.py:287 prints missing lengths like this; treated as "no length"
RATE_LO, RATE_HI, ALPHA_LO, ALPHA_HI, PINV_HI = 1e-3, 1e3, 0.02, 100.0, 0.99
_GOLD = 0.3819660112501051
# the packed model the kernels read, [B, LLH_MODEL] doubles: its slots as in nnj_llh.cuh (MDL_*)
LLH_MODEL = 64
MDL_LAM, MDL_U, MDL_UINV, MDL_FREQ, MDL_RATE, MDL_PINV, MDL_ALPHA, MDL_FLAGS, MDL_GTR = 0, 4, 20, 36, 40, 44, 45, 46, 48
_IUPAC = {"A": 1, "C": 2, "G": 4, "T": 8, "U": 8, "R": 5, "Y": 10, "S": 6, "W": 9, "K": 12, "M": 3, "B": 14, "D": 13, "H": 11, "V": 7}


# ------------------------------------------------------------------ alignment
def sequences_to_masks(seqs: Sequence[str]) -> np.ndarray:
    """DNA strings -> uint8 [R, L] state masks (bit 0 A, 1 C, 2 G, 3 T); gaps, N, ? and anything unknown = 15."""
    lut = np.full(256, 15, dtype=np.uint8)
    for ch, m in _IUPAC.items():
        lut[ord(ch)] = lut[ord(ch.lower())] = m
    return np.stack([lut[np.frombuffer(s.encode("ascii", "replace"), dtype=np.uint8)] for s in seqs])


def onehot_to_masks(data) -> np.ndarray:
    """int8 one-hot [..., R, L, 4] (the encoder's input; gap = 1111, pad = 0000) -> uint8 masks [..., R, L]."""
    d = (data.cpu().numpy() if torch.is_tensor(data) else np.asarray(data)).astype(np.uint8)
    m = d[..., 0] | (d[..., 1] << 1) | (d[..., 2] << 2) | (d[..., 3] << 3)
    m[m == 0] = 15
    return m


def compress_patterns(masks: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """Unique columns + multiplicities (the reference compresses patterns as well, raxmlpy.cpp:1646-1657)."""
    cols, counts = np.unique(masks, axis=1, return_counts=True)
    return np.ascontiguousarray(cols), counts.astype(np.float64)


def empirical_freqs(masks: np.ndarray) -> np.ndarray:
    """Base frequencies counted from the alignment; an ambiguity code spreads its count over its states, 15 is skipped."""
    cnt = np.zeros(4)
    hist = np.bincount(masks.ravel(), minlength=16)
    for m in range(1, 15):
        bits = np.array([(m >> a) & 1 for a in range(4)], dtype=np.float64)
        cnt += hist[m] * bits / bits.sum()
    if cnt.sum() == 0:
        return np.full(4, 0.25)
    f = np.maximum(cnt / cnt.sum(), 1e-4)
    return f / f.sum()


# ------------------------------------------------------------------ model
class SubstModel:
    """Parameters of B trees at once.  `spec` follows raxmlpy's model strings: "JC" or "GTR", optionally "+I", "+G"."""

    def __init__(self, spec: str, freqs: np.ndarray, B: int):
        parts = [p.strip().upper() for p in spec.split("+")]
        if parts[0] not in ("JC", "GTR"):
            raise ValueError(f"unsupported substitution model {spec!r}: use JC or GTR with optional +I / +G")
        bad = [p for p in parts[1:] if p not in ("I", "G", "G4", "F", "FC")]
        if bad:
            raise ValueError(f"unsupported model component(s) {bad} in {spec!r}")
        self.gtr, self.inv, self.gamma = parts[0] == "GTR", "I" in parts[1:], any(p in ("G", "G4") for p in parts[1:])
        self.B = B
        self.rates = np.ones((B, 6))
        self.freqs = np.tile(np.asarray(freqs, dtype=np.float64) if self.gtr else np.full(4, 0.25), (B, 1)) if np.ndim(freqs) == 1 else np.asarray(freqs, dtype=np.float64)
        self.alpha = np.ones(B)
        self.pinv = np.zeros(B)
        self._gamma_cache = {}

    def free_params(self) -> List[Tuple[str, int]]:
        p = [("rate", i) for i in range(5)] if self.gtr else []
        if self.gamma:
            p.append(("alpha", 0))
        if self.inv:
            p.append(("pinv", 0))
        return p

    def pack(self) -> np.ndarray:
        """[B, LLH_MODEL] doubles for the kernels: eigenvalues, U, U^-1, freqs, class rates, p_inv, alpha, flags, the 6 GTR rates (MDL_*)."""
        B, pi = self.B, self.freqs
        r = np.zeros((B, 4, 4))
        for k, (a, b) in enumerate(itertools.combinations(range(4), 2)):
            r[:, a, b] = r[:, b, a] = self.rates[:, k]
        Q = r * pi[:, None, :]
        idx = np.arange(4)
        Q[:, idx, idx] = -Q.sum(2)
        Q /= -(pi * Q[:, idx, idx]).sum(1)[:, None, None]
        sq = np.sqrt(pi)
        S = sq[:, :, None] * Q / sq[:, None, :]
        lam, V = np.linalg.eigh(0.5 * (S + S.transpose(0, 2, 1)))
        U, Ui = V / sq[:, :, None], V.transpose(0, 2, 1) * sq[:, None, :]
        cat = np.ones((B, 4))
        if self.gamma:
            L = _lib.lib()
            buf = (C.c_double * 4)()
            cache = self._gamma_cache
            if len(cache) > 4096:
                cache.clear()
            for b in range(B):
                a = float(self.alpha[b])
                if a not in cache:
                    _lib.check(L.nnj_gamma_rates(a, 4, buf), "nnj_gamma_rates")
                    cache[a] = np.array(buf[:])
                cat[b] = cache[a]
        out = np.zeros((B, LLH_MODEL))
        out[:, MDL_LAM:MDL_LAM + 4], out[:, MDL_U:MDL_U + 16], out[:, MDL_UINV:MDL_UINV + 16] = lam, U.reshape(B, 16), Ui.reshape(B, 16)
        out[:, MDL_FREQ:MDL_FREQ + 4], out[:, MDL_RATE:MDL_RATE + 4] = pi, cat
        out[:, MDL_PINV], out[:, MDL_ALPHA], out[:, MDL_GTR:MDL_GTR + 6] = self.pinv, self.alpha, self.rates
        out[:, MDL_FLAGS] = float((1 if self.gtr else 0) | (2 if self.gamma else 0) | (4 if self.inv else 0))
        return out

    def unpack(self, packed: np.ndarray) -> None:
        """Take the parameters the kernel optimised (nnj_llh_optimize_all) back into this object."""
        self.pinv, self.alpha, self.rates = packed[:, MDL_PINV].copy(), packed[:, MDL_ALPHA].copy(), packed[:, MDL_GTR:MDL_GTR + 6].copy()


# ------------------------------------------------------------------ trees
def tree_arrays_from_tuples(tup, labels: Sequence[str]) -> Tuple[np.ndarray, np.ndarray]:
    """(child, len, child, len[, child, len]) tuples (treestr_to_tuples) -> children int32 [R-1, 2] in join order and
    brlen float64 [2R-2].  A trifurcating (unrooted) top level is rooted on its last branch.  Missing lengths and the
    reference's 0.12345 placeholder become BRLEN_DEFAULT."""
    index = {name: i for i, name in enumerate(labels)}
    R = len(labels)
    children, brlen = [], np.full(2 * R - 2, BRLEN_DEFAULT)

    def split(t):
        kids, lens = [], []
        for item in t:
            if isinstance(item, (tuple, str)):
                kids.append(item)
                lens.append(None)
            else:
                lens[-1] = float(item)
        return kids, lens

    def visit(node) -> int:
        if isinstance(node, str):
            if node not in index:
                raise ValueError(f"tree leaf {node!r} is not among the alignment labels")
            return index[node]
        kids, lens = split(node)
        ids = [visit(k) for k in kids]
        while len(ids) > 2:                    # resolve a multifurcation by joining its first two children with a zero-length branch
            v = R + len(children)
            children.append((ids[0], ids[1]))
            for c, ln in zip(ids[:2], lens[:2]):
                if ln is not None and ln != PLACEHOLDER:
                    brlen[c] = ln
            ids, lens = [v] + ids[2:], [0.0] + lens[2:]
        v = R + len(children)
        children.append((ids[0], ids[1]))
        for c, ln in zip(ids, lens):
            if ln is not None and ln != PLACEHOLDER:
                brlen[c] = ln
        return v

    visit(tup)
    if len(children) != R - 1:
        raise ValueError(f"tree has {len(children) + 1} leaves, the alignment {R}")
    return np.asarray(children, dtype=np.int32), brlen


def children_from_merges(merges, R: int) -> np.ndarray:
    """NJ merge list [R-1, 2] (logical slot indices, slot i <- new node, slot j removed: environment.py:764-768) -> children."""
    cur = list(range(R))
    out = np.zeros((R - 1, 2), dtype=np.int32)
    for k, (i, j) in enumerate(np.asarray(merges).tolist()):
        out[k] = (cur[i], cur[j])
        cur[i] = R + k
        del cur[j]
    return out


def tuples_with_lengths(children: np.ndarray, brlen: np.ndarray, labels: Sequence[str], unrooted: bool):
    """Join-order arrays -> (child, len, child, len) tuples; `unrooted` expands one root child into a trifurcation whose third
    branch carries the whole root branch (what pll_utree_export_newick prints, raxmlpy.cpp:1845-1849)."""
    R = len(labels)

    def sub(v):
        if v < R:
            return labels[v]
        a, b = (int(c) for c in children[v - R])
        return (sub(a), float(brlen[a]), sub(b), float(brlen[b]))

    c1, c2 = (int(c) for c in children[-1])
    if not unrooted:
        return (sub(c1), float(brlen[c1]), sub(c2), float(brlen[c2]))
    t0 = float(brlen[c1] + brlen[c2])
    if c1 >= R:
        return sub(c1) + (sub(c2), t0)
    if c2 >= R:
        return sub(c2) + (sub(c1), t0)
    return (sub(c1), t0 / 2, sub(c2), t0 / 2)


def tuples_to_newick(t) -> str:
    def fmt(n):
        if isinstance(n, str):
            return n
        parts = []
        for k in range(0, len(n), 2):
            parts.append(f"{fmt(n[k])}:{n[k + 1]:.8f}")
        return "(" + ",".join(parts) + ")"
    return fmt(t) + ";"


# ------------------------------------------------------------------ NNI quartets (DESIGN.md 12)
def internal_branches(children) -> List[int]:
    """The R-3 internal branches of a tree as the inner node v below each, in increasing v: every inner node but the root, where
    the root branch counts once, at the first root child c1, and only when both root children are inner."""
    children = np.asarray(children)
    R = len(children) + 1
    c1, c2 = (int(c) for c in children[-1])
    return [v for v in range(R, 2 * R - 2) if v not in (c1, c2) or (v == c1 and c2 >= R)]


def quartet(children, v: int) -> Tuple[Tuple[int, int, int, int], Tuple[int, int, int, int, int]]:
    """The quartet around the branch above v -> ((a, b, c, d), edges).  a, b are v's children, c its sibling and d its parent p,
    whose outer vector is U[p] (the rest of the tree); for the root branch (v = c1) c and d are the children of c2.  `edges` are the
    nodes whose brlen entries hold the central, A, B, C and D lengths (v, a, b, c, p; the root branch is brlen[c1] + brlen[c2])."""
    children = np.asarray(children)
    R = len(children) + 1
    c1, c2 = (int(c) for c in children[-1])
    a, b = (int(c) for c in children[v - R])
    if v == c1:
        c, d = (int(x) for x in children[c2 - R])
        return (a, b, c, d), (v, a, b, c, d)
    p = next(R + k for k, pair in enumerate(children.tolist()) if v in pair)
    pa, pb = (int(x) for x in children[p - R])
    c = pb if pa == v else pa
    return (a, b, c, p), (v, a, b, c, p)


def nni_tree(children, v: int, k: int, brlen=None):
    """Alternative k (1: AC|BD, 2: AD|BC) of the branch above v as a join-order children array; k = 0 is the tree itself (renumbered
    the same way).  Alternative 1 swaps B and C, alternative 2 swaps A and C.  With `brlen`, also returns the lengths carried over:
    the branch above every node keeps its length (the nodes are renumbered, their edges are not)."""
    children = np.asarray(children)
    R = len(children) + 1
    kids = {R + j: [int(x), int(y)] for j, (x, y) in enumerate(children.tolist())}
    (a, b, c, _), _ = quartet(children, v)
    c1, c2 = (int(x) for x in children[-1])
    holder = c2 if v == c1 else next(u for u, pair in kids.items() if v in pair)      # the node c hangs below
    if k in (1, 2):
        mine = b if k == 1 else a
        kids[v][kids[v].index(mine)] = c
        kids[holder][kids[holder].index(c)] = mine
    elif k != 0:
        raise ValueError("k must be 0, 1 or 2")
    new_id, out = {u: u for u in range(R)}, []

    def visit(u):
        stack = [(u, False)]
        while stack:
            x, done = stack.pop()
            if x < R:
                continue
            if done:
                new_id[x] = R + len(out)
                out.append((new_id[kids[x][0]], new_id[kids[x][1]]))
            else:
                stack.append((x, True))
                stack.append((kids[x][1], False))
                stack.append((kids[x][0], False))

    visit(2 * R - 2)
    ch = np.asarray(out, dtype=np.int32)
    if brlen is None:
        return ch
    bl = np.zeros(2 * R - 2)
    for u in range(2 * R - 2):
        bl[new_id[u]] = brlen[u]
    return ch, bl


# ------------------------------------------------------------------ engine
class TreeLikelihood:
    """B trees over alignments of one shape, scored together (one CTA per tree)."""

    def __init__(self, masks: np.ndarray, weights: Optional[np.ndarray] = None, device=None):
        """masks uint8 [B, R, L] (or [R, L]: the same alignment for every tree, expanded lazily); weights [B, L] / [L]."""
        self.device = torch.device(device or "cuda")
        if self.device.type != "cuda":
            raise _lib.NnjError("the tree likelihood runs on a CUDA device only (no CPU fallback)")
        self.masks = np.ascontiguousarray(masks, dtype=np.uint8)
        self.shared = self.masks.ndim == 2
        self.R, self.L = self.masks.shape[-2:]
        if self.R < 3:
            raise ValueError("need at least 3 taxa")
        self.weights = np.ones(self.masks.shape[:-2] + (self.L,)) if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
        self._staged_B, self._staged_tw = None, None      # the device tips and weights of the last tree count
        self._ws = None

    def _staged(self, B: int):
        if self._staged_B != B:
            m = torch.from_numpy(self.masks)
            w = torch.from_numpy(self.weights)
            if self.shared:
                m, w = m.unsqueeze(0).expand(B, -1, -1), w.unsqueeze(0).expand(B, -1)
            elif m.shape[0] != B:
                raise ValueError(f"{m.shape[0]} alignments but {B} trees")
            self._staged_B, self._staged_tw = B, (m.contiguous().to(self.device), w.contiguous().to(self.device))
        return self._staged_tw

    def _workspace(self, need: int, what: str):
        """The grow-only device workspace, at least `need` bytes (what the library's `what` returned; < 0: a shape it refuses)."""
        if need < 0:
            raise _lib.NnjError(f"{what}: bad shape")
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        return self._ws

    def _trees(self, children, brlen, model: SubstModel):
        """-> children int32 [B, R-1, 2], a copy of brlen float64 [B, 2R-2], B; one model row per tree."""
        children = np.ascontiguousarray(children, dtype=np.int32)
        B = children.shape[0]
        brlen = np.ascontiguousarray(brlen, dtype=np.float64).copy()
        if children.shape != (B, self.R - 1, 2) or brlen.shape != (B, 2 * self.R - 2) or model.B != B:
            raise ValueError("children must be [B, R-1, 2], brlen [B, 2R-2], one model row per tree")
        return children, brlen, B

    def _call(self, mode: str, children, brlen, model: SubstModel, max_passes=32, eps=1e-3, lh_eps=1.0, max_rounds=10):
        """One C-ABI call over all B trees: mode "eval" (nnj_llh_eval), "brlen" (nnj_llh_optimize_brlen) or "all" (nnj_llh_optimize_all)."""
        children, brlen, B = self._trees(children, brlen, model)
        tips, w = self._staged(B)
        ws = self._workspace(int(_lib.lib().nnj_llh_workspace_bytes(B, self.R, self.L)), "nnj_llh_workspace_bytes")
        packed = model.pack()
        L = _lib.lib()
        after, before = np.zeros(B), np.zeros(B)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        vp = C.c_void_p
        dev = (vp(tips.data_ptr()), vp(w.data_ptr()), children.ctypes.data_as(vp), brlen.ctypes.data_as(vp), packed.ctypes.data_as(vp), B, self.R, self.L)
        tail = (vp(ws.data_ptr()), ws.numel(), vp(stream))
        with torch.cuda.device(self.device):
            if mode == "eval":
                rc = L.nnj_llh_eval(*dev, after.ctypes.data_as(vp), *tail)
            elif mode == "brlen":
                rc = L.nnj_llh_optimize_brlen(*dev, int(max_passes), float(eps), before.ctypes.data_as(vp), after.ctypes.data_as(vp), *tail)
            else:
                rc = L.nnj_llh_optimize_all(*dev, int(max_passes), float(eps), float(lh_eps), int(max_rounds), before.ctypes.data_as(vp),
                                            after.ctypes.data_as(vp), *tail)
        _lib.check(rc, "nnj_llh_" + mode)
        if mode == "all":
            model.unpack(packed)
        return brlen, before, after

    def loglik(self, children, brlen, model: SubstModel) -> np.ndarray:
        return self._call("eval", children, brlen, model)[2]

    def optimize_branches(self, children, brlen, model: SubstModel, max_passes=32, eps=1e-3):
        """-> (brlen_opt [B, 2R-2], llh_before [B], llh_after [B])"""
        return self._call("brlen", children, brlen, model, max_passes, eps)

    def optimize_all(self, children, brlen, model: SubstModel, lh_eps=1.0, max_rounds=10, max_passes=32, eps=1e-3):
        """Branch lengths, then rounds of (every free model parameter by golden section, branch lengths) until a round gains
        < lh_eps - per tree, entirely inside the kernel (nnj_llh_optimize_all: eigen-system and class rates are rebuilt on the
        device, no host round trips).  Updates `model` in place.  -> (brlen_opt, llh_before, llh_after)"""
        return self._call("all", children, brlen, model, max_passes, eps, lh_eps, max_rounds)


    def nni_support(self, children, brlen, model: SubstModel, n_rell: int, seed: int, rep0: int = 0, site_llh: bool = False) -> dict:
        """Likelihood support of the R-3 internal branches of B trees (nnj_llh_branch_support, DESIGN.md 12) at the given lengths and
        model, which should be optimised already (optimize_all).  -> dict of numpy arrays: branch_node [B, R-3], llh [B, R-3, 3]
        (L0, L1, L2), nni_brlen [B, R-3, 2, 5], sh_count and lbp_count [B, R-3] over replicates rep0 .. rep0+n_rell-1, and with
        site_llh=True the per-pattern log-likelihoods [B, R-3, 3, L] as a device tensor."""
        children, brlen, B = self._trees(children, brlen, model)
        R, L = self.R, self.L
        if not 0 <= int(seed) < 2 ** 64 or int(rep0) < 0 or int(n_rell) < 0:
            raise ValueError("need 0 <= seed < 2^64, rep0 >= 0, n_rell >= 0")
        nb = max(R - 3, 0)
        tips, w = self._staged(B)
        lib = _lib.lib()
        ws = self._workspace(int(lib.nnj_llh_support_workspace_bytes(B, R, L, int(n_rell))), "nnj_llh_support_workspace_bytes")
        packed = model.pack()
        out = dict(branch_node=np.zeros((B, nb), dtype=np.int32), llh=np.zeros((B, nb, 3)), nni_brlen=np.zeros((B, nb, 2, 5)),
                   sh_count=np.zeros((B, nb), dtype=np.int32), lbp_count=np.zeros((B, nb), dtype=np.int32))
        site = torch.empty((B, nb, 3, L), dtype=torch.float64, device=self.device) if site_llh and nb else None
        vp = C.c_void_p
        ptr = [out[k].ctypes.data_as(vp) for k in ("branch_node", "llh", "nni_brlen", "sh_count", "lbp_count")]
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            rc = lib.nnj_llh_branch_support(vp(tips.data_ptr()), vp(w.data_ptr()), children.ctypes.data_as(vp), brlen.ctypes.data_as(vp),
                                            packed.ctypes.data_as(vp), B, R, L, C.c_uint64(int(seed)), int(rep0), int(n_rell), *ptr,
                                            vp(site.data_ptr() if site is not None else 0), vp(ws.data_ptr()), ws.numel(), vp(stream))
        _lib.check(rc, "nnj_llh_branch_support")
        if site_llh:
            out["site_llh"] = site if site is not None else torch.empty((B, 0, 3, L), dtype=torch.float64, device=self.device)
        return out

    def topology_test(self, children, brlen, model: SubstModel, n_boot: int, seed: int, site_llh: bool = False) -> dict:
        """Tree topology test over the K trees (nnj_llh_topology_test, DESIGN.md 13) at the given lengths and models, which should be
        optimised already (optimize_all).  Needs the shared-alignment form (masks [R, L]).  -> dict of numpy arrays: llh [K] (L_k),
        win [10, K] (winner counts per scale), kh, sh [K] (KH / SH counts) and elw [K], over n_boot replicates per scale drawn with
        `seed`; with site_llh=True the per-pattern log-likelihoods [K, L] as a device tensor."""
        if not self.shared:
            raise ValueError("topology_test compares trees of one alignment: construct TreeLikelihood with masks [R, L]")
        children, brlen, K = self._trees(children, brlen, model)
        R, L = self.R, self.L
        if K < 2:
            raise ValueError("topology_test needs at least two trees")
        if R > 4096:
            raise ValueError(f"topology_test: {R} taxa, the tree likelihood supports at most 4096")
        if not 0 <= int(seed) < 2 ** 64 or not 1 <= int(n_boot) <= 10 ** 6:
            raise ValueError("need 0 <= seed < 2^64 and 1 <= n_boot <= 10^6")
        tips = torch.from_numpy(self.masks).to(self.device)
        w = torch.from_numpy(self.weights).to(self.device)
        lib = _lib.lib()
        ws = self._workspace(int(lib.nnj_llh_topotest_workspace_bytes(K, R, L, int(n_boot))), "nnj_llh_topotest_workspace_bytes")
        packed = model.pack()
        out = dict(llh=np.zeros(K), win=np.zeros((10, K), dtype=np.int32), kh=np.zeros(K, dtype=np.int32), sh=np.zeros(K, dtype=np.int32),
                   elw=np.zeros(K))
        site = torch.empty((K, L), dtype=torch.float64, device=self.device) if site_llh else None
        vp = C.c_void_p
        ptr = [out[k].ctypes.data_as(vp) for k in ("llh", "win", "kh", "sh", "elw")]
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            rc = lib.nnj_llh_topology_test(vp(tips.data_ptr()), vp(w.data_ptr()), children.ctypes.data_as(vp), brlen.ctypes.data_as(vp),
                                           packed.ctypes.data_as(vp), K, R, L, C.c_uint64(int(seed)), int(n_boot), *ptr,
                                           vp(site.data_ptr() if site is not None else 0), vp(ws.data_ptr()), ws.numel(), vp(stream))
        _lib.check(rc, "nnj_llh_topology_test")
        if site_llh:
            out["site_llh"] = site
        return out


# ------------------------------------------------------------------ raxmlpy-compatible entry points
def _prepare(tree_str: str, msa: dict, model: str):
    labels, seqs = list(msa["labels"]), list(msa["sequences"])
    masks = sequences_to_masks(seqs)
    children, brlen = tree_arrays_from_tuples(treestr_to_tuples(tree_str), labels)
    pats, w = compress_patterns(masks)
    sm = SubstModel(model, empirical_freqs(masks), 1)
    return labels, TreeLikelihood(pats, w), children[None], brlen[None], sm


def optimize_brlen(tree_str, msa, is_root=False, iters=32, model="JC", opt_model=True, device=None):
    """raxmlpy.optimize_brlen (core.py:6-8): -> (unrooted Newick with optimised lengths, log L before, log L after).
    `iters` bounds the branch-length sweeps like the reference's argument of the same name; `is_root` is accepted for
    signature compatibility (rooted and unrooted inputs are both understood from the string)."""
    labels, eng, ch, bl, sm = _prepare(tree_str, msa, model)
    if opt_model:
        t, before, after = eng.optimize_all(ch, bl, sm)
    else:
        t, before, after = eng.optimize_branches(ch, bl, sm, max_passes=max(1, int(iters)))
    newick = tuples_to_newick(tuples_with_lengths(ch[0], t[0], labels, unrooted=True))
    return newick, float(before[0]), float(after[0])


def compute_llh(tree_str, msa, is_root=False, model="JC", opt_model=True, device=None):
    """raxmlpy.compute_llh (core.py:10-12): log L of the tree as given; with opt_model the model parameters (not the branch
    lengths) are optimised first (raxmlpy.cpp:1783-1787): coordinate golden section from the host, one evaluation per launch."""
    labels, eng, ch, bl, sm = _prepare(tree_str, msa, model)
    best = float(eng.loglik(ch, bl, sm)[0])
    if not opt_model:
        return best
    bounds = {"rate": (np.log(RATE_LO), np.log(RATE_HI)), "alpha": (np.log(ALPHA_LO), np.log(ALPHA_HI)), "pinv": (0.0, PINV_HI)}

    def objective(kind, i, x):
        if kind == "rate":
            sm.rates[:, i] = np.exp(x)
        elif kind == "alpha":
            sm.alpha = np.exp(np.atleast_1d(x))
        else:
            sm.pinv = np.atleast_1d(np.asarray(x, dtype=np.float64))
        return float(eng.loglik(ch, bl, sm)[0])

    for _ in range(10):
        start = best
        for kind, i in sm.free_params():
            a, b = bounds[kind]
            x1, x2 = a + _GOLD * (b - a), b - _GOLD * (b - a)
            f1, f2 = objective(kind, i, x1), objective(kind, i, x2)
            for _it in range(24):
                if f1 >= f2:
                    b, x2, f2 = x2, x1, f1
                    x1 = a + _GOLD * (b - a)
                    f1 = objective(kind, i, x1)
                else:
                    a, x1, f1 = x1, x2, f2
                    x2 = b - _GOLD * (b - a)
                    f2 = objective(kind, i, x2)
            best = objective(kind, i, x1 if f1 > f2 else x2)
        if best - start < 1.0:
            break
    return best


def score_topologies(masks: np.ndarray, children: np.ndarray, labels: Sequence[str], model="GTR+I+G", opt_model=True, device=None):
    """Search-mode scorer: B candidate topologies of ONE alignment (masks [R, L]) optimised together.
    -> (log L [B], brlen [B, 2R-2]).  Used by RL_Search and PhyInferEnv(branch_optimize=True)."""
    pats, w = compress_patterns(masks)
    B = children.shape[0]
    eng = TreeLikelihood(pats, w, device=device)
    sm = SubstModel(model, empirical_freqs(masks), B)
    bl = np.full((B, 2 * masks.shape[0] - 2), BRLEN_DEFAULT)
    if opt_model:
        t, _, ll = eng.optimize_all(children, bl, sm)
    else:
        t, _, ll = eng.optimize_branches(children, bl, sm)
    return ll, t
