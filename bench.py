#!/usr/bin/env python
"""bench.py — trees/sec of Argmax inference on 50-taxa x 1024-site alignments (BASELINE.json metric, configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch 512] [--scaling strong|weak] [--impl ours|reference]
                    [--precision bf16x3|fp32] [--workload config2|config4|config1] [--dump-outputs DIR]

One "step" = one pass of the hot path (encode + 49 learned-NJ steps) over a batch of synthetic MSAs
(config 2: iid tokens over A,C,G,T,gap, seed 1234; weights torch.manual_seed(0) default init — the shipped
checkpoint is a missing blob).  configs[1] reads "batch of 512 ... sharded by alignment over 1/2/4/8 B200", so the default
is STRONG scaling: the 512 alignments of a step are cut into contiguous shards of 512/N per rank (alignments are independent:
no collective on the data path); value = 512 x K / max-over-ranks device time.  `--scaling weak` gives every rank its own
512 (the round-1 line); at N > 1 the default run also measures that and reports it under "weak".

Printed keys beyond the base contract:
  e2e            same metric through the C-ABI host-buffer entry point nnj_rollout_host (pinned host int8 MSA in,
                 merge lists out; H2D/D2H inside the timed region, staged per chunk on a copy stream)
  roofline       the kernel class with the largest share of the step, timed live with CUDA events on the launching
                 stream (nnj_profile_*), algorithmic FLOPs / launch from BASELINE.md section 3
  roofline_step  the whole step: algorithmic TFLOP/s against the sustained bf16 peak, encoder and NJ loop separately, and the
                 NJ loop's DRAM bytes per tree against SURVEY 8(d)'s 334 MB streaming figure
  kernels        per-class milliseconds / launches / share of the profiled step
  latency_b1_ms  one alignment, device-resident input -> merge list (median of 7)
  directory_inference  Argmax_inference over PHYLIP files of the timed batch: per-file loop vs files_per_call=128 (wall clock, host work included)
  tree_llh       the Search-mode scorer: 32 topologies of the batch scored with the GPU likelihood (branch lengths / + model search)
  gpu_eager_baseline  the reference formulation (the oracle restatement) in torch eager on this GPU at B = 1 / 8 / 32 (SURVEY 8d)
  parity_check   after the timed region: alignments of the bench batch replayed on the CPU oracle
  cpu_baseline   the CPU oracle (port of the reference, oracle/nnj_oracle.py) timed on this box's host cores
  --impl reference : the same oracle as the reference arm (the reference itself needs /root/reference, absent on the GPU box)
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

D, H = 64, 8
WORKLOADS = {
    # name: (taxa, sites, default global batch, metric text)
    "config2": (50, 1024, 512, "trees/sec, 50-taxa x 1024-site Argmax inference"),
    "config4": (200, 4096, 4, "trees/sec, 200-taxa x 4096-site Argmax inference"),
}
UNIT = "trees/s"


def synthetic_msa(batch, taxa, sites, seed):
    """Config-2 generator (SURVEY.md 8d): iid tokens, p(A,C,G,T,-) = (.28,.12,.12,.21,.27) -> one-hot int8, gap = 1111."""
    import torch
    g = torch.Generator().manual_seed(seed)
    p = torch.tensor([0.28, 0.12, 0.12, 0.21, 0.27])
    tok = torch.multinomial(p, batch * taxa * sites, replacement=True, generator=g).view(batch, taxa, sites)
    table = torch.tensor([[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 0], [0, 0, 0, 1], [1, 1, 1, 1]], dtype=torch.int8)
    return table[tok]


def algorithmic_flops(R, Cc, layers=6):
    """Per-tree algorithmic FLOPs per kernel class (2*M*N*K per contraction, elementwise excluded; BASELINE.md section 3).
    NJ classes use the folded formulation the kernels implement (W_h and W_q folded per node, DESIGN.md)."""
    F = 4 * D
    pair_evals = [(R * (R - 1) // 2, R)] + [(n, n) for n in range(R - 1, 1, -1)]     # (pairs, nodes) per step
    fl = {
        "embed": 2 * R * Cc * (4 * D + D * D),
        "ln_qkv": layers * 2 * 3 * 2 * R * Cc * D * D,
        "out_proj": layers * 2 * 2 * R * Cc * D * D,
        "row_qk_gemm": layers * 2 * Cc * Cc * R * D,
        "row_pv_gemm": layers * 2 * Cc * Cc * R * D,
        "col_attn": layers * 4 * Cc * R * R * D,
        "ffn": layers * 4 * R * Cc * D * F,
        "alpha": sum(p * 2 * n * Cc * D for p, n in pair_evals if n > 2),
        "pair_score": sum(p * ((2 * n * Cc * D + 2 * Cc * D * D if n > 2 else 0) + 2 * Cc * D * D + 2 * Cc * D) for p, n in pair_evals),
        "merge": sum(2 * 2 * n * Cc * D + 2 * Cc * D * D + 3 * 2 * Cc * D * D for n in range(R, 2, -1)),   # incl. the merge pair's alpha
        "node_derive": R * 3 * 2 * Cc * D * D,
    }
    return fl


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dirpath, arrays, world=1, rank=0):
    """--dump-outputs: the arrays one timed step returned to its caller (first axis = alignment; under several ranks gathered in
    rank order, i.e. the batch order) as dirpath/<name>.npy in float32 - merge indices are small integers, exact in float32.
    Above DUMP_LIMIT_BYTES in all, the same rows of every array are kept: a sorted sample drawn with seed 0, so that two builds
    run with the same arguments write the same alignments."""
    import numpy as np
    host = {k: v.cpu().numpy().astype(np.float32) for k, v in arrays.items()}
    if world > 1:
        import torch.distributed as dist
        parts = [None] * world
        dist.all_gather_object(parts, host)
        host = {k: np.concatenate([p[k] for p in parts]) for k in host}
    if rank != 0:
        return
    n = next(iter(host.values())).shape[0]
    keep = min(n, DUMP_LIMIT_BYTES // sum(v[:1].nbytes for v in host.values()))
    if keep < n:
        rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        host = {k: v[rows] for k, v in host.items()}
    os.makedirs(dirpath, exist_ok=True)
    for k, v in host.items():
        np.save(os.path.join(dirpath, k + ".npy"), v)


ENC_CLASSES = ("embed", "ln_qkv", "out_proj", "row_qk_gemm", "row_softmax", "row_pv_gemm", "col_attn", "ffn")
NJ_CLASSES = ("node_derive", "alpha", "alpha_softmax", "pair_score", "pair_blend", "select", "merge", "misc")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([t.strip() for t in line.split(",")])

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        if not sm:
            return None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


def _oracle():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import nnj_oracle as O
    return O


def cpu_oracle_run(data, mask, want_merges=None):
    """Time the CPU oracle (port of the reference path) on the given alignments, one per call like the reference (B=1), and -
    when `want_merges` is given - check the device's merge lists against it (identical, or a tie-ambiguous step: replay)."""
    import torch
    O = _oracle()
    sd = O.init_state_dict(0)
    n = data.shape[0]
    identical, tie_ok, worst_gap = 0, 0, None
    t0 = time.perf_counter()
    refs = [O.rollout(sd, data[b:b + 1], mask[b:b + 1]) for b in range(n)]
    dt = time.perf_counter() - t0
    if want_merges is not None:
        for b, ref in enumerate(refs):
            got = want_merges[b:b + 1].long()
            if torch.equal(got, ref["merges"]):
                identical += 1
                continue
            rep = O.rollout(sd, data[b:b + 1], mask[b:b + 1], forced_merges=got)     # teacher-forced replay of OUR trajectory
            slack = max(float(((lg.max(1).values - lg.gather(1, a.unsqueeze(1)).squeeze(1)) / lg.abs().max(1).values).max())
                        for lg, a in zip(rep["logits"], rep["actions"]))
            worst_gap = slack if worst_gap is None else max(worst_gap, slack)
            tie_ok += int(slack < 1e-5)
    return n / dt, dt, torch.get_num_threads(), {"trees": n, "identical_merges": identical, "tie_aware_ok": tie_ok,
                                                  "worst_tie_slack": worst_gap, "tie_tolerance": 1e-5}


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path.  /root/reference is not on the GPU box, so this
    is the oracle port (validated against the executed reference, tests/golden) with all host threads torch will use."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    R, L, _, metric = WORKLOADS[args.workload]
    sample = 1
    mask = torch.zeros(sample, L, dtype=torch.bool)
    for _ in range(args.warmup):
        cpu_oracle_run(synthetic_msa(sample, R, L, 1234), mask)
    t0 = time.perf_counter()
    for k in range(args.steps):
        cpu_oracle_run(synthetic_msa(sample, R, L, 1234 + k), mask)
    dt = time.perf_counter() - t0
    tps = args.steps * sample / dt
    cores = torch.get_num_threads()
    line = {
        "impl": "reference", "metric": metric, "value": tps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": f"configs[1]: synthetic MSAs {R} taxa x {L} sites, Argmax; each step = {sample} alignment (bounded sample, B=1 per call as shipped)"},
        "cpu_baseline": {"value": tps, "unit": UNIT, "cores": cores, "kind": "port", "sample": f"{args.steps} x {sample} alignment(s) of the config-2 generator"},
        "e2e": {"value": tps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def llh_scoring_rate(merges, onehot, R):
    """Search-mode scorer (SURVEY 8 f2) on the side: the first 32 topologies of the timed batch scored on ONE alignment with the GPU
    likelihood (GTR+I+G4, csrc/nnj_llh.cu) - branch lengths only, and with the in-kernel model-parameter search."""
    import numpy as np
    import torch
    from neuralnj_b200 import likelihood as LH
    masks = LH.onehot_to_masks(onehot)
    ch = np.stack([LH.children_from_merges(m, R) for m in merges])
    labels = [f"t{i}" for i in range(R)]
    LH.score_topologies(masks, ch[:2], labels, opt_model=False)
    out = {"topologies": int(ch.shape[0]), "model": "GTR+I+G4, empirical frequencies, fp64"}
    for key, full in (("branch_lengths_only", False), ("with_model_search", True)):
        torch.cuda.synchronize()
        t0 = time.time()
        ll, _ = LH.score_topologies(masks, ch, labels, opt_model=full)
        torch.cuda.synchronize()
        dt = time.time() - t0
        out[key] = {"s": round(dt, 3), "trees_per_s": round(ch.shape[0] / dt, 1), "best_llh": round(float(ll.max()), 3)}
    return out


def write_phylip_files(onehot, dirpath):
    """int8 one-hot alignments [n, R, L, 4] (gap = 1111) -> dirpath/msaNNNN.phy, sequential PHYLIP with taxa named taxon1..taxonR."""
    import numpy as np
    d = onehot.numpy()
    n, R, L = d.shape[:3]
    tok = np.where(d.sum(-1) == 4, 4, d.argmax(-1))
    letters = np.frombuffer(b"ACGT-", dtype=np.uint8)
    os.makedirs(dirpath)
    for b in range(n):
        rows = [f"taxon{r + 1} " + letters[tok[b, r]].tobytes().decode() for r in range(R)]
        with open(os.path.join(dirpath, f"msa{b:04d}.phy"), "w") as f:
            f.write(f"{R} {L}\n" + "\n".join(rows) + "\n")


def directory_inference_rate(model, data_host, R, L, dev):
    """The file-level entry point (`Argmax_inference`, finetune_rl_search.py:478-509) on alignments of the timed batch written as
    PHYLIP files: wall clock over everything a user of the entry point pays - parsing and encoding the files, H2D, the rollout,
    the host tree objects, Newick strings and the .tre files.  `files_per_call_128`: equal-shape alignments stacked into one device
    call; `per_file_loop`: the reference's one-alignment-per-call loop (on 16 of the files)."""
    import tempfile
    import torch
    from neuralnj_b200 import Argmax_inference, inference_config
    n = min(128, data_host.shape[0])
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        dirs = {}
        for label, cnt in (("files_per_call_128", n), ("per_file_loop", min(16, n))):
            dirs[label] = os.path.join(tmp, label)
            write_phylip_files(data_host[:cnt], dirs[label])
        cfgs = inference_config()
        trees = {}
        for label, fpc in (("per_file_loop", 1), ("files_per_call_128", 128)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            written = Argmax_inference(dirs[label], os.path.join(tmp, "out_" + label), None, cfgs=cfgs, device=dev, files_per_call=fpc,
                                       policy_network=model)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            out[label] = {"files": len(written), "s": round(dt, 3), "trees_per_s": round(len(written) / dt, 1)}
            trees[label] = [open(w).read() for w in written]
        k = len(trees["per_file_loop"])
        out["same_trees_as_per_file_loop"] = trees["files_per_call_128"][:k] == trees["per_file_loop"]
    out["note"] = "wall clock incl. PHYLIP parsing, H2D, rollout, host tree objects, Newick and .tre writing; one process, host work not overlapped with the device"
    return out


def supervised_eval_rate(model, data, mask, merges, R):
    """Training step, forward half (SURVEY 8 f3) on the side: the first 128 alignments of the timed batch replayed along their own
    merge lists with teacher forcing (NNJ_SELECT_FORCED, logits trace kept) and ranked by the balanced-ELU loss kernel
    (nnj_rank_loss, action set of a step = the action taken).  Device time, CUDA events."""
    import torch
    from neuralnj_b200.supervise import SupervisedRollout, balanced_elu_loss, trace_offsets
    n = min(128, data.shape[0])
    d, m, f = data[:n].contiguous(), mask[:n].contiguous(), merges[:n].contiguous()
    offs = torch.tensor(trace_offsets(R)[:-1], device=d.device)
    nn = R - torch.arange(R - 1, device=d.device)
    i, j = f[..., 0].long(), f[..., 1].long()
    pidx = i * nn - i * (i + 1) // 2 + (j - i - 1) + offs                      # position of every taken action in the logits trace
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    out = {}
    for it in range(2):                                                        # the second pass is the timed one
        ev[0].record()
        mg, slp, trace = model.rollout_fused(d, m, want_logits=True, forced=f)
        ev[1].record()
        flags = torch.zeros(trace.shape, dtype=torch.uint8, device=d.device)
        flags.scatter_(1, pidx, 1)
        roll = SupervisedRollout(([], [], [], [], [], [], slp))
        roll.trace, roll.in_set, roll.taxa = trace, flags, R
        loss = balanced_elu_loss(roll, epoch=0, ratio_factor=0.5)
        ev[2].record()
        torch.cuda.synchronize()
        assert torch.equal(mg, f)
        out = {"alignments": n, "forced_rollout_ms": round(ev[0].elapsed_time(ev[1]), 2), "loss_ms": round(ev[1].elapsed_time(ev[2]), 3),
               "trees_per_s": round(n / (ev[0].elapsed_time(ev[2]) * 1e-3), 1), "loss": round(loss["loss"], 5), "precision": round(loss["precision"], 5),
               "note": "forward only: supervise_rollout(eval=True) + BALANCED_ELU_LOSS (train.py:43-161, 448-545); no backward pass in this library"}
    return out


def gpu_eager_baseline(dev, R, L, budget_s=40.0):
    """SURVEY 8(d) same-box GPU bar: the reference formulation (the oracle restatement, pure torch ops) run in torch eager
    on this B200 at B = 1 / 8 / 32.  Step 0 is pair-chunked for B > 1 (the reference materialises ~3 GB per tree there)."""
    import torch
    O = _oracle()
    sd = {k: v.to(dev) for k, v in O.init_state_dict(0).items()}
    out = {}
    t_start = time.perf_counter()
    for B in (1, 8, 32):
        if time.perf_counter() - t_start > budget_s:
            break
        data = synthetic_msa(B, R, L, 4321).to(dev)
        mask = torch.zeros(B, L, dtype=torch.bool, device=dev)
        try:
            O.rollout(sd, data, mask, pair_chunk=0 if B == 1 else 128)      # warm (cuBLAS handles, allocator)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            O.rollout(sd, data, mask, pair_chunk=0 if B == 1 else 128)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            out[f"B{B}"] = {"trees_per_s": round(B / dt, 3), "s_per_call": round(dt, 3)}
        except Exception as e:   # noqa: BLE001  (an OOM at B = 32 must not take the bench line down)
            out[f"B{B}"] = {"error": type(e).__name__}
            torch.cuda.empty_cache()
    out["note"] = "oracle/nnj_oracle.py on cuda (torch eager, fp32, TF32 off): the reference's formulation on this GPU, not the product path"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=0, help="GLOBAL alignments per step with --scaling strong, per GPU with weak (default: the workload's)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--workload", default="config2", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="bf16x3", choices=["fp32", "bf16x3", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip latency_b1 / gpu_eager_baseline / the weak-scaling second measurement")
    ap.add_argument("--cpu-trees", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the merge lists and selected log-probabilities of the last timed step "
                    "as DIR/<name>.npy (float32, at most 64 MB: a fixed seeded sample of alignments beyond that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the device path computed: it needs --impl ours")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import __graft_entry__ as graft
    graft.build()
    from neuralnj_b200 import PhyloATTN, inference_config, _lib
    from neuralnj_b200.shard import shard_bounds
    L = _lib.lib()
    R_TAXA, L_SITES, default_batch, METRIC = WORKLOADS[args.workload]
    torch.manual_seed(0)
    model = PhyloATTN(inference_config(), precision=args.precision).to(dev).eval()
    G = args.batch or default_batch                     # global batch (strong) / per-GPU batch (weak)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_inputs(scaling):
        """This rank's alignments.  strong: rows [lo, hi) of ONE global batch (same seed on every rank); weak: its own batch."""
        if scaling == "strong":
            lo, hi = shard_bounds(G, rank, world)
            host = synthetic_msa(G, R_TAXA, L_SITES, 1234)[lo:hi].contiguous().pin_memory()
        else:
            host = synthetic_msa(G, R_TAXA, L_SITES, 1234 + rank).pin_memory()
        mask_h = torch.zeros(host.shape[0], L_SITES, dtype=torch.bool).pin_memory()
        return host, mask_h

    def timed(scaling, steps, warmup, clocks_on):
        data_host, mask_host = make_inputs(scaling)
        data, mask = data_host.to(dev), mask_host.to(dev)
        n_global = G if scaling == "strong" else G * world
        for _ in range(warmup):
            model.rollout_fused(data, mask)
        barrier()
        sampler = ClockSampler(local) if (rank == 0 and clocks_on) else None
        if sampler:
            sampler.start()
        L.nnj_launch_count(1)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            merges, slp, _ = model.rollout_fused(data, mask)
        ev1.record()
        barrier()
        clocks = sampler.stop() if sampler else None
        launches = int(L.nnj_launch_count(0))
        ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms_total = float(ms)
        return {"value": n_global * steps / (ms_total / 1e3), "ms_total": ms_total, "launches": launches, "clocks": clocks, "merges": merges,
                "slp": slp, "data_host": data_host, "mask_host": mask_host, "data": data, "mask": mask, "n_global": n_global}

    main_run = timed(args.scaling, args.steps, args.warmup, True)
    value, ms_total, launches, clocks, merges = (main_run[k] for k in ("value", "ms_total", "launches", "clocks", "merges"))
    data_host, mask_host, data, mask = (main_run[k] for k in ("data_host", "mask_host", "data", "mask"))
    B_local = data_host.shape[0]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"merges": merges, "selected_log_ps": main_run["slp"]}, world, rank)

    # ---- end to end through the host-buffer C-ABI entry point
    model.rollout_host(data_host, mask_host)       # warm
    barrier()
    t0 = time.perf_counter()
    e2e_steps = max(1, min(args.steps, 3))
    for _ in range(e2e_steps):
        mh = model.rollout_host(data_host, mask_host)
    torch.cuda.synchronize()
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_val = main_run["n_global"] * e2e_steps / float(e2e_s)
    assert torch.equal(mh, merges.cpu()), "host entry point and device path disagree"

    # ---- per-kernel-class timing (one extra step with CUDA events around every launch)
    n_cls = L.nnj_profile_classes()
    L.nnj_profile_enable(1)
    model.rollout_fused(data, mask)
    cls_ms = (C.c_double * n_cls)()
    cls_n = (C.c_int64 * n_cls)()
    _lib.check(L.nnj_profile_read(n_cls, cls_ms, cls_n))
    L.nnj_profile_enable(0)
    names = [L.nnj_profile_name(i).decode() for i in range(n_cls)]
    tot_ms = sum(cls_ms)
    fl = algorithmic_flops(R_TAXA, L_SITES)
    B = B_local
    kernels = {n: {"ms": round(cls_ms[i], 3), "launches": int(cls_n[i]), "share": round(cls_ms[i] / tot_ms, 4)} for i, n in enumerate(names) if cls_n[i]}
    top = max((n for n in kernels if n in fl), key=lambda n: kernels[n]["ms"])
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except OSError:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)" if peaks else "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"
    top_flops_per_launch = fl[top] * B / kernels[top]["launches"]
    top_ms_per_launch = kernels[top]["ms"] / kernels[top]["launches"]
    achieved = top_flops_per_launch / (top_ms_per_launch * 1e-3) / 1e12
    roofline = {"bound": "tensor", "kernel": top, "achieved": round(achieved, 3), "peak": peak_tf, "unit": "TFLOP/s",
                "frac": round(achieved / peak_tf, 5), "traffic": None, "peak_source": peak_src,
                "flops_per_launch": top_flops_per_launch, "ms_per_launch": round(top_ms_per_launch, 4),
                "note": "algorithmic (1x) FLOPs against the dense bf16 tensor peak; CUDA-core fp32 kernels and 3x split-bf16 tcgen05 kernels both count 1x"}
    for n in kernels:
        if n in fl:
            kernels[n]["tflops"] = round(fl[n] * B / (kernels[n]["ms"] * 1e-3) / 1e12, 3)
    # DRAM traffic.  The NJ kernels stream only the n live node slots of a step, so their bytes change from step to step: the
    # mean over a rollout comes from the algorithmic byte count (node tiles of the live slots + x planes), which the committed
    # `ncu --set full` captures reproduce within 1 % at the captured launches (profiles/r02_traffic_b128.json).
    roofline_hbm = None
    nj_bytes_per_tree = None
    if args.workload == "config2":
        site_bytes = 256 * L_SITES                           # one fp32 [sites x 64] row set: 256 KB at 1024 sites
        P0 = R_TAXA * (R_TAXA - 1) // 2
        step0_pairs = [256] * (P0 // 256) + ([P0 % 256] if P0 % 256 else [])
        alpha_b = [(3 * R_TAXA + p) * site_bytes for p in step0_pairs] + [(3 * n + n) * site_bytes for n in range(R_TAXA - 1, 2, -1)]
        score_b = [(2 * R_TAXA * (2 if p > 128 else 1) + p) * site_bytes for p in step0_pairs] + [(2 * n + n) * site_bytes for n in range(R_TAXA - 1, 1, -1)]
        merge_b = [(n + 4 + 12) * site_bytes + n * site_bytes for n in range(R_TAXA, 2, -1)]     # k_merge (all nodes + pair + new node's planes) + k_alpha1 (K of all nodes)
        derive_b = 8 * R_TAXA * site_bytes
        nj_bytes_per_tree = sum(alpha_b) + sum(score_b) + sum(merge_b) + derive_b
        if top in ("alpha", "pair_score"):
            per = alpha_b if top == "alpha" else score_b
            roofline["traffic"] = round(sum(per) / len(per) * B / max(1, kernels["node_derive"]["launches"]))
            roofline["traffic_source"] = "mean over the launches of a rollout: algorithmic bytes of the live node slots + x planes (= ncu dram__bytes at the captured launches, profiles/r02_traffic_b128.json)"
        if "alpha" in kernels:
            a_ms = kernels["alpha"]["ms"]
            a_bytes = sum(alpha_b) * B
            roofline_hbm = {"bound": "hbm", "kernel": "alpha", "achieved": round(a_bytes / (a_ms * 1e-3) / 1e9, 1), "peak": hbm_peak,
                            "unit": "GB/s", "frac": round(a_bytes / (a_ms * 1e-3) / 1e9 / hbm_peak, 4), "traffic": round(a_bytes / kernels["alpha"]["launches"]),
                            "ms_per_launch": round(a_ms / kernels["alpha"]["launches"], 4),
                            "note": "k_alpha_v3 over a whole rollout: live node slots (X, Y, K') once + x planes per launch; the late steps (few live nodes) are latency-bound, which pulls the mean below the 6.1-6.3 TB/s of the early launches"}
    enc_ms = sum(kernels[n]["ms"] for n in ENC_CLASSES if n in kernels)
    nj_ms = sum(kernels[n]["ms"] for n in NJ_CLASSES if n in kernels)
    enc_fl = sum(fl[n] for n in ENC_CLASSES if n in fl)
    nj_fl = sum(fl[n] for n in NJ_CLASSES if n in fl)
    step_ms = ms_total / args.steps
    roofline_step = {
        "algorithmic_gflop_per_tree": round((enc_fl + nj_fl) / 1e9, 1),
        "step_tflops": round((enc_fl + nj_fl) * B / (step_ms * 1e-3) / 1e12, 2), "step_frac_of_tensor_peak": round((enc_fl + nj_fl) * B / (step_ms * 1e-3) / 1e12 / peak_tf, 4),
        "encoder": {"ms": round(enc_ms, 2), "tflops": round(enc_fl * B / (enc_ms * 1e-3) / 1e12, 2), "frac_of_tensor_peak": round(enc_fl * B / (enc_ms * 1e-3) / 1e12 / peak_tf, 4)},
        "nj_loop": {"ms": round(nj_ms, 2), "tflops": round(nj_fl * B / (nj_ms * 1e-3) / 1e12, 2), "frac_of_tensor_peak": round(nj_fl * B / (nj_ms * 1e-3) / 1e12 / peak_tf, 4)},
        "precision_note": "bf16x3 executes 3 MMAs per algorithmic product: 100 % tensor-pipe utilisation reads as 0.333 here" if args.precision == "bf16x3" else None,
    }
    if nj_bytes_per_tree:
        stream = sum(n * L_SITES * D * 4 for n in range(2, R_TAXA + 1))        # SURVEY 8(d): state re-read once per step
        roofline_step["nj_loop"].update({"dram_bytes_per_tree": nj_bytes_per_tree, "streaming_bytes_per_tree": stream,
                                         "traffic_ratio": round(nj_bytes_per_tree / stream, 2),
                                         "hbm_gbs": round(nj_bytes_per_tree * B / (nj_ms * 1e-3) / 1e9, 1),
                                         "frac_of_hbm_peak": round(nj_bytes_per_tree * B / (nj_ms * 1e-3) / 1e9 / hbm_peak, 4)})

    extras = {}
    if rank == 0 and not args.no_extras:
        d1, m1 = data[:1].contiguous(), mask[:1].contiguous()
        for _ in range(3):
            model.rollout_fused(d1, m1)
        ts = []
        for _ in range(7):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            model.rollout_fused(d1, m1)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        extras["latency_b1_ms"] = round(sorted(ts)[len(ts) // 2], 3)
        if world == 1:
            extras["gpu_eager_baseline"] = gpu_eager_baseline(dev, R_TAXA, L_SITES, budget_s=40.0 if args.workload == "config2" else 0.0)
        if world == 1 and args.workload == "config2":
            try:        # a side measurement: it must never take the headline line down with it
                extras["tree_llh"] = llh_scoring_rate(merges[:32].cpu().numpy(), data_host[0], R_TAXA)
            except Exception as exc:   # noqa: BLE001
                extras["tree_llh"] = {"error": f"{type(exc).__name__}: {exc}"}
            try:
                extras["supervised_eval"] = supervised_eval_rate(model, data, mask, merges, R_TAXA)
            except Exception as exc:   # noqa: BLE001
                extras["supervised_eval"] = {"error": f"{type(exc).__name__}: {exc}"}
            try:
                extras["directory_inference"] = directory_inference_rate(model, data_host, R_TAXA, L_SITES, dev)
            except Exception as exc:   # noqa: BLE001
                extras["directory_inference"] = {"error": f"{type(exc).__name__}: {exc}"}
    if rank == 0 and world == 1 and not args.no_extras and args.workload == "config2" and args.precision == "bf16x3":
        # The north star's "bf16 encoder" (precision="bf16": one tcgen05 product per encoder contraction, NJ loop unchanged) on the same
        # batch: what the encoder kernels reach without the 3-product split.  NOT the headline - the mode does not keep the reference's
        # Argmax topologies with these weights (DESIGN.md 5); reported so that the split's cost is a measured number.
        try:
            m1p = PhyloATTN(inference_config(), precision="bf16").to(dev).eval()
            m1p.load_state_dict(model.state_dict())
            for _ in range(2):
                m1p.rollout_fused(data, mask)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            for _ in range(2):
                m1p_merges, _, _ = m1p.rollout_fused(data, mask)
            b.record()
            torch.cuda.synchronize()
            ms = a.elapsed_time(b) / 2
            same = int((m1p_merges == merges).all(dim=2).all(dim=1).sum())
            extras["bf16_encoder_mode"] = {"value": round(B_local / (ms * 1e-3), 1), "unit": UNIT, "ms_per_step": round(ms, 2), "steps": 2,
                                           "merge_lists_identical_to_bf16x3": f"{same}/{B_local}",
                                           "note": "precision='bf16' (NNJ_PREC_BF16): scores within 1e-2 relative of the reference, topologies not guaranteed"}
            del m1p
        except Exception as exc:   # noqa: BLE001
            extras["bf16_encoder_mode"] = {"error": f"{type(exc).__name__}: {exc}"}
    weak = None
    if world > 1 and args.scaling == "strong" and not args.no_extras:
        w = timed("weak", max(1, min(args.steps, 3)), 1, False)
        weak = {"value": round(w["value"], 3), "unit": UNIT, "scaling": "weak", "per_gpu_batch": G, "steps": max(1, min(args.steps, 3)),
                "ms_per_step": round(w["ms_total"] / max(1, min(args.steps, 3)), 3)}

    cpu_baseline, parity = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.workload == "config2":
        n = min(args.cpu_trees, B_local)
        tps, secs, cores, parity = cpu_oracle_run(data_host[:n], mask_host[:n], merges[:n].cpu())
        cpu_baseline = {"value": round(tps, 4), "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": f"the first {n} alignments of the timed batch, B=1 per call, {secs:.1f} s"}

    if rank == 0:
        shard = f"{G} alignments per step cut into {world} contiguous shard(s) of {B_local}" if args.scaling == "strong" else f"{G} alignments per GPU per step"
        line = {
            "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(step_ms, 3), "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": {"fp32": "f32", "bf16x3": "bf16x3 (split-bf16 tcgen05, fp32 accumulate) + f32",
                      "bf16": "bf16 encoder (one-product tcgen05, fp32 accumulate) + bf16x3 NJ loop + f32"}[args.precision],
            "data": "synthetic",
            "config": {"workload": f"configs[{1 if args.workload == 'config2' else 3}]: synthetic MSAs, {R_TAXA} taxa x {L_SITES} sites, Argmax, sharded by alignment: {shard}",
                       "global_batch": main_run["n_global"], "parallelism": f"alignment-sharded x{world}, no collectives",
                       "weights": "torch.manual_seed(0) default init (checkpoint blob absent)", "precision": args.precision,
                       "l2": f"inputs_larger_than_l2 ({data_host.numel() / 1e6:.0f} MB int8 MSA + {B_local * R_TAXA * L_SITES * 256 / 1e9:.1f} GB fp32 node state per rank per step)"},
            "e2e": {"value": round(e2e_val, 3), "unit": UNIT, "h2d_bytes_per_step": int(data_host.numel() + mask_host.numel()),
                    "d2h_bytes_per_step": int(mh.numel() * 4), "api": "nnj_rollout_host (C ABI, pinned host buffers, per-chunk staging on a copy stream)", "steps": e2e_steps},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": roofline,
            "roofline_hbm": roofline_hbm,
            "roofline_step": roofline_step,
            "kernels": kernels,
            "cpu_baseline": cpu_baseline,
            "parity_check": parity,
        }
        if weak:
            line["weak"] = weak
        line.update(extras)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
