"""Timing of the tree topology test (nnj_llh_topology_test, DESIGN.md 13) on one GPU, with the card's name, power limit and max SM clock
read in the same run.

    python scratch/bench_topotest.py OUT.json [--reps 3]

Shapes: one 50-taxon alignment of 1024 simulated sites, K = 16, 64 and 256 candidate trees (the generating tree and random ones),
N = 10 000 replicates per scale, GTR+I+G.  Per K: optimize_all of the K trees and the whole topology_test call (CUDA events, after one
warm-up call of the same shape), and in a separate profiled call the kernel time of k_topo_totals alone (torch.profiler, CUDA
activities).  Derived: the fp64 multiply-adds of the totals, 11 N K P (ten scales and the second pass over scale 5), over that kernel
time.  Also the numpy oracle's statistics (oracle/topotest_oracle.py) on the K = 64 per-pattern log-likelihoods at N = 200, on the
host CPU."""
import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import llh_oracle as O  # noqa: E402
import topotest_oracle as TO  # noqa: E402

from neuralnj_b200 import likelihood as LH  # noqa: E402

GEN = dict(rates6=(1.2, 3.1, 0.8, 1.1, 4.2, 1.0), freqs=(0.3, 0.2, 0.2, 0.3), alpha=0.7, pinv=0.15)
N = 10000


def model(K):
    sm = LH.SubstModel("GTR+I+G", np.asarray(GEN["freqs"]), K)
    sm.rates[:] = GEN["rates6"]
    sm.alpha[:] = GEN["alpha"]
    sm.pinv[:] = GEN["pinv"]
    return sm


def timed(fn, reps):
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return out


def kernel_ms(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ms, launches = {}, {}
    for ev in prof.events():
        m = re.search(r"\b(k_topo_totals|k_topo_stats|k_topo_sums|k_rell_counts|k_llh)\(", ev.name)
        if m and ev.device_type.name == "CUDA":
            ms[m.group(1)] = ms.get(m.group(1), 0.0) + (ev.device_time if hasattr(ev, "device_time") else ev.cuda_time) / 1000.0
            launches[m.group(1)] = launches.get(m.group(1), 0) + 1
    return ms, launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    res = {"gpu": gpu, "n_boot": N, "shapes": []}
    print(gpu, flush=True)
    rng = np.random.default_rng(5)
    R, L = 50, 1024
    ch0, bl0 = O.random_tree(R, rng)
    tips = O.simulate(ch0, bl0, R, L, O.Model(**GEN), rng, gap_frac=0.05)
    pats, w = O.compress_patterns(tips)
    P = pats.shape[1]
    eng = LH.TreeLikelihood(pats, w)
    for K in (16, 64, 256):
        trees = [(ch0, bl0)] + [O.random_tree(R, rng) for _ in range(K - 1)]
        ch, bl = np.stack([t[0] for t in trees]), np.stack([t[1] for t in trees])
        t_fit = timed(lambda: eng.optimize_all(ch, bl, model(K)), 1 + a.reps)[1:]
        sm = model(K)
        fit, _, _ = eng.optimize_all(ch, bl, sm)
        call = lambda: eng.topology_test(ch, fit, sm, N, 1)      # noqa: E731
        t_warm = timed(call, 1)[0]
        t = timed(call, a.reps)
        ms, launches = kernel_ms(call)
        madds = 11 * N * K * P
        row = dict(R=R, sites=L, patterns=P, K=K, n_boot=N, optimize_all_ms=t_fit, warmup_ms=t_warm, call_ms=t, kernel_ms=ms, launches=launches,
                   totals_mul_add=madds, totals_gmuladd_per_s=madds / (ms["k_topo_totals"] * 1e-3) / 1e9)
        res["shapes"].append(row)
        print(json.dumps(row), flush=True)
        if K == 64:
            site = eng.topology_test(ch, fit, sm, 10, 1, site_llh=True)["site_llh"].cpu().numpy()
            t0 = time.perf_counter()
            TO.topology_test(site, w, 200, 1)
            res["oracle_cpu_K64_N200_s"] = time.perf_counter() - t0
            print(json.dumps({"oracle_cpu_K64_N200_s": res["oracle_cpu_K64_N200_s"]}), flush=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
