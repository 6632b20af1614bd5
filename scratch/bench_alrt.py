"""Timing of likelihood branch support (nnj_llh_branch_support, DESIGN.md 12) on one GPU, with the card's name and power limit read
in the same run.

    python scratch/bench_alrt.py OUT.json [--reps 3]

Shapes: 50 taxa x 1024 patterns at B = 1 and B = 64, 200 x 4096 at B = 1; N = 1000 RELL replicates; simulated data, random trees,
GTR+I+G with fixed parameters.  Per shape: the whole call (CUDA events, after one warm-up call of the same shape), its three stages
from torch.profiler kernel times in a separate profiled call (prepare = llh_prepare's k_llh launch, NNI = k_llh_nni, RELL = k_rell_counts + k_rell),
and beside them optimize_all and optimize_branches of the same trees.  Also the numpy oracle (oracle/alrt_oracle.py) on one
50-taxon tree, on the host CPU."""
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
import alrt_oracle as A  # noqa: E402
import llh_oracle as O  # noqa: E402

from neuralnj_b200 import likelihood as LH  # noqa: E402

GEN = dict(rates6=(1.2, 3.1, 0.8, 1.1, 4.2, 1.0), freqs=(0.3, 0.2, 0.2, 0.3), alpha=0.7, pinv=0.15)
STAGES = {"k_llh": "prepare", "k_llh_nni": "nni", "k_rell_counts": "rell", "k_rell": "rell"}


def data(R, L, B, seed):
    rng = np.random.default_rng(seed)
    ch0, bl0 = O.random_tree(R, rng)
    tips = O.simulate(ch0, bl0, R, L, O.Model(**GEN), rng, gap_frac=0.05)
    chs, bls = zip(*[O.random_tree(R, rng) for _ in range(B - 1)]) if B > 1 else ((), ())
    ch = np.stack([ch0, *chs])
    bl = np.stack([bl0, *bls])
    return tips, ch, bl


def model(B):
    sm = LH.SubstModel("GTR+I+G", np.asarray(GEN["freqs"]), B)
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


def stages(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ms = {"prepare": 0.0, "nni": 0.0, "rell": 0.0}
    for ev in prof.events():
        m = re.search(r"\b(k_llh_nni|k_rell_counts|k_rell|k_llh)\(", ev.name)      # "void nnj::(anonymous namespace)::k_rell(...)"
        if m and ev.device_type.name == "CUDA":
            ms[STAGES[m.group(1)]] += (ev.device_time if hasattr(ev, "device_time") else ev.cuda_time) / 1000.0
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    res = {"gpu": gpu, "n_rell": 1000, "shapes": []}
    print(gpu, flush=True)
    for R, L, B in ((50, 1024, 1), (50, 1024, 64), (200, 4096, 1)):
        tips, ch, bl = data(R, L, B, seed=R + B)
        eng = LH.TreeLikelihood(tips, np.ones(L))
        sm = model(B)
        call = lambda: eng.nni_support(ch, bl, sm, 1000, 1)       # noqa: E731
        t_warm = timed(call, 1)[0]
        t = timed(call, a.reps)
        st = stages(call)
        t_all = timed(lambda: eng.optimize_all(ch, bl, model(B)), a.reps)
        t_br = timed(lambda: eng.optimize_branches(ch, bl, sm), a.reps)
        row = dict(R=R, patterns=L, B=B, branches=R - 3, ctas_nni=2 * B * (R - 3), warmup_ms=t_warm, call_ms=t, stage_ms=st,
                   optimize_all_ms=t_all, optimize_branches_ms=t_br)
        res["shapes"].append(row)
        print(json.dumps(row), flush=True)
    tips, ch, bl = data(50, 1024, 1, seed=51)
    t0 = time.perf_counter()
    A.branch_support(ch[0], bl[0], tips, np.ones(1024), O.Model(**GEN), 1000, 1)
    res["oracle_cpu_50x1024_s"] = time.perf_counter() - t0
    print(json.dumps({"oracle_cpu_50x1024_s": res["oracle_cpu_50x1024_s"]}), flush=True)
    with open(a.out, "w") as f:
        json.dump(res, f)


if __name__ == "__main__":
    main()
