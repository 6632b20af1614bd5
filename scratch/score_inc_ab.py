"""Per-step times of the incremental pair-score launches (k_score_inc / k_score_small) of one 128-tree chunk, two builds alternated.

    python scratch/score_inc_ab.py OLD_LIB NEW_LIB --out FILE [--rounds 2]

Each round runs one child process per build (NNJ_LIB_PATH selects the library): a warm-up rollout of 128 alignments of 50 taxa x 1024
sites, then one rollout under torch.profiler; the child prints the pair-score kernels of that rollout in launch order.  The table gives,
per NJ step (live nodes n = 50 - t), the median over rounds of each build's launch time.  Card name and power limit head the output."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def child():
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import torch
    import nnj_oracle as O
    from neuralnj_b200 import PhyloATTN, inference_config
    torch.manual_seed(0)
    model = PhyloATTN(inference_config(), precision="bf16x3").to("cuda:0").eval()
    data = O.evolved_msa(128, 50, 1024, seed=11).cuda()
    mask = torch.zeros(128, 1024, dtype=torch.bool, device="cuda")
    model.rollout_fused(data, mask)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        model.rollout_fused(data, mask)
        torch.cuda.synchronize()
    ev = [(e.time_range.start, e.name, e.time_range.end - e.time_range.start) for e in prof.events()
          if e.device_type == torch.autograd.DeviceType.CUDA and e.name.startswith(("void nnj::k_score_inc", "void nnj::k_score_small", "nnj::k_score_inc", "nnj::k_score_small"))]
    ev.sort()
    print(json.dumps([[n.split("(")[0].split("<")[0].replace("void ", ""), d] for _, n, d in ev]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    runs = {"old": [], "new": []}
    for _ in range(args.rounds):
        for tag in ("old", "new"):
            env = dict(os.environ, NNJ_LIB_PATH=os.path.abspath(getattr(args, tag)))
            r = subprocess.run([sys.executable, __file__, "--child"], env=env, capture_output=True, text=True, cwd=ROOT)
            if r.returncode:
                sys.exit(f"{tag} child failed:\n{r.stdout}\n{r.stderr}")
            runs[tag].append(json.loads(r.stdout.strip().splitlines()[-1]))
    lines = [f"card: {card}", "128 trees x 50 taxa x 1024 sites, bf16x3; times in us (median over %d rounds per build, builds alternated)" % args.rounds,
             f"{'step':>4} {'n':>3} {'old kernel':>14} {'old us':>8} {'new kernel':>14} {'new us':>8}"]
    steps = min(len(runs["old"][0]), len(runs["new"][0]))
    tot = {"old": 0.0, "new": 0.0}
    for i in range(steps):
        row = {}
        for tag in ("old", "new"):
            row[tag] = (runs[tag][0][i][0], statistics.median(r[i][1] for r in runs[tag]))
            tot[tag] += row[tag][1]
        lines.append(f"{i + 1:>4} {50 - (i + 1):>3} {row['old'][0]:>14} {row['old'][1]:>8.1f} {row['new'][0]:>14} {row['new'][1]:>8.1f}")
    lines.append(f"sum of {steps} launches: old {tot['old'] / 1000:.2f} ms, new {tot['new'] / 1000:.2f} ms")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    if "--child" in sys.argv:
        child()
    else:
        main()
