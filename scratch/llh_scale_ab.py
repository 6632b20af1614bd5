"""A/B of the tree likelihood between two checkouts (e.g. before and after a kernel change), in one process tree on one GPU:
  1. bit-identity: LH.score_topologies on a simulated 50 x 1024 alignment (16 topologies; branch lengths only and with the
     model search) and TreeLikelihood.loglik, from each checkout's own libnnj.so, compared bit for bit;
  2. timing: scratch/llh_time.py and bench.py's tree_llh side figures, the two checkouts alternating.

    python scratch/llh_scale_ab.py OLD_TREE NEW_TREE OUT_DIR [--rounds 2] [--bench-steps 3]

Both trees must be built (python -c "import __graft_entry__ as g; g.build()" in each).  Writes OUT_DIR/ab.json."""
import argparse
import json
import os
import subprocess
import sys

DUMP = r'''
import os, sys
import numpy as np
sys.path.insert(0, os.getcwd()); sys.path.insert(0, os.path.join(os.getcwd(), "oracle"))
import llh_oracle as O
from neuralnj_b200 import likelihood as LH
R, L, B = 50, 1024, 16
rng = np.random.default_rng(9)
gen = O.Model(rates6=(1.2, 3.1, 0.8, 1.1, 4.2, 1.0), freqs=(0.3, 0.2, 0.2, 0.3), alpha=0.7, pinv=0.15)
ch0, bl = O.random_tree(R, rng)
tips = O.simulate(ch0, bl, R, L, gen, rng, gap_frac=0.05)
ch = np.stack([O.random_tree(R, rng)[0] for _ in range(B - 1)] + [ch0])
labels = [f"t{i}" for i in range(R)]
ll_b, t_b = LH.score_topologies(tips, ch, labels, opt_model=False)
ll_a, t_a = LH.score_topologies(tips, ch, labels, opt_model=True)
pats, w = LH.compress_patterns(tips)
sm = LH.SubstModel("GTR+I+G", LH.empirical_freqs(tips), B)
ev = LH.TreeLikelihood(pats, w).loglik(ch, np.stack([bl] * B), sm)
np.savez(sys.argv[1], ll_b=ll_b, t_b=t_b, ll_a=ll_a, t_a=t_a, ev=ev)
'''


def run(cmd, cwd):
    p = subprocess.run(cmd, cwd=cwd, capture_output=True, text=True)
    if p.returncode:
        raise RuntimeError(f"{cmd} in {cwd} failed:\n{p.stdout[-2000:]}\n{p.stderr[-4000:]}")
    return p.stdout


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("out")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--bench-steps", type=int, default=3)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    trees = {"old": os.path.abspath(a.old), "new": os.path.abspath(a.new)}
    res = {"gpu": run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], ".").strip()}
    import numpy as np
    dumps = {}
    for k, tree in trees.items():
        path = os.path.join(os.path.abspath(a.out), f"dump_{k}.npz")
        run([sys.executable, "-c", DUMP, path], tree)
        dumps[k] = np.load(path)
    res["bit_identical"] = {key: bool(np.array_equal(dumps["old"][key], dumps["new"][key])) for key in dumps["old"].files}
    res["max_abs_diff"] = {key: float(np.abs(dumps["old"][key] - dumps["new"][key]).max()) for key in dumps["old"].files}
    print(json.dumps(res), flush=True)
    res["llh_time"], res["bench_tree_llh"] = {"old": [], "new": []}, {"old": [], "new": []}
    for r in range(a.rounds):
        for k, tree in (trees.items() if r % 2 == 0 else reversed(list(trees.items()))):
            res["llh_time"][k].append(run([sys.executable, "scratch/llh_time.py"], tree).strip().splitlines())
            out = run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(a.bench_steps), "--warmup", "1", "--no-cpu-baseline"], tree)
            line = [x for x in out.splitlines() if x.startswith("{")][-1]
            j = json.loads(line)
            res["bench_tree_llh"][k].append({"tree_llh": j.get("tree_llh") or j.get("extras", {}).get("tree_llh"), "value": j.get("value")})
            print(k, r, json.dumps(res["llh_time"][k][-1]), json.dumps(res["bench_tree_llh"][k][-1]), flush=True)
    with open(os.path.join(a.out, "ab.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
