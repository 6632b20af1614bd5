#!/bin/bash
# A/B of the incremental pair-score kernel on one B200: GPU tests of the NJ loop, then per-step launch times and bench.py with the
# parent build (build/ab_old/libnnj.so) and this tree's build alternated, and the benchmark outputs of both compared.
#   bash scratch/r3_score_inc.sh OUT_DIR
set -u
OUT=${1:?usage: r3_score_inc.sh OUT_DIR}
mkdir -p $OUT
OLD=$PWD/build/ab_old/libnnj.so
NEW=$PWD/neuralnj_b200/libnnj.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/card.txt
python -c "import __graft_entry__ as g; g.build()" || exit 1
python -m pytest -q tests/test_gpu_score_inc_tc.py tests/test_gpu_tc_paths.py 2>&1 | tail -40 | tee $OUT/tests.txt
grep -q "failed\|error" $OUT/tests.txt && exit 1
python scratch/score_inc_ab.py $OLD $NEW --rounds 2 --out $OUT/score_inc_ab.txt
for r in 1 2 3; do
  for tag in old new; do
    lib=$OLD; [ $tag = new ] && lib=$NEW
    extra=""; [ $r = 1 ] && extra="--dump-outputs $OUT/dump_$tag"
    NNJ_LIB_PATH=$lib python bench.py --gpus 1 --steps 5 --warmup 3 --no-cpu-baseline --no-extras $extra 2>/dev/null | tail -1 > $OUT/bench_${tag}_$r.json
    echo "$tag $r $(python -c "import json;d=json.load(open('$OUT/bench_${tag}_$r.json'));print(d['value'], d['unit'], 'pair_score', d['kernels']['pair_score']['ms'], 'ms')")"
  done
done
OUT=$OUT python - <<'EOF'
import glob, os, numpy as np
out = os.environ["OUT"]
for f in sorted(glob.glob(os.path.join(out, "dump_old", "*.npy"))):
    a, b = np.load(f), np.load(f.replace("dump_old", "dump_new"))
    rows = (a != b).reshape(a.shape[0], -1).any(1)
    print(os.path.basename(f), "identical" if not rows.any() else
          f"{int(rows.sum())} of {a.shape[0]} alignments differ (rows {np.nonzero(rows)[0][:8].tolist()}), max abs diff {np.abs(a.astype(np.float64) - b).max():.3g}")
EOF
