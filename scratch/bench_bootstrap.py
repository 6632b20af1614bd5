"""Bootstrap support throughput: 1 000 replicates of the 50 x 1024 example alignment (tests/golden/msa/ex50x1024_73.phy), bf16x3,
seed-0 weights.  Prints one JSON line:
  replicates_per_s          wall clock of bootstrap_support(path, model, 1000) after a warm-up call (host parse + reference rollout
                            included, ends in the host read of the totals)
  stage_ms                  CUDA-event milliseconds summed over the chunks of 128 of the same 1 000 replicates: resampling
                            (nnj_bootstrap_columns), rollouts (nnj_rollout), split distances (nnj_split_distances); each stage
                            starts on an idle device, so host launch overhead is included
  per_chunk_call_ms_back_to_back   the resampling / split-distance call of one chunk, 20 calls queued back to back
  resample_write_gb_per_s   bytes written by one resampling call (128 x 50 x 1024 x 4 = 26 MB) over its back-to-back time; the
                            output fits the 126 MB L2, so this is not an HBM figure
  host_alternative_ms       the same supports from the same merge lists on the host: PhyInferEnv.replay_merges of the 1 000 trees,
                            treeutil.bipartitions of each Newick, transfer distances with Python sets
  gpu, power_limit_w        read in the same run"""
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle")]
import support_oracle as SO                                           # noqa: E402
from neuralnj_b200 import PhyInferEnv, PhyloATTN, empty_config, inference_config, load_pi_instance   # noqa: E402
from neuralnj_b200 import support as SUP                              # noqa: E402

N, SEED = 1000, 0
path = os.path.join(ROOT, "tests", "golden", "msa", "ex50x1024_73.phy")
torch.manual_seed(0)
model = PhyloATTN(inference_config(), precision="bf16x3").cuda().eval()

SUP.bootstrap_support(path, model, SUP.CHUNK, seed=SEED + 1)           # warm-up: every shape of the timed window
torch.cuda.synchronize()
t0 = time.perf_counter()
res = SUP.bootstrap_support(path, model, N, seed=SEED)
wall = time.perf_counter() - t0

inst = load_pi_instance(path)
R, L = inst["data"].shape[1:3]
keys = inst["seq_keys"][0]
data = inst["data"][0].cuda()
mask = (inst["seq_weights"][0] == 0).cuda()
l_eff = int((~mask).sum())
splits, _ = SUP.reference_splits(res["tree"], keys)
splits_dev = SUP.split_bitsets(splits, R).cuda()
ms = {"resample": 0.0, "rollout": 0.0, "split_distances": 0.0}
all_merges = []
with torch.no_grad():
    for r0 in range(0, N, SUP.CHUNK):
        n = min(SUP.CHUNK, N - r0)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        reps = SUP.bootstrap_columns(data, l_eff, SEED, r0, n)
        ev[1].record()
        merges, _, _ = model.rollout_fused(reps, mask.expand(n, L))
        ev[2].record()
        d = SUP.split_distances(merges, splits_dev)
        ev[3].record()
        torch.cuda.synchronize()
        for k, name in enumerate(ms):
            ms[name] += ev[k].elapsed_time(ev[k + 1])
        all_merges.append(merges.cpu())
merges = torch.cat(all_merges)

# the two kernels alone: 20 back-to-back calls on one chunk of 128 replicates (no host synchronisation in between)
mg0 = all_merges[0].cuda()
K = 20
per_call = {}
for name, fn in (("resample", lambda: SUP.bootstrap_columns(data, l_eff, SEED, 0, SUP.CHUNK)),
                 ("split_distances", lambda: SUP.split_distances(mg0, splits_dev))):
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(K):
        fn()
    b.record()
    torch.cuda.synchronize()
    per_call[name] = a.elapsed_time(b) / K
resample_gbps = SUP.CHUNK * R * L * 4 / (per_call["resample"] * 1e-3) / 1e9

t0 = time.perf_counter()
env = PhyInferEnv(empty_config(), torch.device("cpu"))
env.init_states(inst["seqs"] * N, inst["seq_keys"] * N, None)
env.replay_merges(merges)
host = SO.support_from_newicks(res["tree"], [st.subtrees[0].utree_op_str for st in env.states])
host_ms = 1e3 * (time.perf_counter() - t0)
same = all((float(f), float(t)) == host[sp] for sp, f, t in zip(res["splits"], res["fbp"], res["tbe"]))

try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
    power = float(q[1])
except Exception:
    power = None
print(json.dumps({"workload": "bootstrap_support ex50x1024_73 (50 taxa x 1024 sites), bf16x3", "n_replicates": N, "chunk": SUP.CHUNK,
                  "replicates_per_s": round(N / wall, 1), "wall_s": round(wall, 3),
                  "stage_ms": {k: round(v, 2) for k, v in ms.items()},
                  "per_chunk_call_ms_back_to_back": {k: round(v, 4) for k, v in per_call.items()},
                  "resample_write_gb_per_s": round(resample_gbps, 1),
                  "host_alternative_ms": round(host_ms, 1), "host_alternative_equal": same,
                  "splits": len(splits), "fbp_mean": round(float(res["fbp"].mean()), 2), "tbe_mean": round(float(res["tbe"].mean()), 4),
                  "gpu": torch.cuda.get_device_name(0), "power_limit_w": power}))
