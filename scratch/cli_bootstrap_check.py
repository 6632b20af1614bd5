"""CLI check of --bootstrap: a directory run with --files_per_call 128 --bootstrap 100 writes the .tre files of a run without
--bootstrap, plus <name>.fbp.tre / <name>.tbe.tre whose labels strip off to the .tre.  Seed-0 weights through a checkpoint so that
both runs use the same model.  Works in a temporary directory; prints one JSON line."""
import json
import os
import shutil
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from neuralnj_b200 import PhyloATTN, inference_config           # noqa: E402
from neuralnj_b200.support import strip_support_labels         # noqa: E402

tmp = tempfile.mkdtemp()
msas = os.path.join(tmp, "msas")
os.makedirs(msas)
names = ["ex50x1024_73", "ex50x1024_71", "t20x256_10", "t20x256_103"]
for n in names:
    shutil.copyfile(os.path.join(ROOT, "tests", "golden", "msa", n + ".phy"), os.path.join(msas, n + ".phy"))
torch.manual_seed(0)
torch.save({"model_state_dict": PhyloATTN(inference_config()).state_dict()}, os.path.join(tmp, "w.pt"))
with open(os.path.join(tmp, "cfg.yaml"), "w") as f:
    f.write(f"instance_path: {msas}\nreload_checkpoint_path: {os.path.join(tmp, 'w.pt')}\nenv:\n  batch_size: 1\n"
            "model:\n  vocab_size: 4\n  patch_size: 1\n  embed_dim: 64\n  num_enc_heads: 8\n  num_enc_layers: 6\n")
out = {}
for tag, extra in (("plain", []), ("boot", ["--bootstrap", "100", "--bootstrap_seed", "3"])):
    wd = os.path.join(tmp, tag)
    os.makedirs(wd)
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-m", "neuralnj_b200.rollout", "--config_path", os.path.join(tmp, "cfg.yaml"), "--files_per_call", "128"]
                       + extra, cwd=wd, env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    out[tag] = os.path.join(wd, "output", "Argmax_dim64_patch1", "msas")
ok = {}
for n in names:
    tre = open(os.path.join(out["plain"], n + ".tre")).read()
    same = open(os.path.join(out["boot"], n + ".tre")).read() == tre
    strips = all(strip_support_labels(open(os.path.join(out["boot"], f"{n}.{k}.tre")).read()) == tre for k in ("fbp", "tbe"))
    ok[n] = same and strips
print(json.dumps({"cli_bootstrap_check": ok, "files": sorted(os.listdir(out["boot"]))}))
shutil.rmtree(tmp)
assert all(ok.values())
