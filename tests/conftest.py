import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

ALL_CASES = ["ex50x1024_73", "ex50x1024_71", "t20x256_10", "t20x256_103", "t20x256_104", "t20x256_117", "t20x256_120",
             "t50x256_a", "t100x256_a", "t20x512_a", "t50x512_a", "batch2_20x256", "padded_20x256",
             "tiny_3x64", "tiny_4x96", "tiny_5x128"]
SMALL_CASES = [c for c in ALL_CASES if not c.startswith(("ex50", "t100", "t50x512"))]


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


class Golden:
    """One record written by oracle/make_golden.py from the executed reference."""

    def __init__(self, name):
        z = np.load(os.path.join(GOLD, name + ".npz"), allow_pickle=False)
        self.name = name
        self.data = torch.from_numpy(z["data"])
        self.mask = torch.from_numpy(z["seq_mask"])
        self.merges = torch.from_numpy(z["merges"]).long()
        off = z["logit_offsets"]
        lg = torch.from_numpy(z["logits"])
        self.logits = [lg[:, off[k]:off[k + 1]] for k in range(len(off) - 1)]
        self.logits_flat = lg
        self.selected_log_ps = torch.from_numpy(z["selected_log_ps"])
        self.state_sample = torch.from_numpy(z["state_sample"])
        self.newick = [str(s) for s in z["newick"]]
        self.seq_keys = [[str(k) for k in row] for row in z["seq_keys"]]


@pytest.fixture(scope="session")
def golden():
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = Golden(name)
        return cache[name]
    return get


@pytest.fixture(scope="session")
def sd0():
    import nnj_oracle as O
    return O.init_state_dict(0)


@pytest.fixture(scope="session")
def gpu_models():
    """One model per precision mode, same seed-0 weights: fp32 CUDA-core path and tcgen05 split-bf16 path."""
    from neuralnj_b200 import PhyloATTN, inference_config
    import __graft_entry__ as g
    g.build()
    out = {}
    for prec in ("fp32", "bf16x3"):
        torch.manual_seed(0)
        out[prec] = PhyloATTN(inference_config(), precision=prec).to("cuda:0").eval()
    return out


@pytest.fixture(scope="session")
def gpu_model(gpu_models):
    return gpu_models["fp32"]


@pytest.fixture(scope="session")
def parity_report():
    """Collects one entry per (case, precision) from the GPU parity tests and, when the session ends, writes them to the file named
    by NNJ_PARITY_REPORT (e.g. profiles/r02_parity.json; unset: nothing is written, so a test run leaves the tree untouched): how
    each case passed ("strict" = merge list identical to the reference / oracle, "tie_aware" = teacher-forced replay), the
    record's own minimum relative top-1/top-2 gap, and the largest relative logit error seen."""
    import json
    rep = {}
    yield rep
    dst = os.environ.get("NNJ_PARITY_REPORT")
    if not rep or not dst:
        return
    out = {"tolerances": {"logit_rel": 2e-5, "tie_rel": {"fp32": 1e-6, "bf16x3": 1e-5}},
           "summary": {}, "cases": dict(sorted(rep.items()))}
    for prec in sorted({v["precision"] for v in rep.values()}):
        rows = [v for v in rep.values() if v["precision"] == prec]
        out["summary"][prec] = {"cases": len(rows), "strict": sum(r["mode"] == "strict" for r in rows),
                                "tie_aware": sum(r["mode"] == "tie_aware" for r in rows),
                                "max_logit_rel_err": max((r["max_logit_rel_err"] for r in rows if r["max_logit_rel_err"] is not None), default=None)}
    os.makedirs(os.path.dirname(os.path.abspath(dst)), exist_ok=True)
    with open(dst, "w") as f:
        json.dump(out, f, indent=1)
