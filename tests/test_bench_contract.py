"""The bench.py JSON contract (driver side): the committed line of the last GPU run and a live `--impl reference` line
carry every key the driver and the judge read.  CPU only — nothing here touches the CUDA library."""
import json
import os
import subprocess
import sys

from conftest import ROOT

BASE_KEYS = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "e2e", "cpu_baseline"]


def _check_common(d):
    for k in BASE_KEYS:
        assert k in d, k
    assert d["unit"] == "trees/s" and d["higher_is_better"] is True and d["scaling"] in ("strong", "weak") and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["vs_baseline"] is None                      # BASELINE.md publishes no number for this metric
    for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert k in d["e2e"], k
    for k in ("value", "unit", "cores", "kind", "sample"):
        assert k in d["cpu_baseline"], k
    assert d["cpu_baseline"]["kind"] in ("port", "reference")


def test_committed_gpu_line_has_the_contract_keys():
    path = os.path.join(ROOT, "profiles", "r02_bench_final.json")
    if not os.path.exists(path):
        path = os.path.join(ROOT, "profiles", "r01_bench_final.json")
    with open(path) as f:
        d = json.loads(f.read().strip().splitlines()[-1])
    _check_common(d)
    assert d["n_gpus"] == 1 and d["warmup"] >= 3 and d["value"] > 0
    assert d["gpu_launches"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert abs(d["value"] - 512 * 1e3 / d["ms_per_step"]) / d["value"] < 1e-3          # value = trees per step / step time
    for k in ("sm_mhz", "sm_max_mhz", "reasons"):
        assert k in d["clocks"], k
    assert not {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(d["clocks"]["reasons"])
    r = d["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in r, k
    assert r["bound"] in ("hbm", "tensor") and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-3
    assert abs(sum(v["share"] for v in d["kernels"].values()) - 1.0) < 0.01


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.strip().splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    _check_common(d)
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1


def test_dump_outputs_writes_float32_arrays_and_samples_the_same_rows(tmp_path, monkeypatch):
    """--dump-outputs: every array as <name>.npy in float32; above the size limit the same seeded rows of every array."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    merges = torch.arange(40 * 3 * 2, dtype=torch.int32).view(40, 3, 2)
    slp = -torch.rand(40, 3)
    bench.dump_outputs(str(tmp_path / "all"), {"merges": merges, "selected_log_ps": slp})
    m, s = np.load(tmp_path / "all" / "merges.npy"), np.load(tmp_path / "all" / "selected_log_ps.npy")
    assert m.dtype == s.dtype == np.float32 and np.array_equal(m, merges.numpy()) and np.array_equal(s, slp.numpy())
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 10 * (6 + 3) * 4)          # room for 10 of the 40 rows
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"merges": merges, "selected_log_ps": slp})
    m, s = np.load(tmp_path / "a" / "merges.npy"), np.load(tmp_path / "a" / "selected_log_ps.npy")
    assert m.shape == (10, 3, 2) and s.shape == (10, 3)
    rows = (m[:, 0, 0] / 6).astype(int)
    assert list(rows) == sorted(set(rows)) and np.array_equal(s, slp.numpy()[rows])
    assert np.array_equal(m, np.load(tmp_path / "b" / "merges.npy"))


def test_directory_inference_side_measurement_on_the_oracle_stand_in(tmp_path, monkeypatch):
    """bench.py's `directory_inference` extra: synthetic alignments -> PHYLIP files -> `Argmax_inference` per file and stacked.
    The files must read back as the one-hot batch they were written from, and the measurement's bookkeeping is exercised with the
    CPU oracle standing in for the device model (test infrastructure; on the GPU box the bench passes its own model)."""
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from neuralnj_b200 import load_pi_instance
    from test_entry_batched_cpu import OracleAgent
    data = bench.synthetic_msa(3, 6, 64, 7)
    bench.write_phylip_files(data, str(tmp_path / "phy"))
    for b in range(3):
        inst = load_pi_instance(str(tmp_path / "phy" / f"msa{b:04d}.phy"))
        assert torch.equal(inst["data"][0], data[b]) and inst["seq_keys"][0] == [f"taxon{r + 1}" for r in range(6)]
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    out = bench.directory_inference_rate(OracleAgent(), data, 6, 64, torch.device("cpu"))
    assert out["files_per_call_128"]["files"] == 3 and out["per_file_loop"]["files"] == 3
    assert out["same_trees_as_per_file_loop"] is True and out["files_per_call_128"]["trees_per_s"] > 0
