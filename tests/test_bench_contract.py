"""The bench line contract (task statement, section 4) checked on the committed round-2 measurement, plus bench.py's CLI."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_committed_bench_line_has_every_contract_key():
    d = json.load(open(os.path.join(ROOT, "profiles", "r02_bench_1gpu.json")))
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"):
        assert k in d, k
    assert d["warmup"] >= 3 and d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert "workload" in d["config"] and d["gpu_launches"] > 0
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in d["roofline"], k
    assert abs(d["roofline"]["frac"] - d["roofline"]["achieved"] / d["roofline"]["peak"]) < 1e-9
    for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert k in d["e2e"], k
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["value"] < d["value"]
    for k in ("value", "unit", "cores", "kind", "sample"):
        assert k in d["cpu_baseline"], k
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    pc = d["precision_check"]                      # the default policy inside the north-star tolerance on every output, W included
    assert pc["ok"] is True and max(pc["rel_fro"].values()) <= pc["tolerance"] == 1e-4 and "tf32" in d["dtype"]
    # value is the whole-job aggregate: pairs x LM iterations / time
    cfg = d["config"]
    assert abs(d["value"] - cfg["global_pairs"] * cfg["lm_iterations_per_step"] / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]


def test_bench_cli_parses():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--precision", "--layout", "--e2e-boundary", "--config", "--motion", "--dump-outputs"):
        assert flag in out.stdout
