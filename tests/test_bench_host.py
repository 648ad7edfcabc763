"""Host-side logic of bench.py and the profiling tools (no GPU): the per-kernel work model and roofline bound, the
JSON contract keys of the reference arm, and the ncu kernel-name -> bench-name mapping."""
import importlib.util
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load(path, name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, path))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


bench = load("bench.py", "bench_mod")
PEAKS = {"hbm_gbs": 6454.0, "bf16_tflops": 1673.6, "bf16_tflops_sustained": 1395.3, "source": "test"}


def test_kernel_work_matches_survey_totals():
    # SURVEY 8d closed forms at G416, one frame, bf16: LKPM = 2 N C k^2 + 16 N C^2, depthwise 870 MFLOP at L1
    dw = bench.kernel_work("dwconv_tc<31>", 1, 2)
    assert abs(dw["flops"] - 2 * 14144 * 32 * 961) < 1 and dw["bound"] == "tensor"
    mlp = bench.kernel_work("lkpm_mlp_tc<32>", 1, 2)
    assert abs(mlp["flops"] - 16 * 14144 * 32 * 32) < 1
    assert bench.kernel_work("layout_kernel", 1, 2)["flops"] == 0
    assert bench.kernel_work("no_such_kernel", 1, 2) is None


def test_roofline_bound_is_the_slower_of_hbm_and_tensor():
    dw = bench.roofline_of("dwconv_tc<31>", 130e-6, 64, 2, PEAKS)          # 961 taps per element: tensor-bound
    assert dw["bound"] == "tensor" and 0.25 < dw["frac"] < 0.35 and dw["unit"] == "TFLOP/s"
    mlp = bench.roofline_of("lkpm_mlp_tc<32>", 90e-6, 64, 2, PEAKS)        # 85 flop/byte < ridge (216): HBM-bound
    assert mlp["bound"] == "hbm" and mlp["unit"] == "GB/s" and 0.25 < mlp["frac"] < 0.35
    lay = bench.roofline_of("layout_kernel", 30e-6, 64, 2, PEAKS)
    assert lay["bound"] == "hbm" and lay["frac"] is not None
    assert bench.roofline_of("unknown", 1e-3, 64, 2, PEAKS)["frac"] is None


def test_committed_traffic_file_names_bench_kernels():
    traffic = bench.load_ncu_traffic()
    assert traffic, "profiles/ncu_traffic.json missing or empty"
    for name in ("dwconv_tc<31>", "lkpm_mlp_tc<32>", "conv3x3_tc<2C->C,32>", "loftr_query_tc<lsa,32>", "kv_state_tc<hist2image,128>",
                 "attn_query_tc<dapm,64>", "layout_kernel", "hist_encoder_tc"):
        assert name in traffic and traffic[name] > 0, name
        assert bench.kernel_work(name, 64, 2) is not None, name          # every captured kernel has a work model


def test_peaks_file_or_fallback():
    p = bench.load_peaks()
    assert p["hbm_gbs"] > 1000 and p["bf16_tflops_sustained"] > 100 and p["source"]


def test_committed_bench_line_carries_the_whole_contract():
    """The driver's contract for the JSON line (keys and their meaning), checked on the committed final line of the
    round; bench.py prints the same dict."""
    import json
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    d = json.load(open(os.path.join(root, "profiles", "r1s_bench_final.json")))
    baseline = json.load(open(os.path.join(root, "BASELINE.json")))
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline"):
        assert k in d, k
    assert baseline["metric"].startswith(d["metric"]) and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["warmup"] >= 3 and d["n_gpus"] == 1 and d["dtype"] == "bf16"
    assert "workload" in d["config"] and "model" not in d["config"] and "l2_policy" in d["config"]
    assert abs(d["value"] - d["config"]["global_batch"] * d["steps"] / (d["ms_per_step"] * d["steps"] * 1e-3)) <= 1e-6 * d["value"]
    e = d["e2e"]
    assert e["unit"] == d["unit"] and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and 0 < e["value"] < d["value"]
    assert d["gpu_launches"] > 0 and d["gpu_launches"] % d["steps"] == 0
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["unit"] in ("GB/s", "TFLOP/s")
    assert abs(r["frac"] - r["achieved"] / r["peak"]) <= 1e-9 and 0 < r["frac"] <= 1 and r["traffic"] is None or r["traffic"] > 0
    c = d["cpu_baseline"]
    assert c["kind"] in ("port", "reference") and c["cores"] >= 1 and c["value"] > 0 and c["unit"] == d["unit"] and c["sample"]


def test_dump_outputs_stays_in_budget_and_repeats(tmp_path, monkeypatch):
    """--dump-outputs: float32 files, full arrays under the budget, above it the same seeded positions on every run."""
    import numpy as np
    import torch
    small = [("a", torch.arange(6, dtype=torch.bfloat16).reshape(2, 3)), ("b", torch.ones(4))]
    assert bench.dump_outputs(str(tmp_path / "full"), small) == 1.0
    a = np.load(tmp_path / "full" / "a.npy")
    assert a.dtype == np.float32 and a.shape == (2, 3) and np.array_equal(a, np.arange(6).reshape(2, 3))
    monkeypatch.setattr(bench, "DUMP_BYTES", 2 * 1024 + 4 * 3000)
    big = [("x", torch.randn(2, 4, 500)), ("y", torch.randn(8000))]
    for run in ("r1", "r2"):
        share = bench.dump_outputs(str(tmp_path / run), big)
        assert 0 < share < 1
    total = 0
    for name, t in big:
        s1, s2 = np.load(tmp_path / "r1" / f"{name}.npy"), np.load(tmp_path / "r2" / f"{name}.npy")
        assert s1.dtype == np.float32 and np.array_equal(s1, s2) and np.isin(s1, t.numpy()).all()
        total += os.path.getsize(tmp_path / "r1" / f"{name}.npy")
    assert total <= bench.DUMP_BYTES


def test_reference_arm_runs_on_rank_zero_only():
    """Under torchrun the CPU arm is rank 0's job: every other rank exits 0 without work and without output."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "1"], env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""
