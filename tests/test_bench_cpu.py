"""bench.py's output contract, checked on CPU through the `--impl reference` arm (the only arm that needs no GPU)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_exactly_one_json_line_with_the_contract_keys():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--gaussians", "2000", "--res", "64", "--views", "4"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "views/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "views/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and "workload" in d["config"]


def test_arguments_that_cannot_be_honoured_are_refused():
    """No timed steps, or an output dump from the CPU arm (which returns no GPU outputs), is an argument error."""
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 2 and "error" in out.stderr, (extra, out.stderr[-2000:])
        assert not os.path.exists(os.path.join(ROOT, "unused"))


def test_clock_sampler_degrades_without_nvidia_smi(monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setenv("PATH", "/nonexistent")
    s = bench.ClockSampler(0)
    s.start(wait_s=0.05)
    s.begin(); s.end()
    c = s.stop()
    assert c["samples"] == 0 and c["sm_mhz"] is None and c["reasons"] == []


def test_roofline_accounting_and_strong_scaling_config():
    """The algorithmic-bytes table (SURVEY.md 8d) and the strong-scaling config block, without a GPU."""
    sys.path.insert(0, ROOT)
    import argparse
    import bench
    args = argparse.Namespace(gaussians=300000, views=64, res=1024, sh_degree=3, scene="sample")
    P, K, HW, V, n_vis, D = 300000, 16, 1024, 64, 18_860_897, 69_468_138
    stages = {"preprocess_fwd": (2.8, 5), "scan": (4.5, 5), "binning": (9.6, 5), "blend_fwd": (39.2, 5), "blend_bwd": (81.1, 5),
              "preprocess_bwd": (5.1, 5)}
    r = bench.roofline(args, stages, 143.4, 28.68, 5, P, K, HW, V, n_vis, D)
    assert r["kernel"] == "blend_bwd" and r["bound"] == "fp32_issue" and r["unit"] == "GB/s"
    want = V * HW * HW * 28 + D * 44 + n_vis * 40
    assert r["algorithmic_bytes_per_launch"] == want and abs(r["achieved"] - want / (81.1 / 5 * 1e-3) / 1e9) < 1e-6
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12 and 0 < r["frac"] < 1
    assert r["issue_active_pct"] and r["traffic"] == int(json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["blend_bwd"]["dram_bytes_per_view"] * V)
    assert set(r["stages"]) == set(stages) and abs(sum(s["share_of_step"] for s in r["stages"].values()) - 142.3 / 143.4) < 1e-9
    c8 = bench.workload_config(args, 8)
    assert c8["views_per_gpu"] == 8 and "strong scaling" in c8["parallelism"] and c8["views_per_step"] == 64
    assert bench.workload_config(args, 1)["parallelism"] == "single GPU"
    assert bench.percentiles([3.0, 1.0, 2.0, 10.0])["median"] == 2.5
