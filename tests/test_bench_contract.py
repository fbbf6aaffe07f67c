"""CPU: bench.py's contract pieces that need no GPU -- workload table, CPU-sample planning, and the reference arm's
JSON line (run as a subprocess on a tiny sample)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_workload_table_covers_the_baseline_configs():
    sys.path.insert(0, ROOT)
    import bench
    from pymc_b200 import models

    assert set(bench.WORKLOADS) == {"radon", "logistic", "stochvol", "mvgauss"}
    for name, wl in bench.WORKLOADS.items():
        assert wl["builder"] in models.BUILDERS and wl["bound"] in ("onchip", "tensor") and wl["scaling"] in ("weak", "strong")
        assert wl["per_eval"] > 0 and wl["chains"] > 0
    # SURVEY 8(d): Radon algorithmic bytes per grad-eval = 919 (8+8+4) + 7 * 175 * 8
    assert bench.WORKLOADS["radon"]["per_eval"] == 28180
    assert bench.WORKLOADS["radon"]["chains"] == 2048 and bench.WORKLOADS["mvgauss"]["scaling"] == "strong"


def test_roofline_objects():
    sys.path.insert(0, ROOT)
    import bench

    wl = bench.WORKLOADS["radon"]
    r = bench.make_roofline("radon", wl, per_launch=9.0e7, k_ms=500.0, fp64=36.0, dmma=37.0, peaks=(6563.9, "measured"),
                            traffic=(5.3e9, "ncu"))
    # the top level is the BINDING resource of the on-chip kernels: the fp64 pipe (VERDICT r1 weak #3)
    assert r["bound"] == "fp64" and r["unit"] == "TFLOP/s" and r["peak"] == 36.0 and r["traffic"] == 5.3e9
    assert abs(r["achieved"] - (919 * 30 + 175 * 12) * 9.0e7 / 0.5 / 1e12) < 1e-9 and abs(r["frac"] - r["achieved"] / 36.0) < 1e-12
    h = r["hbm_by_algorithmic_bytes"]  # SURVEY 8(d)'s second figure, secondary
    assert h["unit"] == "GB/s" and abs(h["achieved"] - 28180 * 9.0e7 / 0.5 / 1e9) < 1e-6 and h["peak_source"] == "measured"
    assert abs(h["frac"] - h["achieved"] / 6563.9) < 1e-12 and h["dram_bytes_measured"] == 5.3e9
    assert bench.make_roofline("radon", wl, 9.0e7, 500.0, None, None, (6650.0, "fallback"), None)["peak"] == 36.0
    t = bench.make_roofline("logistic", bench.WORKLOADS["logistic"], per_launch=4.0e5, k_ms=12000.0, fp64=36.0, dmma=37.0,
                            peaks=(6563.9, "measured"), traffic=None)
    assert t["bound"] == "tensor" and t["unit"] == "TFLOP/s" and abs(t["achieved"] - 512e6 * 4.0e5 / 12.0 / 1e12) < 1e-9
    assert t["peak"] == 37.0 and t["traffic"] is None
    assert bench.make_roofline("mvgauss", bench.WORKLOADS["mvgauss"], 1e5, 1e4, None, None, (6563.9, "measured"), None)["peak"] == 37.0
    json.dumps([r, t])


def test_dump_outputs_writes_a_fixed_bounded_sample(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    import numpy as np
    import torch

    from pymc_b200.engine import NutsResult

    C, T, n = 50, 7, 3
    g = torch.Generator().manual_seed(0)
    res = NutsResult(draws=torch.randn(C, T, n, generator=g, dtype=torch.float64),
                     stats={"tree_size": torch.randint(1, 64, (C, T), generator=g, dtype=torch.int32),
                            "diverging": torch.zeros(C, T, dtype=torch.uint8)},
                     summary={"grad_evals": torch.arange(C, dtype=torch.int64), "final_var": torch.ones(C, n, dtype=torch.float64)},
                     kernel_ms=0.0, launches=1, tune=0, n_draws=T, store_warmup=False)
    bench.dump_outputs(res, str(tmp_path / "all"))
    out = {p.stem: np.load(p) for p in (tmp_path / "all").iterdir()}
    assert set(out) == {"chains", "draws", "stat_tree_size", "stat_diverging", "summary_grad_evals", "summary_final_var"}
    assert all(a.dtype == np.float64 for a in out.values())
    assert np.array_equal(out["chains"], np.arange(C)) and np.array_equal(out["draws"], res.draws.numpy())
    assert np.array_equal(out["stat_tree_size"], res.stats["tree_size"].numpy())
    # above the cap: the same seeded chains in every array, and no more bytes than the cap
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096 * 6 + 10 * 8 * (T * n + 2 * T + 1 + n + 1))
    for d in ("a", "b"):
        bench.dump_outputs(res, str(tmp_path / d))
    a = {p.stem: np.load(p) for p in (tmp_path / "a").iterdir()}
    b = {p.stem: np.load(p) for p in (tmp_path / "b").iterdir()}
    idx = a["chains"].astype(int)
    assert len(idx) == 10 and np.all(np.diff(idx) > 0) and all(np.array_equal(a[k], b[k]) for k in a)
    assert np.array_equal(a["draws"], res.draws.numpy()[idx]) and np.array_equal(a["summary_grad_evals"], idx)
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= bench.DUMP_BYTES


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-chains", "2", "--tune", "6", "--draws", "8"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "leapfrog_grad_evals_per_sec" and line["unit"] == "grad-evals/s"
    assert line["value"] > 0 and line["higher_is_better"] is True and line["gpu_launches"] == 0
    assert line["e2e"]["value"] == line["value"] and line["e2e"]["h2d_bytes_per_step"] == 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    cb = line["cpu_baseline"]  # pinned workers, single-core rate and the linear expectation next to the measured rate
    assert cb["pinned"] and cb["single_core_evals_per_s"] > 0 and 0 < cb["parallel_efficiency"] < 4
    assert line["config"]["workload"].startswith("radon_hierarchical")
    ess = line["cpu_baseline"]["ess"]  # ESS/s of the CPU sample, same estimator as the GPU line
    assert ess["chains"] == 2 and ess["draws"] == 8 and ess["ess_per_sec"] > 0


def test_reference_arm_is_silent_on_nonzero_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
