#!/usr/bin/env python
"""bench.py -- leapfrog gradient-evaluations/sec of the NUTS hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # the CUDA engine (this repo)
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host cores

`--workload {radon,logistic,stochvol,mvgauss}` selects the BASELINE config (default: #2, the one the metric is quoted
on for a single GPU; the defaults of the others are sized so a step takes seconds).
One "step" = one complete sampling run of BASELINE config #2 on each GPU: Radon hierarchical regression
(919 obs, 85 counties, n=175, fp64), 2048 chains x (1000 tune + 1000 draws), jitter+adapt_diag, inside ONE
persistent kernel launch per GPU.  N > 1 shards chains (2048 per GPU, weak scaling, no data-path
collective).  `value` = leapfrog gradient evaluations (sum of the reference's own `tree_size` stat,
hmc/nuts.py:485) of all ranks / device time (CUDA events, max over ranks), inputs resident in HBM.
`e2e` = the same through the public host API with pinned host buffers: H2D of start points / streams
and D2H of draws + sampler stats inside the timed region.  `--dump-outputs DIR` writes what the last timed step
computed as .npy files (the inputs are seeded, so two builds run with the same arguments compare output for output).

The reference arm times oracle/nuts_numpy.py + oracle/logp_numpy.py (the CPU restatement that is
bit-identical to the reference's own NUTS files; PyTensor is not installable, see DESIGN.md) with one
OS process per chain on all host cores -- what pymc/sampling/parallel.py does.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "leapfrog_grad_evals_per_sec"
UNIT = "grad-evals/s"
ALG_BYTES_PER_EVAL = 919 * (8 + 8 + 4) + 7 * 175 * 8  # SURVEY 8(d): observed data + state traffic = 28,180 B

# The bench line (no --workload) is BASELINE config #2, the configuration the metric is quoted on for ONE GPU.
# The other BASELINE configs can be timed with --workload; per-eval algorithmic work follows SURVEY 8(d).
WORKLOADS = {
    "radon": dict(
        builder="radon", args={}, chains=2048, tune=1000, draws=1000, scaling="weak", mass="diag_adapt",
        bound="onchip", per_eval=float(ALG_BYTES_PER_EVAL), kernel="nuts_warp_kernel<RadonModel,6>",
        flops_per_eval=919 * 30.0 + 175 * 12.0,  # SURVEY 8(d): ~30 flop per observation + ~12 per parameter ~ 30 kflop
        desc={"n": 175, "n_obs": 919, "counties": 85}, cpu_procs=0, cpu_tune=300, cpu_draws=200,
        l2="outputs (2.9 GB of draws per step) exceed L2; no explicit flush needed",
        note="observed data is staged once per CTA into shared memory (bulk TMA) and the chain state lives in "
             "registers/shared memory, so DRAM traffic is far below the algorithmic bytes; the binding pipe is fp64"),
    "logistic": dict(  # config #3: 512 chains per GPU (4096 over 8), X replicated
        builder="logistic", args={}, chains=512, tune=60, draws=20, scaling="weak", mass="diag_adapt",
        bound="tensor", per_eval=4.0 * 1e6 * 128, kernel="logistic_fused_kernel<16> (fp64 DMMA)",
        desc={"n": 128, "n_rows": 1_000_000}, cpu_procs=16, cpu_tune=12, cpu_draws=6,
        l2="the design matrix (1.02 GB) is streamed from HBM on every batched leapfrog and exceeds L2",
        note="lock-step batched leapfrog: one fused pass over X per batch (X.beta, sigmoid/softplus, X^T r) on the fp64 "
             "tensor path (mma.sync m8n8k4.f64); flops per grad-eval per chain = 4 N K"),
    "stochvol": dict(  # config #4: 256 chains per GPU (512 over 2), deep trees
        builder="stochvol", args={}, chains=256, tune=300, draws=100, scaling="weak", mass="diag_adapt",
        bound="onchip", per_eval=24000.0 + 7 * 3003 * 8 + 2 * 3003 * 8 * 2, kernel="nuts_warp_kernel<StochVolModel,12,8> (chain = CTA)",
        flops_per_eval=3000 * 40.0,  # SURVEY 8(d): ~40 flop per latent state ~ 120 kflop
        desc={"n": 3003, "T": 3000}, cpu_procs=0, cpu_tune=40, cpu_draws=20,
        l2="tree bookkeeping of 256 chains (53 vectors x 24 KB each) is spread over HBM/L2",
        note="chain = CTA of 8 warps; integrator state in shared memory, pending-subtree stack in HBM/L2"),
    "mvgauss": dict(  # config #5: 256 chains in TOTAL, strong scaling over GPUs, dense mass matrix
        builder="mvgauss", args={}, chains=256, tune=20, draws=10, scaling="strong", mass="dense",
        bound="tensor", per_eval=4.0 * 1e4 * 1e4, kernel="gemm_nt_dmma_kernel (fp64 DMMA)",
        desc={"n": 10000, "mass": "QuadPotentialFull(Sigma)"}, cpu_procs=8, cpu_tune=3, cpu_draws=2,
        l2="precision and covariance (800 MB each) are streamed from HBM on every batched leapfrog and exceed L2",
        note="lock-step batched leapfrog: grad = -P q and w = Sigma g as two NT GEMMs over all chains on the fp64 tensor "
             "path; flops per grad-eval per chain = 4 n^2 (one mass GEMM per leapfrog by linearity)"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="radon", choices=sorted(WORKLOADS))
    ap.add_argument("--chains-per-gpu", type=int, default=0, help="0 = the workload's default")
    ap.add_argument("--tune", type=int, default=-1)
    ap.add_argument("--draws", type=int, default=-1)
    ap.add_argument("--cpu-chains", type=int, default=0, help="reference arm / cpu_baseline: chains per step (0 = host cores)")
    ap.add_argument("--precision", default="fp64", choices=["fp64", "tc_fp16x2"],
                    help="logistic / mvgauss: fp64 DMMA (parity mode) or the tcgen05 split-fp16 tensor-core performance mode")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (draws, per-draw stats, per-chain summary) as DIR/<name>.npy "
                         "in float64; above 64 MB a fixed, seeded sample of chains")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the CUDA engine's outputs: --impl b200")
    args.wl = WORKLOADS[args.workload]
    args.tune = args.wl["tune"] if args.tune < 0 else args.tune
    args.draws = args.wl["draws"] if args.draws < 0 else args.draws
    return args


def workload_name(args, C):
    base = {"radon": "radon_hierarchical", "logistic": "logistic_glm_1e6x128", "stochvol": "stochastic_volatility_T3000",
            "mvgauss": "gaussian_n10000_dense_mass"}[args.workload]
    return f"{base}_{C}chains_{args.tune}tune_{args.draws}draws"


# ---------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port on the host cores, one process per chain
# ---------------------------------------------------------------------------------------------
_CPU_SPEC = {}


def _cpu_chain(job):
    seed, tune, draws, workload, threads = job
    try:  # BLAS threads per chain process (the reference pins 1 per chain, sampling/parallel.py:200-205; the
        from threadpoolctl import threadpool_limits  # BLAS-bound configs get cores/processes threads each)

        threadpool_limits(limits=threads)
    except Exception:
        pass
    from oracle import logp_numpy, nuts_numpy
    from pymc_b200 import models

    wl = WORKLOADS[workload]
    if workload not in _CPU_SPEC:  # built once per worker process
        _CPU_SPEC[workload] = models.BUILDERS[wl["builder"]](**wl["args"])
    spec = _CPU_SPEC[workload]
    # logp/dlogp as COMPILED code where the oracle has a plain-C build (Radon: oracle/c/radon_logp.c, gcc -O3): the reference
    # evaluates this function as a PyTensor C thunk, so the NumPy form (10x slower per call) would flatter the GPU arm
    f = logp_numpy.make_logp(spec, compiled=True)
    rng = np.random.default_rng(seed)
    q0 = spec.initial_point() + rng.uniform(-1, 1, spec.n)
    if wl["mass"] == "dense":
        mass = nuts_numpy.DenseMass(spec.data["cov"])
    else:
        mass = nuts_numpy.DiagMass(np.ones(spec.n), adapt=True, initial_mean=q0.copy(), initial_weight=10)
    o = nuts_numpy.Oracle(f, mass)
    o.setup_chain(np.random.default_rng(seed + 1))
    t0 = time.perf_counter()
    qs, st = o.run(q0, tune, draws)
    return int(st["tree_size"].sum()), time.perf_counter() - t0, qs[tune:, :4096]


def cpu_run(chains, tune, draws, seed0, pool, workload="radon", threads=1):
    t0 = time.perf_counter()
    out = pool.map(_cpu_chain, [(seed0 + 2 * c, tune, draws, workload, threads) for c in range(chains)])
    wall = time.perf_counter() - t0
    evals = sum(o[0] for o in out)
    return evals, wall, np.stack([o[2] for o in out])


def cpu_ess(qs, wall):
    """ESS/s of a CPU sample: rank-normalised bulk ESS (min over parameters) of the post-warm-up draws / wall time of the
    whole sample (warm-up included) -- the same estimator and convention as the GPU line's `ess`."""
    from pymc_b200 import diagnostics

    if qs.shape[0] < 2 or qs.shape[1] < 8:
        return None
    try:
        e = float(np.nanmin(diagnostics.ess_bulk(qs)))
    except Exception:  # a diagnostic must never take the bench line down
        return None
    return {"min_bulk_ess": e, "ess_per_sec": e / wall, "chains": int(qs.shape[0]), "draws": int(qs.shape[1])}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def physical_cpus():
    """One logical CPU id per PHYSICAL core of the CPUs this process may run on (hyper-thread siblings dropped)."""
    try:
        allowed = sorted(os.sched_getaffinity(0))
    except AttributeError:
        return list(range(os.cpu_count() or 1))
    seen, out = set(), []
    for cpu in allowed:
        try:
            with open(f"/sys/devices/system/cpu/cpu{cpu}/topology/thread_siblings_list") as fh:
                key = fh.read().strip()
        except OSError:
            key = str(cpu)
        if key not in seen:
            seen.add(key)
            out.append(cpu)
    return out


def _pin_worker(cpus, procs, counter):
    """Pool initializer: worker i is pinned to its own slice of the physical cores (one core per chain process; the
    BLAS-bound workloads get cores/processes cores each)."""
    with counter.get_lock():
        i = counter.value
        counter.value += 1
    per = max(1, len(cpus) // max(1, procs))
    lo = (i * per) % len(cpus)
    try:
        os.sched_setaffinity(0, cpus[lo:lo + per] or cpus[:1])
    except (AttributeError, OSError):
        pass


def summary_matrix(summary):
    """Per-chain scalar summaries (grad_evals, bad_energy_at, final_step_size, ...) as one [chains, k] float64 matrix for the
    gather to rank 0; per-chain VECTORS (final_var [chains, n], final_cov) stay with the rank that holds the chains."""
    cols = [np.asarray(v, dtype=np.float64) for v in summary.values() if np.ndim(v) == 1]
    return np.stack(cols, axis=1)


def cpu_logp_kind(workload):
    from oracle import logp_numpy
    from pymc_b200 import models

    wl = WORKLOADS[workload]
    if wl["builder"] == "radon" and os.path.isfile(logp_numpy.RadonLogpC.LIB):
        return "compiled C (oracle/c/radon_logp.c, gcc -O3) under the Python NUTS of oracle/nuts_numpy.py"
    return "NumPy/SciPy (oracle/logp_numpy.py) under the Python NUTS of oracle/nuts_numpy.py"


def make_pool(procs):
    import multiprocessing as mp

    ctx = mp.get_context("spawn")
    return ctx.Pool(procs, initializer=_pin_worker, initargs=(physical_cpus(), procs, ctx.Value("i", 0)))


def cpu_plan(args):
    """processes, BLAS threads per process, chains, tune, draws of the bounded CPU sample of this workload.
    One process per PHYSICAL core (pinned), like one chain per core in sampling/parallel.py."""
    cores = len(physical_cpus())
    wl = args.wl
    procs = min(cores, wl["cpu_procs"] or cores)
    chains = args.cpu_chains or procs
    procs = min(procs, chains)
    return procs, max(1, cores // procs), chains, min(args.tune, wl["cpu_tune"]), min(args.draws, wl["cpu_draws"])


def cpu_measure(args, steps, warm=True):
    """The bounded CPU sample: `steps` runs of `chains` chains on pinned workers + the single-process rate on one idle
    core (the linear expectation).  Returns (evals, wall, ess, info); info carries per-core rates and the efficiency, and
    says so loudly when the box delivers less than half of linear (oversubscribed host: VERDICT r1 weak #9)."""
    procs, threads, chains, tune, draws = cpu_plan(args)
    with make_pool(1) as solo:  # one chain alone on one pinned core
        cpu_run(1, 2, 1, 999, solo, args.workload, threads)
        e1, w1, _ = cpu_run(1, tune, draws, 4242, solo, args.workload, threads)
    solo_rate = e1 / w1
    with make_pool(procs) as pool:
        if warm:
            cpu_run(procs, 2, 1, 999, pool, args.workload, threads)  # imports, model build, BLAS warm-up in every worker
        evals, wall, ess = 0, 0.0, None
        for s in range(steps):
            e, w, qs = cpu_run(chains, tune, draws, 1000 * (s + 1), pool, args.workload, threads)
            evals += e
            wall += w
            ess = cpu_ess(qs, w)
    rate = evals / wall
    eff = rate / (solo_rate * procs)
    info = {"processes": procs, "blas_threads": threads, "physical_cores": len(physical_cpus()), "logical_cpus": host_cores(),
            "pinned": True, "per_core_evals_per_s": rate / procs, "single_core_evals_per_s": solo_rate,
            "linear_expectation": solo_rate * procs, "parallel_efficiency": eff,
            "logp": cpu_logp_kind(args.workload)}
    if eff < 0.5:
        info["warning"] = (f"host delivers {eff:.0%} of linear scaling over {procs} pinned processes: the CPU arm is "
                           "memory/SMT/cgroup bound on this box; compare with linear_expectation")
        print("bench.py: " + info["warning"], file=sys.stderr)
    sample = (f"{chains} chains x ({tune} tune + {draws} draws) of the same {args.workload} model per step, {procs} pinned "
              f"processes x {threads} BLAS threads")
    return evals, wall, ess, info, sample, procs * threads


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    evals, wall, ess, info, sample, cores = cpu_measure(args, args.steps, warm=bool(args.warmup))
    value = evals / wall
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args, (args.chains_per_gpu or args.wl["chains"])), **args.wl["desc"],
                   "note": "bounded CPU sample of the same workload"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "ess": ess, **info},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
# clocks sampling during the timed region (B200_PROFILING.md recipe)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def ncu_traffic(workload, evals_per_launch):
    """(DRAM bytes per launch, source) from the committed ncu --set full capture of this workload's kernel
    (profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum per grad-eval of the captured launch, scaled by
    the grad-evals of this launch -- the capture is a shorter launch of the same kernel); None if nothing is committed."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.isfile(p):
        try:
            e = json.load(open(p))[workload]
            return float(e["dram_bytes_per_grad_eval"]) * evals_per_launch, e.get("source", "profiles/traffic.json")
        except Exception:
            return None
    return None


def make_roofline(workload, wl, per_launch, k_ms, fp64, dmma, peaks, traffic):
    """The `roofline` object of the bench line.  per_launch: grad evaluations of one run (start states included);
    k_ms: its CUDA-event duration; fp64 / dmma: TFLOP/s measured in this process (or None); peaks: (HBM GB/s, source);
    traffic: (DRAM bytes per launch or None, how it was obtained).

    The top-level `bound`/`frac` is the BINDING resource.  The persistent kernels keep observed data and chain state on
    chip, so their DRAM traffic is orders of magnitude below the algorithmic bytes and the binding pipe is fp64: the
    HBM-by-algorithmic-bytes figure SURVEY 8(d) asks for is reported as the secondary `hbm_by_algorithmic_bytes` object
    (it is NOT a utilisation of anything), next to the DRAM bytes ncu measured."""
    t_bytes, t_how = traffic if traffic else (None, None)
    if wl["bound"] == "onchip":
        peak, how = peaks
        gbs = wl["per_eval"] * per_launch / (k_ms * 1e-3) / 1e9
        hbm = {"achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak, "peak_source": how,
               "algorithmic_bytes_per_eval": wl["per_eval"], "dram_bytes_measured": t_bytes, "dram_bytes_source": t_how,
               "note": "algorithmic bytes / kernel time; not a DRAM utilisation (data and chain state are on chip)"}
        fpeak = fp64 or 36.0
        tf = wl["flops_per_eval"] * per_launch / (k_ms * 1e-3) / 1e12
        return {"bound": "fp64", "achieved": tf, "peak": fpeak, "unit": "TFLOP/s", "frac": tf / fpeak,
                "traffic": t_bytes, "traffic_source": t_how,
                "peak_source": "DFMA micro-benchmark in this run (b200_measure_fp64_tflops; MEASURED_PEAKS.json has only HBM "
                               "and bf16)" if fp64 else "fallback 36.0 (DFMA peak measured on this pool, profiles/)",
                "algorithmic_flops_per_eval": wl["flops_per_eval"], "kernel": wl["kernel"], "kernel_ms": k_ms,
                "note": wl["note"], "hbm_by_algorithmic_bytes": hbm}
    # dense contraction on the fp64 tensor path: no fp64 entry in MEASURED_PEAKS.json (HBM + bf16 only), so the
    # denominator is the DMMA rate measured in this process by the library's own micro-benchmark
    peak = dmma or 37.0
    achieved = wl["per_eval"] * per_launch / (k_ms * 1e-3) / 1e12
    return {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
            "traffic": t_bytes, "traffic_source": t_how,
            "peak_source": "fp64 DMMA micro-benchmark in this run (MEASURED_PEAKS.json has no fp64 entry)"
            if dmma else "fallback 37.0 (scripts/mb/dmma.cu measured on this pool)",
            "kernel": wl["kernel"], "kernel_ms": k_ms, "algorithmic_flops_per_eval": wl["per_eval"], "note": wl["note"],
            "fp64_dfma_peak_tflops_measured": fp64,
            "time_base": "kernel_ms spans every launch of the lock-step loop (advance kernels and ragged tail included)"}


# ---------------------------------------------------------------------------------------------
# the CUDA engine arm
# ---------------------------------------------------------------------------------------------
DUMP_BYTES = 64_000_000  # everything --dump-outputs writes, .npy headers included


def dump_outputs(res, out_dir):
    """Writes the arrays a caller of the timed path receives from one nuts_run -- draws [C, T, n], every per-draw stat
    [C, T] and every per-chain summary [C, ...] -- as out_dir/<name>.npy in float64, so that two builds run with the same
    arguments can be compared output for output.  When all chains do not fit in DUMP_BYTES, every array keeps the same
    chains: a sample drawn from default_rng(0), listed in chains.npy."""
    import torch

    arrays = {"draws": res.draws, **{"stat_" + k: v for k, v in res.stats.items()},
              **{"summary_" + k: v for k, v in res.summary.items()}}
    C = res.draws.shape[0]
    per_chain = 8 * sum(int(a.numel()) // C for a in arrays.values()) + 8  # float64 values + the chain's index
    budget = DUMP_BYTES - 4096 * (len(arrays) + 1)  # room for the .npy headers
    k = min(C, max(1, budget // per_chain))
    chains = np.arange(C) if k == C else np.sort(np.random.default_rng(0).choice(C, size=k, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "chains.npy"), chains.astype(np.float64))
    for name, a in arrays.items():
        sel = a[torch.as_tensor(chains, device=a.device)] if torch.is_tensor(a) else np.asarray(a)[chains]
        sel = sel.to(torch.float64).cpu().numpy() if torch.is_tensor(sel) else sel.astype(np.float64)
        np.save(os.path.join(out_dir, name + ".npy"), sel)


def pcie_probe(dev, mib=512):
    """Host link of THIS box: one pinned 512 MiB copy each way (CUDA events).  The e2e figure moves with it: the Radon step
    sends 3 GB of draws to the host while the sampling half of the kernel runs."""
    import torch

    h = torch.empty(mib << 20, dtype=torch.uint8, pin_memory=True)
    d = torch.empty(mib << 20, dtype=torch.uint8, device=dev)
    out = {}
    for name, (dst, src) in {"h2d_GBps": (d, h), "d2h_GBps": (h, d)}.items():
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        dst.copy_(src, non_blocking=True)
        b.record()
        torch.cuda.synchronize()
        out[name] = (mib << 20) / (a.elapsed_time(b) * 1e-3) / 1e9
    return out


def b200_arm(args):
    import torch

    from pymc_b200 import _lib, diagnostics, engine, models, parallel
    from pymc_b200 import rng as brng

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # B200_BENCH_ONE_GPU=1: every rank uses GPU 0 and the ranks talk over gloo -- NOT a measurement, a way to run the N > 1 host
    # logic of this file (sharding, the gathers, max-over-ranks timing) on a one-GPU box; the line says so ("debug")
    one_gpu = world > 1 and os.environ.get("B200_BENCH_ONE_GPU") == "1"
    if one_gpu:
        local = 0
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist

        if one_gpu:
            dist.init_process_group("gloo")
        else:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    wl = args.wl
    build_args = dict(wl["args"])
    if args.workload == "mvgauss":  # four 800 MB matrices, a minute of BLAS: built once per box, shared by every rank and run
        build_args["cache_dir"] = os.environ.get("B200_CACHE_DIR", "/dev/shm/b200_cache")
        if world > 1 and rank != 0:
            import torch.distributed as dist

            dist.barrier()  # rank 0 builds (or finds) the cache first
    spec = models.BUILDERS[wl["builder"]](**build_args)
    if args.workload == "mvgauss" and world > 1 and rank == 0:
        import torch.distributed as dist

        dist.barrier()
    cm = engine.CompiledModel(spec, device=local)
    if args.precision != "fp64":
        if args.workload not in ("logistic", "mvgauss"):
            raise SystemExit("--precision tc_fp16x2 applies to the dense contractions: --workload logistic | mvgauss")
        cm.set_precision(args.precision)
    tune, draws, n = args.tune, args.draws, spec.n
    if wl["scaling"] == "strong":  # fixed total number of chains, split over the ranks (BASELINE config #5)
        chains_total = args.chains_per_gpu * world if args.chains_per_gpu else wl["chains"]
        lo, hi = parallel.chain_range(chains_total, rank, world)
        C = hi - lo
    else:
        C = args.chains_per_gpu or wl["chains"]
        chains_total = C * world
        lo = rank * C
    run_kw = dict(mass=wl["mass"])
    # streams and starts exactly as sample_b200_nuts derives them; global chain ids => independent of N
    step_rngs, _, jitter_seeds = brng.chain_generators(20260922, chains_total)
    q0_host = np.stack([spec.initial_point() + np.random.default_rng(s).uniform(-1, 1, n) for s in jitter_seeds[lo:lo + C]])
    mean_all = np.mean([spec.initial_point() + np.random.default_rng(s).uniform(-1, 1, n) for s in jitter_seeds], axis=0)
    mean0_host = np.broadcast_to(mean_all, (C, n)).copy() if wl["mass"] == "diag_adapt" else None
    states0 = brng.pack_pcg64(step_rngs[lo:lo + C])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: inputs resident in HBM, outputs stay in HBM --------------------------------------
    q0_d = torch.as_tensor(q0_host, device=dev)
    mean0_d = None if mean0_host is None else torch.as_tensor(mean0_host, device=dev)
    states = states0.copy()

    def step_device(k):
        return cm.nuts_run(q0_d, states, tune=tune, draws=draws, mean0=mean0_d, store_warmup=False,
                           philox_seed=1000 + k, device_outputs=True, reuse_outputs=True, chain_offset=lo, **run_kw)

    for k in range(args.warmup):
        res = step_device(-1 - k)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    evals_t = torch.zeros((), dtype=torch.int64, device=dev)
    all_evals_t = torch.zeros((), dtype=torch.int64, device=dev)
    kernel_ms, launches = [], 0
    lockstep = args.workload in ("logistic", "mvgauss")
    # start-state evaluations per chain: one per iteration (compute_state, base_hmc.py:202); the lock-step engine carries
    # the accepted proposal's (logp, grad) into the next draw and evaluates only the very first start state
    start_evals = 1 if lockstep else (tune + draws)
    ev0.record()
    for k in range(args.steps):
        res = step_device(k)
        # leapfrog gradient evaluations of ALL iterations (warm-up included): the kernel's own count minus the
        # start-state evaluations
        all_evals_t += res.summary["grad_evals"].sum()
        evals_t += res.summary["grad_evals"].sum() - C * start_evals
        kernel_ms.append(res.kernel_ms)
        launches += res.launches
    ev1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms_total = parallel.max_over_ranks(ev0.elapsed_time(ev1))
    evals = parallel.sum_over_ranks(float(evals_t.item()))
    all_evals = float(all_evals_t.item())
    value = evals / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:  # rank 0's chains when N > 1
        dump_outputs(res, args.dump_outputs)

    # ESS/sec of the last step (rank-normalised bulk ESS over this rank's chains, min over parameters)
    ess = diagnostics.ess_bulk_torch(res.draws)
    ess_min = float(ess.min().item())
    step_s = ms_total * 1e-3 / args.steps
    div_frac = float(res.stats["diverging"].double().mean().item())

    # ---- e2e: public host API, pinned host buffers, H2D + D2H inside the timed region --------------
    e2e = None
    near = parallel.near_gpu(local)
    if not args.no_e2e:
        near.__enter__()  # pinned buffers are allocated on the GPU's NUMA node (restored before the CPU arm runs)
        T = draws
        pin = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=True).numpy()  # noqa: E731
        q0_p = pin((C, n), torch.float64); q0_p[:] = q0_host
        mean0_p = None
        if mean0_host is not None:
            mean0_p = pin((C, n), torch.float64); mean0_p[:] = mean0_host
        n_e2e = args.steps
        st_e = states0.copy()
        # one untimed call: allocates the pooled pinned output buffers the timed calls reuse
        res_h = cm.nuts_run(q0_p, st_e, tune=tune, draws=draws, mean0=mean0_p, store_warmup=False,
                            philox_seed=1999, device_outputs=False, chain_offset=lo, pinned_outputs=True, **run_kw)
        if world > 1:  # NCCL sets the gather's channels up on its first call (100+ ms): not part of a steady-state step
            parallel.gather_chains(summary_matrix(res_h.summary), {}, chains_total, dst=0)
        barrier()
        t0 = time.perf_counter()
        ev_tot = 0
        call_ms, call_kernel_ms = [], []
        for k in range(n_e2e):
            tc0 = time.perf_counter()
            res_h = cm.nuts_run(q0_p, st_e, tune=tune, draws=draws, mean0=mean0_p, store_warmup=False,
                                philox_seed=2000 + k, device_outputs=False, chain_offset=lo, pinned_outputs=True, **run_kw)
            ev_tot += int(res_h.summary["grad_evals"].sum()) - C * start_evals
            call_ms.append(1e3 * (time.perf_counter() - tc0))
            call_kernel_ms.append(res_h.kernel_ms)
            if world > 1:
                # the draws stay SHARDED: every rank's shard is already in its own pinned host buffer on this node (N PCIe
                # links in parallel).  What rank 0 needs of the other ranks for the run's report -- the per-chain summaries
                # (step size, tree statistics, evaluation counts) -- is gathered to rank 0 over NCCL here, inside the timed
                # region.  The cost of gathering the DRAWS themselves to rank 0's HBM is measured separately below.
                summ_all, _ = parallel.gather_chains(summary_matrix(res_h.summary), {}, chains_total, dst=0)
        torch.cuda.synchronize()
        dt = parallel.max_over_ranks(time.perf_counter() - t0)
        ev_all = parallel.sum_over_ranks(float(ev_tot))
        h2d = q0_p.nbytes + (mean0_p.nbytes if mean0_p is not None else 0) + st_e.nbytes
        d2h = res_h.draws.nbytes + sum(v.nbytes for v in res_h.stats.values()) + sum(v.nbytes for v in res_h.summary.values()) + st_e.nbytes
        e2e = {"value": ev_all / dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "steps": n_e2e, "ms_per_step": 1e3 * dt / n_e2e,
               # this rank's calls: wall time of each public-API call and the kernel time inside it (CUDA events)
               "call_ms": call_ms, "call_kernel_ms": call_kernel_ms,
               "warmup_calls": 1,  # one untimed call first: it allocates the pooled pinned output buffers the timed calls reuse
               }
        if rank == 0:
            e2e["host_link"] = pcie_probe(dev)
            e2e["host_numa"] = near.info
        near.__exit__()
        if world > 1:
            e2e["gather"] = ("draws stay sharded: each rank copies its chains to its own pinned host buffer; per-chain "
                             "summaries are gathered to rank 0 over NCCL inside the timed region")

    # ---- N > 1: what gathering every rank's draws to rank 0 costs (NCCL gather over NVLink into rank 0's HBM) ---------
    gather_info = None
    if world > 1:
        # one small untimed gather first: NCCL builds the communicator's gather channels lazily (1-3 s on the first call,
        # which the r2_scale_* lines of the multi-GPU call still include in their gather figure)
        parallel.gather_chains(res.draws[:, :1].contiguous(), {}, chains_total, dst=0)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        gd, _ = parallel.gather_chains(res.draws, {}, chains_total, dst=0)
        g1.record()
        torch.cuda.synchronize()
        g_ms = parallel.max_over_ranks(g0.elapsed_time(g1))
        nbytes = parallel.sum_over_ranks(float(res.draws.numel() * res.draws.element_size() if rank != 0 else 0))
        gather_info = {"ms": g_ms, "bytes_to_rank0": nbytes, "GB_per_s": nbytes / (g_ms * 1e-3) / 1e9,
                       "what": "dist.gather of the last step's device-resident draws to rank 0 (not part of value or e2e: "
                               "the product leaves draws sharded unless sample_b200_nuts(gather='rank0') is asked for)"}
        del gd

    # ---- roofline of the dominant kernel --------------------------------------------------------------
    k_ms = float(np.mean(kernel_ms))
    per_launch = all_evals / args.steps  # grad evaluations of one run on this rank, start states included
    fp64 = dmma = None
    if rank == 0:
        import ctypes

        tf = ctypes.c_double()
        if _lib.load().b200_measure_fp64_tflops(ctypes.byref(tf)) == 0:
            fp64 = tf.value
        if _lib.load().b200_measure_dmma_tflops(ctypes.byref(tf)) == 0:
            dmma = tf.value
    roofline = make_roofline(args.workload, wl, per_launch, k_ms, fp64, dmma, measured_peaks(),
                             ncu_traffic(args.workload, per_launch))
    if args.precision == "tc_fp16x2":
        # tensor-core performance mode: every fp64 product is three fp16 MMAs (hi*hi, hi*lo, lo*hi) -> issued tensor flops =
        # 3 x the algorithmic 4 N K per eval; peak = the dense bf16/fp16 rate in MEASURED_PEAKS.json (sustained figure: the
        # kernel runs inside a long loop), else the nominal 2250
        issued = 3.0 * wl["per_eval"] * per_launch / (k_ms * 1e-3) / 1e12
        tpeak, tsrc = 2250.0, "nominal dense bf16/fp16 (MEASURED_PEAKS.json absent)"
        try:
            mp_ = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            tpeak, tsrc = float(mp_.get("bf16_tflops_sustained") or mp_["bf16_tflops"]), "MEASURED_PEAKS.json bf16_tflops_sustained"
        except Exception:
            pass
        roofline = {"bound": "tensor", "achieved": issued, "peak": tpeak, "unit": "TFLOP/s", "frac": issued / tpeak,
                    "traffic": None, "peak_source": tsrc,
                    "kernel": ("logistic_tc2_kernel" if args.workload == "logistic" else "gemm_tc_kernel") + " (tcgen05.mma kind::f16, TMEM, TMA)",
                    "kernel_ms": k_ms, "algorithmic_flops_per_eval": wl["per_eval"], "issued_tensor_flops_per_eval": 3.0 * wl["per_eval"],
                    "fp64_equivalent_tflops": wl["per_eval"] * per_launch / (k_ms * 1e-3) / 1e12,
                    "accuracy": "gradient <= 1e-6 of its largest entry, logp <= 1e-8 relative vs the fp64 path "
                                "(tests/test_gpu_tc.py; profiles/r2_parity_report.json)",
                    "time_base": "kernel_ms spans every launch of the lock-step loop (advance kernels and ragged tail included)"}

    # ---- cpu_baseline (rank 0, N = 1 only): the oracle port on the host cores, bounded sample -----------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        e, w, ess_c, info, sample, cores = cpu_measure(args, 1)
        cpu = {"value": e / w, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "wall_s": w, "ess": ess_c, **info}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None,
            "dtype": "f64" if args.precision == "fp64" else "f16x2 split operands, f32 accumulate, f64 drains (performance mode)",
            "data": "synthetic",
            "config": {"workload": workload_name(args, C if wl["scaling"] == "weak" else chains_total), **wl["desc"],
                       "precision": args.precision,
                       "chains_per_gpu": C, "chains_total": chains_total, "tune": tune, "draws": draws,
                       "init": "jitter+adapt_diag" if wl["mass"] == "diag_adapt" else "jitter, fixed dense mass matrix",
                       "momentum": "device philox", "l2": wl["l2"]},
            "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "host_ms_between_launches": ms_total / args.steps - k_ms,
            "gather_to_rank0": gather_info,
            "ess": {"min_bulk_ess_last_step": ess_min, "ess_per_sec": ess_min / step_s, "chains": C, "draws": draws},
            "grad_evals_incl_start_state": all_evals * world, "divergent_fraction": div_frac,
        }
        if one_gpu:
            line["debug"] = "B200_BENCH_ONE_GPU=1: all ranks shared GPU 0 over gloo; not a measurement"
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        reference_arm(args)
    else:
        b200_arm(args)


if __name__ == "__main__":
    main()
