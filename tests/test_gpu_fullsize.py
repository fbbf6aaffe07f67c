"""-m gpu: parity of the kernel instantiations the BENCH lines actually run (VERDICT r1, "What's weak" #1).

Round 1 only exercised the small-shape instantiations of the lock-step kernels under test (K = 8 logistic slabs,
n = 60 GEMM tiles).  Here the benchmarked shapes are compared with the oracle and with goldens produced by the
verbatim reference (oracle/make_golden.py fullsize):

  * logistic_fused_kernel<16> (K = 128): 8192 x 128 with 130 chains (two chain-CTAs, row-CTA split), the 3-draw
    fixed-step golden, and points on the real 1e6 x 128 design matrix of BASELINE config #3;
  * gemm_nt_dmma_kernel<8,17|9|5,3>, <4,*>, <2,*> and ls_advance_kernel<16> at n = 10^4 (config #5): logp/grad at
    C in {256, 64, 32} and the 3-draw dense-mass golden;
  * the sharding drift of the fused logistic pass (row-CTA count depends on the chains per launch) is bounded;
  * the bench path of config #2 (device Philox momentum, cold jitter+adapt_diag) against posterior moments of an
    independent oracle CPU run (tests/golden/radon_posterior_oracle.npz), within 4 MCSE.
"""
import json
import os

import numpy as np
import pytest

from b200_helpers import CONTINUOUS, discrete_equal, gpu_free_run, gpu_single_draws, relerr
from conftest import ROOT

pytestmark = pytest.mark.gpu


def _report(key, value):
    """Evidence that travels back from the GPU box (gpurun merges gpurun_out/): first divergent draw indices etc."""
    p = os.path.join(ROOT, "gpurun_out")
    try:
        os.makedirs(p, exist_ok=True)
        f = os.path.join(p, "parity_report.json")
        d = json.load(open(f)) if os.path.isfile(f) else {}
        d[key] = value
        json.dump(d, open(f, "w"), indent=1, sort_keys=True)
    except OSError:
        pass


@pytest.fixture(scope="module")
def logistic128():
    from pymc_b200 import engine, models

    return engine.CompiledModel(models.logistic(n_rows=8192, n_features=128, seed=3))


@pytest.fixture(scope="module")
def logistic_full():
    from pymc_b200 import engine, models

    return engine.CompiledModel(models.logistic())


@pytest.fixture(scope="module")
def mvgauss_full():
    from pymc_b200 import engine, models

    return engine.CompiledModel(models.mvgauss())


def _check_logp_grad(cm, Q, tol):
    from oracle import logp_numpy

    f = logp_numpy.make_logp(cm.spec)
    lp, g = cm.logp_dlogp(Q)
    lo = np.array([f(q)[0] for q in Q])
    go = np.array([f(q)[1] for q in Q])
    assert relerr(lp, lo) <= tol, relerr(lp, lo)
    scale = np.max(np.abs(go), axis=1, keepdims=True)
    assert np.max(np.abs(g - go) / scale) <= tol, np.max(np.abs(g - go) / scale)
    return lp, g, scale


def test_logistic_k128_logp_grad_two_chain_ctas(logistic128):
    """130 chains = two chain-CTAs of logistic_fused_kernel<16>; 8192 rows are split over 74 row-CTAs."""
    cm = logistic128
    rng = np.random.default_rng(0)
    Q = rng.uniform(-0.5, 0.5, (130, cm.n))
    _check_logp_grad(cm, Q, 1e-12)


def test_logistic_k128_fixed_step_golden(logistic128, golden):
    name = "logistic_k128_fixed"
    d = golden(name)
    res, _ = gpu_free_run(logistic128, d, name)
    for c in range(len(d["seeds"])):
        st = {k: v[c] for k, v in res.stats.items()}
        assert discrete_equal(st, d, c).all(), f"{name} chain {c}"
        assert np.max(np.abs(res.draws[c] - d["draws_q"][c])) <= 1e-9
        for k in ("energy", "model_logp", "mean_tree_accept"):
            assert relerr(st[k], d["stat_" + k][c]) <= 1e-8, k


def test_logistic_full_design_matrix_points(logistic_full):
    """BASELINE config #3's own matrix (1e6 x 128): logp ~ -7e5, so 1e-12 relative is 1e-6 absolute."""
    rng = np.random.default_rng(1)
    Q = rng.normal(0.0, 0.3, (4, 128))
    _check_logp_grad(logistic_full, Q, 1e-12)


def test_logistic_sharding_drift_is_bounded(logistic_full):
    """The fused pass splits the rows over 148 / ceil(C/128) row-CTAs, so the partial-sum grouping of a chain's
    gradient depends on how many chains share the launch (DESIGN section 6).  Bound: <= 1e-12 relative."""
    cm = logistic_full
    rng = np.random.default_rng(2)
    Q = rng.normal(0.0, 0.3, (512, 128))
    lp_a, g_a = cm.logp_dlogp(Q[:64])
    lp_b, g_b = cm.logp_dlogp(Q)
    scale = np.max(np.abs(g_b[:64]), axis=1, keepdims=True)
    drift_g = float(np.max(np.abs(g_a - g_b[:64]) / scale))
    drift_l = relerr(lp_a, lp_b[:64])
    _report("logistic_sharding_drift", {"grad_rel": drift_g, "logp_rel": drift_l, "launches": "C=64 vs C=512"})
    assert drift_g <= 1e-12 and drift_l <= 1e-13, (drift_g, drift_l)


@pytest.mark.parametrize("C", [256, 64, 32])
def test_mvgauss_full_logp_grad(mvgauss_full, C):
    """C = 256 -> gemm_nt_dmma_kernel<8,17,3>, 64 -> <4,*>, 32 -> <2,*> (one wave of 148 SMs each)."""
    cm = mvgauss_full
    rng = np.random.default_rng(C)
    L = cm.spec.data["L"]
    Q = (L @ rng.standard_normal((cm.n, C))).T.copy()
    P = cm.spec.data["prec"]
    lp, g = cm.logp_dlogp(Q)
    go = -(Q @ P)
    lo = -0.5 * cm.n * np.log(2 * np.pi) - cm.spec.meta["logdet_L"] + 0.5 * np.einsum("ci,ci->c", Q, go)
    scale = np.max(np.abs(go), axis=1, keepdims=True)
    assert np.max(np.abs(g - go) / scale) <= 1e-12
    assert relerr(lp, lo) <= 1e-12


def test_mvgauss_full_fixed_step_golden(mvgauss_full, golden):
    """n = 10^4 dense mass: ls_advance_kernel<16>, the 2-chain GEMM tiles and the momentum GEMMs against the reference."""
    name = "mvgauss_n10000_fixed"
    d = golden(name)
    res, _ = gpu_free_run(mvgauss_full, d, name)
    for c in range(len(d["seeds"])):
        st = {k: v[c] for k, v in res.stats.items()}
        assert discrete_equal(st, d, c).all(), (name, c, st["tree_size"], d["stat_tree_size"][c])
        assert np.max(np.abs(res.draws[c] - d["draws_q"][c])) <= 1e-8
        for k in ("energy", "model_logp", "mean_tree_accept"):
            assert relerr(st[k], d["stat_" + k][c]) <= 1e-8, k


def test_radon_bench_path_posterior_matches_oracle_run(golden):
    """Config #2 as the bench runs it (device Philox momentum, cold jitter+adapt_diag), 256 chains x (500 + 500):
    posterior means and sds of every parameter agree with an independent 32-chain oracle CPU run within 4 MCSE
    (tests/sampler_fixtures.py style; fixture + generating script: oracle/make_posterior_fixture.py)."""
    from pymc_b200 import diagnostics, engine, models
    from pymc_b200 import rng as brng

    d = golden("radon_posterior_oracle")
    spec = models.radon()
    cm = engine.CompiledModel(spec)
    C = 256
    step_rngs, _, jitter_seeds = brng.chain_generators(777, C)
    q0 = np.stack([spec.initial_point() + np.random.default_rng(s).uniform(-1, 1, spec.n) for s in jitter_seeds])
    res = cm.nuts_run(q0, brng.pack_pcg64(step_rngs), tune=500, draws=500, mean0=np.broadcast_to(q0.mean(0), q0.shape).copy(),
                      store_warmup=False, philox_seed=4242)
    assert np.all(res.summary["bad_energy_at"] == -1)
    x = res.draws
    ess = diagnostics.ess_bulk(x)
    mean, sd = x.mean((0, 1)), x.std((0, 1))
    # MCSE of the mean from the bulk ESS; the VARIANCE estimate has its own Monte Carlo error: (x - mean)^2 is a chain with a
    # smaller effective sample size (heavy-tailed in the funnel directions log sigma_a / log sigma_b)
    n_gpu, n_cpu = x.shape[0] * x.shape[1], int(d["chains"]) * int(d["draws"])
    mcse_mean = np.sqrt(sd**2 / np.minimum(ess, n_gpu) + d["sd"] ** 2 / np.minimum(d["ess"], n_cpu))
    dev2 = (x - mean) ** 2
    var_mcse_gpu = dev2.std((0, 1)) / np.sqrt(np.minimum(diagnostics.ess_bulk(dev2), n_gpu))
    mcse_var = np.sqrt(var_mcse_gpu**2 + d["var_mcse"] ** 2)
    z_mean = np.abs(mean - d["mean"]) / mcse_mean
    z_sd = np.abs(sd**2 - d["var"]) / mcse_var
    worst = int(np.argmax(z_sd))
    _report("radon_posterior_check", {"max_z_mean": float(z_mean.max()), "max_z_var": float(z_sd.max()), "worst_var_param": worst,
                                     "sd_gpu_worst": float(sd[worst]), "sd_oracle_worst": float(d["sd"][worst]),
                                     "min_ess_gpu": float(ess.min()), "gpu_chains": C, "oracle_chains": int(d["chains"])})
    assert z_mean.max() <= 4.0, (int(np.argmax(z_mean)), float(z_mean.max()))
    assert z_sd.max() <= 4.5, (worst, float(z_sd.max()), float(sd[worst]), float(d["sd"][worst]))
    assert res.stats["diverging"].mean() < 0.01


@pytest.mark.parametrize("name", ["eight_schools_adapt", "radon_adapt", "radon_small_adapt", "stochvol_small_adapt",
                                  "logistic_small_adapt"])
def test_report_first_divergent_draw(golden, name):
    """SURVEY section 7: "accept/diagnose rare ulp-flips (report first divergent draw index rather than hiding)".
    Free-running and teacher-forced replays of the adaptive goldens; the indices go to gpurun_out/parity_report.json."""
    from b200_helpers import SPEC_OF
    from pymc_b200 import engine

    cm = engine.CompiledModel(SPEC_OF[name]())
    d = golden(name)
    res, _ = gpu_free_run(cm, d, name)
    st = {k: v[0] for k, v in res.stats.items()}
    ok = discrete_equal(st, d, 0)
    free_first = int(np.argmin(ok)) if not ok.all() else -1
    dq, st1 = gpu_single_draws(cm, d, name, chain=0)
    ok1 = discrete_equal(st1, d, 0)
    forced = [int(i) for i in np.flatnonzero(~ok1)]
    _report("first_divergent_draw/" + name, {"free_running_first_tree_mismatch": free_first, "draws": int(len(ok)),
                                             "teacher_forced_mismatches": forced[:20],
                                             "teacher_forced_identical_fraction": float(ok1.mean())})
    assert free_first == -1 or free_first >= 10


def _lockstep_run(cm, C, *, tune, draws, mass, seed=11, **kw):
    from pymc_b200 import rng as brng

    spec = cm.spec
    step_rngs, _, jit = brng.chain_generators(seed, C)
    q0 = np.stack([spec.initial_point() + np.random.default_rng(s).uniform(-1, 1, spec.n) for s in jit])
    return cm.nuts_run(q0, brng.pack_pcg64(step_rngs), tune=tune, draws=draws, mass=mass, store_warmup=True, philox_seed=5, **kw)


@pytest.mark.parametrize("case", ["logistic_diag", "radon_dense"])
def test_lockstep_row_compaction_changes_nothing(case, monkeypatch):
    """Finished chains give their request rows up (lockstep.cuh: ls_compact_*): with a tile of 8 rows and 40 chains of
    different lengths the batch shrinks several times during a short run; draws, statistics and evaluation counts must be
    the ones of the run without compaction, bit for bit (same chain-block count => same reduction order)."""
    from pymc_b200 import engine, models

    if case == "logistic_diag":
        cm = engine.CompiledModel(models.logistic(n_rows=4096, n_features=8, seed=2))
        kw = dict(tune=25, draws=8, mass="diag_adapt")
    else:
        spec = models.radon(n_obs=200, n_counties=12, seed=4)
        cm = engine.CompiledModel(spec)
        A = np.random.default_rng(0).standard_normal((spec.n, spec.n)) * 0.05
        cm.set_dense_mass(cov=np.eye(spec.n) * 0.05 + A @ A.T)
        kw = dict(tune=20, draws=6, mass="dense")
    monkeypatch.setenv("B200_LS_COMPACT_TILE", "0")
    ref = _lockstep_run(cm, 40, **kw)
    monkeypatch.setenv("B200_LS_COMPACT_TILE", "8")
    got = _lockstep_run(cm, 40, **kw)
    ge = ref.summary["grad_evals"]
    assert ge.max() > 1.2 * ge.min()  # chains do finish at different times
    assert got.launches > ref.launches and (got.launches - ref.launches) % 2 == 0  # two kernels per compaction
    np.testing.assert_array_equal(got.summary["grad_evals"], ge)
    np.testing.assert_array_equal(got.draws, ref.draws)
    for k in ref.stats:
        np.testing.assert_array_equal(got.stats[k], ref.stats[k], err_msg=k)
