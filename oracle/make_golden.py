"""Generates tests/golden/*.npz by running the REFERENCE's own NUTS code (loaded verbatim from
/root/reference by oracle/ref_loader.py) on the NumPy logp/grad restatement.

Run in the builder container only (the reference does not exist on the GPU box):

    python -m oracle.make_golden

Every file stores the inputs (start points, seeds, momentum noise z, mass matrix) next to the
reference's outputs (accepted positions and the per-draw sampler stats of hmc/nuts.py:478-489),
so tests can replay the exact case through oracle/nuts_numpy.py and through the CUDA engine.
"""
from __future__ import annotations

import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import logp_numpy, ref_loader  # noqa: E402
from pymc_b200 import models  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
STAT_KEYS = ["depth", "tree_size", "index_in_trajectory", "diverging", "reached_max_treedepth", "step_size",
             "step_size_bar", "mean_tree_accept", "energy", "energy_error", "max_energy_error", "model_logp"]


def run_reference(spec, q0, *, seed, tune, draws, adapt, var=None, eps=None, nuts_kwargs=None, init_var=None,
                  dense=False):
    """One chain through the verbatim reference.  adapt=True: DiagAdapt(mean=q0, ones, weight 10) + dual
    averaging (what init_nuts builds, mcmc.py:1890-1894); adapt=False: fixed QuadPotentialDiag(var), fixed eps."""
    f = logp_numpy.make_logp(spec)
    qp = ref_loader.quadpotential()
    n = spec.n
    if dense:  # QuadPotentialFull with the model's covariance (quadpotential.py:680-725); `adapt` = step size only
        pot = qp.QuadPotentialFull(spec.data["cov"])
    elif adapt:
        pot = qp.QuadPotentialDiagAdapt(n, q0.copy(), np.ones(n) if init_var is None else np.array(init_var, dtype="d"), 10)
    else:
        pot = qp.QuadPotentialDiag(np.ones(n) if var is None else np.asarray(var, dtype="d"))
    start = {v.name: q0[v.offset : v.offset + v.size].copy() for v in spec.vars}
    kw = dict(nuts_kwargs or {})
    if eps is not None:
        kw["step_scale"] = eps * n**0.25  # base_hmc.py:161 inverts to step_size == eps
    step, _ = ref_loader.make_nuts(f, spec.var_sizes, start, potential=pot, step_rng=0, adapt_step_size=adapt, **kw)
    step.setup_chain(np.random.default_rng(seed), tune, draws)
    if tune == 0:
        step.tune = False
    pt, qs, sts = start, [], []
    pre_rng, pre_var, used_eps = [], [], []
    for i in range(tune + draws):
        if i == tune:
            step.stop_tuning()
        # what a single-draw replay ("teacher forcing") needs: stream position, mass matrix, step size
        s = step.rng.bit_generator.state["state"]
        pre_rng.append([s["state"] >> 64, s["state"] & (2**64 - 1), s["inc"] >> 64, s["inc"] & (2**64 - 1)])
        pre_var.append(np.zeros(1) if dense else np.array(step.potential._var if adapt else step.potential.v))
        pt, st = step.step(pt)
        used_eps.append(float(step.step_size))  # set inside astep: the eps this draw integrated with
        qs.append(np.concatenate([np.ravel(pt[v.name]) for v in spec.vars]))
        sts.append(st[0])
    stats = {k: np.array([s[k] for s in sts]) for k in STAT_KEYS}
    final_var = np.zeros(1) if dense else np.array(step.potential._var if adapt else step.potential.v)
    extra = dict(pre_rng=np.array(pre_rng, dtype=np.uint64), pre_var=np.array(pre_var), used_eps=np.array(used_eps))
    return np.array(qs), stats, final_var, float(step.step_size), extra


def noise(seed, T, n):
    """The momentum normals the reference's potential draws: setup_chain spawns the potential stream
    from the chain stream (base_hmc.py:300-302), then one normal(size=n) per draw (quadpotential.py:325,:619)."""
    g = np.random.default_rng(seed).spawn(1)[0]
    return np.array([g.normal(size=n) for _ in range(T)])


def case(name, spec_name, spec_args, q0s, seeds, *, tune, draws, adapt, var=None, eps=None, nuts_kwargs=None,
         init_var=None, dense=False):
    spec = models.BUILDERS[spec_name](**spec_args)
    C = len(seeds)
    Q, ST, FV, FE, Z, EX = [], [], [], [], [], []
    for c in range(C):
        v = None if var is None else var[c]
        e = None if eps is None else float(eps[c])
        q, st, fv, fe, ex = run_reference(spec, q0s[c], seed=seeds[c], tune=tune, draws=draws, adapt=adapt, var=v,
                                          eps=e, nuts_kwargs=nuts_kwargs,
                                          init_var=None if init_var is None else init_var[c], dense=dense)
        Q.append(q); ST.append(st); FV.append(fv); FE.append(fe); EX.append(ex)
        Z.append(noise(seeds[c], tune + draws, spec.n))
    out = dict(q0=np.array(q0s), seeds=np.array(seeds), tune=tune, draws=draws, adapt=adapt, dense=dense, draws_q=np.array(Q),
               z=np.array(Z), final_var=np.array(FV), final_step_size=np.array(FE),
               var=np.array(var) if var is not None else np.ones((C, spec.n)),
               eps=np.array(eps) if eps is not None else np.full(C, np.nan),
               init_var=np.array(init_var) if init_var is not None else np.ones((C, spec.n)),
               step_scale=(nuts_kwargs or {}).get("step_scale", 0.25))
    for k in EX[0]:
        out[k] = np.array([e[k] for e in EX])
    for k in STAT_KEYS:
        out["stat_" + k] = np.array([s[k] for s in ST])
    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    ts = out["stat_tree_size"]
    print(f"{name}: {C} chains x {tune}+{draws}, grad evals {int(ts.sum())}, mean depth {out['stat_depth'].mean():.2f}, "
          f"divergences {int(out['stat_diverging'].sum())}")
    return out


def main():
    if not ref_loader.available():
        raise SystemExit("reference not present; golden vectors can only be generated in the builder container")
    # --- Eight Schools: the SURVEY 8c loader self-check case (start 0, unit mass, eps0, seed 20240922) ---
    es = models.eight_schools()
    case("eight_schools_fixed", "eight_schools", {}, [np.zeros(10)], [20240922], tune=0, draws=40, adapt=False)
    rng = np.random.default_rng(11)
    q0s = [es.initial_point() + rng.uniform(-1, 1, 10) for _ in range(3)]
    e = case("eight_schools_adapt", "eight_schools", {}, q0s, [101, 102, 103], tune=300, draws=100, adapt=True)
    case("eight_schools_warm_adapt", "eight_schools", {}, [e["draws_q"][0, -1]], [601], tune=250, draws=30, adapt=True,
         init_var=e["final_var"][:1], nuts_kwargs={"step_scale": float(e["final_step_size"][0]) / 10 * 10**0.25})
    # --- std normal n=100, fixed eps ---
    q0s = [rng.standard_normal(100) for _ in range(2)]
    case("std_normal_fixed", "std_normal", {"n": 100}, q0s, [7, 8], tune=0, draws=30, adapt=False)
    # --- Radon: full adaptation from jittered starts, then a fixed-eps/fixed-mass replay from the warm state ---
    rd = models.radon()
    q0s = [rd.initial_point() + rng.uniform(-1, 1, rd.n) for _ in range(2)]
    a = case("radon_adapt", "radon", {}, q0s[:1], [201], tune=400, draws=50, adapt=True)
    b = run_reference(rd, q0s[1], seed=202, tune=400, draws=1, adapt=True)
    warm_q = [a["draws_q"][0, -1], b[0][-1]]
    warm_var = np.array([a["final_var"][0], b[2]])
    warm_eps = np.array([a["final_step_size"][0], b[3]])
    case("radon_fixed", "radon", {}, warm_q, [301, 302], tune=0, draws=40, adapt=False, var=warm_var, eps=warm_eps)
    # adaptation ON from a warm state (tuned mass matrix as initial_diag, eps0 = tuned/10 so mu = log(tuned)):
    # exercises dual averaging and both Welford window switches in the non-chaotic regime
    case("radon_warm_adapt", "radon", {}, warm_q[:1], [501], tune=250, draws=30, adapt=True, init_var=warm_var[:1],
         nuts_kwargs={"step_scale": float(warm_eps[0]) / 10 * rd.n**0.25})
    # small ragged radon (counties with 1..n obs, fewer counties than lanes), early treedepth cap exercised
    q0s = [np.zeros(2 * 7 + 5) + rng.uniform(-1, 1, 19)]
    case("radon_small_adapt", "radon", {"n_obs": 40, "n_counties": 7, "seed": 5}, q0s, [401], tune=250, draws=50,
         adapt=True, nuts_kwargs={"max_treedepth": 6, "early_max_treedepth": 4})


def team_cases():
    """Cases for the chain-per-CTA (team) kernels: std_normal n=300 and stochastic volatility."""
    rng = np.random.default_rng(21)
    q0s = [rng.standard_normal(300) for _ in range(2)]
    case("std_normal_team_fixed", "std_normal", {"n": 300}, q0s, [17, 18], tune=0, draws=20, adapt=False)
    # stochastic volatility, small T: cold adaptive run, then fixed replay from its end state
    sv = models.stochvol(T=100, seed=4)
    q0s = [sv.initial_point() + rng.uniform(-1, 1, sv.n)]
    a = case("stochvol_small_adapt", "stochvol", {"T": 100, "seed": 4}, q0s, [701], tune=300, draws=40, adapt=True)
    case("stochvol_small_fixed", "stochvol", {"T": 100, "seed": 4}, [a["draws_q"][0, -1]], [702], tune=0, draws=30,
         adapt=False, var=a["final_var"], eps=a["final_step_size"])
    # full size (T=3000, n=3003): warm up with the reference, keep only a short fixed replay
    sv = models.stochvol()
    q0 = sv.initial_point() + rng.uniform(-1, 1, sv.n)
    b = run_reference(sv, q0, seed=703, tune=250, draws=1, adapt=True)
    print("stochvol full warm-up: evals", int(b[1]["tree_size"].sum()), "final eps", b[3])
    case("stochvol_fixed", "stochvol", {}, [b[0][-1]], [704], tune=0, draws=6, adapt=False, var=np.array([b[2]]),
         eps=np.array([b[3]]))


def lockstep_cases():
    """Cases for the lock-step (GEMM-shaped) engine: dense mass Gaussian and logistic GLM."""
    rng = np.random.default_rng(31)
    mv = models.mvgauss(n=60, seed=5)
    q0s = [rng.standard_normal(60) for _ in range(2)]
    case("mvgauss_dense_fixed", "mvgauss", {"n": 60, "seed": 5}, q0s, [801, 802], tune=0, draws=30, adapt=False, dense=True)
    case("mvgauss_dense_stepadapt", "mvgauss", {"n": 60, "seed": 5}, q0s[:1], [803], tune=150, draws=30, adapt=True, dense=True)
    lg = models.logistic(n_rows=400, n_features=8, seed=3)
    q0s = [lg.initial_point() + rng.uniform(-1, 1, lg.n)]
    a = case("logistic_small_adapt", "logistic", {"n_rows": 400, "n_features": 8, "seed": 3}, q0s, [811], tune=250, draws=40,
             adapt=True)
    case("logistic_small_fixed", "logistic", {"n_rows": 400, "n_features": 8, "seed": 3}, [a["draws_q"][0, -1]], [812], tune=0,
         draws=40, adapt=False, var=a["final_var"], eps=a["final_step_size"])


def fullsize_cases():
    """Goldens for the kernel instantiations the BENCH lines of configs #3 and #5 run (VERDICT r1, weak #1):
    logistic_fused_kernel<16> (K = 128, several chain-CTAs is the test's job) and gemm_nt_dmma_kernel<8|4|2,*> +
    ls_advance_kernel<16> at n = 10^4.  Short fixed-step replays from a state the reference itself warmed up."""
    rng = np.random.default_rng(41)
    args = {"n_rows": 8192, "n_features": 128, "seed": 3}
    lg = models.logistic(**args)
    q0s = [lg.initial_point() + rng.uniform(-0.2, 0.2, lg.n) for _ in range(3)]
    a = case("logistic_k128_adapt", "logistic", args, q0s[:1], [821], tune=120, draws=4, adapt=True)
    warm = [a["draws_q"][0, -1], a["draws_q"][0, -2], a["draws_q"][0, -3]]
    case("logistic_k128_fixed", "logistic", args, warm, [822, 823, 824], tune=0, draws=3, adapt=False,
         var=np.repeat(a["final_var"], 3, axis=0), eps=np.repeat(a["final_step_size"], 3))
    os.remove(os.path.join(OUT, "logistic_k128_adapt.npz"))  # only the warm state was needed
    # dense Gaussian at full size: start from draws of the target itself (x = L z), fixed eps, mass = Sigma
    mv = models.mvgauss()
    q0s = [mv.data["L"] @ rng.standard_normal(mv.n) for _ in range(2)]
    case("mvgauss_n10000_fixed", "mvgauss", {}, q0s, [831, 832], tune=0, draws=3, adapt=False, dense=True,
         eps=np.array([0.15, 0.15]))
    d = dict(np.load(os.path.join(OUT, "mvgauss_n10000_fixed.npz")))
    for k in ("var", "init_var", "pre_var", "final_var"):  # unused by a dense-mass replay
        d[k] = np.zeros(1)
    np.savez_compressed(os.path.join(OUT, "mvgauss_n10000_fixed.npz"), **d)


def run_reference_generic(spec, q0, *, seed, tune, draws, step_kind="nuts", potential, adapt=True, step_kwargs=None):
    """One chain through the verbatim reference with a caller-built potential and step class (NUTS | HamiltonianMC)."""
    f = logp_numpy.make_logp(spec)
    start = {v.name: q0[v.offset : v.offset + v.size].copy() for v in spec.vars}
    make = ref_loader.make_hmc if step_kind == "hmc" else ref_loader.make_nuts
    step, _ = make(f, spec.var_sizes, start, potential=potential, step_rng=0, adapt_step_size=adapt, **(step_kwargs or {}))
    step.setup_chain(np.random.default_rng(seed), tune, draws)
    if tune == 0:
        step.tune = False
    pt, qs, sts, pre_rng = start, [], [], []
    for i in range(tune + draws):
        if i == tune:
            step.stop_tuning()
        s = step.rng.bit_generator.state["state"]
        pre_rng.append([s["state"] >> 64, s["state"] & (2**64 - 1), s["inc"] >> 64, s["inc"] & (2**64 - 1)])
        pt, st = step.step(pt)
        qs.append(np.concatenate([np.ravel(pt[v.name]) for v in spec.vars]))
        sts.append(st[0])
    return np.array(qs), sts, np.array(pre_rng, dtype=np.uint64), step


def f3_cases():
    """HamiltonianMC (hmc/hmc.py) and init="jitter+adapt_diag_grad" (QuadPotentialDiagAdaptExp) goldens."""
    qp = ref_loader.quadpotential()
    rng = np.random.default_rng(51)
    for name, spec_name, args in [("eight_schools", "eight_schools", {}), ("radon", "radon", {})]:
        spec = models.BUILDERS[spec_name](**args)
        n = spec.n
        C = 2
        q0s = [spec.initial_point() + rng.uniform(-1, 1, n) for _ in range(C)]
        seeds = [901 + c for c in range(C)]
        # -- HMC, adaptive (dual averaging at target 0.65 + DiagAdapt), cold start
        tune, draws = 40, 10
        Q, ST, PR = [], [], []
        for c in range(C):
            pot = qp.QuadPotentialDiagAdapt(n, q0s[c].copy(), np.ones(n), 10)
            q, sts, pre, step = run_reference_generic(spec, q0s[c], seed=seeds[c], tune=tune, draws=draws, step_kind="hmc",
                                                      potential=pot)
            Q.append(q); ST.append(sts); PR.append(pre)
        out = dict(q0=np.array(q0s), seeds=np.array(seeds), tune=tune, draws=draws, draws_q=np.array(Q), pre_rng=np.array(PR),
                   z=np.array([noise(s, tune + draws, n) for s in seeds]))
        for k, kk in [("n_steps", "tree_size"), ("accept", "mean_tree_accept"), ("energy", "energy"), ("energy_error", "energy_error"),
                      ("model_logp", "model_logp"), ("step_size", "step_size"), ("step_size_bar", "step_size_bar"),
                      ("diverging", "diverging"), ("accepted", "accepted")]:
            out["stat_" + kk] = np.array([[s[k] for s in sts] for sts in ST])
        np.savez_compressed(os.path.join(OUT, name + "_hmc_adapt.npz"), **out)
        print(name + "_hmc_adapt", "leapfrogs", int(out["stat_tree_size"].sum()), "accepted", float(out["stat_accepted"].mean()))
        # -- NUTS + DiagAdaptExp(use_grads), short discard window so the gradient-based updates start at draw 21
        tune, draws = 60, 10
        Q, ST, PR, FV = [], [], [], []
        for c in range(C):
            pot = qp.QuadPotentialDiagAdaptExp(n, q0s[c].copy(), alpha=0.02, use_grads=True, stop_adaptation=50, discard_window=10)
            q, sts, pre, step = run_reference_generic(spec, q0s[c], seed=seeds[c] + 50, tune=tune, draws=draws, potential=pot)
            Q.append(q); ST.append(sts); PR.append(pre); FV.append(np.array(step.potential._var))
        out = dict(q0=np.array(q0s), seeds=np.array(seeds) + 50, tune=tune, draws=draws, draws_q=np.array(Q), pre_rng=np.array(PR),
                   z=np.array([noise(s + 50, tune + draws, n) for s in seeds]), final_var=np.array(FV), alpha=0.02,
                   stop_adaptation=50, discard_window=10)
        for k in STAT_KEYS:
            out["stat_" + k] = np.array([[s[k] for s in sts] for sts in ST])
        np.savez_compressed(os.path.join(OUT, name + "_adapt_grad.npz"), **out)
        print(name + "_adapt_grad", "grad evals", int(out["stat_tree_size"].sum()))


def dense_any_cases():
    """QuadPotentialFull / QuadPotentialFullInv on a model that is NOT a Gaussian (Radon): the dense mass matrix is model-
    independent in the reference (quadpotential.py:633-725).  Fixed step size, start and diagonal from the radon_fixed golden,
    plus a rank-5 correlation."""
    qp = ref_loader.quadpotential()
    base = dict(np.load(os.path.join(OUT, "radon_fixed.npz")))
    spec = models.radon()
    n = spec.n
    rng = np.random.default_rng(61)
    var = base["var"][0]
    U = rng.standard_normal((n, 5)) * 0.3 * np.sqrt(var)[:, None]
    cov = np.diag(var) + U @ U.T
    cov = 0.5 * (cov + cov.T)
    A = np.linalg.inv(cov)
    A = 0.5 * (A + A.T)
    eps = float(base["eps"][0]) * 0.8
    for tag, pot_of in (("full", lambda: qp.QuadPotentialFull(cov)), ("fullinv", lambda: qp.QuadPotentialFullInv(A))):
        C, draws = 2, 8
        q0s = [base["q0"][c] for c in range(C)]
        seeds = [951 + c for c in range(C)]
        Q, ST, PR = [], [], []
        for c in range(C):
            q, sts, pre, step = run_reference_generic(spec, q0s[c], seed=seeds[c], tune=0, draws=draws, potential=pot_of(),
                                                      adapt=False, step_kwargs={"step_scale": eps * n**0.25})
            Q.append(q); ST.append(sts); PR.append(pre)
        out = dict(q0=np.array(q0s), seeds=np.array(seeds), tune=0, draws=draws, draws_q=np.array(Q), pre_rng=np.array(PR),
                   z=np.array([noise(s, draws, n) for s in seeds]), cov=cov, A=A, eps=np.full(C, eps), dense=True, adapt=False)
        for k in STAT_KEYS:
            out["stat_" + k] = np.array([[s[k] for s in sts] for sts in ST])
        np.savez_compressed(os.path.join(OUT, f"radon_dense_{tag}_fixed.npz"), **out)
        print(f"radon_dense_{tag}_fixed", "grad evals", int(out["stat_tree_size"].sum()), "mean depth", out["stat_depth"].mean())


def full_adapt_cases():
    """QuadPotentialFullAdapt (quadpotential.py:748-845; init="adapt_full", mcmc.py:1986-2005): cold start from the identity with
    weight 10, covariance and Cholesky refreshed after every tuning draw; the short window of the Eight Schools case runs two
    foreground <- background switches (window 15 -> 30 -> 60)."""
    import warnings
    qp = ref_loader.quadpotential()
    rng = np.random.default_rng(71)
    for name, window, tune, draws in [("eight_schools", 15, 50, 10), ("radon", 101, 30, 6)]:
        spec = models.BUILDERS[name]()
        n = spec.n
        C = 2
        q0s = [spec.initial_point() + rng.uniform(-1, 1, n) for _ in range(C)]
        seeds = [971 + c for c in range(C)]
        Q, ST, PR, COV = [], [], [], []
        for c in range(C):
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                pot = qp.QuadPotentialFullAdapt(n, q0s[c].copy(), np.eye(n), 10, adaptation_window=window)
            q, sts, pre, step = run_reference_generic(spec, q0s[c], seed=seeds[c], tune=tune, draws=draws, potential=pot)
            Q.append(q); ST.append(sts); PR.append(pre); COV.append(np.array(step.potential._cov))
        out = dict(q0=np.array(q0s), seeds=np.array(seeds), tune=tune, draws=draws, draws_q=np.array(Q), pre_rng=np.array(PR),
                   z=np.array([noise(s, tune + draws, n) for s in seeds]), final_cov=np.array(COV), adaptation_window=window)
        for k in STAT_KEYS:
            out["stat_" + k] = np.array([[s[k] for s in sts] for sts in ST])
        np.savez_compressed(os.path.join(OUT, name + "_full_adapt.npz"), **out)
        print(name + "_full_adapt", "grad evals", int(out["stat_tree_size"].sum()), "mean depth", out["stat_depth"].mean())


def reference_chain(spec, f, q0, seed, tune, draws, potential, adapt):
    """One chain of the verbatim reference NUTS from default_rng(seed) -> (positions [T, n], per-draw stats dicts)."""
    start = {v.name: q0[v.offset : v.offset + v.size].copy() for v in spec.vars}
    step, _ = ref_loader.make_nuts(f, spec.var_sizes, start, potential=potential, step_rng=0, adapt_step_size=adapt)
    step.setup_chain(np.random.default_rng(seed), tune, draws)
    if tune == 0:
        step.tune = False
    pt, qs, sts = start, [], []
    for i in range(tune + draws):
        if i == tune:
            step.stop_tuning()
        pt, st = step.step(pt)
        qs.append(np.concatenate([np.ravel(pt[v.name]) for v in spec.vars]))
        sts.append(st[0])
    return np.array(qs), sts, step


def record(out, key, a, limit=2000):
    """out[key] = a, or -- for an array of more than `limit` values -- its shape and the SHA-256 of its float64 bytes
    ('<key>.shape', '<key>.sha256'): enough for a bit-identity check at a fraction of the size."""
    import hashlib
    a = np.asarray(a)
    if a.size <= limit:
        out[key] = a
    else:
        out[key + ".shape"] = np.array(a.shape)
        out[key + ".sha256"] = np.array(hashlib.sha256(np.ascontiguousarray(a, dtype=np.float64).tobytes()).hexdigest())


PORT_STAT_KEYS = ["tree_size", "depth", "index_in_trajectory", "energy", "step_size", "step_size_bar", "mean_tree_accept",
                  "max_energy_error", "model_logp", "diverging", "energy_error"]


def port_cases():
    """ref_port_chains.npz: the reference chains tests/test_oracle_vs_reference.py holds oracle/nuts_numpy.py to, bit for bit
    (keys '<case>/q' and '<case>/<stat>', large arrays as digests, see record())."""
    import warnings
    qp = ref_loader.quadpotential()
    out = {}
    for name, adapt, tune, draws in [("eight_schools", False, 0, 25), ("eight_schools", True, 220, 30), ("radon", True, 130, 10),
                                     ("std_normal", False, 0, 10)]:
        spec = models.std_normal(40) if name == "std_normal" else models.BUILDERS[name]()
        n = spec.n
        q0 = spec.initial_point() + np.random.default_rng(1).uniform(-1, 1, n)
        pot = qp.QuadPotentialDiagAdapt(n, q0.copy(), np.ones(n), 10) if adapt else qp.QuadPotentialDiag(np.ones(n))
        qs, sts, _ = reference_chain(spec, logp_numpy.make_logp(spec), q0, 77, tune, draws, pot, adapt)
        key = f"diag-{name}-{adapt}-{tune}-{draws}"
        record(out, key + "/q", qs)
        for k in PORT_STAT_KEYS:
            record(out, f"{key}/{k}", [s[k] for s in sts])
    # QuadPotentialFull, fixed step size
    spec = models.mvgauss(n=15, seed=2)
    q0 = np.random.default_rng(3).normal(size=15)
    qs, _, _ = reference_chain(spec, logp_numpy.make_logp(spec), q0, 5, 0, 12, qp.QuadPotentialFull(spec.data["cov"]), False)
    record(out, "dense/q", qs)
    # QuadPotentialFullAdapt (init="adapt_full") through the first window switch for Eight Schools
    for name, tune, draws in [("eight_schools", 130, 10), ("radon", 60, 5)]:
        spec = models.BUILDERS[name]()
        n = spec.n
        q0 = spec.initial_point() + np.random.default_rng(4).uniform(-1, 1, n)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            pot = qp.QuadPotentialFullAdapt(n, q0.copy(), np.eye(n), 10)
        qs, sts, step = reference_chain(spec, logp_numpy.make_logp(spec), q0, 91, tune, draws, pot, True)
        key = f"dense_adapt-{name}"
        record(out, key + "/q", qs)
        for k in ("tree_size", "depth", "index_in_trajectory", "energy", "step_size"):
            record(out, f"{key}/{k}", [s[k] for s in sts])
        record(out, key + "/cov", step.potential._cov)
        record(out, key + "/chol", step.potential._chol)
    # the SURVEY 8c known answer of the loader: Eight Schools from 0, unit mass, seed 20240922
    spec = models.eight_schools()
    qs, sts, _ = reference_chain(spec, logp_numpy.make_logp(spec), np.zeros(10), 20240922, 0, 5, qp.QuadPotentialDiag(np.ones(10)),
                                 False)
    assert [(s["depth"], s["tree_size"], s["index_in_trajectory"]) for s in sts] == \
        [(4, 15, -10), (5, 31, -10), (5, 31, -11), (5, 31, 13), (4, 15, 10)], "the reference loader is broken"
    record(out, "self_check/q", qs)
    for k in PORT_STAT_KEYS:
        record(out, f"self_check/{k}", [s[k] for s in sts])
    np.savez_compressed(os.path.join(OUT, "ref_port_chains.npz"), **out)


def step_seam_case():
    """ref_step_seam.npz: the reference NUTS (default potential) driven like _iter_sample drives a step method, the run
    tests/test_step_seam.py drives B200NUTS through: positions, every per-draw stat with a value, the stats keys, and where
    the caller's generator is left."""
    spec = models.eight_schools()
    f = logp_numpy.make_logp(spec)
    q0 = spec.initial_point() + np.random.default_rng(3).uniform(-1, 1, spec.n)
    start = {v.name: q0[v.offset : v.offset + v.size].copy() for v in spec.vars}
    ref, _ = ref_loader.make_nuts(f, spec.var_sizes, start, step_rng=0)  # default potential: DiagAdapt(zeros, ones, 10)
    tune, draws = 60, 25
    ref.setup_chain(np.random.default_rng(20240922), tune, draws)  # the loop of _iter_sample
    ref.tune = True
    ref.reset_tuning()
    point, qs, sts = dict(start), [], []
    for i in range(tune + draws):
        if i == tune:
            ref.stop_tuning()
        point, st = ref.step(point)
        qs.append(np.concatenate([np.ravel(point[k]) for k in start]))
        sts.append(st[0])
    qs = np.array(qs)
    s = ref.rng.bit_generator.state["state"]["state"]
    out = dict(q=qs, rng_after=np.array([s >> 64, s & (2**64 - 1)], dtype=np.uint64),
               stats_keys=np.array(sorted(sts[0])), stats_dtypes_shapes_keys=np.array(sorted(type(ref).stats_dtypes_shapes)))
    for k in ("depth", "tree_size", "index_in_trajectory", "diverging", "reached_max_treedepth", "divergences", "step_size",
              "step_size_bar", "mean_tree_accept", "energy", "energy_error", "max_energy_error", "model_logp"):
        out["stat_" + k] = np.array([x[k] for x in sts])
    np.savez_compressed(os.path.join(OUT, "ref_step_seam.npz"), **out)


def potential_objects():
    """The reference QuadPotential objects tests/test_potentials.py hands to pymc_b200.potentials, keyed by label."""
    import warnings
    qp = ref_loader.quadpotential()
    n = 4
    rng = np.random.default_rng(0)
    v, mean = rng.uniform(0.5, 2.0, n), rng.normal(size=n)
    B = rng.normal(size=(n, n))
    cov = B @ B.T + n * np.eye(n)
    objs = {
        "diag": qp.QuadPotentialDiag(v),
        "diag_adapt": qp.QuadPotentialDiagAdapt(n, mean, v, 7, adaptation_window=33, discard_window=9),
        "diag_adapt_exp": qp.QuadPotentialDiagAdaptExp(n, mean, alpha=0.03, use_grads=True, stop_adaptation=120),
        "diag_adapt_exp_nostop": qp.QuadPotentialDiagAdaptExp(n, mean, alpha=0.03, use_grads=True),
        "full": qp.QuadPotentialFull(cov),
        "full_inv": qp.QuadPotentialFullInv(cov),
        "diag_adapt_early": qp.QuadPotentialDiagAdapt(n, mean, v, 7, early_update=True),
        "diag_adapt_multiplier": qp.QuadPotentialDiagAdapt(n, mean, v, 7, adaptation_window_multiplier=2),
        "diag_adapt_exp_nograds": qp.QuadPotentialDiagAdaptExp(n, mean, alpha=0.03),
        "diag_n3": qp.QuadPotentialDiag(np.ones(3)),
    }
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        objs["full_adapt"] = qp.QuadPotentialFullAdapt(n, mean, np.diag(v), 10, adaptation_window=40,
                                                       adaptation_window_multiplier=3, update_window=5)
        objs["full_adapt_offdiag"] = qp.QuadPotentialFullAdapt(n, mean, cov, 10)
    # the Eight Schools potentials of the whole-run sampler test
    n = 10
    rng = np.random.default_rng(1)
    mean, diag = rng.normal(size=n), rng.uniform(0.5, 2.0, n)
    objs["es_diag_adapt"] = qp.QuadPotentialDiagAdapt(n, mean, diag, 4, adaptation_window=20, discard_window=5)
    objs["es_diag"] = qp.QuadPotentialDiag(diag)
    return objs


def potential_cases():
    """ref_potentials.json: {label: {"__class__": class name, attribute: value}} of the reference QuadPotential objects, every
    plain-valued attribute (numbers, strings, float arrays as lists); generators and running estimators are left out."""
    import json
    out = {}
    for label, obj in potential_objects().items():
        d = out[label] = {"__class__": type(obj).__name__}
        for k, val in vars(obj).items():
            if isinstance(val, np.ndarray) and val.dtype == np.float64:
                d[k] = val.tolist()
            elif isinstance(val, (bool, int, float, str, np.integer, np.floating, np.bool_)):
                d[k] = val.item() if isinstance(val, np.generic) else val
    with open(os.path.join(OUT, "ref_potentials.json"), "w") as fh:
        json.dump(out, fh, indent=1)
        fh.write("\n")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "seams":
        port_cases()
        step_seam_case()
        potential_cases()
        raise SystemExit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "lockstep":
        lockstep_cases()
        raise SystemExit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "dense_any":
        dense_any_cases()
        raise SystemExit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "full_adapt":
        full_adapt_cases()
        raise SystemExit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "f3":
        f3_cases()
        raise SystemExit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "fullsize":
        fullsize_cases()
        raise SystemExit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "team":
        team_cases()
        raise SystemExit(0)
    main()
