"""Shared helpers: model specs per golden file, GPU replay (free-running and single-draw), oracle replay, recorded reference
potential objects."""
import json
import os

import numpy as np

from pymc_b200 import _lib, models

_REF_POTENTIALS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_potentials.json")
_REF_CLASSES = {}

SPEC_OF = {
    "std_normal_fixed": lambda: models.std_normal(100),
    "eight_schools_fixed": models.eight_schools,
    "eight_schools_adapt": models.eight_schools,
    "eight_schools_warm_adapt": models.eight_schools,
    "radon_fixed": models.radon,
    "radon_adapt": models.radon,
    "radon_warm_adapt": models.radon,
    "radon_small_adapt": lambda: models.radon(40, 7, 5),
    "std_normal_team_fixed": lambda: models.std_normal(300),
    "stochvol_small_adapt": lambda: models.stochvol(T=100, seed=4),
    "stochvol_small_fixed": lambda: models.stochvol(T=100, seed=4),
    "stochvol_fixed": models.stochvol,
    "mvgauss_dense_fixed": lambda: models.mvgauss(n=60, seed=5),
    "mvgauss_dense_stepadapt": lambda: models.mvgauss(n=60, seed=5),
    "logistic_small_adapt": lambda: models.logistic(n_rows=400, n_features=8, seed=3),
    "logistic_small_fixed": lambda: models.logistic(n_rows=400, n_features=8, seed=3),
    "logistic_k128_fixed": lambda: models.logistic(n_rows=8192, n_features=128, seed=3),
    "mvgauss_n10000_fixed": models.mvgauss,
}
TREE_KW = {"radon_small_adapt": dict(max_treedepth=6, early_max_treedepth=4)}
DISCRETE = ["depth", "tree_size", "index_in_trajectory", "diverging", "reached_max_treedepth"]
CONTINUOUS = ["step_size", "step_size_bar", "mean_tree_accept", "energy", "energy_error", "max_energy_error", "model_logp"]


def relerr(a, b):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    with np.errstate(invalid="ignore"):
        e = np.abs(a - b) / np.maximum(1e-300, np.maximum(np.abs(a), np.abs(b)))
    e = np.where((a == b) | (np.isnan(a) & np.isnan(b)), 0.0, e)
    return float(np.max(e)) if e.size else 0.0


def start_states(d):
    """PCG64 stream states at the start of every golden chain (pre_rng of draw 0)."""
    return stream_states(d["pre_rng"][:, 0])


def stream_states(arr_u64x4):
    a = np.array(arr_u64x4, dtype=np.uint64, copy=True).reshape(-1, 4)  # copy: the engine advances states in place
    return a.view(_lib.PCG64_DTYPE).reshape(-1)


def gpu_free_run(cm, d, name, draws=None):
    """Replay a golden case through b200_nuts_run with the golden inputs (start, streams, momentum noise)."""
    tune, T = int(d["tune"]), int(d["tune"]) + int(d["draws"])
    if draws is not None:  # only the first `draws` iterations (all must be in one phase)
        assert draws <= tune or tune == 0
        T = draws
    kw = dict(TREE_KW.get(name, {}))
    dense = bool(d["dense"]) if "dense" in d else False
    if dense:
        kw.update(mass="dense", adapt_step_size=bool(d["adapt"]))
        if bool(d["adapt"]):
            t, dr = (T, 0) if draws is not None else (tune, int(d["draws"]))
        else:
            t, dr = 0, T
            if not np.isnan(d["eps"][0]):
                kw["eps0"] = d["eps"]
    elif bool(d["adapt"]):
        kw.update(mass="diag_adapt", mean0=d["q0"], var0=d["init_var"], adapt_step_size=True, step_scale=float(d["step_scale"]))
        t, dr = (T, 0) if draws is not None else (tune, int(d["draws"]))
    else:
        kw.update(mass="diag", var0=d["var"], adapt_step_size=False)
        if not np.isnan(d["eps"][0]):
            kw["eps0"] = d["eps"]
        t, dr = 0, T
    states = start_states(d)
    res = cm.nuts_run(d["q0"], states, tune=t, draws=dr, z=np.ascontiguousarray(d["z"][:, :T]), **kw)
    return res, states


def gpu_single_draws(cm, d, name, chain=0):
    """Teacher forcing: every golden draw t replayed as an independent one-iteration chain started from the
    golden state before it (position, stream position, mass matrix, step size)."""
    T = int(d["tune"]) + int(d["draws"])
    q_prev = np.concatenate([d["q0"][chain][None], d["draws_q"][chain][:-1]])
    states = stream_states(d["pre_rng"][chain])
    kw = dict(TREE_KW.get(name, {}))
    tune = int(d["tune"])
    # draws with iteration index < 200 inside tuning use early_max_treedepth: replay them as tuning iterations
    out = {}
    early = np.arange(T) < min(tune, 200)
    for sel, as_tune in ((early, True), (~early, False)):
        if not sel.any():
            continue
        res = cm.nuts_run(q_prev[sel], states[sel].copy(), tune=1 if as_tune else 0, draws=0 if as_tune else 1,
                          z=np.ascontiguousarray(d["z"][chain][sel][:, None, :]), mass="diag", var0=d["pre_var"][chain][sel],
                          adapt_step_size=False, eps0=d["used_eps"][chain][sel], **kw)
        out[as_tune] = (sel, res)
    n = q_prev.shape[1]
    dq = np.empty((T, n))
    st = {}
    for as_tune, (sel, res) in out.items():
        dq[sel] = res.draws[:, 0]
        for k, v in res.stats.items():
            st.setdefault(k, np.zeros(T, dtype=v.dtype))[sel] = v[:, 0]
    return dq, st


def reference_potential(label):
    """One of the reference's QuadPotential objects as ``pymc_b200.potentials`` sees it: an instance of a class with the
    reference class's name, carrying the plain-valued attributes the reference object had after construction
    (tests/golden/ref_potentials.json, recorded from the verbatim classes by ``python -m oracle.make_golden seams``)."""
    with open(_REF_POTENTIALS) as fh:
        attrs = json.load(fh)[label]
    name = attrs.pop("__class__")
    obj = _REF_CLASSES.setdefault(name, type(name, (), {}))()
    for k, v in attrs.items():
        setattr(obj, k, np.array(v, dtype=np.float64) if isinstance(v, list) else v)
    return obj


def discrete_equal(st, d, chain):
    ok = np.ones(len(st["depth"]), dtype=bool)
    for k in DISCRETE:
        if k == "reached_max_treedepth" :
            continue
        ok &= np.asarray(st[k]).astype(np.int64) == np.asarray(d["stat_" + k][chain]).astype(np.int64)
    return ok


class OracleEngine:
    """CPU stand-in for ``pymc_b200.engine.CompiledModel`` in host-logic tests: same ``nuts_run`` / ``logp_dlogp``
    interface, every chain run through oracle/nuts_numpy.py (bit-identical to the reference).  Lets the seams above the
    C ABI (step method, whole-run sampler, chain sharding over torch.distributed) be tested without a GPU."""

    def __init__(self, spec):
        from oracle import logp_numpy

        self.spec, self.n = spec, spec.n
        self.f = logp_numpy.make_logp(spec)

    def set_dense_mass(self, cov=None, *, inverse=None):
        assert cov is not None, "the stand-in takes QuadPotentialFull(cov) only"
        self.dense_cov = np.array(cov, dtype=np.float64)

    def logp_dlogp(self, q):
        q = np.asarray(q, dtype=np.float64).reshape(-1, self.n)
        out = [self.f(x) for x in q]
        return np.array([o[0] for o in out]), np.array([o[1] for o in out])

    def nuts_run(self, q0, rng_states, *, tune, draws, z=None, mean0=None, var0=None, mass="diag_adapt", store_warmup=True,
                 philox_seed=0, mass_initial_weight=10.0, step_scale=0.25, target_accept=0.8, gamma=0.05, k=0.75, t0=10.0,
                 Emax=1000.0, adapt_step_size=True, max_treedepth=10, early_max_treedepth=8, chain_offset=0, **unused):
        from oracle import nuts_numpy
        from pymc_b200.engine import NutsResult

        assert mass in ("diag", "diag_adapt", "dense_adapt", "dense") and z is not None, "the stand-in draws momentum from the host stream only"
        self.last_q0 = np.array(q0, dtype=np.float64)
        self.last_call = dict(mass=mass, var0=None if var0 is None else np.array(var0), mean0=None if mean0 is None else np.array(mean0),
                              mass_initial_weight=mass_initial_weight)
        q0 = np.asarray(q0, dtype=np.float64).reshape(-1, self.n)
        C, T = q0.shape[0], tune + draws
        qs_all, st_all = [], []
        for c in range(C):
            v0 = np.ones(self.n) if var0 is None else np.asarray(var0)[c]
            m0 = np.zeros(self.n) if mean0 is None else np.asarray(mean0)[c]
            if mass == "dense_adapt":  # QuadPotentialFullAdapt(n, mean, diag(var0), weight): init="adapt_full"
                m = nuts_numpy.DenseAdaptMass(self.n, m0.copy(), np.diag(v0), mass_initial_weight,
                                              adaptation_window=unused.get("adaptation_window", 101))
            elif mass == "diag":  # QuadPotentialDiag(v)
                m = nuts_numpy.DiagMass(v0, adapt=False)
            elif mass == "dense":  # QuadPotentialFull(cov) from set_dense_mass
                m = nuts_numpy.DenseMass(self.dense_cov)
            else:
                m = nuts_numpy.DiagMass(v0, adapt=True, initial_mean=m0.copy(), initial_weight=mass_initial_weight,
                                        adaptation_window=unused.get("adaptation_window", 101),
                                        discard_window=unused.get("discard_window", 50))
            o = nuts_numpy.Oracle(self.f, m, step_scale=step_scale, adapt_step_size=adapt_step_size, target_accept=target_accept,
                                  gamma=gamma, k=k, t0=t0, Emax=Emax, max_treedepth=max_treedepth,
                                  early_max_treedepth=early_max_treedepth)
            g = np.random.default_rng(0)
            st = g.bit_generator.state
            rec = rng_states[c]
            st["state"]["state"] = (int(rec["state_hi"]) << 64) | int(rec["state_lo"])
            st["state"]["inc"] = (int(rec["inc_hi"]) << 64) | int(rec["inc_lo"])
            st["has_uint32"], st["uinteger"] = 0, 0
            g.bit_generator.state = st
            o.rng = g
            qs, stats = o.run(q0[c], tune, draws, z=np.asarray(z)[c])
            s = g.bit_generator.state["state"]
            rng_states[c] = (s["state"] >> 64, s["state"] & (2**64 - 1), s["inc"] >> 64, s["inc"] & (2**64 - 1))
            w = 0 if store_warmup else tune
            qs_all.append(qs[w:])
            st_all.append({k_: np.asarray(v)[w:] for k_, v in stats.items()})
        dt = {"depth": np.int32, "tree_size": np.int32, "index_in_trajectory": np.int32, "diverging": np.uint8,
              "reached_max_treedepth": np.uint8}
        names = [nm for nm, _ in _lib.STAT_FIELDS]  # exactly the arrays b200_stats carries
        stats = {k_: np.stack([s[k_] for s in st_all]).astype(dt.get(k_, np.float64)) for k_ in names}
        return NutsResult(draws=np.stack(qs_all), stats=stats, summary={"bad_energy_at": np.full(C, -1, dtype=np.int32)},
                          kernel_ms=0.0, launches=0, tune=tune, n_draws=draws, store_warmup=store_warmup)
