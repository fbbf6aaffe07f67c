"""CPU: seam B2 inbound -- the reference's own QuadPotential objects (class name and attribute values, recorded from the
verbatim classes in tests/golden/ref_potentials.npz) are read and mapped onto the engine's mass kinds (pymc_b200/potentials.py),
and ``sample_b200_nuts(nuts_kwargs={"potential": obj})`` runs the chain that potential defines (checked on the oracle-backed
engine, which is bit-identical to the reference)."""
import numpy as np
import pytest

from b200_helpers import OracleEngine, reference_potential
from pymc_b200 import models, potentials, sampling


def test_reference_potential_objects_map_onto_the_engine_kinds():
    # the objects were built from these values (oracle/make_golden.py, potential_objects)
    n = 4
    rng = np.random.default_rng(0)
    v, mean = rng.uniform(0.5, 2.0, n), rng.normal(size=n)
    k = potentials.engine_kwargs(reference_potential("diag"), n)  # QuadPotentialDiag(v)
    assert k["mass"] == "diag" and np.array_equal(k["var0"], v)
    # QuadPotentialDiagAdapt(n, mean, v, 7, adaptation_window=33, discard_window=9)
    k = potentials.engine_kwargs(reference_potential("diag_adapt"), n)
    assert (k["mass"], k["mass_initial_weight"], k["adaptation_window"], k["discard_window"]) == ("diag_adapt", 7.0, 33, 9)
    assert np.array_equal(k["var0"], v) and np.array_equal(k["mean0"], mean)
    # QuadPotentialDiagAdaptExp(n, mean, alpha=0.03, use_grads=True, stop_adaptation=120), then without stop_adaptation
    k = potentials.engine_kwargs(reference_potential("diag_adapt_exp"), n)
    assert (k["mass"], k["mass_alpha"], k["stop_adaptation"], k["discard_window"]) == ("diag_adapt_grad", 0.03, 120, 50)
    assert potentials.engine_kwargs(reference_potential("diag_adapt_exp_nostop"), n)["stop_adaptation"] is None
    B = rng.normal(size=(n, n))
    cov = B @ B.T + n * np.eye(n)
    k = potentials.engine_kwargs(reference_potential("full"), n)  # QuadPotentialFull(cov)
    assert k["mass"] == "dense" and np.array_equal(k["dense_cov"], cov)
    k = potentials.engine_kwargs(reference_potential("full_inv"), n)  # QuadPotentialFullInv(cov)
    assert k["mass"] == "dense" and np.allclose(k["dense_inverse"], cov, rtol=1e-13, atol=1e-13)
    # QuadPotentialFullAdapt(n, mean, diag(v), 10, adaptation_window=40, adaptation_window_multiplier=3, update_window=5)
    k = potentials.engine_kwargs(reference_potential("full_adapt"), n)
    assert (k["mass"], k["mass_initial_weight"], k["adaptation_window"], k["window_multiplier"], k["update_window"]) == \
           ("dense_adapt", 10.0, 40, 3.0, 5)
    assert np.array_equal(k["var0"], v) and np.array_equal(k["mean0"], mean)
    with pytest.raises(NotImplementedError, match="non-diagonal"):  # QuadPotentialFullAdapt(n, mean, cov, 10)
        potentials.engine_kwargs(reference_potential("full_adapt_offdiag"), n)
    # options the kernels do not implement are refused by name, never ignored
    with pytest.raises(NotImplementedError, match="early_update"):  # QuadPotentialDiagAdapt(n, mean, v, 7, early_update=True)
        potentials.engine_kwargs(reference_potential("diag_adapt_early"), n)
    with pytest.raises(NotImplementedError, match="multiplier"):  # ... adaptation_window_multiplier=2
        potentials.engine_kwargs(reference_potential("diag_adapt_multiplier"), n)
    with pytest.raises(NotImplementedError, match="use_grads"):  # QuadPotentialDiagAdaptExp(n, mean, alpha=0.03)
        potentials.engine_kwargs(reference_potential("diag_adapt_exp_nograds"), n)

    base = reference_potential("diag")

    class Mine(type(base)):  # the user-subclass case of tests/step_methods/hmc/test_quadpotential.py:138-157
        def velocity(self, x, out=None):
            return x

    mine = Mine()
    vars(mine).update(vars(base))
    with pytest.raises(NotImplementedError, match="subclass"):
        potentials.engine_kwargs(mine, n)
    with pytest.raises(ValueError, match="expected 4 values"):  # QuadPotentialDiag(np.ones(3))
        potentials.engine_kwargs(reference_potential("diag_n3"), n)


def test_a_potential_object_defines_the_chain_the_sampler_runs():
    """nuts_kwargs={"potential": QuadPotentialDiagAdapt(...)}: every chain equals the reference chain under that potential."""
    from oracle import logp_numpy, nuts_numpy
    from pymc_b200 import rng as brng

    spec = models.eight_schools()
    n, chains, seed, tune, draws = spec.n, 2, 6, 45, 8
    rng = np.random.default_rng(1)
    mean, diag = rng.normal(size=n), rng.uniform(0.5, 2.0, n)
    pot = reference_potential("es_diag_adapt")  # QuadPotentialDiagAdapt(n, mean, diag, 4, adaptation_window=20, discard_window=5)
    res = sampling.sample_b200_nuts(draws, tune=tune, chains=chains, random_seed=seed, model=OracleEngine(spec), momentum="numpy",
                                    keep_untransformed=True, nuts_kwargs={"potential": pot})
    step_rngs, pot_rngs, jitter_seeds = brng.chain_generators(seed, chains)
    q0 = sampling.initial_points(spec, chains, jitter_seeds)
    f = logp_numpy.make_logp(spec)
    for c in range(chains):
        m = nuts_numpy.DiagMass(diag, adapt=True, initial_mean=mean.copy(), initial_weight=4, adaptation_window=20, discard_window=5)
        o = nuts_numpy.Oracle(f, m)
        o.rng, o.mass.rng = step_rngs[c], pot_rngs[c]
        qs, _ = o.run(q0[c], tune, draws)
        assert np.array_equal(qs[tune:], res.unconstrained[c])
    fixed = sampling.sample_b200_nuts(draws, tune=tune, chains=1, random_seed=seed, model=OracleEngine(spec), momentum="numpy",
                                      keep_untransformed=True, nuts_kwargs={"potential": reference_potential("es_diag")})
    m = nuts_numpy.DiagMass(diag, adapt=False)
    o = nuts_numpy.Oracle(f, m)
    sr, pr, js = brng.chain_generators(seed, 1)
    o.rng, o.mass.rng = sr[0], pr[0]
    qs, _ = o.run(sampling.initial_points(spec, 1, js)[0], tune, draws)
    assert np.array_equal(qs[tune:], fixed.unconstrained[0])
    with pytest.raises(ValueError, match="contradicts"):
        sampling.sample_b200_nuts(2, tune=2, chains=1, random_seed=1, model=OracleEngine(spec), momentum="numpy",
                                  nuts_kwargs={"potential": pot, "adaptation_window": 99})
