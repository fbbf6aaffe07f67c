"""CPU: oracle/nuts_numpy.py must be BIT-IDENTICAL to the reference's own nuts.py / integration.py / quadpotential.py /
step_sizes.py.  The reference chains were recorded from those files loaded verbatim (oracle/ref_loader.py) into
tests/golden/ref_port_chains.npz by ``python -m oracle.make_golden seams``; every case below replays the same start, seed
and potential through the port.  Arrays of more than 2000 values are recorded as their shape and the SHA-256 of their
float64 bytes, which pins them bit for bit as well."""
import hashlib

import numpy as np
import pytest

from oracle import logp_numpy, nuts_numpy
from pymc_b200 import models


@pytest.fixture(scope="module")
def ref(golden):
    return golden("ref_port_chains")


def assert_recorded(ref, key, got):
    """`got` equals the recorded reference array `key` bit for bit."""
    if key in ref:
        assert np.array_equal(ref[key], got), key
    else:
        got = np.ascontiguousarray(got, dtype=np.float64)
        assert tuple(ref[key + ".shape"]) == got.shape, key
        assert hashlib.sha256(got.tobytes()).hexdigest() == str(ref[key + ".sha256"]), key


def _port_chain(spec, f, q0, seed, tune, draws, adapt):
    mass = nuts_numpy.DiagMass(np.ones(spec.n), adapt=adapt, initial_mean=q0.copy(), initial_weight=10)
    o = nuts_numpy.Oracle(f, mass, adapt_step_size=adapt)
    o.setup_chain(np.random.default_rng(seed))
    if tune == 0:
        o.tune = False
    return o.run(q0, tune, draws)


STAT_KEYS = ("tree_size", "depth", "index_in_trajectory", "energy", "step_size", "step_size_bar", "mean_tree_accept",
             "max_energy_error", "model_logp", "diverging", "energy_error")


@pytest.mark.parametrize("name,adapt,tune,draws", [
    ("eight_schools", False, 0, 25), ("eight_schools", True, 220, 30), ("radon", True, 130, 10), ("std_normal", False, 0, 10),
])
def test_port_is_bit_identical_to_reference(ref, name, adapt, tune, draws):
    """QuadPotentialDiagAdapt(n, q0, ones, 10) + dual averaging (adapt) or QuadPotentialDiag(ones), seed 77."""
    spec = models.std_normal(40) if name == "std_normal" else models.BUILDERS[name]()
    f = logp_numpy.make_logp(spec)
    q0 = spec.initial_point() + np.random.default_rng(1).uniform(-1, 1, spec.n)
    key = f"diag-{name}-{adapt}-{tune}-{draws}"
    qo, so = _port_chain(spec, f, q0, 77, tune, draws, adapt)
    assert_recorded(ref, key + "/q", qo)
    for k in STAT_KEYS:
        assert_recorded(ref, f"{key}/{k}", so[k])


def test_dense_mass_matches_reference(ref):
    """QuadPotentialFull (quadpotential.py:680-725) vs DenseMass, fixed step size."""
    spec = models.mvgauss(n=15, seed=2)
    f = logp_numpy.make_logp(spec)
    q0 = np.random.default_rng(3).normal(size=15)
    o = nuts_numpy.Oracle(f, nuts_numpy.DenseMass(spec.data["cov"]), adapt_step_size=False)
    o.setup_chain(np.random.default_rng(5))
    o.tune = False
    qo, _ = o.run(q0, 0, 12)
    assert_recorded(ref, "dense/q", qo)


@pytest.mark.parametrize("name,tune,draws", [("eight_schools", 130, 10), ("radon", 60, 5)])
def test_dense_adapt_mass_matches_reference(ref, name, tune, draws):
    """QuadPotentialFullAdapt (quadpotential.py:748-845, init="adapt_full": mcmc.py:1986-1996) vs DenseAdaptMass, through the
    first window switch for Eight Schools (foreground <- background at delta = 101)."""
    spec = models.BUILDERS[name]()
    n = spec.n
    f = logp_numpy.make_logp(spec)
    q0 = spec.initial_point() + np.random.default_rng(4).uniform(-1, 1, n)
    o = nuts_numpy.Oracle(f, nuts_numpy.DenseAdaptMass(n, q0.copy(), np.eye(n), 10))
    o.setup_chain(np.random.default_rng(91))
    qo, so = o.run(q0, tune, draws)
    key = f"dense_adapt-{name}"
    assert qo.shape == (tune + draws, n)
    assert_recorded(ref, key + "/q", qo)
    for k in ("tree_size", "depth", "index_in_trajectory", "energy", "step_size"):
        assert_recorded(ref, f"{key}/{k}", so[k])
    assert_recorded(ref, key + "/cov", o.mass.cov)
    assert_recorded(ref, key + "/chol", o.mass.chol)


def test_loader_self_check_known_answer(ref):
    """SURVEY 8c: five Eight-Schools draws of the verbatim reference (depth, tree_size, index_in_trajectory), as recorded, and
    the port on the same case."""
    sr = {k: ref["self_check/" + k] for k in STAT_KEYS}
    qr = ref["self_check/q"]
    got = [(int(d), int(t), int(i)) for d, t, i in zip(sr["depth"], sr["tree_size"], sr["index_in_trajectory"])]
    assert got == [(4, 15, -10), (5, 31, -10), (5, 31, -11), (5, 31, 13), (4, 15, 10)]
    assert abs(sr["energy"][0] - 48.33000583528482) < 1e-10
    assert abs(qr[0][0] - (-0.4558081288677123)) < 1e-12 and abs(qr[0][1] - 2.267682240205048) < 1e-12
    spec = models.eight_schools()
    qo, so = _port_chain(spec, logp_numpy.make_logp(spec), np.zeros(10), 20240922, 0, 5, False)
    assert_recorded(ref, "self_check/q", qo)
    for k in STAT_KEYS:
        assert_recorded(ref, "self_check/" + k, so[k])
