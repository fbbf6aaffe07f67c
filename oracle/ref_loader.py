"""TEST INFRASTRUCTURE ONLY -- loads the reference's own HMC/NUTS sources verbatim.

The reference sampler (tree building, leapfrog, mass matrix, step-size adaptation) is pure
NumPy/SciPy.  ``import pymc`` fails in this image because PyTensor / xarray / arviz are absent,
but the HMC files themselves run unmodified once a few stub modules stand in for those imports
(SURVEY.md section 8c).  This module builds those stubs in ``sys.modules`` and executes the
reference files *from where they lie* under ``/root/reference`` -- nothing is copied.

It is used for one thing: ``oracle/make_golden.py`` generates the committed golden vectors in
``tests/golden/`` with it, among them the recorded reference chains, step-method run and potential
objects the tests compare with.  The tests themselves never need the reference tree.

Callers must check ``available()`` first.
Nothing in ``pymc_b200`` imports this file.
"""
from __future__ import annotations

import importlib
import importlib.util
import os
import sys
import types

import numpy as np

REFERENCE_ROOT = os.environ.get("B200_REFERENCE_ROOT", "/root/reference")

# load order matters: each file only imports names that are already registered
_FILES = [
    ("pymc.exceptions", "pymc/exceptions.py"),
    ("pymc.vartypes", "pymc/vartypes.py"),
    ("pymc.blocking", "pymc/blocking.py"),
    ("pymc.util", "pymc/util.py"),
    ("pymc.stats.convergence", "pymc/stats/convergence.py"),
    ("pymc.step_methods.state", "pymc/step_methods/state.py"),
    ("pymc.step_methods.compound", "pymc/step_methods/compound.py"),
    ("pymc.step_methods.arraystep", "pymc/step_methods/arraystep.py"),
    ("pymc.step_methods.step_sizes", "pymc/step_methods/step_sizes.py"),
    ("pymc.step_methods.hmc.quadpotential", "pymc/step_methods/hmc/quadpotential.py"),
    ("pymc.step_methods.hmc.integration", "pymc/step_methods/hmc/integration.py"),
    ("pymc.step_methods.hmc.base_hmc", "pymc/step_methods/hmc/base_hmc.py"),
    ("pymc.step_methods.hmc.nuts", "pymc/step_methods/hmc/nuts.py"),
    ("pymc.step_methods.hmc.hmc", "pymc/step_methods/hmc/hmc.py"),
]

_loaded: dict[str, types.ModuleType] | None = None


def available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "pymc/step_methods/hmc/nuts.py"))


def _pkg(name: str) -> types.ModuleType:
    m = types.ModuleType(name)
    m.__path__ = []  # mark as package
    sys.modules[name] = m
    return m


def _install_stubs() -> None:
    # ---- pytensor: only config.floatX, shared(), utils.lazy_scipy_module and two type names
    pt = _pkg("pytensor")
    pt.config = types.SimpleNamespace(floatX="float64")

    class _Shared:
        def __init__(self, value):
            self._v = value

        def set_value(self, v, borrow=False):
            self._v = v

        def get_value(self, borrow=False):
            return self._v

    pt.shared = lambda value, **kw: _Shared(value)
    ptu = types.ModuleType("pytensor.utils")
    ptu.lazy_scipy_module = lambda name: importlib.import_module("scipy." + name)
    sys.modules["pytensor.utils"] = ptu
    pt.utils = ptu
    ptc = types.ModuleType("pytensor.compile")
    ptc.SharedVariable = _Shared
    sys.modules["pytensor.compile"] = ptc
    ptg = _pkg("pytensor.graph")
    ptgb = types.ModuleType("pytensor.graph.basic")

    class Variable:  # noqa: D401 - placeholder type
        pass

    ptgb.Variable = Variable
    sys.modules["pytensor.graph.basic"] = ptgb
    ptg.basic = ptgb

    # ---- xarray: two type names used in annotations / isinstance
    xr = types.ModuleType("xarray")
    xr.Dataset = type("Dataset", (), {})
    xr.DataTree = type("DataTree", (), {})
    sys.modules["xarray"] = xr

    # ---- pymc package shells
    pm = _pkg("pymc")
    _pkg("pymc.stats")
    sm = _pkg("pymc.step_methods")
    hm = _pkg("pymc.step_methods.hmc")
    pm.step_methods = sm
    sm.hmc = hm

    model = types.ModuleType("pymc.model")
    model.modelcontext = lambda m: m
    model.Point = lambda *a, **k: dict(*a)
    sys.modules["pymc.model"] = model
    ptf = types.ModuleType("pymc.pytensorf")
    ptf.floatX = lambda x: np.asarray(x, dtype="float64")
    sys.modules["pymc.pytensorf"] = ptf
    tun = types.ModuleType("pymc.tuning")
    tun.guess_scaling = lambda *a, **k: (_ for _ in ()).throw(NotImplementedError("guess_scaling"))
    sys.modules["pymc.tuning"] = tun


def load() -> dict[str, types.ModuleType]:
    """Execute the reference HMC files under stubs; returns {module name: module}."""
    global _loaded
    if _loaded is not None:
        return _loaded
    if not available():
        raise RuntimeError(f"reference not found under {REFERENCE_ROOT}")
    if "pymc" in sys.modules and not hasattr(sys.modules["pymc"], "__b200_stub__"):
        raise RuntimeError("a real 'pymc' is already imported; the stub loader must run first")
    _install_stubs()
    sys.modules["pymc"].__b200_stub__ = True
    out = {}
    for name, rel in _FILES:
        spec = importlib.util.spec_from_file_location(name, os.path.join(REFERENCE_ROOT, rel))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
        parent, _, leaf = name.rpartition(".")
        setattr(sys.modules[parent], leaf, mod)
        out[name] = mod
    _loaded = out
    return out


# --------------------------------------------------------------------------------------------
# Minimal stand-ins for the model-side objects the reference step method touches.
# --------------------------------------------------------------------------------------------
class _ValueVar:
    def __init__(self, name, size):
        self.name = name
        self.dtype = "float64"
        self.size = size


class FakeModel:
    """Only what ``BaseHMC.__init__``/``astep`` read: value vars and an initial point."""

    def __init__(self, var_sizes: dict[str, int], start: dict[str, np.ndarray]):
        self.value_vars = [_ValueVar(k, s) for k, s in var_sizes.items()]
        self.continuous_value_vars = self.value_vars
        self.rvs_to_values = {}
        self._start = {k: np.asarray(v, dtype="float64") for k, v in start.items()}

    def initial_point(self, *a, **k):
        return dict(self._start)

    def point_logps(self):
        return {}


class LogpDlogp:
    """Satisfies seam B1 (SURVEY 8b): ``_pytensor_function(q) -> (logp, dlogp)`` on a raveled q."""

    def __init__(self, fn):
        self._pytensor_function = fn
        self._raveled_inputs = True
        self.dtype = "float64"
        self._extra_vars_shared = {}
        self.trust_input = True
        self.n_calls = 0

    def set_extra_values(self, point):
        pass


def make_nuts(logp_dlogp, var_sizes, start_point, *, potential=None, step_rng=0, **nuts_kwargs):
    """Build the reference ``NUTS`` step method around a NumPy ``q -> (logp, grad)`` callable."""
    mods = load()
    NUTS = mods["pymc.step_methods.hmc.nuts"].NUTS
    model = FakeModel(var_sizes, start_point)
    func = LogpDlogp(logp_dlogp)
    step = NUTS(
        vars=model.value_vars,
        model=model,
        potential=potential,
        logp_dlogp_func=func,
        initial_point=model.initial_point(),
        rng=step_rng,
        **nuts_kwargs,
    )
    return step, model


def make_hmc(logp_dlogp, var_sizes, start_point, *, potential=None, step_rng=0, **hmc_kwargs):
    """Build the reference ``HamiltonianMC`` step method (hmc/hmc.py) around a NumPy ``q -> (logp, grad)`` callable."""
    mods = load()
    HMC = mods["pymc.step_methods.hmc.hmc"].HamiltonianMC
    model = FakeModel(var_sizes, start_point)
    func = LogpDlogp(logp_dlogp)
    step = HMC(vars=model.value_vars, model=model, potential=potential, logp_dlogp_func=func,
               initial_point=model.initial_point(), rng=step_rng, **hmc_kwargs)
    return step, model


def quadpotential():
    return load()["pymc.step_methods.hmc.quadpotential"]
