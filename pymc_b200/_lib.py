"""ctypes binding of libb200nuts.so (C ABI declared in include/b200nuts.h).

The library is the product: there is NO CPU fallback.  ``load()`` raises if the shared object is
missing, and every compute entry point raises ``B200Error`` when no CUDA device is visible.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200nuts.so")

MEM_HOST, MEM_DEVICE = 0, 1
MASS_DIAG, MASS_DIAG_ADAPT, MASS_DENSE, MASS_DIAG_ADAPT_GRAD, MASS_DENSE_ADAPT = 0, 1, 2, 3, 4
SAMPLER_NUTS, SAMPLER_HMC = 0, 1
MOMENTUM_DEVICE_PHILOX, MOMENTUM_HOST_BUFFER = 0, 1
PRECISION_FP64, PRECISION_TC_FP16X2 = 0, 1


class B200Error(RuntimeError):
    pass


class ModelDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("n", C.c_int32),
        ("n_obs", C.c_int64),
        ("n_groups", C.c_int32),
        ("x", C.c_void_p),
        ("y", C.c_void_p),
        ("aux", C.c_void_p),
        ("idx", C.c_void_p),
        ("y_u8", C.c_void_p),
        ("scalar0", C.c_double),
        ("m1", C.c_void_p),
        ("m2", C.c_void_p),
        ("ir", C.c_void_p),
    ]


# ---- ModelSpec IR (include/b200nuts.h: b200_ir_*) ---------------------------------------------------------------------
MODEL_IR = 6


class IrParam(C.Structure):
    _fields_ = [("kind", C.c_int32), ("ref", C.c_int32), ("value", C.c_double)]


class IrVar(C.Structure):
    _fields_ = [("offset", C.c_int32), ("size", C.c_int32), ("transform", C.c_int32), ("reserved", C.c_int32),
                ("lo", C.c_double), ("hi", C.c_double)]


class IrPrior(C.Structure):
    _fields_ = [("dist", C.c_int32), ("var", C.c_int32), ("p", IrParam * 3)]


class IrFactor(C.Structure):
    _fields_ = [("offset", C.c_int32), ("size", C.c_int32), ("idx", C.c_void_p)]


class IrTerm(C.Structure):
    _fields_ = [("coef", C.c_void_p), ("n_factors", C.c_int32), ("reserved", C.c_int32), ("f", IrFactor * 3)]


class IrLik(C.Structure):
    _fields_ = [("dist", C.c_int32), ("n_terms", C.c_int32), ("N", C.c_int64), ("y", C.c_void_p), ("terms", C.c_void_p),
                ("sigma_kind", C.c_int32), ("reserved", C.c_int32), ("sigma", IrParam), ("sigma_obs", C.c_void_p),
                ("nu", C.c_double)]


class IrAr1(C.Structure):
    _fields_ = [("var", C.c_int32), ("reserved", C.c_int32), ("phi", IrParam), ("sigma", IrParam), ("init_sigma", C.c_double)]


class Ir(C.Structure):
    _fields_ = [("n_vars", C.c_int32), ("n_priors", C.c_int32), ("n_liks", C.c_int32), ("n_ar1", C.c_int32),
                ("vars", C.c_void_p), ("priors", C.c_void_p), ("liks", C.c_void_p), ("ar1", C.c_void_p)]


def build_ir(low):
    """pymc_b200.ir.LoweredIR -> (ctypes b200_ir, keep-alive list).  Pointers reference NumPy arrays held in `keep`."""
    keep = []

    def param(t):
        kind, value, ref = t
        return IrParam(int(kind), int(ref), float(value))

    def addr(a):
        if a is None:
            return None
        keep.append(a)
        return a.ctypes.data

    nv = len(low.vars)
    vars_ = (IrVar * nv)()
    for k in range(nv):
        o, sz, tr = (int(x) for x in low.vars[k])
        vars_[k] = IrVar(o, sz, tr, 0, float(low.var_bounds[k][0]), float(low.var_bounds[k][1]))
    pri = (IrPrior * max(1, len(low.priors)))()
    for k, (dist, var, pars) in enumerate(low.priors):
        pri[k].dist, pri[k].var = int(dist), int(var)
        for a in range(3):
            pri[k].p[a] = param(pars[a])
    liks = (IrLik * max(1, len(low.liks)))()
    for k, L in enumerate(low.liks):
        terms = (IrTerm * len(L["terms"]))()
        for t, T in enumerate(L["terms"]):
            terms[t].coef = addr(T["coef"])
            terms[t].n_factors = len(T["factors"])
            for f, (o, sz, idx) in enumerate(T["factors"]):
                terms[t].f[f] = IrFactor(int(o), int(sz), addr(idx))
        keep.append(terms)
        liks[k].dist, liks[k].n_terms, liks[k].N = int(L["dist"]), len(L["terms"]), int(L["N"])
        liks[k].y, liks[k].terms = addr(L["y"]), C.addressof(terms)
        liks[k].sigma_kind = int(L["sigma_kind"])
        liks[k].sigma = IrParam(1 if L["sigma_kind"] == 2 else 0, int(L["sigma_ref"]), float(L["sigma_value"]))
        liks[k].sigma_obs, liks[k].nu = addr(L["sigma_obs"]), float(L["nu"])
    ars = (IrAr1 * max(1, len(low.ar1)))()
    for k, (var, phi, sigma, init_sigma) in enumerate(low.ar1):
        ars[k].var, ars[k].phi, ars[k].sigma, ars[k].init_sigma = int(var), param(phi), param(sigma), float(init_sigma)
    ir = Ir(nv, len(low.priors), len(low.liks), len(low.ar1), C.addressof(vars_), C.addressof(pri), C.addressof(liks),
            C.addressof(ars))
    keep += [vars_, pri, liks, ars]
    return ir, keep


class Pcg64State(C.Structure):
    _fields_ = [("state_hi", C.c_uint64), ("state_lo", C.c_uint64), ("inc_hi", C.c_uint64), ("inc_lo", C.c_uint64)]


PCG64_DTYPE = np.dtype([("state_hi", "<u8"), ("state_lo", "<u8"), ("inc_hi", "<u8"), ("inc_lo", "<u8")])


STATE_FIELDS = [  # b200_chain_state: (name, dtype, per-chain vector?)
    ("q", np.float64, True), ("log_step", np.float64, False), ("log_bar", np.float64, False), ("hbar", np.float64, False),
    ("da_count", np.int32, False), ("n_samples", np.int32, False), ("window", np.int32, False), ("var", np.float64, True),
    ("fg_n", np.float64, False), ("fg_mean", np.float64, True), ("fg_m2", np.float64, True), ("bg_n", np.float64, False),
    ("bg_mean", np.float64, True), ("bg_m2", np.float64, True), ("n_grad", np.int64, False),
]


class ChainStateC(C.Structure):
    _fields_ = [(name, C.c_void_p) for name, _, _ in STATE_FIELDS]


class NutsCfg(C.Structure):
    _fields_ = [
        ("chains", C.c_int32),
        ("tune", C.c_int32),
        ("draws", C.c_int32),
        ("max_treedepth", C.c_int32),
        ("early_max_treedepth", C.c_int32),
        ("adapt_step_size", C.c_int32),
        ("mass_kind", C.c_int32),
        ("momentum_source", C.c_int32),
        ("store_warmup", C.c_int32),
        ("chain_offset", C.c_int32),
        ("step_scale", C.c_double),
        ("target_accept", C.c_double),
        ("gamma", C.c_double),
        ("k", C.c_double),
        ("t0", C.c_double),
        ("Emax", C.c_double),
        ("mass_initial_weight", C.c_double),
        ("adaptation_window", C.c_int32),
        ("discard_window", C.c_int32),
        ("philox_seed", C.c_uint64),
        ("sampler", C.c_int32),
        ("max_steps", C.c_int32),
        ("path_length", C.c_double),
        ("mass_alpha", C.c_double),
        ("stop_adaptation", C.c_int32),
        ("iter_begin", C.c_int32),
        ("iter_count", C.c_int32),
        ("resume", C.c_void_p),
        ("save", C.c_void_p),
        ("constrain_draws", C.c_int32),
        ("mass_update_window", C.c_int32),
        ("adaptation_window_multiplier", C.c_double),
    ]


STAT_FIELDS = [
    ("depth", np.int32),
    ("tree_size", np.int32),
    ("index_in_trajectory", np.int32),
    ("diverging", np.uint8),
    ("reached_max_treedepth", np.uint8),
    ("step_size", np.float64),
    ("step_size_bar", np.float64),
    ("mean_tree_accept", np.float64),
    ("energy", np.float64),
    ("energy_error", np.float64),
    ("max_energy_error", np.float64),
    ("model_logp", np.float64),
]


class Stats(C.Structure):
    _fields_ = [(name, C.c_void_p) for name, _ in STAT_FIELDS]


SUMMARY_FIELDS = [
    ("grad_evals", np.int64),
    ("bad_energy_at", np.int32),
    ("final_step_size", np.float64),
    ("final_var", np.float64),
    ("final_cov", np.float64),
]


class ChainSummary(C.Structure):
    _fields_ = [(name, C.c_void_p) for name, _ in SUMMARY_FIELDS]


# every symbol include/b200nuts.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("b200_version", C.c_int, []),
    ("b200_last_error", C.c_char_p, []),
    ("b200_struct_size", C.c_int, [C.c_int]),
    ("b200_device_count", C.c_int, []),
    ("b200_set_device", C.c_int, [C.c_int]),
    ("b200_model_create", C.c_int, [C.POINTER(ModelDesc), C.POINTER(C.c_void_p)]),
    ("b200_model_destroy", None, [C.c_void_p]),
    ("b200_model_n", C.c_int, [C.c_void_p]),
    ("b200_model_set_precision", C.c_int, [C.c_void_p, C.c_int32]),
    ("b200_model_set_transforms", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("b200_model_set_dense_mass", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("b200_logp_dlogp", C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    (
        "b200_leapfrog",
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32] + [C.c_void_p] * 7 + [C.c_int32, C.c_void_p],
    ),
    (
        "b200_nuts_run",
        C.c_int,
        [C.c_void_p, C.POINTER(NutsCfg)] + [C.c_void_p] * 7 + [C.POINTER(Stats), C.POINTER(ChainSummary), C.c_int32, C.c_void_p],
    ),
    ("b200_pointwise_loglik", C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p]),
    ("b200_last_kernel_ms", C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    ("b200_measure_fp64_tflops", C.c_int, [C.POINTER(C.c_double)]),
    ("b200_measure_dmma_tflops", C.c_int, [C.POINTER(C.c_double)]),
]

_lib = None


def load() -> C.CDLL:
    """dlopen the engine; raises if it has not been built (run ``./build.sh`` or ``__graft_entry__.build()``)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise B200Error(f"{LIB_PATH} is missing: build the CUDA engine first (./build.sh); there is no CPU fallback")
        lib = C.CDLL(LIB_PATH)
        for name, restype, argtypes in SYMBOLS:
            fn = getattr(lib, name)
            fn.restype = restype
            fn.argtypes = argtypes
        mirrors = [ModelDesc, NutsCfg, Stats, ChainSummary, Pcg64State, Ir, IrVar, IrPrior, IrTerm, IrLik, IrAr1, IrParam, IrFactor,
                   ChainStateC]
        for which, cls in enumerate(mirrors):
            if lib.b200_struct_size(which) != C.sizeof(cls):
                raise B200Error(f"ABI mismatch: {cls.__name__} is {C.sizeof(cls)} bytes here, {lib.b200_struct_size(which)} in "
                                f"{LIB_PATH} (rebuild with ./build.sh)")
        _lib = lib
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise B200Error(load().b200_last_error().decode())


def require_gpu() -> None:
    if load().b200_device_count() < 1:
        raise B200Error("no CUDA device visible: the B200 engine has no CPU fallback")


def ptr(a) -> int | None:
    """Raw address of a NumPy array or torch tensor (None passes NULL)."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a.data_ptr()  # torch.Tensor


def last_kernel_ms() -> tuple[float, int]:
    ms, n = C.c_double(), C.c_int32()
    load().b200_last_kernel_ms(C.byref(ms), C.byref(n))
    return ms.value, n.value
