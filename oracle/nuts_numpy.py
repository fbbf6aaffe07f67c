"""TEST INFRASTRUCTURE ONLY -- CPU restatement (NumPy/SciPy) of the reference NUTS hot path.

This is the oracle the CUDA path is checked against, and the "port" timed as ``cpu_baseline``.
It restates, function by function, what the reference does for one NUTS transition:

  * ``Oracle.draw``          <- BaseHMC.astep            pymc/step_methods/hmc/base_hmc.py:196-288
  * ``Oracle._transition``   <- NUTS._hamiltonian_step   pymc/step_methods/hmc/nuts.py:204-225
  * ``_Trajectory.double``   <- _Tree.extend             nuts.py:334-392
  * ``_Trajectory._grow``    <- _Tree._build_subtree     nuts.py:442-476
  * ``_Trajectory._leaf``    <- _Tree._single_step       nuts.py:394-440
  * ``Oracle._leapfrog``     <- CpuLeapfrogIntegrator._step   hmc/integration.py:109-145
  * ``Oracle._start_state``  <- CpuLeapfrogIntegrator.compute_state   integration.py:68-75
  * ``DualAveraging``        <- DualAverageAdaptation    pymc/step_methods/step_sizes.py:41-84
  * ``DiagMass``             <- QuadPotentialDiag / QuadPotentialDiagAdapt + _WeightedVariance
                                hmc/quadpotential.py:582-630, :211-355, :405-448
  * ``DenseMass``            <- QuadPotentialFull        quadpotential.py:680-725
  * ``DenseAdaptMass``       <- QuadPotentialFullAdapt + _WeightedCovariance   quadpotential.py:748-907
  * ``DiagMassExp``          <- QuadPotentialDiagAdaptExp + _ExpWeightedVariance   quadpotential.py:458-579
  * ``Oracle.hmc_draw``      <- HamiltonianMC._hamiltonian_step + unif step jitter   hmc/hmc.py:35-36, :143-200

It performs the same floating-point operations with the same NumPy/BLAS calls in the same order
and consumes the two per-chain PCG64 streams in the same order (SURVEY.md 8a row a15), so that on
the same NumPy/SciPy it is *bit-identical* to the reference files loaded verbatim
(``oracle/ref_loader.py``); ``tests/test_oracle_vs_reference.py`` asserts that against reference
chains recorded in ``tests/golden/ref_port_chains.npz``, and the other ``tests/golden/*.npz`` (all
made by ``oracle/make_golden.py`` from the verbatim reference) pin it further.  PARITY STATUS: pinned.

Only tests/, bench.py's cpu_baseline / --impl reference legs and __graft_entry__.smoke() may
import this module; nothing under pymc_b200/ does.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import scipy.linalg as sl

_axpy = sl.blas.daxpy  # the reference fetches BLAS axpy for float64 (integration.py:110)


# ------------------------------------------------------------------------------------------------
# mass matrices
# ------------------------------------------------------------------------------------------------
class _Welford:
    """_WeightedVariance (quadpotential.py:405-448): running mean / raw second moment, divisor n."""

    def __init__(self, n, mean=None, var=None, weight=0.0):
        self.count = float(weight)
        self.mean = np.zeros(n) if mean is None else np.array(mean, dtype="d", copy=True)
        self.m2 = np.zeros(n) if var is None else np.array(var, dtype="d", copy=True)
        self.m2[:] *= self.count

    def add(self, x):
        self.count += 1
        before = x - self.mean
        self.mean[:] += before / self.count
        after = x - self.mean
        self.m2[:] += before * after


class DiagMass:
    """Diagonal inverse-mass ("var").  adapt=False -> QuadPotentialDiag; adapt=True -> DiagAdapt."""

    def __init__(self, var, *, adapt=False, initial_mean=None, initial_weight=0.0,
                 adaptation_window=101, discard_window=50, multiplier=1.0):
        self.n = len(var)
        self.adapt = adapt
        self._init = (np.array(var, dtype="d"), None if initial_mean is None else np.array(initial_mean, dtype="d"),
                      float(initial_weight), int(adaptation_window), int(discard_window), float(multiplier))
        self.rng = None
        self.reset()

    def reset(self):
        var, mean, weight, window, discard, mult = self._init
        self.var = var.copy()
        self.std = np.sqrt(var)
        self.inv_std = 1.0 / self.std
        self.window, self.discard, self.mult = window, discard, mult
        self.k = 0
        if self.adapt:
            self.fg = _Welford(self.n, np.zeros(self.n) if mean is None else mean, var, weight)
            self.bg = _Welford(self.n)

    def velocity(self, p, out=None):
        # QuadPotentialDiag multiplies (x, v), DiagAdapt (var, x): commutative, same bits
        return np.multiply(self.var, p, out=out)

    def kinetic(self, p, v):
        return 0.5 * np.dot(p, v)

    def momentum(self, z):
        return self.inv_std * z if self.adapt else z * self.inv_std

    def update(self, q, grad, tune):
        """QuadPotentialDiagAdapt.update (quadpotential.py:335-355)."""
        if not (self.adapt and tune):
            return
        if self.k > self.discard:
            self.fg.add(q)
            self.bg.add(q)
        if self.k > self.window:
            self.var = np.clip(self.fg.m2 / self.fg.count, 1e-12, 1e12)
            self.std = np.sqrt(self.var)
            self.inv_std = 1.0 / self.std
        if self.k > 0 and self.k % self.window == 0:
            self.fg = self.bg
            self.bg = _Welford(self.n)
            self.window = int(self.window * self.mult)
        self.k += 1


class DiagMassExp(DiagMass):
    """QuadPotentialDiagAdaptExp (quadpotential.py:493-579) with use_grads=True: exponentially weighted variances of the
    draws and of their gradients (_ExpWeightedVariance :458-483); var = sqrt(var_draws / var_grads) after 2 * discard
    draws; what init="jitter+adapt_diag_grad" builds (pymc/sampling/mcmc.py:1895-1912: alpha=0.02, stop = tune - 50)."""

    def __init__(self, n, *, alpha=0.02, stop_adaptation=None, discard_window=50, initial_mean=None):
        self.alpha, self.stop = float(alpha), (np.inf if stop_adaptation is None else stop_adaptation)
        super().__init__(np.ones(n), adapt=True, initial_mean=initial_mean, initial_weight=0.0, discard_window=discard_window)

    def reset(self):
        super().reset()
        self.est = self.est_g = None

    def _add(self, e, value):
        mean, var = e
        delta = value - mean
        mean[...] += self.alpha * delta
        var[...] = (1 - self.alpha) * (var + self.alpha * delta**2)

    def update(self, q, grad, tune):
        if tune and self.k < self.stop:
            if self.k > self.discard:
                self._add(self.est, q)
                self._add(self.est_g, grad)
            elif self.k == self.discard:
                self.est = [q.copy(), np.zeros_like(q)]
                self.est_g = [grad.copy(), np.zeros_like(grad)]
            if self.k > 2 * self.discard:
                self.var = np.sqrt(self.est[1] / self.est_g[1])
                self.std = np.sqrt(self.var)
                self.inv_std = 1.0 / self.std
            self.k += 1


class DenseMass:
    """QuadPotentialFull (quadpotential.py:680-725): v = cov @ p ; p0 = solve(chol^T, z)."""

    adapt = False

    def __init__(self, cov):
        self.cov = np.array(cov, dtype="d", copy=True)
        self.chol = sl.cholesky(self.cov, lower=True)
        self.n = len(self.cov)
        self.rng = None

    def reset(self):
        pass

    def velocity(self, p, out=None):
        return np.dot(self.cov, p, out=out)

    def kinetic(self, p, v):
        return 0.5 * np.dot(p, v)

    def momentum(self, z):
        return sl.solve_triangular(self.chol.T, z, overwrite_b=False)

    def update(self, q, grad, tune):
        pass


class DenseInvMass(DenseMass):
    """QuadPotentialFullInv (quadpotential.py:633-677): A = inverse covariance; v = cho_solve(chol(A), p); p0 = chol(A) z."""

    def __init__(self, A):
        self.L = sl.cholesky(np.array(A, dtype="d"), lower=True)
        self.n = len(self.L)
        self.rng = None

    def velocity(self, p, out=None):
        vel = sl.cho_solve((self.L, True), p)
        if out is None:
            return vel
        out[:] = vel
        return out

    def momentum(self, z):
        return np.dot(self.L, z)


class _WelfordCov:
    """_WeightedCovariance (quadpotential.py:855-907): running mean / raw scatter matrix, divisor n - 1."""

    def __init__(self, n, mean=None, cov=None, weight=0.0):
        self.count = float(weight)
        self.mean = np.zeros(n) if mean is None else np.array(mean, dtype="d", copy=True)
        self.raw = np.eye(n) if cov is None else np.array(cov, dtype="d", copy=True)
        self.raw[:] *= self.count

    def add(self, x):
        x = np.asarray(x)
        self.count += 1
        before = x - self.mean
        self.mean[:] += before / self.count
        after = x - self.mean
        self.raw[:] += after[:, None] * before[None, :]


class DenseAdaptMass(DenseMass):
    """QuadPotentialFullAdapt (quadpotential.py:748-845): foreground / background sample covariances; the covariance and its
    Cholesky factor are refreshed every `update_window` tuning draws, the windows grow by `multiplier`."""

    adapt = True

    def __init__(self, n, initial_mean, initial_cov=None, initial_weight=0, adaptation_window=101, multiplier=2,
                 update_window=1):
        if initial_cov is None:
            initial_cov, initial_weight = np.eye(n), 1
        self.n = n
        self._init = (np.array(initial_mean, dtype="d"), np.array(initial_cov, dtype="d"), initial_weight,
                      int(adaptation_window), float(multiplier), int(update_window))
        self.rng = None
        self.reset()

    def reset(self):
        mean, cov, weight, window, mult, upd = self._init
        self.prev = 0
        self.cov = cov.copy()
        self.chol = sl.cholesky(self.cov, lower=True)
        self.chol_error = None
        self.fg = _WelfordCov(self.n, mean, cov, weight)
        self.bg = _WelfordCov(self.n)
        self.k = 0
        self.window, self.mult, self.upd = window, mult, upd

    def update(self, q, grad, tune):
        if not tune:
            return
        delta = self.k - self.prev
        self.fg.add(q)
        self.bg.add(q)
        if (delta + 1) % self.upd == 0:
            np.divide(self.fg.raw, self.fg.count - 1, out=self.cov)
            try:
                self.chol = sl.cholesky(self.cov, lower=True)
            except (sl.LinAlgError, ValueError) as e:  # kept and raised by raise_ok in the reference
                self.chol_error = e
        if delta >= self.window:
            self.fg = self.bg
            self.bg = _WelfordCov(self.n)
            self.prev = self.k
            self.window = int(self.window * self.mult)
        self.k += 1


# ------------------------------------------------------------------------------------------------
# step-size adaptation
# ------------------------------------------------------------------------------------------------
class DualAveraging:
    """Nesterov dual averaging exactly as step_sizes.py:50-84."""

    def __init__(self, eps0, target=0.8, gamma=0.05, k=0.75, t0=10):
        self.eps0, self.target, self.gamma, self.kappa, self.t0 = eps0, target, gamma, k, t0
        self.reset()

    def reset(self):
        self.log_step = np.log(self.eps0)
        self.log_bar = self.log_step
        self.hbar = 0.0
        self.count = 1
        self.mu = np.log(10 * self.eps0)

    def current(self, tuning):
        return np.exp(self.log_step) if tuning else np.exp(self.log_bar)

    def update(self, accept, tuning):
        if not tuning:
            return
        c = self.count
        w = 1.0 / (c + self.t0)
        self.hbar = (1 - w) * self.hbar + w * (self.target - accept)
        self.log_step = self.mu - self.hbar * np.sqrt(c) / self.gamma
        m = c ** -self.kappa
        self.log_bar = m * self.log_step + (1 - m) * self.log_bar
        self.count += 1


# ------------------------------------------------------------------------------------------------
# trajectory
# ------------------------------------------------------------------------------------------------
@dataclass
class Phase:
    """integration.State (integration.py:27-34)."""

    q: np.ndarray
    p: np.ndarray
    v: np.ndarray
    grad: np.ndarray
    energy: float
    logp: float
    idx: int


@dataclass
class Span:
    """nuts.Subtree (nuts.py:264-267); ``pick`` is the Proposal (a Phase; only q/grad/energy/logp/idx used)."""

    left: Phase | None
    right: Phase | None
    p_sum: np.ndarray | None
    pick: Phase | None
    log_w: float


def _uturn(s, va, vb):
    return (s.dot(va) <= 0) or (s.dot(vb) <= 0)


class _Trajectory:
    def __init__(self, oracle, start: Phase, eps: float, rng):
        self.o, self.eps, self.rng = oracle, eps, rng
        self.e0 = start.energy
        self.left = self.right = start
        self.pick = start
        self.depth = 0
        self.log_w = 0.0
        self.log_accept = -np.inf
        self.n_leaves = 0
        self.p_sum = start.p.copy()
        self.max_de = 0.0

    # nuts.py:394-440
    def _leaf(self, frm: Phase, eps):
        new = self.o._leapfrog(eps, frm)
        self.n_leaves += 1
        if new is None:  # IntegrationError branch (only reachable with scipy.linalg potentials)
            return Span(None, None, None, None, -np.inf), True, False
        de = new.energy - self.e0
        if np.isnan(de):
            de = np.inf
        self.log_accept = np.logaddexp(self.log_accept, (-de if de > 0 else 0))
        if np.abs(de) > np.abs(self.max_de):
            self.max_de = de
        if de < self.o.Emax:
            return Span(new, new, new.p, new, -de), False, False
        return Span(None, None, None, None, -np.inf), True, False

    # nuts.py:442-476
    def _grow(self, frm: Phase, height: int, eps):
        if height == 0:
            return self._leaf(frm, eps)
        a, div, turn = self._grow(frm, height - 1, eps)
        if div or turn:
            return a, div, turn
        b, div, turn = self._grow(a.right, height - 1, eps)
        if not (div or turn):
            ps = a.p_sum + b.p_sum
            turn = _uturn(ps, a.left.v, b.right.v)
            if (not turn) and (height - 1 > 0):
                s1 = a.p_sum + b.left.p
                turn = _uturn(s1, a.left.v, b.left.v)
                if not turn:
                    s2 = a.right.p + b.p_sum
                    turn = _uturn(s2, a.right.v, b.right.v)
            log_w = np.logaddexp(a.log_w, b.log_w)
            pick = b.pick if np.log(self.rng.random()) < (b.log_w - log_w) else a.pick
        else:
            ps, log_w, pick = a.p_sum, a.log_w, a.pick
        return Span(a.left, b.right, ps, pick, log_w), div, turn

    # nuts.py:334-392
    def double(self, direction):
        if direction > 0:
            sub, div, turn = self._grow(self.right, self.depth, np.asarray(self.eps, dtype="float64"))
            lo_begin, lo_end = self.left, self.right
            hi_begin, hi_end = sub.left, sub.right
            lo_sum, hi_sum = self.p_sum.copy(), sub.p_sum
            self.right = sub.right
        else:
            sub, div, turn = self._grow(self.left, self.depth, np.asarray(-self.eps, dtype="float64"))
            lo_begin, lo_end = sub.right, sub.left
            hi_begin, hi_end = self.left, self.right
            lo_sum, hi_sum = sub.p_sum, self.p_sum.copy()
            self.left = sub.right
        self.depth += 1
        if div or turn:
            return div, turn
        if np.log(self.rng.random()) < (sub.log_w - self.log_w):
            self.pick = sub.pick
        self.log_w = np.logaddexp(sub.log_w, self.log_w)
        self.p_sum[:] += sub.p_sum
        turn = _uturn(self.p_sum, self.left.v, self.right.v)
        if not turn:
            s1 = lo_sum + hi_begin.p
            turn = _uturn(s1, lo_begin.v, hi_begin.v)
        if not turn:
            s2 = lo_end.p + hi_sum
            turn = _uturn(s2, lo_end.v, hi_end.v)
        return div, turn


class BadInitialEnergy(RuntimeError):
    """SamplingError("Bad initial energy") of base_hmc.py:205-224."""


class Oracle:
    """One chain of the reference NUTS sampler.

    ``logp_dlogp``: q -> (logp, grad).  ``mass``: DiagMass | DenseMass.  Defaults are the
    reference's (base_hmc.py:82-98, nuts.py:132)."""

    def __init__(self, logp_dlogp, mass, *, step_scale=0.25, adapt_step_size=True, target_accept=0.8,
                 gamma=0.05, k=0.75, t0=10, Emax=1000.0, max_treedepth=10, early_max_treedepth=8, sampler="nuts",
                 path_length=2.0, max_steps=1024):
        self.sampler, self.path_length, self.max_steps = sampler, path_length, max_steps
        self.f = logp_dlogp
        self.mass = mass
        self.n = mass.n
        self.Emax = Emax
        self.max_treedepth, self.early_max_treedepth = max_treedepth, early_max_treedepth
        self.adapt_step_size = adapt_step_size
        self.eps0 = step_scale / (self.n ** 0.25)  # base_hmc.py:161
        self.da = DualAveraging(self.eps0, target_accept, gamma, k, t0)
        self.tune = True
        self.iter_count = 0
        self.divergences = 0
        self.n_grad = 0
        self.rng = None

    def setup_chain(self, rng: np.random.Generator):
        """BlockedStep.setup_chain + BaseHMC.setup_chain (compound.py:233-250, base_hmc.py:300-302)."""
        self.rng = rng
        self.mass.rng = rng.spawn(1)[0]

    # integration.py:68-75
    def _start_state(self, q, p):
        logp, grad = self.f(q)
        self.n_grad += 1
        v = self.mass.velocity(p)
        energy = self.mass.kinetic(p, v) - logp
        return Phase(q, p, v, grad, energy, logp, 0)

    # integration.py:109-145
    def _leapfrog(self, eps, s: Phase):
        q = s.q.copy()
        p = s.p.copy()
        v = np.empty_like(q)
        dt = 0.5 * eps
        _axpy(s.grad, p, a=dt)
        self.mass.velocity(p, out=v)
        _axpy(v, q, a=eps)
        logp, grad = self.f(q)
        self.n_grad += 1
        _axpy(grad, p, a=dt)
        self.mass.velocity(p, out=v)
        energy = self.mass.kinetic(p, v) - logp
        return Phase(q, p, v, grad, energy, logp, s.idx + int(np.sign(eps)))

    # nuts.py:204-225
    def _transition(self, start, eps):
        limit = self.early_max_treedepth if (self.tune and self.iter_count < 200) else self.max_treedepth
        tr = _Trajectory(self, start, eps, self.rng)
        hit_max = False
        div = turn = False
        for _ in range(limit):
            direction = (self.rng.random() < 0.5) * 2 - 1
            div, turn = tr.double(direction)
            if div or turn:
                break
        else:
            hit_max = not self.tune
        return tr, div, hit_max

    # hmc.py:143-200 (HamiltonianMC._hamiltonian_step); the step size is jittered by unif() (hmc.py:35-36) in astep
    def _hmc_transition(self, start, eps):
        n_steps = max(1, int(self.path_length / eps))
        n_steps = min(self.max_steps, n_steps)
        state = start
        for _ in range(n_steps):
            state = self._leapfrog(eps, state)
        div = False
        if not np.isfinite(state.energy):
            div = True
        de = state.energy - start.energy
        if np.isnan(de):
            de = np.inf
        if np.abs(de) > self.Emax:
            div = True
        accept = min(1, np.exp(-de))
        if div or self.rng.random() >= accept:
            end, accepted = start, False
        else:
            end, accepted = state, True
        return end, state, n_steps, accept, de, div, accepted

    def hmc_draw(self, q0, z=None):
        """One HamiltonianMC transition (BaseHMC.astep with step_rand = unif, hmc.py:141)."""
        q0 = np.asarray(q0, dtype="float64")
        if z is None:
            z = self.mass.rng.normal(size=self.n)
        p0 = self.mass.momentum(z)
        start = self._start_state(q0, p0)
        if not np.isfinite(start.energy):
            raise BadInitialEnergy(f"Bad initial energy at iteration {self.iter_count}")
        adapting = self.tune and self.adapt_step_size
        eps = self.da.current(adapting)
        eps_j = self.rng.uniform(0.85, 1.15) * eps
        end, last, n_steps, accept, de, div, accepted = self._hmc_transition(start, eps_j)
        self.da.update(accept, adapting)
        self.mass.update(end.q, end.grad, self.tune)
        if not self.tune:
            self.divergences += bool(div)
        self.iter_count += 1
        stats = {
            "depth": 0, "step_size": float(np.exp(self.da.log_step)), "step_size_bar": float(np.exp(self.da.log_bar)),
            "mean_tree_accept": float(accept), "tree_size": n_steps, "diverging": bool(div), "divergences": self.divergences,
            "energy_error": de, "energy": last.energy, "max_energy_error": de, "model_logp": last.logp,
            "index_in_trajectory": n_steps if accepted else 0, "reached_max_treedepth": False, "tune": self.tune,
        }
        return end.q, stats

    # base_hmc.py:196-288
    def draw(self, q0, z=None):
        if self.sampler == "hmc":
            return self.hmc_draw(q0, z)
        """One transition from q0.  ``z``: optional pre-drawn N(0,1)^n momentum noise (otherwise drawn
        from the potential stream exactly like ``potential.random()``)."""
        q0 = np.asarray(q0, dtype="float64")
        if z is None:
            z = self.mass.rng.normal(size=self.n)
        p0 = self.mass.momentum(z)
        start = self._start_state(q0, p0)
        if not np.isfinite(start.energy):
            raise BadInitialEnergy(f"Bad initial energy at iteration {self.iter_count}")
        adapting = self.tune and self.adapt_step_size
        eps = self.da.current(adapting)
        tr, div, hit_max = self._transition(start, eps)
        accept = np.exp(tr.log_accept) / tr.n_leaves
        self.da.update(accept, adapting)
        self.mass.update(tr.pick.q, tr.pick.grad, self.tune)
        if not self.tune:
            self.divergences += bool(div)
        self.iter_count += 1
        stats = {
            "depth": tr.depth,
            "step_size": float(np.exp(self.da.log_step)),
            "step_size_bar": float(np.exp(self.da.log_bar)),
            "mean_tree_accept": float(accept),
            "tree_size": tr.n_leaves,
            "diverging": bool(div),
            "divergences": self.divergences,
            "energy_error": tr.pick.energy - start.energy,
            "energy": tr.pick.energy,
            "max_energy_error": tr.max_de,
            "model_logp": tr.pick.logp,
            "index_in_trajectory": tr.pick.idx,
            "reached_max_treedepth": hit_max,
            "tune": self.tune,
        }
        return tr.pick.q, stats

    def stop_tuning(self):
        self.tune = False

    def run(self, q0, tune, draws, z=None):
        """The chain loop of _iter_sample (sampling/mcmc.py:1549-1583): tune+draws transitions, stop_tuning at i==tune."""
        T = tune + draws
        qs = np.empty((T, self.n))
        stats = []
        q = np.asarray(q0, dtype="float64")
        for i in range(T):
            if i == tune:
                self.stop_tuning()
            q, st = self.draw(q, None if z is None else z[i])
            qs[i] = q
            stats.append(st)
        keys = stats[0].keys()
        return qs, {k: np.array([s[k] for s in stats]) for k in keys}
