"""Seam B3 (SURVEY 8b): ``B200NUTS`` driven exactly like ``_iter_sample`` drives a step method
(pymc/sampling/mcmc.py:1503-1578), against the VERBATIM reference ``NUTS`` on the same generator (its run recorded in
tests/golden/ref_step_seam.npz by ``python -m oracle.make_golden seams``).

CPU: the device engine is replaced by a stand-in with the ``CompiledModel.nuts_run`` interface that runs the oracle
(bit-identical to the reference, tests/test_oracle_vs_reference.py), which pins the protocol glue: stream derivation
(``rng`` / ``rng.spawn(1)[0]``), tune/draw schedule, point (un)raveling, stats keys.  GPU: the real engine."""
import numpy as np
import pytest

from b200_helpers import OracleEngine
from pymc_b200 import models
from pymc_b200.step import B200NUTS


def drive(step, start, rng, tune, draws):
    """The loop of _iter_sample."""
    step.setup_chain(rng, tune, draws)
    step.tune = bool(tune)
    step.reset_tuning()
    point, out, stats = start, [], []
    for i in range(tune + draws):
        if i == tune:
            step.stop_tuning()
        point, st = step.step(point)
        out.append(np.concatenate([np.ravel(point[k]) for k in start]))
        stats.append(st[0])
    return np.array(out), stats


def test_b200nuts_protocol_matches_reference_nuts_with_oracle_engine(golden):
    spec = models.eight_schools()
    q0 = spec.initial_point() + np.random.default_rng(3).uniform(-1, 1, spec.n)
    start = {v.name: q0[v.offset : v.offset + v.size].copy() for v in spec.vars}
    tune, draws, seed = 60, 25, 20240922

    # the reference NUTS with its default potential, DiagAdapt(zeros, ones, 10), driven by drive() from default_rng(seed)
    want = golden("ref_step_seam")
    hi, lo = (int(x) for x in want["rng_after"])
    rng_ref_after = (hi << 64) | lo

    mine = B200NUTS(OracleEngine(spec))
    rng = np.random.default_rng(seed)
    got_q, got_st = drive(mine, dict(start), rng, tune, draws)

    assert np.array_equal(got_q, want["q"])
    for k in ("depth", "tree_size", "index_in_trajectory", "diverging", "reached_max_treedepth", "divergences"):
        assert [s[k] for s in got_st] == want["stat_" + k].tolist(), k
    for k in ("step_size", "step_size_bar", "mean_tree_accept", "energy", "energy_error", "max_energy_error", "model_logp"):
        np.testing.assert_allclose([s[k] for s in got_st], want["stat_" + k], rtol=1e-12, atol=1e-12, err_msg=k)
    assert set(B200NUTS.stats_dtypes_shapes) == set(want["stats_dtypes_shapes_keys"].tolist())
    assert set(got_st[0]) == set(want["stats_keys"].tolist())
    # the caller's generator is left exactly where the reference leaves its own
    assert rng.bit_generator.state["state"]["state"] == rng_ref_after
    # shape of a point entry is preserved, other keys pass through
    p, _ = B200NUTS(OracleEngine(spec)), None
    p.setup_chain(np.random.default_rng(1), 0, 2)
    p.tune = False
    out, _ = p.step({**start, "extra": 7})
    assert out["extra"] == 7 and out["theta_t"].shape == (8,) and out["mu"].shape == (1,)


def test_b200nuts_requires_setup_chain_and_respects_schedule():
    spec = models.eight_schools()
    s = B200NUTS(OracleEngine(spec))
    start = {v.name: np.zeros(v.size) for v in spec.vars}
    with pytest.raises(RuntimeError, match="setup_chain"):
        s.step(start)
    s.setup_chain(np.random.default_rng(2), 3, 2)
    s.reset_tuning()
    pt = start
    for i in range(5):
        if i == 3:
            s.stop_tuning()
        pt, st = s.step(pt)
        assert s.tune == (i < 3)
    with pytest.raises(RuntimeError, match="more often"):
        s.step(pt)
    s2 = B200NUTS(OracleEngine(spec))
    s2.setup_chain(np.random.default_rng(2), 3, 2)
    s2.step(start)
    with pytest.raises(RuntimeError, match="stop_tuning"):
        s2.stop_tuning()  # iteration 1, but the device chain was tuned for 3
    assert B200NUTS.competence(type("V", (), {"dtype": "float64"})(), True) == 3
    assert B200NUTS.competence(type("V", (), {"dtype": "int64"})(), True) == 0


def _golden_prefix_through_step_seam(golden, make_engine):
    d = golden("eight_schools_adapt")
    spec = models.eight_schools()
    s = B200NUTS(make_engine(spec), potential_mean=d["q0"][0], potential_var=d["init_var"][0],
                 step_scale=float(d["step_scale"]))
    tune, T = int(d["tune"]), 12
    q0 = d["q0"][0]
    pt = {v.name: q0[v.offset : v.offset + v.size].copy() for v in spec.vars}
    s.setup_chain(np.random.default_rng(int(d["seeds"][0])), tune, int(d["draws"]))
    s.tune = True
    s.reset_tuning()
    for i in range(T):
        pt, st = s.step(pt)
        q = np.concatenate([np.ravel(pt[v.name]) for v in spec.vars])
        assert st[0]["tree_size"] == d["stat_tree_size"][0][i] and st[0]["depth"] == d["stat_depth"][0][i]
        assert np.max(np.abs(q - d["draws_q"][0][i])) <= 1e-7
        assert abs(st[0]["step_size"] - d["stat_step_size"][0][i]) <= 1e-9 * d["stat_step_size"][0][i]


def test_b200nuts_reproduces_golden_adaptive_prefix_oracle_engine(golden):
    """The golden chain was produced by the verbatim reference from default_rng(seed): the step-method seam must land on
    it when it derives its streams from the same generator (here with the oracle-backed engine)."""
    _golden_prefix_through_step_seam(golden, OracleEngine)


@pytest.mark.gpu
def test_b200nuts_on_device_reproduces_golden_adaptive_prefix(golden):
    """The real engine behind the step-method seam: first iterations of the reference's adaptive Eight Schools chain."""
    from pymc_b200 import engine

    _golden_prefix_through_step_seam(golden, engine.CompiledModel)


@pytest.mark.gpu
def test_b200nuts_sampling_state_and_changed_point_on_device(golden):
    """sampling_state carries the step-size and potential state (hmc/base_hmc.py:61-71); a driver that changes the point
    between calls gets a re-launch from ITS point (ADVICE r1), never stale draws."""
    import warnings

    from pymc_b200 import engine

    spec = models.eight_schools()
    s = B200NUTS(engine.CompiledModel(spec))
    s.setup_chain(np.random.default_rng(3), 30, 10)
    s.reset_tuning()
    pt = {v.name: np.zeros(v.size) for v in spec.vars}
    for i in range(5):
        pt, st = s.step(pt)
    state = s.sampling_state
    assert state["iter_count"] == 5 and state["step_adapt"]["count"] >= 30 and state["launched_through_iteration"] == 40
    assert state["potential"]["_var"].shape == (spec.n,) and np.all(state["potential"]["_var"] > 0)
    assert state["potential"]["_foreground_var"]["mean"].shape == (spec.n,)
    moved = {k: v + 0.25 for k, v in pt.items()}
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        pt2, st2 = s.step(moved)
    assert any("re-launching" in str(x.message) for x in w)
    assert s.iter_count == 6 and np.isfinite(st2[0]["energy"])
    for i in range(6, 40):
        if i == 30:
            s.stop_tuning()
        pt2, st2 = s.step(pt2)
    with pytest.raises(RuntimeError):
        s.step(pt2)
