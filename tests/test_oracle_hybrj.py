"""Pins the oracle's analytic-Jacobian path (modelOrder == 1: variational integration,
shooting::ShootingFunctionJacobian, hybrj) against the UNMODIFIED reference (oracle/_ref) and against
the known answers of SURVEY.md section 8c (DI solve: nfev 30 / njev 4, tf = 27.655974527562883)."""
import numpy as np
import pytest

import scenarios as S
from oracle import pyref
from backends import OracleBackend

needs_ref = pytest.mark.skipif(not pyref.available(), reason="reference build (oracle/_ref) not present")


def di_wp_spec():
    """tests/testDoubleIntegrator_WP.cpp:34-51: two segments, every time FREE but the first, interior
    velocity CONTINUOUS and position FIXED."""
    n = 6
    mode_t = [S.FIXED, S.FREE, S.FREE]
    mode_X = [[S.FIXED] * n, [S.FIXED] * 3 + [S.CONTINUOUS] * 3, [S.FIXED] * n]
    time = [0.0, 8.0, 16.0]
    Xb = np.zeros((3, n))
    Xb[1, :3] = [5.0, 10.0, 1.0]
    Xb[2, :3] = [10.0, 15.0, 0.0]
    x0 = np.zeros(2 * 12 + 2)
    x0[6:12] = 0.01
    x0[12:15] = Xb[1, :3]
    x0[15:18] = [0.5, 0.6, 0.0]
    x0[18:24] = 0.01
    x0[24:] = [8.0, 16.0]
    return S.make_spec(S.DI, 2, mode_t, mode_X, time, Xb, x0, 1e-8, name="di_wp")


def ref_shooting(spec):
    from backends import RefBackend
    be = RefBackend()
    m = pyref.RefModel(S.DI, model_order=1, step_nbr=0)
    for name, v in zip(S.PARAMS[S.DI], spec["mparams"]):
        m.set(name, v)
    s = pyref.RefShooting(m, spec["M"], 1)
    s.set_precision(spec["xtol"])
    s.set_mode(spec["mode_t"], spec["mode_X"])
    n, M = 6, spec["M"]
    x0 = np.asarray(spec["x0"], dtype=np.float64)
    vt = np.array(spec["time"], dtype=np.float64)
    k = 2 * n * M
    for j in range(M + 1):
        if spec["mode_t"][j] == S.FREE:
            vt[j] = x0[k]
            k += 1
    vX = np.zeros((M + 1, 2 * n))
    for j in range(M):
        vX[j] = x0[2 * n * j:2 * n * (j + 1)]
    vX[M, :n] = spec["Xb"][M]
    s.init_v(vt, vX)
    Xd = np.zeros((M + 1, 2 * n))
    Xd[:, :n] = np.asarray(spec["Xb"], dtype=np.float64)
    s.desired_v(np.array(spec["time"], dtype=np.float64), Xd)
    return m, s


@needs_ref
def test_variational_trajectory_bit_exact(oracle_lib):
    m = pyref.RefModel(S.DI, model_order=1, step_nbr=0)
    p = OracleBackend().problem(S.di_problem())
    rng = np.random.default_rng(3)
    for _ in range(4):
        X = np.zeros(156)
        X[:12] = rng.uniform(-1, 1, 12)
        X[12:] = np.eye(12).reshape(-1) + 0.1 * rng.uniform(-1, 1, 144)
        tf = float(rng.uniform(1, 20))
        assert np.array_equal(p.traj_var(0.0, X, tf), m.traj(0.0, X, tf, is_jac=1))


@needs_ref
@pytest.mark.parametrize("make", [S.di_problem, di_wp_spec])
def test_analytic_jacobian_bit_exact(oracle_lib, make):
    spec = make()
    p = OracleBackend().problem(spec)
    _, s = ref_shooting(spec)
    rng = np.random.default_rng(11)
    x = np.array(spec["x0"], dtype=np.float64)
    for k in range(3):
        xx = x * (1 + 0.05 * k * rng.uniform(-1, 1, x.size))
        want = s.jacobian(xx)
        got = p.jacobian(xx)
        assert np.array_equal(got, want), np.argwhere(got != want)[:5]


def test_analytic_jacobian_is_the_derivative_of_the_residual(oracle_lib):
    """Central differences of the residual at the points of test_analytic_jacobian_bit_exact.  Only for the one-segment
    problem: with interpolated interior times the reference's Jacobian is its own."""
    spec = S.di_problem()
    p = OracleBackend().problem(spec)
    rng = np.random.default_rng(11)
    x = np.array(spec["x0"], dtype=np.float64)
    for k in range(3):
        xx = x * (1 + 0.05 * k * rng.uniform(-1, 1, x.size))
        got = p.jacobian(xx)
        fd = np.zeros_like(got)
        for j in range(x.size):
            h = 1e-6 * max(1.0, abs(xx[j]))
            e = np.zeros(x.size); e[j] = h
            fd[:, j] = (p.residual(xx + e) - p.residual(xx - e)) / (2 * h)
        assert np.max(np.abs(fd - got)) <= 1e-6 * max(1.0, np.max(np.abs(got)))


def test_hybrj_solve_matches_reference_and_survey(oracle_lib):
    """The known answers of SURVEY.md section 8c, and the reference itself where its build is present."""
    spec = S.di_problem()
    p = OracleBackend().problem(spec)
    o = p.solve_hybrj(spec["x0"], xtol=spec["xtol"])
    assert (o["info"], o["nfev"], o["njev"]) == (1, 30, 4)                       # SURVEY.md section 8c, DI solve 1
    assert o["x"][12] == pytest.approx(27.655974527562883, rel=1e-14)
    if not pyref.available():
        return
    _, s = ref_shooting(spec)
    assert s.solve(0.0) == 1
    assert s.call_number() == (30, 4)
    assert np.array_equal(s.params(), o["x"])                                    # bit-exact against the reference


@needs_ref
def test_hybrj_two_segments_matches_reference(oracle_lib):
    spec = di_wp_spec()
    p = OracleBackend().problem(spec)
    o = p.solve_hybrj(spec["x0"], xtol=spec["xtol"])
    _, s = ref_shooting(spec)
    info = s.solve(0.0)
    assert info == o["info"]
    assert s.call_number() == (o["nfev"], o["njev"])
    if info == 1:
        assert np.array_equal(s.params(), o["x"])


def _golden_hybrj():
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_hybrj.json")) as f:
        return json.load(f)


def _unhex(v):
    return np.array([float.fromhex(s) for s in v])


def test_oracle_matches_golden_hybrj(oracle_lib):
    """The committed vectors (tests/golden/golden_hybrj.json, recorded from the unmodified reference by
    tests/golden/make_golden_hybrj.py) pin the oracle where the reference build is not available."""
    g = _golden_hybrj()
    p = OracleBackend().problem(S.di_problem())
    for e in g["traj_var"]:
        assert np.array_equal(p.traj_var(0.0, _unhex(e["X0"]), float.fromhex(e["tf"])), _unhex(e["Xf"]))
    for e, make in zip(g["jacobian"], (S.di_problem, di_wp_spec)):
        spec = make()
        x = _unhex(e["x"])
        J = OracleBackend().problem(spec).jacobian(x)
        assert np.array_equal(J.reshape(-1), _unhex(e["J"]))
    for e, make in zip(g["solve"], (S.di_problem, di_wp_spec)):
        spec = make()
        o = OracleBackend().problem(spec).solve_hybrj(spec["x0"], xtol=spec["xtol"])
        assert (o["info"], o["nfev"], o["njev"]) == (e["info"], e["nfev"], e["njev"])
        if e["info"] == 1:          # (SOCP keeps tab_param unchanged when the solve fails, shooting.cpp:588)
            assert np.array_equal(o["x"], _unhex(e["x"]))
    assert (g["solve"][0]["nfev"], g["solve"][0]["njev"]) == (30, 4)
