"""GPU parity of the trajectory dump (socp_trace_batch) = the observer form of odeTools::integrate
(odeTools.cpp:103-123) with the row layout of model::Trace (model.hpp:446-462):
t, X[0..N), control, H [, model extra] -- one row at t0 and one after every RK4 step."""
import numpy as np
import pytest

import scenarios as S

pytestmark = pytest.mark.gpu

NCTRL = {S.GODDARD: 3, S.DI: 3, S.COVID19: 1, S.VTOL: 3, S.INTERCEPTOR: 2}
CASES = {
    S.GODDARD: (S.GODDARD_XI, 0.0, 0.1, 10),
    S.DI: (np.r_[np.zeros(6), 0.01 * np.ones(6)], 0.0, 8.0, 30),
    S.COVID19: (S.COVID_XI, 0.0, 1.5, 50),
    S.VTOL: (np.array([20, 8, 5, 0.3, 0.2, 0.1, -0.03, 0.013, -0.003, -0.29, 0.1, -0.03]), 0.0, 5.0, 20),
}


@pytest.fixture(scope="module")
def eng():
    import socp_b200 as sb
    e = sb.Engine(0)
    o = S.VTOL_OBSTACLES
    e.set_obstacles(o["type"], o["pos"], o["rad"])
    return e


@pytest.mark.parametrize("model", sorted(CASES))
def test_trace_rows_match_oracle(eng, oracle_lib, model):
    from backends import OracleBackend
    import oracle.pyoracle as O
    from backends import oracle_obstacles
    ora = OracleBackend()
    X0, t0, tf, steps = CASES[model]
    mp = np.array(S.DEFAULTS[model], dtype=np.float64)
    if model == S.GODDARD:
        mp[6] = 1.0
    N, nc = 2 * S.DIM[model], NCTRL[model]
    rows, nrows, Xf = eng.trace_batch(model, mp, t0, np.tile(X0, (3, 1)), tf, steps)
    assert rows.shape[2] == N + nc + 3
    assert list(nrows) == [steps + 1] * 3
    assert np.array_equal(rows[0], rows[1]) and np.array_equal(rows[0], rows[2])
    r = rows[0, :steps + 1]
    # first row = the initial point, last row = the end point of socp_traj_batch (same arithmetic)
    assert r[0, 0] == t0 and np.array_equal(r[0, 1:1 + N], X0)
    end = eng.traj_batch(model, mp, t0, X0[None, :], tf, steps)[0]
    assert np.array_equal(Xf[0], r[-1, 1:1 + N])
    # (the trace is compute_traj with an observer: the same step loop as traj_kernel)
    assert np.array_equal(Xf[0], end)
    # times: repeated t += dt (odeTools.cpp:111-121)
    t, dt = t0, (tf - t0) / steps
    for k in range(steps + 1):
        assert r[k, 0] == t
        t += dt
    # every step against the oracle's RK4 (one step from the previous row), controls and H at the row
    p = O.OracleProblem(model, 1, step_nbr=1, obstacles=oracle_obstacles() if model == S.VTOL else None)
    for k, v in enumerate(mp):
        p.set_param(k, v)
    for k in range(steps):
        want = ora.traj(model, mp, r[k, 0], r[k, 1:1 + N], r[k, 0] + dt, 1)
        scale = np.max(np.abs(want))
        assert np.max(np.abs(r[k + 1, 1:1 + N] - want)) <= 1e-12 * scale, (model, k)     # the path's RK4 tolerance
    for k in range(steps + 1):
        u = np.asarray(p.control(r[k, 0], r[k, 1:1 + N]))[:nc]
        H = p.hamiltonian(r[k, 0], r[k, 1:1 + N])
        assert np.allclose(r[k, 1 + N:1 + N + nc], u, rtol=1e-11, atol=1e-13), (model, k)
        assert abs(r[k, 1 + N + nc] - H) <= 1e-11 * max(1.0, abs(H), np.max(np.abs(r[k, 1:1 + N]))), (model, k)
    if model == S.GODDARD:      # goddard::Trace appends the switching function (goddard.cpp:337-339)
        X = r[:, 1:1 + N]
        sw = mp[5] - mp[1] * X[:, 13] - mp[0] / X[:, 6] * np.sqrt(X[:, 10] ** 2 + X[:, 11] ** 2 + X[:, 12] ** 2)
        assert np.allclose(r[:, -1], sw, rtol=1e-13, atol=1e-15)


def test_trace_interceptor_two_stages(eng):
    """interceptor::ComputeTraj traces both stages (interceptor.cpp:165-220): 2 x (S+1) rows when the
    flight crosses the burn-out time, the chart id in the last column."""
    mp = np.array(S.DEFAULTS[S.INTERCEPTOR], dtype=np.float64)
    X0 = np.array(S.INTERCEPTOR_INIT_XI + [0.01, -1, 0.5, 0.2, 100., 50.])
    t1 = mp[4] / mp[6]
    rows, nrows, Xf = eng.trace_batch(S.INTERCEPTOR, mp, 0.0, np.tile(X0, (2, 1)), np.array([t1 + 5.0, t1 - 5.0]), 50)
    assert list(nrows) == [102, 51]
    assert rows[0, 50, 0] == pytest.approx(t1) and rows[0, 51, 0] == t1
    assert np.array_equal(rows[0, 50, 1:13], rows[0, 51, 1:13])        # stage 2 starts where stage 1 ended
    assert set(np.unique(rows[0, :102, -1])) <= {1.0, 2.0}
    end = eng.traj_batch(S.INTERCEPTOR, mp, 0.0, np.tile(X0, (2, 1)), np.array([t1 + 5.0, t1 - 5.0]), 50)
    assert np.array_equal(Xf, end)
