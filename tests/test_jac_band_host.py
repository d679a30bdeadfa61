"""The structural band of the shooting Jacobian (socp_jac_band) on the Goddard shapes: the solver's Jacobian phase
stores only these rows of every column, so (a) the forward-difference Jacobian must be an exact zero outside them, and
(b) a Householder QR without pivoting (MINPACK qrfac's arithmetic) must keep R and its reflectors inside them.
No GPU: the band is host code and the Jacobian comes from the oracle port."""
import ctypes

import numpy as np
import pytest

import scenarios as S
from backends import OracleBackend


def jac_band(spec):
    import socp_b200 as sb
    from socp_b200 import _lib
    shape = sb.make_shape(spec["model"], spec["M"], spec["mode_t"], spec["mode_X"], spec["steps"])
    P = S.num_param(spec)
    lo = (ctypes.c_int * P)()
    end = (ctypes.c_int * P)()
    rc = _lib.lib().socp_jac_band(ctypes.byref(shape), lo, end)
    assert rc in (0, 1)
    return rc == 1, np.array(lo), np.array(end)


def outside(lo, end, n):
    rows = np.arange(n)[:, None]
    return (rows < lo[None, :]) | (rows >= end[None, :])


def goddard_spec(M, k):
    ora = OracleBackend()
    Xi, xf0 = S.goddard_batch_inputs(8)
    return S.goddard_problem(lambda mp, a, b, c: ora.traj(S.GODDARD, mp, a, b, c, 10), M=M, Xi=Xi[k], xf0=xf0[k])


def qr_steps(J):
    """MINPACK qrfac without pivoting on a copy of J; yields the working matrix after every reflector (R above the
    diagonal, the reflectors on and below it)."""
    a = J.copy()
    n = a.shape[0]
    for j in range(n):
        v = a[j:, j]
        ajnorm = np.linalg.norm(v)
        if ajnorm != 0.0:
            if v[0] < 0.0:
                ajnorm = -ajnorm
            v /= ajnorm
            v[0] += 1.0
            for k in range(j + 1, n):
                s = v @ a[j:, k]
                if s != 0.0:
                    a[j:, k] -= (s / v[0]) * v
        yield a


# (the benchmark's shape: M = 6, P = 85; scenarios.goddard_problem at M = 6 and at M = 12, P = 169)
@pytest.mark.parametrize("M,k", [(6, 0), (6, 5), (12, 3)])
def test_goddard_jacobian_stays_in_its_band(M, k):
    spec = goddard_spec(M, k)
    P = S.num_param(spec)
    banded, lo, end = jac_band(spec)
    assert banded == (P <= 96)
    assert np.all(lo <= np.arange(P)) and np.all(end > np.arange(P))
    off = outside(lo, end, P)
    ora = OracleBackend()
    rng = np.random.default_rng(k)
    x0 = np.asarray(spec["x0"], dtype=np.float64)
    for x in (x0, x0 * (1 + 1e-3 * rng.standard_normal(P))):
        J = ora.fdjac(spec, x)
        assert np.count_nonzero(J) > P
        assert np.all(J[off] == 0.0), "forward-difference Jacobian non-zero outside the band"
        for step, a in enumerate(qr_steps(J)):
            assert np.all(a[off] == 0.0), "Householder QR fills a row outside the band (reflector %d)" % step


def test_band_of_the_benchmark_shape():
    """P = 85: the first block keeps its two blocks of rows, the middle blocks three, and the last block and the final
    time are dense (the final conditions of the last segment are rows of the first block)."""
    spec = goddard_spec(6, 0)
    banded, lo, end = jac_band(spec)
    assert banded
    N = 14
    for j in range(85):
        p = j // N
        if p == 0:
            assert (lo[j], end[j]) == (0, 2 * N)
        elif p < 5:
            assert (lo[j], end[j]) == (0 if p == 1 else N * (p - 1), N * (p + 2))
        else:
            assert (lo[j], end[j]) == (0, 85)


def test_free_interior_time_keeps_the_dense_kernel():
    import socp_b200 as sb
    mode_t, mode_X = sb.default_modes(sb.GODDARD, 6, sb.FREE, S.GODDARD_MODE_XF)
    mode_t = list(mode_t)
    mode_t[3] = sb.FREE
    spec = dict(model=S.GODDARD, M=6, mode_t=mode_t, mode_X=mode_X, steps=10)
    P = S.num_param(spec)
    assert P == 86
    banded, _, _ = jac_band(spec)
    assert not banded
