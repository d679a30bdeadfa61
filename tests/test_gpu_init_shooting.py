"""GPU checks of the initial guess of a batch (socp_init_shooting_batch, Engine.init_shooting_batch): every interior
node bit for bit the socp_traj_batch / socp_traj_adaptive_batch of (ti, Xi, node time), on all five models; the guess
bench.py builds by hand; the unmodified reference's InitShooting (where its build is present) and the plain-C oracle;
the time line; HOST / DEVICE modes, batch position, M == 1, B == 0 and argument checks; and the C++ mirror's batched
InitShooting against the single-problem class.

Tolerance against the checkers: the trajectory rule of test_gpu_traj.py (1e-12 norm-relative, relaxed for Goddard and
the interceptor only as far as the oracle shows a trajectory amplifies rounding-level differences)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import scenarios as S
from gpu_util import engine
from test_gpu_traj import TOL, check_traj, conditioned_tol, errors

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "cpp", "build", "bin")

# per model: initial state and costate, final time (ti = 0); the interceptor's M = 4 grid puts node 3 past burn-out
# (propellant_mass / q = 20 s), so that node integrates across the stage change
XI = {S.GODDARD: S.GODDARD_XI, S.DI: np.r_[np.zeros(6), 0.01 * np.ones(6)], S.COVID19: S.COVID_XI,
      S.VTOL: np.array([20, 8, 5, 0.3, 0.2, 0.1, -0.03, 0.013, -0.003, -0.29, 0.1, -0.03]),
      S.INTERCEPTOR: np.array(S.INTERCEPTOR_INIT_XI + [0.01, -1, 0.5, 0.2, 100., 50.])}
TF = {S.GODDARD: 0.1, S.DI: 8.0, S.COVID19: 20.0, S.VTOL: 5.0, S.INTERCEPTOR: 40.0}


def mparams_of(model):
    mp = np.array(S.DEFAULTS[model], dtype=np.float64)
    if model == S.GODDARD:
        mp[6], mp[2] = 1.0, 0.0                  # mu2 = 1, KD = 0 (tests/testGoddard.cpp:94)
    return mp


def inputs(model, B, seed=0):
    """B perturbed copies of the model's (ti, Xi, tf, Xf); problem 0 unperturbed"""
    rng = np.random.default_rng(20261022 + 31 * model + seed)
    n = S.DIM[model]
    Xi = XI[model] * (1 + 1e-3 * rng.uniform(-1, 1, size=(B, 2 * n)))
    Xi[0] = XI[model]
    ti = 1e-3 * TF[model] * rng.uniform(0, 1, size=B)
    tf = TF[model] * (1 + 1e-2 * rng.uniform(-1, 1, size=B))
    ti[0], tf[0] = 0.0, TF[model]
    Xf = np.ascontiguousarray(Xi[:, :n] * (1 + 0.1 * rng.uniform(-1, 1, size=(B, n))))
    return ti, np.ascontiguousarray(Xi), tf, Xf


def shape_for(model, M, free=(), ode_tol=0.0):
    """SetMode(FREE, FIXED) plus FREE interior node times at the nodes in `free`"""
    import socp_b200 as sb
    mode_t, mode_X = S.default_modes(model, M, S.FREE, [S.FIXED] * S.DIM[model])
    for j in free:
        mode_t[j] = S.FREE
    return sb.make_shape(model, M, mode_t, mode_X, 0, ode_tol=ode_tol)


def grid(ti, tf, M):
    """time[b][i] = ti + i * (tf - ti) / M, the reference's expression"""
    return np.stack([ti + i * (tf - ti) / M for i in range(M + 1)], axis=1)


def c(a):
    return np.ascontiguousarray(a)


# (model, M, B): vtolUAV at a batch whose B (M - 1) items take the four-lane cooperative kernel and at one that does not
CASES = [(S.GODDARD, 6, 64), (S.DI, 4, 64), (S.COVID19, 5, 32), (S.VTOL, 4, 16), (S.VTOL, 4, 8000), (S.INTERCEPTOR, 4, 64)]


@pytest.mark.parametrize("adaptive", [False, True], ids=["rk4", "dopri5"])
@pytest.mark.parametrize("model,M,B", CASES)
def test_nodes_are_traj_bit_for_bit(model, M, B, adaptive):
    tol = 1e-8 if adaptive else 0.0
    ti, Xi, tf, Xf = inputs(model, B)
    mp = mparams_of(model)
    eng = engine()
    time, Xb, x = eng.init_shooting_batch(shape_for(model, M, ode_tol=tol), mp, ti, Xi, tf, Xf)
    n, N = S.DIM[model], 2 * S.DIM[model]
    assert np.array_equal(time, grid(ti, tf, M))
    for i in range(1, M):
        if adaptive and model != S.INTERCEPTOR:
            want, ns = eng.traj_adaptive_batch(model, mp, ti, Xi, c(time[:, i]), tol)
            assert np.all(ns[:, 0] > 0)
        else:
            want = eng.traj_batch(model, mp, ti, Xi, c(time[:, i]))
        # the interceptor keeps its fixed-step loop with SOCP_DOPRI5 (interceptor.cpp:104-130), and its node is the
        # socp_traj_batch integration: socp_traj_adaptive_batch runs the same loop from a kernel instance the compiler
        # contracts differently, and the stage change at node 2 (t = 20 s, burn-out) turns those last bits into
        # different trajectories
        assert np.array_equal(x[:, N * i:N * (i + 1)], want), (model, i)
        assert np.array_equal(Xb[:, i], want[:, :n]), (model, i)
    assert np.array_equal(x[:, :N], Xi) and np.array_equal(Xb[:, 0], Xi[:, :n]) and np.array_equal(Xb[:, M], Xf)
    assert np.array_equal(x[:, N * M], time[:, M]) and x.shape[1] == N * M + 1


def test_goddard_explicit_switching_times():
    """With mu2 = 0 the thrust is 1, 0.5 and 0 between the switching times: sw [B][2] reaches every node, and a
    node is the socp_traj_batch of the same sw."""
    B, M = 64, 6
    ti, Xi, tf, Xf = inputs(S.GODDARD, B)
    mp = mparams_of(S.GODDARD)
    mp[6], mp[7] = 0.0, 0.5                      # mu2 = 0: thrust 1 up to sw[0], 0.5 up to sw[1], then 0
    rng = np.random.default_rng(4)
    sw = c(np.stack([0.03 + 0.005 * rng.uniform(-1, 1, B), 0.07 + 0.005 * rng.uniform(-1, 1, B)], axis=1))
    eng = engine()
    shape = shape_for(S.GODDARD, M)
    time, Xb, x = eng.init_shooting_batch(shape, mp, ti, Xi, tf, Xf, sw=sw)
    _, _, x0 = eng.init_shooting_batch(shape, mp, ti, Xi, tf, Xf)
    for i in range(1, M):
        want = eng.traj_batch(S.GODDARD, mp, ti, Xi, c(time[:, i]), sw=sw)
        assert np.array_equal(x[:, 14 * i:14 * (i + 1)], want), i
    assert not np.array_equal(x, x0)             # the default switching times give another guess


def test_bench_goddard_guess():
    """bench.goddard_workload's hand-written node loop and the batched call build the same time line and node blocks,
    and the same boundary states at nodes 0 and M.  Two entries differ, where the bench departs from InitShooting:
      * the FREE final time: the bench writes tf = 0.1, InitShooting takes node M of the time line,
        0 + 6 (0.1 - 0) / 6 = 0.10000000000000002, one ulp above;
      * the interior rows of Xb: the bench leaves them at zero, InitShooting stores the node states there.  The residual
        reads no boundary state of a CONTINUOUS node: with the bench's final time both give the same residual."""
    import bench
    B, seed = 4096, 3
    eng = engine()
    shape, mp, time_b, Xb_b, x_b = bench.goddard_workload(eng, B, seed)
    Xi, xf0 = S.goddard_batch_inputs(B, seed=seed)
    Xf = np.zeros((B, 7))
    Xf[:, 0] = xf0
    mp_init = np.array(S.DEFAULTS[S.GODDARD])
    mp_init[6] = 1.0
    time, Xb, x = eng.init_shooting_batch(shape, mp_init, 0.0, Xi, 0.1, Xf)
    Xb_b = Xb_b.reshape(B, 7, 7)
    assert np.array_equal(time, time_b) and np.array_equal(x[:, :84], x_b[:, :84])
    assert np.all(x[:, 84] == time[:, 6]) and np.all(x_b[:, 84] == 0.1) and np.all(time[:, 6] == np.nextafter(0.1, 1))
    assert np.array_equal(Xb[:, [0, 6]], Xb_b[:, [0, 6]]) and not np.any(Xb_b[:, 1:6])
    assert np.array_equal(Xb[:, 1:6], x[:, 14:84].reshape(B, 5, 14)[:, :, :7])
    x[:, 84] = 0.1
    assert np.array_equal(eng.residual_batch(shape, mp, time, c(Xb.reshape(B, -1)), x),
                          eng.residual_batch(shape, mp, time_b, c(Xb_b.reshape(B, -1)), x_b))


# the guesses the checkers restate: M >= 3, and one shape with a FREE interior time
REF_CASES = [(S.GODDARD, 6, ()), (S.GODDARD, 6, (3,)), (S.DI, 4, ()), (S.COVID19, 5, (2,)), (S.VTOL, 3, ()),
             (S.INTERCEPTOR, 4, ())]


def node_tol(model, mp, t0, X0, t):
    if model not in (S.GODDARD, S.INTERCEPTOR):
        return (TOL, TOL)
    from backends import OracleBackend
    return conditioned_tol(OracleBackend(), model, mp, t0, X0, t)


@pytest.mark.parametrize("model,M,free", REF_CASES)
def test_reference_init_shooting(model, M, free):
    """RefShooting.init(ti, Xi, tf, Xf) -> params() of the unmodified reference, problem by problem: 1e-12
    norm-relative (the interceptor: the bound test_gpu_traj.py derives for its trajectories)."""
    from oracle import pyref
    if not pyref.available():
        pytest.skip("reference build (oracle/_ref) not present")
    from backends import RefBackend
    B = 4
    ti, Xi, tf, Xf = inputs(model, B)
    mp = mparams_of(model)
    shape = shape_for(model, M, free)
    time, _, x = engine().init_shooting_batch(shape, mp, ti, Xi, tf, Xf)
    be = RefBackend()
    N = 2 * S.DIM[model]
    for b in range(B):
        m = be.model(model, mp)
        s = pyref.RefShooting(m, M, 1)
        s.set_mode(list(shape.mode_t)[:M + 1], [list(shape.mode_X[j])[:S.DIM[model]] for j in range(M + 1)])
        s.init(ti[b], Xi[b], tf[b], np.r_[Xf[b], np.zeros(S.DIM[model])])
        want = s.params()
        assert want.size == x.shape[1]
        assert np.array_equal(x[b, :N], want[:N]) and np.array_equal(x[b, N * M:], want[N * M:]), (model, b)
        if model == S.INTERCEPTOR:
            for i in range(1, M):
                check_traj(x[b, N * i:N * (i + 1)], want[N * i:N * (i + 1)], "interceptor problem %d node %d" % (b, i),
                           node_tol(model, mp, ti[b], Xi[b], time[b, i]))
        else:
            assert errors(x[b], want)[0] <= TOL, (model, b, errors(x[b], want))


@pytest.mark.parametrize("model,M,free", REF_CASES)
def test_oracle_nodes(model, M, free):
    """Every interior node against the plain-C oracle's integration of (ti, Xi) to the node time."""
    from backends import OracleBackend
    ora = OracleBackend()
    B = 8
    ti, Xi, tf, Xf = inputs(model, B, seed=1)
    mp = mparams_of(model)
    time, _, x = engine().init_shooting_batch(shape_for(model, M, free), mp, ti, Xi, tf, Xf)
    N = 2 * S.DIM[model]
    for b in range(B):
        for i in range(1, M):
            want = ora.traj(model, mp, ti[b], Xi[b], time[b, i])
            check_traj(x[b, N * i:N * (i + 1)], want, "model %d problem %d node %d" % (model, b, i),
                       node_tol(model, mp, ti[b], Xi[b], time[b, i]))


def test_time_line():
    """Node M is the grid expression, bit for bit, not tf; the FREE times follow the node blocks in node order."""
    B, M = 256, 7
    rng = np.random.default_rng(12)
    ti, Xi, _, Xf = inputs(S.DI, B)
    tf = ti + rng.uniform(0.1, 10.0, B)
    time, Xb, x = engine().init_shooting_batch(shape_for(S.DI, M, free=(5, 2)), mparams_of(S.DI), ti, Xi, tf, Xf)
    last = ti + M * (tf - ti) / M
    assert np.array_equal(time[:, M], last) and np.any(last != tf)
    assert np.array_equal(time, grid(ti, tf, M))
    assert np.array_equal(x[:, 12 * M:], time[:, [2, 5, M]])


def test_host_and_device_modes():
    """Torch CUDA tensors (produced on a side stream) give tensors with the HOST bits."""
    import torch
    B, M = 512, 6
    ti, Xi, tf, Xf = inputs(S.GODDARD, B)
    mp = np.tile(mparams_of(S.GODDARD), (B, 1))
    sw = c(np.tile([0.03, 0.07], (B, 1)))
    shape = shape_for(S.GODDARD, M, free=(2,))
    eng = engine()
    want = eng.init_shooting_batch(shape, mp, ti, Xi, tf, Xf, sw=sw)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        dev = lambda a: torch.from_numpy(c(a)).pin_memory().to("cuda", non_blocking=True)
        got = eng.init_shooting_batch(shape, dev(mp), dev(ti), dev(Xi), dev(tf), dev(Xf), sw=dev(sw))
        host = [g.cpu() for g in got]
    eng.use_torch_stream()
    assert all(torch.is_tensor(g) and g.is_cuda for g in got)
    for h, w in zip(host, want):
        assert np.array_equal(h.numpy(), w)


@pytest.mark.parametrize("model", [S.GODDARD, S.VTOL, S.INTERCEPTOR])
def test_independent_of_batch(model):
    """A problem's guess does not depend on its position or on B: B = 1 per problem against a shuffled B = 4096."""
    B, M = 8, 4
    ti, Xi, tf, Xf = inputs(model, B, seed=2)
    mp = mparams_of(model)
    shape = shape_for(model, M)
    eng = engine()
    single = [eng.init_shooting_batch(shape, mp, ti[b:b + 1], Xi[b:b + 1], tf[b:b + 1], Xf[b:b + 1]) for b in range(B)]
    idx = np.random.default_rng(0).permutation(np.tile(np.arange(B), 4096 // B))
    big = eng.init_shooting_batch(shape, mp, c(ti[idx]), c(Xi[idx]), c(tf[idx]), c(Xf[idx]))
    for k in range(idx.size):
        for got, one in zip(big, single[idx[k]]):
            assert np.array_equal(got[k], one[0]), (model, k)


def test_one_segment_and_empty_batch():
    """M == 1 copies only (no integration); B == 0 does nothing."""
    B = 5
    ti, Xi, tf, Xf = inputs(S.COVID19, B)
    eng = engine()
    eng.reset_stats()
    time, Xb, x = eng.init_shooting_batch(shape_for(S.COVID19, 1), mparams_of(S.COVID19), ti, Xi, tf, Xf)
    assert eng.stats()["rk4_steps"] == 0
    assert np.array_equal(time, grid(ti, tf, 1)) and np.array_equal(x, np.c_[Xi, time[:, 1]])
    assert np.array_equal(Xb[:, 0], Xi[:, :4]) and np.array_equal(Xb[:, 1], Xf)
    time, Xb, x = eng.init_shooting_batch(shape_for(S.COVID19, 3), mparams_of(S.COVID19), ti[:0], Xi[:0], tf[:0], Xf[:0])
    assert time.shape == (0, 4) and Xb.shape == (0, 4, 4) and x.shape == (0, 25)


def test_edges():
    """B = 0 leaves the outputs alone; NULL arguments, a negative B and a bad shape are SOCP_ERR_ARG."""
    import socp_b200 as sb
    B, M = 2, 3
    ti, Xi, tf, Xf = inputs(S.DI, B)
    mp = c(np.tile(mparams_of(S.DI), (B, 1)))
    shape = shape_for(S.DI, M)
    eng = engine()
    L, h = eng._L, eng._h
    d = lambda a: ctypes.c_void_p(a.ctypes.data)
    time, Xb, x = np.full((B, M + 1), 7.0), np.full((B, M + 1, 6), 7.0), np.full((B, 12 * M + 1), 7.0)
    sh = ctypes.byref(shape)
    args = [d(mp), d(ti), d(Xi), d(tf), d(Xf), d(time), d(Xb), d(x)]
    call = lambda s, B_, a: L.socp_init_shooting_batch(h, s, B_, a[0], None, *a[1:], 0)
    assert call(sh, 0, args) == 0
    assert np.all(time == 7.0) and np.all(Xb == 7.0) and np.all(x == 7.0)
    for k in range(len(args)):
        a = list(args)
        a[k] = None
        assert call(sh, B, a) == -1, k
    assert call(sh, -1, args) == -1
    assert call(None, B, args) == -1
    assert L.socp_init_shooting_batch(None, sh, B, args[0], None, *args[1:], 0) == -1
    for bad in ("model", "mode_t", "continuous_end", "num_multi", "integrator"):
        s2 = shape_for(S.DI, M)
        if bad == "model":
            s2.model_id = 9
        elif bad == "mode_t":
            s2.mode_t[1] = 7
        elif bad == "continuous_end":
            s2.mode_t[0] = S.CONTINUOUS
        elif bad == "num_multi":
            s2.num_multi = 0
        else:
            s2.integrator = 5
        assert call(ctypes.byref(s2), B, args) == -1, bad
    assert np.all(time == 7.0) and np.all(Xb == 7.0) and np.all(x == 7.0)
    with pytest.raises(ValueError):
        eng.init_shooting_batch(shape, mparams_of(S.DI), ti, Xi, tf, c(Xi))
    s2 = shape_for(S.DI, M)
    s2.mode_t[0] = S.CONTINUOUS
    with pytest.raises(sb.SocpError):
        eng.init_shooting_batch(s2, mparams_of(S.DI), ti, Xi, tf, Xf)


def test_mirror_demo():
    """shooting_batch::InitShooting then GetParameters(k) equals shooting::InitShooting bit for bit for every member:
    Goddard with switching times set on the model, and the double integrator with the adaptive integrator."""
    exe = os.path.join(BIN, "demo_init_shooting")
    assert os.access(exe, os.X_OK), "run __graft_entry__.build() first"
    r = subprocess.run([exe, "64"], capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "goddard: 64 of 64 members identical to shooting::InitShooting" in r.stdout, r.stdout
    assert "di: 64 of 64 members identical to shooting::InitShooting" in r.stdout, r.stdout
