"""GPU checks of Move(t) and GetSolution for a batch of solved problems (socp_move_batch, socp_solution_batch),
and of the re-mesh they serve: the golden Goddard stage 4 and interceptor scenario data, a Python restatement of
shooting::Move(tf) on the plain-C oracle for all five models, bit-identity with socp_traj_batch, HOST / DEVICE
modes, argument checks and the four-stage Goddard pipeline demo of the C++ mirror.

Tolerance: the trajectory rule of test_gpu_traj.py (1e-12 norm- and component-relative, relaxed for Goddard and
the interceptor only as far as the oracle shows a trajectory amplifies rounding-level differences)."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import scenarios as S
from golden_util import by_name, spec_from_hex, unhex
from gpu_util import engine, shape_of
from test_gpu_traj import TOL, check_traj, conditioned_tol

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "cpp", "build", "bin")
S1, S2 = 0.0227, 0.08


def stage4_times(tf):
    return np.array([0.0, S1 / 2, S1, (S2 + S1) / 2, S2, (S2 + tf) / 2, tf])


def solved(kind, name, goal_param=True):
    """spec, solution x and the model parameters it was solved with"""
    e = by_name(kind, name)
    spec = spec_from_hex(e["spec"])
    mp = np.array(spec["mparams"])
    if kind == "cont_param" and goal_param:
        mp[S.pidx(spec["model"], e["pname"])] = unhex(e["goal"])
    return spec, unhex(e["x"]), mp


def oracle_problem(spec, mp, ode_tol=0.0):
    from backends import OracleBackend
    p = OracleBackend().problem(dict(spec, mparams=list(mp)))
    if ode_tol > 0:
        p.p.integrator, p.p.ode_tol = 1, ode_tol
    return p


def oracle_move(p, x, tq, M, N):
    """shooting::Move(tf) (cpp/src/socp/shooting.cpp:146-160) on the oracle: returns (state, t_seg, seg, target)"""
    tl = p.timeline(x)                           # ComputeTimeLine: also the switching times of the model
    t0, t_end = tl[0], tl[M]
    target = tq if (tq >= t0 and tq <= t_end) else t_end
    seg = 0
    while tl[seg + 1] < target:
        seg += 1
    return p.traj(tl[seg], x[N * seg:N * seg + N], target), tl[seg], seg, target


# one solved problem per model (golden), perturbed into a batch; Goddard's stage 4 has FREE interior times
CASES = {S.GODDARD: ("solve", "goddard_stage4_singular"), S.DI: ("solve", "di_free_tf"),
         S.COVID19: ("solve", "covid_stage1"), S.VTOL: ("solve", "vtol_wp1"),
         S.INTERCEPTOR: ("solve", "interceptor_init")}


def batch_case(model, B=16, seed=0):
    spec, x, mp = solved(*CASES[model])
    rng = np.random.default_rng(20261000 + 17 * model + seed)
    X = x * (1 + 1e-6 * rng.uniform(-1, 1, size=(B, x.size)))
    X[0] = x
    return spec, X, mp


def queries(p, x, M, rng):
    """Q = 7: t0, node time t_1, t_end, below t0, above t_end, an interior time, the node time t_{M-1}"""
    tl = p.timeline(x)
    return np.array([tl[0], tl[1], tl[M], tl[0] - 1.0, tl[M] + 1.0, tl[0] + rng.uniform(0.05, 0.95) * (tl[M] - tl[0]),
                     tl[max(M - 1, 1)]])


def tol_for(model, mp, t0, X0, tf, steps, sw):
    if model not in (S.GODDARD, S.INTERCEPTOR):
        return (TOL, TOL)
    from backends import OracleBackend
    return conditioned_tol(OracleBackend(), model, mp, t0, X0, tf, steps, sw)


def test_golden_goddard_stage4():
    """The re-mesh of tests/testGoddard.cpp:115-145 from the golden stage-3 solution reproduces the golden stage-4
    spec (its x0 node blocks and Xb, Xb[6] = Move(tf)); solving it gives the golden stage-4 solution."""
    spec3, x3, mp3 = solved("cont_param", "goddard_stage3_mu2")
    shape3 = shape_of(spec3)
    eng = engine()
    vt, vX = eng.solution_batch(shape3, mp3, np.array([spec3["time"]]), x3[None])
    assert vt[0, 6] == x3[-1] and np.array_equal(vX[0, :6], x3[:84].reshape(6, 14))
    e4 = by_name("solve", "goddard_stage4_singular")
    g4 = spec_from_hex(e4["spec"])
    vt4 = stage4_times(vt[0, 6])
    assert np.array_equal(vt4, g4["time"])
    Xq = eng.move_batch(shape3, mp3, np.array([spec3["time"]]), x3[None], vt4[None])[0]
    assert np.array_equal(Xq[6], vX[0, 6])                            # GetSolution's last node is Move(t_end)
    p = oracle_problem(spec3, mp3)
    x0, Xb = np.array(g4["x0"]), np.array(g4["Xb"])
    for i in range(7):
        _, t_seg, seg, target = oracle_move(p, x3, vt4[i], 6, 14)
        tol = tol_for(S.GODDARD, mp3, t_seg, x3[14 * seg:14 * seg + 14], target, spec3["steps"], None)
        want = np.r_[x0[14 * i:14 * i + 14]] if i < 6 else Xb[6]
        check_traj(Xq[i, :want.size], want, "stage-4 node %d" % i, tol)
        check_traj(Xq[i, :7], Xb[i], "stage-4 Xb %d" % i, tol)
    # solve the re-meshed problem
    import socp_b200 as sb
    shape4 = shape_of(g4)
    x, Xb4 = sb.unknowns_from_nodes(shape4, vt4[None], Xq[None])
    r = eng.solve_batch(shape4, np.array(g4["mparams"]), vt4[None], Xb4.reshape(1, -1), np.ascontiguousarray(x), xtol=g4["xtol"])
    xg = unhex(e4["x"])
    assert r["info"][0] == 1
    assert np.linalg.norm(r["x"][0] - xg) <= g4["xtol"] * np.linalg.norm(xg)


def test_golden_interceptor_get_solution():
    """GetSolution after the mu_gft continuation gives the previous boundary data of the scenario continuations
    (tests/testInterceptor.cpp:194-199): x0 = [vX[0], vt[1]] (copies, bit-exact), Xb[1] = vX[1][:6] = Move(t_end)."""
    spec, x, mp = solved("cont_param", "interceptor_mu_gft")
    vt, vX = engine().solution_batch(shape_of(spec), mp, np.array([spec["time"]]), x[None])
    tol = tol_for(S.INTERCEPTOR, mp, vt[0, 0], x[:12], vt[0, 1], spec["steps"], None)
    for sc in ("S1", "S2", "S3"):
        s = spec_from_hex(by_name("cont_boundary", "interceptor_" + sc)["spec"])
        assert np.array_equal(np.r_[vX[0, 0], vt[0, 1]], s["x0"]), sc
        assert np.array_equal(vt[0], s["time"]) and np.array_equal(vX[0, 0, :6], s["Xb"][0]), sc
        check_traj(vX[0, 1, :6], np.array(s["Xb"][1]), "interceptor %s Xb[1]" % sc, tol)
    check_traj(vX[0, 1], oracle_move(oracle_problem(spec, mp), x, vt[0, 1], 1, 12)[0], "interceptor Move(t_end)", tol)


def _move_case(model, ode_tol=0.0, B=16):
    spec, X, mp = batch_case(model, B)
    import socp_b200 as sb
    shape = sb.make_shape(spec["model"], spec["M"], spec["mode_t"], spec["mode_X"], spec["steps"], ode_tol=ode_tol)
    time = np.tile(spec["time"], (B, 1))
    return spec, shape, X, mp, time


@pytest.mark.parametrize("model", sorted(CASES))
def test_move_vs_oracle(model):
    spec, shape, X, mp, time = _move_case(model)
    M, N = spec["M"], 2 * len(spec["Xb"][0])
    rng = np.random.default_rng(7 + model)
    p = oracle_problem(spec, mp)
    tq = np.array([queries(p, X[b], M, rng) for b in range(X.shape[0])])
    got = engine().move_batch(shape, mp, time, X, tq)
    assert got.shape == (X.shape[0], 7, N)
    for b in range(X.shape[0]):
        for q in range(7):
            want, t_seg, seg, target = oracle_move(p, X[b], tq[b, q], M, N)
            sw = [p.p.sw[0], p.p.sw[1]] if model == S.GODDARD else None
            tol = tol_for(model, mp, t_seg, X[b, N * seg:N * seg + N], target, spec["steps"], sw)
            check_traj(got[b, q], want, "model %d problem %d query %d" % (model, b, q), tol)


def test_move_dopri5_vs_oracle():
    """An adaptive (SOCP_DOPRI5) shape: every Move integrates with the oracle's Dormand-Prince restatement."""
    spec, shape, X, mp, time = _move_case(S.DI, ode_tol=1e-9)
    M, N = spec["M"], 12
    rng = np.random.default_rng(3)
    p = oracle_problem(spec, mp, ode_tol=1e-9)
    tq = np.array([queries(p, X[b], M, rng) for b in range(X.shape[0])])
    got = engine().move_batch(shape, mp, time, X, tq)
    for b in range(X.shape[0]):
        for q in range(7):
            check_traj(got[b, q], oracle_move(p, X[b], tq[b, q], M, N)[0], "dopri5 problem %d query %d" % (b, q))


def _sw_of(shape, vt):
    """the switching times the device derives: the first two FREE interior node times (defaults otherwise)"""
    sw = np.tile([S1, S2], (vt.shape[0], 1))
    free = [j for j in range(1, shape.num_multi) if shape.mode_t[j] == S.FREE][:2]
    for k, j in enumerate(free):
        sw[:, k] = vt[:, j]
    return np.ascontiguousarray(sw)


@pytest.mark.parametrize("model", sorted(CASES))
def test_move_is_traj_bit_for_bit(model):
    """Move == socp_traj_batch on the same segment start, node state, target, switching times and S; a query at
    node time t_{j+1} returns the end of segment j, not node j+1."""
    spec, shape, X, mp, time = _move_case(model)
    M, N, B = spec["M"], 2 * len(spec["Xb"][0]), X.shape[0]
    eng = engine()
    vt, vX = eng.solution_batch(shape, mp, time, X)
    assert np.array_equal(vX[:, :M], X[:, :N * M].reshape(B, M, N))
    sw = _sw_of(shape, vt)
    rng = np.random.default_rng(11)
    for j in range(M):
        # an interior time of segment j, and its end node time t_{j+1}
        for at_node, tq in ((False, vt[:, j] + rng.uniform(0.1, 0.9, B) * (vt[:, j + 1] - vt[:, j])), (True, vt[:, j + 1])):
            got = eng.move_batch(shape, mp, time, X, np.ascontiguousarray(tq[:, None]))[:, 0]
            want = eng.traj_batch(model, mp, np.ascontiguousarray(vt[:, j]), np.ascontiguousarray(X[:, N * j:N * j + N]),
                                  np.ascontiguousarray(tq), spec["steps"], sw=sw)
            assert np.array_equal(got, want), (model, j, at_node)
            if at_node and j < M - 1:            # the perturbed solutions are not continuous at the nodes
                assert not np.any([np.array_equal(got[b], X[b, N * (j + 1):N * (j + 2)]) for b in range(1, B)])
    # GetSolution's last node is Move(t_end) is the end of the last segment
    want = eng.traj_batch(model, mp, np.ascontiguousarray(vt[:, M - 1]), np.ascontiguousarray(X[:, N * (M - 1):N * M]),
                          np.ascontiguousarray(vt[:, M]), spec["steps"], sw=sw)
    assert np.array_equal(vX[:, M], want)


@pytest.mark.parametrize("model", sorted(CASES))
def test_move_independent_of_batch(model):
    """B = 1 against B = 4096 (every problem at many positions): the same bits.  For vtolUAV the small batches run
    the cooperative four-lane kernel and the large one the one-thread kernel."""
    spec, shape, X, mp, time = _move_case(model, B=8)
    M, B = spec["M"], X.shape[0]
    rng = np.random.default_rng(5)
    p = oracle_problem(spec, mp)
    tq = np.array([queries(p, X[b], M, rng) for b in range(B)])
    eng = engine()
    single = np.array([eng.move_batch(shape, mp, time[:1], X[b:b + 1], tq[b:b + 1])[0] for b in range(B)])
    reps = 4096 // B
    big = eng.move_batch(shape, mp, np.tile(time, (reps, 1)), np.tile(X, (reps, 1)), np.tile(tq, (reps, 1)))
    for r in range(reps):
        assert np.array_equal(big[r * B:(r + 1) * B], single), (model, r)
    vt1, vX1 = eng.solution_batch(shape, mp, time[:1], X[:1])
    vt, vX = eng.solution_batch(shape, mp, np.tile(time, (reps, 1)), np.tile(X, (reps, 1)))
    assert np.array_equal(vt[::B], np.tile(vt1, (reps, 1))) and np.array_equal(vX[::B], np.tile(vX1, (reps, 1, 1)))


def test_host_and_device_modes():
    """DEVICE mode (torch tensors, on a non-default stream the inputs were produced on) gives the HOST bits; the
    whole stage-4 re-mesh runs on the device and solves to the same bits as on the host."""
    import torch
    import socp_b200 as sb
    spec, shape, X, mp, time = _move_case(S.GODDARD, B=64)
    rng = np.random.default_rng(9)
    p = oracle_problem(spec, mp)
    tq = np.array([queries(p, X[b], 6, rng) for b in range(X.shape[0])])
    eng = engine()
    want = eng.move_batch(shape, mp, time, X, tq)
    vt_h, vX_h = eng.solution_batch(shape, mp, time, X)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().to("cuda", non_blocking=True)
        mp_d, time_d, X_d, tq_d = dev(np.tile(mp, (64, 1))), dev(time), dev(X), dev(tq)
        out = eng.move_batch(shape, mp_d, time_d, X_d, tq_d)
        vt_d, vX_d = eng.solution_batch(shape, mp_d, time_d, X_d)
        got, vt_g, vX_g = out.cpu(), vt_d.cpu(), vX_d.cpu()
    assert torch.is_tensor(out) and np.array_equal(got.numpy(), want)
    assert np.array_equal(vt_g.numpy(), vt_h) and np.array_equal(vX_g.numpy(), vX_h)
    # stage 4 of tests/testGoddard.cpp, host and device
    spec3, x3, mp3 = solved("cont_param", "goddard_stage3_mu2")
    g4 = spec_from_hex(by_name("solve", "goddard_stage4_singular")["spec"])
    shape3, shape4 = shape_of(spec3), shape_of(g4)
    B = 4
    x3b = x3 * (1 + 1e-7 * np.random.default_rng(1).uniform(-1, 1, (B, x3.size)))
    t3 = np.tile(spec3["time"], (B, 1))
    results = []
    for mem in ("host", "device"):
        conv = (lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()) if mem == "device" else (lambda a: a)
        mp3b, mp4b = conv(np.tile(mp3, (B, 1))), conv(np.tile(g4["mparams"], (B, 1)))
        vt, vX = eng.solution_batch(shape3, mp3b, conv(t3), conv(x3b))
        vt4 = conv(np.stack([stage4_times(t) for t in vt[:, 6].tolist()]))
        Xq = eng.move_batch(shape3, mp3b, conv(t3), conv(x3b), vt4)
        x, Xb = sb.unknowns_from_nodes(shape4, vt4, Xq)
        r = eng.solve_batch(shape4, mp4b, vt4, Xb.reshape(B, -1), x if mem == "device" else np.ascontiguousarray(x),
                            xtol=g4["xtol"])
        results.append([np.asarray(v.cpu()) if torch.is_tensor(v) else v for v in (Xq, r["x"], r["info"])])
    eng.use_torch_stream()                       # back to the default stream for the tests that follow
    for h, d in zip(*results):
        assert np.array_equal(h, d)
    assert np.all(results[0][2] == 1)


def test_edges():
    """B = 0 and Q = 0 are no-ops; NULL arguments, a bad shape and a negative Q are SOCP_ERR_ARG."""
    import socp_b200 as sb
    spec, shape, X, mp, time = _move_case(S.DI, B=2)
    eng = engine()
    L, h = eng._L, eng._h
    d = lambda a: ctypes.c_void_p(a.ctypes.data)
    mpb = np.ascontiguousarray(np.tile(mp, (2, 1)))
    tq = np.zeros((2, 3))
    Xq = np.full((2, 3, 12), 7.0)
    vt, vX = np.full((2, spec["M"] + 1), 7.0), np.full((2, spec["M"] + 1, 12), 7.0)
    sh = ctypes.byref(shape)
    assert L.socp_move_batch(h, sh, 0, d(mpb), d(time), d(X), 3, d(tq), d(Xq), 0) == 0
    assert L.socp_move_batch(h, sh, 2, d(mpb), d(time), d(X), 0, d(tq), d(Xq), 0) == 0
    assert L.socp_solution_batch(h, sh, 0, d(mpb), d(time), d(X), d(vt), d(vX), 0) == 0
    assert np.all(Xq == 7.0) and np.all(vt == 7.0) and np.all(vX == 7.0)
    assert L.socp_move_batch(h, sh, 2, d(mpb), d(time), d(X), -1, d(tq), d(Xq), 0) == -1
    args = [d(mpb), d(time), d(X), d(tq), d(Xq)]
    for k in range(5):
        a = list(args)
        a[k] = None
        assert L.socp_move_batch(h, sh, 2, a[0], a[1], a[2], 3, a[3], a[4], 0) == -1
    args = [d(mpb), d(time), d(X), d(vt), d(vX)]
    for k in range(5):
        a = list(args)
        a[k] = None
        assert L.socp_solution_batch(h, sh, 2, *a, 0) == -1
    assert L.socp_move_batch(h, None, 2, *args[:3], 3, d(tq), d(Xq), 0) == -1
    assert L.socp_move_batch(None, sh, 2, *args[:3], 3, d(tq), d(Xq), 0) == -1
    for bad in ("model", "mode_t", "continuous_end"):
        s2 = sb.make_shape(spec["model"], spec["M"], spec["mode_t"], spec["mode_X"], spec["steps"])
        if bad == "model":
            s2.model_id = 9
        elif bad == "mode_t":
            s2.mode_t[1] = 7
        else:
            s2.mode_t[0] = S.CONTINUOUS
        assert L.socp_move_batch(h, ctypes.byref(s2), 2, *args[:3], 3, d(tq), d(Xq), 0) == -1, bad
        assert L.socp_solution_batch(h, ctypes.byref(s2), 2, *args, 0) == -1, bad
    assert np.all(Xq == 7.0)


def _demo(*args):
    exe = os.path.join(BIN, "demo_goddard_pipeline")
    assert os.access(exe, os.X_OK), "run __graft_entry__.build() first"
    r = subprocess.run([exe] + list(args), capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    return r.stdout


@pytest.mark.parametrize("devices", ["1", "0"])
def test_goddard_pipeline_demo(devices):
    """The four Goddard stages on a batch of 128 (numDevice 0: every visible GPU shares it): member 0 is bit for bit
    the single-problem run, and its stage 4 converges to the golden singular-arc final time."""
    out = _demo("128", devices)
    assert "batch member 0 identical to the single run: yes" in out, out
    rows = re.findall(r"stage (\d) \(.*?\): (\d+) of 128 converged", out)
    assert [r[0] for r in rows] == ["1", "2", "3", "4"], out
    assert all(int(r[1]) > 0 for r in rows), out
    m = re.search(r"problem 0 stage 4: info (\d+) nfev \d+ tf (\S+)", out)
    assert m and int(m.group(1)) == 1, out
    tf = unhex(by_name("solve", "goddard_stage4_singular")["x"])[-1]
    assert abs(float(m.group(2)) - tf) <= 1e-6 * tf, (m.group(2), tf)
