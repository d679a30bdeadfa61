"""GPU checks of shooting::Trace for a batch of solved problems (socp_solution_trace_batch): bit-identity with
socp_trace_batch on every segment, the reference's row semantics, the oracle's controls and Hamiltonian, independence
from batch size and position, HOST / DEVICE modes, the RK4 observer of an adaptive shape, argument checks, a batch
whose row buffer passes 2^31 values, and the batch-trace demo of the C++ mirror."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import scenarios as S
from gpu_util import engine
from test_gpu_move import BIN, CASES, _move_case, _sw_of, oracle_problem

pytestmark = pytest.mark.gpu


def timelines(spec, shape, mp, X):
    """the oracle's ComputeTimeLine of every problem: tl [B][M+1], and the switching times sw [B][2] the device derives
    from it (only goddard reads them; they are the oracle's own there)"""
    p = oracle_problem(spec, mp)
    tl, osw = [], []
    for x in X:
        tl.append(p.timeline(x))
        osw.append([p.p.sw[0], p.p.sw[1]])
    tl = np.array(tl)
    sw = _sw_of(shape, tl)
    if spec["model"] == S.GODDARD:
        assert np.array_equal(sw, osw)
    return tl, sw


def segment_rows(eng, model, mp, tl, sw, X, j, N, steps):
    """socp_trace_batch of segment j of every problem"""
    rows, nrows, _ = eng.trace_batch(model, mp, np.ascontiguousarray(tl[:, j]), np.ascontiguousarray(X[:, N * j:N * j + N]),
                                     np.ascontiguousarray(tl[:, j + 1]), steps, sw=sw)
    return rows, nrows


@pytest.mark.parametrize("model", sorted(CASES))
def test_segments_are_trace_batch_bit_for_bit(model):
    spec, shape, X, mp, time = _move_case(model)
    M, N, B = spec["M"], 2 * len(spec["Xb"][0]), X.shape[0]
    eng = engine()
    rows, nrows = eng.solution_trace_batch(shape, mp, time, X)
    R, W = eng._L.socp_trace_max_rows(model, spec["steps"]), eng._L.socp_trace_width(model)
    assert rows.shape == (B, M, R, W) and nrows.shape == (B, M) and nrows.dtype == np.int32
    tl, sw = timelines(spec, shape, mp, X)
    vt, _ = eng.solution_batch(shape, mp, time, X)
    assert np.array_equal(tl, vt)
    for j in range(M):
        want, wn = segment_rows(eng, model, mp, tl, sw, X, j, N, spec["steps"])
        assert np.array_equal(nrows[:, j], wn), (model, j)
        for b in range(B):
            assert np.array_equal(rows[b, j, :wn[b]], want[b, :wn[b]]), (model, b, j)


@pytest.mark.parametrize("model", sorted(CASES))
def test_reference_semantics(model):
    """First row of segment j = (tl[j], node j); row times are repeated t += dt (each interceptor stage on its own);
    S+1 rows, 2(S+1) for an interceptor segment across burn-out; the last row of the last segment is Move(t_end)."""
    spec, shape, X, mp, time = _move_case(model)
    M, N, B, S_ = spec["M"], 2 * len(spec["Xb"][0]), X.shape[0], spec["steps"]
    eng = engine()
    rows, nrows = eng.solution_trace_batch(shape, mp, time, X)
    tl, _ = timelines(spec, shape, mp, X)
    _, vX = eng.solution_batch(shape, mp, time, X)
    t_burn = mp[4] / mp[6] if model == S.INTERCEPTOR else None
    crossed = 0
    for b in range(B):
        for j in range(M):
            r = rows[b, j]
            assert r[0, 0] == tl[b, j] and np.array_equal(r[0, 1:1 + N], X[b, N * j:N * j + N]), (model, b, j)
            stages = [(tl[b, j], tl[b, j + 1])]
            if t_burn is not None and tl[b, j] < t_burn < tl[b, j + 1]:
                stages = [(tl[b, j], t_burn), (t_burn, tl[b, j + 1])]
                crossed += 1
            assert nrows[b, j] == len(stages) * (S_ + 1), (model, b, j)
            k = 0
            for t0, tf in stages:
                t, dt = t0, (tf - t0) / S_
                for _ in range(S_ + 1):
                    assert r[k, 0] == t, (model, b, j, k)
                    t += dt
                    k += 1
        last = rows[b, M - 1, nrows[b, M - 1] - 1]
        # an interceptor row in chart 2 holds the other chart's coordinates; Move(t_end) converts back to chart 1
        if model != S.INTERCEPTOR or last[-1] == 1.0:
            end = vX[b, M]
            assert np.max(np.abs(last[1:1 + N] - end)) <= 1e-14 * np.max(np.abs(end)), (model, b)
    if model == S.INTERCEPTOR:
        assert crossed == B
    if model == S.GODDARD:
        # goddard::Trace's extra column is the switching function; the control is bang (|u| = 1) up to the first
        # switching time, singular up to the second, off after it (tests/testGoddard.cpp stage 4)
        Xr = rows[..., 1:1 + N]
        sf = mp[5] - mp[1] * Xr[..., 13] - mp[0] / Xr[..., 6] * np.sqrt(Xr[..., 10] ** 2 + Xr[..., 11] ** 2 + Xr[..., 12] ** 2)
        assert np.allclose(rows[..., -1], sf, rtol=1e-13, atol=1e-15)
        _, sw = timelines(spec, shape, mp, X)
        t, unorm = rows[..., 0], np.linalg.norm(rows[..., 1 + N:4 + N], axis=-1)
        for b in range(B):
            assert np.allclose(unorm[b][t[b] <= sw[b, 0]], 1.0, rtol=1e-12)
            assert np.all(unorm[b][t[b] > sw[b, 1]] == 0.0)
            mid = unorm[b][(t[b] > sw[b, 0]) & (t[b] <= sw[b, 1])]
            assert mid.size > 0 and np.all(mid <= 1.0 + 1e-12)


def test_controls_and_hamiltonian_vs_oracle():
    """Every row of the double integrator against the oracle's control and H, tolerances of test_gpu_trace.py."""
    spec, shape, X, mp, time = _move_case(S.DI)
    M, N, nc = spec["M"], 12, 3
    rows, nrows = engine().solution_trace_batch(shape, mp, time, X)
    p = oracle_problem(spec, mp)
    for b in range(X.shape[0]):
        p.timeline(X[b])
        for j in range(M):
            for r in rows[b, j, :nrows[b, j]]:
                u = np.asarray(p.control(r[0], r[1:1 + N]))[:nc]
                H = p.hamiltonian(r[0], r[1:1 + N])
                assert np.allclose(r[1 + N:1 + N + nc], u, rtol=1e-11, atol=1e-13), (b, j)
                assert abs(r[1 + N + nc] - H) <= 1e-11 * max(1.0, abs(H), np.max(np.abs(r[1:1 + N]))), (b, j)


def _written(rows, nrows):
    return [rows[b, j, :nrows[b, j]] for b in range(nrows.shape[0]) for j in range(nrows.shape[1])]


def test_independent_of_batch():
    """Problem b alone gives the rows it has inside a batch of 10^4, wherever it sits."""
    spec, shape, X, mp, time = _move_case(S.GODDARD, B=16)
    eng = engine()
    reps = 10000 // 16
    big_r, big_n = eng.solution_trace_batch(shape, mp, np.tile(time, (reps, 1)), np.tile(X, (reps, 1)))
    for b in range(16):
        r1, n1 = eng.solution_trace_batch(shape, mp, time[b:b + 1], X[b:b + 1])
        for pos in (b, b + 16 * 311, b + 16 * (reps - 1)):
            assert np.array_equal(big_n[pos], n1[0]), (b, pos)
            for w, g in zip(_written(r1, n1), _written(big_r[pos:pos + 1], big_n[pos:pos + 1])):
                assert np.array_equal(w, g), (b, pos)


def test_host_and_device_modes():
    import torch
    spec, shape, X, mp, time = _move_case(S.INTERCEPTOR, B=64)
    eng = engine()
    rows_h, n_h = eng.solution_trace_batch(shape, mp, time, X)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    rows_d, n_d = eng.solution_trace_batch(shape, dev(np.tile(mp, (64, 1))), dev(time), dev(X))
    assert torch.is_tensor(rows_d) and rows_d.is_cuda and n_d.dtype == torch.int32
    rows_d, n_d = rows_d.cpu().numpy(), n_d.cpu().numpy()
    assert np.array_equal(n_d, n_h)
    for w, g in zip(_written(rows_h, n_h), _written(rows_d, n_d)):
        assert np.array_equal(w, g)


def test_dopri5_shape_traces_with_rk4():
    """An adaptive shape is traced with the fixed-step RK4 observer: the rows of the RK4 shape."""
    import socp_b200 as sb
    spec, shape, X, mp, time = _move_case(S.DI)
    adaptive = sb.make_shape(spec["model"], spec["M"], spec["mode_t"], spec["mode_X"], spec["steps"], ode_tol=1e-9)
    eng = engine()
    r1, n1 = eng.solution_trace_batch(shape, mp, time, X)
    r2, n2 = eng.solution_trace_batch(adaptive, mp, time, X)
    assert np.array_equal(n1, n2) and np.all(n1 == spec["steps"] + 1)
    for w, g in zip(_written(r1, n1), _written(r2, n2)):
        assert np.array_equal(w, g)


def test_edges():
    """B == 0 writes nothing; NULL arrays, a negative B and a bad shape are SOCP_ERR_ARG."""
    import socp_b200 as sb
    spec, shape, X, mp, time = _move_case(S.DI, B=2)
    eng = engine()
    L, h = eng._L, eng._h
    d = lambda a: ctypes.c_void_p(a.ctypes.data)
    mpb = np.ascontiguousarray(np.tile(mp, (2, 1)))
    R, W = L.socp_trace_max_rows(S.DI, spec["steps"]), L.socp_trace_width(S.DI)
    rows, nrows = np.full((2, spec["M"], R, W), 7.0), np.full((2, spec["M"]), 7, dtype=np.int32)
    sh = ctypes.byref(shape)
    args = [d(mpb), d(time), d(X), d(rows), d(nrows)]
    assert L.socp_solution_trace_batch(h, sh, 0, *args, 0) == 0
    assert np.all(rows == 7.0) and np.all(nrows == 7)
    for k in range(5):
        a = list(args)
        a[k] = None
        assert L.socp_solution_trace_batch(h, sh, 2, *a, 0) == -1, k
    assert L.socp_solution_trace_batch(h, sh, -1, *args, 0) == -1
    assert L.socp_solution_trace_batch(h, None, 2, *args, 0) == -1
    assert L.socp_solution_trace_batch(None, sh, 2, *args, 0) == -1
    for bad in ("model", "mode_t", "continuous_end", "integrator"):
        s2 = sb.make_shape(spec["model"], spec["M"], spec["mode_t"], spec["mode_X"], spec["steps"])
        if bad == "model":
            s2.model_id = 9
        elif bad == "mode_t":
            s2.mode_t[1] = 7
        elif bad == "continuous_end":
            s2.mode_t[0] = S.CONTINUOUS
        else:
            s2.integrator = 5
        assert L.socp_solution_trace_batch(h, ctypes.byref(s2), 2, *args, 0) == -1, bad
    assert np.all(rows == 7.0) and np.all(nrows == 7)


def test_rows_past_2_31_values():
    """Goddard, 1.7e6 problems: B*M*R*W = 2.24e9 doubles (18 GB) in device mode; problems at the far end match
    socp_trace_batch."""
    import torch
    spec, shape, X, mp, time = _move_case(S.GODDARD, B=16)
    B, M, N = 1_700_000, spec["M"], 14
    eng = engine()
    R, W = eng._L.socp_trace_max_rows(S.GODDARD, spec["steps"]), eng._L.socp_trace_width(S.GODDARD)
    assert B * M * R * W > 2 ** 31
    reps = B // 16 + 1
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    x_d = dev(X).repeat(reps, 1)[:B].contiguous()
    t_d = dev(time).repeat(reps, 1)[:B].contiguous()
    mp_d = dev(np.tile(mp, (B, 1)))
    rows_d, n_d = eng.solution_trace_batch(shape, mp_d, t_d, x_d)
    picks = [B - 1, B - 2, B - 17, B - 16 * 1000 - 5, 1_627_000]
    tl, sw = timelines(spec, shape, mp, X)
    for pos in picks:
        got, gn = rows_d[pos].cpu().numpy(), n_d[pos].cpu().numpy()
        b = pos % 16
        for j in range(M):
            want, wn = segment_rows(eng, S.GODDARD, mp, tl[b:b + 1], sw[b:b + 1], X[b:b + 1], j, N, spec["steps"])
            assert gn[j] == wn[0] and np.array_equal(got[j, :wn[0]], want[0, :wn[0]]), (pos, j)
    del rows_d, n_d, x_d, t_d, mp_d
    torch.cuda.empty_cache()


def test_batch_trace_demo(tmp_path):
    """The C++ mirror: shooting_batch::Trace(k) writes the text shooting::Trace writes for the same problem."""
    exe = os.path.join(BIN, "demo_goddard_trace")
    assert os.access(exe, os.X_OK), "run __graft_entry__.build() first"
    r = subprocess.run([exe, "64"], capture_output=True, text=True, timeout=1200, cwd=str(tmp_path))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "all traces identical: yes" in r.stdout, r.stdout
