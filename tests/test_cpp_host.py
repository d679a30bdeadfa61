"""The C++ host mirror (cpp/): SOCP's own `model` / `shooting` API on top of the C ABI.

CPU part: the mirror builds, the reference's own demo programs compile against it UNCHANGED (when the
reference tree is present), and the host-only closed-form costate guess (interceptor::InitAnalytical)
matches the unmodified reference.  GPU part: the demos run and reproduce the reference's results.
"""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import scenarios as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CPP = os.path.join(ROOT, "cpp")
BIN = os.path.join(CPP, "build", "bin")
REF_DEMOS = ["testDoubleIntegrator", "testDoubleIntegrator_WP", "testGoddard", "testCovid19", "testInterceptor",
             "testVtolUAV"]


@pytest.fixture(scope="module")
def built():
    from socp_b200 import build
    build.build()
    subprocess.check_call(["make", "-s", "-C", CPP])
    return True


def test_mirror_builds_and_links(built):
    for name in ("demo_double_integrator", "demo_goddard_batch"):
        assert os.access(os.path.join(BIN, name), os.X_OK)
    out = subprocess.run(["ldd", os.path.join(BIN, "demo_double_integrator")], capture_output=True, text=True).stdout
    assert "libsocp_host.so" in out and "libsocp_b200.so" in out and "not found" not in out
    # the only way the mirror computes: through the C ABI (no second implementation of the hot path)
    syms = subprocess.run(["nm", "-D", "--undefined-only", os.path.join(CPP, "build", "libsocp_host.so")],
                          capture_output=True, text=True).stdout
    for s in ("socp_create", "socp_solve_batch", "socp_traj_batch", "socp_trace_batch", "socp_point_batch",
              "socp_continuation_param_batch", "socp_continuation_boundary_batch"):
        assert s in syms, s


@pytest.mark.skipif(not os.path.isdir("/root/reference/tests"), reason="reference tree not present")
def test_reference_demos_compile_unchanged(built):
    """tests/test*.cpp of the reference, symlinked (never copied), compile against the mirror headers."""
    subprocess.check_call(["make", "-s", "-C", CPP, "refdemos"])
    for t in REF_DEMOS:
        assert os.access(os.path.join(BIN, "ref_" + t), os.X_OK), t
        src = os.path.join(CPP, "build", "ref", "tests", t + ".cpp")
        assert os.path.islink(src) and os.path.realpath(src).startswith("/root/reference/")
    # the include "../src/socp/shooting.hpp" of the demos resolved to the mirror, not to the reference
    out = subprocess.run(["g++", "-std=gnu++11", "-w", "-H", "-fsyntax-only",
                          os.path.join(CPP, "build", "ref", "tests", "testGoddard.cpp")], capture_output=True, text=True).stderr
    hdr = [l for l in out.splitlines() if l.strip(". ").endswith("shooting.hpp")]
    assert hdr and all("/cpp/" in l for l in hdr), hdr


def _close_to_reference(got, want):
    # the azimuth of the line of sight is an acos() next to 1 (interceptor.cpp:905-911): rounding
    # differences of the projected position are amplified to ~sqrt(ulp) in p_chi, p_L, p_l
    scale = np.max(np.abs(want))
    return np.all(np.abs(got - want) <= 1e-7 * np.abs(want) + 1e-12 * scale)


def test_init_analytical_matches_reference(built):
    """interceptor::InitAnalytical (interceptor.cpp:844-955) is host glue in both code bases.  Where the reference
    build is absent, the mirror is compared with the guess tests/golden/make_golden.py recorded from it (the
    initialisation problem of tests/testInterceptor.cpp: mu_gft = 0, tf = 10 s)."""
    from oracle import pyref
    L = ctypes.CDLL(os.path.join(CPP, "build", "libsocp_host.so"))
    L.socp_host_interceptor_init_analytical.argtypes = [ctypes.c_void_p, ctypes.c_double, ctypes.c_void_p,
                                                        ctypes.c_double, ctypes.c_void_p]
    if not pyref.available():
        import golden_util as G
        want = G.unhex(G.golden()["interceptor_costate_guess"])
        mp = np.array(S.DEFAULTS[S.INTERCEPTOR], dtype=np.float64)
        mp[13] = 0.0
        a = np.r_[S.INTERCEPTOR_INIT_XI, np.zeros(6)]
        b = np.r_[S.INTERCEPTOR_INIT_XF, np.zeros(6)]
        got = a.copy()
        L.socp_host_interceptor_init_analytical(mp.ctypes.data, 0.0, got.ctypes.data, 10.0, b.ctypes.data)
        assert np.array_equal(got[:6], a[:6])
        assert np.all(np.isfinite(want)) and _close_to_reference(got[6:], want), (got[6:], want)
        return
    rng = np.random.default_rng(5)
    cases = [(np.array(S.INTERCEPTOR_INIT_XI), np.array(S.INTERCEPTOR_INIT_XF))]
    for _ in range(6):
        amp = np.array([0.2, 0.2, 0.2, 0.2, 1e-4, 1e-4])      # keep the rendez-vous point within reach
        Xi = np.array(S.INTERCEPTOR_INIT_XI) * (1 + amp * rng.uniform(-1, 1, 6))
        Xf = np.array(S.INTERCEPTOR_INIT_XF) * (1 + amp * rng.uniform(-1, 1, 6))
        cases.append((Xi, Xf))
    for mu_gft in (0.0, 1.0):
        mp = np.array(S.DEFAULTS[S.INTERCEPTOR], dtype=np.float64)
        mp[13] = mu_gft
        ref = pyref.RefModel(S.INTERCEPTOR, model_order=0, step_nbr=0)
        ref.set("mu_gft", mu_gft)
        keep = [k for k in range(17) if k not in (11, 12)]        # r_2p, t_2p: never initialised by the reference's constructor
        assert np.allclose(ref.params()[keep], mp[keep])
        for Xi, Xf in cases:
            a = np.r_[Xi, np.zeros(6)]
            b = np.r_[Xf, np.zeros(6)]
            want_i, _ = ref.init_analytical(0.0, a.copy(), 20.0, b.copy())
            got = a.copy()
            bb = b.copy()
            L.socp_host_interceptor_init_analytical(mp.ctypes.data, 0.0, got.ctypes.data, 20.0, bb.ctypes.data)
            assert np.array_equal(got[:6], a[:6])
            assert np.all(np.isfinite(want_i[6:])), want_i
            assert _close_to_reference(got[6:], want_i[6:]), (got[6:], want_i[6:])


def _run(name, *args, cwd=None):
    r = subprocess.run([os.path.join(BIN, name)] + list(args), capture_output=True, text=True, timeout=600, cwd=cwd)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return r.stdout


@pytest.mark.gpu
def test_double_integrator_demo_matches_reference():
    """Three stages of tests/testDoubleIntegrator.cpp (solve, boundary continuation, parameter
    continuation) through the mirror classes; reference results with the forward-difference solver
    (SURVEY.md section 8c, `modelOrder = 0` row): nfev 82 / 25 / 151."""
    assert os.access(os.path.join(BIN, "demo_double_integrator"), os.X_OK), "run __graft_entry__.build() first"
    out = _run("demo_double_integrator")
    rows = re.findall(r"stage (\d) info (\d+) nfev (\d+) njev \d+ tf (\S+) p0 (.*)", out)
    assert len(rows) == 3, out
    want = [(82, 27.655974527562908, [-0.0056730204147606, -0.0085095306215938124]),
            (25, 30.80070288243714, [-0.0041067603843020425, -0.0082135207686335095]),
            (151, 25.900200641181858, [-0.0069067201709498496, -0.013813440341899698])]
    for (stage, info, nfev, tf, p0), (w_nfev, w_tf, w_p) in zip(rows, want):
        p = [float(v) for v in p0.split()]
        assert int(info) == 1 and int(nfev) == w_nfev, (stage, info, nfev)
        assert abs(float(tf) - w_tf) <= 1e-8 * w_tf
        assert abs(p[0] - w_p[0]) <= 1e-7 * abs(w_p[0]) and abs(p[1] - w_p[1]) <= 1e-7 * abs(w_p[1])


@pytest.mark.gpu
def test_double_integrator_demo_hybrj_matches_reference():
    """The same three stages with modelOrder = 1, as tests/testDoubleIntegrator.cpp runs them: analytic
    Jacobian + hybrj.  Reference (SURVEY.md section 8c): nfev/njev 30/4, 12/1, 125/2."""
    out = _run("demo_double_integrator", "1")
    rows = re.findall(r"stage (\d) info (\d+) nfev (\d+) njev (\d+) tf (\S+) p0", out)
    assert len(rows) == 3, out
    want = [(30, 4, 27.655974527562883), (12, 1, 30.800702882437143), (125, 2, 25.900200641161657)]
    for (stage, info, nfev, njev, tf), (w_nfev, w_njev, w_tf) in zip(rows, want):
        assert int(info) == 1 and (int(nfev), int(njev)) == (w_nfev, w_njev), (stage, info, nfev, njev)
        assert abs(float(tf) - w_tf) <= 1e-8 * w_tf


@pytest.mark.gpu
def test_goddard_batch_demo():
    out = _run("demo_goddard_batch", "128")
    assert "identical to the single solve: yes" in out, out
    m = re.search(r"batch 128 solved: (\d+) converged", out)
    assert m and int(m.group(1)) > 0
    # problem 0 is the reference's own Goddard stage 1 (golden: nfev 1184, tf = 0.21965083876703931; the
    # solve from the trivial guess is chaotic in the reference itself, so only success is asserted here)
    m = re.search(r"problem 0: info (\d+) nfev (\d+) tf (\S+)", out)
    assert m, out


@pytest.mark.gpu
@pytest.mark.skipif(not os.access(os.path.join(BIN, "ref_testDoubleIntegrator"), os.X_OK),
                    reason="reference demos not built (reference tree absent at build time)")
def test_reference_demo_binaries_run(tmp_path):
    """The reference's own demo mains, compiled unchanged against the mirror, run on the GPU engine and
    report success ("Algo returned 1").  They write traces to ../../trace/<model>/ relative to the cwd."""
    run = tmp_path / "bin" / "Release"
    run.mkdir(parents=True)
    for m in ("doubleIntegrator", "goddard", "covid19", "interceptor", "vtolUAV"):
        (tmp_path / "trace" / m).mkdir(parents=True)
    out = _run("ref_testDoubleIntegrator", cwd=str(run))
    assert out.count("Algo returned 1") >= 3, out
    trace = (tmp_path / "trace" / "doubleIntegrator" / "trace.dat").read_text().splitlines()
    assert len(trace) >= 31 and len(trace[0].split("\t")) == 1 + 12 + 3 + 1
    # tests/testGoddard.cpp: solve (KD = 0), continuation KD -> 310, continuation mu2 -> 0.2, re-meshed
    # solve with the true singular control: four "OK = 1"
    out = _run("ref_testGoddard", cwd=str(run))
    assert out.count("OK = 1") == 4, out
    trace = (tmp_path / "trace" / "goddard" / "trace.dat").read_text().splitlines()
    assert len(trace[0].split("\t")) == 1 + 14 + 3 + 1 + 1          # t, X, control, H, switching function
    # tests/testCovid19.cpp: solve + two continuations on the boundary data (M = 20, 1000 steps/segment)
    out = _run("ref_testCovid19", cwd=str(run))
    assert out.count("OK = 1") == 3, out
    # tests/testDoubleIntegrator_WP.cpp: two segments, free interior time, waypoint continuation
    out = _run("ref_testDoubleIntegrator_WP", cwd=str(run))
    assert "Algo returned 1" in out and "OK = 1" in out, out


@pytest.mark.gpu
@pytest.mark.skipif(not os.access(os.path.join(BIN, "ref_testInterceptor"), os.X_OK),
                    reason="reference demos not built (reference tree absent at build time)")
def test_reference_interceptor_and_vtol_demos_run(tmp_path):
    """tests/testInterceptor.cpp (analytic guess, mu_gft homotopy, three scenarios; S1 fails in the
    reference too, SURVEY.md section 8c) and tests/testVtolUAV.cpp (waypoint-by-waypoint path continuation
    through the obstacle field, M grows to 32) -- the demo mains of the reference, unchanged."""
    run = tmp_path / "bin" / "Release"
    run.mkdir(parents=True)
    for m in ("interceptor", "vtolUAV"):
        (tmp_path / "trace" / m).mkdir(parents=True)
    out = _run("ref_testInterceptor", cwd=str(run))
    assert out.count("OK = 1") >= 2, out                 # scenarios S2 and S3
    # the vtolUAV demo reads data/vtolUAV/{obstacles,waypoints} relative to the cwd
    import backends
    d = tmp_path / "data" / "vtolUAV"
    d.mkdir(parents=True)
    backends._obstacle_files(str(d))                      # writes d/obstacles and d/waypoints
    out = _run("ref_testVtolUAV", cwd=str(run))
    assert out.count("OK = 1") == 4, out


@pytest.mark.gpu
def test_goddard_batch_demo_over_every_visible_gpu():
    """shooting_batch(model, numMulti, batch, numDevice = 0): one host thread and one engine context per GPU,
    contiguous blocks of the batch (on a one-GPU box this is the single-device path through the same code)."""
    out = _run("demo_goddard_batch", "256", "0")
    assert "identical to the single solve: yes" in out, out
    m = re.search(r"batch of 256 problems on (\d+) GPU", out)
    assert m and int(m.group(1)) >= 1, out
    one = _run("demo_goddard_batch", "256", "1")
    # the same problems give the same answers whatever the number of devices
    assert re.search(r"batch 256 solved: (\d+)", out).group(1) == re.search(r"batch 256 solved: (\d+)", one).group(1)
    assert re.search(r"problem 0: .*", out).group(0) == re.search(r"problem 0: .*", one).group(0)
