#!/usr/bin/env python
"""bench.py -- headline benchmark of the batched shooting engine (BASELINE.json metric).

Default workload (BASELINE.json configs[1], SURVEY.md section 8d "C2"): the Goddard rocket problem with
free final time (tests/testGoddard.cpp:28-99: multiple shooting M=6, P=85 unknowns, 10 RK4 steps per
segment, xtol 1e-6, KD=0, mu2=1), a batch of 1e5 perturbed initial conditions per GPU, trivial costate
guess 0.1.  One "step" = one batched solve of the whole batch (socp_solve_batch).

  python bench.py --gpus N --steps K --warmup W             (torchrun for N > 1, one rank per GPU)
  python bench.py --impl reference ...                      (the reference's CPU solver, all cores)
  python bench.py --scaling strong --global-batch 1000000   (fixed total work split over the ranks)
  python bench.py --workload goddard_warm|interceptor|covid19|vtol_rk45   (the other BASELINE configs)
  python bench.py --dump-outputs DIR ...                    (what the last timed step returned, as DIR/<name>.npy)

Prints ONE JSON line (rank 0).  `value` = shooting solves per second with the inputs resident in HBM;
`e2e` = the same through the public API with pinned HOST buffers (H2D + D2H inside the timed region);
`roofline` = the kernel with the largest share of the step, every kernel of the round under
`roofline.kernels` (measured in a separate profiled pass, not inside the `value` region);
`cpu_baseline` = the unmodified reference (oracle/_ref) timed on the host cores on a bounded sample;
`parity` = per-problem comparison of the GPU results with that reference on the same sample;
`stage2` = SURVEY C2 stage 2, the well-conditioned part of the Goddard pipeline: warm-started solves
(the reference's converged x* + each problem's perturbed boundary data) and the KD 0 -> 310 continuation
on the converged batch, each with its own throughput and parity object.
oracle/ is used here only as the CPU baseline / parity checker / reference arm.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# nominal flops per RK4 step, SURVEY.md 8(d) / BASELINE.md section 3 (as written in the reference, no CSE credit)
FLOPS_PER_RK4_STEP = {"goddard": 1100.0, "interceptor": 1704.0, "covid19": 256.0, "vtol": 2736.0, "di": 264.0}
METRIC = "shooting solves/sec (Goddard free-tf, M=6, P=85; RK4 steps/sec and % of FP64 roofline alongside)"
TRAFFIC_FILE = os.path.join(ROOT, "profiles", "r2_traffic.json")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="goddard", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="problems per GPU (0 = the workload's default)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--global-batch", type=int, default=0, help="--scaling strong: total problems over all ranks")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--parity-sample", type=int, default=1024, help="problems compared with oracle/_ref (rank 0, N = 1)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="problems in the CPU baseline sample (0 = the parity sample)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip cpu_baseline, parity and stage2 parity")
    ap.add_argument("--no-stage2", action="store_true")
    ap.add_argument("--no-profile-pass", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float64, at most 64 MB in all)")
    return ap.parse_args()


# ---------------------------------------------------------------------------------------------
# workload construction (host side, untimed)
# ---------------------------------------------------------------------------------------------
class Workload:
    """Arrays of one batch as the C ABI takes them + what the CPU checkers need to rebuild problem k."""

    def __init__(self, name, model, shape, mp, time_, Xb, x0, xtol, steps, flops_key, label, mode_t, mode_X, M,
                 kind="solve", cont=None, ode_tol=0.0):
        self.name, self.model, self.shape = name, model, shape
        self.mp, self.time, self.Xb, self.x0 = mp, time_, Xb, x0
        self.xtol, self.steps, self.flops_key, self.label = xtol, steps, flops_key, label
        self.mode_t, self.mode_X, self.M = mode_t, mode_X, M
        # kind: "solve" (one root solve per problem), "cont_boundary" (homotopy on the boundary data: cont = dict(step,
        # time_des[B][M+1], Xb_des[B][(M+1) dim])), "cont_param" (homotopy on a model parameter: cont = dict(step, pname, goal[B]))
        self.kind, self.cont, self.ode_tol = kind, cont, ode_tol
        self.unit = "solves/s" if kind == "solve" else "homotopies/s"

    @property
    def B(self):
        return self.x0.shape[0]

    @property
    def P(self):
        return self.x0.shape[1]

    def spec(self, k, x0=None, mparams=None):
        """Problem k as a scenario spec for the CPU checkers (tests/scenarios.py)."""
        import scenarios as S
        n = S.DIM[self.model]
        sp = S.make_spec(self.model, self.M, self.mode_t, self.mode_X, self.time[k], self.Xb[k].reshape(self.M + 1, n),
                         self.x0[k] if x0 is None else x0, self.xtol,
                         mparams=self.mp[k] if mparams is None else mparams, steps=self.steps,
                         name="%s_%d" % (self.name, k))
        if self.ode_tol > 0:
            sp["ode_tol"] = self.ode_tol
        if self.kind == "cont_boundary":
            sp["cont"] = dict(step=self.cont["step"], timed=[float(v) for v in self.cont["time_des"][k]],
                              Xd=[[float(v) for v in r] for r in self.cont["Xb_des"][k].reshape(self.M + 1, n)])
        elif self.kind == "cont_param":
            sp["cont"] = dict(step=self.cont["step"], pname=self.cont["pname"], goal=float(self.cont["goal"][k]))
        return sp


def goddard_workload(eng, B, seed):
    """Config C2 arrays for B problems: (shape, mparams, time, Xb, x0).  The initial guess follows
    shooting::InitShooting (shooting.cpp:202-245): interior node states by integrating from the
    initial state with the constructor's KD=310 (tests/testGoddard.cpp sets KD=0 afterwards)."""
    import socp_b200 as sb
    import scenarios as S
    M, n, N = 6, 7, 14
    Xi, xf0 = S.goddard_batch_inputs(B, seed=seed)
    mode_t, mode_X = sb.default_modes(sb.GODDARD, M, sb.FREE, S.GODDARD_MODE_XF)
    shape = sb.make_shape(sb.GODDARD, M, mode_t, mode_X, 10)
    mp_init = np.array(S.DEFAULTS[S.GODDARD]); mp_init[6] = 1.0          # mu2 = 1, KD = 310
    ti, tf = 0.0, 0.1
    time_ = np.tile(np.array([ti + i * (tf - ti) / M for i in range(M + 1)]), (B, 1))
    x0 = np.zeros((B, N * M + 1))
    x0[:, :N] = Xi
    for i in range(1, M):
        x0[:, N * i:N * (i + 1)] = eng.traj_batch(sb.GODDARD, mp_init, ti, Xi, time_[:, i], 10)
    x0[:, N * M] = tf
    mp = np.tile(mp_init, (B, 1)); mp[:, 2] = 0.0                        # KD = 0
    Xb = np.zeros((B, M + 1, n))
    Xb[:, 0, :] = Xi[:, :n]
    Xb[:, M, 0] = xf0
    return shape, mp, time_, Xb.reshape(B, -1), x0


def spec_of(k, mp, time_, Xb, x0):
    """Problem k of the Goddard batch as a scenario spec for the CPU checkers."""
    import scenarios as S
    mode_t, mode_X = S.default_modes(S.GODDARD, 6, S.FREE, S.GODDARD_MODE_XF)
    return S.make_spec(S.GODDARD, 6, mode_t, mode_X, time_[k], Xb[k].reshape(7, 7), x0[k], 1e-6,
                       mparams=mp[k], steps=10, name="goddard_batch_%d" % k)


def reference_xstar():
    """The reference's converged unknowns of the UNPERTURBED stage-1 problem (tests/testGoddard.cpp:94-99,
    info 1 after 1184 evaluations), recorded from oracle/_ref as hex floats in tests/golden/golden.json."""
    import golden_util as G
    e = G.by_name("solve", "goddard_stage1")
    assert e["info"] == 1
    return np.asarray(G.unhex(e["x"]), dtype=np.float64)


def wl_goddard(eng, B, seed):
    import scenarios as S
    shape, mp, time_, Xb, x0 = goddard_workload(eng, B, seed)
    mode_t, mode_X = S.default_modes(S.GODDARD, 6, S.FREE, S.GODDARD_MODE_XF)
    return Workload("goddard", S.GODDARD, shape, mp, time_, Xb, x0, 1e-6, 10, "goddard",
                    "goddard_free_tf_M6_P85_batch (BASELINE configs[1], SURVEY C2 stage 1: trivial costate guess)",
                    mode_t, mode_X, 6)


def wl_goddard_warm(eng, B, seed):
    """SURVEY C2 stage 2, first half: the same perturbed problems, each started from the reference's
    converged x* of the unperturbed problem (a warm start as SolveShooting does between two SolveOCP calls,
    shooting.cpp:568-595).  Well conditioned: (info, nfev) are reproducible problem for problem."""
    w = wl_goddard(eng, B, seed)
    w.name = "goddard_warm"
    w.label = "goddard_warm_start_M6_P85_batch (SURVEY C2 stage 2: reference x* + perturbed boundary data)"
    w.x0 = np.tile(reference_xstar(), (B, 1))
    return w


def _golden_spec(kind, name):
    import golden_util as G
    e = G.by_name(kind, name)
    return e, G.spec_from_hex(e["spec"])


def wl_interceptor(eng, B, seed):
    """BASELINE configs[2] / SURVEY C3: interceptor guidance shooting (P = 13).  Every problem is the boundary
    continuation of tests/testInterceptor.cpp:137-139 (step 0.1: eleven solves) from the solved initialisation
    problem (`initState`, :152-199, mu_gft 0 -> 1; shared by all problems, recorded from oracle/_ref in
    tests/golden/golden.json) to scenario S3 (:84-97) with a perturbed target: altitude +-500 m, heading +-0.05 rad,
    latitude / longitude +-2 km."""
    import socp_b200 as sb
    import scenarios as S
    import golden_util as G
    e, spec = _golden_spec("cont_boundary", "interceptor_S3")
    timed, Xd0 = np.asarray(G.unhex(e["timed"])), np.asarray(G.unhex(e["Xd"]))
    rng = np.random.default_rng(seed)
    Xd = np.tile(Xd0.reshape(1, 2, 6), (B, 1, 1))
    Xd[:, 1, 0] += rng.uniform(-500, 500, B)
    Xd[:, 1, 3] += rng.uniform(-0.05, 0.05, B)
    Xd[:, 1, 4] += rng.uniform(-2000, 2000, B) / S.R_EARTH
    Xd[:, 1, 5] += rng.uniform(-2000, 2000, B) / S.R_EARTH
    shape = sb.make_shape(sb.INTERCEPTOR, 1, spec["mode_t"], spec["mode_X"], spec["steps"])
    return Workload("interceptor", S.INTERCEPTOR, shape, np.tile(np.array(spec["mparams"]), (B, 1)),
                    np.tile(np.array(spec["time"]), (B, 1)), np.tile(np.array(spec["Xb"]).reshape(1, -1), (B, 1)),
                    np.tile(np.array(spec["x0"]), (B, 1)), spec["xtol"], spec["steps"], "interceptor",
                    "interceptor_S3_boundary_continuation_P13_batch (BASELINE configs[2], SURVEY C3: 11 solves per problem)",
                    spec["mode_t"], spec["mode_X"], 1, kind="cont_boundary",
                    cont=dict(step=0.1, time_des=np.tile(timed, (B, 1)), Xb_des=Xd.reshape(B, -1)))


def wl_covid19(eng, B, seed):
    """BASELINE configs[4] / SURVEY C5: Covid-19 SEIR control (M = 20 segments x 1000 RK4 steps, P = 160), a
    continuation sweep over the cost weight of the ICU constraint: every problem starts from the reference's
    solution of tests/testCovid19.cpp:42-93 (muI = 1; recorded from oracle/_ref) and runs the parameter homotopy
    of shooting.cpp:695-778 on muI to its own goal, log-uniform in [0.1, 10], step 0.5."""
    import socp_b200 as sb
    import scenarios as S
    import golden_util as G
    e, spec = _golden_spec("solve", "covid_stage1")
    assert e["info"] == 1
    xs = np.asarray(G.unhex(e["x"]))
    rng = np.random.default_rng(seed)
    goal = np.exp(rng.uniform(np.log(0.1), np.log(10.0), B))
    shape = sb.make_shape(sb.COVID19, 20, spec["mode_t"], spec["mode_X"], spec["steps"])
    return Workload("covid19", S.COVID19, shape, np.tile(np.array(spec["mparams"]), (B, 1)),
                    np.tile(np.array(spec["time"]), (B, 1)), np.tile(np.array(spec["Xb"]).reshape(1, -1), (B, 1)),
                    np.tile(xs, (B, 1)), spec["xtol"], spec["steps"], "covid19",
                    "covid19_muI_continuation_sweep_M20_P160_batch (BASELINE configs[4], SURVEY C5)",
                    spec["mode_t"], spec["mode_X"], 20, kind="cont_param", cont=dict(step=0.5, pname="muI", goal=goal))


def wl_vtol_rk45(eng, B, seed):
    """BASELINE configs[3] / SURVEY C4: vtolUAV with the obstacle map of data/vtolUAV, adaptive Dormand-Prince
    segments (the reference's -D_USE_BOOST build: xtol 1e-4, odeIntTol 1e-5, tests/testVtolUAV.cpp:65-66): the first
    leg of the waypoint path (:163-214, WP0 -> WP1, free final time) with the start point jittered by +-0.5 m."""
    import socp_b200 as sb
    import scenarios as S
    o = S.VTOL_OBSTACLES
    if eng is not None:
        eng.set_obstacles(o["type"], o["pos"], o["rad"])
    v = S.vtol_first_problem()
    rng = np.random.default_rng(seed)
    jit = rng.uniform(-0.5, 0.5, (B, 3))
    Xb = np.tile(np.array(v["Xb"]).reshape(1, -1), (B, 1))
    x0 = np.tile(np.array(v["x0"]), (B, 1))
    Xb[:, 0:3] += jit
    x0[:, 0:3] += jit
    shape = sb.make_shape(sb.VTOL_UAV, 1, v["mode_t"], v["mode_X"], v["steps"], ode_tol=1e-5)
    return Workload("vtol_rk45", S.VTOL, shape, np.tile(np.array(v["mparams"]), (B, 1)), np.tile(np.array(v["time"]), (B, 1)),
                    Xb, x0, v["xtol"], v["steps"], "vtol",
                    "vtolUAV_first_leg_dopri5_P13_batch (BASELINE configs[3], SURVEY C4: adaptive RK45, odeIntTol 1e-5)",
                    v["mode_t"], v["mode_X"], 1, ode_tol=1e-5)


WORKLOADS = {"goddard": (wl_goddard, 100000), "goddard_warm": (wl_goddard_warm, 100000),
             "interceptor": (wl_interceptor, 1000000), "covid19": (wl_covid19, 4096), "vtol_rk45": (wl_vtol_rk45, 1000000)}


# ---------------------------------------------------------------------------------------------
# CPU reference (oracle/_ref = unmodified reference sources; falls back to the C port)
# ---------------------------------------------------------------------------------------------
def _cpu_backend():
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle import pyref
    import backends
    return backends.RefBackend() if pyref.available() else backends.OracleBackend()


def _cpu_worker(job):
    """job = (kind, payload): solve / continuation / ensemble for a chunk of specs on one core."""
    kind, specs, extra = job
    be = _cpu_backend()
    out = []
    for s in specs:
        if kind == "run":
            # whatever the workload's unit of work is; (info, nfev or nfev_total, x, solver calls)
            if s.get("ode_tol"):
                # adaptive Dormand-Prince: the reference needs Boost.Odeint for it (absent): the C port stands in
                import backends
                p = backends.OracleBackend().problem(s)
                p.p.integrator, p.p.ode_tol = 1, s["ode_tol"]
                q = p.solve(s["x0"], xtol=s["xtol"])
                out.append((int(q["info"]), int(q["nfev"]), np.asarray(q["x"], dtype=np.float64), 1))
            elif "cont" in s and "timed" in s["cont"]:
                c = s["cont"]
                r = be.continuation_boundary(s, c["step"], np.asarray(c["timed"]), np.asarray(c["Xd"]))
                out.append((int(r["info"]), int(r["nfev_total"]), np.asarray(r["x"], dtype=np.float64), int(r["solver_calls"])))
            elif "cont" in s:
                c = s["cont"]
                r = be.continuation_param(s, c["step"], c["pname"], c["goal"])
                out.append((int(r["info"]), int(r["nfev_total"]), np.asarray(r["x"], dtype=np.float64), int(r["solver_calls"])))
            else:
                r = be.solve(s)
                out.append((int(r["info"]), int(r["nfev"]), np.asarray(r["x"], dtype=np.float64), 1))
        elif kind == "solve":
            r = be.solve(s)
            out.append((int(r["info"]), int(r["nfev"]), np.asarray(r["x"], dtype=np.float64)))
        elif kind == "cont_param":
            r = be.continuation_param(s, extra["step"], extra["pname"], extra["goal"])
            out.append((int(r["info"]), int(r["solver_calls"]), int(r["nfev_total"]), np.asarray(r["x"], dtype=np.float64)))
        elif kind == "ensemble":
            # the C port with its conditioning probe: every RHS evaluation moved by +-2 ulp
            import backends
            ora = backends.OracleBackend()
            runs = []
            for seed in range(extra["runs"]):
                p = ora.problem(s)
                p.p.noise_ulps = 0.0 if seed == 0 else 2.0
                p.p.noise_state = seed
                q = p.solve(s["x0"], xtol=s["xtol"])
                runs.append((int(q["info"]), int(q["nfev"])))
            out.append(runs)
    return out


class CpuPool:
    """One process per host core, each with its own copy of the reference library."""

    def __init__(self, cores=None):
        import multiprocessing as mp
        self.cores = cores or len(os.sched_getaffinity(0))
        self.pool = mp.get_context("spawn").Pool(self.cores)
        from oracle import pyref
        self.kind = "reference" if pyref.available() else "port"

    def run(self, kind, specs, extra=None):
        chunks = [(kind, specs[i::self.cores], extra) for i in range(self.cores)]
        chunks = [c for c in chunks if c[1]]
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_worker, chunks)
        dt = time.perf_counter() - t0
        flat = [None] * len(specs)
        for i, c in enumerate(res):
            for j, r in enumerate(c):
                flat[i + j * self.cores] = r
        return dt, flat

    def solve(self, specs):
        dt, res = self.run("solve", specs)
        return dt, res

    def work(self, specs):
        """One unit of work of the workload per spec (a solve or a whole homotopy): [(info, nfev, x, solver calls)]."""
        return self.run("run", specs)

    def close(self):
        self.pool.close()
        self.pool.join()


def parity_solve(gpu_info, gpu_nfev, gpu_x, ref, xtol):
    """Per-problem comparison of GPU results with the reference on the same problems.
    ref = [(info, nfev, x)].  The reference keeps its guess when info != 1 (shooting.cpp:588), so unknowns
    are compared where both report success."""
    n = len(ref)
    r_info = np.array([r[0] for r in ref]); r_nfev = np.array([r[1] for r in ref])
    g_info = np.asarray(gpu_info[:n]); g_nfev = np.asarray(gpu_nfev[:n])
    same_info = g_info == r_info
    same_both = same_info & (g_nfev == r_nfev)
    both_ok = (g_info == 1) & (r_info == 1)
    rel = np.array([np.linalg.norm(gpu_x[k] - ref[k][2]) / np.linalg.norm(ref[k][2]) for k in range(n) if both_ok[k]])
    pg, pr = float((g_info == 1).mean()), float((r_info == 1).mean())
    pooled = 0.5 * (pg + pr)
    z = (pg - pr) / np.sqrt(max(2 * pooled * (1 - pooled) / n, 1e-300))
    return {
        "sample": n, "checker": "oracle/_ref (unmodified reference + clean-room MINPACK)",
        "identical_info": float(same_info.mean()), "identical_info_nfev": float(same_both.mean()),
        "gpu_converged": pg, "ref_converged": pr, "converged_rate_z": float(z),
        "both_converged": int(both_ok.sum()),
        "x_within_xtol": float((rel <= xtol).mean()) if rel.size else None,
        "x_rel_err_max": float(rel.max()) if rel.size else None,
        "x_rel_err_median": float(np.median(rel)) if rel.size else None,
        "mean_nfev_gpu": float(g_nfev.mean()), "mean_nfev_ref": float(r_nfev.mean()),
        "max_abs_nfev_diff": int(np.abs(g_nfev - r_nfev).max()),
    }


def parity_ensemble(gpu_info, gpu_nfev, ref, runs):
    """Trivial-guess workload: the reference's own outcome is not reproducible under a +-2-ulp change of the
    arithmetic (DESIGN.md section 3), so membership in the outcome ensemble of the C port with its
    conditioning probe is reported, for the GPU and -- as calibration -- for the reference itself."""
    n = len(runs)
    def member(info, nfev, ens):
        infos = {e[0] for e in ens}
        nf = [e[1] for e in ens]
        return info in infos and 0.9 * min(nf) <= nfev <= 1.1 * max(nf)
    stable = [len(set(e)) == 1 for e in runs]
    g = [member(int(gpu_info[k]), int(gpu_nfev[k]), runs[k]) for k in range(n)]
    r = [member(ref[k][0], ref[k][1], runs[k]) for k in range(n)]
    return {"sample": n, "runs_per_problem": len(runs[0]), "probe": "+-2 ulp on every RHS evaluation (oracle port)",
            "reference_stable_fraction": float(np.mean(stable)),
            "gpu_in_ensemble": float(np.mean(g)), "reference_in_ensemble": float(np.mean(r)),
            "membership": "info in the ensemble's info set and nfev within [0.9 min, 1.1 max] of it"}


# ---------------------------------------------------------------------------------------------
def hbm_peak_gbs():
    """Measured copy bandwidth of this pool's B200s (driver-written MEASURED_PEAKS.json), else the
    fallback stated in B200_PROFILING.md."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md; MEASURED_PEAKS.json absent)"


def source_digest():
    """Digest of the CUDA sources: ties the ncu traffic record to the build it was captured from."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "socp_b200", "csrc")
    for f in sorted(os.listdir(d)):
        with open(os.path.join(d, f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def ncu_traffic(workload="goddard", P=85):
    """DRAM bytes per unit of work of each solver kernel, extracted by tools/summarize_r2.py from the committed
    `ncu --set full` captures (profiles/r2_*_raw.csv).  Only used when it was captured from the sources being run
    (digest match) on the workload being run (the bytes per Broyden iteration or per factorisation scale with P^2);
    otherwise traffic is reported as null."""
    try:
        with open(TRAFFIC_FILE) as f:
            t = json.load(f)
    except Exception:
        return {}, "no ncu capture on record (profiles/r2_traffic.json absent)"
    if t.get("source_digest") != source_digest():
        return {}, "ncu capture on record is from other sources (digest %s, running %s)" % (t.get("source_digest"), source_digest())
    if t.get("P", 85) != P or not workload.startswith(t.get("workload", "goddard")):
        return {}, "ncu capture on record is of the %s workload (P = %d), not of this one" % (t.get("workload", "goddard"), t.get("P", 85))
    return t.get("kernels", {}), "profiles/r2_traffic.json (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [v.strip() for v in out.strip().split(",")]
                if len(f) >= 7:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(s[3 + k].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]),
                "power_w_max": max(float(s[2]) for s in self.samples), "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
def run_reference(args, rank):
    """The reference's own CPU implementation (oracle/_ref) on the host cores, same workload."""
    if rank != 0:
        return
    import scenarios as S
    from backends import OracleBackend
    pool = CpuPool()
    per_step = args.cpu_sample or 8 * pool.cores
    n = per_step * (args.steps + args.warmup)
    batch = args.batch or WORKLOADS[args.workload][1]
    # build the same problems as the GPU arm (same seed); the guess integration runs on the CPU port
    if args.workload in ("goddard", "goddard_warm"):
        ora = OracleBackend()
        Xi, xf0 = S.goddard_batch_inputs(batch, seed=20260002)
        xstar = reference_xstar() if args.workload == "goddard_warm" else None
        specs = []
        for k in range(n):
            kk = k % batch
            s = S.goddard_problem(lambda mp, a, b, c: ora.traj(S.GODDARD, mp, a, b, c, 10), Xi=Xi[kk], xf0=xf0[kk])
            if xstar is not None:
                s["x0"] = [float(v) for v in xstar]
            specs.append(s)
        unit, steps_per_nfev = "solves/s", 60.0
    else:
        w = WORKLOADS[args.workload][0](None, min(n, batch), 20260002)
        specs = [w.spec(k % w.B) for k in range(n)]
        unit, steps_per_nfev = w.unit, float(w.M * w.steps)
    for wu in range(args.warmup):
        pool.work(specs[wu * per_step:(wu + 1) * per_step])
    t_total, res = 0.0, []
    for st in range(args.steps):
        lo = (args.warmup + st) * per_step
        dt, r = pool.work(specs[lo:lo + per_step])
        t_total += dt
        res += r
    pool.close()
    value = per_step * args.steps / t_total
    nfev = sum(r[1] for r in res)
    line = {
        "impl": "reference", "metric": METRIC if args.workload.startswith("goddard") else "shooting %s (%s)" % (unit.replace("/s", "/sec"), WORKLOAD_LABELS[args.workload]),
        "value": value, "unit": unit, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD_LABELS.get(args.workload, args.workload), "batch_per_gpu": batch,
                   "sample_per_step": per_step},
        "rk4_steps_per_s": nfev * steps_per_nfev / t_total,
        "converged_fraction": sum(1 for r in res if r[0] == 1) / len(res),
        "cpu_baseline": {"value": value, "unit": unit, "cores": pool.cores,
                         "kind": "port" if args.workload == "vtol_rk45" else pool.kind,
                         "sample": "%d problems of the batch per step, one process per core" % per_step},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# the CPU side of the heavier workloads is bounded to ~10-30 s of host work
PARITY_CAP = {"covid19": 32, "interceptor": 1024, "vtol_rk45": 1024}

WORKLOAD_LABELS = {
    "interceptor": "interceptor_S3_boundary_continuation_P13_batch (configs[2])",
    "covid19": "covid19_muI_continuation_sweep_M20_P160_batch (configs[4])",
    "vtol_rk45": "vtolUAV_first_leg_dopri5_P13_batch (configs[3])",
    "goddard": "goddard_free_tf_M6_P85_batch (configs[1])",
    "goddard_warm": "goddard_warm_start_M6_P85_batch (SURVEY C2 stage 2)",
}


# ---------------------------------------------------------------------------------------------
def la_flops_per_iteration(P):
    """Nominal linear-algebra flops of one Powell-hybrid (Broyden) iteration, MINPACK as written: Q^T f 2P^2,
    two R v products 2P^2, r1updt two Givens sweeps over the packed factor 6P^2, r1mpyq 2(P-1) rotations on
    P rows of Q 12P^2, dogleg (back substitution, gradient, R g) 3P^2."""
    return 25.0 * P * P


def device_arrays(torch, dev, w):
    def dv(a):
        return torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    d = dict(mp=dv(w.mp), time=dv(w.time), Xb=dv(w.Xb), x0=dv(w.x0))
    d["x"] = torch.empty_like(d["x0"])
    d["info"] = torch.empty(w.B, dtype=torch.int32, device=dev)
    d["nfev"] = torch.empty(w.B, dtype=torch.int32, device=dev)
    d["fnorm"] = torch.empty(w.B, dtype=torch.float64, device=dev)
    if w.kind != "solve":
        d["calls"] = torch.empty((w.B, 2), dtype=torch.int32, device=dev)
    if w.kind == "cont_boundary":
        d["time_des"], d["Xb_des"] = dv(w.cont["time_des"]), dv(w.cont["Xb_des"])
    if w.kind == "cont_param":
        d["goal"], d["mpw"] = dv(w.cont["goal"]), torch.empty_like(d["mp"])
    return d


def unit_of_work(eng, w, a, x, mp=None, info=None, nfev=None, fnorm=None, calls=None):
    """One unit of work of the workload for every problem through the public API: a root solve, or a whole
    homotopy.  `a` holds host (numpy) or device (torch) arrays; x is updated in place."""
    import scenarios as S
    if w.kind == "solve":
        return eng.solve_batch(w.shape, a["mp"], a["time"], a["Xb"], x, xtol=w.xtol, maxfev=10000, info=info, nfev=nfev, fnorm=fnorm)
    if w.kind == "cont_boundary":
        return eng.continuation_boundary_batch(w.shape, a["mp"], a["time"], a["Xb"], a["time_des"], a["Xb_des"], x, w.cont["step"],
                                               xtol=w.xtol, info=info, calls=calls)
    return eng.continuation_param_batch(w.shape, mp, a["time"], a["Xb"], x, w.cont["step"], S.pidx(w.model, w.cont["pname"]),
                                        a["goal"], xtol=w.xtol, info=info, calls=calls)


def timed_solves(eng, torch, dist, world, dev, w, d, steps, warmup, gather):
    """`warmup` untimed + `steps` timed units of work for the whole batch, device resident; returns ms for the timed steps."""
    def step():
        d["x"].copy_(d["x0"])
        if w.kind == "cont_param":
            d["mpw"].copy_(d["mp"])                      # the homotopy rewrites its parameter in place
        unit_of_work(eng, w, d, d["x"], mp=d.get("mpw"), info=d["info"], nfev=d["nfev"], fnorm=d["fnorm"], calls=d.get("calls"))
        if w.kind != "solve":
            d["nfev"].copy_(d["calls"][:, 1])
        if gather and world > 1:
            # the only exchange of the path: gather converged unknowns + status over NVLink
            from socp_b200 import sharding
            sharding.gather_results(d["x"], d["info"], d["nfev"])

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), step


DUMP_BYTES = 64 * 10 ** 6          # --dump-outputs writes at most this much


def step_outputs(w, d):
    """The arrays a caller of the timed path receives after one unit of work (device tensors, one row per problem):
    unknowns and status, |F| of a solve, the solver-call counts of a homotopy and the parameter block it rewrites."""
    out = {"x": d["x"], "info": d["info"]}
    if w.kind == "solve":
        out.update(nfev=d["nfev"], fnorm=d["fnorm"])
    else:
        out["calls"] = d["calls"]
    if w.kind == "cont_param":
        out["mparams"] = d["mpw"]
    return out


def dump_outputs(torch, outputs, path):
    """Write every output as <path>/<name>.npy in float64.  Where all of them together would exceed DUMP_BYTES, the
    same fixed, seeded sample of problems is taken from each, and its row indices are written as sample_rows.npy."""
    os.makedirs(path, exist_ok=True)
    B = outputs["x"].shape[0]
    if B == 0:                      # --scaling strong with fewer problems than ranks: this rank's block is empty
        return 0
    row_bytes = sum(8 * t.numel() // B for t in outputs.values())
    n = min(B, (DUMP_BYTES - 4096) // (row_bytes + 8))         # 4 KB for the .npy headers
    idx = None
    if n < B:
        rows = np.sort(np.random.default_rng(0).choice(B, n, replace=False))
        np.save(os.path.join(path, "sample_rows.npy"), rows.astype(np.float64))
        idx = torch.from_numpy(rows).to(outputs["x"].device)
    for name, t in outputs.items():
        if idx is not None:
            t = t.index_select(0, idx)
        np.save(os.path.join(path, name + ".npy"), t.to(torch.float64).cpu().numpy())
    return n


def e2e_solves(eng, torch, dist, world, dev, w, steps):
    """The same work through the C ABI with HOST buffers (mem = SOCP_HOST): pinned host memory, H2D and D2H inside the
    timed region (wall clock around the calls, max over ranks)."""
    src = dict(mp=w.mp, time=w.time, Xb=w.Xb, x0=w.x0)
    if w.kind == "cont_boundary":
        src.update(time_des=w.cont["time_des"], Xb_des=w.cont["Xb_des"])
    if w.kind == "cont_param":
        src.update(goal=w.cont["goal"])
    h = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in src.items()}
    hn = {k: v.numpy() for k, v in h.items()}
    hx = torch.empty_like(h["x0"]).pin_memory()
    hmp = torch.empty_like(h["mp"]).pin_memory()
    h_info = torch.empty(w.B, dtype=torch.int32).pin_memory()
    h_nfev = torch.empty(w.B, dtype=torch.int32).pin_memory()
    h_fn = torch.empty(w.B, dtype=torch.float64).pin_memory()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        hx.copy_(h["x0"])
        if w.kind == "solve":
            unit_of_work(eng, w, hn, hx.numpy(), info=h_info.numpy(), nfev=h_nfev.numpy(), fnorm=h_fn.numpy())
        else:
            hmp.copy_(h["mp"])
            unit_of_work(eng, w, hn, hx.numpy(), mp=hmp.numpy())     # the host form returns fresh result arrays
    dt = time.perf_counter() - t0
    tt = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dt = float(tt.item())
    h2d = sum(v.nbytes for v in src.values())
    d2h = (w.x0.nbytes + 4 * w.B + 4 * w.B + 8 * w.B)
    return {"value": world * w.B * steps / dt, "unit": w.unit, "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": d2h, "steps": steps,
            "api": {"solve": "socp_solve_batch", "cont_boundary": "socp_continuation_boundary_batch",
                    "cont_param": "socp_continuation_param_batch"}[w.kind] + "(mem=SOCP_HOST) via socp_b200.Engine, pinned host buffers"}


def kernel_rooflines(st, ms_profiled, P, flops_step, peak_tf, hbm_peak, traffic, N=14, M=6):
    """Per kernel of the solver round: CUDA-event time of the profiled pass, algorithmic work from the device
    counters, and the roofline that bounds it (DESIGN.md section 5)."""
    LR = P * (P + 1) // 2
    it, jac = st["iterations"], st["jac_evals"]
    nres = st.get("res_evals", 0.0)
    kern = {}

    def add(name, bound, ms, work, unit, peak, per_unit, units, note):
        if ms <= 0:
            return
        ach = work / (ms * 1e-3) / (1e12 if unit == "TFLOP/s" else 1e9)
        k = {"bound": bound, "ms": ms, "unit": unit, "peak": peak, "achieved": ach, "frac": ach / peak,
             "share_of_step": ms / ms_profiled if ms_profiled > 0 else None,
             "algorithmic_per_unit": per_unit, "units": units, "unit_of_work": note}
        tr = traffic.get(name)
        k["traffic_per_unit"] = tr["dram_bytes_per_unit"] if tr else None
        kern[name] = k

    if st["rk4_steps"] > 0:
        add("integrate_worklist", "fp64", st["integrate_ms"], st["rk4_steps"] * flops_step, "TFLOP/s", peak_tf, flops_step,
            st["rk4_steps"], "RK4 step")
    else:
        # adaptive Dormand-Prince: an accepted step is six new right-hand sides (the seventh is the next step's first)
        # and ~40 N flops of stage algebra; rejected attempts are not counted (nominal, like the RK4 figure)
        rhs = (flops_step - 12.0 * N) / 4.0
        fl = 6.0 * rhs + 40.0 * N
        add("integrate_worklist(dopri5)", "fp64", st["integrate_ms"], st["dopri_steps"] * fl, "TFLOP/s", peak_tf, fl,
            st["dopri_steps"], "accepted Dormand-Prince step")
    # Broyden phase.  Split build: a streaming pass over Q (apply the pending 2(P-1) rotations, form Q^T f:
    # Q read + written once) and a chain kernel (R read + written once, work vectors).  Fused build: one kernel.
    bytes_q = 8.0 * (2 * P * P + 6 * P)
    bytes_chain = 8.0 * (2 * LR + 16 * P)
    if st.get("qpass_ms", 0.0) > 0.02 * st["res_ms"]:           # the split build (the record between two events is never 0)
        add("hybrd_qpass_kernel", "hbm", st["qpass_ms"], it * bytes_q, "GB/s", hbm_peak, bytes_q, it, "Broyden iteration of one problem")
        add("hybrd_chain_kernel", "hbm", st["res_ms"] - st["qpass_ms"], it * bytes_chain, "GB/s", hbm_peak, bytes_chain, it,
            "Broyden iteration of one problem")
    else:
        add("hybrd_res_kernel", "hbm", st["res_ms"], it * (bytes_q + bytes_chain), "GB/s", hbm_peak, bytes_q + bytes_chain, it,
            "Broyden iteration of one problem")
    flops_jac = 8.0 / 3.0 * P ** 3
    add("hybrd_jac_kernel", "fp64", st["jac_ms"], jac * flops_jac, "TFLOP/s", peak_tf, flops_jac, jac,
        "Jacobian factorisation (Householder QR + accumulation of Q, dense count)")
    # assembly: per Jacobian request the segment end points in (nJ + M records of N + 2 doubles), P columns of
    # at most 2N + 1 reachable rows out, plus the zero fill of the P x P matrix; per residual M records in, P out
    nfree = P - N * M
    nJ = N * M + nfree * M                       # perturbed segment integrations of one forward-difference Jacobian
    bytes_asm_jac = 8.0 * ((nJ + M) * (N + 2) + P * (2 * N + 1) + P * P + 2 * P)
    bytes_asm_res = 8.0 * (M * (N + 2) + 2 * P)
    add("assemble_kernel(+zero_fjac)", "hbm", st["assemble_ms"], jac * bytes_asm_jac + nres * bytes_asm_res, "GB/s", hbm_peak,
        bytes_asm_jac, jac, "forward-difference Jacobian assembled (residual requests counted at %d B each)" % bytes_asm_res)
    return kern


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    # stdout carries exactly ONE JSON line: anything libraries print there (NCCL's version banner, ...) goes
    # to stderr instead
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    import socp_b200 as sb
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the engine has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    single = rank == 0 and world == 1

    # CPU pool first (spawned before the heavy CUDA work; rank 0, N = 1 only)
    pool = CpuPool() if single and not args.no_cpu_baseline else None

    eng = sb.Engine(local)
    peak_gflops, clk = eng.measure_fp64_peak()
    build, default_B = WORKLOADS[args.workload]
    if args.scaling == "strong":
        total = args.global_batch or 1000000
        from socp_b200 import sharding
        lo, hi = sharding.shard_bounds(total, rank, world)
        B, first = hi - lo, lo
    else:
        B = args.batch or default_B
        total, first = world * B, rank * B
    seed = 20260002 + (rank if args.scaling == "weak" else 0) + int(os.environ.get("SOCP_BENCH_SEED_OFFSET", "0"))
    if args.scaling == "strong":
        # one global batch, every rank takes its contiguous block of it
        w = _strong_block(build, eng, total, lo, hi, seed)
    else:
        w = build(eng, B, seed)
    P = w.P
    d = device_arrays(torch, dev, w)

    # ---- value: device-resident timed region, no profiling events inside it -------------------------------
    sampler = ClockSampler(local)
    sampler.start()
    eng.reset_stats()
    ms, step = timed_solves(eng, torch, dist, world, dev, w, d, args.steps, args.warmup, gather=True)
    st = eng.stats()
    sampler.stop_flag = True
    sampler.join(timeout=2)
    if args.dump_outputs:
        # the buffers still hold the last timed step: nothing has run since
        path = args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, "rank%d" % rank)
        n = dump_outputs(torch, step_outputs(w, d), path)
        print("outputs of the last timed step (%d of %d problems) written to %s" % (n, B, path), file=sys.stderr)

    if world > 1:
        print("rank %d: %.1f ms for %d step(s), %d solver rounds" % (rank, ms, args.steps, st["solver_rounds"]), file=sys.stderr)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    # steps executed in the timed region only: warm-up steps are excluded by the reset below
    agg = torch.tensor([0.0, float((d["info"] == 1).sum().item()), float(d["nfev"].sum().item()),
                        float(((d["info"] == 1) & (d["fnorm"] < 1e-5)).sum().item()), float(B)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(agg, op=dist.ReduceOp.SUM)
    ms = float(t.item())
    ms_per_step = ms / args.steps
    total_B = float(agg[4].item())
    value = total_B / (ms_per_step * 1e-3)

    # ---- separate profiled pass: CUDA events around every kernel of every round (rank-local) -----------------
    flops = FLOPS_PER_RK4_STEP[w.flops_key]
    peak_tf = peak_gflops / 1e3
    hbm_peak, hbm_src = hbm_peak_gbs()
    traffic, traffic_src = ncu_traffic(w.name, P)
    roofline, whole = None, None
    if not args.no_profile_pass:
        eng.reset_stats()
        eng.set_profiling(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step()
        e1.record()
        torch.cuda.synchronize()
        ms_prof = e0.elapsed_time(e1)
        sp = eng.stats()
        eng.set_profiling(False)
        import scenarios as S
        kern = kernel_rooflines(sp, ms_prof, P, flops, peak_tf, hbm_peak, traffic, N=2 * S.DIM[w.model], M=w.M)
        dom = max(kern, key=lambda k: kern[k]["ms"])
        dk = kern[dom]
        n_launch = max(sp["solver_rounds"], 1.0)
        roofline = {"kernel": dom, "bound": dk["bound"], "achieved": dk["achieved"], "peak": dk["peak"], "unit": dk["unit"],
                    "frac": dk["frac"],
                    "traffic": (dk["traffic_per_unit"] * dk["units"] / n_launch) if dk["traffic_per_unit"] else None,
                    "traffic_source": traffic_src,
                    "algorithmic_per_launch": dk["algorithmic_per_unit"] * dk["units"] / n_launch,
                    "avg_launch_ms": dk["ms"] / n_launch, "launches": n_launch, "share_of_step": dk["share_of_step"],
                    "profiled_step_ms": ms_prof,
                    "note": "per-kernel CUDA events of ONE extra solve of the same batch after the timed region "
                            "(profiling events are not recorded inside `value`)",
                    "peak_source": {"hbm": hbm_src, "fp64": "measured on this GPU: register-resident DFMA chain "
                                    "(socp_measure_fp64_peak); MEASURED_PEAKS.json has no FP64 entry"},
                    "flops_per_rk4_step": flops, "kernels": kern}
        # whole-solve FP64 fraction: (RK4 flops + nominal linear algebra flops) / step time / FP64 peak
        la = sp["iterations"] * la_flops_per_iteration(P) + sp["jac_evals"] * 8.0 / 3.0 * P ** 3
        rk = sp["rk4_steps"] * flops
        whole = {"fp64_frac": (rk + la) / (ms_prof * 1e-3) / 1e12 / peak_tf, "rk4_tflop": rk / 1e12, "la_tflop": la / 1e12,
                 "rk4_only_frac": rk / (ms_prof * 1e-3) / 1e12 / peak_tf, "peak_tflops": peak_tf,
                 "la_flops_per_iteration": la_flops_per_iteration(P), "la_flops_per_jacobian": 8.0 / 3.0 * P ** 3,
                 "rk4_steps": sp["rk4_steps"], "iterations": sp["iterations"], "jacobians": sp["jac_evals"],
                 "solver_rounds": sp["solver_rounds"]}
        rk4_steps_per_step = sp["rk4_steps"]
    else:
        rk4_steps_per_step = st["rk4_steps"] / max(args.steps + args.warmup, 1)
    rk4_rate = rk4_steps_per_step * world / (ms_per_step * 1e-3)

    # keep the stage-1 results of the sample for the parity object before anything overwrites them
    n_par = min(args.parity_sample, B, PARITY_CAP.get(w.name, 1 << 30)) if pool is not None else 0
    g1 = (d["info"][:n_par].cpu().numpy(), d["nfev"][:n_par].cpu().numpy(), d["x"][:n_par].cpu().numpy()) if n_par else None

    # ---- the RK4 trajectory kernel alone (BASELINE metric "RK4 steps/sec, % of FP64 roofline") ---------------
    rk4_kernel = None
    if w.model == sb.GODDARD:
        Bt = 1 << 20
        reps = 6
        Xi_t = torch.from_numpy(np.tile(w.x0[:1, :14], (Bt, 1)) * (1 + 1e-3 * np.random.default_rng(7).uniform(-1, 1, (Bt, 14)))).to(dev)
        mp_t = d["mp"][:1].repeat(Bt, 1).contiguous()
        t0_t = torch.zeros(Bt, dtype=torch.float64, device=dev)
        tf_t = torch.full((Bt,), 0.1 / 6, dtype=torch.float64, device=dev)
        out_t = torch.empty_like(Xi_t)
        for _ in range(3):
            eng.traj_batch(sb.GODDARD, mp_t, t0_t, Xi_t, tf_t, 10, out=out_t)
        eng.sync()
        eng.reset_stats()
        eng.timer_start()
        for _ in range(reps):
            eng.traj_batch(sb.GODDARD, mp_t, t0_t, Xi_t, tf_t, 10, out=out_t)
        t_ms = eng.timer_stop()
        steps_t = eng.stats()["rk4_steps"]
        tf_ach = steps_t * flops / (t_ms * 1e-3) / 1e12
        rk4_kernel = {"kernel": "traj_kernel<goddard>", "trajectories": Bt, "rk4_steps_per_s": steps_t / (t_ms * 1e-3),
                      "ms_per_launch": t_ms / reps, "achieved": tf_ach, "peak": peak_tf, "unit": "TFLOP/s",
                      "frac": tf_ach / peak_tf, "bound": "fp64", "flops_per_rk4_step": flops,
                      "note": "inputs 117 MB + outputs 117 MB per launch (> L2 together with the solver workspace)"}
        del Xi_t, mp_t, t0_t, tf_t, out_t

    # ---- end to end through the public API with pinned host buffers ------------------------------------------
    e2e = e2e_solves(eng, torch, dist, world, dev, w, args.e2e_steps)

    # ---- CPU baseline + parity on the same sample (rank 0, N = 1) --------------------------------------------
    cpu_baseline, parity, stage2 = None, None, None
    if pool is not None:
        n_s = max(args.cpu_sample or n_par, n_par)
        specs = [w.spec(k) for k in range(n_s)]
        dt, res = pool.work(specs)
        nf = sum(r[1] for r in res)
        cpu_baseline = {"value": len(res) / dt, "unit": w.unit, "cores": pool.cores,
                        "kind": "port" if w.ode_tol > 0 else pool.kind,
                        "sample": "first %d problems of the same batch, one process per core, wall time" % len(res),
                        "rk4_steps_per_s": (nf * w.M * w.steps / dt) if w.ode_tol == 0 else None,
                        "converged_fraction": sum(1 for r in res if r[0] == 1) / len(res)}
        if w.ode_tol > 0:
            cpu_baseline["note"] = ("adaptive Dormand-Prince is the reference's -D_USE_BOOST build; Boost.Odeint is absent, so the "
                                    "checker is the C port of the same algorithm (parity unpinned against Boost itself)")
        parity = parity_solve(g1[0], g1[1], g1[2], res[:n_par], w.xtol)
        parity["workload"] = w.name
        if w.kind != "solve":
            gc = d["calls"][:n_par, 0].cpu().numpy()
            parity["identical_solver_calls"] = float(np.mean(gc == np.array([r[3] for r in res[:n_par]])))
            parity["nfev_is"] = "total over the solver calls of a homotopy"
        if w.name == "goddard":
            n_e = min(128, n_par)
            _, ens = pool.run("ensemble", specs[:n_e], dict(runs=5))
            parity["ensemble"] = parity_ensemble(g1[0], g1[1], res, ens)
            parity["note"] = ("from the trivial costate guess the reference's own (info, nfev) change under a +-2-ulp change of "
                              "the arithmetic (its FMA and non-FMA CPU builds agree on 0 of 32 problems), so per-problem identity "
                              "is not expected here; it is on the warm-started stage (stage2.parity)")

    # ---- stage 2 (SURVEY C2): warm-started solves + KD continuation on the converged batch ------------------
    if single and w.name == "goddard" and not args.no_stage2:
        stage2 = run_stage2(args, eng, torch, dist, dev, w, pool)
    if pool is not None:
        pool.close()

    if rank == 0:
        conv = float(agg[1].item()) / total_B
        line = {
            "metric": METRIC if w.name.startswith("goddard") else "shooting %s (%s)" % (w.unit.replace("/s", "/sec"), w.label),
            "value": value, "unit": w.unit, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": w.label,
                       "batch_per_gpu": B, "global_batch": int(total_B), "xtol": w.xtol, "rk4_steps_per_segment": w.steps,
                       "parallelism": "problems sharded, %d rank(s), no data-path collective; results all-gathered" % world,
                       "l2": "working set %.1f GB per GPU >> 126 MB L2, no flush needed" % (st["device_bytes"] / 1e9)},
            "rk4_steps_per_s": rk4_rate, "rk4_steps_per_step": rk4_steps_per_step * world,
            "converged_fraction": conv,                                            # info == 1, what SOCP accepts
            "converged_solves_per_s": value * conv,
            "true_root_fraction": (float(agg[3].item()) / total_B) if w.kind == "solve" else None,   # info == 1 and |F| < 1e-5
            "mean_nfev": float(agg[2].item()) / total_B,
            "mean_solver_calls": float(d["calls"][:, 0].double().mean().item()) if w.kind != "solve" else 1.0,
            "solver_rounds_per_step": st["solver_rounds"] / (args.steps + args.warmup),
            "gpu_launches": int(st["kernel_launches"] * args.steps / (args.steps + args.warmup)),
            "roofline": roofline, "whole_solve": whole, "rk4_kernel": rk4_kernel, "e2e": e2e, "cpu_baseline": cpu_baseline,
            "parity": parity, "stage2": stage2,
            "clocks": sampler.summary(), "fp64_peak_probe_sm_mhz": clk,
        }
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


_PER_PROBLEM_CONT = ("time_des", "Xb_des", "goal")          # continuation data with one row per problem


def _slice(w, lo, hi):
    w.mp, w.time, w.Xb, w.x0 = (np.ascontiguousarray(a[lo:hi]) for a in (w.mp, w.time, w.Xb, w.x0))
    if w.cont:
        w.cont = {k: (np.ascontiguousarray(v[lo:hi]) if k in _PER_PROBLEM_CONT else v) for k, v in w.cont.items()}
    return w


def _strong_block(build, eng, total, lo, hi, seed):
    """Rows [lo, hi) of a large global batch without building all of it: the batch is defined as consecutive
    blocks of 100000 problems drawn with seeds seed, seed + 1, ... (independent of the world size)."""
    blk = 100000
    parts = []
    b0 = (lo // blk) * blk
    while b0 < hi:
        wb = build(eng, min(blk, total - b0), seed + b0 // blk)
        a, b = max(lo, b0) - b0, min(hi, b0 + blk) - b0
        parts.append(_slice(wb, a, b))
        b0 += blk
    w = parts[0]
    if len(parts) > 1:
        w.mp, w.time, w.Xb, w.x0 = (np.ascontiguousarray(np.concatenate([getattr(p, k) for p in parts])) for k in ("mp", "time", "Xb", "x0"))
        if w.cont:
            w.cont = {k: (np.ascontiguousarray(np.concatenate([p.cont[k] for p in parts])) if k in _PER_PROBLEM_CONT else v)
                      for k, v in w.cont.items()}
    return w


def run_stage2(args, eng, torch, dist, dev, w1, pool):
    """SURVEY C2 stage 2 on the same batch.  (a) warm-started solves: x0 = the reference's converged x* of the
    unperturbed problem; (b) the KD 0 -> 310 continuation (tests/testGoddard.cpp:105, step 1) from the members
    converged in (a).  Both are compared problem for problem with oracle/_ref on the parity sample."""
    import scenarios as S
    out = {}
    w = Workload("goddard_warm", w1.model, w1.shape, w1.mp, w1.time, w1.Xb, np.tile(reference_xstar(), (w1.B, 1)),
                 w1.xtol, w1.steps, w1.flops_key,
                 "goddard_warm_start_M6_P85_batch (SURVEY C2 stage 2: reference x* + perturbed boundary data)",
                 w1.mode_t, w1.mode_X, w1.M)
    d = device_arrays(torch, dev, w)
    eng.reset_stats()
    ms, _ = timed_solves(eng, torch, dist, 1, dev, w, d, args.steps, 1, gather=False)
    st = eng.stats()
    info, nfev, x = d["info"].cpu().numpy(), d["nfev"].cpu().numpy(), d["x"].cpu().numpy()
    fn = d["fnorm"].cpu().numpy()
    e2e = e2e_solves(eng, torch, dist, 1, dev, w, args.e2e_steps)
    warm = {"workload": w.label, "value": w.B * args.steps / (ms * 1e-3), "unit": "solves/s", "ms_per_step": ms / args.steps,
            "steps": args.steps, "converged_fraction": float((info == 1).mean()),
            "true_root_fraction": float(((info == 1) & (fn < 1e-5)).mean()), "mean_nfev": float(nfev.mean()),
            "solver_rounds_per_step": st["solver_rounds"] / (args.steps + 1), "e2e": e2e}
    n_par = min(args.parity_sample, w.B) if pool is not None else 0
    ref_warm = None
    if n_par:
        specs = [w.spec(k) for k in range(n_par)]
        dt, ref_warm = pool.solve(specs)
        warm["parity"] = parity_solve(info, nfev, x, ref_warm, w.xtol)
        warm["cpu_baseline"] = {"value": n_par / dt, "unit": "solves/s", "cores": pool.cores, "kind": pool.kind,
                                "sample": "first %d problems of the same batch, one process per core, wall time" % n_par}
    out["warm_start"] = warm

    # (b) continuation KD 0 -> 310, step 1 (shooting.cpp:695-778) on the members that converged in (a).
    # Device resident: the warm-started solutions stay in HBM and the homotopy state machines run on the device
    # (socp_continuation_param_batch, mem = SOCP_DEVICE); the host-buffer form is timed beside it as e2e.
    ok = np.flatnonzero(info == 1)
    if ok.size:
        kd = S.pidx(S.GODDARD, "KD")
        okd = torch.from_numpy(ok).to(dev)
        sel_d = lambda t: t.index_select(0, okd).contiguous()
        c_mp0, c_time, c_Xb, c_x0 = sel_d(d["mp"]), sel_d(d["time"]), sel_d(d["Xb"]), sel_d(d["x"])
        c_goal = torch.full((ok.size,), 310.0, dtype=torch.float64, device=dev)
        c_info = torch.empty(ok.size, dtype=torch.int32, device=dev)
        c_calls = torch.empty((ok.size, 2), dtype=torch.int32, device=dev)
        c_mp, c_x = torch.empty_like(c_mp0), torch.empty_like(c_x0)

        def cont_step():
            c_mp.copy_(c_mp0); c_x.copy_(c_x0)
            eng.continuation_param_batch(w.shape, c_mp, c_time, c_Xb, c_x, 1.0, kd, c_goal, xtol=w.xtol, info=c_info, calls=c_calls)
        cont_step()                                                         # warm-up
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.e2e_steps):
            cont_step()
        e1.record()
        torch.cuda.synchronize()
        dt = e0.elapsed_time(e1) * 1e-3 / args.e2e_steps
        r = dict(info=c_info.cpu().numpy(), calls=c_calls.cpu().numpy(), x=c_x.cpu().numpy())
        # the same through host buffers (staged once in, once out by the library)
        h_args = (w.shape, np.ascontiguousarray(w.mp[ok]), np.ascontiguousarray(w.time[ok]), np.ascontiguousarray(w.Xb[ok]),
                  np.ascontiguousarray(x[ok]), 1.0, kd, np.full(ok.size, 310.0))
        t0 = time.perf_counter()
        rh = eng.continuation_param_batch(*h_args, xtol=w.xtol)
        dth = time.perf_counter() - t0
        cont = {"workload": "goddard continuation KD 0 -> 310, step 1 (tests/testGoddard.cpp:105) on the %d members converged "
                            "in the warm-started stage" % ok.size,
                "value": ok.size / dt, "unit": "continuations/s", "seconds": dt,
                "api": "socp_continuation_param_batch(mem=SOCP_DEVICE): homotopy state machines on the device, no problem data over PCIe",
                "e2e": {"value": ok.size / dth, "unit": "continuations/s", "api": "socp_continuation_param_batch(mem=SOCP_HOST)",
                        "same_outcome_as_device": bool(np.array_equal(rh["info"], r["info"]) and np.array_equal(rh["calls"], r["calls"])
                                                       and np.array_equal(rh["x"], r["x"]))},
                "converged_fraction": float((r["info"] == 1).mean()),
                "mean_solver_calls": float(r["calls"][:, 0].mean()), "mean_nfev_total": float(r["calls"][:, 1].mean())}
        if n_par:
            sel = [k for k in range(n_par) if info[k] == 1 and ref_warm[k][0] == 1]
            # each side continues from ITS OWN stage-(a) solution, as the reference's pipeline does
            specs = [w.spec(k, x0=ref_warm[k][2]) for k in sel]
            dtc, ref_c = pool.run("cont_param", specs, dict(step=1.0, pname="KD", goal=310.0))
            pos = {k: i for i, k in enumerate(ok)}
            gi = np.array([r["info"][pos[k]] for k in sel]); gc = np.array([r["calls"][pos[k]] for k in sel])
            gx = np.array([r["x"][pos[k]] for k in sel])
            ri = np.array([c[0] for c in ref_c]); rc = np.array([[c[1], c[2]] for c in ref_c])
            both = (gi == 1) & (ri == 1)
            rel = np.array([np.linalg.norm(gx[i] - ref_c[i][3]) / np.linalg.norm(ref_c[i][3]) for i in range(len(sel)) if both[i]])
            cont["parity"] = {
                "sample": len(sel), "checker": "oracle/_ref",
                "identical_info": float((gi == ri).mean()), "identical_solver_calls": float((gc[:, 0] == rc[:, 0]).mean()),
                "identical_info_calls_nfev": float(((gi == ri) & (gc[:, 0] == rc[:, 0]) & (gc[:, 1] == rc[:, 1])).mean()),
                "mean_nfev_total_gpu": float(gc[:, 1].mean()), "mean_nfev_total_ref": float(rc[:, 1].mean()),
                "x_within_xtol": float((rel <= w.xtol).mean()) if rel.size else None,
                "x_rel_err_max": float(rel.max()) if rel.size else None,
                "x_rel_err_median": float(np.median(rel)) if rel.size else None,
                "note": "KD = 310 from the KD = 0 solution in one step is ill conditioned in the reference itself: its FMA and "
                        "non-FMA CPU builds (same code, gcc) agree on nfev for 15 of 32 problems, always on info, and their "
                        "unknowns differ by 4.1e-6 (median) / 4.5e-5 (worst) relative, 25 % within xtol (DESIGN.md section 3)",
            }
            cont["cpu_baseline"] = {"value": len(sel) / dtc, "unit": "continuations/s", "cores": pool.cores, "kind": pool.kind}
        out["continuation_KD"] = cont
    return out


if __name__ == "__main__":
    main()
