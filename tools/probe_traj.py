"""Quick device probe: FP64 peak + RK4 trajectory kernel throughput per model (device-resident)."""
import json, sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np, torch
import socp_b200 as sb
import scenarios as S
FLOPS_PER_STEP = {0: 1100, 1: 264, 2: 256, 3: 2736, 4: 1704}
eng = sb.Engine(0)
o = S.VTOL_OBSTACLES; eng.set_obstacles(o["type"], o["pos"], o["rad"])
peak, clk = eng.measure_fp64_peak()
print(json.dumps(dict(fp64_peak_gflops=peak, sm_clock_mhz=clk)))
eng.use_torch_stream()
B = int(sys.argv[1]) if len(sys.argv) > 1 else 1 << 20
base = {0: S.GODDARD_XI, 1: np.r_[np.zeros(6), 0.01*np.ones(6)], 2: S.COVID_XI,
        3: np.array([20, 8, 5, 0.3, 0.2, 0.1, -0.03, 0.013, -0.003, -0.29, 0.1, -0.03]),
        4: np.array(S.INTERCEPTOR_INIT_XI + [0.01, -1, 0.5, 0.2, 100., 50.])}
tfs = {0: 0.1, 1: 8.0, 2: 1.5, 3: 5.0, 4: 10.0}
rng = np.random.default_rng(0)
only = [int(v) for v in sys.argv[2].split(",")] if len(sys.argv) > 2 else list(range(5))     # model ids, e.g. "3" = vtolUAV
print(json.dumps(dict(lib=os.environ.get("SOCP_LIB", "default"))))
for model in only:
    Bm = B if model != 2 else B // 16
    mp = np.array(S.DEFAULTS[model]);
    if model == 0: mp[6], mp[2] = 1.0, 0.0
    X0 = base[model] * (1 + 0.01 * rng.uniform(-1, 1, size=(Bm, base[model].size)))
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    dX0, dmp = d(X0), d(np.tile(mp, (Bm, 1)))
    dt0, dtf = torch.zeros(Bm, dtype=torch.float64, device="cuda"), torch.full((Bm,), tfs[model], dtype=torch.float64, device="cuda")
    out = torch.empty_like(dX0)
    for _ in range(2): eng.traj_batch(model, dmp, dt0, dX0, dtf, out=out)
    eng.sync(); eng.reset_stats()
    reps = 5
    eng.timer_start()
    for _ in range(reps): eng.traj_batch(model, dmp, dt0, dX0, dtf, out=out)
    ms = eng.timer_stop() / reps
    steps = eng.stats()["rk4_steps"] / reps
    gf = steps * FLOPS_PER_STEP[model] / (ms * 1e-3) / 1e9
    print(json.dumps(dict(model=sb.MODEL_NAMES[model], B=Bm, ms=ms, rk4_steps_per_s=steps / (ms * 1e-3), nominal_gflops=gf, frac_of_peak=gf / peak)))
