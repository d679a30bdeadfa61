"""Throughput of tracing solved problems on the device (socp_solution_trace_batch) next to the kernels it restates.

  python tools/trace_rate.py [B=100000] [reps=10]

B perturbed copies of the golden Goddard stage-3 solution (M = 6 segments, S = 10 RK4 steps, W = 20 columns):
B * M * S RK4 steps and B * M * (S + 1) rows of output (1.06 GB at B = 1e5).  Timed with CUDA events, after a
warm-up, the arms alternated twice:
  * socp_solution_trace_batch on the B solutions;
  * socp_trace_batch on the same B * M segments in one launch (start, node state, end, switching times and S the same;
    the time line is computed before the timed region);
  * socp_traj_batch on the same segments (the integration without the observer).
Every array lives on the device (torch tensors, DEVICE mode); the output is far larger than the 126 MB L2.  For each
it prints the kernel time, RK4 steps/s and output GB/s, the output rate as a fraction of the 6458 GB/s copy
bandwidth of DESIGN.md section 5, and the fraction of the trajectory kernel's steps/s.  One JSON line per
measurement, the first with the GPU's name and power limit."""
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import socp_b200 as sb  # noqa: E402
from golden_util import by_name, spec_from_hex, unhex  # noqa: E402

COPY_GBS = 6458.0


def gpu_facts():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 100000
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
    print(json.dumps(dict(gpu=gpu_facts(), B=B, reps=reps)), flush=True)
    eng = sb.Engine(0)
    eng.use_torch_stream()
    L, h = eng._L, eng._h
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    e3 = by_name("cont_param", "goddard_stage3_mu2")
    spec = spec_from_hex(e3["spec"])
    mp1 = np.array(spec["mparams"])
    mp1[6] = unhex(e3["goal"])
    shape = sb.make_shape(spec["model"], spec["M"], spec["mode_t"], spec["mode_X"], spec["steps"])
    M, N, S = spec["M"], 14, spec["steps"]
    R, W = L.socp_trace_max_rows(sb.GODDARD, S), L.socp_trace_width(sb.GODDARD)
    x1 = unhex(e3["x"])
    Xh = x1 * (1 + 1e-7 * np.random.default_rng(0).uniform(-1, 1, size=(B, x1.size)))
    X, mp, time = d(Xh), d(np.tile(mp1, (B, 1))), d(np.tile(spec["time"], (B, 1)))
    rows = torch.empty((B, M, R, W), dtype=torch.float64, device="cuda")
    nrows = torch.empty((B, M), dtype=torch.int32, device="cuda")

    # the B * M segments as socp_trace_batch / socp_traj_batch inputs, from the time line of GetSolution
    vt, _ = eng.solution_batch(shape, mp, time, X)
    t0, tf = vt[:, :M].reshape(-1).contiguous(), vt[:, 1:].reshape(-1).contiguous()
    X0 = X[:, :N * M].reshape(B * M, N).contiguous()
    mpM = mp.repeat_interleave(M, dim=0).contiguous()
    sw = d(np.tile([0.0227, 0.08], (B * M, 1)))         # no FREE interior time: the defaults
    rows2, nrows2 = torch.empty_like(rows).view(B * M, R, W), torch.empty_like(nrows).view(B * M)
    Xf = torch.empty_like(X0)

    def solution_trace():                  # Engine.solution_trace_batch without its output allocation
        eng._check(L.socp_solution_trace_batch(h, ctypes.byref(shape), B, p(mp), p(time), p(X), p(rows), p(nrows), 1))

    def trace():
        eng._check(L.socp_trace_batch(h, sb.GODDARD, S, B * M, p(mpM), p(sw), p(t0), p(tf), p(X0), p(rows2), p(nrows2),
                                      None, 1))

    def traj():
        eng.traj_batch(sb.GODDARD, mpM, t0, X0, tf, S, sw=sw, out=Xf)

    solution_trace()
    trace()
    torch.cuda.synchronize()
    same = bool(torch.equal(nrows.view(-1), nrows2) and torch.equal(rows.view(B * M, R, W), rows2))
    print(json.dumps(dict(check="solution_trace == trace_batch bit for bit", ok=same)), flush=True)

    steps = B * M * S
    out_bytes = B * M * (S + 1) * W * 8 + B * M * 4

    def rate(f, what, bytes_out):
        for _ in range(3):
            f()
        eng.sync()
        runs = []
        for _ in range(reps):
            eng.timer_start()
            f()
            runs.append(eng.timer_stop())
        ms = float(np.median(runs))
        r = dict(what=what, segments=B * M, rk4_steps=steps, out_bytes=bytes_out, ms_median=ms, ms_min=float(min(runs)),
                 ms_max=float(max(runs)), rk4_steps_per_s=steps / (ms * 1e-3), out_GB_per_s=bytes_out / (ms * 1e-3) / 1e9)
        r["out_share_of_copy_bw"] = r["out_GB_per_s"] / COPY_GBS
        print(json.dumps(r), flush=True)
        return r

    res = {"solution_trace": [], "trace": [], "traj": []}
    for _ in range(2):
        res["solution_trace"].append(rate(solution_trace, "socp_solution_trace_batch", out_bytes))
        res["trace"].append(rate(trace, "socp_trace_batch, same segments", out_bytes))
        res["traj"].append(rate(traj, "socp_traj_batch, same segments", B * M * N * 8))
    med = {k: float(np.median([r["ms_median"] for r in v])) for k, v in res.items()}
    print(json.dumps(dict(solution_trace_over_trace_time=med["solution_trace"] / med["trace"],
                          solution_trace_steps_per_s_over_traj=med["traj"] / med["solution_trace"],
                          write_bound_ms=out_bytes / (COPY_GBS * 1e9) * 1e3, traj_ms=med["traj"])), flush=True)


if __name__ == "__main__":
    main()
