"""Throughput of sampling solved problems on the device, and the cost of a re-mesh next to the solve it feeds.

  python tools/move_rate.py [B=100000] [reps=10]

Goddard stage 4 of tests/testGoddard.cpp for B perturbed copies of the golden stage-3 solution (M = 6):
  * socp_solution_batch + socp_move_batch at the Q = M + 1 = 7 stage-4 node times: RK4 steps/s (device counter over
    CUDA-event time), next to socp_traj_batch integrating exactly the same 8 B segments (same start, node state,
    target, switching times, S);
  * the wall time of the stage-4 re-mesh (GetSolution, Move, unknowns_from_nodes, all device-resident) against the
    stage-4 solve it prepares.
Every array lives on the device (torch tensors, DEVICE mode); the traj inputs (8 B x 38 doubles, 240 MB at B = 1e5)
exceed the 126 MB L2.  Prints one JSON line per measurement, the first with the GPU's name and power limit."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import socp_b200 as sb  # noqa: E402
from golden_util import by_name, spec_from_hex, unhex  # noqa: E402

S1, S2 = 0.0227, 0.08


def gpu_facts():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))


def shape_of(spec):
    return sb.make_shape(spec["model"], spec["M"], spec["mode_t"], spec["mode_X"], spec["steps"])


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 100000
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
    print(json.dumps(dict(gpu=gpu_facts(), B=B, reps=reps)), flush=True)
    eng = sb.Engine(0)
    eng.use_torch_stream()
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    e3 = by_name("cont_param", "goddard_stage3_mu2")
    spec3 = spec_from_hex(e3["spec"])
    mp3 = np.array(spec3["mparams"])
    mp3[6] = unhex(e3["goal"])
    g4 = spec_from_hex(by_name("solve", "goddard_stage4_singular")["spec"])
    shape3, shape4 = shape_of(spec3), shape_of(g4)
    x3 = unhex(e3["x"])
    rng = np.random.default_rng(0)
    X = d(x3 * (1 + 1e-7 * rng.uniform(-1, 1, size=(B, x3.size))))
    mp, time3 = d(np.tile(mp3, (B, 1))), d(np.tile(spec3["time"], (B, 1)))
    mp4 = d(np.tile(g4["mparams"], (B, 1)))
    M, N, Q = 6, 14, 7
    s = torch.tensor([0.0, S1 / 2, S1, (S2 + S1) / 2, S2], dtype=torch.float64, device="cuda")

    def remesh():
        vt, vX = eng.solution_batch(shape3, mp, time3, X)
        tf = vt[:, M:M + 1]
        vt4 = torch.cat([s.expand(B, 5), (S2 + tf) / 2, tf], dim=1).contiguous()
        Xq = eng.move_batch(shape3, mp, time3, X, vt4)
        x4, Xb4 = sb.unknowns_from_nodes(shape4, vt4, Xq)
        return vt, vX, vt4, Xq, x4, Xb4

    # the segments the moves integrate, for socp_traj_batch: 7 queries + Move(t_end) per problem
    vt, vX, vt4, Xq, x4, Xb4 = remesh()
    torch.cuda.synchronize()
    tl, targets = vt.cpu().numpy(), vt4.cpu().numpy()
    seg = np.argmax(tl[:, None, 1:] >= targets[:, :, None], axis=2)           # seg = 0; while (tl[seg+1] < t) ++seg
    seg = np.concatenate([seg, np.full((B, 1), M - 1)], axis=1)
    tq = np.concatenate([targets, tl[:, M:]], axis=1)
    Xn = X.cpu().numpy()[:, :N * M].reshape(B, M, N)
    t0 = d(np.take_along_axis(tl, seg, axis=1).reshape(-1))
    X0 = d(np.take_along_axis(Xn, seg[:, :, None], axis=1).reshape(-1, N))
    tf_ = d(tq.reshape(-1))
    mp8 = d(np.repeat(np.tile(mp3, (B, 1)), Q + 1, axis=0))
    sw = d(np.tile([S1, S2], (B * (Q + 1), 1)))
    out = torch.empty_like(X0)

    def traj():
        eng.traj_batch(sb.GODDARD, mp8, t0, X0, tf_, spec3["steps"], sw=sw, out=out)

    def sample():
        eng.solution_batch(shape3, mp, time3, X)
        eng.move_batch(shape3, mp, time3, X, vt4, out=Xq)

    # same answers: the moves are the traj kernel's integrations
    sample()
    traj()
    torch.cuda.synchronize()
    o = out.view(B, Q + 1, N)
    same = bool(torch.equal(o[:, :Q], Xq) and torch.equal(o[:, Q], vX[:, M]))
    print(json.dumps(dict(check="move == traj bit for bit", ok=same)), flush=True)

    def rate(f, what, trajectories):
        for _ in range(2):
            f()
        eng.sync()
        eng.reset_stats()
        runs = []
        for _ in range(reps):
            eng.timer_start()
            f()
            runs.append(eng.timer_stop())
        steps = eng.stats()["rk4_steps"] / reps
        ms = float(np.median(runs))
        r = dict(what=what, trajectories=trajectories, rk4_steps=steps, ms_median=ms, ms_min=float(min(runs)),
                 ms_max=float(max(runs)), rk4_steps_per_s=steps / (ms * 1e-3))
        print(json.dumps(r), flush=True)
        return r

    res = []
    for _ in range(2):                      # alternate the two, twice, for the spread
        res.append(rate(sample, "solution_batch + move_batch (Q = 7)", B * (Q + 1)))
        res.append(rate(traj, "traj_batch, same segments", B * (Q + 1)))
    mv = np.median([r["rk4_steps_per_s"] for r in res[0::2]])
    tr = np.median([r["rk4_steps_per_s"] for r in res[1::2]])
    print(json.dumps(dict(move_over_traj_steps_per_s=mv / tr)), flush=True)

    # the stage-4 re-mesh next to the stage-4 solve (wall clock, each ended by a device synchronise)
    walls = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        vt, vX, vt4, Xq, x4, Xb4 = remesh()
        torch.cuda.synchronize()
        walls.append(time.perf_counter() - t)
    x = x4.clone()
    torch.cuda.synchronize()
    t = time.perf_counter()
    r = eng.solve_batch(shape4, mp4, vt4, Xb4.reshape(B, -1), x, xtol=g4["xtol"])
    torch.cuda.synchronize()
    solve_s = time.perf_counter() - t
    info = r["info"].cpu().numpy()
    print(json.dumps(dict(what="stage-4 re-mesh vs stage-4 solve", remesh_s_median=float(np.median(walls)),
                          remesh_s_min=float(min(walls)), solve_s=solve_s, converged=int((info == 1).sum()),
                          remesh_share_of_stage=float(np.median(walls)) / (float(np.median(walls)) + solve_s))), flush=True)


if __name__ == "__main__":
    main()
