"""Throughput of the batched initial guess (socp_init_shooting_batch) next to the trajectory calls it replaces.

  python tools/init_rate.py [reps=10] [B_goddard=100000] [B_covid19=10000]

Two workloads, RK4:
  * Goddard, M = 6, S = 10: the guess of bench.py's goddard_workload (B problems of tests/testGoddard.cpp);
  * covid19, M = 20, S = 1000 (tests/testCovid19.cpp's mesh and step count).
For each, three ways to build the B (M - 1) interior nodes, every array on the device (torch tensors, DEVICE mode):
  * init    socp_init_shooting_batch: the whole guess (time, Xb, x), one call;
  * loop    one socp_traj_batch of B trajectories per interior node, as the C++ mirror and bench.py used to do;
  * single  one socp_traj_batch over the same B (M - 1) segments (inputs laid out node-major beforehand, not timed).
Times are CUDA events on the engine's stream around INNER = 10 back-to-back call sequences (the host enqueues ahead of
the device, as in a pipeline, so the Python and launch overhead of one call is not device idle time), per sequence, the
median of `reps` such windows, the three variants alternated twice for the spread.  Prints one JSON line per
measurement, the first with the GPU's name and power limit.  The Goddard inputs (B x 14 doubles) fit the 126 MB L2; both workloads are bound by the integration, not by memory."""
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
import scenarios as S  # noqa: E402

INNER = 10


def gpu_facts():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))


def workload(name, B):
    """(model, shape, mparams [np], ti [B], Xi [B][2dim], tf [B], Xf [B][dim]) on the host"""
    if name == "goddard":
        M, S_ = 6, 10
        Xi, xf0 = S.goddard_batch_inputs(B)
        mp = np.array(S.DEFAULTS[S.GODDARD])
        mp[6] = 1.0
        Xf = np.zeros((B, 7))
        Xf[:, 0] = xf0
        model, ti, tf, mode_Xf = S.GODDARD, 0.0, 0.1, S.GODDARD_MODE_XF
    else:
        M, S_ = 20, 1000
        rng = np.random.default_rng(0)
        Xi = S.COVID_XI * (1 + 1e-2 * rng.uniform(-1, 1, size=(B, 8)))
        mp = np.array(S.DEFAULTS[S.COVID19])
        Xf = np.tile(S.COVID_XI[:4], (B, 1))
        model, ti, tf, mode_Xf = S.COVID19, 0.0, 20.0, [S.FREE] * 4
    mode_t, mode_X = sb.default_modes(model, M, sb.FIXED, mode_Xf)
    shape = sb.make_shape(model, M, mode_t, mode_X, S_)
    return model, shape, mp, np.full(B, ti), np.ascontiguousarray(Xi), np.full(B, tf), np.ascontiguousarray(Xf)


def measure(eng, name, B, reps):
    model, shape, mp, ti, Xi, tf, Xf = workload(name, B)
    M, S_, N = shape.num_multi, shape.step_nbr, Xi.shape[1]
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    mp_d, ti_d, Xi_d, tf_d, Xf_d = d(np.tile(mp, (B, 1))), d(ti), d(Xi), d(tf), d(Xf)
    nodes = [d(ti + i * (tf - ti) / M) for i in range(1, M)]
    outs = [torch.empty_like(Xi_d) for _ in nodes]
    K = B * (M - 1)                                   # the segments, node-major
    mp_k, ti_k, Xi_k = d(np.tile(mp, (K, 1))), d(np.tile(ti, M - 1)), d(np.tile(Xi, (M - 1, 1)))
    tf_k = torch.cat(nodes).contiguous()
    out_k = torch.empty_like(Xi_k)
    res = {}

    def init():
        res["init"] = eng.init_shooting_batch(shape, mp_d, ti_d, Xi_d, tf_d, Xf_d)

    def loop():
        for t, o in zip(nodes, outs):
            eng.traj_batch(model, mp_d, ti_d, Xi_d, t, S_, out=o)

    def single():
        eng.traj_batch(model, mp_k, ti_k, Xi_k, tf_k, S_, out=out_k)

    init(), loop(), single()
    torch.cuda.synchronize()
    x = res["init"][2]
    same = all(torch.equal(x[:, N * i:N * (i + 1)], outs[i - 1]) for i in range(1, M)) and \
        torch.equal(torch.stack(outs), out_k.view(M - 1, B, N))
    print(json.dumps(dict(workload=name, check="init nodes == loop == single traj, bit for bit", ok=bool(same))), flush=True)

    def rate(f, what):
        for _ in range(2):
            f()
        eng.sync()
        eng.reset_stats()
        runs = []
        for _ in range(reps):
            eng.timer_start()
            for _ in range(INNER):
                f()
            runs.append(eng.timer_stop() / INNER)
        steps = eng.stats()["rk4_steps"] / (reps * INNER)
        ms = float(np.median(runs))
        r = dict(workload=name, what=what, B=B, M=M, S=S_, trajectories=K, rk4_steps=steps, ms_median=ms,
                 ms_min=float(min(runs)), ms_max=float(max(runs)), rk4_steps_per_s=steps / (ms * 1e-3))
        print(json.dumps(r), flush=True)
        return r

    rows = []
    for _ in range(2):
        rows += [rate(init, "init_shooting_batch"), rate(loop, "traj_batch per interior node"),
                 rate(single, "one traj_batch, same segments")]
    med = lambda k: float(np.median([r["ms_median"] for r in rows[k::3]]))
    print(json.dumps(dict(workload=name, init_ms=med(0), loop_ms=med(1), single_ms=med(2),
                          init_over_single_time=med(0) / med(2), init_over_loop_time=med(0) / med(1))), flush=True)


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 10
    Bg = int(sys.argv[2]) if len(sys.argv) > 2 else 100000
    Bc = int(sys.argv[3]) if len(sys.argv) > 3 else 10000
    print(json.dumps(dict(gpu=gpu_facts(), reps=reps)), flush=True)
    eng = sb.Engine(0)
    eng.use_torch_stream()
    measure(eng, "goddard", Bg, reps)
    measure(eng, "covid19", Bc, reps)


if __name__ == "__main__":
    main()
