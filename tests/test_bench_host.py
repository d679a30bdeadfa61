"""Host-side logic of bench.py that needs no GPU: the CPU pool keeps the order of its problems, and the
parity objects report what they say."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_cpu_pool_keeps_problem_order(oracle_lib):
    import bench
    import scenarios as S
    from backends import OracleBackend
    specs = []
    for k in range(5):
        s = S.di_problem()
        s["Xb"][1][1] = 15.0 + k
        specs.append(s)
    pool = bench.CpuPool(cores=3)
    try:
        _, res = pool.solve(specs)
    finally:
        pool.close()
    ora = OracleBackend()
    for s, r in zip(specs, res):
        o = ora.solve(s)
        assert (r[0], r[1]) == (o["info"], o["nfev"])
        assert np.linalg.norm(r[2] - o["x"]) <= 1e-8 * np.linalg.norm(o["x"])
    # the problems differ, so a permutation would show
    assert len({tuple(np.round(r[2], 6)) for r in res}) == 5


def test_parity_solve_counts():
    import bench
    x = np.ones((4, 3))
    ref = [(1, 10, x[0]), (1, 11, x[1] * (1 + 1e-3)), (4, 50, x[2]), (1, 12, x[3])]
    p = bench.parity_solve(np.array([1, 1, 1, 5]), np.array([10, 11, 40, 12]), x, ref, 1e-6)
    assert p["sample"] == 4
    assert p["identical_info"] == 0.5 and p["identical_info_nfev"] == 0.5
    assert p["both_converged"] == 2 and p["x_within_xtol"] == 0.5
    assert abs(p["x_rel_err_max"] - 1e-3 / (1 + 1e-3)) < 1e-9
    assert p["max_abs_nfev_diff"] == 10


def test_parity_ensemble_membership():
    import bench
    runs = [[(1, 100), (1, 120), (4, 300)], [(1, 90), (1, 90), (1, 90)]]
    ref = [(1, 100, None), (1, 90, None)]
    p = bench.parity_ensemble(np.array([4, 1]), np.array([310, 120]), ref, runs)
    assert p["reference_stable_fraction"] == 0.5
    assert p["gpu_in_ensemble"] == 0.5 and p["reference_in_ensemble"] == 1.0


def test_reference_xstar_is_the_golden_solution():
    import bench
    x = bench.reference_xstar()
    assert x.shape == (85,) and abs(x[84] - 0.21965083876703931) < 1e-15      # SURVEY 8c: tf of Goddard stage 1


def test_strong_scaling_blocks_carry_every_per_problem_array():
    """bench.py --scaling strong: a rank's block of the global batch is cut out of 100000-problem blocks drawn with
    fixed seeds; every per-problem array -- the continuation targets too -- must follow the cut, whatever the
    world size (a rank whose block spans two seed blocks included)."""
    import bench
    total = 250000
    for build in (bench.wl_interceptor, bench.wl_covid19):
        full = bench._strong_block(build, None, total, 0, total, 7)
        assert full.B == total
        for world in (2, 8):
            per = -(-total // world)
            for rank in (0, world - 1, world // 2):
                lo, hi = min(rank * per, total), min(rank * per + per, total)
                w = bench._strong_block(build, None, total, lo, hi, 7)
                assert w.B == hi - lo
                assert np.array_equal(w.x0, full.x0[lo:hi]) and np.array_equal(w.Xb, full.Xb[lo:hi])
                for k in bench._PER_PROBLEM_CONT:
                    if k in w.cont:
                        assert w.cont[k].shape[0] == hi - lo, (k, w.cont[k].shape)
                        assert np.array_equal(w.cont[k], full.cont[k][lo:hi]), k
                s0 = w.spec(0)
                assert s0["cont"]["step"] == w.cont["step"]


def test_dump_outputs_writes_float64_within_budget(tmp_path):
    """bench.py --dump-outputs: every output of the step as <name>.npy in float64; a batch too large for the budget
    is sampled on the same fixed rows in every array, and the sample is the same from run to run."""
    import torch
    import bench
    B, P = 200000, 85
    w = bench.Workload("goddard", 0, None, None, None, None, np.zeros((B, P)), 1e-6, 10, "goddard", "", None, None, 6)
    d = {"x": torch.arange(B * P, dtype=torch.float64).reshape(B, P), "info": torch.arange(B, dtype=torch.int32),
         "nfev": torch.full((B,), 7, dtype=torch.int32), "fnorm": torch.zeros(B, dtype=torch.float64)}
    outs = bench.step_outputs(w, d)
    assert sorted(outs) == ["fnorm", "info", "nfev", "x"]
    n = bench.dump_outputs(torch, outs, str(tmp_path / "a"))
    assert 0 < n < B
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["fnorm.npy", "info.npy", "nfev.npy", "sample_rows.npy", "x.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_BYTES
    rows = np.load(tmp_path / "a" / "sample_rows.npy").astype(np.int64)
    x, info = np.load(tmp_path / "a" / "x.npy"), np.load(tmp_path / "a" / "info.npy")
    assert x.dtype == np.float64 and info.dtype == np.float64 and x.shape == (n, P)
    assert np.array_equal(info, rows) and np.array_equal(x[:, 0], rows * P)
    bench.dump_outputs(torch, outs, str(tmp_path / "b"))
    assert np.array_equal(np.load(tmp_path / "b" / "sample_rows.npy"), rows)
    # a small batch is written whole; a homotopy returns its solver calls and the rewritten parameters
    wc = bench.Workload("covid19", 2, None, None, None, None, np.zeros((8, 3)), 1e-6, 10, "covid19", "", None, None, 20,
                        kind="cont_param")
    dc = {"x": torch.ones(8, 3, dtype=torch.float64), "info": torch.ones(8, dtype=torch.int32),
          "calls": torch.ones(8, 2, dtype=torch.int32), "mpw": torch.ones(8, 5, dtype=torch.float64)}
    outs = bench.step_outputs(wc, dc)
    assert sorted(outs) == ["calls", "info", "mparams", "x"]
    assert bench.dump_outputs(torch, outs, str(tmp_path / "c")) == 8
    assert "sample_rows.npy" not in os.listdir(tmp_path / "c")
    assert np.load(tmp_path / "c" / "calls.npy").shape == (8, 2)
    # an empty block (a rank of a strong-scaling run with fewer problems than ranks) writes nothing
    outs = bench.step_outputs(wc, {k: v[:0] for k, v in dc.items()})
    assert bench.dump_outputs(torch, outs, str(tmp_path / "e")) == 0 and os.listdir(tmp_path / "e") == []


def test_ncu_traffic_record_applies_only_to_its_sources(monkeypatch):
    """roofline.traffic is taken from profiles/r2_traffic.json only when that record was captured from the CUDA sources
    being run (digest of socp_b200/csrc) and on the workload being run.  The record carries a measured figure for the
    kernels of the Broyden and Jacobian phases; from any other sources bench.py reports no traffic and says why."""
    import json
    import bench
    with open(bench.TRAFFIC_FILE) as f:
        t = json.load(f)
    for name in ("hybrd_chain_kernel", "hybrd_qpass_kernel", "hybrd_jac_kernel"):
        k = t["kernels"][name]
        assert k["dram_bytes_per_unit"] > 1e4 and k["units"] > 100, name
    # the sources the record was captured from
    monkeypatch.setattr(bench, "source_digest", lambda: t["source_digest"])
    kernels, src = bench.ncu_traffic()
    assert kernels == t["kernels"] and "r2_traffic.json" in src
    # the record is of the Goddard batch (P = 85): it is not applied to the kernels of another workload
    assert bench.ncu_traffic("goddard_warm", 85)[0] == kernels
    other, why = bench.ncu_traffic("covid19", 160)
    assert other == {} and "not of this one" in why
    # the sources being run: the record applies only if it was captured from them
    monkeypatch.undo()
    now, why = bench.ncu_traffic()
    if bench.source_digest() == t["source_digest"]:
        assert now == kernels
    else:
        assert now == {} and "from other sources" in why
