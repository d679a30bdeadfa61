"""Host side of re-meshing a batch (no GPU needed): unknowns_from_nodes restates shooting::InitShooting(vt, vX)
(guess_from_nodes, cpp/src/socp/shooting.cpp:88-114) for a whole batch, and the C++ mirror with Move /
GetSolution / Resize and the Goddard pipeline demo builds and links."""
import os
import subprocess

import numpy as np
import pytest

import scenarios as S
from golden_util import by_name, spec_from_hex

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CPP = os.path.join(ROOT, "cpp")


@pytest.fixture(scope="module")
def sb():
    from socp_b200 import build
    build.build()
    import socp_b200
    return socp_b200


def nodes(B, M, N):
    """vt[b][i] and vX[b][i][k] that name their own position"""
    vt = np.array([[b + 0.125 * i for i in range(M + 1)] for b in range(B)])
    vX = np.array([[[1000.0 * b + 10.0 * i + k for k in range(N)] for i in range(M + 1)] for b in range(B)])
    return vt, vX


def test_free_interior_times_reproduce_golden_stage4(sb):
    """The stage-4 Goddard unknowns of tests/golden/make_golden.py: the six node blocks, then vt[2], vt[4], vt[6]."""
    spec = spec_from_hex(by_name("solve", "goddard_stage4_singular")["spec"])
    shape = sb.make_shape(spec["model"], spec["M"], spec["mode_t"], spec["mode_X"], spec["steps"])
    x0, Xb = np.array(spec["x0"]), np.array(spec["Xb"])
    vX = np.zeros((1, 7, 14))
    vX[0, :6] = x0[:84].reshape(6, 14)
    vX[0, 6, :7] = Xb[6]
    vX[0, 6, 7:] = np.nan                      # the last node's costate is not an unknown
    x, Xb_out = sb.unknowns_from_nodes(shape, np.array([spec["time"]]), vX)
    assert x.shape == (1, 87) and np.array_equal(x[0], x0)
    assert np.array_equal(Xb_out[0, :6], vX[0, :6, :7]) and np.array_equal(Xb_out[0, 6], Xb[6])


@pytest.mark.parametrize("mode_t", [
    [S.FIXED, S.CONTINUOUS, S.CONTINUOUS, S.FIXED],                 # no free time
    [S.FIXED, S.FREE, S.CONTINUOUS, S.FREE],                        # free interior and final times
    [S.FREE, S.CONTINUOUS, S.FIXED, S.CONTINUOUS, S.FREE],          # free t0, continuous nodes on both sides
])
def test_unknowns_from_nodes(sb, mode_t):
    M, dim = len(mode_t) - 1, 4
    N = 2 * dim
    mode_X = [[S.FIXED] * dim] + [[S.CONTINUOUS] * dim] * (M - 1) + [[S.FIXED] * dim]
    shape = sb.make_shape(sb.COVID19, M, mode_t, mode_X)
    B = 3
    vt, vX = nodes(B, M, N)
    x, Xb = sb.unknowns_from_nodes(shape, vt, vX)
    free = [j for j in range(M + 1) if mode_t[j] == S.FREE]
    assert x.shape == (B, sb.num_param(shape)) == (B, N * M + len(free))
    for b in range(B):
        # guess_from_nodes: param[j N + i] = X[j][i] for j < M, then the FREE node times in node order
        for j in range(M):
            for i in range(N):
                assert x[b, j * N + i] == 1000.0 * b + 10.0 * j + i
        assert list(x[b, N * M:]) == [b + 0.125 * j for j in free]
        assert np.array_equal(Xb[b], vX[b, :, :dim])
    assert Xb.flags["C_CONTIGUOUS"] and x.flags["C_CONTIGUOUS"]
    # torch tensors give tensors with the same values
    import torch
    xt, Xbt = sb.unknowns_from_nodes(shape, torch.from_numpy(vt), torch.from_numpy(vX))
    assert torch.is_tensor(xt) and np.array_equal(xt.numpy(), x) and np.array_equal(Xbt.numpy(), Xb)
    assert Xbt.is_contiguous() and xt.is_contiguous()


def test_unknowns_from_nodes_checks_shapes(sb):
    mode_t, mode_X = sb.default_modes(sb.COVID19, 2, S.FIXED, [S.FIXED] * 4)
    shape = sb.make_shape(sb.COVID19, 2, mode_t, mode_X)
    vt, vX = nodes(2, 2, 8)
    with pytest.raises(ValueError):
        sb.unknowns_from_nodes(shape, vt, vX[:, :2])
    with pytest.raises(ValueError):
        sb.unknowns_from_nodes(shape, vt[:1], vX)
    with pytest.raises(ValueError):
        sb.unknowns_from_nodes(shape, vt, vX[..., :4])


def test_mirror_builds_with_pipeline_demo(sb):
    subprocess.check_call(["make", "-s", "-C", CPP])
    demo = os.path.join(CPP, "build", "bin", "demo_goddard_pipeline")
    assert os.access(demo, os.X_OK)
    out = subprocess.run(["ldd", demo], capture_output=True, text=True).stdout
    assert "libsocp_host.so" in out and "libsocp_b200.so" in out and "not found" not in out
    syms = subprocess.run(["nm", "-D", "--undefined-only", os.path.join(CPP, "build", "libsocp_host.so")],
                          capture_output=True, text=True).stdout
    for s in ("socp_move_batch", "socp_solution_batch"):
        assert s in syms, s
