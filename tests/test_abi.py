"""The C-ABI library loads and exports every symbol include/socp_b200.h declares (no compute
calls here: this runs without a GPU), and refuses to work without a device."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "socp_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(socp_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from socp_b200 import _lib, build
    build.build()
    L = ctypes.CDLL(_lib.SO_PATH)
    syms = header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(L, s), "missing symbol " + s
    assert sorted(_lib.SYMBOLS) == syms


def test_static_facts():
    import socp_b200 as sb
    assert [sb.model_dim(m) for m in range(5)] == [7, 6, 4, 6, 6]
    assert [sb.default_steps(m) for m in range(5)] == [10, 30, 1000, 100, 50]
    import scenarios as S
    for m in range(5):
        assert list(sb.default_params(m)) == pytest.approx(S.DEFAULTS[m])
        assert sb.PARAM_NAMES[m] == S.PARAMS[m]
        assert sb.model_nparams(m) == len(S.DEFAULTS[m])
    # the caller's trace buffer is sized from these: a row is model::Trace (t, X, controls, H, extra), 2 dim + nctrl + 3
    from socp_b200 import _lib
    L = _lib.lib()
    assert [L.socp_trace_width(m) for m in range(5)] == [20, 18, 12, 18, 17]
    # one integration of S steps gives S + 1 rows; the interceptor's trace has two stages
    assert L.socp_trace_max_rows(sb.INTERCEPTOR, 10) == 22
    assert L.socp_trace_max_rows(sb.GODDARD, 10) == 11
    mode_t, mode_X = sb.default_modes(sb.GODDARD, 6, sb.FREE, S.GODDARD_MODE_XF)
    assert sb.num_param(sb.make_shape(sb.GODDARD, 6, mode_t, mode_X)) == 85


def test_no_cpu_fallback():
    """Without a CUDA device the engine must fail loudly instead of computing on the CPU."""
    import torch
    import socp_b200 as sb
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(sb.SocpError):
        sb.Engine(0)


def test_product_does_not_touch_the_oracle():
    """Only tests/, bench.py and __graft_entry__.smoke() may use oracle/."""
    pkg = os.path.join(ROOT, "socp_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".inl", ".h", ".hpp", ".cpp")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("the oracle", "").lower() or f == "models.cuh" and "oracle/" not in src, f
