"""socp_b200 -- B200-native batched shooting engine for the hot path of bherisse/socp.

Python host over libsocp_b200.so (hand-written sm_100a CUDA behind a C ABI, include/socp_b200.h).
"""
from .engine import (Engine, SocpError, make_shape, default_modes, num_param, model_dim, model_nparams,  # noqa: F401
                     default_steps, default_params, unknowns_from_nodes, PARAM_NAMES, MODEL_NAMES,
                     GODDARD, DOUBLE_INTEGRATOR, COVID19, VTOL_UAV, INTERCEPTOR, FIXED, FREE, CONTINUOUS)
