"""Python host over the C ABI (include/socp_b200.h): one `Engine` per GPU.

Arrays may be numpy arrays (host buffers: the library stages H2D/D2H itself) or torch CUDA
tensors (device buffers: passed by pointer, stream-ordered on the engine's stream).
PyTorch is only plumbing here (device memory / streams); all computation happens in
libsocp_b200.so.  There is no CPU path: constructing an Engine without a GPU raises.
"""
import ctypes

import numpy as np

from . import _lib
from ._lib import DEVICE, HOST, Shape, SocpError, Stats

GODDARD, DOUBLE_INTEGRATOR, COVID19, VTOL_UAV, INTERCEPTOR = range(5)
FIXED, FREE, CONTINUOUS = 0, 1, 2
MODEL_NAMES = ["goddard", "doubleIntegrator", "covid19", "vtolUAV", "interceptor"]
PARAM_NAMES = {
    GODDARD: ["C", "b", "KD", "kr", "u_max", "mu1", "mu2", "singularControl"],
    DOUBLE_INTEGRATOR: ["u_max", "a_max", "muT"],
    COVID19: ["R0", "Tinf", "Tinc", "N", "Imax", "muI", "umin", "umax"],
    VTOL_UAV: ["u_max", "a_max", "alphaT", "alphaV", "invSigmaXwp", "Vd", "ca", "nWP_tot", "nWP",
               "phiObs", "psiWP", "muObs", "sigmaWP"],
    INTERCEPTOR: ["c0", "hr", "d0", "eta", "propellant_mass", "empty_mass", "q", "ve", "alpha_max",
                  "u_max", "a_max", "r_2p", "t_2p", "mu_gft", "muT", "muV", "muC"],
}


def model_dim(model_id):
    return _lib.lib().socp_model_dim(model_id)


def model_nparams(model_id):
    return _lib.lib().socp_model_nparams(model_id)


def default_steps(model_id):
    return _lib.lib().socp_model_default_steps(model_id)


def default_params(model_id):
    out = np.zeros(model_nparams(model_id))
    _lib.lib().socp_model_default_params(model_id, out.ctypes.data)
    return out


def make_shape(model_id, num_multi, mode_t, mode_X, step_nbr=0, ode_tol=0.0):
    """shooting::SetMode(mode_t, mode_X) (shooting.cpp:185-199) as a plain struct.  ode_tol > 0 selects
    the adaptive Dormand-Prince integrator of the reference's Boost build (abs = rel = ode_tol)."""
    s = Shape()
    s.integrator, s.ode_tol = (1, float(ode_tol)) if ode_tol and ode_tol > 0 else (0, 0.0)
    s.model_id, s.num_multi, s.step_nbr = int(model_id), int(num_multi), int(step_nbr or 0)
    dim = model_dim(model_id)
    if len(mode_t) != num_multi + 1 or len(mode_X) != num_multi + 1:
        raise ValueError("mode_t / mode_X need numMulti+1 entries")
    for i in range(num_multi + 1):
        s.mode_t[i] = int(mode_t[i])
        for j in range(dim):
            s.mode_X[i][j] = int(mode_X[i][j])
    return s


def default_modes(model_id, num_multi, mode_tf, mode_Xf):
    """shooting::SetMode(mode_tf, mode_Xf) (shooting.cpp:165-182)."""
    n = model_dim(model_id)
    mode_t = [FIXED] + [CONTINUOUS] * (num_multi - 1) + [int(mode_tf)]
    mode_X = [[FIXED] * n] + [[CONTINUOUS] * n for _ in range(num_multi - 1)] + [list(mode_Xf)]
    return mode_t, mode_X


def num_param(shape):
    return _lib.lib().socp_num_param(ctypes.byref(shape))


def unknowns_from_nodes(shape, vt, vX):
    """shooting::InitShooting(vt, vX) (shooting.cpp:88-114) for B problems of one shape: the unknowns x[B][P] (the
    M node blocks vX[:, :M], then the FREE node times in node order) and the boundary / waypoint states
    Xb = vX[..., :dim].  vt is [B][M+1], vX [B][M+1][2dim]; numpy arrays give numpy results, torch tensors give
    tensors on the same device (no copy through the host).  The node times of the new problem are vt itself."""
    M, dim = shape.num_multi, model_dim(shape.model_id)
    N = 2 * dim
    free = [j for j in range(M + 1) if shape.mode_t[j] == FREE]
    if tuple(vX.shape[1:]) != (M + 1, N) or tuple(vt.shape[1:]) != (M + 1,) or vt.shape[0] != vX.shape[0]:
        raise ValueError("vt must be [B][%d] and vX [B][%d][%d]" % (M + 1, M + 1, N))
    B = vX.shape[0]
    if _is_torch(vX):
        import torch
        x = torch.cat([vX[:, :M].reshape(B, M * N), vt[:, free]], dim=1)
        return x, vX[..., :dim].contiguous()
    vt, vX = np.asarray(vt, dtype=np.float64), np.asarray(vX, dtype=np.float64)
    x = np.concatenate([vX[:, :M].reshape(B, M * N), vt[:, free]], axis=1)
    return x, np.ascontiguousarray(vX[..., :dim])


def _is_torch(a):
    return a is not None and type(a).__module__.startswith("torch")


class _Arg:
    """Resolve an array argument to (pointer, keepalive) for host or device memory.  Device tensors are
    checked before their pointer crosses the C ABI (dtype, contiguity, device): the library reinterprets
    the memory as float64 / int32 on the engine's GPU."""

    def __init__(self, mem, device=None):
        self.mem = mem
        self.device = device
        self.keep = []

    def _device_ptr(self, a, dtype):
        import torch
        want = {np.float64: torch.float64, np.int32: torch.int32}[dtype]
        if not _is_torch(a) or not a.is_cuda:
            raise ValueError("device mode needs torch CUDA tensors for every array argument")
        if a.dtype != want:
            raise ValueError("device tensor has dtype %s, the library reads %s" % (a.dtype, want))
        if not a.is_contiguous():
            raise ValueError("device tensors must be contiguous")
        if self.device is not None and a.device.index != self.device:
            raise ValueError("tensor lives on cuda:%s, the engine on cuda:%s" % (a.device.index, self.device))
        return ctypes.c_void_p(a.data_ptr())

    def inp(self, a, dtype=np.float64):
        if a is None:
            return None
        if self.mem == DEVICE:
            return self._device_ptr(a, dtype)
        arr = np.ascontiguousarray(a, dtype=dtype)
        self.keep.append(arr)
        return ctypes.c_void_p(arr.ctypes.data)

    def out(self, a, dtype=np.float64):
        if a is None:
            return None
        if self.mem == DEVICE:
            return self._device_ptr(a, dtype)
        if not (isinstance(a, np.ndarray) and a.flags["C_CONTIGUOUS"] and a.dtype == np.dtype(dtype)):
            raise ValueError("output buffers must be contiguous numpy arrays of dtype %s" % np.dtype(dtype))
        return ctypes.c_void_p(a.ctypes.data)


class Engine:
    """One socp_ctx: a GPU, a stream, a workspace."""

    def __init__(self, device=0):
        self._L = _lib.lib()
        h = ctypes.c_void_p()
        rc = self._L.socp_create(int(device), ctypes.byref(h))
        if rc != 0:
            raise SocpError("socp_create failed: %s" % self._L.socp_last_error(None).decode())
        self._h = h
        self.device = int(device)
        self._bound_stream = None

    def close(self):
        if getattr(self, "_h", None):
            self._L.socp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise SocpError("libsocp_b200 error %d: %s" % (rc, self._L.socp_last_error(self._h).decode()))

    # -- plumbing -------------------------------------------------------------------------------
    def use_torch_stream(self):
        """Run on torch's current stream of the engine's device.  DEVICE-mode calls do this by themselves
        (see _arg), so tensors produced on torch's stream are ordered before the library reads them."""
        import torch
        st = torch.cuda.current_stream(self.device).cuda_stream
        if st != self._bound_stream:
            self._check(self._L.socp_set_stream(self._h, ctypes.c_void_p(st)))
            self._bound_stream = st

    def _arg(self, mem):
        """Argument resolver of one call.  In DEVICE mode the engine first binds to torch's CURRENT stream:
        the library then reads and writes the tensors in stream order with whatever produced them."""
        if mem == DEVICE:
            self.use_torch_stream()
        return _Arg(mem, self.device)

    def sync(self):
        self._check(self._L.socp_sync(self._h))

    def stats(self):
        s = Stats()
        self._check(self._L.socp_get_stats(self._h, ctypes.byref(s)))
        return dict(rk4_steps=s.rk4_steps, kernel_launches=s.kernel_launches,
                    solver_rounds=s.solver_rounds, device_bytes=s.device_bytes,
                    integrate_ms=s.integrate_ms, integrate_launches=s.integrate_launches,
                    advance_ms=s.advance_ms, advance_launches=s.advance_launches, assemble_ms=s.assemble_ms, jac_ms=s.jac_ms, iterations=s.iterations, jac_evals=s.jac_evals,
                    dopri_steps=s.dopri_steps, qpass_ms=s.qpass_ms, res_evals=s.res_evals,
                    res_ms=s.advance_ms - s.jac_ms)

    def set_profiling(self, on=True):
        self._check(self._L.socp_set_profiling(self._h, int(bool(on))))

    def reset_stats(self):
        self._check(self._L.socp_reset_stats(self._h))

    def timer_start(self):
        self._check(self._L.socp_timer_start(self._h))

    def timer_stop(self):
        ms = ctypes.c_float()
        self._check(self._L.socp_timer_stop(self._h, ctypes.byref(ms)))
        return ms.value

    def measure_fp64_peak(self):
        g, c = ctypes.c_double(), ctypes.c_double()
        self._check(self._L.socp_measure_fp64_peak(self._h, ctypes.byref(g), ctypes.byref(c)))
        return g.value, c.value

    def set_obstacles(self, types, pos, rad):
        t = np.ascontiguousarray(types, dtype=np.float64)
        p = np.ascontiguousarray(pos, dtype=np.float64)
        r = np.ascontiguousarray(rad, dtype=np.float64)
        self._check(self._L.socp_set_obstacles(self._h, t.size, t.ctypes.data, p.ctypes.data, r.ctypes.data))

    @staticmethod
    def _mem(*arrays):
        return DEVICE if any(_is_torch(a) for a in arrays) else HOST

    @staticmethod
    def _bcast_params(mparams, B, np_):
        if _is_torch(mparams):
            return mparams
        m = np.asarray(mparams, dtype=np.float64)
        if m.ndim == 1:
            m = np.tile(m, (B, 1))
        if m.shape != (B, np_):
            raise ValueError("mparams must be [B][%d]" % np_)
        return m

    # -- hot path -------------------------------------------------------------------------------
    def traj_batch(self, model_id, mparams, t0, X0, tf, step_nbr=0, sw=None, out=None):
        """model::ComputeTraj for B trajectories (socp_traj_batch)."""
        mem = self._mem(X0)
        B = X0.shape[0]
        N = 2 * model_dim(model_id)
        if mem == HOST:
            mparams = self._bcast_params(mparams, B, model_nparams(model_id))
            t0 = np.broadcast_to(np.asarray(t0, dtype=np.float64), (B,))
            tf = np.broadcast_to(np.asarray(tf, dtype=np.float64), (B,))
            if out is None:
                out = np.empty((B, N))
        elif out is None:
            import torch
            out = torch.empty_like(X0)
        a = self._arg(mem)
        self._check(self._L.socp_traj_batch(self._h, model_id, int(step_nbr or 0), B, a.inp(mparams), a.inp(sw),
                                            a.inp(t0), a.inp(tf), a.inp(X0), a.out(out), mem))
        return out

    def traj_adaptive_batch(self, model_id, mparams, t0, X0, tf, tol, step_nbr=0, sw=None):
        """ComputeTraj with the adaptive Dormand-Prince integrator (socp_traj_adaptive_batch); host arrays.
        Returns (Xf[B][N], nsteps[B][2] = accepted steps, rejected attempts)."""
        X0 = np.ascontiguousarray(X0, dtype=np.float64)
        B, N = X0.shape
        mparams = self._bcast_params(mparams, B, model_nparams(model_id))
        t0 = np.broadcast_to(np.asarray(t0, dtype=np.float64), (B,))
        tf = np.broadcast_to(np.asarray(tf, dtype=np.float64), (B,))
        Xf, ns = np.empty((B, N)), np.zeros((B, 2), dtype=np.int32)
        a = _Arg(HOST)
        self._check(self._L.socp_traj_adaptive_batch(self._h, model_id, int(step_nbr or 0), B, a.inp(mparams), a.inp(sw),
                                                     a.inp(t0), a.inp(tf), a.inp(X0), float(tol), a.out(Xf), a.out(ns, np.int32), HOST))
        return Xf, ns

    def trace_batch(self, model_id, mparams, t0, X0, tf, step_nbr=0, sw=None):
        """The observer form of ComputeTraj (socp_trace_batch): rows[B][R][W] = {t, X, control, H, extra}
        as model::Trace writes them (model.hpp:446-462), nrows[B], Xf[B][N].  Host arrays."""
        X0 = np.ascontiguousarray(X0, dtype=np.float64)
        B, N = X0.shape
        mparams = self._bcast_params(mparams, B, model_nparams(model_id))
        t0 = np.broadcast_to(np.asarray(t0, dtype=np.float64), (B,))
        tf = np.broadcast_to(np.asarray(tf, dtype=np.float64), (B,))
        W = self._L.socp_trace_width(model_id)
        R = self._L.socp_trace_max_rows(model_id, int(step_nbr or 0))
        rows, nrows, Xf = np.zeros((B, R, W)), np.zeros(B, dtype=np.int32), np.empty((B, N))
        a = _Arg(HOST)
        self._check(self._L.socp_trace_batch(self._h, model_id, int(step_nbr or 0), B, a.inp(mparams), a.inp(sw),
                                             a.inp(t0), a.inp(tf), a.inp(X0), a.out(rows), a.out(nrows, np.int32), a.out(Xf), HOST))
        return rows, nrows, Xf

    def point_batch(self, model_id, mparams, t, X, sw=None, chart_stage=None):
        """odeTools::Model, model::Control, model::Hamiltonian at B points (host arrays)."""
        X = np.ascontiguousarray(X, dtype=np.float64)
        B, N = X.shape
        mparams = self._bcast_params(mparams, B, model_nparams(model_id))
        t = np.broadcast_to(np.asarray(t, dtype=np.float64), (B,))
        rhs, ctl, H = np.empty((B, N)), np.empty((B, 4)), np.empty(B)
        a = _Arg(HOST)
        self._check(self._L.socp_point_batch(self._h, model_id, B, a.inp(mparams), a.inp(sw),
                                             a.inp(chart_stage, np.int32), a.inp(t), a.inp(X), a.out(rhs),
                                             a.out(ctl), a.out(H), HOST))
        return rhs, ctl, H

    def _problem_args(self, shape, mparams, time, Xb, x):
        mem = self._mem(x)
        B = x.shape[0]
        if mem == HOST:
            mparams = self._bcast_params(mparams, B, model_nparams(shape.model_id))
        return mem, B, mparams

    def residual_batch(self, shape, mparams, time, Xb, x, out=None):
        """shooting::ShootingFunction for B problems (socp_residual_batch)."""
        mem, B, mparams = self._problem_args(shape, mparams, time, Xb, x)
        P = num_param(shape)
        if out is None:
            if mem == HOST:
                out = np.empty((B, P))
            else:
                import torch
                out = torch.empty_like(x)
        a = self._arg(mem)
        self._check(self._L.socp_residual_batch(self._h, ctypes.byref(shape), B, a.inp(mparams), a.inp(time),
                                                a.inp(Xb), a.inp(x), a.out(out), mem))
        return out

    def fdjac_batch(self, shape, mparams, time, Xb, x, epsfcn=1e-15, out=None):
        """MINPACK fdjac1 on the shooting residual; returns [B][P][P] with J[b, i, j] = dF_i/dx_j."""
        mem, B, mparams = self._problem_args(shape, mparams, time, Xb, x)
        P = num_param(shape)
        if mem != HOST:
            raise ValueError("fdjac_batch takes host arrays")
        buf = np.empty((B, P * P))
        a = _Arg(mem)
        self._check(self._L.socp_fdjac_batch(self._h, ctypes.byref(shape), B, a.inp(mparams), a.inp(time),
                                             a.inp(Xb), a.inp(x), float(epsfcn), a.out(buf), mem))
        return buf.reshape(B, P, P).transpose(0, 2, 1).copy()

    def solve_batch(self, shape, mparams, time, Xb, x, xtol=1e-8, maxfev=10000, info=None, nfev=None,
                    fnorm=None):
        """shooting::SolveShootingFunction for B problems; x is updated in place."""
        mem, B, mparams = self._problem_args(shape, mparams, time, Xb, x)
        if mem == HOST:
            if not (isinstance(x, np.ndarray) and x.dtype == np.float64 and x.flags["C_CONTIGUOUS"]):
                raise ValueError("x must be a contiguous float64 array (updated in place)")
            info = np.empty(B, dtype=np.int32) if info is None else info
            nfev = np.empty(B, dtype=np.int32) if nfev is None else nfev
            fnorm = np.empty(B) if fnorm is None else fnorm
        else:
            import torch
            info = torch.empty(B, dtype=torch.int32, device=x.device) if info is None else info
            nfev = torch.empty(B, dtype=torch.int32, device=x.device) if nfev is None else nfev
            fnorm = torch.empty(B, dtype=torch.float64, device=x.device) if fnorm is None else fnorm
        a = self._arg(mem)
        self._check(self._L.socp_solve_batch(self._h, ctypes.byref(shape), B, a.inp(mparams), a.inp(time),
                                             a.inp(Xb), a.out(x), float(xtol), int(maxfev), a.out(info, np.int32),
                                             a.out(nfev, np.int32), a.out(fnorm), mem))
        return dict(x=x, info=info, nfev=nfev, fnorm=fnorm)

    def move_batch(self, shape, mparams, time, x, tq, out=None):
        """shooting::Move(tf) of B solutions x at Q times each (socp_move_batch): tq [B][Q] (host arrays: a [Q]
        vector is shared by every problem); returns Xq [B][Q][2dim].  A time outside [t0, t_end] gives the
        state at t_end, as in the reference."""
        mem, B, mparams = self._problem_args(shape, mparams, time, None, x)
        N = 2 * model_dim(shape.model_id)
        if mem == HOST:
            tq = np.asarray(tq, dtype=np.float64)
            tq = np.ascontiguousarray(np.broadcast_to(tq, (B, tq.shape[-1])) if tq.ndim == 1 else tq)
            Q = tq.shape[1]
            if out is None:
                out = np.empty((B, Q, N))
        else:
            Q = tq.shape[1]
            if out is None:
                import torch
                out = torch.empty((B, Q, N), dtype=torch.float64, device=x.device)
        if tuple(tq.shape) != (B, Q):
            raise ValueError("tq must be [B][Q]")
        a = self._arg(mem)
        self._check(self._L.socp_move_batch(self._h, ctypes.byref(shape), B, a.inp(mparams), a.inp(time), a.inp(x),
                                            int(Q), a.inp(tq), a.out(out), mem))
        return out

    def solution_batch(self, shape, mparams, time, x):
        """shooting::GetSolution for B solutions (socp_solution_batch): returns (vt [B][M+1], vX [B][M+1][2dim]),
        vX[:, M] = Move(t_end).  Numpy arrays or torch CUDA tensors, like solve_batch."""
        mem, B, mparams = self._problem_args(shape, mparams, time, None, x)
        M, N = shape.num_multi, 2 * model_dim(shape.model_id)
        if mem == HOST:
            vt, vX = np.empty((B, M + 1)), np.empty((B, M + 1, N))
        else:
            import torch
            vt = torch.empty((B, M + 1), dtype=torch.float64, device=x.device)
            vX = torch.empty((B, M + 1, N), dtype=torch.float64, device=x.device)
        a = self._arg(mem)
        self._check(self._L.socp_solution_batch(self._h, ctypes.byref(shape), B, a.inp(mparams), a.inp(time), a.inp(x),
                                                a.out(vt), a.out(vX), mem))
        return vt, vX

    def solution_trace_batch(self, shape, mparams, time, x):
        """shooting::Trace for B solutions (socp_solution_trace_batch): returns (rows [B][M][R][W], nrows [B][M]),
        rows[b, j, :nrows[b, j]] = the observer rows {t, X, control, H, extra} of segment j of problem b, RK4 for
        every shape.  Numpy arrays or torch CUDA tensors, like solution_batch."""
        mem, B, mparams = self._problem_args(shape, mparams, time, None, x)
        M = shape.num_multi
        W = self._L.socp_trace_width(shape.model_id)
        R = self._L.socp_trace_max_rows(shape.model_id, int(shape.step_nbr))
        if mem == HOST:
            rows, nrows = np.empty((B, M, R, W)), np.empty((B, M), dtype=np.int32)
        else:
            import torch
            rows = torch.empty((B, M, R, W), dtype=torch.float64, device=x.device)
            nrows = torch.empty((B, M), dtype=torch.int32, device=x.device)
        a = self._arg(mem)
        self._check(self._L.socp_solution_trace_batch(self._h, ctypes.byref(shape), B, a.inp(mparams), a.inp(time),
                                                      a.inp(x), a.out(rows), a.out(nrows, np.int32), mem))
        return rows, nrows

    def init_shooting_batch(self, shape, mparams, ti, Xi, tf, Xf, sw=None):
        """shooting::InitShooting(ti, Xi, tf, Xf) for B new problems of one shape (socp_init_shooting_batch): the
        uniform time grid, node 0 = Xi, node M = Xf, every interior node integrated from (ti, Xi) with the shape's
        integrator.  Xi is [B][2dim], Xf [B][dim], ti / tf [B], sw an optional [B][2] of goddard switching times.
        Returns (time [B][M+1], Xb [B][M+1][dim], x [B][P]), the problem inputs of solve_batch.  Numpy arrays give numpy
        results (scalar ti / tf and a 1-D mparams are broadcast); torch CUDA tensors give tensors on their device."""
        M, dim, P = shape.num_multi, model_dim(shape.model_id), num_param(shape)
        if P < 0:
            raise ValueError("bad shape (model id / numMulti)")
        mem = self._mem(Xi)
        B = Xi.shape[0]
        if mem == HOST:
            Xi, Xf = np.asarray(Xi, dtype=np.float64), np.asarray(Xf, dtype=np.float64)
            mparams = self._bcast_params(mparams, B, model_nparams(shape.model_id))
            ti = np.broadcast_to(np.asarray(ti, dtype=np.float64), (B,))
            tf = np.broadcast_to(np.asarray(tf, dtype=np.float64), (B,))
            time, Xb, x = np.empty((B, M + 1)), np.empty((B, M + 1, dim)), np.empty((B, P))
        else:
            import torch
            time = torch.empty((B, M + 1), dtype=torch.float64, device=Xi.device)
            Xb = torch.empty((B, M + 1, dim), dtype=torch.float64, device=Xi.device)
            x = torch.empty((B, P), dtype=torch.float64, device=Xi.device)
        if tuple(Xi.shape) != (B, 2 * dim) or tuple(Xf.shape) != (B, dim):
            raise ValueError("Xi must be [B][%d] and Xf [B][%d]" % (2 * dim, dim))
        a = self._arg(mem)
        self._check(self._L.socp_init_shooting_batch(self._h, ctypes.byref(shape), B, a.inp(mparams), a.inp(sw), a.inp(ti),
                                                     a.inp(Xi), a.inp(tf), a.inp(Xf), a.out(time), a.out(Xb), a.out(x), mem))
        return time, Xb, x

    # -- analytic-Jacobian path (modelOrder == 1; the double integrator, as in the reference) -----
    def traj_var_batch(self, model_id, mparams, t0, X0, tf, step_nbr=0):
        """model::ComputeTraj(isJac = 1) for B extended states [(2dim+1) 2dim] (host arrays)."""
        X0 = np.ascontiguousarray(X0, dtype=np.float64)
        B = X0.shape[0]
        mparams = self._bcast_params(mparams, B, model_nparams(model_id))
        t0 = np.broadcast_to(np.asarray(t0, dtype=np.float64), (B,))
        tf = np.broadcast_to(np.asarray(tf, dtype=np.float64), (B,))
        out = np.empty_like(X0)
        a = _Arg(HOST)
        self._check(self._L.socp_traj_var_batch(self._h, model_id, int(step_nbr or 0), B, a.inp(mparams), a.inp(t0),
                                                a.inp(tf), a.inp(X0), a.out(out), HOST))
        return out

    def jacobian_batch(self, shape, mparams, time, Xb, x):
        """shooting::ShootingFunctionJacobian; returns [B][P][P] with J[b, i, j] = dF_i/dx_j (host arrays)."""
        mem, B, mparams = self._problem_args(shape, mparams, time, Xb, x)
        P = num_param(shape)
        buf = np.empty((B, P * P))
        a = _Arg(HOST)
        self._check(self._L.socp_jacobian_batch(self._h, ctypes.byref(shape), B, a.inp(mparams), a.inp(time),
                                                a.inp(Xb), a.inp(x), a.out(buf), HOST))
        return buf.reshape(B, P, P).transpose(0, 2, 1).copy()

    def solve_hybrj_batch(self, shape, mparams, time, Xb, x, xtol=1e-8, maxfev=10000):
        """shooting::SolveShootingFunction with modelOrder == 1 (hybrj); x updated in place (host arrays)."""
        mem, B, mparams = self._problem_args(shape, mparams, time, Xb, x)
        if not (isinstance(x, np.ndarray) and x.dtype == np.float64 and x.flags["C_CONTIGUOUS"]):
            raise ValueError("x must be a contiguous float64 array (updated in place)")
        info, nfev, njev = (np.empty(B, dtype=np.int32) for _ in range(3))
        fnorm = np.empty(B)
        a = _Arg(HOST)
        self._check(self._L.socp_solve_hybrj_batch(self._h, ctypes.byref(shape), B, a.inp(mparams), a.inp(time),
                                                   a.inp(Xb), a.out(x), float(xtol), int(maxfev), a.out(info, np.int32),
                                                   a.out(nfev, np.int32), a.out(njev, np.int32), a.out(fnorm), HOST))
        return dict(x=x, info=info, nfev=nfev, njev=njev, fnorm=fnorm)

    def continuation_param_batch(self, shape, mparams, time, Xb, x, step, param_idx, goal, xtol=1e-8,
                                 maxfev=10000, step_min=1e-12, info=None, calls=None):
        """shooting::SolveShootingContinuation(step, Rdata, Rgoal) for B problems.
        Host arrays: works on copies, returns dict(x, info, calls, mparams).  Torch CUDA tensors: x and mparams are
        updated IN PLACE on the device (goal, info, calls are device tensors too; info/calls are created when None)
        and no problem data crosses PCIe."""
        B = x.shape[0]
        mem = self._mem(x)
        if mem == HOST:
            mparams = np.ascontiguousarray(self._bcast_params(mparams, B, model_nparams(shape.model_id))).copy()
            x = np.ascontiguousarray(x, dtype=np.float64).copy()
            goal = np.ascontiguousarray(np.broadcast_to(np.asarray(goal, dtype=np.float64), (B,)))
            info = np.empty(B, dtype=np.int32)
            calls = np.empty((B, 2), dtype=np.int32)
        else:
            import torch
            info = torch.empty(B, dtype=torch.int32, device=x.device) if info is None else info
            calls = torch.empty((B, 2), dtype=torch.int32, device=x.device) if calls is None else calls
        a = self._arg(mem)
        self._check(self._L.socp_continuation_param_batch(
            self._h, ctypes.byref(shape), B, a.out(mparams), a.inp(time), a.inp(Xb), a.out(x), float(xtol),
            int(maxfev), float(step), int(param_idx), a.inp(goal), float(step_min), a.out(info, np.int32),
            a.out(calls, np.int32), mem))
        return dict(x=x, info=info, calls=calls, mparams=mparams)

    def continuation_boundary_batch(self, shape, mparams, time_prec, Xb_prec, time_des, Xb_des, x, step,
                                    xtol=1e-8, maxfev=10000, step_min=1e-12, info=None, calls=None):
        """shooting::SolveShootingContinuation(step) on the boundary data for B problems (host arrays: works on a
        copy of x; torch CUDA tensors: x updated in place on the device)."""
        B = x.shape[0]
        mem = self._mem(x)
        if mem == HOST:
            mparams = self._bcast_params(mparams, B, model_nparams(shape.model_id))
            x = np.ascontiguousarray(x, dtype=np.float64).copy()
            info = np.empty(B, dtype=np.int32)
            calls = np.empty((B, 2), dtype=np.int32)
        else:
            import torch
            info = torch.empty(B, dtype=torch.int32, device=x.device) if info is None else info
            calls = torch.empty((B, 2), dtype=torch.int32, device=x.device) if calls is None else calls
        a = self._arg(mem)
        self._check(self._L.socp_continuation_boundary_batch(
            self._h, ctypes.byref(shape), B, a.inp(mparams), a.inp(time_prec), a.inp(Xb_prec),
            a.inp(time_des), a.inp(Xb_des), a.out(x), float(xtol), int(maxfev), float(step),
            float(step_min), a.out(info, np.int32), a.out(calls, np.int32), mem))
        return dict(x=x, info=info, calls=calls)
