// socp_b200/csrc/integrate.cuh -- fixed-step RK4 on registers, one thread per trajectory.
//
// Restates odeTools::RK4 (/root/reference/src/socp/odeTools.cpp:89-98), odeTools::integrate
// (:128-146, non-Boost branch), model::ModelInt (src/socp/model.hpp:395-414) and
// interceptor::ComputeTraj / ModelInt (src/models/interceptor/interceptor.cpp:165-220, :104-130).
// The state/costate vector, the stage slopes and the model constants stay in registers for the
// whole segment; nothing is written until the end point.
#pragma once
#include "models.cuh"

namespace socp {

// ---- cooperative thread groups (north_star (1): "a warp-cooperative group for wider models such as vtolUAV") ------
// Coop<MODEL>::LANES lanes of a warp own ONE trajectory: every lane carries the whole state (the RK4 / dopri5
// algebra is replicated, it is a few dozen flops) and the expensive, separable part of the right-hand side is split
// over the lanes and combined with shuffles -- for vtolUAV the sum over the obstacles of the penalty map (27 exp per
// evaluation, 85 % of the RHS): lane q takes the obstacles i = q (mod 4).  The adaptive integrator's error norm is
// reduced the same way (each lane the components i = q (mod LANES), then a shuffle max over the group).  The results
// are bit for bit those of the one-thread-per-trajectory kernels (obstacle_eval fixes one summation order for both),
// so which kernel integrates a trajectory is purely a scheduling decision: the group form is used when the batch is
// too small to fill the GPU with one thread per trajectory (the tail of a batched solve, small batches).
template <int MODEL> struct Coop {
    static constexpr int LANES = 1;
    SOCP_DEV static void set(typename Model<MODEL>::Ctx &, int) {}
    SOCP_DEV static bool owns(const typename Model<MODEL>::Ctx &, int) { return true; }
    SOCP_DEV static double group_max(const typename Model<MODEL>::Ctx &, double v) { return v; }
};
template <> struct Coop<VTOL_UAV> {
    static constexpr int LANES = 4;
    // lane q of the group of LANES consecutive lanes of the warp that holds this thread
    SOCP_DEV static void set(Model<VTOL_UAV>::Ctx &c, int q) {
        c.coop_lanes = LANES;
        c.cq = q;
        c.cmask = ((1u << LANES) - 1u) << ((threadIdx.x & 31) & ~(LANES - 1));
    }
    SOCP_DEV static bool owns(const Model<VTOL_UAV>::Ctx &c, int i) { return c.coop_lanes == 1 || (i & (LANES - 1)) == c.cq; }
    // max over the group with MINPACK-free NaN semantics: a NaN anywhere gives NaN (the step is rejected)
    SOCP_DEV static double group_max(const Model<VTOL_UAV>::Ctx &c, double v) {
        if (c.coop_lanes == 1) return v;
#pragma unroll
        for (int off = LANES / 2; off > 0; off >>= 1) {
            const double o = __shfl_xor_sync(c.cmask, v, off);
            v = (v != v || o != o) ? nan("") : fmax(v, o);
        }
        return v;
    }
};

// One classical RK4 step with the reference's combination order
//   X <- X + (h/6) * (F1 + (F4 + 2*(F2 + F3)))          (odeTools.cpp:97)
template <int MODEL>
SOCP_DEV void rk4_step(const typename Model<MODEL>::Ctx &c, double t, double *X, double h) {
    typedef Model<MODEL> M;
    constexpr int N = M::N;
    double F1[N], F23[N], F[N], Y[N];
    const double h2 = h / 2.0;
    M::rhs(c, t, X, F1);
#pragma unroll
    for (int i = 0; i < N; ++i) Y[i] = X[i] + h2 * F1[i];
    M::rhs(c, t + h2, Y, F23);                       // F2
#pragma unroll
    for (int i = 0; i < N; ++i) Y[i] = X[i] + h2 * F23[i];
    M::rhs(c, t + h2, Y, F);                         // F3
#pragma unroll
    for (int i = 0; i < N; ++i) { F23[i] = F23[i] + F[i]; Y[i] = X[i] + h * F[i]; }
    M::rhs(c, t + h, Y, F);                          // F4
    const double h6 = h / 6.0;
#pragma unroll
    for (int i = 0; i < N; ++i) X[i] = X[i] + h6 * (F1[i] + (F[i] + 2.0 * F23[i]));
}

// What a fixed-step integration reports besides its end point: nothing (NoRows), or the observer rows of a trace
// (TraceRows, below).  Called at the start point and after every step.
struct NoRows {
    template <class C> SOCP_DEV void operator()(const C &, double, const double *) {}
};

// odeTools::integrate: `while (t < tf - dt/2)` with `t += dt` and a last-step clamp, so that
// tf <= t0 performs zero steps.  Returns the number of RK4 steps taken.
template <int MODEL, class OBS>
SOCP_DEV int integrate_fixed(const typename Model<MODEL>::Ctx &c, double *X, double t0, double tf, double dt, OBS &obs) {
    double t = t0;
    int steps = 0;
    obs(c, t, X);
    while (t < (tf - dt / 2)) {
        rk4_step<MODEL>(c, t, X, (t + dt > tf) ? tf - t : dt);     // one inlined copy of the step
        t += dt;
        ++steps;
        obs(c, t, X);
    }
    return steps;
}

// ---- adaptive Dormand-Prince 5(4): the reference's -D_USE_BOOST build -----------------------------
// odeTools.cpp:131-134: integrate_adaptive(make_dense_output<runge_kutta_dopri5>(tol, tol), model, X,
// t0, tf, dt).  Restated from the published Boost.Odeint algorithm (runge_kutta_dopri5::do_step_impl,
// default_error_checker, default_step_adjuster, integrate_adaptive for dense-output steppers); Boost is
// not available to pin against, so parity is checked against the CPU restatement of the same algorithm only.
// One thread owns the trajectory: state, the seven stage slopes and the step-size controller live in
// registers; the error norm is a max over the thread's own components.
template <int MODEL>
SOCP_DEV void dopri5_try(const typename Model<MODEL>::Ctx &c, double t, const double *in, const double *k1, double dt,
                         double *out, double *k7, double &err, double tol) {
    typedef Model<MODEL> M;
    constexpr int N = M::N;
    const double a2 = 1.0 / 5, a3 = 3.0 / 10, a4 = 4.0 / 5, a5 = 8.0 / 9;
    const double b21 = 1.0 / 5, b31 = 3.0 / 40, b32 = 9.0 / 40, b41 = 44.0 / 45, b42 = -56.0 / 15, b43 = 32.0 / 9,
                 b51 = 19372.0 / 6561, b52 = -25360.0 / 2187, b53 = 64448.0 / 6561, b54 = -212.0 / 729,
                 b61 = 9017.0 / 3168, b62 = -355.0 / 33, b63 = 46732.0 / 5247, b64 = 49.0 / 176, b65 = -5103.0 / 18656;
    const double c1 = 35.0 / 384, c3 = 500.0 / 1113, c4 = 125.0 / 192, c5 = -2187.0 / 6784, c6 = 11.0 / 84;
    const double dc1 = c1 - 5179.0 / 57600, dc3 = c3 - 7571.0 / 16695, dc4 = c4 - 393.0 / 640,
                 dc5 = c5 - (-92097.0 / 339200), dc6 = c6 - 187.0 / 2100, dc7 = -1.0 / 40;
    double k2[N], k3[N], k4[N], k5[N], k6[N], y[N];
#pragma unroll
    for (int i = 0; i < N; ++i) y[i] = in[i] + dt * b21 * k1[i];
    M::rhs(c, t + dt * a2, y, k2);
#pragma unroll
    for (int i = 0; i < N; ++i) y[i] = in[i] + dt * b31 * k1[i] + dt * b32 * k2[i];
    M::rhs(c, t + dt * a3, y, k3);
#pragma unroll
    for (int i = 0; i < N; ++i) y[i] = in[i] + dt * b41 * k1[i] + dt * b42 * k2[i] + dt * b43 * k3[i];
    M::rhs(c, t + dt * a4, y, k4);
#pragma unroll
    for (int i = 0; i < N; ++i) y[i] = in[i] + dt * b51 * k1[i] + dt * b52 * k2[i] + dt * b53 * k3[i] + dt * b54 * k4[i];
    M::rhs(c, t + dt * a5, y, k5);
#pragma unroll
    for (int i = 0; i < N; ++i)
        y[i] = in[i] + dt * b61 * k1[i] + dt * b62 * k2[i] + dt * b63 * k3[i] + dt * b64 * k4[i] + dt * b65 * k5[i];
    M::rhs(c, t + dt, y, k6);
#pragma unroll
    for (int i = 0; i < N; ++i)
        out[i] = in[i] + dt * c1 * k1[i] + dt * c3 * k3[i] + dt * c4 * k4[i] + dt * c5 * k5[i] + dt * c6 * k6[i];
    M::rhs(c, t + dt, out, k7);
    // error norm (Boost's default_error_checker: max_i |xerr_i| / (eps_abs + eps_rel (|x_i| + dt |dxdt_i|))): every lane
    // of a cooperative group takes its share of the components, a shuffle max over the group drives the step control
    err = 0.;
#pragma unroll
    for (int i = 0; i < N; ++i) {
        if (!Coop<MODEL>::owns(c, i)) continue;
        const double xe = dt * dc1 * k1[i] + dt * dc3 * k3[i] + dt * dc4 * k4[i] + dt * dc5 * k5[i] + dt * dc6 * k6[i] + dt * dc7 * k7[i];
        const double e = fabs(xe) / (tol + tol * (fabs(in[i]) + fabs(dt) * fabs(k1[i])));
        if (e > err || e != e) err = e;
    }
    err = Coop<MODEL>::group_max(c, err);
}

// returns accepted steps; rejected attempts are added to `rejected`
template <int MODEL>
SOCP_DEV int integrate_adaptive(const typename Model<MODEL>::Ctx &c, double *X, double t0, double tf, double dt, double tol,
                                int &rejected) {
    constexpr int N = Model<MODEL>::N;
    const double eps = 2.220446049250313e-16;
    double t = t0, k1[N], out[N], k7[N];
    bool have_deriv = false;
    int steps = 0;
    if (!(dt > 0.)) return 0;
    while (tf - t > eps) {
        while ((t + dt) - tf <= eps) {
            if (!have_deriv) { Model<MODEL>::rhs(c, t, X, k1); have_deriv = true; }
            int failed = 0;
            bool ok = false;
            while (!ok && failed < 500) {
                double err;
                dopri5_try<MODEL>(c, t, X, k1, dt, out, k7, err, tol);
                if (err > 1.0 || err != err) {
                    const double f = 0.9 * pow(err, -1.0 / 3.0);
                    dt *= (f > 0.2 && f == f) ? f : 0.2;
                    ++failed;
                    ++rejected;
                } else {
                    t += dt;
                    if (err < 0.5) {
                        const double e5 = 1.0 / 3125.0;          // 5^-5
                        dt *= 0.9 * pow(fmax(err, e5), -1.0 / 5.0);
                    }
                    ok = true;
                }
            }
            if (!ok) return steps;
#pragma unroll
            for (int i = 0; i < N; ++i) { X[i] = out[i]; k1[i] = k7[i]; }
            ++steps;
        }
        dt = tf - t;
        have_deriv = false;
    }
    return steps;
}

template <class OBS>
SOCP_DEV int interceptor_model_int(Model<INTERCEPTOR>::Ctx &c, double *X, double t0, double tf, int S, OBS &obs) {
    double t = t0;
    const double dt = (tf - t0) / S;
    obs(c, t, X);
    for (int i = 0; i < S; ++i) {
        Model<INTERCEPTOR>::set_chart(c, X);
        rk4_step<INTERCEPTOR>(c, t, X, dt);
        t += dt;
        obs(c, t, X);
    }
    return S;
}

// model::ComputeTraj for one segment.  For the interceptor `c.chart` / `c.stage` are updated and
// left as the reference leaves its hidden state (the final state is converted back to chart 1
// but currentChart is not reset, interceptor.cpp:214-216).
template <int MODEL, class OBS = NoRows>
SOCP_DEV int compute_traj(typename Model<MODEL>::Ctx &c, double *X, double t0, double tf, int S, OBS &&obs = OBS()) {
    if constexpr (MODEL == INTERCEPTOR) {
        int steps = 0;
        c.chart = 1;
        const double t1 = c.mprop / c.q;
        if (t0 < t1) {
            c.stage = 1;
            if (tf > t1) {
                steps += interceptor_model_int(c, X, t0, t1, S, obs);
                c.stage = 0;
                steps += interceptor_model_int(c, X, t1, tf, S, obs);
            } else {
                steps += interceptor_model_int(c, X, t0, tf, S, obs);
            }
        } else {
            c.stage = 0;
            steps += interceptor_model_int(c, X, t0, tf, S, obs);
        }
        if (c.chart == 2) Model<INTERCEPTOR>::convert(2, X);
        return steps;
    } else {
        return integrate_fixed<MODEL>(c, X, t0, tf, (tf - t0) / S, obs);
    }
}

// model::ComputeTraj with the adaptive integrator (the reference's Boost build).  The interceptor keeps
// its own fixed-step loop there too (interceptor.cpp:104-130 calls RK4 directly).
template <int MODEL>
SOCP_DEV int compute_traj_adaptive(typename Model<MODEL>::Ctx &c, double *X, double t0, double tf, int S, double tol, int &rejected) {
    if constexpr (MODEL == INTERCEPTOR) return compute_traj<MODEL>(c, X, t0, tf, S);
    else return integrate_adaptive<MODEL>(c, X, t0, tf, (tf - t0) / S, tol, rejected);
}

template <int MODEL> SOCP_DEV void get_chart_stage(const typename Model<MODEL>::Ctx &, int &chart, int &stage) { chart = 1; stage = 0; }
template <> SOCP_DEV void get_chart_stage<INTERCEPTOR>(const Model<INTERCEPTOR>::Ctx &c, int &chart, int &stage) { chart = c.chart; stage = c.stage; }
template <int MODEL> SOCP_DEV void set_chart_stage(typename Model<MODEL>::Ctx &, int, int) {}
template <> SOCP_DEV void set_chart_stage<INTERCEPTOR>(Model<INTERCEPTOR>::Ctx &c, int chart, int stage) { c.chart = chart; c.stage = stage; }

// warp-aggregated add of per-thread step counts into a device counter
SOCP_DEV void count_steps(unsigned long long *counter, int steps) {
    unsigned mask = __activemask();
    int total = steps;
    for (int off = 16; off > 0; off >>= 1) total += __shfl_down_sync(mask, total, off);
    // lanes outside the mask contribute garbage only if the mask is not full; handle that case
    if (mask != 0xffffffffu) {
        atomicAdd(counter, (unsigned long long)steps);
    } else if ((threadIdx.x & 31) == 0) {
        atomicAdd(counter, (unsigned long long)total);
    }
}

// ---- kernel: B independent trajectories ------------------------------------------------------
#define SOCP_TRAJ_THREADS 128      // threads per CTA of the trajectory kernels
// L = 1: one thread per trajectory.  L = Coop<MODEL>::LANES: a cooperative group of L lanes per trajectory.
template <int MODEL, bool ADAPTIVE, int L = 1>
__global__ void __launch_bounds__(SOCP_TRAJ_THREADS, Model<MODEL>::MINB)
traj_kernel(long B, int S, const double *__restrict__ mparams, const double *__restrict__ sw,
            const double *__restrict__ t0, const double *__restrict__ tf,
            const double *__restrict__ X0, double *__restrict__ Xf, unsigned long long *counter,
            double ode_tol, int *__restrict__ nsteps) {
    typedef Model<MODEL> M;
    constexpr int N = M::N;
    // (State I/O is per thread, N strided 8-byte accesses: staging the block's states through a shared tile for coalesced
    // traffic was measured -- 0.662 vs 0.582 ms for 2^20 Goddard trajectories, 51 vs 58 % of the FP64 peak: the two block
    // barriers and the tile cost more than the 74 % excess sectors of a kernel that moves 300 B per 11 kflop.)
    const long gt = (long)blockIdx.x * blockDim.x + threadIdx.x;
    const long b = gt / L;
    const int q = (int)(threadIdx.x % L);
    int steps = 0;
    if (b < B) {
        typename M::Ctx c;
        M::load(c, mparams + b * M::NP, sw ? sw + 2 * b : nullptr);
        if (L > 1) Coop<MODEL>::set(c, q);
        double X[N];
#pragma unroll
        for (int i = 0; i < N; ++i) X[i] = X0[b * N + i];
        int rej = 0;
        if (ADAPTIVE) steps = compute_traj_adaptive<MODEL>(c, X, t0[b], tf[b], S, ode_tol, rej);
        else steps = compute_traj<MODEL>(c, X, t0[b], tf[b], S);
        if (q == 0) {
#pragma unroll
            for (int i = 0; i < N; ++i) Xf[b * N + i] = X[i];
            if (nsteps) { nsteps[2 * b] = steps; nsteps[2 * b + 1] = rej; }
        } else steps = 0;
    }
    count_steps(counter + (ADAPTIVE ? 3 : 0), steps);
}

// ---- kernel: trajectories with the observer (model::Trace rows) ----------------------------------
// Restates the observer form of odeTools::integrate (odeTools.cpp:103-123): one row at t0 and one
// after every RK4 step.  Row layout = model::Trace (model.hpp:446-462): t, X[0..N), control[0..NCTRL),
// H, extra -- extra is the switching function of goddard::Trace (goddard.cpp:337-339), the chart id
// of interceptor::Trace (interceptor.cpp:151), 0 otherwise.
template <int MODEL> SOCP_DEV double trace_extra(const typename Model<MODEL>::Ctx &, const double *) { return 0.0; }
template <> SOCP_DEV double trace_extra<GODDARD>(const Model<GODDARD>::Ctx &c, const double *X) {
    return c.mu1 - c.b * X[13] - c.C / X[6] * sqrt(X[10] * X[10] + X[11] * X[11] + X[12] * X[12]);
}
template <> SOCP_DEV double trace_extra<INTERCEPTOR>(const Model<INTERCEPTOR>::Ctx &c, const double *) { return (double)c.chart; }

template <int MODEL>
__device__ __noinline__ void trace_row(const typename Model<MODEL>::Ctx &c, double t, const double *X, double *row) {
    typedef Model<MODEL> M;
    constexpr int N = M::N;
    row[0] = t;
    for (int i = 0; i < N; ++i) row[1 + i] = X[i];
    double u[4] = {0, 0, 0, 0};
    M::control(c, t, X, u);
    for (int k = 0; k < M::NCTRL; ++k) row[1 + N + k] = u[k];
    row[1 + N + M::NCTRL] = M::hamiltonian(c, t, X);
    row[2 + N + M::NCTRL] = trace_extra<MODEL>(c, X);
}

template <int MODEL> struct TraceRows {
    double *rows;
    int W, n;
    SOCP_DEV void operator()(const typename Model<MODEL>::Ctx &c, double t, const double *X) {
        trace_row<MODEL>(c, t, X, rows + (size_t)(n++) * W);
    }
};

// compute_traj with the observer on: returns the rows written (S + 1 per integration)
template <int MODEL>
SOCP_DEV int trace_traj(typename Model<MODEL>::Ctx &c, double *X, double t0, double tf, int S, double *rows, int W) {
    TraceRows<MODEL> obs{rows, W, 0};
    compute_traj<MODEL>(c, X, t0, tf, S, obs);
    return obs.n;
}

// rows: [B][max_rows][W]; nrows[b] = rows written (S+1 per integration, two integrations for a
// two-stage interceptor flight); Xf as traj_kernel.
template <int MODEL>
__global__ void __launch_bounds__(64)
trace_kernel(long B, int S, int max_rows, const double *__restrict__ mparams, const double *__restrict__ sw,
             const double *__restrict__ t0, const double *__restrict__ tf, const double *__restrict__ X0,
             double *__restrict__ rows, int *__restrict__ nrows, double *__restrict__ Xf) {
    typedef Model<MODEL> M;
    constexpr int N = M::N, W = N + M::NCTRL + 3;
    long b = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    typename M::Ctx c;
    M::load(c, mparams + b * M::NP, sw ? sw + 2 * b : nullptr);
    double X[N];
    for (int i = 0; i < N; ++i) X[i] = X0[b * N + i];
    const int nr = trace_traj<MODEL>(c, X, t0[b], tf[b], S, rows + (size_t)b * max_rows * W, W);
    nrows[b] = nr;
    if (Xf) for (int i = 0; i < N; ++i) Xf[b * N + i] = X[i];
}

// ---- kernel: RHS / control / Hamiltonian at B points -----------------------------------------
template <int MODEL>
__global__ void point_kernel(long B, const double *__restrict__ mparams, const double *__restrict__ sw,
                             const int *__restrict__ chart_stage, const double *__restrict__ t,
                             const double *__restrict__ X, double *rhs, double *control, double *H) {
    typedef Model<MODEL> M;
    constexpr int N = M::N;
    long b = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    typename M::Ctx c;
    M::load(c, mparams + b * M::NP, sw ? sw + 2 * b : nullptr);
    if (chart_stage) set_chart_stage<MODEL>(c, chart_stage[2 * b], chart_stage[2 * b + 1]);
    double x[N], out[N];
    for (int i = 0; i < N; ++i) x[i] = X[b * N + i];
    if (rhs) {
        M::rhs(c, t[b], x, out);
        for (int i = 0; i < N; ++i) rhs[b * N + i] = out[i];
    }
    if (control) {
        double u[4] = {0, 0, 0, 0};
        M::control(c, t[b], x, u);
        for (int i = 0; i < 4; ++i) control[b * 4 + i] = u[i];
    }
    if (H) H[b] = M::hamiltonian(c, t[b], x);
}

// ---- FP64 peak probe: register-resident DFMA chains ------------------------------------------
__global__ void __launch_bounds__(256) dfma_peak_kernel(double *out, int iters, double a, double b) {
    double x0 = threadIdx.x * 1e-3, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5,
           x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
            x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
        }
    }
    out[(long)blockIdx.x * blockDim.x + threadIdx.x] = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
}

}  // namespace socp
