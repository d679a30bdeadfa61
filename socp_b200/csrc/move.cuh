// socp_b200/csrc/move.cuh -- shooting::Move(tf), shooting::GetSolution and shooting::Trace for a batch of solved
// problems, and shooting::InitShooting(ti, Xi, tf, Xf) for a batch of new ones.
//
// Restates shooting::Move(tf) (src/socp/shooting.cpp:383-437; cpp/src/socp/shooting.cpp:146-160) and
// shooting::UpdateSolution (:1462-1508): the state of a solution at time t is the integration of the shooting
// segment that contains t, from its node state.  One thread (or one cooperative group, integrate.cuh) per
// (problem, query); the time line is never materialised: timeline_pair yields the node times on demand, so
// the kernel is as register-resident as traj_kernel.
#pragma once
#include "solver.cuh"

namespace socp {

// What a Move needs of a socp_shape: passed by value, so mode_t is read from the constant bank.
struct MoveShape {
    int M, P, S;
    int mode_t[SOCP_MAX_NODES];
    double ode_tol;                        // > 0: adaptive Dormand-Prince (socp_shape::integrator == SOCP_DOPRI5)
};

// Xq[b * ostride + q * N ..] = Move(tq[b * Q + q]) of problem b for q < Q; tq == nullptr: Move(t_end) (Q = 1).
// The integration is compute_traj / compute_traj_adaptive with the arguments traj_kernel gives it, so a Move
// is bit for bit the socp_traj_batch of (t_seg, node state, target, switching times, S).  One work item per
// thread (group) and a grid that covers them all, as traj_kernel: a grid-stride loop keeps its induction state
// live across the integration and made Goddard spill (32 B with -Xptxas -v; none without it).
template <int MODEL, bool ADAPTIVE, int L = 1>
__global__ void __launch_bounds__(SOCP_TRAJ_THREADS, Model<MODEL>::MINB)
move_kernel(MoveShape sh, long B, int Q, const double *__restrict__ mparams, const double *__restrict__ time,
            const double *__restrict__ x, const double *__restrict__ tq, double *__restrict__ Xq, long ostride,
            unsigned long long *counter) {
    typedef Model<MODEL> M;
    constexpr int N = M::N;
    const long total = B * Q;
    const int lane = (int)(threadIdx.x % L);
    int steps = 0;
    const long w = ((long)blockIdx.x * blockDim.x + threadIdx.x) / L;
    if (w < total) {
        const long b = w / Q;
        const int q = (int)(w % Q);
        const double *xb = x + b * sh.P;
        const double *time_b = time + b * (sh.M + 1);
        const int nm = N * sh.M;
        auto xfree = [&](int k) { return xb[nm + k]; };
        // ComputeTimeLine first, as the reference's Move does: t0, t_end and the switching times
        double t1, t2, t_end, sw[2] = {Model<GODDARD>::SW0_GUESS, Model<GODDARD>::SW1_GUESS}, sw_unused[2];
        timeline_pair(sh, time_b, xfree, sh.M - 1, t1, t_end, sw);
        timeline_pair(sh, time_b, xfree, 0, t1, t2, sw_unused);
        // a query outside [t0, t_end] (NaN included) is answered at t_end
        const double tv = tq ? tq[w] : t_end;
        const double target = (tv >= t1 && tv <= t_end) ? tv : t_end;
        // seg = 0; while (tl[seg + 1] < target) ++seg;   (target <= t_end = tl[M] stops it at M - 1)
        int seg = 0;
        while (seg < sh.M - 1 && t2 < target) {
            ++seg;
            timeline_pair(sh, time_b, xfree, seg, t1, t2, sw_unused);
        }
        typename M::Ctx c;
        M::load(c, mparams + b * M::NP, sw);
        if (L > 1) Coop<MODEL>::set(c, lane);
        double X[N];
#pragma unroll
        for (int i = 0; i < N; ++i) X[i] = xb[N * seg + i];
        int st, rej = 0;
        if (ADAPTIVE) st = compute_traj_adaptive<MODEL>(c, X, t1, target, sh.S, sh.ode_tol, rej);
        else st = compute_traj<MODEL>(c, X, t1, target, sh.S);
        if (lane == 0) {
            double *out = Xq + b * ostride + (long)q * N;
#pragma unroll
            for (int i = 0; i < N; ++i) out[i] = X[i];
            steps += st;
        }
    }
    count_steps(counter + (ADAPTIVE ? 3 : 0), steps);
}

// The copies of GetSolution: vt[b] = the time line, vX[b][i] = node i of x[b] for i < M (vX[b][M] is the
// move_kernel's Move(t_end)).  One thread per output value.
__global__ void __launch_bounds__(256)
solution_nodes_kernel(MoveShape sh, long B, int N, const double *__restrict__ time, const double *__restrict__ x,
                      double *__restrict__ vt, double *__restrict__ vX) {
    const long nt = B * (sh.M + 1), nx = B * sh.M * N;
    for (long w = (long)blockIdx.x * blockDim.x + threadIdx.x; w < nt + nx; w += (long)gridDim.x * blockDim.x) {
        if (w < nt) {
            const long b = w / (sh.M + 1);
            const int j = (int)(w % (sh.M + 1));
            const double *xb = x + b * sh.P;
            const int nm = N * sh.M;
            double t1, t2, sw[2];
            // node j is the start of segment j, or the end of segment M - 1
            timeline_pair(sh, time + b * (sh.M + 1), [&](int k) { return xb[nm + k]; },
                          j < sh.M ? j : sh.M - 1, t1, t2, sw);
            vt[w] = j < sh.M ? t1 : t2;
        } else {
            const long v = w - nt, per = (long)sh.M * N;
            const long b = v / per, r = v % per;
            vX[b * (per + N) + r] = x[b * sh.P + r];
        }
    }
}

// shooting::Trace (src/socp/shooting.cpp:496-544): every segment of every solution re-integrated with the observer on.
// rows[b][j] (R rows of W) = the rows of segment j of problem b, nrows[b * M + j] = their count: the trace_traj of
// (tl[j], node j of x[b], tl[j + 1], switching times, S), so a segment is bit for bit the socp_trace_batch of the same
// arguments.  The observer is the fixed-step RK4 one for every shape, SOCP_DOPRI5 included, as model::ModelInt's
// trace branch (odeTools.cpp:103-123).  One thread per (problem, segment), 64-thread CTAs as trace_kernel.
template <int MODEL>
__global__ void __launch_bounds__(64)
solution_trace_kernel(MoveShape sh, long B, int R, const double *__restrict__ mparams, const double *__restrict__ time,
                      const double *__restrict__ x, double *__restrict__ rows, int *__restrict__ nrows) {
    typedef Model<MODEL> M;
    constexpr int N = M::N, W = N + M::NCTRL + 3;
    const long w = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= B * sh.M) return;
    const long b = w / sh.M;
    const int j = (int)(w % sh.M);
    const double *xb = x + b * sh.P;
    const int nm = N * sh.M;
    double t1, t2;
    typename M::Ctx c;
    segment_setup<MODEL>(sh, time + b * (sh.M + 1), [&](int k) { return xb[nm + k]; }, j, mparams + b * M::NP, t1, t2, c);
    double X[N];
    for (int i = 0; i < N; ++i) X[i] = xb[N * j + i];
    nrows[w] = trace_traj<MODEL>(c, X, t1, t2, sh.S, rows + w * R * W, W);
}

// shooting::InitShooting(ti, Xi, tf, Xf) (src/socp/shooting.cpp:202-245; cpp/src/socp/shooting.cpp:118-127): node i of
// the uniform grid, with the reference's expression, so node M is this value and not tf.
SOCP_DEV double init_node_time(double ti, double tf, int i, int M) { return ti + i * (tf - ti) / M; }

// The time line and the copies of InitShooting: time[b] = the grid, node 0 = Xi[b] (x and Xb), Xb node M = Xf[b], and
// the FREE node times after the node blocks of x[b], in node order.  One thread per output value: per problem, M + 1
// times, N values of node 0, dim of node M, nfree times.  (One warp per problem, a lane per value, was measured slower:
// 47 against 29 us for 10^5 Goddard problems on a B200 at its 1000 W power limit.)
__global__ void __launch_bounds__(256)
init_copies_kernel(MoveShape sh, long B, int n, const double *__restrict__ ti, const double *__restrict__ Xi,
                   const double *__restrict__ tf, const double *__restrict__ Xf, double *__restrict__ time,
                   double *__restrict__ Xb, double *__restrict__ x) {
    const int N = 2 * n, nt = sh.M + 1, nfree = sh.P - N * sh.M;
    const int per = nt + N + n + nfree;
    for (long w = (long)blockIdx.x * blockDim.x + threadIdx.x; w < B * per; w += (long)gridDim.x * blockDim.x) {
        const long b = w / per;
        int r = (int)(w % per);
        if (r < nt) {
            time[b * nt + r] = init_node_time(ti[b], tf[b], r, sh.M);
        } else if ((r -= nt) < N) {
            const double v = Xi[b * N + r];
            x[b * sh.P + r] = v;
            if (r < n) Xb[b * nt * n + r] = v;
        } else if ((r -= N) < n) {
            Xb[(b * nt + sh.M) * n + r] = Xf[b * n + r];
        } else {
            r -= n;
            int j = -1;                             // the node of the r-th FREE time
            for (int k = 0; k <= r; ++k) do ++j; while (sh.mode_t[j] != SOCP_FREE);
            x[b * sh.P + N * sh.M + r] = init_node_time(ti[b], tf[b], j, sh.M);
        }
    }
}

// Interior node i (1 <= i < M) of problem b: the integration of (ti[b], Xi[b]) to time[b][i], written to x[b][i] and its
// first dim values to Xb[b][i]; time is init_copies_kernel's output.  compute_traj / compute_traj_adaptive with
// traj_kernel's arguments, so a node is bit for bit the socp_traj_batch (socp_traj_adaptive_batch) of (ti, Xi, node time,
// sw, S).  One work item per thread (group), node-major: blockIdx.y = i - 1, so the items of a warp share the interval
// length (the adaptive step counts of a warp diverge less) and no thread divides its index by B.
template <int MODEL, bool ADAPTIVE, int L = 1>
__global__ void __launch_bounds__(SOCP_TRAJ_THREADS, Model<MODEL>::MINB)
init_nodes_kernel(MoveShape sh, long B, const double *__restrict__ mparams, const double *__restrict__ sw,
                  const double *__restrict__ ti, const double *__restrict__ Xi, const double *__restrict__ time,
                  double *__restrict__ Xb, double *__restrict__ x, unsigned long long *counter) {
    typedef Model<MODEL> M;
    constexpr int N = M::N, n = M::DIM;
    const int i = 1 + (int)blockIdx.y;
    const int lane = (int)(threadIdx.x % L);
    int steps = 0;
    const long b = ((long)blockIdx.x * blockDim.x + threadIdx.x) / L;
    if (b < B) {
        typename M::Ctx c;
        M::load(c, mparams + b * M::NP, sw ? sw + 2 * b : nullptr);
        if (L > 1) Coop<MODEL>::set(c, lane);
        double X[N];
#pragma unroll
        for (int k = 0; k < N; ++k) X[k] = Xi[b * N + k];
        int st, rej = 0;
        if (ADAPTIVE) st = compute_traj_adaptive<MODEL>(c, X, ti[b], time[b * (sh.M + 1) + i], sh.S, sh.ode_tol, rej);
        else st = compute_traj<MODEL>(c, X, ti[b], time[b * (sh.M + 1) + i], sh.S);
        if (lane == 0) {
            double *xo = x + b * sh.P + (long)N * i, *Xo = Xb + (b * (sh.M + 1) + i) * n;
#pragma unroll
            for (int k = 0; k < N; ++k) xo[k] = X[k];
#pragma unroll
            for (int k = 0; k < n; ++k) Xo[k] = X[k];
            steps += st;
        }
    }
    count_steps(counter + (ADAPTIVE ? 3 : 0), steps);
}

}  // namespace socp
