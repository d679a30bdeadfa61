// socp_b200/csrc/move.cuh -- shooting::Move(tf), shooting::GetSolution and shooting::Trace for a batch of solved
// problems.
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
        double t1, t2, t_end, sw[2] = {0.0227, 0.08}, sw_unused[2];
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
        if (L > 1) Coop<MODEL>::set(c, lane, ((1u << L) - 1u) << ((threadIdx.x & 31) & ~(L - 1)));
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
    double t1, t2, sw[2] = {0.0227, 0.08};
    timeline_pair(sh, time + b * (sh.M + 1), [&](int k) { return xb[nm + k]; }, j, t1, t2, sw);
    typename M::Ctx c;
    M::load(c, mparams + b * M::NP, sw);
    double X[N];
    for (int i = 0; i < N; ++i) X[i] = xb[N * j + i];
    nrows[w] = trace_traj<MODEL>(c, X, t1, t2, sh.S, rows + w * R * W, W);
}

}  // namespace socp
