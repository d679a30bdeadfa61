// socp_b200/csrc/solver.cuh -- batched shooting residual, FD Jacobian and Powell-hybrid solve.
//
// Lock-step reverse-communication design: every problem of the batch carries its own MINPACK
// `hybrd` state (phase, trust radius, counters, QR factors) in HBM.  One ROUND is two kernels:
//
//   integrate_worklist   one thread per (problem, segment[, perturbed column]) work item: RK4 over
//                        one shooting segment with the state in registers.  A residual request is
//                        M items, a forward-difference Jacobian request is 2*dim*M + nfree*M items
//                        (only the segment a perturbed unknown can influence is re-integrated; the
//                        other entries of that column are exactly zero in the reference too).
//   advance              one thread group per problem: assemble the residual / Jacobian from the
//                        segment end points (boundary functions, continuity, free-time conditions),
//                        run the hybrd state machine up to its next function evaluation and append
//                        the problem to the next round's work list -- or retire it (converged /
//                        failed), which is the convergence mask.
//
// Restates: shooting::ShootingFunction (src/socp/shooting.cpp:918-993), ComputeTimeLine
// (:1579-1617), MultipleShootingFunction (:1511-1576, isJac == 0), the boundary functions of
// model.hpp:90-255 with the model overrides (interceptor.cpp:223-272, vtolUAV.cpp:223-283,
// goddard.cpp:343-370), and MINPACK hybrd/fdjac1/qrfac/qform/dogleg/r1updt/r1mpyq as called from
// shooting.cpp:803-826 (ml = mu = n-1, epsfcn = 1e-15, mode = 1, factor = 1).
#pragma once
#include <cuda_runtime.h>
#include <cuda_pipeline.h>
#include <float.h>
#include "../../include/socp_b200.h"
#include "models.cuh"
#include "integrate.cuh"

namespace socp {

enum { PH_IDLE = 0, PH_F0 = 1, PH_JAC = 2, PH_TRIAL = 3 };
enum { RUN_SOLVE = 0, RUN_RESIDUAL = 1, RUN_FDJAC = 2 };
// per-problem integer state
// I_PEND: the rotations of the last Broyden update (scr) have not been applied to Q yet (split build)
enum { I_PHASE = 0, I_ITER, I_NCSUC, I_NCFAIL, I_NSLOW1, I_NSLOW2, I_JEVAL, I_NFEV, I_INFO, I_BASE, I_NJEV, I_PEND, I_COUNT = 12 };
// per-problem scalar state
enum { D_DELTA = 0, D_XNORM, D_FNORM, D_PNORM, D_COUNT = 4 };

struct SolverDev {
    // shape
    int model_id, dim, N, M, S, P, nfree, np, nJ, REC, LR;
    int LRS;                               // doubles between the packed factors of two problems: LR rounded up to even (bulk copies)
    int QS;                                // doubles between the Q / fjac matrices of two problems: P*P rounded up to an
                                           // even count, so that every matrix starts 16-byte aligned (bulk copies)
    int mode_t[SOCP_MAX_NODES];
    int mode_X[SOCP_MAX_NODES][SOCP_MAX_DIM];
    const int *jac_col, *jac_seg;          // [nJ] work item -> (column, segment)
    const int *col_item0, *col_nseg;       // [P] first item of a column; 1 or M segments
    const int *band_lo, *band_off;         // [P], [P + 1] structural band of the Jacobian (jac_band): column k keeps the
                                           // rows band_lo[k] .. band_lo[k] + band_off[k + 1] - band_off[k] - 1
    int band_doubles;                      // > 0: the Jacobian phase runs hybrd_jac_band_kernel on a band of this size
    // problem data
    long B;
    const double *mparams, *time, *Xb;
    // solver settings
    double xtol, epsfcn, factor;
    int maxfev, run_mode;
    double ode_tol;                        // > 0: adaptive Dormand-Prince segments (socp_shape::ode_tol)
    int analytic;                          // 1: hybrj -- Jacobian requests are served by the variational integration
    // persistent state
    double *x, *xe, *fvec, *diag, *qtf, *wa1, *wa2, *wa3, *wa4, *scr, *fjac, *r, *ends, *jends, *dstate;
    int *istate;
    // work lists, double buffered: list[2][2][B], count[2][2]
    int *lists;
    int *counts;
    unsigned long long *counters;      // [0] RK4 steps, [1] Broyden iterations, [2] Jacobian factorisations, [3] dopri steps,
                                       // [4] residual requests, [5] Q passes, [16+k] / [32+k] phase clocks
    const SolverDev *self;             // this struct in GLOBAL memory: what non-inlined device functions take by reference
                                       // (a reference to the kernel parameter would make every thread copy the 2.5 KB
                                       // struct to its local-memory frame)
    int sm_count;                      // multiprocessors of the device (seq_warp)
    int phase_clocks;                  // debugging aid (SOCP_PHASE_CLOCKS=1): accumulate clock64() per phase
};

#define EPSMCH DBL_EPSILON

// phase timing of the Powell-hybrid kernels (debugging aid, off unless SolverDev::phase_clocks)
#define SOCP_PHASE(base, k)                                                                   \
    do {                                                                                      \
        if (D.phase_clocks && (threadIdx.x % G) == 0) {                                       \
            const long long now_ = clock64();                                                 \
            atomicAdd(D.counters + (base) + (k), (unsigned long long)(now_ - phase_t0));      \
            phase_t0 = now_;                                                                  \
        }                                                                                     \
    } while (0)

// finer marks inside a phase (same clock, slots 48..63); sub_t0 is the caller's running time stamp
#define SOCP_SUB(k)                                                                           \
    do {                                                                                      \
        if (clk_on && (threadIdx.x % G) == 0) {                                               \
            const long long now_ = clock64();                                                 \
            atomicAdd(clk_counters + 48 + (k), (unsigned long long)(now_ - sub_t0));          \
            sub_t0 = now_;                                                                    \
        }                                                                                     \
    } while (0)

// Which warp of a thread group runs the strictly sequential phases (Givens sweeps, back substitution).
// Warp w of every CTA is scheduled on sub-partition w % 4 of its SM, so if every resident CTA used warp 0
// all the sequential chains of an SM would share ONE scheduler and FP64 pipe while three idle (measured:
// 1.7x slower per problem with 4 co-resident CTAs).  Co-resident CTAs are b, b + #SMs, b + 2 #SMs, ...:
// rotate by blockIdx.x / #SMs.
template <int G> SOCP_DEV int seq_warp(int sm_count) {
    return (G == 32) ? 0 : (int)((blockIdx.x / (unsigned)sm_count) % (G / 32));
}

// ---- group helpers ---------------------------------------------------------------------------
template <int G> SOCP_DEV void gsync() { if (G == 32) __syncwarp(); else __syncthreads(); }

SOCP_DEV double warp_sum_d(double v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}
SOCP_DEV double warp_max_d(double v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, off));
    return v;
}

// MINPACK enorm on one warp: x[0..n) (stride 1, visible to the whole warp).  Components in the
// intermediate range are summed as plain squares; small (<= rdwarf) and large (>= rgiant/n) ones are
// scaled by their maximum as MINPACK does, but with the maximum found first (a reduction) instead
// of by running rescaling, so nothing is sequential.  Every lane returns the same value.
// enorm_rows: the same norm of an n-vector whose components outside [lo, end) are zeros and not stored
// (x[i - lo] is component i).  Component i stays on lane i % 32, so the bits are those of the full vector: a
// zero adds nothing to any of the sums.
SOCP_DEV double enorm_rows(int n, const double *x, int lo, int end) {
    const double rdwarf = 3.834e-20, rgiant = 1.304e19;
    // MINPACK's agiant = rgiant / n; the range test is written xabs * n < rgiant so that no call pays a
    // divide (the two differ only for a component within an ulp of the threshold, where either
    // accumulation is safe)
    const double dn = (double)n;
    const int lane = threadIdx.x & 31;
    const int first = lo + ((lane - lo) & 31);
    double s2 = 0., small_max = 0., big_max = 0.;
    bool isnan_ = false;
    for (int i = first; i < end; i += 32) {
        const double xabs = fabs(x[i - lo]);
        if (xabs > rdwarf && xabs * dn < rgiant) s2 = fma(xabs, xabs, s2);
        else if (xabs <= rdwarf) small_max = fmax(small_max, xabs);
        else if (xabs == xabs) big_max = fmax(big_max, xabs);
        else isnan_ = true;
    }
    s2 = warp_sum_d(s2);
    if (__any_sync(0xffffffffu, isnan_)) return s2 + nan("");      // MINPACK's enorm propagates a NaN
    const bool special = __any_sync(0xffffffffu, small_max != 0. || big_max != 0.);
    if (!special) return sqrt(s2);
    const double x1max = warp_max_d(big_max), x3max = warp_max_d(small_max);
    double s1 = 0., s3 = 0.;
    for (int i = first; i < end; i += 32) {
        const double xabs = fabs(x[i - lo]);
        if (xabs > rdwarf && xabs * dn < rgiant) continue;
        if (xabs <= rdwarf) { if (xabs != 0.) { const double q = xabs / x3max; s3 = fma(q, q, s3); } }
        else { const double q = xabs / x1max; s1 = fma(q, q, s1); }
    }
    s1 = warp_sum_d(s1);
    s3 = warp_sum_d(s3);
    if (s1 != 0.) return x1max * sqrt(s1 + (s2 / x1max) / x1max);
    if (s2 != 0.) {
        if (s2 >= x3max) return sqrt(s2 * (1. + (x3max / s2) * (x3max * s3)));
        return sqrt(x3max * ((s2 / x3max) + (x3max * s3)));
    }
    return x3max * sqrt(s3);
}
SOCP_DEV double enorm_warp(int n, const double *x) { return enorm_rows(n, x, 0, n); }

// Euclidean norm over a thread group: every warp of the group evaluates enorm_warp on the whole
// vector (n is a few hundred at most), so no block-level reduction or barrier is needed and every
// thread gets the same bits.  The caller guarantees x is visible (a barrier after its last write).
template <int G> SOCP_DEV double enorm_g(int n, const double *x, double *) {
    return enorm_warp(n, x);
}

// ---- time line (shooting.cpp:1579-1617) --------------------------------------------------------
// Node times from the fixed times and the FREE-time unknowns, linear interpolation for CONTINUOUS
// nodes.  xfree(k) returns the k-th free-time unknown (already perturbed if needed).
// sw[2] receives the first two FREE interior times (SwitchingTimesUpdate, goddard.cpp:373).
// t1, t2 = the two node times of segment s, without materialising the whole line.  SH is any shape with M and
// mode_t[M + 1]: SolverDev for the solver kernels, MoveShape for the move kernels (move.cuh).
template <class SH, class XF>
SOCP_DEV void timeline_pair(const SH &D, const double *time_b, XF xfree, int s, double &t1, double &t2, double *sw) {
    int k = 0, cur = 0, nsw = 0;
    double tcur = 0;
    t1 = t2 = 0;
    for (int j = 0; j <= D.M; ++j) {
        const int m = D.mode_t[j];
        if (m == SOCP_FIXED || m == SOCP_FREE) {
            double tj;
            if (m == SOCP_FIXED) tj = time_b[j];
            else {
                tj = xfree(k++);
                if (j < D.M && nsw < 2) sw[nsw++] = tj;
            }
            if (s > cur && s < j) t1 = tcur + (s - cur) * (tj - tcur) / (j - cur);
            else if (s == j) t1 = tj;
            if (s + 1 > cur && s + 1 < j) t2 = tcur + (s + 1 - cur) * (tj - tcur) / (j - cur);
            else if (s + 1 == j) t2 = tj;
            cur = j;
            tcur = tj;
        }
    }
}

// Segment s of a problem as its integration starts: the node times t1, t2 and the model context loaded from the
// parameter block mp with the switching times of the time line (Goddard's guesses while it has fewer than two FREE
// interior times; the other models ignore them).
template <int MODEL, class SH, class XF>
SOCP_DEV void segment_setup(const SH &D, const double *time_b, XF xfree, int s, const double *mp, double &t1, double &t2,
                            typename Model<MODEL>::Ctx &c) {
    double sw[2] = {Model<GODDARD>::SW0_GUESS, Model<GODDARD>::SW1_GUESS};
    timeline_pair(D, time_b, xfree, s, t1, t2, sw);
    Model<MODEL>::load(c, mp, sw);
}

// MINPACK fdjac1 step for unknown value v
SOCP_DEV double fd_step(double v, double epsfcn) {
    double eps = sqrt(fmax(epsfcn, EPSMCH));
    double h = eps * fabs(v);
    if (h == 0.) h = eps;
    return h;
}

// ---- kernel 1: integrate every requested shooting segment --------------------------------------
// L lanes per work item: 1, or Coop<MODEL>::LANES (a cooperative group per segment, used when the round has too few
// items to fill the GPU with one thread each -- the tail of a batched solve; same bits either way, integrate.cuh)
template <int MODEL, bool ADAPTIVE, int L = 1>
__global__ void __launch_bounds__(128, Model<MODEL>::MINB)
integrate_worklist(SolverDev D, int cur) {
    typedef Model<MODEL> M;
    constexpr int N = M::N;
    const int nres = D.counts[cur * 2 + 0], njac = D.analytic ? 0 : D.counts[cur * 2 + 1];
    const int *res_list = D.lists + (size_t)(cur * 2 + 0) * D.B;
    const int *jac_list = D.lists + (size_t)(cur * 2 + 1) * D.B;
    if (blockIdx.x == 0 && threadIdx.x == 0) {       // next-next round's counters
        D.counts[(1 - cur) * 2 + 0] = 0;
        D.counts[(1 - cur) * 2 + 1] = 0;
    }
    const long total = (long)nres * D.M + (long)njac * D.nJ;
    int steps = 0;
    const int cq = (int)(threadIdx.x % L);
    for (long w = ((long)blockIdx.x * blockDim.x + threadIdx.x) / L; w < total; w += ((long)gridDim.x * blockDim.x) / L) {
        long b;
        int s, col;
        double *out;
        if (w < (long)nres * D.M) {
            b = res_list[w / D.M];
            s = (int)(w % D.M);
            col = -1;
            const int trial = 1 - D.istate[b * I_COUNT + I_BASE];
            out = D.ends + ((b * 2 + trial) * D.M + s) * D.REC;
        } else {
            const long w2 = w - (long)nres * D.M;
            b = jac_list[w2 / D.nJ];
            const int k = (int)(w2 % D.nJ);
            col = D.jac_col[k];
            s = D.jac_seg[k];
            out = D.jends + (b * D.nJ + k) * D.REC;
        }
        const double *xe = D.xe + b * D.P;
        const double h = (col >= 0) ? fd_step(xe[col], D.epsfcn) : 0.0;
        const int nm = N * D.M;
        double t1, t2;
        typename M::Ctx c;
        segment_setup<MODEL>(D, D.time + b * (D.M + 1), [&](int k) { int idx = nm + k; return xe[idx] + ((idx == col) ? h : 0.0); },
                             s, D.mparams + b * M::NP, t1, t2, c);
        if (L > 1) Coop<MODEL>::set(c, cq);
        double X[N];
#pragma unroll
        for (int i = 0; i < N; ++i) X[i] = xe[N * s + i];
        if (col >= 0 && col < nm && col / N == s) {
            const int kk = col - N * s;
#pragma unroll
            for (int i = 0; i < N; ++i) if (i == kk) X[i] += h;
        }
        int st;
        if (ADAPTIVE) { int rej = 0; st = compute_traj_adaptive<MODEL>(c, X, t1, t2, D.S, D.ode_tol, rej); }
        else st = compute_traj<MODEL>(c, X, t1, t2, D.S);
        if (cq == 0) {
            steps += st;
#pragma unroll
            for (int i = 0; i < N; ++i) out[i] = X[i];
            int chart, stage;
            get_chart_stage<MODEL>(c, chart, stage);
            out[N] = (double)chart;
            out[N + 1] = (double)stage;
        }
    }
    count_steps(D.counters + (ADAPTIVE ? 3 : 0), steps);
}

// ---- residual assembly (one thread) ------------------------------------------------------------
// Writes every entry of F(xe + h e_col) (col < 0: the base point) to out[0..P).
// Deliberately ONE non-inlined function: the base residual and every perturbed column run the
// same machine code, so entries a perturbation cannot reach are bitwise equal to the base and
// their forward difference is exactly zero, as in the reference.
template <int MODEL>
__device__ __noinline__ void assemble(const SolverDev &D, long b, int col, double h, const double *base_ends,
                                      const double *jends_b, double *out, int seg_lo, int seg_hi, const double *base) {
    // Only the segments seg_lo..seg_hi are evaluated (the caller knows which ones a perturbed unknown can
    // reach; every other entry of a forward-difference column is an exact zero, as in the reference, and the
    // column was zero-filled beforehand); the free-time row counter still runs over all of them.
    // base != nullptr: emit the forward difference (F_i(x + h e_col) - base_i) / h instead of F_i.
    // (F_i(x + h e_col) - F_i(x)) / h: one reciprocal per column, then quotient, exact residual and one
    // correction per entry (the correctly rounded quotient short of pathological mantissas of h; a full
    // divide per entry was a third of this kernel's instructions)
    const double rh = base ? 1. / h : 0.;
    auto emit = [&](int i, double v) {
        if (base) {
            const double d = v - base[i], q = d * rh;
            out[i] = (d == 0.) ? 0. : (fabs(q) < DBL_MAX) ? fma(fma(-q, h, d), rh, q) : d / h;
        } else out[i] = v;
    };
    typedef Model<MODEL> M;
    constexpr int N = M::N, n = M::DIM;
    const double *xe = D.xe + b * D.P;
    const double *Xb = D.Xb + b * (D.M + 1) * n;
    const double *mp = D.mparams + b * M::NP;
    auto xv = [&](int idx) { return xe[idx] + ((idx == col) ? h : 0.0); };
    auto rec = [&](int s) -> const double * {
        if (col < 0) return base_ends + s * D.REC;
        if (D.col_nseg[col] == 1) {
            const int seg0 = D.jac_seg[D.col_item0[col]];
            return (s == seg0) ? jends_b + (size_t)D.col_item0[col] * D.REC : base_ends + s * D.REC;
        }
        return jends_b + (size_t)(D.col_item0[col] + s) * D.REC;
    };
    // node times on demand (timeline_pair per evaluated segment: no per-thread array of M + 1 times in local memory);
    // the first call also yields the switching times the model context needs
    const int nm = N * D.M;
    const double *time_b = D.time + b * (D.M + 1);
    auto xfree = [&](int k) { return xv(nm + k); };
    double t_lo, t_hi;
    typename M::Ctx c;
    segment_setup<MODEL>(D, time_b, xfree, seg_lo, mp, t_lo, t_hi, c);
    int nbr = nm;
    double X1[N], Xtf[N], Xp[N];
    for (int i = 0; i < D.M; ++i) {
        if (i < seg_lo || i > seg_hi) {
            if (i == 0 && D.mode_t[0] != SOCP_FIXED) nbr += 1;
            if (i < D.M - 1 && D.mode_t[i + 1] == SOCP_FREE) nbr += 1;
            if (i == D.M - 1 && D.mode_t[D.M] != SOCP_FIXED) nbr += 1;
            continue;
        }
        double t1, t2, sw_unused[2];
        if (i == seg_lo) { t1 = t_lo; t2 = t_hi; }
        else timeline_pair(D, time_b, xfree, i, t1, t2, sw_unused);
        const double *e = rec(i);
#pragma unroll
        for (int k = 0; k < N; ++k) { Xtf[k] = e[k]; X1[k] = xv(N * i + k); }
        set_chart_stage<MODEL>(c, (int)e[N], (int)e[N + 1]);
        const int index = N * (i + 1);
        if (i == 0) {
            // model::InitialFunction (model.hpp:196-213) / InitialHFunction (:239-255)
            for (int k = 0; k < n; ++k)
                emit(k, (D.mode_X[0][k] == SOCP_FREE) ? X1[k + n] : X1[k] - Xb[k]);
            if (D.mode_t[0] != SOCP_FIXED) {
                emit(nm, M::hamiltonian(c, t1, X1));
                nbr += 1;
            }
        }
        if (i < D.M - 1) {
#pragma unroll
            for (int k = 0; k < N; ++k) Xp[k] = xv(index + k);
            if (D.mode_t[i + 1] == SOCP_FREE) {
                // SwitchingTimesFunction: H(X) - H(Xp) (model.hpp:299-305); goddard: H(X) (goddard.cpp:343-370)
                double Hx = M::hamiltonian(c, t2, Xtf);
                if (MODEL != GODDARD) Hx -= M::hamiltonian(c, t2, Xp);
                emit(nbr, Hx);
                nbr += 1;
            }
            // shooting::MultipleShootingFunction (shooting.cpp:1511-1576, isJac == 0)
            const double *Xd = Xb + (i + 1) * n;
            for (int k = 0; k < n; ++k) {
                const int m = D.mode_X[i + 1][k];
                if (m == SOCP_FIXED) {
                    emit(index + k, Xtf[k] - Xd[k]);
                    emit(index + k + n, Xp[k] - Xd[k]);
                } else if (m == SOCP_FREE) {
                    // model::SwitchingStateFunction: empty by default (model.hpp:339);
                    // vtolUAV.cpp:273-283 adds the waypoint penalty to the costate jump
                    if (MODEL == VTOL_UAV) {
                        emit(index + k, Xtf[k] - Xp[k]);
                        emit(index + k + n, (Xtf[k + n] - Xp[k + n]) - mp[4] * (Xtf[k] - Xd[k]));
                    } else {
                        emit(index + k, 0.0);
                        emit(index + k + n, 0.0);
                    }
                } else {
                    emit(index + k, Xtf[k] - Xp[k]);
                    emit(index + k + n, Xtf[k + n] - Xp[k + n]);
                }
            }
        }
        if (i == D.M - 1) {
            // model::FinalFunction (model.hpp:90-103) and overrides interceptor.cpp:223-245,
            // vtolUAV.cpp:223-241; FinalHFunction adds H (+ muT for the interceptor, :270)
            const double *Xf = Xb + D.M * n;
            for (int k = 0; k < n; ++k) {
                double f;
                if (D.mode_X[D.M][k] == SOCP_FREE) {
                    f = Xtf[k + n];
                    if (MODEL == INTERCEPTOR && k == 1) f = Xtf[k + n] + mp[15];
                    if (MODEL == VTOL_UAV) {
                        const int nWP_tot = (int)mp[7], nWP = (int)mp[8];
                        f = Xtf[k + n] - mp[4] * (nWP_tot - nWP) * (Xtf[k] - Xf[k]) - 0.02 * (Xtf[k] - Xf[k]);
                    }
                } else {
                    f = Xtf[k] - Xf[k];
                    if (MODEL == INTERCEPTOR) {
                        if (k == 0) f = f / mp[1];
                        if (k == 3 && fabs(cos(Xf[2])) < 1e-5) f = Xtf[k + n];
                    }
                }
                emit(k + n, f);
            }
            if (D.mode_t[D.M] != SOCP_FIXED) {
                double H = M::hamiltonian(c, t2, Xtf);
                if (MODEL == INTERCEPTOR) H += mp[14];
                emit(nbr, H);
                nbr += 1;
            }
        }
    }
}

// ---- kernel 2a0: zero the Jacobians about to be assembled (coalesced; the column threads of
// assemble_kernel then write only the rows a perturbed unknown can reach) -----------------------------
__global__ void __launch_bounds__(256) zero_fjac_kernel(SolverDev D, int cur) {
    const int njac = D.analytic ? 0 : D.counts[cur * 2 + 1];
    const int *jac_list = D.lists + (size_t)(cur * 2 + 1) * D.B;
    const long pp = (long)D.P * D.P;
    for (long w = (long)blockIdx.x * blockDim.x + threadIdx.x; w < (long)njac * pp; w += (long)gridDim.x * blockDim.x)
        D.fjac[(size_t)jac_list[w / pp] * D.QS + (w % pp)] = 0.;
}

// ---- kernel 2a: assemble residuals and forward-difference Jacobian columns ----------------------
// One thread per residual request, one thread per (Jacobian request, column).  This is the only
// solver kernel besides integrate_worklist that contains model code.
constexpr int ASM_MINB = 3;        // resident CTAs per SM asked of assemble_kernel (register cap 168; measured per 1e5-problem step: 191 ms uncapped at 230 registers, 174 ms at 168, 171 ms at 128 with more spills)
template <int MODEL>
__global__ void __launch_bounds__(128, ASM_MINB)
assemble_kernel(SolverDev D, int cur) {
    const int nres = D.counts[cur * 2 + 0], njac = D.analytic ? 0 : D.counts[cur * 2 + 1];
    const int *res_list = D.lists + (size_t)(cur * 2 + 0) * D.B;
    const int *jac_list = D.lists + (size_t)(cur * 2 + 1) * D.B;
    const int n = D.P;
    const long total = (long)nres + (long)njac * n;
    if (blockIdx.x == 0 && threadIdx.x == 0 && nres > 0) atomicAdd(D.counters + 4, (unsigned long long)nres);
    for (long w = (long)blockIdx.x * blockDim.x + threadIdx.x; w < total; w += (long)gridDim.x * blockDim.x) {
        if (w < nres) {
            const long b = res_list[w];
            const int *is = D.istate + b * I_COUNT;
            const int trial = 1 - is[I_BASE];
            const double *te = D.ends + ((b * 2 + trial) * D.M) * D.REC;
            double *out = (is[I_PHASE] == PH_F0) ? D.fvec + b * n : D.wa4 + b * n;
            assemble<MODEL>(*D.self, b, -1, 0.0, te, D.jends + (size_t)b * D.nJ * D.REC, out, 0, D.M - 1, nullptr);
        } else {
            const long w2 = w - nres;
            const long b = jac_list[w2 / n];
            const int j = (int)(w2 % n);
            const int *is = D.istate + b * I_COUNT;
            const double *be = D.ends + ((b * 2 + is[I_BASE]) * D.M) * D.REC;
            const double h = fd_step(D.xe[b * n + j], D.epsfcn);
            double *colj = D.fjac + (size_t)b * D.QS + (size_t)j * n;
            const double *fvec = D.fvec + b * n;
            // an unknown of node s enters segment s - 1 (as the right-hand state of its continuity rows) and
            // segment s (as its start point); a free time moves every segment
            const int N2 = 2 * Model<MODEL>::DIM, node = j / N2;
            const bool state_col = j < N2 * D.M;
            // fdjac1: the column was zero-filled (zero_fjac_kernel); only the reachable rows are written
            assemble<MODEL>(*D.self, b, j, h, be, D.jends + (size_t)b * D.nJ * D.REC, colj,
                            state_col ? max(node - 1, 0) : 0, state_col ? node : D.M - 1, fvec);
        }
    }
}

// ---- analytic-Jacobian path (modelOrder == 1, hybrj): variational segments ----------------------
// Restates model::ComputeTraj(isJac = 1) for the double integrator (doubleIntegrator.cpp:113-213): the
// extended state is X[0..N) plus the sensitivity rows X[N(k+1) + i] = dX_k / dX0_i, seeded with the
// identity (shooting.cpp:1003-1005).  Every sensitivity COLUMN obeys the same linear system, so a group
// of 16 lanes owns one segment: lane i < N integrates (X, Phi[:, i]) -- the state redundantly, identical
// in every lane -- with the same RK4 and combination order as the plain trajectory.
template <int MODEL> struct Variational { static constexpr bool HAS = false; };
template <> struct Variational<DOUBLE_INTEGRATOR> {
    static constexpr bool HAS = true;
    // (df/dX) phi with the reference's constant matrix (doubleIntegrator.cpp:161-172: -1 on the p_v
    // columns of the velocity rows whatever a_max and the saturation)
    SOCP_DEV static void rhs(const double *phi, double *d) {
        d[0] = phi[3]; d[1] = phi[4]; d[2] = phi[5];
        d[3] = -phi[9]; d[4] = -phi[10]; d[5] = -phi[11];
        d[6] = 0.; d[7] = 0.; d[8] = 0.;
        d[9] = -phi[6]; d[10] = -phi[7]; d[11] = -phi[8];
    }
    // doubleIntegrator::Hamiltonian(isJac = 1): (dH/dX, dH/dt)  (doubleIntegrator.cpp:293-296)
    SOCP_DEV static void hgrad(const double *X, double *g) {
        g[0] = 0.; g[1] = 0.; g[2] = 0.; g[3] = X[6]; g[4] = X[7]; g[5] = X[8];
        g[6] = X[3]; g[7] = X[4]; g[8] = X[5]; g[9] = -X[9]; g[10] = -X[10]; g[11] = -X[11]; g[12] = 0.;
    }
};

// one lane: (X, phi) over [t0, tf] with S RK4 steps; returns steps
template <int MODEL>
SOCP_DEV int var_traj_lane(const typename Model<MODEL>::Ctx &c, double *X, double *phi, double t0, double tf, int S) {
    typedef Model<MODEL> M;
    typedef Variational<MODEL> V;
    constexpr int N = M::N;
    const double dt = (tf - t0) / S;
    double t = t0;
    int steps = 0;
    while (t < (tf - dt / 2)) {
        const double h = (t + dt > tf) ? tf - t : dt, h2 = h / 2.0, h6 = h / 6.0;
        double F1[N], F23[N], F[N], Y[N], G1[N], G23[N], G[N], Z[N];
        M::rhs(c, t, X, F1); V::rhs(phi, G1);
#pragma unroll
        for (int i = 0; i < N; ++i) { Y[i] = X[i] + h2 * F1[i]; Z[i] = phi[i] + h2 * G1[i]; }
        M::rhs(c, t + h2, Y, F23); V::rhs(Z, G23);
#pragma unroll
        for (int i = 0; i < N; ++i) { Y[i] = X[i] + h2 * F23[i]; Z[i] = phi[i] + h2 * G23[i]; }
        M::rhs(c, t + h2, Y, F); V::rhs(Z, G);
#pragma unroll
        for (int i = 0; i < N; ++i) {
            F23[i] = F23[i] + F[i]; Y[i] = X[i] + h * F[i];
            G23[i] = G23[i] + G[i]; Z[i] = phi[i] + h * G[i];
        }
        M::rhs(c, t + h, Y, F); V::rhs(Z, G);
#pragma unroll
        for (int i = 0; i < N; ++i) {
            X[i] = X[i] + h6 * (F1[i] + (F[i] + 2.0 * F23[i]));
            phi[i] = phi[i] + h6 * (G1[i] + (G[i] + 2.0 * G23[i]));
        }
        t += dt;
        ++steps;
    }
    return steps;
}

// B extended trajectories (socp_traj_var_batch): 16 lanes per trajectory
template <int MODEL>
__global__ void __launch_bounds__(128)
traj_var_kernel(long B, int S, const double *__restrict__ mparams, const double *__restrict__ t0,
                const double *__restrict__ tf, const double *__restrict__ X0, double *__restrict__ Xf,
                unsigned long long *counter) {
    typedef Model<MODEL> M;
    constexpr int N = M::N, NV = N * (N + 1);
    const long b = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    const int i = threadIdx.x & 15;
    int steps = 0;
    if (b < B && i < N) {
        typename M::Ctx c;
        M::load(c, mparams + b * M::NP, nullptr);
        double X[N], phi[N];
#pragma unroll
        for (int k = 0; k < N; ++k) { X[k] = X0[b * NV + k]; phi[k] = X0[b * NV + N * (k + 1) + i]; }
        steps = var_traj_lane<MODEL>(c, X, phi, t0[b], tf[b], S);
#pragma unroll
        for (int k = 0; k < N; ++k) Xf[b * NV + N * (k + 1) + i] = phi[k];
        if (i == 0) {
#pragma unroll
            for (int k = 0; k < N; ++k) Xf[b * NV + k] = X[k];
        } else steps = 0;
    }
    count_steps(counter, steps);
}

// kernel 1': variational integration of every segment of the problems that asked for a Jacobian
// (hybrj).  vends = D.jends reinterpreted: [problem][segment][N (N + 1)].
template <int MODEL>
__global__ void __launch_bounds__(128)
integrate_var_worklist(SolverDev D, int cur) {
    typedef Model<MODEL> M;
    constexpr int N = M::N, NV = N * (N + 1);
    const int njac = D.counts[cur * 2 + 1];
    const int *jac_list = D.lists + (size_t)(cur * 2 + 1) * D.B;
    const long total = (long)njac * D.M;
    const int i = threadIdx.x & 15;
    int steps = 0;
    for (long w = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 4; w < total; w += ((long)gridDim.x * blockDim.x) >> 4) {
        const long b = jac_list[w / D.M];
        const int s = (int)(w % D.M);
        if (i >= N) continue;
        const double *xe = D.xe + b * D.P;
        const int nm = N * D.M;
        double t1, t2;
        typename M::Ctx c;
        segment_setup<MODEL>(D, D.time + b * (D.M + 1), [&](int k) { return xe[nm + k]; }, s, D.mparams + b * M::NP, t1, t2, c);
        double X[N], phi[N];
#pragma unroll
        for (int k = 0; k < N; ++k) { X[k] = xe[N * s + k]; phi[k] = (k == i) ? 1. : 0.; }
        const int st = var_traj_lane<MODEL>(c, X, phi, t1, t2, D.S);
        double *out = D.jends + ((size_t)b * D.M + s) * NV;
#pragma unroll
        for (int k = 0; k < N; ++k) out[N * (k + 1) + i] = phi[k];
        if (i == 0) {
#pragma unroll
            for (int k = 0; k < N; ++k) out[k] = X[k];
            steps += st;
        }
    }
    count_steps(D.counters, steps);
}

// kernel 2a': shooting::ShootingFunctionJacobian (shooting.cpp:996-1130) from the segment sensitivities,
// written column-major as StaticShootingFunctionJacobian transposes it (:889-893).  One thread per problem.
template <int MODEL>
__global__ void __launch_bounds__(128)
assemble_jac_kernel(SolverDev D, int cur) {
    typedef Model<MODEL> M;
    typedef Variational<MODEL> V;
    constexpr int N = M::N, n = M::DIM, NV = N * (N + 1);
    const int njac = D.counts[cur * 2 + 1];
    const int *jac_list = D.lists + (size_t)(cur * 2 + 1) * D.B;
    const int P = D.P;
    for (long w = (long)blockIdx.x * blockDim.x + threadIdx.x; w < njac; w += (long)gridDim.x * blockDim.x) {
        const long b = jac_list[w];
        const double *xe = D.xe + b * P;
        double *J = D.fjac + (size_t)b * D.QS;
        auto put = [&](int row, int col, double v) { J[row + (size_t)col * P] = v; };     // dF_row / dx_col
        for (int e = 0; e < P * P; ++e) J[e] = 0.;
        const int nm = N * D.M;
        const double *time_b = D.time + b * (D.M + 1);
        auto xfree = [&](int k) { return xe[nm + k]; };
        typename M::Ctx c;
        double t1, t2;      // the node times of segment i in the loop below
        segment_setup<MODEL>(D, time_b, xfree, 0, D.mparams + b * M::NP, t1, t2, c);
        int nbr = nm;
        // rows of a boundary function: FIXED component j -> sensitivity row j, FREE -> row j + n; with a
        // free time one more column (the flow) and one more row (dH) (model.hpp:104-120, :149-183)
        auto boundary = [&](const double *Xs, const double *Phi, double t, const int *mode, bool identity, int row0, int col0,
                            bool withH) {
            double f[N], g[N + 1];
            if (withH) { M::rhs(c, t, Xs, f); V::hgrad(Xs, g); }
            for (int j = 0; j < n; ++j) {
                const int r = (mode[j] == SOCP_FREE) ? j + n : j;
                for (int q = 0; q < N; ++q) put(row0 + j, col0 + q, identity ? (q == r ? 1. : 0.) : Phi[N * r + q]);
                if (withH) put(row0 + j, nbr, f[r]);
            }
            if (withH) {
                for (int q = 0; q < N; ++q) {
                    double acc = 0.;
                    for (int k = 0; k < N; ++k) acc += g[k] * (identity ? (k == q ? 1. : 0.) : Phi[N * k + q]);
                    put(nbr, col0 + q, acc);
                }
                double acc = 0.;
                for (int k = 0; k < N; ++k) acc += g[k] * f[k];
                put(nbr, nbr, acc + g[N]);
            }
        };
        for (int i = 0; i < D.M; ++i) {
            double sw_unused[2];
            timeline_pair(D, time_b, xfree, i, t1, t2, sw_unused);
            const double *seg = D.jends + ((size_t)b * D.M + i) * NV;     // X(t2) and Phi = dX(t2)/dX(t1)
            const double *Xtf = seg, *Phi = seg + N;                      // Phi[N k + q] = dX_k / dX0_q
            const int index = N * (i + 1);
            if (i == 0) {
                const bool withH = D.mode_t[0] != SOCP_FIXED;
                boundary(xe, nullptr, t1, D.mode_X[0], true, 0, 0, withH);
                if (withH) nbr += 1;
            }
            if (i < D.M - 1) {
                const double *Xp = xe + index;
                const bool free_t = D.mode_t[i + 1] == SOCP_FREE;
                double fxt[N], fxp[N];
                M::rhs(c, t2, Xtf, fxt);
                M::rhs(c, t2, Xp, fxp);
                // shooting::MultipleShootingFunction(isJac = 1), shooting.cpp:1511-1576.  The derivative with
                // respect to the free node time goes to that time's column -- and, as the reference copies a
                // (4 dim + 1)-wide block (shooting.cpp:1063-1067), also to column index + N (a stray entry
                // unless that IS the time column, as in the two-segment demo); reproduced for parity.
                auto tcol = [&](int row, double v) { if (index + N < P) put(row, index + N, v); put(row, nbr, v); };
                for (int j = 0; j < n; ++j) {
                    const int m = D.mode_X[i + 1][j];
                    if (m == SOCP_FIXED) {
                        for (int q = 0; q < N; ++q) {
                            put(index + j, index - N + q, Phi[N * j + q]);
                            put(index + j + n, index + q, (q == j) ? 1. : 0.);
                        }
                        if (free_t) { tcol(index + j, fxt[j]); tcol(index + j + n, fxp[j]); }
                    } else if (m == SOCP_CONTINUOUS) {
                        for (int q = 0; q < N; ++q) {
                            put(index + j, index - N + q, Phi[N * j + q]);
                            put(index + j, index + q, (q == j) ? -1. : -0.);
                            put(index + j + n, index - N + q, Phi[N * (j + n) + q]);
                            put(index + j + n, index + q, (q == j + n) ? -1. : -0.);
                        }
                        if (free_t) { tcol(index + j, fxt[j] - fxp[j]); tcol(index + j + n, fxt[j + n] - fxp[j + n]); }
                    }
                }
                if (free_t) {
                    // model::SwitchingTimesFunction(isJac = 1), model.hpp:306-327
                    double gX[N + 1], gP[N + 1];
                    V::hgrad(Xtf, gX);
                    V::hgrad(Xp, gP);
                    for (int q = 0; q < N; ++q) {
                        double a1 = 0., a2 = 0.;
                        for (int k = 0; k < N; ++k) { a1 += gX[k] * Phi[N * k + q]; a2 -= gP[k] * ((k == q) ? 1. : 0.); }
                        put(nbr, index - N + q, a1);
                        put(nbr, index + q, a2);
                    }
                    double a = 0.;
                    for (int k = 0; k < N; ++k) a += gX[k] * fxt[k] - gP[k] * fxp[k];
                    put(nbr, nbr, a + (gX[N] - gP[N]));
                    nbr += 1;
                }
            }
            if (i == D.M - 1) {
                const bool withH = D.mode_t[D.M] != SOCP_FIXED;
                boundary(Xtf, Phi, t2, D.mode_X[D.M], false, n, N * i, withH);
                if (withH) nbr += 1;
            }
        }
    }
}

// ---- MINPACK linear algebra on a thread group --------------------------------------------------
// Q (fjac) is column-major with leading dimension ldq, r is the packed upper triangle stored by
// rows (cminpack conventions).  The pointers may be shared or global memory.  Thread mappings are
// chosen so that a group touches consecutive addresses (coalesced in HBM, conflict-free in shared
// memory when ldq is odd).  Every routine starts and ends with a group barrier.

// copy with eight independent loads in flight per thread (a plain loop serialises on the memory latency)
template <int G> SOCP_DEV void gcopy(double *dst, const double *src, int n) {
    const int tid = threadIdx.x % G;
    for (int base = 0; base < n; base += 8 * G) {
        double t[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) { const int i = base + k * G + tid; t[k] = (i < n) ? src[i] : 0.; }
#pragma unroll
        for (int k = 0; k < 8; ++k) { const int i = base + k * G + tid; if (i < n) dst[i] = t[k]; }
    }
}

// global -> shared with cp.async (LDGSTS): every element of the copy is in flight at once, no register
// staging; complete with gcopy_async_wait() + a barrier.  dst must be shared memory.
template <int G> SOCP_DEV void gcopy_async(double *dst, const double *src, int n) {
    for (int i = threadIdx.x % G; i < n; i += G) __pipeline_memcpy_async(dst + i, src + i, sizeof(double));
}
SOCP_DEV void gcopy_async_wait() {
    __pipeline_commit();
    __pipeline_wait_prior(0);
}

// ask L2 for [p, p + bytes): one prefetch per 128-byte line, spread over the group
template <int G> SOCP_DEV void l2_prefetch(const void *p, size_t bytes) {
    const char *c = (const char *)p;
    for (size_t off = (size_t)(threadIdx.x % G) * 128; off < bytes; off += (size_t)G * 128)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(c + off));
}

SOCP_DEV double warp_sum(double v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

SOCP_DEV int rowstart(int n, int j) { return j * n - (j * (j - 1)) / 2; }

// dot product with four independent accumulators (the 8-cycle DFMA latency would otherwise pace a
// single running sum); fixed summation tree, so the result is deterministic
SOCP_DEV double dot4(const double *a, const double *b, int m) {
    double s0 = 0., s1 = 0., s2 = 0., s3 = 0.;
    int i = 0;
    for (; i + 3 < m; i += 4) {
        s0 = fma(a[i], b[i], s0); s1 = fma(a[i + 1], b[i + 1], s1);
        s2 = fma(a[i + 2], b[i + 2], s2); s3 = fma(a[i + 3], b[i + 3], s3);
    }
    for (; i < m; ++i) s0 = fma(a[i], b[i], s0);
    return (s0 + s1) + (s2 + s3);
}

// y[i] -= t * x[i] with the operands of four elements fetched before the first store (x and y never
// overlap here, which the compiler cannot know: the plain loop serialises load -> FMA -> store per element)
SOCP_DEV void axpy_sub4(double *y, const double *x, double t, int m) {
    int i = 0;
    for (; i + 3 < m; i += 4) {
        const double x0 = x[i], x1 = x[i + 1], x2 = x[i + 2], x3 = x[i + 3];
        const double y0 = y[i], y1 = y[i + 1], y2 = y[i + 2], y3 = y[i + 3];
        y[i] = __fma_rn(-t, x0, y0); y[i + 1] = __fma_rn(-t, x1, y1); y[i + 2] = __fma_rn(-t, x2, y2); y[i + 3] = __fma_rn(-t, x3, y3);
    }
    for (; i < m; ++i) y[i] = __fma_rn(-t, x[i], y[i]);
}

// Column layouts of the matrix the Jacobian phase factors.  at(k, i) is the element in row i of column k; the rows of
// column k outside [lo(k), end(k)) are exact zeros and are not stored.
struct DenseCols {                       // column-major, leading dimension lda
    double *a;
    int lda, n;
    SOCP_DEV double *at(int k, int i) const { return a + i + (size_t)k * lda; }
    SOCP_DEV int lo(int) const { return 0; }
    SOCP_DEV int end(int) const { return n; }
};
struct BandCols {                        // the structural band of SolverDev::band_lo / band_off, columns back to back
    double *a;
    const int *lo_, *off_;
    SOCP_DEV double *at(int k, int i) const { return a + off_[k] + (i - lo_[k]); }
    SOCP_DEV int lo(int k) const { return lo_[k]; }
    SOCP_DEV int end(int k) const { return lo_[k] + (off_[k + 1] - off_[k]); }
};

// qrfac (no pivoting) fused with "qtf = Q^T fvec" (the Householder reflections are applied to
// qtf as one more column); rdiag/acnorm as in MINPACK.  One thread per column.
// Both routines skip work on EXACT zeros: hi[k] is the last row of column k that is not an exact zero
// (the shooting Jacobian is block bidiagonal plus a border, and Householder reflections keep the
// lower band), so reflector j only spans rows j..hi[j] and a column whose dot product with it is an
// exact zero is left alone.  The skipped operations would add or subtract exact zeros: the factors are
// the ones the dense MINPACK loops produce (up to the sign of a zero).
// With a BandCols layout, a column whose stored rows do not hold all of rows j..hi[j] is one the reflector cannot
// reach (the band holds every row that fill-in can reach, jac_band): its dot product would be an exact zero.
template <int G, class C>
__device__ void qrfac_g(int n, C a, double *rdiag, double *acnorm, double *qtf, double *red, int rot, int *hi) {
    // `rot` rotates the warp that owns the first columns: the active columns always start at thread 0, so
    // without it the co-resident CTAs of an SM would all load the same scheduler (see seq_warp)
    const int tid = (threadIdx.x + 32 * rot) % G;
    gsync<G>();
    for (int j = tid >> 5; j < n; j += G / 32) {       // column norms, one warp per column
        const double v = enorm_rows(n, a.at(j, a.lo(j)), a.lo(j), a.end(j));
        if ((tid & 31) == 0) acnorm[j] = v;
    }
    for (int k = tid; k <= n; k += G) {                // last non-zero row of every column (qtf: dense)
        int last = (k < n) ? 0 : n - 1;
        if (k < n) {
            const int lo = a.lo(k);
            const double *ck = a.at(k, lo);
            for (int i = a.end(k) - 1; i > 0 && i >= lo; --i) if (ck[i - lo] != 0.) { last = i; break; }
        }
        hi[k] = last;
    }
    gsync<G>();
    for (int j = 0; j < n; ++j) {
        double *cj = a.at(j, j);                       // rows j .. hj of the reflector
        const int hj = max(hi[j], j), len = hj - j + 1;
        double ajnorm = enorm_g<G>(len, cj, red);
        if (ajnorm != 0.) {
            if (cj[0] < 0.) ajnorm = -ajnorm;
            gsync<G>();
            for (int i = tid; i < len; i += G) {
                double v = cj[i] / ajnorm;
                if (i == 0) v += 1.;
                cj[i] = v;
            }
            gsync<G>();
            const double ajj = cj[0];
            for (int k = j + 1 + tid; k <= n; k += G) {  // remaining columns, and qtf as column n
                if (k < n && (j < a.lo(k) || hj >= a.end(k))) continue;
                double *ck = (k < n) ? a.at(k, j) : qtf + j;
                const double sum = dot4(cj, ck, len);
                if (sum != 0.) {
                    const double temp = sum / ajj;
                    axpy_sub4(ck, cj, temp, len);
                    if (hi[k] < hj) hi[k] = hj;
                }
            }
        }
        if (tid == 0) rdiag[j] = -ajnorm;
        gsync<G>();
    }
}

// ---- register-window accumulation of Q (block-bidiagonal + border Jacobians) ------------------------------------
// The shooting Jacobian of a problem without free interior times is block bidiagonal (blocks of NB = 2 dim rows and
// columns) plus a border, and Householder reflector k then spans at most the rows of TWO blocks: k .. c0(k) + W - 1,
// c0(k) = NB (k / NB) the first column of its panel, W = 2 NB.  window_ok() checks exactly that on the matrix at hand
// (last non-zero row of every column); when it holds, a thread can keep the W rows of ITS column that a whole panel
// of NB reflectors can touch in registers -- static indices, everything unrolled -- instead of walking shared memory
// one barrier-separated reflector at a time.
//   qform_p : accumulation of Q.  Column j of Q starts as e_j and only ever sees reflectors k <= j, every column is
//             independent of the others: NO barrier in the whole routine.  The reflectors stay where qrfac left them
//             (shared memory, read-only here); the finished rows of a column go straight to GLOBAL memory, block of NB
//             rows by block, so Q never passes through shared memory again.
// Summation order: a reflector's dot product runs over the window rows kk .. W-1 with four running sums ((t - kk) & 3);
// rows past the reflector's last non-zero row add exact zeros.  Same values as qform_g up to the association of the
// last partial group of four (qform_g sends a tail of up to three elements to its first sum).
template <int G>
SOCP_DEV bool window_ok(int n, int NB, const int *hi, int *flag) {
    const int tid = threadIdx.x % G;
    if (tid == 0) *flag = 1;
    gsync<G>();
    for (int k = tid; k < n; k += G)
        if (max(hi[k], k) >= (k / NB) * NB + 2 * NB) *flag = 0;
    gsync<G>();
    return *flag != 0;
}

// dot4 over the window: sum_{i < len} x[i] y[i] with dot4's association (four running sums over complete groups of four,
// the incomplete last group on the first sum).  x(t), y(t) give element t of the window (static t), kk is the window
// index of element 0; `len` is uniform over the threads, so the branches are uniform too.
#define SOCP_WIN_DOT4(W, kk, len, X, Y, sum)                                                      \
    do {                                                                                          \
        double s0_ = 0., s1_ = 0., s2_ = 0., s3_ = 0.;                                            \
        _Pragma("unroll") for (int g_ = 0; g_ < ((W) - (kk) + 3) / 4; ++g_) {                      \
            const int t_ = (kk) + 4 * g_;                                                         \
            if (4 * g_ + 3 < (len)) {                                                             \
                if (t_ + 3 < (W)) {                                                               \
                    s0_ = fma(X(t_), Y(t_), s0_); s1_ = fma(X(t_ + 1), Y(t_ + 1), s1_);           \
                    s2_ = fma(X(t_ + 2), Y(t_ + 2), s2_); s3_ = fma(X(t_ + 3), Y(t_ + 3), s3_);   \
                }                                                                                 \
            } else {                                                                              \
                if (4 * g_ < (len) && t_ < (W)) s0_ = fma(X(t_), Y(t_), s0_);                     \
                if (4 * g_ + 1 < (len) && t_ + 1 < (W)) s0_ = fma(X(t_ + 1), Y(t_ + 1), s0_);     \
                if (4 * g_ + 2 < (len) && t_ + 2 < (W)) s0_ = fma(X(t_ + 2), Y(t_ + 2), s0_);     \
            }                                                                                     \
        }                                                                                         \
        (sum) = (s0_ + s1_) + (s2_ + s3_);                                                        \
    } while (0)

template <int G, int NB, class C>
__device__ void qform_p(int n, C a, const int *hi, double *gq) {
    constexpr int W = 2 * NB;
    const int j = threadIdx.x % G;                 // this thread's column of Q
    if (j >= n) return;
    int p = j / NB;
    double c[W];
#pragma unroll
    for (int t = 0; t < W; ++t) c[t] = (t == j - p * NB) ? 1. : 0.;
    double *out = gq + (size_t)j * n;
    // rows below the first window are zeros of e_j for good
    for (int r = p * NB + W; r < n; ++r) out[r] = 0.;
#pragma unroll 1
    for (; p >= 0; --p) {
        const int c0 = p * NB;
        // reflectors of this panel that act on column j: k = min(j, c0 + NB - 1) .. c0, highest first
#pragma unroll
        for (int kk = NB - 1; kk >= 0; --kk) {
            const int k = c0 + kk;
            if (k > j || k >= n) continue;
            const double *v = a.at(k, k) - kk;                 // v[t] = reflector k at row c0 + t (t >= kk)
            const double wk = v[kk];
            if (wk == 0.) continue;                            // the identity
            const int len = max(hi[k], k) - k + 1;             // rows k .. hk; exact zeros below
#define SOCP_CX(t) c[t]
#define SOCP_VX(t) v[t]
            double sum;
            SOCP_WIN_DOT4(W, kk, len, SOCP_CX, SOCP_VX, sum);
            if (sum != 0.) {
                const double temp = sum / wk;
#pragma unroll
                for (int t = kk; t < W; ++t) if (t - kk < len) c[t] = __fma_rn(-temp, v[t], c[t]);
            }
        }
        // rows c0 + NB .. c0 + W - 1 are final (lower panels stop at row c0 + NB - 1): out they go, and the window moves up
#pragma unroll
        for (int t = NB; t < W; ++t) if (c0 + t < n) out[c0 + t] = c[t];
        if (p == 0) {
#pragma unroll
            for (int t = 0; t < NB; ++t) if (t < n) out[t] = c[t];
        } else {
#pragma unroll
            for (int t = W - 1; t >= NB; --t) c[t] = c[t - NB];
#pragma unroll
            for (int t = 0; t < NB; ++t) c[t] = 0.;
        }
    }
}

// copy R into packed storage (upper triangle by rows), diagonal from rdiag; the rows above a column's stored
// ones are zeros
template <int G, class C>
__device__ void pack_r_g(int n, C a, const double *rdiag, double *r) {
    const int tid = threadIdx.x % G;
    for (int j = tid; j < n; j += G) {
        int l = j;
        const int lo = a.lo(j);
        for (int i = 0; i < j; ++i) { r[l] = (i < lo) ? 0. : *a.at(j, i); l += n - 1 - i; }
        r[l] = rdiag[j];
    }
    gsync<G>();
}

// qform: accumulate Q (n x n) in place from the Householder vectors; wa is scratch [n]
template <int G>
__device__ void qform_g(int n, double *q, int lda, double *wa, int rot, const int *hi) {
    const int tid = (threadIdx.x + 32 * rot) % G;
    for (int j = 1 + tid; j < n; j += G)
        for (int i = 0; i < j; ++i) q[i + (size_t)j * lda] = 0.;
    gsync<G>();
    for (int l = 0; l < n; ++l) {
        const int k = n - 1 - l;
        double *ck = q + (size_t)k * lda;
        const int hk = max(hi[k], k), len = hk - k + 1;    // reflector k spans rows k..hk (zeros below)
        for (int i = k + tid; i <= hk; i += G) { wa[i] = ck[i]; ck[i] = (i == k) ? 1. : 0.; }
        gsync<G>();
        const double wk = wa[k];
        if (wk != 0.) {
            for (int j = k + tid; j < n; j += G) {
                double *cj = q + (size_t)j * lda;
                const double sum = dot4(cj + k, wa + k, len);
                if (sum != 0.) {
                    const double temp = sum / wk;
                    axpy_sub4(cj + k, wa + k, temp, len);
                }
            }
        }
        gsync<G>();
    }
}

// y[i] = add[i] + sum_{j >= i} R(i,j) v[j]   (one thread per packed row, four running sums: a row per
// warp with a shuffle reduction per row cost 10x the instructions -- 85 reductions per call, two calls
// per Broyden iteration -- and was the top line of the kernel's profile)
template <int G>
__device__ void rmulv_g(int n, const double *r, const double *v, const double *add, double *y) {
    const int tid = threadIdx.x % G;
    gsync<G>();
    for (int i = tid; i < n; i += G)
        y[i] = (add ? add[i] : 0.) + dot4(r + rowstart(n, i), v + i, n - i);
    gsync<G>();
}

// steps j = min(32 PH + 31, n - 1) .. 32 PH of dogleg's back substitution for n <= 96 (see dogleg_g)
template <int PH>
SOCP_DEV void backsub_phase(int n, const double *r, const double *dinvs, const double *ds, int lane,
                            double &b0, double &b1, double &b2, int &p0, int &p1, int &p2) {
    for (int j = min(32 * PH + 31, n - 1); j >= 32 * PH; --j) {
        const double bj = (PH == 0) ? b0 : (PH == 1) ? b1 : b2;
        const double d = ds[j], dinv = dinvs[j];
        const double q0 = bj * dinv;
        const double xj = __shfl_sync(0xffffffffu, fma(fma(-q0, d, bj), dinv, q0), j & 31);
        // rows i < j: every row of the slots below PH, the rows i < j of slot PH
        const double r0 = (PH > 0 || lane < j) ? r[p0] : 0.;
        b0 = fma(-r0, xj, b0);
        if (PH >= 1) { const double r1 = (PH > 1 || lane + 32 < j) ? r[p1] : 0.; b1 = fma(-r1, xj, b1); }
        if (PH == 2) { const double r2 = (lane + 64 < j) ? r[p2] : 0.; b2 = fma(-r2, xj, b2); }
        if (lane == (j & 31)) { if (PH == 0) b0 = xj; else if (PH == 1) b1 = xj; else b2 = xj; }
        --p0; --p1; --p2;
    }
}

// dogleg: x <- step; wa1, wa2 scratch
template <int G>
__device__ void dogleg_g(int n, const double *r, const double *diag, const double *qtb, double delta,
                         double *x, double *wa1, double *wa2, double *red, int seqw, bool clk_on = false,
                         unsigned long long *clk_counters = nullptr) {
    long long sub_t0 = clock64();
    const int tid = threadIdx.x % G;
    const int lane = threadIdx.x & 31;
    gsync<G>();
    // Gauss-Newton direction R x = qtb by back substitution, column-oriented so that the only value
    // on the sequential chain is x[j] itself: each lane of warp 0 owns the rows i = lane (mod 32) and
    // keeps their running right-hand sides in x[i]; x[j] travels by one shuffle per step and the
    // right-hand side of the next pivot row is carried in a register.  The effective diagonal
    // (MINPACK replaces a zero pivot by epsmch * max|column|) is prepared in wa2 by all threads.
    for (int j = tid; j < n; j += G) {
        double temp = r[rowstart(n, j)];
        if (temp == 0.) {
            int l = j;
            for (int i = 0; i <= j; ++i) { temp = fmax(temp, fabs(r[l])); l += n - 1 - i; }
            temp = EPSMCH * temp;
            if (temp == 0.) temp = EPSMCH;
        }
        wa2[j] = temp;
        wa1[j] = 1. / temp;
        x[j] = qtb[j];
    }
    gsync<G>();
    if ((tid >> 5) == seqw) {
        if (n <= 96) {
            // every lane keeps the running right-hand sides of its rows i = lane, lane + 32, lane + 64 in
            // registers; per step: corrected quotient in the owner lane, one shuffle, three predicated FMAs
            double b0 = (lane < n) ? x[lane] : 0., b1 = (lane + 32 < n) ? x[lane + 32] : 0., b2 = (lane + 64 < n) ? x[lane + 64] : 0.;
            // p_k: index of R(i_k, j) in the packed rows, moves one to the left per step
            int p0 = rowstart(n, lane) + (n - 1 - lane), p1 = rowstart(n, lane + 32) + (n - 1 - lane - 32),
                p2 = rowstart(n, lane + 64) + (n - 1 - lane - 64);
            // three phases of 32 steps (pivots in slot 2, 1, 0): the slots above the pivot's are finished, the
            // ones below are active in every step
            backsub_phase<2>(n, r, wa1, wa2, lane, b0, b1, b2, p0, p1, p2);
            backsub_phase<1>(n, r, wa1, wa2, lane, b0, b1, b2, p0, p1, p2);
            backsub_phase<0>(n, r, wa1, wa2, lane, b0, b1, b2, p0, p1, p2);
            if (lane < n) x[lane] = b0;
            if (lane + 32 < n) x[lane + 32] = b1;
            if (lane + 64 < n) x[lane + 64] = b2;
        } else {
        double bj = x[n - 1];                                  // rhs of the pivot row (owner lane)
        for (int j = n - 1; j >= 0; --j) {
            const int owner = j & 31, next_owner = (j - 1) & 31;
            double cr = 0., cx = 0.;                           // next pivot row: fetched before x[j] is known
            if (j > 0 && lane == next_owner) { cr = r[rowstart(n, j - 1) + 1]; cx = x[j - 1]; }
            // x[j] = bj / d without a divide on the chain: reciprocal (prepared above), residual, correction
            const double d = wa2[j], dinv = wa1[j];
            const double q0 = bj * dinv;
            const double xj = __shfl_sync(0xffffffffu, fma(fma(-q0, d, bj), dinv, q0), owner);
            if (lane == owner) x[j] = xj;
            if (j > 0 && lane == next_owner) { bj = cx - cr * xj; x[j - 1] = bj; }
            for (int i = lane; i < j - 1; i += 32) x[i] -= r[rowstart(n, i) + (j - i)] * xj;
        }
        }
    }
    gsync<G>();
    SOCP_SUB(5);
    for (int j = tid; j < n; j += G) { wa1[j] = 0.; wa2[j] = diag[j] * x[j]; }
    gsync<G>();
    const double qnorm = enorm_g<G>(n, wa2, red);
    if (qnorm <= delta) { gsync<G>(); return; }
    // scaled gradient direction: wa1 = (R^T qtb) / diag   (one thread per column)
    for (int i = tid; i < n; i += G) {
        double s = 0.;
        int l = i;                                             // R(j, i) in the packed rows
        for (int j = 0; j <= i; ++j) { s += r[l] * qtb[j]; l += n - 1 - j; }
        wa1[i] = s / diag[i];
    }
    gsync<G>();
    const double gnorm = enorm_g<G>(n, wa1, red);
    double sgnorm = 0., alpha = delta / qnorm;
    if (gnorm != 0.) {
        gsync<G>();
        for (int j = tid; j < n; j += G) wa1[j] = (wa1[j] / gnorm) / diag[j];
        rmulv_g<G>(n, r, wa1, nullptr, wa2);
        double temp = enorm_g<G>(n, wa2, red);
        sgnorm = (gnorm / temp) / temp;
        alpha = 0.;
        if (sgnorm < delta) {
            const double bnorm = enorm_g<G>(n, qtb, red);
            temp = (bnorm / gnorm) * (bnorm / qnorm) * (sgnorm / delta);
            const double dq = delta / qnorm, sd = sgnorm / delta;
            temp = temp - dq * (sd * sd) + sqrt((temp - dq) * (temp - dq) + (1. - dq * dq) * (1. - sd * sd));
            alpha = (dq * (1. - sd * sd)) / temp;
        }
    }
    const double temp = (1. - alpha) * fmin(sgnorm, delta);
    gsync<G>();
    for (int j = tid; j < n; j += G) x[j] = temp * wa1[j] + alpha * x[j];
    gsync<G>();
    SOCP_SUB(6);
}

// Givens rotation that maps (a, b) to (rho, 0) with MINPACK's conventions (r1updt): the coefficient
// of the larger operand is positive.  One rsqrt instead of MINPACK's divide / sqrt / divide keeps
// the sequential chains short; when a square could leave the double range the ratio form is used.
SOCP_DEV void givens(double a, double b, double &c, double &sgl) {
    const double mx = fmax(fabs(a), fabs(b));
    if (mx < 1e140 && mx > 1e-140) {
        const double rinv = rsqrt(a * a + b * b);
        if (fabs(a) < fabs(b)) { sgl = fabs(b) * rinv; c = copysign(a * rinv, a) * copysign(1., b); }
        else { c = fabs(a) * rinv; sgl = copysign(b * rinv, b) * copysign(1., a); }
    } else if (fabs(a) < fabs(b)) {
        const double cotan = a / b;
        sgl = .5 / sqrt(.25 + .25 * (cotan * cotan));
        c = sgl * cotan;
    } else {
        const double tn = b / a;
        c = .5 / sqrt(.25 + .25 * (tn * tn));
        sgl = c * tn;
    }
}
// what r1mpyq needs to rebuild the rotation (MINPACK's tau)
SOCP_DEV double givens_tau(double a, double b, double c, double sgl) {
    if (fabs(a) < fabs(b)) return (fabs(c) * DBL_MAX > 1.) ? 1. / c : 1.;
    return sgl;
}

// steps j = 32 PH .. j_end - 1 of the second sweep of r1updt for n <= 96 (see r1updt_g): w in registers, three
// slots per lane (i = lane, lane + 32, lane + 64)
template <int PH>
SOCP_DEV void sweep2_phase(int n, double *s, double *cs, double *sn, double *tmp, int lane, int j_end,
                           double &w0, double &w1, double &w2, double &wj, double &sjj, int &jj) {
    const unsigned FULL = 0xffffffffu;
    const int i0 = lane, i1 = lane + 32, i2 = lane + 64;
    const bool in1 = i1 < n, in2 = i2 < n;
    for (int j = 32 * PH; j < j_end; ++j) {
        const bool a0 = PH == 0 && i0 > j && i0 < n;
        const bool a1 = PH == 0 ? in1 : (PH == 1 && i1 > j && in1);
        const bool a2 = PH <= 1 ? in2 : (i2 > j && in2);
        const int base = jj - j;
        double s0 = 0., s1 = 0., s2 = 0.;
        if (PH == 0) s0 = a0 ? s[base + i0] : 0.;
        if (PH <= 1) s1 = a1 ? s[base + i1] : 0.;
        s2 = a2 ? s[base + i2] : 0.;
        const int jjn = jj + (n - j);
        const double sjj_next = s[jjn];
        double c = 1., sgl = 0.;
        const bool rot = wj != 0.;                         // uniform
        if (rot) givens(sjj, wj, c, sgl);
        if (rot) {
            if (PH == 0 && a0) s[base + i0] = fma(c, s0, sgl * w0);
            if (PH <= 1 && a1) s[base + i1] = fma(c, s1, sgl * w1);
            if (a2) s[base + i2] = fma(c, s2, sgl * w2);
            if (PH == 0 && a0) w0 = fma(c, w0, -sgl * s0);
            if (PH <= 1 && a1) w1 = fma(c, w1, -sgl * s1);
            if (a2) w2 = fma(c, w2, -sgl * s2);
        }
        if (lane == (j & 31)) {
            if (rot) { s[jj] = fma(c, sjj, sgl * wj); cs[j] = c; sn[j] = sgl; }
            tmp[j] = rot ? ((fabs(sjj) < fabs(wj)) ? 1. : 0.) : 2.;
        }
        // the next pivot w[j + 1] sits in slot PH, or in the next slot at the end of the phase
        const bool wrap = ((j + 1) & 31) == 0;
        const double pick = (PH == 0) ? (wrap ? w1 : w0) : (PH == 1) ? (wrap ? w2 : w1) : w2;
        wj = __shfl_sync(FULL, pick, (j + 1) & 31);
        sjj = sjj_next;
        jj = jjn;
    }
}

// r1updt on the packed upper-triangular factor (m == n): (R + u v^T) -> R' with the 2(n-1) Givens
// rotations recorded in v and w for r1mpyq.  cs/sn are scratch [n] each, tmp is scratch [2n].
template <int G>
__device__ void r1updt_g(int n, double *s, const double *u, double *v, double *w, double *cs, double *sn, double *tmp,
                         int seqw, bool clk_on = false, unsigned long long *clk_counters = nullptr) {
    long long sub_t0 = clock64();
    const int tid = threadIdx.x % G;
    const int lane = threadIdx.x & 31;
    const unsigned FULL = 0xffffffffu;
    gsync<G>();
    // First sweep (j = n-2 .. 0).  Rotation j is built from v[j] and the running value vn, which
    // before step j is +-sqrt(sum_{k > j} v[k]^2) carrying the sign of the entry that last dominated
    // (|vn| < |v[k]|), or of v[n-1].  Both are suffix scans, so warp 0 forms all rotations at once
    // instead of walking the scalar recurrence.
    if ((tid >> 5) == seqw) {
        double *SS = tmp;                              // SS[k] = sum_{q >= k} v[q]^2
        int *IDX = (int *)(tmp + n);                   // smallest dominating index above k within the lane's chunk
        double *TAU = w;                               // w is written only after this phase
        const int per = (n + 31) >> 5;                 // contiguous chunk of indices per lane
        const int lo = min(lane * per, n), hi = min(lo + per, n);
        double vmax = 0.;
        for (int k = lo; k < hi; ++k) vmax = fmax(vmax, fabs(v[k]));
        for (int off = 16; off > 0; off >>= 1) vmax = fmax(vmax, __shfl_xor_sync(FULL, vmax, off));
        if (vmax < 1e140 && (vmax > 1e-140 || vmax == 0.)) {
            double acc = 0.;
            for (int k = hi - 1; k >= lo; --k) { acc += v[k] * v[k]; SS[k] = acc; }
            double run = acc;                          // inclusive suffix scan over the lanes
            for (int off = 1; off < 32; off <<= 1) {
                const double t = __shfl_down_sync(FULL, run, off);
                if (lane + off < 32) run += t;
            }
            double above = __shfl_down_sync(FULL, run, 1);
            if (lane == 31) above = 0.;
            for (int k = lo; k < hi; ++k) SS[k] += above;
            __syncwarp();
            int best = n - 1;                          // smallest dominating index in this chunk so far
            for (int k = min(hi - 1, n - 2); k >= lo; --k) {
                IDX[k] = best;
                if (v[k] != 0. && sqrt(SS[k + 1]) < fabs(v[k])) best = k;
            }
            int runm = best;
            for (int off = 1; off < 32; off <<= 1) {
                const int t = __shfl_down_sync(FULL, runm, off);
                if (lane + off < 32) runm = min(runm, t);
            }
            int upm = __shfl_down_sync(FULL, runm, 1); // smallest dominating index above this chunk
            if (lane == 31) upm = n - 1;
            for (int k = min(hi - 1, n - 2); k >= lo; --k) {
                const double vj = v[k];
                double c = 2., sgl = 0., tau = 0.;     // c == 2 marks "no rotation"
                if (vj != 0.) {
                    const int src = (IDX[k] != n - 1) ? IDX[k] : upm;
                    const double m = copysign(sqrt(SS[k + 1]), v[src]);
                    givens(m, vj, c, sgl);
                    tau = givens_tau(m, vj, c, sgl);
                }
                cs[k] = c; sn[k] = sgl; TAU[k] = tau;
            }
            double vn_final = 0.;
            if (lane == 0) vn_final = copysign(sqrt(SS[0]), v[runm]);
            __syncwarp();                              // every read of v is done
            for (int k = min(hi - 1, n - 2); k >= lo; --k) if (cs[k] < 1.5) v[k] = TAU[k];
            if (lane == 0) v[n - 1] = vn_final;
        } else if (lane == 0) {
            // badly scaled vector: MINPACK's scalar recurrence
            double vn = v[n - 1];
            for (int j = n - 2; j >= 0; --j) {
                const double vj = v[j];
                double c = 2., sgl = 0.;
                if (vj != 0.) {
                    givens(vn, vj, c, sgl);
                    v[j] = givens_tau(vn, vj, c, sgl);
                    vn = sgl * vj + c * vn;
                }
                cs[j] = c; sn[j] = sgl;
            }
            v[n - 1] = vn;
        }
    }
    gsync<G>();
    SOCP_SUB(2);
    // apply to the columns: column i is touched by rotations j = min(i, n-2) .. 0
    if (G == 32 && n <= 96) {
        // one warp, three columns per lane (i = lane, lane + 32, lane + 64): the three dependent chains (one per
        // column, through its w) advance together row by row instead of one after the other; per column the
        // operations and their order are those of the loop below
        const int i0 = lane, i1 = lane + 32, i2 = lane + 64;
        const double slast = s[rowstart(n, n - 1)];
        double w0 = (i0 == n - 1) ? slast : 0., w1 = (i1 == n - 1) ? slast : 0., w2 = (i2 == n - 1) ? slast : 0.;
        int rs = rowstart(n, n - 2);                               // packed index of S(j, j)
        for (int j = n - 2; j >= 0; --j) {
            const double c = cs[j], sg = sn[j];
            if (!(c > 1.5)) {                                      // uniform: c == 2 marks "no rotation"
                const bool a0 = i0 >= j && i0 < n, a1 = i1 >= j && i1 < n, a2 = i2 >= j && i2 < n;
                const double x0 = a0 ? s[rs + i0 - j] : 0., x1 = a1 ? s[rs + i1 - j] : 0., x2 = a2 ? s[rs + i2 - j] : 0.;
                const double n0 = c * x0 - sg * w0, n1 = c * x1 - sg * w1, n2 = c * x2 - sg * w2;
                const double v0 = sg * x0 + c * w0, v1 = sg * x1 + c * w1, v2 = sg * x2 + c * w2;
                if (a0) { s[rs + i0 - j] = n0; w0 = v0; }
                if (a1) { s[rs + i1 - j] = n1; w1 = v1; }
                if (a2) { s[rs + i2 - j] = n2; w2 = v2; }
            }
            rs -= n - j + 1;                                       // rowstart(j - 1) = rowstart(j) - (n - (j - 1))
        }
        const double vl = v[n - 1];
        if (i0 < n) w[i0] = w0 + vl * u[i0];
        if (i1 < n) w[i1] = w1 + vl * u[i1];
        if (i2 < n) w[i2] = w2 + vl * u[i2];
    } else
    for (int i = tid; i < n; i += G) {
        double wi = (i == n - 1) ? s[rowstart(n, n - 1)] : 0.;
        const int jtop = (i < n - 1 ? i : n - 2);
        int l = rowstart(n, jtop) + (i - jtop);                // S(j, i) in the packed rows, one row up per step
        // "no rotation" (c == 2) is a predicated no-op rather than a branch, and the operands of four steps are
        // fetched before the dependent chain on wi runs through them
        auto step = [&](double c, double sg, double sl, int at) {
            const double ns = c * sl - sg * wi, nw = sg * sl + c * wi;
            if (!(c > 1.5)) { s[at] = ns; wi = nw; }
        };
        int j = jtop;
        for (; j >= 3; j -= 4) {
            const int l0 = l, l1 = l0 - (n - j), l2 = l1 - (n - j + 1), l3 = l2 - (n - j + 2);
            const double x0 = s[l0], x1 = s[l1], x2 = s[l2], x3 = s[l3];
            const double ca = cs[j], cb = cs[j - 1], cc = cs[j - 2], cd = cs[j - 3];
            const double sa = sn[j], sb = sn[j - 1], sc = sn[j - 2], sd = sn[j - 3];
            step(ca, sa, x0, l0); step(cb, sb, x1, l1); step(cc, sc, x2, l2); step(cd, sd, x3, l3);
            l = l3 - (n - j + 3);
        }
        for (; j >= 0; l -= n - j, --j) step(cs[j], sn[j], s[l], l);
        w[i] = wi + v[n - 1] * u[i];                 // add the spike from the rank-1 update
    }
    gsync<G>();
    SOCP_SUB(3);
    // Second sweep: eliminate the spike; rotation j depends on w[j] after rotations 0..j-1, strictly
    // sequential in j.  Warp 0: each lane owns the columns i = lane (mod 32) for the whole sweep (no
    // barrier inside the loop); the pivot w[j+1] is carried in a register and broadcast by one shuffle.
    if ((tid >> 5) == seqw) {
        if (n <= 96) {
            // w lives in registers (three slots per lane: i = lane, lane + 32, lane + 64); row j of s is read
            // and written once; everything is predicated (no divergent branch in the step) and the pivot
            // for the next step is picked from the right slot and broadcast by one shuffle
            double w0 = (lane < n) ? w[lane] : 0., w1 = (lane + 32 < n) ? w[lane + 32] : 0., w2 = (lane + 64 < n) ? w[lane + 64] : 0.;
            double wj = __shfl_sync(FULL, w0, 0);
            double sjj = s[0];
            int jj = 0;                                            // rowstart(n, j)
            // three phases of 32 steps: in phase p the slots below p are finished (no loads, no FMAs for them)
            // and the slots above p are active in every step
            sweep2_phase<0>(n, s, cs, sn, tmp, lane, min(32, n - 1), w0, w1, w2, wj, sjj, jj);
            sweep2_phase<1>(n, s, cs, sn, tmp, lane, min(64, n - 1), w0, w1, w2, wj, sjj, jj);
            sweep2_phase<2>(n, s, cs, sn, tmp, lane, n - 1, w0, w1, w2, wj, sjj, jj);
            // w[j] for j < n - 1 is replaced by tau below; only the last entry keeps its value
            if (lane == ((n - 1) & 31)) w[n - 1] = ((n - 1) >> 5) == 0 ? w0 : ((n - 1) >> 5) == 1 ? w1 : w2;
            for (int j = lane; j < n - 1; j += 32) if (tmp[j] == 2.) w[j] = 0.;
        } else {
        double wj = w[0];
        double sjj = s[0];
        for (int j = 0; j < n - 1; ++j) {
            const int jj = rowstart(n, j);
            const int nown = (j + 1) & 31;                         // owner of the next pivot
            double c1 = 0., c2 = 0.;
            if (lane == nown) { c1 = s[jj + 1]; c2 = w[j + 1]; }   // fetched before the rotation is known
            const double sjj_next = s[rowstart(n, j + 1)];         // row j+1 is untouched until step j+1
            double carry = c2;
            if (wj != 0.) {                                        // uniform: wj is the same in every lane
                double c, sgl;
                givens(sjj, wj, c, sgl);
                if (lane == (j & 31)) {
                    s[jj] = c * sjj + sgl * wj;
                    cs[j] = c; sn[j] = sgl; tmp[j] = (fabs(sjj) < fabs(wj)) ? 1. : 0.;     // tau is formed after the sweep
                }
                if (lane == nown) { s[jj + 1] = c * c1 + sgl * c2; carry = -sgl * c1 + c * c2; w[j + 1] = carry; }
                for (int i = j + 2 + ((lane - j - 2) & 31); i < n; i += 32) {
                    const int l = jj + (i - j);
                    const double sl = s[l], wi = w[i];
                    s[l] = c * sl + sgl * wi;
                    w[i] = -sgl * sl + c * wi;
                }
            }
            else if (lane == (j & 31)) tmp[j] = 2.;                 // no rotation: w[j] stays zero
            wj = __shfl_sync(FULL, carry, nown);
            sjj = sjj_next;
        }
        }
        // MINPACK's tau for r1mpyq (one divide each, off the sequential chain); entries written by this lane
        for (int j = lane; j < n - 1; j += 32) {
            if (tmp[j] == 1.) w[j] = (fabs(cs[j]) * DBL_MAX > 1.) ? 1. / cs[j] : 1.;
            else if (tmp[j] == 0.) w[j] = sn[j];
        }
        if (lane == ((n - 1) & 31)) s[rowstart(n, n - 1)] = w[n - 1];
    }
    gsync<G>();
    SOCP_SUB(4);
}

// Rotation coefficients as r1mpyq reconstructs them from the stored tau values: scr = [c1 s1 c2 s2][n]
template <int G>
__device__ void r1coef_g(int n, const double *v, const double *w, double *scr) {
    const int tid = threadIdx.x % G;
    gsync<G>();
    for (int j = tid; j < n - 1; j += G) {
        double c, s;
        if (fabs(v[j]) > 1.) { c = 1. / v[j]; s = sqrt(1. - c * c); }
        else { s = v[j]; c = sqrt(1. - s * s); }
        scr[j] = c; scr[n + j] = s;
        if (fabs(w[j]) > 1.) { c = 1. / w[j]; s = sqrt(1. - c * c); }
        else { s = w[j]; c = sqrt(1. - s * s); }
        scr[2 * n + j] = c; scr[3 * n + j] = s;
    }
    gsync<G>();
}

// One step of r1mpyq on the pair (a_j, a_n).  Explicit roundings (no contraction left to the compiler): the
// fused Broyden kernel and the split Q pass must produce the same bits from the same rotations.
SOCP_DEV void rot_first(double c, double s, double aj, double &an, double &out) {      // first set, j = n-2 .. 0
    out = __fma_rn(c, aj, -__dmul_rn(s, an));
    an = __fma_rn(s, aj, __dmul_rn(c, an));
}
SOCP_DEV void rot_second(double c, double s, double aj, double &an, double &out) {     // second set, j = 0 .. n-2
    out = __fma_rn(c, aj, __dmul_rn(s, an));
    an = __fma_rn(-s, aj, __dmul_rn(c, an));
}

// r1mpyq: apply the recorded rotations to A (m x n, column-major, lda): one thread per row, the
// row streamed through registers in chunks of 8 columns so that the loads overlap the chain.
// `extra` (length n, stride 1) is transformed as one more row (r1mpyq(1, n, qtf, 1, ...) of hybrd).
template <int G>
__device__ void r1mpyq_g(int m, int n, double *a, int lda_a, const double *scr, double *extra) {
    const int tid = threadIdx.x % G;
    const double *c1 = scr, *s1 = scr + n, *c2 = scr + 2 * n, *s2 = scr + 3 * n;
    constexpr int CH = 8;
    gsync<G>();
    for (int i = tid; i < m + 1; i += G) {
        double *row = (i < m) ? a + i : extra;
        const int lda = (i < m) ? lda_a : 1;
        double an = row[(size_t)(n - 1) * lda];
        double buf[CH];
        for (int j0 = n - 2; j0 >= 0; j0 -= CH) {             // first set: j = n-2 .. 0
#pragma unroll
            for (int k = 0; k < CH; ++k) if (j0 - k >= 0) buf[k] = row[(size_t)(j0 - k) * lda];
#pragma unroll
            for (int k = 0; k < CH; ++k) if (j0 - k >= 0) rot_first(c1[j0 - k], s1[j0 - k], buf[k], an, buf[k]);
#pragma unroll
            for (int k = 0; k < CH; ++k) if (j0 - k >= 0) row[(size_t)(j0 - k) * lda] = buf[k];
        }
        for (int j0 = 0; j0 < n - 1; j0 += CH) {               // second set: j = 0 .. n-2
#pragma unroll
            for (int k = 0; k < CH; ++k) if (j0 + k < n - 1) buf[k] = row[(size_t)(j0 + k) * lda];
#pragma unroll
            for (int k = 0; k < CH; ++k) if (j0 + k < n - 1) rot_second(c2[j0 + k], s2[j0 + k], buf[k], an, buf[k]);
#pragma unroll
            for (int k = 0; k < CH; ++k) if (j0 + k < n - 1) row[(size_t)(j0 + k) * lda] = buf[k];
        }
        row[(size_t)(n - 1) * lda] = an;
    }
    gsync<G>();
}

// ---- bulk copies (TMA engine, non-tensor form) and their mbarrier -----------------------------------------
SOCP_DEV unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
SOCP_DEV void mbar_init(unsigned long long *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
SOCP_DEV void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
SOCP_DEV bool mbar_try_wait(unsigned long long *bar, unsigned parity) {
    unsigned ok;
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// global -> shared, completion counted in bytes on the mbarrier; 16-byte aligned addresses, size % 16 == 0
SOCP_DEV void bulk_g2s(void *smem_dst, const void *gmem_src, unsigned bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// shared -> global as one bulk group; bulk_wait_read() returns when the shared source may be overwritten
SOCP_DEV void bulk_s2g(void *gmem_dst, const void *smem_src, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
SOCP_DEV void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
SOCP_DEV void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// order this thread's generic-proxy accesses to shared memory before later async-proxy (bulk copy) accesses
SOCP_DEV void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- kernel 2b-1 (split build): one streaming pass over Q per Broyden iteration ---------------------------
// For every problem whose trial residual arrived: bring Q (P x P, column major) into shared memory with ONE
// bulk copy, apply the 2(P-1) Givens rotations the previous Broyden update recorded but did not apply
// (MINPACK r1mpyq, deferred by one iteration: I_PEND), write Q back with one bulk copy, and form
// sum = Q^T F(x + p) from the copy in shared memory.  Q is read once and written once per iteration
// (the fused kernel read it twice: once for Q^T f, once for r1mpyq) and nothing here is a cross-thread
// dependent chain: one thread per row for the rotations, one warp per column for the dot products.
// The chain kernel (hybrd_res_kernel, SPLIT) consumes `sum` (D.wa2) and records the next rotations (D.scr).
__global__ void __launch_bounds__(128)
hybrd_qpass_kernel(SolverDev D, int cur) {
    extern __shared__ __align__(128) double qp_smem[];
    const int n = D.P, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NT = 128, NW = 4;
    double *Qs = qp_smem;                               // [QS]
    double *wv = Qs + D.QS;                             // [n]  F(x + p)
    double *cf = wv + ((n + 1) & ~1);                   // [4n] c1 s1 c2 s2 (r1coef layout)
    unsigned long long *bar = (unsigned long long *)(cf + 4 * n);
    const int nres = D.counts[cur * 2 + 0];
    const int *res_list = D.lists + (size_t)(cur * 2 + 0) * D.B;
    const unsigned qbytes = (unsigned)D.QS * 8u;
    if (tid == 0) mbar_init(bar, 1);
    __syncthreads();
    unsigned parity = 0;
    // the index chain of a problem (list entry -> phase, pending flag) is two dependent global loads in front of the
    // bulk copy: the next problem's is fetched while the current one is being worked on
    long b_next = -1;
    int phase_next = PH_IDLE, pend_next = 0;
    if ((long)blockIdx.x < nres) {
        b_next = res_list[blockIdx.x];
        phase_next = D.istate[b_next * I_COUNT + I_PHASE];
        pend_next = D.istate[b_next * I_COUNT + I_PEND];
    }
    for (long g = blockIdx.x; g < nres; g += gridDim.x) {
        const long b = b_next;
        const int phase = phase_next, pend = pend_next;
        int *is = D.istate + b * I_COUNT;
        if (g + gridDim.x < nres) {
            b_next = res_list[g + gridDim.x];
            phase_next = D.istate[b_next * I_COUNT + I_PHASE];
            pend_next = D.istate[b_next * I_COUNT + I_PEND];
        }
        if (phase != PH_TRIAL) continue;                // first residual of a solve: nothing to do (uniform)
        double *Qg = D.fjac + (size_t)b * D.QS;
        if (tid == 0) {
            mbar_expect_tx(bar, qbytes);
            bulk_g2s(Qs, Qg, qbytes, bar);
        }
        // F(x + p) and the coefficient vectors with cp.async: every element in flight at once, next to the bulk copy
        gcopy_async<NT>(wv, D.wa4 + b * n, n);
        if (pend) gcopy_async<NT>(cf, D.scr + b * 4 * (size_t)n, 4 * n);
        gcopy_async_wait();
        __syncthreads();
        while (!mbar_try_wait(bar, parity)) {}
        parity ^= 1u;
        if (pend) {
            const double *c1 = cf, *s1 = cf + n, *c2 = cf + 2 * n, *s2 = cf + 3 * n;
            for (int i = tid; i < n; i += NT) {         // one thread per row; consecutive threads, consecutive words
                double *row = Qs + i;
                double an = row[(size_t)(n - 1) * n];
                for (int j = n - 2; j >= 0; --j) { double o; rot_first(c1[j], s1[j], row[(size_t)j * n], an, o); row[(size_t)j * n] = o; }
                for (int j = 0; j < n - 1; ++j) { double o; rot_second(c2[j], s2[j], row[(size_t)j * n], an, o); row[(size_t)j * n] = o; }
                row[(size_t)(n - 1) * n] = an;
            }
            fence_async_smem();
            __syncthreads();
            if (tid == 0) bulk_s2g(Qg, Qs, qbytes);
        }
        // sum_j = Q(:, j) . F(x + p): one warp per column, four columns in flight; per lane the rows
        // lane, lane + 32, lane + 64 of a 96-row block accumulate in that order, then the xor butterfly
        // 16, 8, 4, 2, 1 (the summation tree of the fused kernel: the two builds agree bit for bit)
        for (int j0 = 4 * warp; j0 < n; j0 += 4 * NW) {
            double p0 = 0., p1 = 0., p2 = 0., p3 = 0.;
            for (int i0 = 0; i0 < n; i0 += 96) {
#pragma unroll
                for (int u = 0; u < 3; ++u) {
                    const int i = i0 + 32 * u + lane;
                    const double wi = (i < n) ? wv[i] : 0.;
                    const double q0 = (i < n) ? Qs[(size_t)j0 * n + i] : 0.;
                    const double q1 = (i < n && j0 + 1 < n) ? Qs[(size_t)(j0 + 1) * n + i] : 0.;
                    const double q2 = (i < n && j0 + 2 < n) ? Qs[(size_t)(j0 + 2) * n + i] : 0.;
                    const double q3 = (i < n && j0 + 3 < n) ? Qs[(size_t)(j0 + 3) * n + i] : 0.;
                    p0 = fma(q0, wi, p0); p1 = fma(q1, wi, p1); p2 = fma(q2, wi, p2); p3 = fma(q3, wi, p3);
                }
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                p0 += __shfl_xor_sync(0xffffffffu, p0, off); p1 += __shfl_xor_sync(0xffffffffu, p1, off);
                p2 += __shfl_xor_sync(0xffffffffu, p2, off); p3 += __shfl_xor_sync(0xffffffffu, p3, off);
            }
            if (lane < 4 && j0 + lane < n) D.wa2[b * n + j0 + lane] = (lane == 0) ? p0 : (lane == 1) ? p1 : (lane == 2) ? p2 : p3;
        }
        if (tid == 0) {
            atomicAdd(D.counters + 5, 1ULL);                    // problems through the Q pass
            if (pend) { is[I_PEND] = 0; bulk_wait_read(); }     // the copy out has read the shared buffer
        }
        fence_async_smem();
        __syncthreads();                                        // buffer free for the next problem's bulk load
    }
    if (tid == 0) bulk_wait_all();
}

// ---- shared state of one problem inside the Powell-hybrid kernels ------------------------------
struct Work {
    double *x, *xe, *fvec, *diag, *qtf, *wa1, *wa2, *wa3, *wa4, *scr, *r, *q;
    int ldq;
};

// dogleg step from the current factors, trial point xe = x + p, and the request for F(xe)
template <int G>
__device__ void dogleg_and_request(const SolverDev &D, long b, const Work &W, int *is, double *ds, double *red,
                                   int *next_res, int *next_cnt) {
    const int n = D.P, tid = threadIdx.x % G;
    const double delta = ds[D_DELTA];
    dogleg_g<G>(n, W.r, W.diag, W.qtf, delta, W.wa1, W.wa2, W.wa3, red, seq_warp<G>(D.sm_count), D.phase_clocks, D.counters);
    for (int j = tid; j < n; j += G) {
        const double pj = -W.wa1[j];
        W.wa1[j] = pj;
        W.xe[j] = W.x[j] + pj;            // trial point (MINPACK's wa2)
        W.wa3[j] = W.diag[j] * pj;
    }
    gsync<G>();
    const double pnorm = enorm_g<G>(n, W.wa3, red);
    gsync<G>();
    if (tid == 0) {
        ds[D_PNORM] = pnorm;
        if (is[I_ITER] == 1) ds[D_DELTA] = fmin(delta, pnorm);
        is[I_PHASE] = PH_TRIAL;
        next_res[atomicAdd(&next_cnt[0], 1)] = (int)b;
    }
}

// shared-memory carve for one group: [13 P vectors][R][Q]
template <int G>
SOCP_DEV double *group_smem(const SolverDev &D, int per_group_doubles) {
    extern __shared__ __align__(128) double smem_all[];
    const int grp = (G == 32) ? (threadIdx.x >> 5) : 0;
    return smem_all + (size_t)grp * per_group_doubles;
}

// ---- kernel 2b: problems whose residual arrived (first evaluation or trial point) ---------------
// SPLIT = false: the fused kernel (one group does everything of a Broyden iteration, Q swept twice from
// global memory).  SPLIT = true: the chain kernel of the split build -- Q never appears here: sum = Q^T F(x + p)
// was left in D.wa2 by hybrd_qpass_kernel, the 2(P-1) rotations of this update go to D.scr for the next Q pass
// (I_PEND) and only qtf is rotated on the spot.
template <int G, bool STAGE_R, bool SPLIT>
SOCP_DEV void res_loop(const SolverDev &D, int cur, int per_group_doubles) {
    static_assert(!SPLIT || (G == 32 && STAGE_R), "the chain kernel runs one warp per problem with R staged");
    const int GROUPS = (G == 32) ? (int)(blockDim.x >> 5) : 1;
    const int grp = (G == 32) ? (threadIdx.x >> 5) : 0;
    const int tid = threadIdx.x % G;
    const int n = D.P;
    double *sm = group_smem<G>(D, per_group_doubles);
    double *red = sm;                                    // 8 doubles
    double *vec = sm + 8;
    const int nres = D.counts[cur * 2 + 0];
    const int *res_list = D.lists + (size_t)(cur * 2 + 0) * D.B;
    int *next_res = D.lists + (size_t)((1 - cur) * 2 + 0) * D.B;
    int *next_jac = D.lists + (size_t)((1 - cur) * 2 + 1) * D.B;
    int *next_cnt = D.counts + (1 - cur) * 2;
    const double p1 = .1, p5 = .5, p001 = .001, p0001 = 1e-4;
    bool lean_bar_ready = false;
    unsigned lean_parity = 0;

    for (long g = (long)blockIdx.x * GROUPS + grp; g < nres; g += (long)gridDim.x * GROUPS) {
        const long b = res_list[g];
        int *is = D.istate + b * I_COUNT;
        double *ds = D.dstate + b * D_COUNT;
        gsync<G>();
        const int phase = is[I_PHASE];
        if (phase == PH_F0) {
            // first residual: fvec = F(x) was written by assemble_kernel
            const double fnorm = enorm_g<G>(n, D.fvec + b * n, red);
            gsync<G>();
            if (tid == 0) {
                is[I_BASE] = 1 - is[I_BASE];
                is[I_NFEV] = 1;
                ds[D_FNORM] = fnorm;
                is[I_ITER] = 1; is[I_NCSUC] = 0; is[I_NCFAIL] = 0; is[I_NSLOW1] = 0; is[I_NSLOW2] = 0;
                if (D.run_mode == RUN_RESIDUAL) is[I_PHASE] = PH_IDLE;
                else {
                    is[I_PHASE] = PH_JAC;
                    next_jac[atomicAdd(&next_cnt[1], 1)] = (int)b;
                }
            }
            continue;
        }
        // ---- trial point evaluated: wa4 = F(x + p) ----
        long long phase_t0 = clock64();
        Work W;
        // LEAN (the chain kernel): only what the dependent chains touch lives in shared memory --
        // R and nine vectors; x, xe, fvec and F(x + p) are read and written element-wise and stay in global
        // memory.  35 KB per problem instead of 38: six problems per SM instead of five.  R travels by bulk copy.
        constexpr bool LEAN = SPLIT;
        if (LEAN) {
            W.x = D.x + b * n; W.xe = D.xe + b * n; W.fvec = D.fvec + b * n; W.wa4 = D.wa4 + b * n;
            W.diag = vec; W.qtf = vec + n; W.wa1 = vec + 2 * n; W.wa2 = vec + 3 * n; W.wa3 = vec + 4 * n; W.scr = vec + 5 * n;
            W.r = sm + ((8 + 9 * n + 1) & ~1);                 // 16-byte aligned
        } else {
            W.x = vec; W.xe = vec + n; W.fvec = vec + 2 * n; W.diag = vec + 3 * n; W.qtf = vec + 4 * n;
            W.wa1 = vec + 5 * n; W.wa4 = vec + 6 * n; W.wa2 = vec + 7 * n; W.wa3 = vec + 8 * n; W.scr = vec + 9 * n;
            W.r = STAGE_R ? vec + 13 * n : D.r + (size_t)b * D.LRS;
        }
        W.q = D.fjac + (size_t)b * D.QS;
        W.ldq = n;
        if (!SPLIT) l2_prefetch<G>(W.q, (size_t)n * n * sizeof(double));      // Q is first touched ~20 us from now
        if (LEAN) {
            unsigned long long *bar = (unsigned long long *)(sm + 7);
            if (tid == 0) {
                if (!lean_bar_ready) mbar_init(bar, 1);
                bulk_wait_read();                              // the previous visit's copy out has read the buffer
                mbar_expect_tx(bar, (unsigned)D.LRS * 8u);
                bulk_g2s(W.r, D.r + (size_t)b * D.LRS, (unsigned)D.LRS * 8u, bar);
            }
            lean_bar_ready = true;
            gcopy_async<G>(W.diag, D.diag + b * n, n); gcopy_async<G>(W.qtf, D.qtf + b * n, n); gcopy_async<G>(W.wa1, D.wa1 + b * n, n);
            gcopy_async_wait();
            __syncwarp();
            while (!mbar_try_wait(bar, lean_parity)) {}
            lean_parity ^= 1u;
        } else {
            gcopy_async<G>(W.x, D.x + b * n, n); gcopy_async<G>(W.xe, D.xe + b * n, n); gcopy_async<G>(W.fvec, D.fvec + b * n, n);
            gcopy_async<G>(W.diag, D.diag + b * n, n); gcopy_async<G>(W.qtf, D.qtf + b * n, n); gcopy_async<G>(W.wa1, D.wa1 + b * n, n);
            gcopy_async<G>(W.wa4, D.wa4 + b * n, n);
            if (STAGE_R) gcopy_async<G>(W.r, D.r + (size_t)b * D.LRS, D.LR);
            gcopy_async_wait();
        }
        gsync<G>();
        SOCP_PHASE(16, 0);

        const double fnorm1 = enorm_g<G>(n, W.wa4, red);
        double fnorm = ds[D_FNORM], delta = ds[D_DELTA], xnorm = ds[D_XNORM];
        const double pnorm = ds[D_PNORM];
        int iter = is[I_ITER], ncsuc = is[I_NCSUC], ncfail = is[I_NCFAIL], nslow1 = is[I_NSLOW1], nslow2 = is[I_NSLOW2];
        const int jeval = is[I_JEVAL];
        const int nfev = is[I_NFEV] + 1;
        const int trial = 1 - is[I_BASE];
        double actred = -1.;
        if (fnorm1 < fnorm) { const double q = fnorm1 / fnorm; actred = 1. - q * q; }
        // predicted reduction: wa3 = qtf + R * wa1
        rmulv_g<G>(n, W.r, W.wa1, W.qtf, W.wa3);
        const double temp = enorm_g<G>(n, W.wa3, red);
        double prered = 0.;
        if (temp < fnorm) { const double q = temp / fnorm; prered = 1. - q * q; }
        double ratio = 0.;
        if (prered > 0.) ratio = actred / prered;
        if (ratio < p1) {
            ncsuc = 0; ++ncfail; delta = p5 * delta;
        } else {
            ncfail = 0; ++ncsuc;
            if (ratio >= p5 || ncsuc > 1) delta = fmax(delta, pnorm / p5);
            if (fabs(ratio - 1.) <= p1) delta = pnorm / p5;
        }
        int base = is[I_BASE];
        gsync<G>();
        SOCP_PHASE(16, 1);
        if (ratio >= p0001) {
            // successful iteration: x <- x + p, fvec <- wa4
            for (int j = tid; j < n; j += G) {
                const double xj = W.xe[j];
                W.x[j] = xj;
                W.wa2[j] = W.diag[j] * xj;
                W.fvec[j] = W.wa4[j];
            }
            gsync<G>();
            xnorm = enorm_g<G>(n, W.wa2, red);
            fnorm = fnorm1;
            ++iter;
            base = trial;
        }
        ++nslow1;
        if (actred >= p001) nslow1 = 0;
        if (jeval) ++nslow2;
        if (actred >= p1) nslow2 = 0;
        int info = 0;
        if (delta <= D.xtol * xnorm || fnorm == 0.) info = 1;
        if (info == 0) {
            if (nfev >= D.maxfev) info = 2;
            if (p1 * fmax(p1 * delta, pnorm) <= EPSMCH * xnorm) info = 3;
            if (nslow2 == 5) info = 4;
            if (nslow1 == 10) info = 5;
        }
        gsync<G>();
        if (tid == 0) {
            is[I_ITER] = iter; is[I_NCSUC] = ncsuc; is[I_NCFAIL] = ncfail; is[I_NSLOW1] = nslow1; is[I_NSLOW2] = nslow2;
            is[I_NFEV] = nfev; is[I_BASE] = base;
            ds[D_FNORM] = fnorm; ds[D_DELTA] = delta; ds[D_XNORM] = xnorm;
        }
        bool store_r = false;
        if (info != 0) {
            if (tid == 0) { is[I_INFO] = info; is[I_PHASE] = PH_IDLE; }      // retire (convergence mask)
        } else if (ncfail == 2) {
            // re-evaluate the Jacobian at x
            for (int j = tid; j < n; j += G) W.xe[j] = W.x[j];
            if (tid == 0) {
                is[I_PHASE] = PH_JAC;
                next_jac[atomicAdd(&next_cnt[1], 1)] = (int)b;
            }
        } else {
            // rank-one (Broyden) update of the QR factors: sum_j = Q(:,j) . wa4, one warp per
            // column, four columns in flight so that the HBM/L2 loads of Q overlap
            SOCP_PHASE(16, 2);
            if (!SPLIT) {
                const int lane = threadIdx.x & 31, warp = tid >> 5;
                constexpr int NW = G / 32, NC = 8;
                const bool clk_on = D.phase_clocks; unsigned long long *clk_counters = D.counters; long long sub_t0 = clock64();
                for (int j0 = warp * NC; j0 < n; j0 += NW * NC) {
                    double part[NC];
#pragma unroll
                    for (int k = 0; k < NC; ++k) part[k] = 0.;
                    for (int i0 = 0; i0 < n; i0 += 96) {          // 3 x 8 loads in flight per lane
                        double q[3][NC];
#pragma unroll
                        for (int u = 0; u < 3; ++u) {
                            const int i = i0 + 32 * u + lane;
#pragma unroll
                            for (int k = 0; k < NC; ++k)
                                q[u][k] = (i < n && j0 + k < n) ? W.q[(size_t)(j0 + k) * W.ldq + i] : 0.;
                        }
#pragma unroll
                        for (int u = 0; u < 3; ++u) {
                            const int i = i0 + 32 * u + lane;
                            const double wi = (i < n) ? W.wa4[i] : 0.;
#pragma unroll
                            for (int k = 0; k < NC; ++k) part[k] = fma(q[u][k], wi, part[k]);
                        }
                    }
                    SOCP_SUB(0);
                    // transposing butterfly: 9 shuffles leave the sum of column j0 + (lane >> 2) in every lane
                    // (8 separate reductions take 40), then eight lanes finish their columns in parallel
                    double q4[4], q2[2];
                    {
                        const bool up = lane & 16;
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const double recv = __shfl_xor_sync(0xffffffffu, up ? part[k] : part[k + 4], 16);
                            q4[k] = (up ? part[k + 4] : part[k]) + recv;
                        }
                    }
                    {
                        const bool up = lane & 8;
#pragma unroll
                        for (int k = 0; k < 2; ++k) {
                            const double recv = __shfl_xor_sync(0xffffffffu, up ? q4[k] : q4[k + 2], 8);
                            q2[k] = (up ? q4[k + 2] : q4[k]) + recv;
                        }
                    }
                    double sum;
                    {
                        const bool up = lane & 4;
                        const double recv = __shfl_xor_sync(0xffffffffu, up ? q2[0] : q2[1], 4);
                        sum = (up ? q2[1] : q2[0]) + recv;
                    }
                    sum += __shfl_xor_sync(0xffffffffu, sum, 2);
                    sum += __shfl_xor_sync(0xffffffffu, sum, 1);
                    {
                        const int j = j0 + (lane >> 2);
                        if (j < n && (lane & 3) == 0) {
                            W.wa2[j] = (sum - W.wa3[j]) / pnorm;
                            W.wa1[j] = W.diag[j] * ((W.diag[j] * W.wa1[j]) / pnorm);
                            if (ratio >= p0001) W.qtf[j] = sum;
                        }
                    }
                    SOCP_SUB(1);
                }
            } else {
                // split build: sum = Q^T F(x + p) comes from the Q pass (same summation tree, same bits)
                const double *sumv = D.wa2 + b * n;
                for (int j = tid; j < n; j += G) {
                    const double sum = sumv[j];
                    W.wa2[j] = (sum - W.wa3[j]) / pnorm;
                    W.wa1[j] = W.diag[j] * ((W.diag[j] * W.wa1[j]) / pnorm);
                    if (ratio >= p0001) W.qtf[j] = sum;
                }
            }
            if (tid == 0) atomicAdd(D.counters + 1, 1ULL);
            gsync<G>();
            SOCP_PHASE(16, 3);
            r1updt_g<G>(n, W.r, W.wa1, W.wa2, W.wa3, W.scr, W.scr + n, W.scr + 2 * n, seq_warp<G>(D.sm_count), D.phase_clocks, D.counters);
            SOCP_PHASE(16, 4);
            r1coef_g<G>(n, W.wa2, W.wa3, W.scr);
            if (SPLIT) {
                // qtf is needed by the dogleg right away: rotate it here (one row); Q waits for the next Q pass
                r1mpyq_g<G>(0, n, W.q, W.ldq, W.scr, W.qtf);
                gcopy<G>(D.scr + (size_t)b * 4 * n, W.scr, 4 * n);
                if (tid == 0) is[I_PEND] = 1;
            } else r1mpyq_g<G>(n, n, W.q, W.ldq, W.scr, W.qtf);
            SOCP_PHASE(16, 5);
            if (tid == 0) is[I_JEVAL] = 0;
            dogleg_and_request<G>(D, b, W, is, ds, red, next_res, next_cnt);
            store_r = true;
            SOCP_PHASE(16, 6);
        }
        gsync<G>();
        if (LEAN) {
            gcopy<G>(D.qtf + b * n, W.qtf, n); gcopy<G>(D.wa1 + b * n, W.wa1, n);
            if (store_r) {
                fence_async_smem();
                __syncwarp();
                if (tid == 0) bulk_s2g(D.r + (size_t)b * D.LRS, W.r, (unsigned)D.LRS * 8u);
            }
        } else {
            gcopy<G>(D.x + b * n, W.x, n); gcopy<G>(D.xe + b * n, W.xe, n); gcopy<G>(D.fvec + b * n, W.fvec, n);
            gcopy<G>(D.qtf + b * n, W.qtf, n); gcopy<G>(D.wa1 + b * n, W.wa1, n);
            if (STAGE_R && store_r) gcopy<G>(D.r + (size_t)b * D.LRS, W.r, D.LR);
        }
        gsync<G>();
        SOCP_PHASE(16, 7);
    }
    if (SPLIT && tid == 0) bulk_wait_all();
}

// 4 CTAs/SM: after the instruction-level pass the kernel fits 128 registers without spills and the fourth
// co-resident problem is worth -12 % kernel time (before it, the 128-register build spilled and 3 CTAs/SM
// at 167 registers measured the same; 5 CTAs/SM were worse -- DESIGN.md section 5)
template <int G, bool STAGE_R>
__global__ void __launch_bounds__(128, 4)
hybrd_res_kernel(SolverDev D, int cur, int per_group_doubles) {
    res_loop<G, STAGE_R, false>(D, cur, per_group_doubles);
}

// The chain kernel of the split build: ONE WARP per problem (no CTA barrier anywhere: every wait is a
// __syncwarp), as many problems per SM as shared memory holds (R + 13 work vectors per problem).  What is left
// of a Broyden iteration once Q is gone are the dependent chains (Givens sweeps, back substitution, norms);
// their latency is hidden by the other warps of the SM instead of by idle threads of the same CTA.
__global__ void __launch_bounds__(32, 5)
hybrd_chain_kernel(SolverDev D, int cur, int per_group_doubles) {
    res_loop<32, true, true>(D, cur, per_group_doubles);
}

// ---- kernel 2c: problems whose forward-difference Jacobian arrived ------------------------------
// BAND: the matrix is staged as its structural band (SolverDev::band_lo / band_off) after the 13 P work vectors, then
// the two tables; R stays in global memory and qform_p writes Q there.
template <int G, bool STAGE_R, bool STAGE_Q, bool BAND>
SOCP_DEV void jac_loop(const SolverDev &D, int cur, int per_group_doubles) {
    static_assert(!BAND || (STAGE_Q && !STAGE_R), "the banded Jacobian phase stages the matrix and leaves R in global memory");
    const int GROUPS = (G == 32) ? (int)(blockDim.x >> 5) : 1;
    const int grp = (G == 32) ? (threadIdx.x >> 5) : 0;
    const int tid = threadIdx.x % G;
    const int n = D.P;
    double *sm = group_smem<G>(D, per_group_doubles);
    double *red = sm;
    double *vec = sm + 8;
    const int njac = D.counts[cur * 2 + 1];
    const int *jac_list = D.lists + (size_t)(cur * 2 + 1) * D.B;
    int *next_res = D.lists + (size_t)((1 - cur) * 2 + 0) * D.B;
    int *next_cnt = D.counts + (1 - cur) * 2;
    const int ldq_s = n | 1;                               // odd leading dimension in shared memory
    // 128-thread CTA, Q staged: Q travels by bulk copy when its shared layout equals the global one (odd P)
    const bool bulk = (G == 128) && STAGE_Q && !BAND && ldq_s == n;
    int *band_lo = (int *)(vec + 13 * n + D.band_doubles), *band_off = band_lo + n;
    if (BAND) {
        for (int k = tid; k <= n; k += G) {
            if (k < n) band_lo[k] = D.band_lo[k];
            band_off[k] = D.band_off[k];
        }
    }
    const BandCols band{vec + 13 * n, band_lo, band_off};
    __shared__ unsigned long long jac_bar;
    unsigned jac_parity = 0;
    if (bulk) {
        if (threadIdx.x == 0) mbar_init(&jac_bar, 1);
        __syncthreads();
    }

    for (long g = (long)blockIdx.x * GROUPS + grp; g < njac; g += (long)gridDim.x * GROUPS) {
        const long b = jac_list[g];
        int *is = D.istate + b * I_COUNT;
        double *ds = D.dstate + b * D_COUNT;
        gsync<G>();
        if (D.run_mode == RUN_FDJAC) {                     // the Jacobian itself was the request
            if (tid == 0) is[I_PHASE] = PH_IDLE;
            continue;
        }
        Work W;
        W.x = vec; W.xe = vec + n; W.fvec = vec + 2 * n; W.diag = vec + 3 * n; W.qtf = vec + 4 * n;
        W.wa1 = vec + 5 * n; W.wa4 = vec + 6 * n; W.wa2 = vec + 7 * n; W.wa3 = vec + 8 * n; W.scr = vec + 9 * n;
        double *after = vec + 13 * n;
        W.r = STAGE_R ? after : D.r + (size_t)b * D.LRS;
        if (STAGE_R) after += D.LR;
        double *gq = D.fjac + (size_t)b * D.QS;
        if (STAGE_Q) after = sm + (((after - sm) + 1) & ~(ptrdiff_t)1);      // Q starts 16-byte aligned (bulk copies)
        W.q = STAGE_Q ? after : gq;
        W.ldq = STAGE_Q ? ldq_s : n;
        long long phase_t0 = clock64();
        gcopy_async<G>(W.x, D.x + b * n, n); gcopy_async<G>(W.fvec, D.fvec + b * n, n); gcopy_async<G>(W.diag, D.diag + b * n, n);
        if (bulk) {
            if (tid == 0) {
                bulk_wait_read();                          // the previous problem's copy out has read the buffer
                mbar_expect_tx(&jac_bar, (unsigned)D.QS * 8u);
                bulk_g2s(W.q, gq, (unsigned)D.QS * 8u, &jac_bar);
            }
        } else if (BAND)
            for (int c = tid >> 5; c < n; c += G / 32) {
                const int lo = band_lo[c], len = band_off[c + 1] - band_off[c];
                for (int i = tid & 31; i < len; i += 32) __pipeline_memcpy_async(band.a + band_off[c] + i, gq + lo + i + (size_t)c * n, sizeof(double));
            }
        else if (STAGE_Q)
            for (int c = tid >> 5; c < n; c += G / 32)
                for (int i = tid & 31; i < n; i += 32) __pipeline_memcpy_async(W.q + i + (size_t)c * ldq_s, gq + i + (size_t)c * n, sizeof(double));
        gcopy_async_wait();
        if (bulk) {
            while (!mbar_try_wait(&jac_bar, jac_parity)) {}
            jac_parity ^= 1u;
        }
        gsync<G>();
        SOCP_PHASE(32, 0);
        if (tid == 0) {
            if (D.analytic) is[I_NJEV] += 1;               // hybrj counts Jacobian calls apart (njev)
            else is[I_NFEV] += n;                          // hybrd: fdjac1 costs n residual evaluations
            is[I_JEVAL] = 1;
            is[I_PEND] = 0;                                // Q is rebuilt from scratch: nothing pending
            atomicAdd(D.counters + 2, 1ULL);
        }
        for (int i = tid; i < n; i += G) W.qtf[i] = W.fvec[i];
        // wa1 = rdiag, wa2 = acnorm
        int *hi = (int *)W.scr;                            // [n + 1] last non-zero row per column (scr is free here)
        // Register-window accumulation of Q when the Jacobian at hand has the block-bidiagonal + border structure
        // (every sub-column fits the two-block window; fill-in stays inside it): decided per matrix, from its own zeros.
        // (the banded layout holds only for shapes whose every reflector fits the window, jac_band)
        bool win = BAND;
        // (instantiated for the layout the 32 < P <= ~150 problems run with -- Q staged, R in global memory -- and the
        // block size of the benchmark model, 14; every other shape takes the barrier-per-reflector qform_g)
        if ((G == 128) && STAGE_Q && !STAGE_R && !BAND && D.N == 14 && n < G) {
            for (int k = tid; k < n; k += G) {
                const double *ck = W.q + (size_t)k * W.ldq;
                int last = 0;
                for (int i = n - 1; i > 0; --i) if (ck[i] != 0.) { last = i; break; }
                hi[k] = last;
            }
            win = window_ok<G>(n, D.N, hi, (int *)red);
        }
        const DenseCols dense{W.q, W.ldq, n};
        if constexpr (BAND) qrfac_g<G>(n, band, W.wa1, W.wa2, W.qtf, red, seq_warp<G>(D.sm_count), hi);
        else qrfac_g<G>(n, dense, W.wa1, W.wa2, W.qtf, red, seq_warp<G>(D.sm_count), hi);
        SOCP_PHASE(32, 1);
        if (is[I_ITER] == 1) {
            for (int j = tid; j < n; j += G) {
                double dj = W.wa2[j];
                if (dj == 0.) dj = 1.;
                W.diag[j] = dj;
                W.wa3[j] = dj * W.x[j];
            }
            gsync<G>();
            const double xnorm = enorm_g<G>(n, W.wa3, red);
            double delta = D.factor * xnorm;
            if (delta == 0.) delta = D.factor;
            gsync<G>();
            if (tid == 0) { ds[D_XNORM] = xnorm; ds[D_DELTA] = delta; }
        }
        if constexpr (BAND) pack_r_g<G>(n, band, W.wa1, W.r);
        else pack_r_g<G>(n, dense, W.wa1, W.r);
        SOCP_PHASE(32, 2);
        // register-window accumulation of Q when every reflector fits the two-block window (checked on this matrix):
        // no barrier, Q goes straight to global memory
        bool q_in_global = false;
        if constexpr (BAND) {
            qform_p<G, 14>(n, band, hi, gq);
            gsync<G>();
            q_in_global = true;
        } else if ((G == 128) && STAGE_Q && !STAGE_R && win) {
            qform_p<G, 14>(n, dense, hi, gq);
            gsync<G>();
            q_in_global = true;
        } else qform_g<G>(n, W.q, W.ldq, W.wa1, seq_warp<G>(D.sm_count), hi);
        SOCP_PHASE(32, 3);
        for (int j = tid; j < n; j += G) W.diag[j] = fmax(W.diag[j], W.wa2[j]);
        gsync<G>();
        dogleg_and_request<G>(D, b, W, is, ds, red, next_res, next_cnt);
        gsync<G>();
        gcopy<G>(D.xe + b * n, W.xe, n); gcopy<G>(D.diag + b * n, W.diag, n);
        gcopy<G>(D.qtf + b * n, W.qtf, n); gcopy<G>(D.wa1 + b * n, W.wa1, n);
        if (STAGE_R) gcopy<G>(D.r + (size_t)b * D.LRS, W.r, D.LR);
        SOCP_PHASE(32, 5);
        if (q_in_global) {
            // qform_p wrote Q to global memory column by column
        } else if (bulk) {
            // the accumulated Q leaves with one bulk copy; the next problem's copy in waits for it to have read the buffer
            fence_async_smem();
            gsync<G>();
            if (tid == 0) bulk_s2g(gq, W.q, (unsigned)D.QS * 8u);
        } else if (STAGE_Q)
            for (int c = tid >> 5; c < n; c += G / 32)
                for (int i = tid & 31; i < n; i += 32) gq[i + (size_t)c * n] = W.q[i + (size_t)c * ldq_s];
        gsync<G>();
        SOCP_PHASE(32, 6);
    }
    if (bulk && threadIdx.x == 0) bulk_wait_all();
}

template <int G, bool STAGE_R, bool STAGE_Q>
__global__ void __launch_bounds__(128, 3)      // three CTAs per SM is what shared memory allows at P = 85: 168 registers
hybrd_jac_kernel(SolverDev D, int cur, int per_group_doubles) {
    jac_loop<G, STAGE_R, STAGE_Q, false>(D, cur, per_group_doubles);
}

// The Jacobian phase of the shapes with a structural band (SolverDev::band_doubles > 0, 32 < P <= 96, blocks of 14):
// three warps, one thread per column, and the band instead of the dense matrix in shared memory (P = 85: 41 740 B instead
// of 72 160 B per problem), so that five problems share an SM.  At five CTAs (15 warps, four on one SM sub-partition)
// the register cap is 128: the kernel spills 96 bytes, of indices and pointers that stay fixed over a problem.
// Four CTAs at 168 registers do not spill but were no faster than the dense kernel over a whole solve.
__global__ void __launch_bounds__(96, 5)
hybrd_jac_band_kernel(SolverDev D, int cur, int per_group_doubles) {
    jac_loop<96, false, true, true>(D, cur, per_group_doubles);
}

// ---- small kernels -------------------------------------------------------------------------------
__global__ void solver_init(SolverDev D, const double *x_in, long first, const int *active) {
    // problems [first, first + B): copy the unknowns, reset the state, enqueue the first residual.
    // active != nullptr (continuation passes): only the problems whose flag is set take part; the others keep
    // PH_IDLE and are never listed.  counts[] was zeroed by the caller; the list order is the order of the atomics
    // (a problem's result does not depend on its position in any list).
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < D.B * D.P) {
        const double v = x_in[first * D.P + i];
        D.x[i] = v;
        D.xe[i] = v;
    }
    if (i < D.B) {
        int *is = D.istate + i * I_COUNT;
        for (int k = 0; k < I_COUNT; ++k) is[k] = 0;
        for (int k = 0; k < D_COUNT; ++k) D.dstate[i * D_COUNT + k] = 0.;
        if (!active) {
            is[I_PHASE] = PH_F0;
            D.lists[i] = (int)i;                                   // lists[0][0] = residual requests of round 0
            if (i == 0) D.counts[0] = (int)D.B;
        } else if (active[first + i]) {
            is[I_PHASE] = PH_F0;
            D.lists[atomicAdd(&D.counts[0], 1)] = (int)i;
        }
    }
}

__global__ void solver_finish(SolverDev D, long first, double *x_out, double *fvec_out, double *fjac_out,
                              int *info, int *nfev, double *fnorm, int *njev, const int *active) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (x_out && i < D.B * D.P && (!active || active[first + i / D.P])) x_out[first * D.P + i] = D.x[i];
    if (fvec_out && i < D.B * D.P) fvec_out[first * D.P + i] = D.fvec[i];
    if (fjac_out && i < D.B * (long)D.P * D.P) {
        const long pp = (long)D.P * D.P;
        fjac_out[first * pp + i] = D.fjac[(i / pp) * D.QS + (i % pp)];
    }
    if (i < D.B && (!active || active[first + i])) {
        const int *is = D.istate + i * I_COUNT;
        // a problem still in flight when the round limit is hit is NOT a hybrd outcome: it gets its own code
        // (SOCP_INFO_UNFINISHED, negative like hybrd's user-abort codes), distinct from a genuine maxfev (2)
        if (info) info[first + i] = (is[I_PHASE] == PH_IDLE) ? is[I_INFO] : SOCP_INFO_UNFINISHED;
        if (nfev) nfev[first + i] = is[I_NFEV];
        if (njev) njev[first + i] = is[I_NJEV];
        if (fnorm) fnorm[first + i] = D.dstate[i * D_COUNT + D_FNORM];
    }
}

// ---- continuation on the device (shooting.cpp:598-692 boundary data, :695-778 model parameter) -----------------
// Every problem runs the reference's homotopy loop with its own (b, b_prec): all state lives in HBM, the host
// only launches passes and reads ONE counter (problems still in their loop) after each.
struct ContDev {
    long B;
    int P, np, nt, nx;                 // unknowns, parameter block, M + 1 node times, (M + 1) dim boundary values
    int param_idx;                     // >= 0: homotopy on mparams[param_idx]; < 0: on the boundary data
    double step, step_min;
    double *b, *b_prec, *rstart;       // [B] homotopy state (rstart: parameter value at b = 0)
    const double *goal;                // [B] parameter goal
    int *active;                       // [B] 1 while the problem is in its loop
    int *n_active;                     // [1]
    double *x;                         // [B][P] last accepted solution (the caller's array: result)
    double *xw;                        // [B][P] guess in / solution out of the current pass
    double *mparams;                   // [B][np] (param homotopy: entry param_idx is rewritten every pass)
    const double *time_prec, *Xb_prec, *time_des, *Xb_des;     // boundary homotopy end points
    double *time_w, *Xb_w;             // [B][nt], [B][nx] boundary data of the current pass
    int *info_w, *nfev_w;              // [B] outcome of the current pass
    int *info, *calls;                 // [B], [B][2] results (calls may be null)
};

// first pass set-up: b = min(step, 1), b_prec = 0, every problem active, xw = x
__global__ void cont_begin(ContDev C) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < C.B * C.P) C.xw[i] = C.x[i];
    if (i < C.B) {
        C.b[i] = fmin(C.step, 1.0);
        C.b_prec[i] = 0.;
        C.active[i] = 1;
        C.info[i] = 0;
        if (C.calls) { C.calls[2 * i] = 0; C.calls[2 * i + 1] = 0; }
        if (C.param_idx >= 0) C.rstart[i] = C.mparams[i * C.np + C.param_idx];
        if (i == 0) *C.n_active = (int)C.B;
    }
}

// data of the next solve for every active problem: (1 - b) prev + b desired  (shooting.cpp:609-611, :707)
__global__ void cont_setup(ContDev C) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (C.param_idx >= 0) {
        if (i < C.B && C.active[i]) {
            const double bk = C.b[i];
            C.mparams[i * C.np + C.param_idx] = (1 - bk) * C.rstart[i] + bk * C.goal[i];
        }
        return;
    }
    const int per = C.nt + C.nx;
    if (i >= C.B * per) return;
    const long k = i / per;
    const int e = (int)(i % per);
    if (!C.active[k]) return;
    const double bk = C.b[k];
    if (e < C.nt) C.time_w[k * C.nt + e] = (1 - bk) * C.time_prec[k * C.nt + e] + bk * C.time_des[k * C.nt + e];
    else C.Xb_w[k * C.nx + e - C.nt] = (1 - bk) * C.Xb_prec[k * C.nx + e - C.nt] + bk * C.Xb_des[k * C.nx + e - C.nt];
}

// the homotopy state machine after a pass; one warp per problem (the P-wide copies are coalesced)
__global__ void cont_update(ContDev C) {
    const long k = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (k >= C.B || !C.active[k]) return;
    const int ret = C.info_w[k];
    double b = C.b[k], b_prec = C.b_prec[k];
    int still = 1;
    double *x = C.x + k * C.P, *xw = C.xw + k * C.P;
    if (ret != 1) {
        // failure: halve the step and restart from the last accepted solution (shooting.cpp:627-640, :731-742)
        if (fabs(b - b_prec) < C.step_min) still = 0;
        b = b_prec + (b - b_prec) / 2;
        for (int j = lane; j < C.P; j += 32) xw[j] = x[j];
    } else {
        // success: accept, advance b by the step (capped at 1); b == 1 exactly ends the loop (:651-660, :751-759)
        for (int j = lane; j < C.P; j += 32) x[j] = xw[j];
        if (b == 1) still = 0;
        else { b_prec = b; b = fmin(b + C.step, 1.0); }
    }
    if (lane == 0) {
        C.info[k] = ret;
        if (C.calls) { C.calls[2 * k] += 1; C.calls[2 * k + 1] += C.nfev_w[k]; }
        C.b[k] = b; C.b_prec[k] = b_prec;
        // the parameter follows b on every path but the final success, as in the reference (:635-637, :757)
        if (C.param_idx >= 0 && !(ret == 1 && still == 0))
            C.mparams[k * C.np + C.param_idx] = (1 - b) * C.rstart[k] + b * C.goal[k];
        if (!still) { C.active[k] = 0; atomicSub(C.n_active, 1); }
    }
}

// ---- host-side workspace ---------------------------------------------------------------------------
struct SolverWorkspace {
    void *blob = nullptr;
    size_t cap = 0;
    int *h_counts = nullptr;          // pinned
    cudaEvent_t ev = nullptr;
    void release() {
        if (blob) cudaFree(blob);
        blob = nullptr; cap = 0;
        if (h_counts) cudaFreeHost(h_counts);
        h_counts = nullptr;
        if (ev) cudaEventDestroy(ev);
        ev = nullptr;
    }
    double bytes() const { return (double)cap; }
};

}  // namespace socp
