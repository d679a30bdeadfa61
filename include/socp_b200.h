/*
 * socp_b200.h -- C ABI of the B200 batched shooting engine (libsocp_b200.so).
 *
 * Drop-in boundary for the hot path of bherisse/socp.  The reference has no FFI of its own; its
 * seams are (i) the C++ `model` / `shooting` classes and (ii) the cminpack callback ABI
 * (`int fcn(void*, int, const real*, real*, int)`, src/socp/shooting.hpp:282, called from
 * `hybrd` at src/socp/shooting.cpp:803-826).  Each entry point below names the reference code it
 * replaces for a whole batch of independent problems.  The C++ host mirror of `model`/`shooting`
 * (include/socp/) and the Python host (socp_b200/) both sit on top of exactly these symbols.
 *
 * Conventions: plain pointers and sizes only; the caller owns every buffer; int status return
 * (0 = ok, <0 = error, message via socp_last_error); no exceptions cross the boundary; all work is
 * ordered on the context's CUDA stream; one context per GPU and per host thread.
 * `mem` selects where the caller's buffers live: SOCP_HOST (the library stages H2D / D2H itself)
 * or SOCP_DEVICE (device pointers on the context's device; results are ordered on the context
 * stream: socp_sync() before reading them from another stream).  The batched solves and continuations
 * block the calling host thread intermittently: the round loop reads device-side work counters every
 * few rounds to know when the last problem has retired; the trajectory / residual / Jacobian / Move / GetSolution / Trace calls only enqueue.  There is no CPU fallback: without a CUDA device
 * socp_create fails.
 *
 * Data layouts (all double unless noted, row-major, one problem after another):
 *   mparams [B][np]          model parameter block, index maps below (np = socp_model_nparams)
 *   time    [B][M+1]         shooting::data_struct::time   (fixed node times)
 *   Xb      [B][M+1][dim]    data->X[i][0..dim): boundary / waypoint states
 *   x       [B][P]           unknowns (tab_param): M blocks of (state, costate), then FREE times
 *   fvec    [B][P]           residual, layout of shooting::ShootingFunction (shooting.cpp:918-993)
 *   fjac    [B][P*P]         column-major d fvec_i / d x_j at [i + j*P] (cminpack convention)
 */
#ifndef SOCP_B200_H
#define SOCP_B200_H

#ifdef __cplusplus
extern "C" {
#endif

/* model ids: src/models/{goddard,doubleIntegrator,covid19,vtolUAV,interceptor} */
enum { SOCP_GODDARD = 0, SOCP_DOUBLE_INTEGRATOR = 1, SOCP_COVID19 = 2, SOCP_VTOL_UAV = 3,
       SOCP_INTERCEPTOR = 4, SOCP_NUM_MODELS = 5 };
/* model::FIXED / FREE / CONTINUOUS (src/socp/model.hpp:34-38) */
enum { SOCP_FIXED = 0, SOCP_FREE = 1, SOCP_CONTINUOUS = 2 };
enum { SOCP_HOST = 0, SOCP_DEVICE = 1 };
/* integrator of model::ModelInt: fixed-step RK4 (the reference's default build, odeTools.cpp:135-144)
 * or adaptive Dormand-Prince 5(4) (its -D_USE_BOOST build, odeTools.cpp:131-134) */
enum { SOCP_RK4 = 0, SOCP_DOPRI5 = 1 };
enum { SOCP_OK = 0, SOCP_ERR_ARG = -1, SOCP_ERR_CUDA = -2, SOCP_ERR_NOMEM = -3, SOCP_ERR_UNSUPPORTED = -4 };
/* per-problem `info` values are MINPACK's (0 bad input, 1 converged, 2 maxfev, 3 xtol too small, 4/5 slow
 * progress); one more value exists only here: the batch driver stopped (its round limit) while the problem
 * was still iterating -- it cannot happen with the default round limit of maxfev + 8 */
#define SOCP_INFO_UNFINISHED (-2)

#define SOCP_MAX_NODES 64
#define SOCP_MAX_DIM 7

/* parameter block indices
 * goddard (goddard.hpp:29-36):        C b KD kr u_max mu1 mu2 singularControl
 * doubleIntegrator (.hpp:27-31):      u_max a_max muT
 * covid19 (covid19.hpp:29-38):        R0 Tinf Tinc N Imax muI umin umax
 * vtolUAV (vtolUAV.hpp:27-37) + obstacle (obstacle.hpp:24-29):
 *                                     u_max a_max alphaT alphaV invSigmaXwp Vd ca nWP_tot nWP
 *                                     phiObs psiWP muObs sigmaWP
 * interceptor (interceptor.hpp:30-48): c0 hr d0 eta propellant_mass empty_mass q ve alpha_max
 *                                     u_max a_max r_2p t_2p mu_gft muT muV muC                   */

typedef struct socp_ctx socp_ctx;

/* Shape shared by every problem of a batch = what shooting::SetMode / Resize fix
 * (shooting.cpp:123-199).  step_nbr <= 0 selects the model's own stepNbr. */
typedef struct {
    int model_id;
    int num_multi;
    int step_nbr;
    int mode_t[SOCP_MAX_NODES];
    int mode_X[SOCP_MAX_NODES][SOCP_MAX_DIM];
    int integrator;          /* SOCP_RK4 (0, default) or SOCP_DOPRI5 */
    double ode_tol;          /* SOCP_DOPRI5: absolute = relative tolerance (odeTools::odeIntTol, odeTools.hpp:62) */
} socp_shape;

typedef struct {
    double rk4_steps;        /* RK4 steps executed by integration kernels since the last reset */
    double kernel_launches;  /* kernels of this library launched since the last reset */
    double solver_rounds;    /* lock-step rounds of the batched Powell-hybrid state machine */
    double device_bytes;     /* workspace currently held on the device */
    /* filled only while profiling is on (socp_set_profiling): CUDA-event time of the two kernels
     * of the solver rounds, on the context stream */
    double integrate_ms, integrate_launches;   /* integrate_worklist */
    double advance_ms, advance_launches;       /* hybrd_res_kernel + hybrd_jac_kernel (Powell-hybrid step) */
    double assemble_ms;                        /* assemble_kernel (residual / FD Jacobian assembly) */
    double jac_ms;                             /* hybrd_jac_kernel alone (included in advance_ms) */
    double iterations;                         /* problem-iterations of hybrd_res_kernel (Broyden steps), device counter */
    double jac_evals;                          /* Jacobian factorisations of hybrd_jac_kernel, device counter */
    double dopri_steps;                        /* accepted Dormand-Prince steps of the adaptive integration kernels */
    double qpass_ms;                           /* hybrd_qpass_kernel alone (included in advance_ms; 0 in the fused build) */
    double res_evals;                          /* residual requests assembled (base + trial points), device counter */
} socp_stats;

/* ---- context ------------------------------------------------------------------------------ */
int socp_create(int device, socp_ctx **ctx);
void socp_destroy(socp_ctx *ctx);
const char *socp_last_error(const socp_ctx *ctx);      /* ctx may be NULL: last create error */
int socp_set_stream(socp_ctx *ctx, void *cuda_stream); /* run on a caller-owned cudaStream_t */
int socp_sync(socp_ctx *ctx);
int socp_get_stats(socp_ctx *ctx, socp_stats *out);
int socp_reset_stats(socp_ctx *ctx);
/* per-kernel CUDA-event timing of the solver rounds (adds two event records per launch) */
int socp_set_profiling(socp_ctx *ctx, int on);
/* wall-clock-free timing of the library's own kernels: CUDA events on the context stream */
int socp_timer_start(socp_ctx *ctx);
int socp_timer_stop(socp_ctx *ctx, float *ms);

/* static facts */
int socp_model_dim(int model_id);        /* model::GetDim (model.hpp:66) */
int socp_model_nparams(int model_id);
int socp_model_default_steps(int model_id);
int socp_model_default_params(int model_id, double *out);     /* constructor defaults */
int socp_num_param(const socp_shape *shape);                   /* shooting.cpp:179,196 */

/* obstacle table of the vtolUAV penalty map (src/maps/obstacle/obstacle.cpp:24-36): type 0 ellipsoid,
 * 1 box; pos/rad are [n][3], host pointers.  The table lives in constant memory of the DEVICE: it is
 * shared by every context of the process on that device (empty until first set; creating another
 * context does not reset it); setting it synchronises the whole DEVICE first (cudaDeviceSynchronize), so no
 * kernel of another context can observe a half-written table. */
int socp_set_obstacles(socp_ctx *ctx, int n, const double *type, const double *pos, const double *rad);

/* ---- hot path ------------------------------------------------------------------------------ */

/* model::ComputeTraj (model.hpp:77; interceptor.cpp:165) for B independent trajectories:
 * fixed-step RK4 (odeTools.cpp:89-98, :128-146), S = step_nbr steps per segment.
 * sw: optional [B][2] goddard switching times (goddard.cpp:27-29, :373), NULL = defaults. */
int socp_traj_batch(socp_ctx *ctx, int model_id, int step_nbr, long B, const double *mparams,
                    const double *sw, const double *t0, const double *tf, const double *X0,
                    double *Xf, int mem);

/* The same with the adaptive integrator of the reference's -D_USE_BOOST build (odeTools.cpp:131-134):
 * Boost.Odeint integrate_adaptive with a dense-output Dormand-Prince 5(4) stepper, abs = rel = tol, first
 * trial step (tf - t0) / step_nbr.  nsteps: optional [B][2] = {accepted steps, rejected attempts}.
 * The interceptor integrates with its own fixed-step loop in that build too (interceptor.cpp:104-130). */
int socp_traj_adaptive_batch(socp_ctx *ctx, int model_id, int step_nbr, long B, const double *mparams,
                             const double *sw, const double *t0, const double *tf, const double *X0,
                             double tol, double *Xf, int *nsteps, int mem);

/* The observer form of the same integration (odeTools.cpp:103-123 with model::Trace,
 * model.hpp:446-462; shooting::Trace re-integrates every segment this way, shooting.cpp:496-544):
 * one row at t0 and one after every RK4 step.  rows is [B][R][W], W = socp_trace_width(model) =
 * 1 + 2dim + ncontrol + 1 + 1 columns {t, X, control, H, extra}, extra = goddard's switching function
 * (goddard.cpp:337) / interceptor's chart id (interceptor.cpp:151) / 0; R = socp_trace_max_rows.
 * nrows[B] receives the rows written per trajectory.  Xf (end points) may be NULL. */
int socp_trace_width(int model_id);
int socp_trace_max_rows(int model_id, int step_nbr);
int socp_trace_batch(socp_ctx *ctx, int model_id, int step_nbr, long B, const double *mparams,
                     const double *sw, const double *t0, const double *tf, const double *X0,
                     double *rows, int *nrows, double *Xf, int mem);

/* odeTools::Model / model::Control / model::Hamiltonian at B points (rhs [B][2dim], control
 * [B][4], H [B]); any output may be NULL.  chart_stage: optional [B][2] ints (interceptor). */
int socp_point_batch(socp_ctx *ctx, int model_id, long B, const double *mparams, const double *sw,
                     const int *chart_stage, const double *t, const double *X, double *rhs,
                     double *control, double *H, int mem);

/* shooting::ShootingFunction (shooting.cpp:918-993) for B problems. */
int socp_residual_batch(socp_ctx *ctx, const socp_shape *shape, long B, const double *mparams,
                        const double *time, const double *Xb, const double *x, double *fvec, int mem);

/* MINPACK fdjac1 (dense) as hybrd applies it to the shooting residual: column j is
 * (F(x + h_j e_j) - F(x)) / h_j, h_j = sqrt(epsfcn)|x_j| (or sqrt(epsfcn) if x_j == 0). */
int socp_fdjac_batch(socp_ctx *ctx, const socp_shape *shape, long B, const double *mparams,
                     const double *time, const double *Xb, const double *x, double epsfcn,
                     double *fjac, int mem);

/* shooting::SolveShootingFunction (shooting.cpp:781-856, modelOrder 0): Powell hybrid with the
 * reference's settings (maxfev given, ml = mu = P-1, epsfcn = 1e-15, mode = 1, factor = 1).
 * x is updated in place for EVERY problem (as hybrd does); info/nfev/fnorm are [B].
 * SOCP accepts a solve iff info == 1 (shooting.cpp:588). */
int socp_solve_batch(socp_ctx *ctx, const socp_shape *shape, long B, const double *mparams,
                     const double *time, const double *Xb, double *x, double xtol, int maxfev,
                     int *info, int *nfev, double *fnorm, int mem);

/* The analytic-Jacobian path, modelOrder == 1 (shooting.cpp:830-851: hybrj on
 * StaticShootingFunctionJacobian, :877-915).  Only the double integrator has variational equations
 * (doubleIntegrator.cpp:113-213), as in the reference; other models return SOCP_ERR_UNSUPPORTED.
 *   socp_traj_var_batch     model::ComputeTraj(isJac = 1): X0/Xf are [B][(2dim+1) 2dim] extended states
 *                           (state, then the sensitivity rows X[2dim (k+1) + i] = dX_k/dX0_i, shooting.cpp:1003)
 *   socp_jacobian_batch     shooting::ShootingFunctionJacobian (shooting.cpp:996-1130), column-major like fjac
 *   socp_solve_hybrj_batch  the Powell hybrid with that Jacobian; nfev counts residuals, njev Jacobians */
int socp_traj_var_batch(socp_ctx *ctx, int model_id, int step_nbr, long B, const double *mparams,
                        const double *t0, const double *tf, const double *X0, double *Xf, int mem);
int socp_jacobian_batch(socp_ctx *ctx, const socp_shape *shape, long B, const double *mparams,
                        const double *time, const double *Xb, const double *x, double *fjac, int mem);
int socp_solve_hybrj_batch(socp_ctx *ctx, const socp_shape *shape, long B, const double *mparams,
                           const double *time, const double *Xb, double *x, double xtol, int maxfev,
                           int *info, int *nfev, int *njev, double *fnorm, int mem);

/* shooting::SolveShootingContinuation on a model parameter (shooting.cpp:695-778), every problem
 * running its own homotopy b in (0,1] with step halving.  mparams is updated in place (entry
 * param_idx ends at goal[b] on success).  goal is [B].  calls is [B][2] = {solver calls, total
 * nfev} (may be NULL).  The per-problem state machines (b, b_prec, the accepted solution, the data of the next
 * pass) live on the device: with mem == SOCP_DEVICE no problem data crosses PCIe at all, with SOCP_HOST the
 * arrays are staged once before the first pass and fetched once after the last.  The call returns when every
 * homotopy has ended (the host reads one counter per pass). */
int socp_continuation_param_batch(socp_ctx *ctx, const socp_shape *shape, long B, double *mparams,
                                  const double *time, const double *Xb, double *x, double xtol,
                                  int maxfev, double step, int param_idx, const double *goal,
                                  double step_min, int *info, int *calls, int mem);

/* shooting::SolveShootingContinuation on the boundary data (shooting.cpp:598-692): homotopy from
 * (time_prec, Xb_prec) to (time_des, Xb_des).  Same conventions. */
int socp_continuation_boundary_batch(socp_ctx *ctx, const socp_shape *shape, long B,
                                     const double *mparams, const double *time_prec,
                                     const double *Xb_prec, const double *time_des,
                                     const double *Xb_des, double *x, double xtol, int maxfev,
                                     double step, double step_min, int *info, int *calls, int mem);

/* Sampling a solution (the unknowns x [B][P] of a solve, with the time [B][M+1] and mparams it was solved with).
 * shooting::Move(tf) (shooting.cpp:383-437) of B solutions x at Q query times each: tq [B][Q], Xq [B][Q][2dim].
 * The time line is ComputeTimeLine's (FREE times from x, CONTINUOUS nodes interpolated), which also sets goddard's
 * switching times; the state is the integration of the segment that holds the target from its node state:
 * seg = 0; while (tl[seg+1] < target) ++seg -- so a query at node time tl[j+1] returns the end of segment j, not
 * node j+1.  A query outside [t0, t_end] (NaN included) is answered at t_end, as in the reference.  A Move is bit
 * for bit the socp_traj_batch (or, with SOCP_DOPRI5, socp_traj_adaptive_batch) of the same segment start, node
 * state, target and switching times.  Q == 0 or B == 0: nothing is done. */
int socp_move_batch(socp_ctx *ctx, const socp_shape *shape, long B, const double *mparams, const double *time,
                    const double *x, int Q, const double *tq, double *Xq, int mem);
/* shooting::GetSolution (shooting.cpp:481-488, UpdateSolution :1462-1508): vt [B][M+1] node times of the
 * solution, vX [B][M+1][2dim] node states (vX[i] = node i of x for i < M, vX[M] = Move(t_end)).  The result is the
 * node data of a re-mesh: Move at the new node times, then InitShooting(vt, vX). */
int socp_solution_batch(socp_ctx *ctx, const socp_shape *shape, long B, const double *mparams, const double *time,
                        const double *x, double *vt, double *vX, int mem);
/* shooting::Trace (shooting.cpp:496-544): every segment of B solutions re-integrated with the observer on.
 * rows [B][M][R][W] and nrows [B][M] (int): rows[b][j] holds the nrows[b][j] rows of segment j of problem b in the
 * layout of socp_trace_batch (R = socp_trace_max_rows(model, step_nbr), W = socp_trace_width(model)); rows past
 * nrows[b][j] are unspecified.  Segment j runs from node time tl[j] (ComputeTimeLine's, as for a Move) and node
 * state j of x to tl[j+1], so it is bit for bit the socp_trace_batch of the same start, node state, end, switching
 * times and step_nbr: S+1 rows, 2(S+1) for an interceptor segment that crosses the burn-out time.  The first row of
 * segment j+1 repeats the node time tl[j+1] that ends segment j, as in the reference's trace file.  A SOCP_DOPRI5
 * shape is traced with the fixed-step RK4 observer too (odeTools.cpp:103-123): the reference has no adaptive
 * observer.  B == 0: nothing is done. */
int socp_solution_trace_batch(socp_ctx *ctx, const socp_shape *shape, long B, const double *mparams, const double *time,
                              const double *x, double *rows, int *nrows, int mem);

/* FP64 FMA peak of the device measured with a register-resident DFMA chain (GFLOP/s). */
int socp_measure_fp64_peak(socp_ctx *ctx, double *gflops, double *sm_clock_mhz);

#ifdef __cplusplus
}
#endif
#endif
