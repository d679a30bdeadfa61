// socp_b200/csrc/api.cu -- C ABI of libsocp_b200.so (see include/socp_b200.h).
// Host-side plumbing only: argument checks, staging of host buffers, kernel launches on the
// context stream, statistics.  All arithmetic of the hot path lives in the kernels.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <string>
#include <vector>
#include <algorithm>
#include <map>
#include <type_traits>

#include "../../include/socp_b200.h"
#include "models.cuh"
#include "integrate.cuh"
#include "solver.cuh"
#include "move.cuh"

using namespace socp;

namespace {
std::string g_create_error;

// Calls f(std::integral_constant<int, MODEL>) with the compile-time model of a valid SOCP_* model id.
template <typename F>
void with_model(int id, F &&f) {
    switch (id) {
    case SOCP_GODDARD: f(std::integral_constant<int, GODDARD>()); break;
    case SOCP_DOUBLE_INTEGRATOR: f(std::integral_constant<int, DOUBLE_INTEGRATOR>()); break;
    case SOCP_COVID19: f(std::integral_constant<int, COVID19>()); break;
    case SOCP_VTOL_UAV: f(std::integral_constant<int, VTOL_UAV>()); break;
    case SOCP_INTERCEPTOR: f(std::integral_constant<int, INTERCEPTOR>()); break;
    }
}

bool valid_model(int id) { return id >= 0 && id < SOCP_NUM_MODELS; }

struct ModelFacts {
    int dim, np, steps;
    int trace_width;                     // a trace row as trace_kernel writes it: t, X[N], control[NCTRL], H, extra
};
ModelFacts model_facts(int id) {
    ModelFacts f{};
    with_model(id, [&](auto m) {
        using Mo = Model<decltype(m)::value>;
        f = {Mo::DIM, Mo::NP, Mo::DEFAULT_STEPS, Mo::N + Mo::NCTRL + 3};
    });
    return f;
}

const double kPi = 3.14159265358979323846;
const double kDefaults[SOCP_NUM_MODELS][17] = {
    {3.5, 7.0, 310.0, 500.0, 1.0, 1.0, 0.0, -1.0},                       // goddard.hpp:29-36
    {1.0, 1.0, 0.01},                                                    // doubleIntegrator.cpp:30-32
    {4.0, 10.0, 5.0, 1.0, 0.1, 1.0, -10.0, 20.0},                        // covid19.cpp:29-36
    {10.0, 0.3, 0.05, 0.0, 1.0 / 60, 1.0, 0.0, 0.0, 0.0, 1.0, 0.03, 1.0, 2.5},  // vtolUAV.cpp:27-35
    {0.00075, 7500.0, 0.00005, 0.442, 200.0, 200.0, 10.0, 1500.0, kPi / 6, 1.0, 1500.0, 0.0, 0.0,
     1.0, 0.0, 1.0, 0.0},                                                // interceptor.cpp:36-50
};
}  // namespace

// A grow-only device buffer
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};

struct socp_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t stream2 = nullptr;      // Jacobian phase of a solver round, forked from / joined to `stream` with the two events
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    std::string err;
    std::vector<DevBuf> pool;            // workspace slots
    unsigned long long *d_counters = nullptr;   // [0] rk4 steps
    double launches = 0, rounds = 0;
    double steps_base = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    int sm_count = 0;
    int profile = 0;
    double integrate_ms = 0, integrate_launches = 0, advance_ms = 0, advance_launches = 0, assemble_ms = 0, jac_ms = 0, qpass_ms = 0;
    std::vector<cudaEvent_t> prof_events;
    SolverWorkspace solver;              // persistent state of the batched solver (solver.cuh)
    std::map<const void *, size_t> smem_configured;   // opt-in dynamic shared memory per kernel, on THIS device
    int launch_error = 0;                // set by a failed launch configuration inside a solver round
};

#define CUDA_TRY(ctx, call)                                                              \
    do {                                                                                 \
        cudaError_t e_ = (call);                                                         \
        if (e_ != cudaSuccess) {                                                         \
            (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e_);             \
            return SOCP_ERR_CUDA;                                                        \
        }                                                                                \
    } while (0)

static int fail(socp_ctx *ctx, int code, const std::string &msg) {
    if (ctx) ctx->err = msg;
    return code;
}

// error return after host buffers may have been staged: no asynchronous copy from (or to) a caller buffer
// is left in flight when the call returns an error
static int bail(socp_ctx *ctx, int rc) {
    if (ctx) cudaStreamSynchronize(ctx->stream);
    return rc;
}

// SOCP_ERR_CUDA, with the error text in ctx->err, when a launch (or an earlier runtime call) of this thread failed
static int last_launch(socp_ctx *ctx) {
    CUDA_TRY(ctx, cudaGetLastError());
    return SOCP_OK;
}

// the last step of a batch call: with host buffers, the outputs have arrived when it returns
static int finish(socp_ctx *ctx, int mem) {
    if (mem == SOCP_HOST) CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return SOCP_OK;
}

// workspace slot `slot` with at least `bytes` bytes
static void *ws(socp_ctx *ctx, size_t slot, size_t bytes) {
    if (ctx->pool.size() <= slot) ctx->pool.resize(slot + 1);
    DevBuf &b = ctx->pool[slot];
    if (b.cap < bytes) {
        if (b.p) cudaFree(b.p);
        b.p = nullptr;
        b.cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        if (cudaMalloc(&b.p, want) != cudaSuccess) {
            cudaGetLastError();
            ctx->err = "cudaMalloc failed for " + std::to_string(want) + " bytes";
            return nullptr;
        }
        b.cap = want;
    }
    return b.p;
}

// Stage a caller buffer: returns a device pointer (the caller's own when mem == DEVICE).
template <typename T>
static const T *stage_in(socp_ctx *ctx, size_t slot, const T *src, size_t count, int mem, int *rc) {
    if (!src || count == 0) return nullptr;
    if (mem == SOCP_DEVICE) return src;
    T *d = (T *)ws(ctx, slot, count * sizeof(T));
    if (!d) { *rc = SOCP_ERR_NOMEM; return nullptr; }
    cudaError_t e = cudaMemcpyAsync(d, src, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); *rc = SOCP_ERR_CUDA; return nullptr; }
    return d;
}
template <typename T>
static T *stage_out(socp_ctx *ctx, size_t slot, T *dst, size_t count, int mem, int *rc) {
    if (!dst || count == 0) return nullptr;
    if (mem == SOCP_DEVICE) return dst;
    T *d = (T *)ws(ctx, slot, count * sizeof(T));
    if (!d) { *rc = SOCP_ERR_NOMEM; return nullptr; }
    return d;
}
template <typename T>
static int fetch_out(socp_ctx *ctx, T *dst, const T *dev, size_t count, int mem) {
    if (!dst || mem == SOCP_DEVICE || count == 0) return SOCP_OK;
    CUDA_TRY(ctx, cudaMemcpyAsync(dst, dev, count * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
    return SOCP_OK;
}

enum { SLOT_MPARAMS = 0, SLOT_SW, SLOT_T0, SLOT_TF, SLOT_X0, SLOT_XF, SLOT_AUX0, SLOT_AUX1, SLOT_AUX2,
       SLOT_TIME, SLOT_XB, SLOT_X, SLOT_FVEC, SLOT_FJAC, SLOT_INFO, SLOT_NFEV, SLOT_FNORM, SLOT_PEAK,
       SLOT_CONT, SLOT_CONT_A, SLOT_CONT_B, SLOT_SOLVER_BASE };

// The inputs of the trajectory-family calls on the device: mparams [B][np], sw [B][2], t0 [B], tf [B] and
// X0 [B][nx] (null where the call has no such input).
struct TrajIn {
    const double *mp, *sw, *t0, *tf, *X0;
};
static TrajIn stage_traj(socp_ctx *ctx, long B, int np, int nx, const double *mparams, const double *sw,
                         const double *t0, const double *tf, const double *X0, int mem, int *rc) {
    return {stage_in(ctx, SLOT_MPARAMS, mparams, (size_t)B * np, mem, rc), stage_in(ctx, SLOT_SW, sw, (size_t)B * 2, mem, rc),
            stage_in(ctx, SLOT_T0, t0, (size_t)B, mem, rc), stage_in(ctx, SLOT_TF, tf, (size_t)B, mem, rc),
            stage_in(ctx, SLOT_X0, X0, (size_t)B * nx, mem, rc)};
}

// cooperative groups (Coop<MODEL>::LANES lanes per trajectory) when one thread per trajectory cannot fill the GPU:
// fewer threads than the device holds at the kernel's occupancy.
static bool use_coop(socp_ctx *ctx, long items, int lanes) {
    if (lanes <= 1) return false;
    return items * lanes <= (long)ctx->sm_count * 128 * 4;
}

template <int MODEL>
static void launch_traj(socp_ctx *ctx, long B, int S, const TrajIn &in, double *Xf, double tol, int *nsteps) {
    const int threads = SOCP_TRAJ_THREADS;
    constexpr int L = Coop<MODEL>::LANES;
    if (use_coop(ctx, B, L)) {
        const long blocks = (B * L + threads - 1) / threads;
        if (tol > 0.)
            traj_kernel<MODEL, true, L><<<(unsigned)blocks, threads, 0, ctx->stream>>>(B, S, in.mp, in.sw, in.t0, in.tf, in.X0, Xf, ctx->d_counters, tol, nsteps);
        else
            traj_kernel<MODEL, false, L><<<(unsigned)blocks, threads, 0, ctx->stream>>>(B, S, in.mp, in.sw, in.t0, in.tf, in.X0, Xf, ctx->d_counters, 0., nullptr);
        ctx->launches += 1;
        return;
    }
    long blocks = (B + threads - 1) / threads;
    if (tol > 0.)
        traj_kernel<MODEL, true><<<(unsigned)blocks, threads, 0, ctx->stream>>>(B, S, in.mp, in.sw, in.t0, in.tf, in.X0, Xf, ctx->d_counters, tol, nsteps);
    else
        traj_kernel<MODEL, false><<<(unsigned)blocks, threads, 0, ctx->stream>>>(B, S, in.mp, in.sw, in.t0, in.tf, in.X0, Xf, ctx->d_counters, 0., nullptr);
    ctx->launches += 1;
}

// fixed-step (tol = 0) or adaptive (tol > 0) trajectories; `what` names the entry point in the error text
static int traj_batch(socp_ctx *ctx, const char *what, int model_id, int step_nbr, long B, const double *mparams,
                      const double *sw, const double *t0, const double *tf, const double *X0, double tol, double *Xf,
                      int *nsteps, int mem) {
    if (!ctx) return SOCP_ERR_ARG;
    if (!valid_model(model_id) || B < 0 || !mparams || !t0 || !tf || !X0 || !Xf)
        return fail(ctx, SOCP_ERR_ARG, std::string(what) + ": bad arguments");
    if (B == 0) return SOCP_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const ModelFacts m = model_facts(model_id);
    const int N = 2 * m.dim, S = step_nbr > 0 ? step_nbr : m.steps;
    int rc = SOCP_OK;
    const TrajIn in = stage_traj(ctx, B, m.np, N, mparams, sw, t0, tf, X0, mem, &rc);
    double *d_Xf = stage_out(ctx, SLOT_XF, Xf, (size_t)B * N, mem, &rc);
    int *d_ns = stage_out(ctx, SLOT_INFO, nsteps, (size_t)B * 2, mem, &rc);
    if (rc != SOCP_OK) return bail(ctx, rc);
    with_model(model_id, [&](auto mo) { launch_traj<decltype(mo)::value>(ctx, B, S, in, d_Xf, tol, d_ns); });
    if ((rc = last_launch(ctx)) != SOCP_OK || (rc = fetch_out(ctx, Xf, d_Xf, (size_t)B * N, mem)) != SOCP_OK ||
        (rc = fetch_out(ctx, nsteps, d_ns, (size_t)B * 2, mem)) != SOCP_OK)
        return bail(ctx, rc);
    return finish(ctx, mem);
}

extern "C" {

// ---- static facts ---------------------------------------------------------------------------
int socp_model_dim(int id) { return valid_model(id) ? model_facts(id).dim : SOCP_ERR_ARG; }
int socp_model_nparams(int id) { return valid_model(id) ? model_facts(id).np : SOCP_ERR_ARG; }
int socp_model_default_steps(int id) { return valid_model(id) ? model_facts(id).steps : SOCP_ERR_ARG; }
int socp_model_default_params(int id, double *out) {
    if (!valid_model(id) || !out) return SOCP_ERR_ARG;
    std::copy_n(kDefaults[id], model_facts(id).np, out);
    return SOCP_OK;
}
int socp_num_param(const socp_shape *s) {
    if (!s || !valid_model(s->model_id) || s->num_multi < 1 || s->num_multi >= SOCP_MAX_NODES)
        return SOCP_ERR_ARG;
    int nfree = 0;
    for (int j = 0; j <= s->num_multi; ++j)
        if (s->mode_t[j] == SOCP_FREE) ++nfree;
    return 2 * model_facts(s->model_id).dim * s->num_multi + nfree;
}

// ---- context --------------------------------------------------------------------------------
int socp_create(int device, socp_ctx **out) {
    if (!out) return SOCP_ERR_ARG;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        g_create_error = std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count is 0") +
                         " (libsocp_b200 has no CPU fallback)";
        cudaGetLastError();
        return SOCP_ERR_CUDA;
    }
    if (device < 0 || device >= n) { g_create_error = "bad device index"; return SOCP_ERR_ARG; }
    socp_ctx *ctx = new socp_ctx;
    ctx->device = device;
    if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) {
        g_create_error = cudaGetErrorString(e);
        delete ctx;
        return SOCP_ERR_CUDA;
    }
    ctx->own_stream = true;
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    ctx->sm_count = prop.multiProcessorCount;
    // every allocation of the context is checked: a half-built context is destroyed, never returned
    if ((e = cudaMalloc(&ctx->d_counters, 64 * sizeof(unsigned long long))) != cudaSuccess ||
        (e = cudaMemset(ctx->d_counters, 0, 64 * sizeof(unsigned long long))) != cudaSuccess ||
        (e = cudaEventCreate(&ctx->ev0)) != cudaSuccess || (e = cudaEventCreate(&ctx->ev1)) != cudaSuccess ||
        (e = cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming)) != cudaSuccess) {
        g_create_error = std::string("socp_create: ") + cudaGetErrorString(e);
        const int code = (e == cudaErrorMemoryAllocation) ? SOCP_ERR_NOMEM : SOCP_ERR_CUDA;
        cudaGetLastError();
        socp_destroy(ctx);
        return code;
    }
    *out = ctx;
    return SOCP_OK;
}

void socp_destroy(socp_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto &b : ctx->pool)
        if (b.p) cudaFree(b.p);
    ctx->solver.release();
    if (ctx->d_counters) cudaFree(ctx->d_counters);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    if (ctx->stream2) { cudaStreamSynchronize(ctx->stream2); cudaStreamDestroy(ctx->stream2); }
    for (auto e : ctx->prof_events) cudaEventDestroy(e);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char *socp_last_error(const socp_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int socp_set_stream(socp_ctx *ctx, void *s) {
    if (!ctx) return SOCP_ERR_ARG;
    cudaStreamSynchronize(ctx->stream);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    ctx->stream = (cudaStream_t)s;
    ctx->own_stream = false;
    return SOCP_OK;
}

int socp_sync(socp_ctx *ctx) {
    if (!ctx) return SOCP_ERR_ARG;
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return SOCP_OK;
}

int socp_get_stats(socp_ctx *ctx, socp_stats *out) {
    if (!ctx || !out) return SOCP_ERR_ARG;
    unsigned long long c[64];
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    CUDA_TRY(ctx, cudaMemcpy(c, ctx->d_counters, sizeof c, cudaMemcpyDeviceToHost));
    out->rk4_steps = (double)c[0];
    out->kernel_launches = ctx->launches;
    out->solver_rounds = ctx->rounds;
    double bytes = 0;
    for (auto &b : ctx->pool) bytes += (double)b.cap;
    out->device_bytes = bytes + ctx->solver.bytes();
    out->integrate_ms = ctx->integrate_ms; out->integrate_launches = ctx->integrate_launches;
    out->advance_ms = ctx->advance_ms; out->advance_launches = ctx->advance_launches;
    out->assemble_ms = ctx->assemble_ms;
    out->jac_ms = ctx->jac_ms;
    out->iterations = (double)c[1];
    out->jac_evals = (double)c[2];
    out->dopri_steps = (double)c[3];
    out->res_evals = (double)c[4];
    out->qpass_ms = ctx->qpass_ms;
    if (getenv("SOCP_PHASE_CLOCKS")) {
        fprintf(stderr, "phase clocks (cycles): res");
        for (int k = 0; k < 8; ++k) fprintf(stderr, " %llu", c[16 + k]);
        fprintf(stderr, " | jac");
        for (int k = 0; k < 8; ++k) fprintf(stderr, " %llu", c[32 + k]);
        fprintf(stderr, " | sub");
        for (int k = 0; k < 8; ++k) fprintf(stderr, " %llu", c[48 + k]);
        fprintf(stderr, " | iterations %llu jac_evals %llu\n", c[1], c[2]);
    }
    return SOCP_OK;
}

int socp_reset_stats(socp_ctx *ctx) {
    if (!ctx) return SOCP_ERR_ARG;
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_counters, 0, 64 * sizeof(unsigned long long), ctx->stream));
    ctx->launches = 0;
    ctx->rounds = 0;
    ctx->integrate_ms = ctx->integrate_launches = ctx->advance_ms = ctx->advance_launches = ctx->assemble_ms = ctx->jac_ms = ctx->qpass_ms = 0;
    return SOCP_OK;
}

int socp_set_profiling(socp_ctx *ctx, int on) {
    if (!ctx) return SOCP_ERR_ARG;
    ctx->profile = on ? 1 : 0;
    return SOCP_OK;
}

int socp_timer_start(socp_ctx *ctx) {
    if (!ctx) return SOCP_ERR_ARG;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    return SOCP_OK;
}
int socp_timer_stop(socp_ctx *ctx, float *ms) {
    if (!ctx || !ms) return SOCP_ERR_ARG;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    CUDA_TRY(ctx, cudaEventSynchronize(ctx->ev1));
    CUDA_TRY(ctx, cudaEventElapsedTime(ms, ctx->ev0, ctx->ev1));
    return SOCP_OK;
}

int socp_set_obstacles(socp_ctx *ctx, int n, const double *type, const double *pos, const double *rad) {
    if (!ctx || n < 0 || n > SOCP_MAX_OBS || (n > 0 && (!type || !pos || !rad))) return fail(ctx, SOCP_ERR_ARG, "socp_set_obstacles: bad arguments");
    double tab[SOCP_MAX_OBS * 7];
    for (int i = 0; i < n; ++i) {
        tab[i * 7] = type[i];
        for (int k = 0; k < 3; ++k) { tab[i * 7 + 1 + k] = pos[i * 3 + k]; tab[i * 7 + 4 + k] = rad[i * 3 + k]; }
    }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    // the table is shared by every context of this device: wait for ALL of its streams, not only ours,
    // so that no in-flight vtolUAV kernel of another context reads a half-updated table
    CUDA_TRY(ctx, cudaDeviceSynchronize());
    if (n) CUDA_TRY(ctx, cudaMemcpyToSymbol(c_obstacles, tab, sizeof(double) * 7 * n));
    CUDA_TRY(ctx, cudaMemcpyToSymbol(c_num_obstacles, &n, sizeof(int)));
    return SOCP_OK;
}

// ---- trajectories ---------------------------------------------------------------------------
int socp_traj_batch(socp_ctx *ctx, int model_id, int step_nbr, long B, const double *mparams,
                    const double *sw, const double *t0, const double *tf, const double *X0,
                    double *Xf, int mem) {
    return traj_batch(ctx, "socp_traj_batch", model_id, step_nbr, B, mparams, sw, t0, tf, X0, 0., Xf, nullptr, mem);
}

int socp_traj_adaptive_batch(socp_ctx *ctx, int model_id, int step_nbr, long B, const double *mparams,
                             const double *sw, const double *t0, const double *tf, const double *X0,
                             double tol, double *Xf, int *nsteps, int mem) {
    if (!(tol > 0.)) return fail(ctx, SOCP_ERR_ARG, "socp_traj_adaptive_batch: bad arguments");
    return traj_batch(ctx, "socp_traj_adaptive_batch", model_id, step_nbr, B, mparams, sw, t0, tf, X0, tol, Xf, nsteps, mem);
}

int socp_trace_width(int id) { return valid_model(id) ? model_facts(id).trace_width : SOCP_ERR_ARG; }
int socp_trace_max_rows(int id, int step_nbr) {
    if (!valid_model(id)) return SOCP_ERR_ARG;
    const int S = step_nbr > 0 ? step_nbr : model_facts(id).steps;
    return (S + 1) * (id == SOCP_INTERCEPTOR ? 2 : 1);
}

int socp_trace_batch(socp_ctx *ctx, int model_id, int step_nbr, long B, const double *mparams,
                     const double *sw, const double *t0, const double *tf, const double *X0,
                     double *rows, int *nrows, double *Xf, int mem) {
    if (!ctx) return SOCP_ERR_ARG;
    if (!valid_model(model_id) || B < 0 || !mparams || !t0 || !tf || !X0 || !rows || !nrows)
        return fail(ctx, SOCP_ERR_ARG, "socp_trace_batch: bad arguments");
    if (B == 0) return SOCP_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const ModelFacts m = model_facts(model_id);
    const int N = 2 * m.dim, S = step_nbr > 0 ? step_nbr : m.steps;
    const int W = m.trace_width, R = socp_trace_max_rows(model_id, S);
    int rc = SOCP_OK;
    const TrajIn in = stage_traj(ctx, B, m.np, N, mparams, sw, t0, tf, X0, mem, &rc);
    double *d_rows = stage_out(ctx, SLOT_AUX0, rows, (size_t)B * R * W, mem, &rc);
    int *d_nr = stage_out(ctx, SLOT_INFO, nrows, (size_t)B, mem, &rc);
    double *d_Xf = stage_out(ctx, SLOT_XF, Xf, (size_t)B * N, mem, &rc);
    if (rc != SOCP_OK) return bail(ctx, rc);
    with_model(model_id, [&](auto mo) {
        trace_kernel<decltype(mo)::value><<<(unsigned)((B + 63) / 64), 64, 0, ctx->stream>>>(
            B, S, R, in.mp, in.sw, in.t0, in.tf, in.X0, d_rows, d_nr, d_Xf);
    });
    ctx->launches += 1;
    if ((rc = last_launch(ctx)) != SOCP_OK || (rc = fetch_out(ctx, rows, d_rows, (size_t)B * R * W, mem)) != SOCP_OK ||
        (rc = fetch_out(ctx, nrows, d_nr, (size_t)B, mem)) != SOCP_OK || (rc = fetch_out(ctx, Xf, d_Xf, (size_t)B * N, mem)) != SOCP_OK)
        return bail(ctx, rc);
    return finish(ctx, mem);
}

int socp_point_batch(socp_ctx *ctx, int model_id, long B, const double *mparams, const double *sw,
                     const int *chart_stage, const double *t, const double *X, double *rhs,
                     double *control, double *H, int mem) {
    if (!ctx) return SOCP_ERR_ARG;
    if (!valid_model(model_id) || B < 0 || !mparams || !t || !X)
        return fail(ctx, SOCP_ERR_ARG, "socp_point_batch: bad arguments");
    if (B == 0) return SOCP_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const ModelFacts m = model_facts(model_id);
    const int N = 2 * m.dim;
    int rc = SOCP_OK;
    const TrajIn in = stage_traj(ctx, B, m.np, N, mparams, sw, t, nullptr, X, mem, &rc);
    const int *d_cs = stage_in(ctx, SLOT_INFO, chart_stage, (size_t)B * 2, mem, &rc);
    double *d_rhs = stage_out(ctx, SLOT_AUX0, rhs, (size_t)B * N, mem, &rc);
    double *d_ctl = stage_out(ctx, SLOT_AUX1, control, (size_t)B * 4, mem, &rc);
    double *d_H = stage_out(ctx, SLOT_AUX2, H, (size_t)B, mem, &rc);
    if (rc != SOCP_OK) return bail(ctx, rc);
    with_model(model_id, [&](auto mo) {
        point_kernel<decltype(mo)::value><<<(unsigned)((B + 127) / 128), 128, 0, ctx->stream>>>(
            B, in.mp, in.sw, d_cs, in.t0, in.X0, d_rhs, d_ctl, d_H);
    });
    ctx->launches += 1;
    if ((rc = last_launch(ctx)) != SOCP_OK || (rc = fetch_out(ctx, rhs, d_rhs, (size_t)B * N, mem)) != SOCP_OK ||
        (rc = fetch_out(ctx, control, d_ctl, (size_t)B * 4, mem)) != SOCP_OK || (rc = fetch_out(ctx, H, d_H, (size_t)B, mem)) != SOCP_OK)
        return bail(ctx, rc);
    return finish(ctx, mem);
}

// ---- FP64 peak probe ------------------------------------------------------------------------
int socp_measure_fp64_peak(socp_ctx *ctx, double *gflops, double *sm_clock_mhz) {
    if (!ctx || !gflops) return SOCP_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const int threads = 256, blocks = ctx->sm_count * 8, iters = 4096;
    double *out = (double *)ws(ctx, SLOT_PEAK, sizeof(double) * threads * blocks);
    if (!out) return SOCP_ERR_NOMEM;
    float best = 1e30f;
    for (int rep = 0; rep < 6; ++rep) {
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
        dfma_peak_kernel<<<blocks, threads, 0, ctx->stream>>>(out, iters, 0.999999, 1e-9);
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
        CUDA_TRY(ctx, cudaEventSynchronize(ctx->ev1));
        float ms = 0;
        CUDA_TRY(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        if (rep > 0 && ms < best) best = ms;
    }
    ctx->launches += 6;
    double fmas = (double)threads * blocks * (double)iters * 64.0;
    *gflops = 2.0 * fmas / (best * 1e-3) / 1e9;
    if (sm_clock_mhz) {
        int khz = 0;
        cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, ctx->device);
        *sm_clock_mhz = khz / 1000.0;
    }
    return SOCP_OK;
}

}  // extern "C"

#include "solver_api.inl"
