// cpp/src/socp/shooting_batch.cpp -- see shooting_batch.hpp.  Host bookkeeping only; the numerical
// work is socp_init_shooting_batch / socp_solve_batch / socp_continuation_*_batch / socp_move_batch /
// socp_solution_batch / socp_solution_trace_batch (include/socp_b200.h).
#include <cstdlib>
#include <cstring>
#include <functional>
#include <iostream>
#include <thread>

#include "shooting_batch.hpp"
#include "../../../include/socp_b200.h"

struct shooting_batch::data_struct {
	long B;
	int dim, numMulti, numParam;
	socp_shape shape;
	real xtol, stepMin;
	int maxfev;
	std::vector<real> mparams;				// [B][np]
	std::vector<real> time, timed, time_prec;	// [B][M+1]
	std::vector<real> X, Xd, X_prec;		// [B][M+1][dim]   (boundary / waypoint states)
	std::vector<real> param;				// [B][P]
	std::vector<int> info, nfev, calls;
	std::vector<real> fnorm;
	int np;
	int numDevice;
	std::vector<int> devices;				// CUDA device of every block

	// run f(ctx, lo, hi) for the contiguous block [lo, hi) of every device, one host thread per device
	// (a context is used by one thread at a time: the blocks are disjoint and each thread has its own context)
	void for_each_block(std::function<void(socp_ctx *, long, long)> f) const {
		const int G = numDevice;
		const long per = (B + G - 1) / G;
		if (G == 1) { f(model::Context(devices[0]), 0, B); return; }
		std::vector<std::thread> pool;
		for (int g = 0; g < G; g++) {
			const long lo = std::min<long>(g * per, B), hi = std::min<long>(lo + per, B);
			if (hi <= lo) continue;
			socp_ctx *ctx = model::Context(devices[g]);		// created here, in the calling thread, in device order
			pool.push_back(std::thread(f, ctx, lo, hi));
		}
		for (size_t t = 0; t < pool.size(); t++) pool[t].join();
	}
};

static void fail(socp_ctx *ctx, const char *what) {
	std::cerr << std::endl << "socp_b200: " << what << ": " << socp_last_error(ctx) << std::endl;
	exit(1);
}

shooting_batch::shooting_batch(model & model, int numMulti, long batch, int numDevice) : myModel(model) {
	if (numMulti < 1 || numMulti >= SOCP_MAX_NODES || batch < 1 || model.DeviceModelId() < 0) {
		std::cerr << std::endl << "ERROR : shooting_batch needs 1 <= numMulti < " << SOCP_MAX_NODES
		          << ", batch >= 1 and a model with a device implementation" << std::endl;
		exit(1);
	}
	data = new data_struct;
	data->B = batch;
	{
		const int visible = (numDevice == 1) ? 1 : model::DeviceCount();
		data->numDevice = (numDevice <= 0) ? visible : std::min(numDevice, visible);
		if (data->numDevice < 1) data->numDevice = 1;
		const char *dev = getenv("SOCP_DEVICE");
		for (int g = 0; g < data->numDevice; g++) data->devices.push_back(data->numDevice == 1 && dev ? atoi(dev) : g);
	}
	data->dim = model.GetDim();
	data->xtol = 1e-8;						// shooting.cpp:95-101
	data->maxfev = 10000;
	data->stepMin = 1e-12;
	memset(&data->shape, 0, sizeof data->shape);
	data->shape.model_id = model.DeviceModelId();
	data->shape.step_nbr = model.DeviceSteps();
	data->shape.integrator = model.deviceAdaptive ? SOCP_DOPRI5 : SOCP_RK4;
	data->shape.ode_tol = model.odeIntTol;
	const std::vector<real> block = model.DeviceParams();
	data->np = (int)block.size();
	data->mparams.resize((size_t)batch * data->np);
	for (long k = 0; k < batch; k++) std::copy(block.begin(), block.end(), data->mparams.begin() + k * data->np);
	Resize(numMulti);
	data->info.assign(batch, 0); data->nfev.assign(batch, 0); data->calls.assign(batch, 0);
	data->fnorm.assign(batch, 0);
	std::vector<int> fixed(data->dim, model::FIXED);
	SetMode(model::FIXED, fixed);
}

shooting_batch::~shooting_batch() { delete data; }

void shooting_batch::Resize(int numMulti) {
	if (numMulti < 1 || numMulti >= SOCP_MAX_NODES) {
		std::cerr << std::endl << "ERROR : shooting_batch needs 1 <= numMulti < " << SOCP_MAX_NODES << std::endl;
		exit(1);
	}
	data->numMulti = numMulti;
	data->shape.num_multi = numMulti;
	const size_t nodes = numMulti + 1;
	data->time.assign(data->B * nodes, 0); data->timed = data->time; data->time_prec = data->time;
	data->X.assign(data->B * nodes * data->dim, 0); data->Xd = data->X; data->X_prec = data->X;
}

long shooting_batch::GetBatch() const { return data->B; }
int shooting_batch::GetNumDevice() const { return data->numDevice; }
int shooting_batch::GetNumParam() const { return data->numParam; }

void shooting_batch::SetMode(int const& mode_tf, std::vector<int> const& mode_Xf) {
	const int M = data->numMulti;
	std::vector<int> mode_t(M + 1, model::CONTINUOUS);
	std::vector< std::vector<int> > mode_X(M + 1, std::vector<int>(data->dim, model::CONTINUOUS));
	mode_t[0] = model::FIXED;
	mode_X[0].assign(data->dim, model::FIXED);
	mode_t[M] = mode_tf;
	mode_X[M] = mode_Xf;
	SetMode(mode_t, mode_X);
}

void shooting_batch::SetMode(std::vector<int> const& mode_t, std::vector< std::vector<int> > const& mode_X) {
	for (int j = 0; j <= data->numMulti; j++) {
		data->shape.mode_t[j] = mode_t[j];
		for (int k = 0; k < data->dim; k++) data->shape.mode_X[j][k] = mode_X[j][k];
	}
	data->numParam = socp_num_param(&data->shape);
	data->param.assign((size_t)data->B * data->numParam, 0);
}

void shooting_batch::SetModelParameters(long k, std::vector<real> const& block) {
	std::copy(block.begin(), block.begin() + data->np, data->mparams.begin() + k * data->np);
}

std::vector<real> shooting_batch::GetModelParameters(long k) const {
	return std::vector<real>(data->mparams.begin() + k * data->np, data->mparams.begin() + (k + 1) * data->np);
}

void shooting_batch::InitShooting(std::vector<real> const& ti, std::vector<model::mstate> const& Xi,
                                  std::vector<real> const& tf, std::vector<model::mstate> const& Xf) {
	const long B = data->B;
	const int n = data->dim, N = 2 * n, P = data->numParam, np = data->np;
	const size_t nodes = data->numMulti + 1;
	std::vector<real> X0((size_t)B * N), XM((size_t)B * n), sw((size_t)B * 2);
	// the switching times model::ComputeTraj integrates with (model.cpp:105-106)
	const std::vector<real> & st = myModel.deviceSwitchingTimes;
	const real sw0 = st.size() >= 2 ? st[0] : 0.0227, sw1 = st.size() >= 2 ? st[1] : 0.08;
	for (long k = 0; k < B; k++) {
		std::copy(Xi[k].begin(), Xi[k].begin() + N, X0.begin() + k * N);
		std::copy(Xf[k].begin(), Xf[k].begin() + n, XM.begin() + k * n);
		sw[2 * k] = sw0; sw[2 * k + 1] = sw1;
	}
	data_struct *d = data;
	data->for_each_block([&, d](socp_ctx *ctx, long lo, long hi) {
		if (socp_init_shooting_batch(ctx, &d->shape, hi - lo, d->mparams.data() + lo * np, sw.data() + 2 * lo, ti.data() + lo,
		                             X0.data() + lo * N, tf.data() + lo, XM.data() + lo * n, d->time.data() + lo * nodes,
		                             d->X.data() + lo * nodes * n, d->param.data() + lo * P, SOCP_HOST) != SOCP_OK)
			fail(ctx, "socp_init_shooting_batch");
	});
	data->timed = data->time;
	data->time_prec = data->time;
	data->Xd = data->X;
	data->X_prec = data->X;
}

void shooting_batch::InitShooting(long k, std::vector<real> const& vt, std::vector<model::mstate> const& vX) {
	const int M = data->numMulti, n = data->dim, N = 2 * n, P = data->numParam, nodes = M + 1;
	for (int i = 0; i <= M; i++) {
		data->time[k * nodes + i] = data->timed[k * nodes + i] = data->time_prec[k * nodes + i] = vt[i];
		for (int j = 0; j < n; j++)
			data->X[(k * nodes + i) * n + j] = data->Xd[(k * nodes + i) * n + j] = data->X_prec[(k * nodes + i) * n + j] = vX[i][j];
	}
	for (int i = 0; i < M; i++)
		for (int j = 0; j < N; j++) data->param[k * P + N * i + j] = vX[i][j];
	int q = N * M;
	for (int j = 0; j <= M; j++)
		if (data->shape.mode_t[j] == model::FREE) data->param[k * P + q++] = vt[j];
}

void shooting_batch::InitShooting(std::vector< std::vector<real> > const& vt, std::vector< std::vector<model::mstate> > const& vX) {
	for (long k = 0; k < data->B; k++) InitShooting(k, vt[k], vX[k]);
}

void shooting_batch::SetDesiredState(long k, real const& ti, model::mstate const& Xi, real const& tf, model::mstate const& Xf) {
	const int M = data->numMulti, n = data->dim, nodes = M + 1;
	data->timed[k * nodes] = ti;
	data->timed[k * nodes + M] = tf;
	for (int j = 0; j < n; j++) {
		data->Xd[(k * nodes) * n + j] = Xi[j];
		data->Xd[(k * nodes + M) * n + j] = Xf[j];
	}
}

void shooting_batch::SetDesiredState(long k, std::vector<real> const& vt, std::vector<model::mstate> const& vX) {
	const int n = data->dim, nodes = data->numMulti + 1;
	for (size_t i = 0; i < vt.size(); i++) {
		data->timed[k * nodes + i] = vt[i];
		for (int j = 0; j < n; j++) data->Xd[(k * nodes + i) * n + j] = vX[i][j];
	}
}

void shooting_batch::SetPrecision(real const& xtol) { data->xtol = xtol; }
void shooting_batch::SetContinuationMinStep(real const& step) { data->stepMin = step; }

static long count_ok(std::vector<int> const& info) {
	long ok = 0;
	for (size_t k = 0; k < info.size(); k++) ok += (info[k] == 1);
	return ok;
}

long shooting_batch::SolveOCP(real const& continuationStep) {
	const long B = data->B;
	const int P = data->numParam, np = data->np;
	const size_t nodes = data->numMulti + 1, n = data->dim;
	data_struct *d = data;
	if (continuationStep <= 0) {
		// SolveShooting (shooting.cpp:568-595): current data <- desired data, accept iff info == 1
		data->time = data->timed;
		data->X = data->Xd;
		std::vector<real> trial(data->param);
		data->for_each_block([&, d](socp_ctx *ctx, long lo, long hi) {
			if (socp_solve_batch(ctx, &d->shape, hi - lo, d->mparams.data() + lo * np, d->time.data() + lo * nodes,
			                     d->X.data() + lo * nodes * n, trial.data() + lo * P, d->xtol, d->maxfev, d->info.data() + lo,
			                     d->nfev.data() + lo, d->fnorm.data() + lo, SOCP_HOST) != SOCP_OK)
				fail(ctx, "socp_solve_batch");
		});
		for (long k = 0; k < B; k++) {
			data->calls[k] = 1;
			if (data->info[k] == 1) std::copy(trial.begin() + k * P, trial.begin() + (k + 1) * P, data->param.begin() + k * P);
		}
		return count_ok(data->info);
	}
	std::vector<int> calls(2 * B);
	data->for_each_block([&, d](socp_ctx *ctx, long lo, long hi) {
		if (socp_continuation_boundary_batch(ctx, &d->shape, hi - lo, d->mparams.data() + lo * np, d->time_prec.data() + lo * nodes,
		                                     d->X_prec.data() + lo * nodes * n, d->timed.data() + lo * nodes,
		                                     d->Xd.data() + lo * nodes * n, d->param.data() + lo * P, d->xtol, d->maxfev,
		                                     continuationStep, d->stepMin, d->info.data() + lo, calls.data() + 2 * lo,
		                                     SOCP_HOST) != SOCP_OK)
			fail(ctx, "socp_continuation_boundary_batch");
	});
	for (long k = 0; k < B; k++) {
		data->calls[k] = calls[2 * k];
		data->nfev[k] = calls[2 * k + 1];
		if (data->info[k] == 1) {				// the homotopy arrived: desired data become the current and previous data
			std::copy(data->timed.begin() + k * nodes, data->timed.begin() + (k + 1) * nodes, data->time.begin() + k * nodes);
			std::copy(data->Xd.begin() + k * nodes * n, data->Xd.begin() + (k + 1) * nodes * n, data->X.begin() + k * nodes * n);
			std::copy(data->timed.begin() + k * nodes, data->timed.begin() + (k + 1) * nodes, data->time_prec.begin() + k * nodes);
			std::copy(data->Xd.begin() + k * nodes * n, data->Xd.begin() + (k + 1) * nodes * n, data->X_prec.begin() + k * nodes * n);
		}
	}
	return count_ok(data->info);
}

long shooting_batch::SolveOCP(real const& continuationStep, int paramIndex, std::vector<real> const& goal) {
	const long B = data->B;
	const int P = data->numParam, np = data->np;
	const size_t nodes = data->numMulti + 1, n = data->dim;
	data_struct *d = data;
	data->time = data->timed;
	data->X = data->Xd;
	std::vector<int> calls(2 * B);
	data->for_each_block([&, d](socp_ctx *ctx, long lo, long hi) {
		if (socp_continuation_param_batch(ctx, &d->shape, hi - lo, d->mparams.data() + lo * np, d->time.data() + lo * nodes,
		                                  d->X.data() + lo * nodes * n, d->param.data() + lo * P, d->xtol, d->maxfev,
		                                  continuationStep <= 0 ? 1.0 : continuationStep, paramIndex, goal.data() + lo, d->stepMin,
		                                  d->info.data() + lo, calls.data() + 2 * lo, SOCP_HOST) != SOCP_OK)
			fail(ctx, "socp_continuation_param_batch");
	});
	for (long k = 0; k < B; k++) { data->calls[k] = calls[2 * k]; data->nfev[k] = calls[2 * k + 1]; }
	return count_ok(data->info);
}

int shooting_batch::GetInfo(long k) const { return data->info[k]; }

std::vector<int> shooting_batch::GetCallNumber(long k) const {
	std::vector<int> c(2);
	c[0] = data->nfev[k]; c[1] = data->calls[k];
	return c;
}

real shooting_batch::GetResidualNorm(long k) const { return data->fnorm[k]; }

void shooting_batch::GetParameters(long k, std::vector<real> & paramVector) const {
	paramVector.assign(data->param.begin() + k * data->numParam, data->param.begin() + (k + 1) * data->numParam);
}

real shooting_batch::GetParameters(long k, int i) const { return data->param[k * data->numParam + i]; }

void shooting_batch::Move(std::vector<real> const& tf, std::vector<model::mstate> & Xf) const {
	const long B = data->B;
	const int P = data->numParam, np = data->np, N = 2 * data->dim;
	const size_t nodes = data->numMulti + 1;
	std::vector<real> Xq((size_t)B * N);
	const data_struct *d = data;
	data->for_each_block([&, d](socp_ctx *ctx, long lo, long hi) {
		if (socp_move_batch(ctx, &d->shape, hi - lo, d->mparams.data() + lo * np, d->time.data() + lo * nodes,
		                    d->param.data() + lo * P, 1, tf.data() + lo, Xq.data() + lo * N, SOCP_HOST) != SOCP_OK)
			fail(ctx, "socp_move_batch");
	});
	Xf.resize(B);
	for (long k = 0; k < B; k++) Xf[k].assign(Xq.begin() + k * N, Xq.begin() + (k + 1) * N);
}

void shooting_batch::GetSolution(std::vector< std::vector<real> > & vt, std::vector< std::vector<model::mstate> > & vX) const {
	const long B = data->B;
	const int P = data->numParam, np = data->np, N = 2 * data->dim, M = data->numMulti;
	const size_t nodes = M + 1;
	std::vector<real> t((size_t)B * nodes), X((size_t)B * nodes * N);
	const data_struct *d = data;
	data->for_each_block([&, d](socp_ctx *ctx, long lo, long hi) {
		if (socp_solution_batch(ctx, &d->shape, hi - lo, d->mparams.data() + lo * np, d->time.data() + lo * nodes,
		                        d->param.data() + lo * P, t.data() + lo * nodes, X.data() + lo * nodes * N, SOCP_HOST) != SOCP_OK)
			fail(ctx, "socp_solution_batch");
	});
	vt.resize(B);
	vX.resize(B);
	for (long k = 0; k < B; k++) {
		vt[k].assign(t.begin() + k * nodes, t.begin() + (k + 1) * nodes);
		vX[k].resize(nodes);
		for (size_t i = 0; i < nodes; i++) vX[k][i].assign(X.begin() + (k * nodes + i) * N, X.begin() + (k * nodes + i + 1) * N);
	}
}

void shooting_batch::Trace(std::vector<real> & rows, std::vector<int> & nrows) const {
	const long B = data->B;
	const int P = data->numParam, np = data->np, M = data->numMulti;
	const size_t nodes = M + 1;
	const size_t per = (size_t)M * socp_trace_max_rows(data->shape.model_id, data->shape.step_nbr) * socp_trace_width(data->shape.model_id);
	rows.resize(B * per);
	nrows.resize((size_t)B * M);
	const data_struct *d = data;
	data->for_each_block([&, d](socp_ctx *ctx, long lo, long hi) {
		if (socp_solution_trace_batch(ctx, &d->shape, hi - lo, d->mparams.data() + lo * np, d->time.data() + lo * nodes,
		                              d->param.data() + lo * P, rows.data() + lo * per, nrows.data() + lo * M, SOCP_HOST) != SOCP_OK)
			fail(ctx, "socp_solution_trace_batch");
	});
}

void shooting_batch::Trace(long k) const {
	const int P = data->numParam, np = data->np, M = data->numMulti;
	const size_t nodes = M + 1;
	const int R = socp_trace_max_rows(data->shape.model_id, data->shape.step_nbr);
	std::vector<real> rows((size_t)M * R * socp_trace_width(data->shape.model_id));
	std::vector<int> nrows(M);
	socp_ctx *ctx = model::Context(data->devices[0]);
	if (socp_solution_trace_batch(ctx, &data->shape, 1, data->mparams.data() + k * np, data->time.data() + k * nodes,
	                              data->param.data() + k * P, rows.data(), nrows.data(), SOCP_HOST) != SOCP_OK)
		fail(ctx, "socp_solution_trace_batch");
	myModel.AppendTrace(rows.data(), nrows.data(), M, R);
}
