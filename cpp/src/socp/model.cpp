// cpp/src/socp/model.cpp -- host side of the `model` mirror (reference: src/socp/model.hpp:16-479).
// Every numerical entry point forwards to the device through the C ABI (include/socp_b200.h) with a
// batch of one; there is no host arithmetic of the hot path here and no CPU fallback.
#include <cstdio>
#include <cstdlib>
#include <iostream>
#include <sstream>
#include <map>
#include <mutex>
#include <vector>

#include "model.hpp"
#include "../../../include/socp_b200.h"

namespace {
// one engine context per CUDA device, created on first use
std::mutex g_mutex;
std::map<int, socp_ctx *> g_ctx;
struct ObstacleTable { int n; std::vector<real> type, pos, rad; bool set; ObstacleTable() : n(0), set(false) {} } g_obs;

void die(const char *what, socp_ctx *ctx) {
	std::cerr << std::endl << "socp_b200: " << what << ": " << socp_last_error(ctx) << std::endl;
	exit(1);
}

int default_device() {
	const char *dev = getenv("SOCP_DEVICE");
	return dev ? atoi(dev) : 0;
}
}

socp_ctx *model::Context() { return Context(default_device()); }

socp_ctx *model::Context(int device) {
	std::lock_guard<std::mutex> lock(g_mutex);
	std::map<int, socp_ctx *>::iterator it = g_ctx.find(device);
	if (it != g_ctx.end()) return it->second;
	socp_ctx *ctx = nullptr;
	if (socp_create(device, &ctx) != SOCP_OK) die("socp_create", nullptr);
	if (g_obs.set && socp_set_obstacles(ctx, g_obs.n, g_obs.type.data(), g_obs.pos.data(), g_obs.rad.data()) != SOCP_OK)
		die("socp_set_obstacles", ctx);
	g_ctx[device] = ctx;
	return ctx;
}

int model::DeviceCount() {
	// the engine is the only CUDA user of this library: ask it by creating contexts until one fails would be
	// wasteful, so the count comes from the environment the runtime itself honours, else from a probe
	int n = 0;
	socp_ctx *probe = nullptr;
	while (n < 64) {
		{
			std::lock_guard<std::mutex> lock(g_mutex);
			if (g_ctx.count(n)) { ++n; continue; }
		}
		if (socp_create(n, &probe) != SOCP_OK) break;
		{
			std::lock_guard<std::mutex> lock(g_mutex);
			if (g_obs.set) socp_set_obstacles(probe, g_obs.n, g_obs.type.data(), g_obs.pos.data(), g_obs.rad.data());
			g_ctx[n] = probe;
		}
		++n;
	}
	return n;
}

void model::SetDeviceObstacles(int n, const real *type, const real *pos, const real *rad) {
	std::lock_guard<std::mutex> lock(g_mutex);
	g_obs.n = n; g_obs.set = true;
	g_obs.type.assign(type, type + n); g_obs.pos.assign(pos, pos + 3 * n); g_obs.rad.assign(rad, rad + 3 * n);
	if (g_ctx.empty()) {
		socp_ctx *ctx = nullptr;
		if (socp_create(default_device(), &ctx) != SOCP_OK) die("socp_create", nullptr);
		g_ctx[default_device()] = ctx;
	}
	for (std::map<int, socp_ctx *>::iterator it = g_ctx.begin(); it != g_ctx.end(); ++it)
		if (socp_set_obstacles(it->second, n, type, pos, rad) != SOCP_OK) die("socp_set_obstacles", it->second);
}

model::model(int const& _stateDim, int _modelOrder, int _stepNbr, std::string _fileTrace)
	: dim(_stateDim), modelOrder(_modelOrder), strFileTrace(_fileTrace), stepNbr(_stepNbr), deviceAdaptive(0) {
	// the reference truncates the trace file in the constructor (model.hpp:51-54)
	std::ofstream fileTrace;
	fileTrace.open(strFileTrace.c_str(), std::ios::trunc);
	fileTrace.close();
}

model::~model() {}

// -------------------------------------------------------------------------------------------------
// device plumbing shared by the entry points below
namespace {
struct DevCall {
	socp_ctx *ctx;
	int id;
	std::vector<real> mp;
	real sw[2];
	bool has_sw;
	DevCall(const model &m) : ctx(model::Context()), id(m.DeviceModelId()), mp(m.DeviceParams()), has_sw(false) {
		if (id < 0) {
			std::cerr << std::endl << "ERROR : this model has no device implementation (DeviceModelId() < 0); "
			          << "the B200 engine has no CPU fallback" << std::endl;
			exit(1);
		}
		sw[0] = 0.0227; sw[1] = 0.08;					// goddard.cpp:27-29
		if (m.deviceSwitchingTimes.size() >= 2) { sw[0] = m.deviceSwitchingTimes[0]; sw[1] = m.deviceSwitchingTimes[1]; has_sw = true; }
	}
};
}

model::mstate model::ComputeTraj(real const& t0, mstate const& X0, real const& tf, int isTrace, int isJac) {
	return ModelInt(t0, X0, tf, isTrace, isJac);
}

model::mstate model::ModelInt(real const& t0, mstate const& X, real const& tf, int isTrace, int isJac) {
	DevCall dc(*this);
	const int N = 2 * dim;
	mstate Xs(X);
	if (isJac) {
		// variational integration (state + sensitivities): device kernel for the models that have the
		// equations -- the double integrator, as in the reference (doubleIntegrator.cpp:113-213)
		if ((int)X.size() != (N + 1) * N) { std::cerr << std::endl << "ERROR : isJac = 1 needs a (2n+1)*2n state" << std::endl; exit(1); }
		if (socp_traj_var_batch(dc.ctx, dc.id, DeviceSteps(), 1, dc.mp.data(), &t0, &tf, X.data(), Xs.data(), SOCP_HOST) != SOCP_OK)
			die("socp_traj_var_batch", dc.ctx);
		return Xs;
	}
	std::vector<real> Xin(X.begin(), X.begin() + N), Xout(N);
	if (isTrace) {
		const int W = socp_trace_width(dc.id), R = socp_trace_max_rows(dc.id, DeviceSteps());
		std::vector<real> rows((size_t)W * R);
		int nrows = 0;
		if (socp_trace_batch(dc.ctx, dc.id, DeviceSteps(), 1, dc.mp.data(), dc.sw, &t0, &tf, Xin.data(), rows.data(), &nrows,
		                     Xout.data(), SOCP_HOST) != SOCP_OK)
			die("socp_trace_batch", dc.ctx);
		AppendTrace(rows.data(), &nrows, 1, R);
	} else if (deviceAdaptive) {
		if (socp_traj_adaptive_batch(dc.ctx, dc.id, DeviceSteps(), 1, dc.mp.data(), dc.sw, &t0, &tf, Xin.data(), odeIntTol,
		                             Xout.data(), nullptr, SOCP_HOST) != SOCP_OK)
			die("socp_traj_adaptive_batch", dc.ctx);
	} else {
		if (socp_traj_batch(dc.ctx, dc.id, DeviceSteps(), 1, dc.mp.data(), dc.sw, &t0, &tf, Xin.data(), Xout.data(), SOCP_HOST) != SOCP_OK)
			die("socp_traj_batch", dc.ctx);
	}
	for (int i = 0; i < N; i++) Xs[i] = Xout[i];
	return Xs;
}

// point evaluations: odeTools::Model / model::Control / model::Hamiltonian on the device
model::mstate model::Model(real const& t, mstate const& X, int isJac) const {
	DevCall dc(*this);
	mstate out(2 * dim);
	if (socp_point_batch(dc.ctx, dc.id, 1, dc.mp.data(), dc.sw, nullptr, &t, X.data(), out.data(), nullptr, nullptr, SOCP_HOST) != SOCP_OK)
		die("socp_point_batch", dc.ctx);
	return out;
}

model::mcontrol model::Control(real const& t, mstate const& X) const {
	DevCall dc(*this);
	real u[4] = {0, 0, 0, 0};
	if (socp_point_batch(dc.ctx, dc.id, 1, dc.mp.data(), dc.sw, nullptr, &t, X.data(), nullptr, u, nullptr, SOCP_HOST) != SOCP_OK)
		die("socp_point_batch", dc.ctx);
	const int nc = socp_trace_width(dc.id) - 2 * dim - 3;
	return mcontrol(u, u + nc);
}

model::mstate model::Hamiltonian(real const& t, mstate const& X, int isJac) const {
	DevCall dc(*this);
	real H = 0;
	if (socp_point_batch(dc.ctx, dc.id, 1, dc.mp.data(), dc.sw, nullptr, &t, X.data(), nullptr, nullptr, &H, SOCP_HOST) != SOCP_OK)
		die("socp_point_batch", dc.ctx);
	return mstate(1, H);
}

// -------------------------------------------------------------------------------------------------
// boundary functions, value form (isJac == 0) of model.hpp:90-339.  The shooting residual evaluates
// the same conditions on the device (assemble<MODEL>, socp_b200/csrc/solver.cuh); these serve callers
// that use the model interface directly.
static void fixed_or_transversal(int dim, model::mstate const& Xt, model::mstate const& Xd, std::vector<int> const& mode_X,
                                 std::vector<real> & fvec) {
	for (int j = 0; j < dim; j++)
		fvec[j] = (mode_X[j] == model::FREE) ? Xt[j + dim] : Xt[j] - Xd[j];
}

void model::FinalFunction(real const&, mstate const& X_tf, mstate const& Xf, std::vector<int> const& mode_X, std::vector<real> & fvec, int isJac) const {
	if (isJac) { std::cerr << "ERROR : host boundary functions provide the value form only" << std::endl; exit(1); }
	fixed_or_transversal(dim, X_tf, Xf, mode_X, fvec);
}
void model::FinalHFunction(real const& tf, mstate const& X_tf, mstate const& Xf, std::vector<int> const& mode_X, std::vector<real> & fvec, int isJac) const {
	FinalFunction(tf, X_tf, Xf, mode_X, fvec, isJac);
	fvec[dim] = Hamiltonian(tf, X_tf, 0)[0];
}
void model::InitialFunction(real const&, mstate const& X_t0, mstate const& X0, std::vector<int> const& mode_X, std::vector<real> & fvec, int isJac) const {
	if (isJac) { std::cerr << "ERROR : host boundary functions provide the value form only" << std::endl; exit(1); }
	fixed_or_transversal(dim, X_t0, X0, mode_X, fvec);
}
void model::InitialHFunction(real const& t0, mstate const& X_t0, mstate const& X0, std::vector<int> const& mode_X, std::vector<real> & fvec, int isJac) const {
	InitialFunction(t0, X_t0, X0, mode_X, fvec, isJac);
	fvec[dim] = Hamiltonian(t0, X_t0, 0)[0];
}
model::mstate model::SwitchingTimesFunction(real const& t, mstate const& X, mstate const& Xp, int isJac) const {
	if (isJac) { std::cerr << "ERROR : host boundary functions provide the value form only" << std::endl; exit(1); }
	return mstate(1, Hamiltonian(t, X, 0)[0] - Hamiltonian(t, Xp, 0)[0]);
}
void model::SwitchingTimesUpdate(std::vector<real> const& switchingTimes) { deviceSwitchingTimes = switchingTimes; }

// -------------------------------------------------------------------------------------------------
void model::TraceTail(real H, real, std::ostream & file) const { file << H << std::endl; }

void model::AppendTrace(const real *rows, const int *nrows, int nseg, int R) const {
	// same text as model::Trace (model.hpp:446-462): default ostream precision, tab separated
	const int N = 2 * dim, W = socp_trace_width(DeviceModelId()), nc = W - N - 3;
	std::stringstream ss;
	for (int s = 0; s < nseg; s++)
		for (int r = 0; r < nrows[s]; r++) {
			const real *row = rows + ((size_t)s * R + r) * W;
			ss << row[0] << "\t";
			for (int k = 0; k < N; k++) ss << row[1 + k] << "\t";
			for (int k = 0; k < nc; k++) ss << row[1 + N + k] << "\t";
			TraceTail(row[1 + N + nc], row[2 + N + nc], ss);
		}
	std::ofstream fileTrace;
	fileTrace.open(strFileTrace.c_str(), std::ios::app);
	fileTrace << ss.str();
	fileTrace.close();
}

template <class S> static void trace_point(const model &m, real const& t, model::mstate const& X, S & file) {
	model::mcontrol u = m.Control(t, X);
	real H = m.Hamiltonian(t, X, 0)[0];
	file << t << "\t";
	for (int k = 0; k < 2 * m.dim; k++) file << X[k] << "\t";
	for (size_t k = 0; k < u.size(); k++) file << u[k] << "\t";
	file << H << std::endl;
}
void model::Trace(real const& t, mstate const& X, std::ofstream & file) const { trace_point(*this, t, X, file); }
void model::Trace(real const& t, mstate const& X, std::stringstream & file) const { trace_point(*this, t, X, file); }
