// cpp/src/socp/shooting.cpp -- host side of the `shooting` mirror (reference:
// src/socp/shooting.{hpp,cpp}).  Same public API and bookkeeping (tab_param, time/X, time_prec/X_prec,
// timed/Xd, warm starts, continuation with step halving); the root solve itself is one call into the
// device library (socp_solve_batch / socp_solve_hybrj_batch with a batch of one).  For many problems
// at once use shooting_batch (shooting_batch.hpp): same data, leading batch dimension.
#include <cmath>
#include <cstdlib>
#include <algorithm>

#include "shooting.hpp"
#include "../../../include/socp_b200.h"

struct shooting::data_struct {
	int dim, numMulti, numThread, numParam;
	std::vector<real> timed, time, time_prec;			// desired / current / previous node times
	std::vector<model::mstate> Xd, X, X_prec;			// desired / current / previous node states
	std::vector<real> tab_param, tab_param_temp;		// unknowns and their working copy
	std::vector<int> mode_t;
	std::vector< std::vector<int> > mode_X;
	real continuationStepMin, xtol;
	int maxfev, info, nfev, njev;
	real fnorm;
};

static void check_sizes(int numMulti, int numThread) {
	// shooting.cpp:62-77: bad arguments end the program
	const char *msg = 0;
	if (numMulti < 1) msg = "ERROR : numMulti should be superior or equal to 1";
	else if (numThread < 1) msg = "ERROR : numThread should be superior or equal to 1";
	else if (numMulti >= SOCP_MAX_NODES) msg = "ERROR : numMulti exceeds SOCP_MAX_NODES of the device engine";
	if (msg) { std::cerr << std::endl << msg << std::endl; exit(1); }
}

// the device shape of the current modes, with the model's integrator and step count
static socp_shape device_shape(model const& m, int numMulti, std::vector<int> const& mode_t,
                               std::vector< std::vector<int> > const& mode_X) {
	if (m.DeviceModelId() < 0) {
		std::cerr << std::endl << "ERROR : this model has no device implementation; the B200 engine has no CPU fallback" << std::endl;
		exit(1);
	}
	socp_shape shape = socp_shape();
	shape.model_id = m.DeviceModelId();
	shape.integrator = m.deviceAdaptive ? SOCP_DOPRI5 : SOCP_RK4;
	shape.ode_tol = m.odeIntTol;
	shape.num_multi = numMulti;
	shape.step_nbr = m.DeviceSteps();
	for (int j = 0; j <= numMulti; j++) {
		shape.mode_t[j] = mode_t[j];
		for (int k = 0; k < m.GetDim(); k++) shape.mode_X[j][k] = mode_X[j][k];
	}
	return shape;
}

shooting::shooting(model & model, int numMulti, int numThread) : myModel(model) {
	check_sizes(numMulti, numThread);
	data = new data_struct;
	data->dim = myModel.GetDim();
	data->continuationStepMin = 1e-12;				// shooting.cpp:89
	data->maxfev = 10000;							// shooting.cpp:95-101 (epsfcn, mode, factor are fixed inside the engine)
	data->xtol = 1e-8;
	myModel.SetODEIntPrecision(data->xtol);
	data->info = data->nfev = data->njev = 0;
	data->fnorm = 0;
	Resize(numMulti, numThread);
}

shooting::~shooting() { delete data; }

void shooting::Resize(int numMulti, int numThread) const {
	check_sizes(numMulti, numThread);
	data->numMulti = numMulti;
	data->numThread = numThread;					// the batch dimension replaces the reference's thread-per-segment fan-out
	const int nodes = numMulti + 1;
	data->time_prec.resize(nodes); data->time.resize(nodes); data->timed.resize(nodes);
	data->X_prec.resize(nodes); data->X.resize(nodes); data->Xd.resize(nodes);
	data->mode_X.resize(nodes); data->mode_t.resize(nodes);
	data->numParam = 2 * data->dim * numMulti + nodes;		// upper bound until SetMode
	data->tab_param.reserve(data->numParam);
	data->tab_param_temp.reserve(data->numParam);
}

void shooting::SetMode(int const& mode_tf, std::vector<int> const& mode_Xf) const {
	const int M = data->numMulti;
	data->mode_t[0] = model::FIXED;
	data->mode_X[0].assign(data->dim, model::FIXED);
	for (int i = 1; i < M; i++) {
		data->mode_t[i] = model::CONTINUOUS;
		data->mode_X[i].assign(data->dim, model::CONTINUOUS);
	}
	data->mode_t[M] = mode_tf;
	data->mode_X[M] = mode_Xf;
	data->numParam = 2 * data->dim * M + mode_tf;			// as the reference: mode_tf itself is added (shooting.cpp:172)
	data->tab_param.resize(data->numParam);
	data->tab_param_temp.resize(data->numParam);
}

void shooting::SetMode(std::vector<int> const& mode_t, std::vector< std::vector<int> > const& mode_X) const {
	for (int i = 0; i <= data->numMulti; i++) data->mode_X[i] = mode_X[i];
	data->mode_t = mode_t;
	int nfree = 0;
	for (size_t i = 0; i < data->mode_t.size(); i++) if (data->mode_t[i] == model::FREE) nfree++;
	data->numParam = 2 * data->dim * data->numMulti + nfree;
	data->tab_param.resize(data->numParam);
	data->tab_param_temp.resize(data->numParam);
}

// unknowns from the node data: M blocks of (state, costate), then the FREE node times in node order
static void guess_from_nodes(int dim, int M, std::vector<model::mstate> const& X, std::vector<real> const& time,
                             std::vector<int> const& mode_t, std::vector<real> & param) {
	const int N = 2 * dim;
	for (int j = 0; j < M; j++)
		for (int i = 0; i < N; i++) param[j * N + i] = X[j][i];
	int k = N * M;
	for (int j = 0; j <= M; j++)
		if (mode_t[j] == model::FREE) param[k++] = time[j];
}

void shooting::InitShooting(real const& ti, model::mstate const& Xi, real const& tf, model::mstate const& Xf) const {
	const int M = data->numMulti;
	for (int i = 0; i <= M; i++)
		data->time[i] = data->timed[i] = data->time_prec[i] = ti + i * (tf - ti) / M;
	data->X[0] = data->Xd[0] = data->X_prec[0] = Xi;
	for (int i = 1; i < M; i++)					// interior nodes: integrate the guess forward (shooting.cpp:218-222)
		data->X[i] = data->Xd[i] = data->X_prec[i] = Move(ti, Xi, data->time[i]);
	data->X[M] = data->Xd[M] = data->X_prec[M] = Xf;
	guess_from_nodes(data->dim, M, data->X, data->time, data->mode_t, data->tab_param);
}

void shooting::InitShooting(std::vector<real> const& vt, std::vector<model::mstate> const& vX) const {
	const int M = (int)vt.size() - 1;
	data->time_prec = vt; data->time = vt; data->timed = vt;
	data->X_prec = vX; data->X = vX; data->Xd = vX;
	guess_from_nodes(data->dim, M, data->X, data->time, data->mode_t, data->tab_param);
}

void shooting::SetDesiredState(real const& ti, model::mstate const& Xi, real const& tf, model::mstate const& Xf) const {
	data->timed[0] = ti; data->Xd[0] = Xi;
	data->timed[data->numMulti] = tf; data->Xd[data->numMulti] = Xf;
}

void shooting::SetDesiredState(std::vector<real> const& vt, std::vector<model::mstate> const& vX) const {
	for (size_t i = 0; i < vt.size(); i++) { data->timed[i] = vt[i]; data->Xd[i] = vX[i]; }
}

int shooting::SolveOCP(real const& continuationStep) const {
	return (continuationStep <= 0) ? SolveShooting() : SolveShootingContinuation(continuationStep);
}

int shooting::SolveOCP(real const& continuationStep, double const&) const {
	return SolveOCP(continuationStep);
}

int shooting::SolveOCP(real const& continuationStep, real & Rdata, real const& Rgoal) const {
	return SolveShootingContinuation(continuationStep <= 0 ? 1.0 : continuationStep, Rdata, Rgoal);
}

model::mstate shooting::Move(real const& ti, model::mstate const& Xi, real const& tf, int isJac) const {
	return myModel.ComputeTraj(ti, Xi, tf, 0, isJac);
}

void shooting::Move(real const& ti, model::mstate const& Xi, real const& tf, model::mstate & Xf, int isJac) const {
	Xf = myModel.ComputeTraj(ti, Xi, tf, 0, isJac);
}

// state of the current solution at time tf (clamped to the trajectory), shooting.cpp:383-437
model::mstate shooting::Move(real const& tf, int isJac) const {
	const int M = data->numMulti, N = 2 * data->dim;
	std::vector<real> timeLine(M + 1);
	ComputeTimeLine(data->tab_param, timeLine);
	const real t0 = (data->mode_t[0] == model::FIXED) ? data->time[0] : data->tab_param[N * M];
	const real tEnd = (data->mode_t[M] == model::FIXED) ? data->time[M] : data->tab_param[data->numParam - 1];
	const real target = (tf >= t0 && tf <= tEnd) ? tf : tEnd;
	int seg = 0;
	while (timeLine[seg + 1] < target) seg++;
	model::mstate X1 = data->X[0];
	for (int i = 0; i < N; i++) X1[i] = data->tab_param[i];
	if (seg > 0 && seg < M)
		for (int i = 0; i < N; i++) X1[i] = data->tab_param[N * seg + i];
	return Move(timeLine[seg], X1, target, isJac);
}

void shooting::Move(real const& tf, model::mstate & Xf, int) const { Xf = Move(tf); }		// isJac dropped, as shooting.cpp:440-444

void shooting::SetPrecision(real const& xtol) const {
	data->xtol = xtol;
	myModel.SetODEIntPrecision(xtol);
}

void shooting::SetContinuationMinStep(real const& step) const { data->continuationStepMin = step; }

real shooting::GetParameters(int const& k) const { return data->tab_param[k]; }

real *shooting::GetParameters() const {
	real *param = new real[data->numParam];
	std::copy(data->tab_param.begin(), data->tab_param.begin() + data->numParam, param);
	return param;
}

void shooting::GetParameters(std::vector<real> & paramVector) const {
	paramVector.assign(data->tab_param.begin(), data->tab_param.begin() + data->numParam);
}

void shooting::GetSolution(std::vector<real> & vt, std::vector<model::mstate> & vX) const {
	UpdateSolution();
	vt = data->time;
	for (int i = 0; i <= data->numMulti; i++) vX[i] = data->X[i];		// vX must be pre-sized (shooting.cpp:485-487)
}

std::vector<int> shooting::GetCallNumber() const {
	std::vector<int> calls(2);
	calls[0] = data->nfev; calls[1] = data->njev;
	return calls;
}

real shooting::GetResidualNorm() const { return data->fnorm; }

model & shooting::GetModel() const { return myModel; }

// re-integrate every segment with the observer on (shooting.cpp:496-544): one socp_solution_trace_batch of this problem
void shooting::Trace() const {
	const int M = data->numMulti;
	UpdateSolution();					// its ComputeTimeLine leaves the model's switching times as the reference does
	const socp_shape shape = device_shape(myModel, M, data->mode_t, data->mode_X);
	const int R = socp_trace_max_rows(shape.model_id, shape.step_nbr), W = socp_trace_width(shape.model_id);
	std::vector<real> mp = myModel.DeviceParams(), rows((size_t)M * R * W);
	std::vector<int> nrows(M);
	socp_ctx *ctx = model::Context();
	if (socp_solution_trace_batch(ctx, &shape, 1, mp.data(), data->time.data(), data->tab_param.data(), rows.data(),
	                              nrows.data(), SOCP_HOST) != SOCP_OK) {
		std::cerr << std::endl << "socp_b200: socp_solution_trace_batch: " << socp_last_error(ctx) << std::endl;
		exit(1);
	}
	myModel.AppendTrace(rows.data(), nrows.data(), M, R);
}

// ---- solve ----------------------------------------------------------------------------------------
int shooting::SolveShooting() const {
	data->tab_param_temp = data->tab_param;
	for (int i = 0; i <= data->numMulti; i++) {
		data->time[i] = data->timed[i];
		for (int j = 0; j < data->dim; j++) data->X[i][j] = data->Xd[i][j];
	}
	const int ret = SolveShootingFunction(data->numParam, data->tab_param_temp);
	if (ret == 1) data->tab_param = data->tab_param_temp;			// SOCP keeps a solution only if info == 1 (shooting.cpp:588)
	return ret;
}

// homotopy on the boundary data (shooting.cpp:598-692): b in (0,1], halve on failure, stop when b == 1
int shooting::SolveShootingContinuation(real const& continuationStep) const {
	const int M = data->numMulti;
	const real bStep = continuationStep;
	real b = (std::min<real>)(continuationStep, 1.0), b_prec = 0;
	struct { const shooting::data_struct *d; int M; void operator()(real b, shooting::data_struct *dd) const {
		for (int i = 0; i <= M; i++) {
			dd->time[i] = (1 - b) * dd->time_prec[i] + b * dd->timed[i];
			for (int j = 0; j < dd->dim; j++) dd->X[i][j] = (1 - b) * dd->X_prec[i][j] + b * dd->Xd[i][j];
		}
	} } blend = { data, M };
	blend(b, data);
	data->tab_param_temp = data->tab_param;
	int ret = 0;
	for (bool running = true; running; ) {
		ret = SolveShootingFunction(data->numParam, data->tab_param_temp);
		if (ret != 1) {
			if (fabs(b - b_prec) < data->continuationStepMin) running = false;
			b = b_prec + (b - b_prec) / 2;
			data->tab_param_temp = data->tab_param;
			blend(b, data);
		} else if (b == 1) {
			running = false;
		} else {
			b_prec = b;
			b = (std::min<real>)(b + bStep, 1.0);
			data->tab_param = data->tab_param_temp;
			blend(b, data);
		}
	}
	if (ret == 1) {
		data->tab_param = data->tab_param_temp;
		for (int i = 0; i <= M; i++) {
			data->time_prec[i] = data->timed[i];
			for (int j = 0; j < data->dim; j++) data->X_prec[i][j] = data->Xd[i][j];
		}
	}
	return ret;
}

// homotopy on any real datum the model reads (shooting.cpp:695-778)
int shooting::SolveShootingContinuation(real const& continuationStep, real & Rdata, real const& Rgoal) const {
	const real Rstart = Rdata, bStep = continuationStep;
	real b = (std::min<real>)(continuationStep, 1.0), b_prec = 0;
	Rdata = (1 - b) * Rstart + b * Rgoal;
	data->tab_param_temp = data->tab_param;
	for (int i = 0; i <= data->numMulti; i++) {
		data->time[i] = data->timed[i];
		for (int j = 0; j < data->dim; j++) data->X[i][j] = data->Xd[i][j];
	}
	int ret = 0;
	for (bool running = true; running; ) {
		ret = SolveShootingFunction(data->numParam, data->tab_param_temp);
		if (ret != 1) {
			if (fabs(b - b_prec) < data->continuationStepMin) running = false;
			b = b_prec + (b - b_prec) / 2;
			data->tab_param_temp = data->tab_param;
			Rdata = (1 - b) * Rstart + b * Rgoal;
		} else if (b == 1) {
			running = false;
		} else {
			b_prec = b;
			b = (std::min<real>)(b + bStep, 1.0);
			data->tab_param = data->tab_param_temp;
			Rdata = (1 - b) * Rstart + b * Rgoal;
		}
	}
	if (ret == 1) data->tab_param = data->tab_param_temp;
	return ret;
}

// The one call that leaves the host: shooting.cpp:781-856 (hybrd for modelOrder 0, hybrj for 1)
int shooting::SolveShootingFunction(int const & numParam, std::vector<real> & param) const {
	socp_ctx *ctx = model::Context();
	const socp_shape shape = device_shape(myModel, data->numMulti, data->mode_t, data->mode_X);
	if (socp_num_param(&shape) != numParam) {
		std::cerr << std::endl << "ERROR : numParam does not match the modes (SetMode before InitShooting)" << std::endl;
		exit(1);
	}
	std::vector<real> mp = myModel.DeviceParams(), Xb;
	for (int j = 0; j <= data->numMulti; j++)
		Xb.insert(Xb.end(), data->X[j].begin(), data->X[j].begin() + data->dim);
	int rc;
	if (myModel.modelOrder == 0) {
		data->njev = 0;
		rc = socp_solve_batch(ctx, &shape, 1, mp.data(), data->time.data(), Xb.data(), param.data(), data->xtol, data->maxfev,
		                      &data->info, &data->nfev, &data->fnorm, SOCP_HOST);
	} else {
		// analytic Jacobian from the variational integration (hybrj, shooting.cpp:830-851)
		rc = socp_solve_hybrj_batch(ctx, &shape, 1, mp.data(), data->time.data(), Xb.data(), param.data(), data->xtol, data->maxfev,
		                            &data->info, &data->nfev, &data->njev, &data->fnorm, SOCP_HOST);
	}
	if (rc != SOCP_OK && rc != SOCP_ERR_ARG) {
		std::cerr << std::endl << "socp_b200: " << socp_last_error(ctx) << std::endl;
		exit(1);
	}
	// the reference pushes the switching times into the model while it evaluates the residual
	// (shooting.cpp:1615); leave the model in the state the last evaluation would have left it
	std::vector<real> timeLine(data->numMulti + 1);
	ComputeTimeLine(param, timeLine);
	return data->info;
}

// node times from the fixed times and the FREE-time unknowns; CONTINUOUS nodes are interpolated
// between their FIXED/FREE neighbours (shooting.cpp:1579-1617)
void shooting::ComputeTimeLine(std::vector<real> const& param, std::vector<real> & timeLine) const {
	const int M = data->numMulti;
	int k = 2 * data->dim * M, last = 0;
	std::vector<real> switchingTimes;
	for (int j = 0; j <= M; j++) {
		if (data->mode_t[j] == model::CONTINUOUS) continue;
		if (data->mode_t[j] == model::FIXED) timeLine[j] = data->time[j];
		else {
			timeLine[j] = param[k++];
			if (j < M) switchingTimes.push_back(timeLine[j]);
		}
		for (int q = last + 1; q < j; q++)
			timeLine[q] = timeLine[last] + (q - last) * (timeLine[j] - timeLine[last]) / (j - last);
		last = j;
	}
	myModel.SwitchingTimesUpdate(switchingTimes);
}

// node times and states of the current solution into data->time / data->X (shooting.cpp:1462-1508)
void shooting::UpdateSolution() const {
	const int M = data->numMulti, N = 2 * data->dim;
	std::vector<real> timeLine(M + 1);
	ComputeTimeLine(data->tab_param, timeLine);
	const real tEnd = (data->mode_t[M] == model::FIXED) ? data->time[M] : data->tab_param[data->numParam - 1];
	model::mstate X1 = data->X[0];
	for (int i = 0; i < N; i++) X1[i] = data->tab_param[i];
	for (int i = 0; i <= M; i++) {
		data->time[i] = timeLine[i];
		data->X[i] = X1;
		if (i < M - 1)
			for (int j = 0; j < N; j++) X1[j] = data->tab_param[N * (i + 1) + j];
		else
			X1 = Move(tEnd, 0);
	}
}
