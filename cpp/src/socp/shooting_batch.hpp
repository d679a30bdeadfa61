// cpp/src/socp/shooting_batch.hpp -- the batch driver the reference does not have: B independent
// shooting problems that share one model type and one mode layout, solved together on the GPU.
// Same vocabulary and semantics as `shooting` (shooting.hpp), with a leading problem index:
// Resize / SetMode / InitShooting / SetDesiredState / SolveOCP / GetParameters, Move / GetSolution to
// sample the solutions and re-mesh them, and Trace.  One call of SolveOCP is one socp_solve_batch (or one batched
// continuation) over all B problems; one Move, GetSolution or Trace is one socp_move_batch / socp_solution_batch /
// socp_solution_trace_batch.
#include <vector>

#include "model.hpp"

#ifndef _SHOOTING_BATCH_H_
#define _SHOOTING_BATCH_H_

class shooting_batch
{
public:
	/// numDevice GPUs share the batch (contiguous blocks, one host thread + one engine context per device,
	/// no communication during the solve) -- the batch analogue of the reference's `numThread` constructor
	/// argument (shooting.hpp ctor, shooting.cpp:1133).  numDevice <= 0: every visible device.
	shooting_batch(model & model, int numMulti, long batch, int numDevice = 1);
	~shooting_batch();

	long GetBatch() const;
	int GetNumDevice() const;
	int GetNumParam() const;

	/// shooting::Resize(numMulti) for every problem: the node arrays take the new size (their contents are
	/// reset) and, as in the reference, SetMode must follow before InitShooting
	void Resize(int numMulti);

	void SetMode(int const& mode_tf, std::vector<int> const& mode_Xf);
	void SetMode(std::vector<int> const& mode_t, std::vector< std::vector<int> > const& mode_X);

	/// model parameter block of problem k (layout of include/socp_b200.h); every problem starts with
	/// the model's current parameters
	void SetModelParameters(long k, std::vector<real> const& block);
	std::vector<real> GetModelParameters(long k) const;

	/// shooting::InitShooting(ti, Xi, tf, Xf) for every problem: uniform time grid, interior nodes by
	/// integrating the guess forward (one batched trajectory call per interior node)
	void InitShooting(std::vector<real> const& ti, std::vector<model::mstate> const& Xi,
	                  std::vector<real> const& tf, std::vector<model::mstate> const& Xf);
	/// shooting::InitShooting(vt, vX) for problem k
	void InitShooting(long k, std::vector<real> const& vt, std::vector<model::mstate> const& vX);
	/// shooting::InitShooting(vt, vX) for every problem: vt[k] has M+1 node times, vX[k] M+1 node states
	void InitShooting(std::vector< std::vector<real> > const& vt, std::vector< std::vector<model::mstate> > const& vX);
	void SetDesiredState(long k, real const& ti, model::mstate const& Xi, real const& tf, model::mstate const& Xf);
	void SetDesiredState(long k, std::vector<real> const& vt, std::vector<model::mstate> const& vX);

	void SetPrecision(real const& xtol);
	void SetContinuationMinStep(real const& step);

	/// shooting::SolveOCP(continuationStep) for every problem; returns the number of problems with
	/// info == 1.  continuationStep <= 0: plain solve towards the desired data; > 0: homotopy on the
	/// boundary data from the previous solution (shooting.cpp:598-692), every problem with its own b.
	long SolveOCP(real const& continuationStep);
	/// shooting::SolveOCP(continuationStep, Rdata, Rgoal) on entry paramIndex of the parameter blocks
	long SolveOCP(real const& continuationStep, int paramIndex, std::vector<real> const& goal);

	int GetInfo(long k) const;
	std::vector<int> GetCallNumber(long k) const;			///< {nfev of the last solve (total over a continuation), solver calls}
	real GetResidualNorm(long k) const;
	void GetParameters(long k, std::vector<real> & paramVector) const;
	real GetParameters(long k, int i) const;

	/// shooting::Move(tf) for every problem: Xf[k] = state of solution k at tf[k] (a time outside [t0, t_end] gives
	/// the state at t_end)
	void Move(std::vector<real> const& tf, std::vector<model::mstate> & Xf) const;
	/// shooting::GetSolution for every problem: vt[k] = the M+1 node times, vX[k] = the node states, vX[k][M] = Move(t_end)
	void GetSolution(std::vector< std::vector<real> > & vt, std::vector< std::vector<model::mstate> > & vX) const;
	/// shooting::Trace for every problem: every segment re-integrated with the observer on, in the layout of
	/// socp_solution_trace_batch -- rows [B][M][R][W] (R = socp_trace_max_rows, W = socp_trace_width), nrows [B][M]
	void Trace(std::vector<real> & rows, std::vector<int> & nrows) const;
	/// shooting::Trace of problem k: its rows appended to the model's trace file, the text shooting::Trace writes
	void Trace(long k) const;

private:
	model & myModel;
	struct data_struct;
	data_struct *data;
};

#endif //_SHOOTING_BATCH_H_
