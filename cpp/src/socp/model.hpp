// cpp/src/socp/model.hpp -- mirror of the reference's abstract `model` (src/socp/model.hpp:16-479)
// for the B200 engine.  Same public data (dim, modelOrder, parameters, strFileTrace, stepNbr) and
// the same virtual interface; the five shipped models implement it by calling the device through
// the C ABI (include/socp_b200.h).  A model is usable by `shooting` only if it names a device
// implementation (DeviceModelId() >= 0): a host-only RHS cannot run on the GPU, and there is no
// CPU fallback.
#include <fstream>
#include <map>
#include <string>

#include "odeTools.hpp"

#ifndef _MODEL_H_
#define _MODEL_H_

struct socp_ctx;

class model : public odeTools
{
public:
	typedef odeTools::odeVector mstate;
	typedef odeTools::odeVector mcontrol;

	enum {
		FIXED,		///< fixed time or state
		FREE,		///< free time or state
		CONTINUOUS	///< standard continuity conditions (interior points of multiple shooting)
	};

	model(int const& _stateDim, int _modelOrder = 0, int _stepNbr = 10, std::string _fileTrace = std::string(""));
	virtual ~model();

	virtual int GetDim() const {return dim;};

	/// model.hpp:77 -- one shooting segment, integrated on the GPU (socp_traj_batch, batch of 1)
	virtual mstate ComputeTraj(real const& t0, mstate const& X0, real const& tf, int isTrace, int isJac);

	/// Boundary functions (model.hpp:90-339).  The shooting residual evaluates them on the device
	/// (socp_b200/csrc/solver.cuh); these host entry points serve the isJac == 0 form for callers
	/// that use them directly.
	virtual void FinalFunction(real const& tf, mstate const& X_tf, mstate const& Xf, std::vector<int> const& mode_X, std::vector<real> & fvec, int isJac) const;
	virtual void FinalHFunction(real const& tf, mstate const& X_tf, mstate const& Xf, std::vector<int> const& mode_X, std::vector<real> & fvec, int isJac) const;
	virtual void InitialFunction(real const& t0, mstate const& X_t0, mstate const& X0, std::vector<int> const& mode_X, std::vector<real> & fvec, int isJac) const;
	virtual void InitialHFunction(real const& t0, mstate const& X_t0, mstate const& X0, std::vector<int> const& mode_X, std::vector<real> & fvec, int isJac) const;
	virtual mstate SwitchingTimesFunction(real const& t, mstate const& X, mstate const& Xp, int isJac) const;
	virtual void SwitchingStateFunction(real const& t, int const& stateID, mstate const& X, mstate const& Xp, mstate const& Xd, mstate & fvec, int isJac) const {};
	virtual void SwitchingTimesUpdate(std::vector<real> const& switchingTimes);
	virtual void SetODEIntPrecision(real const& xtol) { odeIntTol = xtol; };

	int dim;									///< state dimension
	int modelOrder;								///< 0 if jacobian is not provided, 1 otherwise
	std::map<std::string,real> parameters;		///< parameters for continuation
	std::string strFileTrace;					///< trace file
	int  stepNbr;								///< step number for ModelInt

	/// evaluated on the device (socp_point_batch, batch of 1)
	virtual mstate Model(real const& t, mstate const& X, int isJac = 0) const;
	virtual mcontrol Control(real const& t, mstate const& X) const;
	virtual mstate Hamiltonian(real const& t, mstate const& X, int isJac) const;
	virtual mstate ModelInt(real const& t0, mstate const& X, real const& tf, int isTrace, int isJac);
	virtual void Trace(real const& t, mstate const& X, std::ofstream & file) const;
	virtual void Trace(real const& t, mstate const& X, std::stringstream & file) const;
	virtual int GetMode(real const& t, mstate const& X) const {return 0;};

	// ---- B200 engine hooks (not in the reference) ---------------------------------------------
	/// id of the device implementation (SOCP_GODDARD ...), -1 for a host-only model
	virtual int DeviceModelId() const { return -1; }
	/// current parameter block in the layout of include/socp_b200.h
	virtual std::vector<real> DeviceParams() const { return std::vector<real>(); }
	/// RK4 steps per segment the device should use (the model's own stepNbr)
	virtual int DeviceSteps() const { return stepNbr; }
	/// 0 (default): fixed-step RK4, the reference's default build; 1: adaptive Dormand-Prince with
	/// abs = rel = odeIntTol, the reference's -D_USE_BOOST build (odeTools.cpp:131-134)
	int deviceAdaptive;
	void SetAdaptiveIntegration(bool on) { deviceAdaptive = on ? 1 : 0; }
	/// switching times pushed by shooting::ComputeTimeLine (goddard.cpp:373)
	std::vector<real> deviceSwitchingTimes;
	/// end of a trace row: H, then whatever the model appends (goddard: switching function,
	/// goddard.cpp:337; interceptor: chart id, interceptor.cpp:151); `extra` is the device's last column
	virtual void TraceTail(real H, real extra, std::ostream & file) const;
	/// trace rows in the layout of socp_trace_batch (rows [nseg][R][socp_trace_width], nrows [nseg]) appended to
	/// strFileTrace as model::Trace writes them; ModelInt's trace branch, shooting::Trace and shooting_batch::Trace(k)
	/// all write through it
	void AppendTrace(const real *rows, const int *nrows, int nseg, int R) const;
	static socp_ctx* Context();					///< engine context of the default device (device 0 or $SOCP_DEVICE)
	/// engine context of CUDA device `device` (one context per device, created on first use; thread safe).
	/// The obstacle table set through SetDeviceObstacles is replayed on every context created later.
	static socp_ctx* Context(int device);
	static int DeviceCount();					///< CUDA devices visible to this process
	/// vtolUAV penalty map on every engine context of the process (existing and future ones)
	static void SetDeviceObstacles(int n, const real *type, const real *pos, const real *rad);

private:
	model() {};
};

#endif //_MODEL_H_
