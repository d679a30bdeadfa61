// cpp/demos/demo_init_shooting.cpp -- shooting_batch::InitShooting(ti, Xi, tf, Xf) gives every member of a batch the
// initial guess that shooting::InitShooting(ti, Xi, tf, Xf) gives the same problem alone: the same integrator and the
// same switching times as model::ComputeTraj.  Two cases:
//   goddard   RK4, mu2 = 0 with switching times set on the model (0.03, 0.07): the thrust of every interior node
//             integration depends on them
//   di        the double integrator with the adaptive Dormand-Prince integrator (SOCP_DOPRI5)
// Prints "<case>: <k> of <B> members identical to shooting::InitShooting" per case; exit status 0 iff all are.
//   usage: demo_init_shooting [B=64]
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "socp/shooting.hpp"
#include "socp/shooting_batch.hpp"
#include "models/goddard/goddard.hpp"
#include "models/doubleIntegrator/doubleIntegrator.hpp"

static double unit(unsigned long long & s) {		// uniform in [-1, 1]
	s = s * 6364136223846793005ULL + 1442695040888963407ULL;
	return ((double)(s >> 11) / 9007199254740992.0) * 2.0 - 1.0;
}

// InitShooting of B perturbed copies of (ti, Xi, tf, Xf), batched and one by one; returns the members that match
static long compare(const char *name, model & m, int M, long B, real ti, model::mstate const& Xi, real tf,
                    model::mstate const& Xf, int mode_tf, unsigned long long seed) {
	const int dim = m.GetDim();
	std::vector<int> mode_Xf(dim, model::FIXED);
	shooting single(m, M, 1);
	single.SetMode(mode_tf, mode_Xf);
	shooting_batch batch(m, M, B);
	batch.SetMode(mode_tf, mode_Xf);
	std::vector<real> vti(B), vtf(B);
	std::vector<model::mstate> vXi(B, Xi), vXf(B, Xf);
	for (long k = 0; k < B; k++) {
		vti[k] = ti + (k ? 1e-3 * (tf - ti) * unit(seed) : 0.0);
		vtf[k] = tf * (1 + (k ? 1e-2 * unit(seed) : 0.0));
		for (int j = 0; j < 2 * dim; j++) vXi[k][j] *= 1 + (k ? 1e-3 * unit(seed) : 0.0);
		for (int j = 0; j < dim; j++) vXf[k][j] *= 1 + (k ? 1e-3 * unit(seed) : 0.0);
	}
	batch.InitShooting(vti, vXi, vtf, vXf);
	long same = 0;
	std::vector<real> p;
	for (long k = 0; k < B; k++) {
		single.InitShooting(vti[k], vXi[k], vtf[k], vXf[k]);
		batch.GetParameters(k, p);
		bool eq = (int)p.size() == batch.GetNumParam();
		for (int i = 0; eq && i < batch.GetNumParam(); i++) eq = single.GetParameters(i) == p[i];
		same += eq;
	}
	printf("%s: %ld of %ld members identical to shooting::InitShooting\n", name, same, B);
	return same;
}

int main(int argc, char **argv) {
	const long B = argc > 1 ? atol(argv[1]) : 64;
	bool ok = true;
	{
		// tests/testGoddard.cpp:53-76 with mu2 = 0: thrust 1 up to the first switching time, 0.5 up to the second
		goddard g("", 10);
		const int dim = g.GetDim();
		model::mstate Xi(2 * dim, 0.1), Xf(2 * dim, 0.0);
		Xi[0] = 0.999949994; Xi[1] = 0.0001; Xi[2] = 0.01; Xi[3] = 1e-10; Xi[4] = 1e-10; Xi[5] = 1e-10; Xi[6] = 1.0;
		Xf[0] = 1.01;
		g.SetParameterDataName("mu2", 0.0);
		g.SetParameterDataName("singularControl", 0.5);
		g.SwitchingTimesUpdate(std::vector<real>{0.03, 0.07});
		ok = compare("goddard", g, 6, B, 0.0, Xi, 0.1, Xf, model::FREE, 20261022ULL) == B && ok;
	}
	{
		// tests/testDoubleIntegrator.cpp:25-40, four segments, adaptive integration
		doubleIntegrator di(0, "");
		const int dim = di.GetDim();
		di.SetAdaptiveIntegration(true);
		model::mstate Xi(2 * dim), Xf(2 * dim, 0.0);
		for (int i = 0; i < dim; i++) { Xi[i] = 0; Xi[dim + i] = 0.01; }
		Xf[0] = 10; Xf[1] = 15;
		ok = compare("di", di, 4, B, 0.0, Xi, 10.0, Xf, model::FREE, 20261023ULL) == B && ok;
	}
	return ok ? 0 : 1;
}
