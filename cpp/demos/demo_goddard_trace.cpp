// cpp/demos/demo_goddard_trace.cpp -- shooting::Trace for members of a solved batch.  A batch of perturbed Goddard
// problems (the perturbation of demo_goddard_batch) is solved with KD = 0 (tests/testGoddard.cpp:94).  Two members at
// different batch positions are traced with shooting_batch::Trace(k); the same solutions, loaded into the
// single-problem class with InitShooting(vt, vX), are traced with shooting::Trace(); the rows of the whole-batch
// shooting_batch::Trace(rows, nrows) are written out as well.  The demo exits non-zero unless the three trace files
// of each member are byte-identical.
//   usage: demo_goddard_trace [B=256] [numDevice=1]      (numDevice 0: every visible GPU shares the batch)
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <sstream>
#include <vector>

#include "socp/shooting.hpp"
#include "socp/shooting_batch.hpp"
#include "models/goddard/goddard.hpp"
#include "../../include/socp_b200.h"

static double unit(unsigned long long & s) {		// uniform in [-1, 1]
	s = s * 6364136223846793005ULL + 1442695040888963407ULL;
	return ((double)(s >> 11) / 9007199254740992.0) * 2.0 - 1.0;
}

static std::string slurp(std::string const& path) {
	std::ifstream f(path.c_str(), std::ios::binary);
	std::stringstream ss;
	ss << f.rdbuf();
	return ss.str();
}

// point the model's trace file at `path`, emptied
static void trace_to(model & m, std::string const& path) {
	m.strFileTrace = path;
	std::ofstream f(path.c_str(), std::ios::trunc);
}

int main(int argc, char **argv) {
	const long B = argc > 1 ? atol(argv[1]) : 256;
	const int numDevice = argc > 2 ? atoi(argv[2]) : 1;
	const int M = 6;
	if (B < 2) { std::cerr << "B must be at least 2" << std::endl; return 2; }
	goddard my_goddard("", 10);
	const int dim = my_goddard.GetDim();
	std::vector<int> mode_Xf(dim, model::FREE);
	mode_Xf[0] = mode_Xf[1] = mode_Xf[2] = model::FIXED;

	// reference problem data (tests/testGoddard.cpp:53-76), perturbed for members k > 0
	model::mstate Xi0(2 * dim, 0.1), Xf0(2 * dim, 0.0);
	Xi0[0] = 0.999949994; Xi0[1] = 0.0001; Xi0[2] = 0.01; Xi0[3] = 1e-10; Xi0[4] = 1e-10; Xi0[5] = 1e-10; Xi0[6] = 1.0;
	Xf0[0] = 1.01;
	my_goddard.SetParameterDataName("mu2", 1.0);
	shooting_batch batch(my_goddard, M, B, numDevice);
	batch.SetPrecision(1e-6);
	batch.SetMode(model::FREE, mode_Xf);
	std::vector<real> vti(B, 0.0), vtf(B, 0.1);
	std::vector<model::mstate> vXi(B, Xi0), vXf(B, Xf0);
	unsigned long long seed = 20260002ULL;
	for (long k = 1; k < B; k++) {
		for (int j = 0; j < 3; j++) vXi[k][j] *= 1 + 1e-3 * unit(seed);
		vXi[k][6] *= 1 + 1e-2 * unit(seed);
		vXf[k][0] = 1.01 + 0.002 * unit(seed);
	}
	batch.InitShooting(vti, vXi, vtf, vXf);		// the guess is integrated with KD = 310, the solve uses KD = 0
	for (long k = 0; k < B; k++) {
		std::vector<real> block = batch.GetModelParameters(k);
		block[2] = 0.0;
		batch.SetModelParameters(k, block);
	}
	my_goddard.SetParameterDataName("KD", 0.0);
	const long ok = batch.SolveOCP(0.0);
	printf("batch of %ld problems on %d GPU(s): %ld converged\n", B, batch.GetNumDevice(), ok);

	std::vector< std::vector<real> > vt;
	std::vector< std::vector<model::mstate> > vX;
	batch.GetSolution(vt, vX);
	std::vector<real> rows;
	std::vector<int> nrows;
	batch.Trace(rows, nrows);
	const size_t per = rows.size() / B;
	bool same = true;
	const long members[2] = {1, B - 1};
	for (int m = 0; m < 2; m++) {
		const long k = members[m];
		std::ostringstream tag;
		tag << k;
		trace_to(my_goddard, "trace_batch_" + tag.str() + ".dat");
		batch.Trace(k);
		shooting single(my_goddard, M, 1);
		single.SetMode(model::FREE, mode_Xf);
		single.InitShooting(vt[k], vX[k]);
		trace_to(my_goddard, "trace_single_" + tag.str() + ".dat");
		single.Trace();
		trace_to(my_goddard, "trace_rows_" + tag.str() + ".dat");
		my_goddard.AppendTrace(rows.data() + k * per, nrows.data() + k * M, M, (int)(per / M / socp_trace_width(SOCP_GODDARD)));
		const std::string a = slurp("trace_batch_" + tag.str() + ".dat"), b = slurp("trace_single_" + tag.str() + ".dat"),
		                  c = slurp("trace_rows_" + tag.str() + ".dat");
		const bool eq = !a.empty() && a == b && a == c;
		printf("problem %ld (info %d): %zu bytes of trace, Trace(k), shooting::Trace and Trace(rows, nrows) identical: %s\n",
		       k, batch.GetInfo(k), a.size(), eq ? "yes" : "NO");
		same = same && eq;
	}
	printf("all traces identical: %s\n", same ? "yes" : "NO");
	return same ? 0 : 1;
}
