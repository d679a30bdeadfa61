// cpp/demos/demo_goddard_pipeline.cpp -- the reference's whole Goddard pipeline (tests/testGoddard.cpp:28-156) on a
// batch of perturbed instances (the perturbation of demo_goddard_batch):
//   1. KD = 0 solve;   2. continuation KD -> 310;   3. continuation mu2 1 -> 0.2;
//   4. the true singular arc: GetSolution, new node times [0, s1/2, s1, (s1+s2)/2, s2, (s2+tf)/2, tf] around the
//      switching times s1 = 0.0227, s2 = 0.08, Move at those times, SetMode with two FREE interior times,
//      InitShooting(vt, vX), mu2 = 0 and singularControl = -1, solve.
// Problem 0 is the unperturbed reference problem; it also runs the four stages alone through `shooting`, and the
// demo reports whether the batch member is bit for bit the single-problem result after every stage.
//   usage: demo_goddard_pipeline [B=256] [numDevice=1]      (numDevice 0: every visible GPU shares the batch)
#include <cstdio>
#include <cstdlib>
#include <iostream>
#include <vector>

#include "socp/shooting.hpp"
#include "socp/shooting_batch.hpp"
#include "models/goddard/goddard.hpp"

static double unit(unsigned long long & s) {		// uniform in [-1, 1]
	s = s * 6364136223846793005ULL + 1442695040888963407ULL;
	return ((double)(s >> 11) / 9007199254740992.0) * 2.0 - 1.0;
}

// the re-meshed node times of stage 4 (tests/testGoddard.cpp:115-130)
static std::vector<real> stage4_times(real tf) {
	const real s1 = 0.0227, s2 = 0.08;
	real t[] = {0.0, s1 / 2, s1, (s2 + s1) / 2, s2, (s2 + tf) / 2, tf};
	return std::vector<real>(t, t + 7);
}

static bool same_as_single(shooting_batch const& batch, shooting const& single, int info1, int P) {
	bool same = (info1 == batch.GetInfo(0)) && P == batch.GetNumParam();
	for (int i = 0; same && i < P; i++) same = single.GetParameters(i) == batch.GetParameters(0, i);
	return same;
}

int main(int argc, char **argv) {
	const long B = argc > 1 ? atol(argv[1]) : 256;
	const int numDevice = argc > 2 ? atoi(argv[2]) : 1;
	const int M = 6;
	goddard my_goddard("", 10);
	const int dim = my_goddard.GetDim();
	std::vector<int> mode_Xf(dim, model::FREE);
	mode_Xf[0] = mode_Xf[1] = mode_Xf[2] = model::FIXED;
	// stage 4 modes (tests/testGoddard.cpp:132-140)
	std::vector<int> mode_t4(M + 1, model::CONTINUOUS);
	mode_t4[0] = model::FIXED; mode_t4[2] = mode_t4[4] = mode_t4[6] = model::FREE;
	std::vector< std::vector<int> > mode_X4(M + 1, std::vector<int>(dim, model::CONTINUOUS));
	mode_X4[0].assign(dim, model::FIXED);
	mode_X4[M] = mode_Xf;

	// reference problem data (tests/testGoddard.cpp:53-76)
	model::mstate Xi0(2 * dim, 0.1), Xf0(2 * dim, 0.0);
	Xi0[0] = 0.999949994; Xi0[1] = 0.0001; Xi0[2] = 0.01; Xi0[3] = 1e-10; Xi0[4] = 1e-10; Xi0[5] = 1e-10; Xi0[6] = 1.0;
	Xf0[0] = 1.01;
	const real ti = 0, tf = 0.1;

	// the guess for the interior nodes is integrated with the constructor's KD = 310; the solve uses KD = 0
	my_goddard.SetParameterDataName("mu2", 1.0);
	shooting_batch batch(my_goddard, M, B, numDevice);
	printf("batch of %ld problems on %d GPU(s)\n", B, batch.GetNumDevice());
	batch.SetPrecision(1e-6);
	batch.SetMode(model::FREE, mode_Xf);
	std::vector<real> vti(B, ti), vtf(B, tf);
	std::vector<model::mstate> vXi(B, Xi0), vXf(B, Xf0);
	unsigned long long seed = 20260002ULL;
	for (long k = 1; k < B; k++) {
		for (int j = 0; j < 3; j++) vXi[k][j] *= 1 + 1e-3 * unit(seed);
		vXi[k][6] *= 1 + 1e-2 * unit(seed);
		vXf[k][0] = 1.01 + 0.002 * unit(seed);
	}
	batch.InitShooting(vti, vXi, vtf, vXf);
	shooting single(my_goddard, M, 1);
	single.SetPrecision(1e-6);
	single.SetMode(model::FREE, mode_Xf);
	single.InitShooting(ti, Xi0, tf, Xf0);
	for (long k = 0; k < B; k++) {
		std::vector<real> block = batch.GetModelParameters(k);
		block[2] = 0.0;									// KD = 0
		batch.SetModelParameters(k, block);
	}
	my_goddard.SetParameterDataName("KD", 0.0);
	bool same = true;
	int info1;

	// stage 1: KD = 0
	long ok = batch.SolveOCP(0.0);
	info1 = single.SolveOCP(0.0);
	same = same_as_single(batch, single, info1, 2 * dim * M + 1) && same;
	printf("stage 1 (KD = 0): %ld of %ld converged, member 0 identical: %s\n", ok, B, same ? "yes" : "NO");

	// stage 2: continuation KD -> 310 (tests/testGoddard.cpp:105)
	ok = batch.SolveOCP(1.0, 2, std::vector<real>(B, 310.0));
	info1 = single.SolveOCP(1.0, my_goddard.GetParameterDataName("KD"), 310.0);
	same = same_as_single(batch, single, info1, 2 * dim * M + 1) && same;
	printf("stage 2 (KD -> 310): %ld of %ld converged, member 0 identical: %s\n", ok, B, same ? "yes" : "NO");

	// stage 3: continuation mu2 1 -> 0.2 (tests/testGoddard.cpp:110)
	ok = batch.SolveOCP(1.0, 6, std::vector<real>(B, 0.2));
	info1 = single.SolveOCP(1.0, my_goddard.GetParameterDataName("mu2"), 0.2);
	same = same_as_single(batch, single, info1, 2 * dim * M + 1) && same;
	printf("stage 3 (mu2 -> 0.2): %ld of %ld converged, member 0 identical: %s\n", ok, B, same ? "yes" : "NO");

	// stage 4: re-mesh on the switching times, then the true singular control (tests/testGoddard.cpp:115-156)
	std::vector< std::vector<real> > vt, vt4(B);
	std::vector< std::vector<model::mstate> > vX, vX4(B, std::vector<model::mstate>(M + 1));
	batch.GetSolution(vt, vX);
	for (long k = 0; k < B; k++) vt4[k] = stage4_times(vt[k][M]);
	for (int i = 0; i <= M; i++) {
		std::vector<real> tq(B);
		std::vector<model::mstate> Xq;
		for (long k = 0; k < B; k++) tq[k] = vt4[k][i];
		batch.Move(tq, Xq);
		for (long k = 0; k < B; k++) vX4[k][i] = Xq[k];
	}
	batch.SetMode(mode_t4, mode_X4);
	batch.InitShooting(vt4, vX4);
	for (long k = 0; k < B; k++) {
		std::vector<real> block = batch.GetModelParameters(k);
		block[6] = 0.0;									// mu2 = 0
		block[7] = -1.0;								// singularControl = -1
		batch.SetModelParameters(k, block);
	}
	ok = batch.SolveOCP(0.0);

	std::vector<real> vt1(M + 1);
	std::vector<model::mstate> vX1(M + 1);
	single.GetSolution(vt1, vX1);
	bool same_remesh = vt1 == vt[0];
	std::vector<real> vt41 = stage4_times(vt1[M]);
	std::vector<model::mstate> vX41(M + 1);
	for (int i = 0; i <= M; i++) {
		vX41[i] = single.Move(vt41[i]);
		same_remesh = same_remesh && vX41[i] == vX4[0][i];
	}
	single.SetMode(mode_t4, mode_X4);
	single.InitShooting(vt41, vX41);
	my_goddard.SetParameterDataName("mu2", 0.0);
	my_goddard.SetParameterDataName("singularControl", -1.0);
	info1 = single.SolveOCP(0.0);
	same = same_remesh && same_as_single(batch, single, info1, 2 * dim * M + 3) && same;
	printf("stage 4 (re-mesh, singular arc): %ld of %ld converged, re-mesh of member 0 identical: %s, member 0 identical: %s\n",
	       ok, B, same_remesh ? "yes" : "NO", same ? "yes" : "NO");
	printf("problem 0 stage 4: info %d nfev %d tf %.17g\n", batch.GetInfo(0), batch.GetCallNumber(0)[0],
	       batch.GetParameters(0, 2 * dim * M + 2));
	printf("single    stage 4: info %d nfev %d tf %.17g\n", info1, single.GetCallNumber()[0], single.GetParameters(2 * dim * M + 2));
	printf("batch member 0 identical to the single run: %s\n", same ? "yes" : "NO");
	return same ? 0 : 1;
}
