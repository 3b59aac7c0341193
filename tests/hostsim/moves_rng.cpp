// moves_rng.cpp -- TEST INFRASTRUCTURE.  Compiles the differential-evolution moves' draws, partner picks and move
// choice (magprop_rng.cuh, the functions the kernels and the entry points call) for the host, so tests/test_moves.py
// can pin them against the NumPy restatement without a GPU.  Built by that test into a temporary directory; never
// part of the package.
#include <cmath>

#include "../../magprop_b200/csrc/magprop_rng.cuh"

using namespace mp;

extern "C" void mr_move_draws(unsigned long long seed, unsigned long long hs, unsigned me, double* u4) {
  const MoveDraws d = move_draws(seed, hs, me);
  for (int k = 0; k < 4; ++k) u4[k] = d.u[k];
}
extern "C" void mr_de_pair(double uj, double uk, unsigned nc, unsigned* jk) { de_pair(uj, uk, nc, jk, jk + 1); }
extern "C" void mr_snooker_triple(double uz, double u1, double u2, unsigned nc, unsigned* zr) {
  snooker_triple(uz, u1, u2, nc, zr, zr + 1, zr + 2);
}
extern "C" int mr_choose_move(unsigned long long seed, unsigned long long step, const double* weights, int n) {
  return choose_move(seed, step, weights, n);
}
