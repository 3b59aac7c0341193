// tempered_rng.cpp -- TEST INFRASTRUCTURE.  Compiles parallel tempering's mover -> row mapping and swap decision
// (magprop_rng.cuh, the functions the kernels call) for the host, so tests/test_tempered.py can pin them against
// the NumPy restatement without a GPU.  Built by that test into a temporary directory; never part of the package.
#include <cmath>

#include "../../magprop_b200/csrc/magprop_rng.cuh"

using namespace mp;

// temperature, row and partner row (for the given partner draws pj) of every mover of half-step `split`
extern "C" void tr_tempered_rows(int n, int ntemps, unsigned long long seed, unsigned long long step, int split,
                                 int randomize, const int* pj, int* t_out, int* row_out, int* partner_out) {
  const SplitPerm p = make_split_perm(n, seed, step, randomize);
  const uint32_t half = (uint32_t)n / 2u;
  for (uint32_t g = 0; g < (uint32_t)ntemps * half; ++g) {
    const TemperedMover m = tempered_mover(p, (uint32_t)split * half, g);
    t_out[g] = (int)m.t;
    row_out[g] = (int)m.row;
    partner_out[g] = (int)tempered_partner(p, (uint32_t)(1 - split) * half, m.t, (uint32_t)pj[g]);
  }
}
extern "C" int tr_pt_swap_accept(unsigned long long seed, unsigned long long step, unsigned row_hot, double beta_cold,
                                 double beta_hot, double lnp_hot, double lnp_cold) {
  return pt_swap_accept(seed, step, row_hot, beta_cold, beta_hot, lnp_hot, lnp_cold) ? 1 : 0;
}
