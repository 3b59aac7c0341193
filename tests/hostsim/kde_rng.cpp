// kde_rng.cpp -- TEST INFRASTRUCTURE.  Compiles the KDE move's draws (gauss_pair, kde_centre_uniform, kde_gaussians
// and accept_uniform of magprop_rng.cuh, the functions magprop_kde.cu and the accept step call) for the host, so
// tests/test_kde.py can pin them against the NumPy restatement without a GPU.  Built by that test with
// -ffp-contract=off (the library is built with -fmad=false) into a temporary directory; never part of the package.
#include <cmath>

#include "../../magprop_b200/csrc/magprop_rng.cuh"

using namespace mp;

extern "C" void kr_gauss_pair(const double* u1, const double* u2, long n, double* z0, double* z1) {
  for (long i = 0; i < n; ++i) gauss_pair(u1[i], u2[i], z0 + i, z1 + i);
}
// Rows me0 .. me0 + n - 1 of half-step hs: u_c [n], z [n][ndim], the KDE accept uniform [n].
extern "C" void kr_draws(unsigned long long seed, unsigned long long hs, unsigned me0, long n, int ndim, double* uc,
                         double* z, double* ua) {
  for (long i = 0; i < n; ++i) {
    const uint32_t me = me0 + (uint32_t)i;
    uc[i] = kde_centre_uniform(seed, hs, me);
    kde_gaussians(seed, hs, me, ndim, z + i * ndim);
    ua[i] = accept_uniform(4, seed, hs, me);
  }
}
