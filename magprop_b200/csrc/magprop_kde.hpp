// magprop_kde.hpp -- the kernel-density move's two launches (magprop_kde.cu), as the ensemble half-step
// (magprop_kernels.cu) calls them.  Host only, internal.  Semantics: MP_MOVE_KDE in include/magprop_b200.h.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "magprop_abi.hpp"
#include "magprop_rng.cuh"

namespace mp {

// One half-step's KDE move over T temperatures of n walkers (T = 1 without a ladder): the movers are the tempered_mover
// rows of positions pos0 + [0, n/2), the centres of temperature t the rows t*n + P(cpos0 + [0, M)).
struct KdeMove {
  const double* coords;   // [T*n][ndim]
  SplitPerm perm;
  int pos0, cpos0, T, n, ndim, M;
  double h;               // the bandwidth factor
  uint64_t seed, hs;      // hs: the half-step counter
  double* stats;          // [T][kKdeStats] work space: mu, L, the ok flag
  double* white;          // [T][M][ndim] work space: the whitened centres y(c_j)
};
constexpr int kKdeStats = 96;       // mu at 0, the ok flag at 9, L (row-major 9 x 9) at 12

// Once per half-step, before the slab loop: every temperature's mu, L, ok flag and whitened centres.
int kde_prepare(const KdeMove& k, cudaStream_t stream);
// Per slab: q and ln f of movers mover0 + [0, count) into prop[0, count) and lnf[0, count).
int kde_propose(const KdeMove& k, int mover0, int count, double* prop, double* lnf, cudaStream_t stream);

}  // namespace mp
