// smc_rng.cpp -- TEST INFRASTRUCTURE.  Compiles the SMC stage uniform (smc_stage_uniform in magprop_rng.cuh, the
// function mp_smc_resample calls) for the host, so tests/test_smc.py can pin it against the NumPy restatement without
// a GPU.  Built by that test into a temporary directory; never part of the package.
#include <cmath>

#include "../../magprop_b200/csrc/magprop_rng.cuh"

using namespace mp;

extern "C" double sr_stage_uniform(unsigned long long seed, unsigned long long stage) {
  return smc_stage_uniform(seed, stage);
}
