// magprop_constants.hpp -- the physical constants of the reference model, in cgs units (funcs.py:12-18,
// magnetar/funcs.py:7-13).  Apart from magprop_core.cuh, which includes it, the reference restatements of
// magprop_models.cu read it: they need the constants without the disc tables that come with the core.
#pragma once

namespace mp {

constexpr double kG = 6.674e-8;
constexpr double kC = 3.0e10;
constexpr double kR = 1.0e6;
constexpr double kMsol = 1.99e33;
constexpr double kM = 1.4 * kMsol;
constexpr double kGM = kG * kM;
constexpr double kTwoPi = 6.283185307179586476925286766559;

}  // namespace mp
