// magprop_rng.cuh -- counter-based random numbers of the ensemble move: Philox4x32-10 draws, the keyed
// permutation that defines the per-step random halves, and parallel tempering's mover -> row mapping and swap
// decision.  Plain C++ apart from the qualifiers, so the CPU tests can compile it for the host and pin it against
// their NumPy restatement.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define MP_RNG_HD __host__ __device__ inline
#else
#define MP_RNG_HD inline
#endif

namespace mp {

// ---- counter-based RNG: Philox4x32-10 (Salmon et al. 2011) -------------------
struct Philox {
  uint32_t c[4];
};
MP_RNG_HD Philox philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    const uint32_t n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    const uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += W0; k1 += W1;
  }
  Philox o;
  o.c[0] = c0; o.c[1] = c1; o.c[2] = c2; o.c[3] = c3;
  return o;
}
// 53-bit uniform in (0,1): never 0 so log() is finite
MP_RNG_HD double u01(uint32_t hi, uint32_t lo) {
  const uint64_t v = (((uint64_t)hi << 32) | lo) >> 11;
  return ((double)v + 0.5) * (1.0 / 9007199254740992.0);
}

// ---- the ensemble order: a keyed pseudo-random permutation of [0, n) -----------------------------
// emcee's RedBlueMove re-draws the two halves every step (`inds = arange(n) % 2; random.shuffle(inds)`,
// SURVEY.md appendix C).  Here position g of the ensemble order holds walker P(g) and the halves are
// g < n/2 and g >= n/2; P is a balanced Feistel network on 2*hb bits (4^hb >= n) walked until it lands
// inside [0, n) -- a bijection any thread of any rank evaluates for one index in a few dozen integer
// instructions, so the split needs no index arrays, no sort and no communication.  Keys: one Philox block
// of (seed, step).  randomize = 0: P = identity (fixed halves).
struct SplitPerm {
  uint32_t n, k0, k1, mask;
  int hb, randomize;
};
MP_RNG_HD uint32_t mix32(uint32_t x) {   // an avalanching 32-bit hash ("lowbias32")
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  return x;
}
MP_RNG_HD uint32_t perm_at(const SplitPerm& p, uint32_t g) {
  if (!p.randomize) return g;
  uint32_t x = g;
  do {
    uint32_t L = x >> p.hb, R = x & p.mask;
    for (uint32_t r = 0; r < 6u; ++r) {
      const uint32_t F = mix32((R + r * 0x9E3779B9u) ^ ((r & 1u) ? p.k1 : p.k0)) & p.mask;
      const uint32_t nL = R;
      R = L ^ F;
      L = nL;
    }
    x = (L << p.hb) | R;
  } while (x >= p.n);
  return x;
}
// The inverse: at which position of the ensemble order walker w sits.  (Cycle-walking is symmetric: undo the
// rounds, and walk on while the result is outside [0, n).)
MP_RNG_HD uint32_t perm_inv(const SplitPerm& p, uint32_t w) {
  if (!p.randomize) return w;
  uint32_t x = w;
  do {
    uint32_t L = x >> p.hb, R = x & p.mask;
    for (int r = 5; r >= 0; --r) {
      const uint32_t F = mix32((L + (uint32_t)r * 0x9E3779B9u) ^ ((r & 1) ? p.k1 : p.k0)) & p.mask;
      const uint32_t pR = L;
      L = R ^ F;
      R = pR;
    }
    x = (L << p.hb) | R;
  } while (x >= p.n);
  return x;
}

inline SplitPerm make_split_perm(int n, uint64_t seed, uint64_t step, int randomize) {
  SplitPerm p;
  p.n = (uint32_t)n;
  p.randomize = randomize ? 1 : 0;
  p.hb = 1;
  while ((1ull << (2 * p.hb)) < (unsigned long long)n) ++p.hb;
  p.mask = (1u << p.hb) - 1u;
  const Philox k = philox4x32_10((uint32_t)step, (uint32_t)(step >> 32), 0u, 2u, (uint32_t)seed, (uint32_t)(seed >> 32));
  p.k0 = k.c[0];
  p.k1 = k.c[1];
  return p;
}

// ---- parallel tempering: T temperatures x n walkers, row r = t*n + w -----------------------------------
// Every temperature is one ensemble moved as above, all sharing the split P of the step.  Mover g of a tempered
// half-step is the (g mod n/2)-th mover of temperature g / (n/2); its partner is drawn from the same temperature.
struct TemperedMover {
  uint32_t t, row;
};
MP_RNG_HD TemperedMover tempered_mover(const SplitPerm& p, uint32_t pos0, uint32_t g) {
  const uint32_t half = p.n / 2u;
  TemperedMover m;
  m.t = g / half;
  m.row = m.t * p.n + perm_at(p, pos0 + (g - m.t * half));
  return m;
}
MP_RNG_HD uint32_t tempered_partner(const SplitPerm& p, uint32_t cpos0, uint32_t t, uint32_t pj) {
  return t * p.n + perm_at(p, cpos0 + pj);
}
// The replica exchange of column j between temperature t (row_hot = t*n + j) and t-1, at MCMC step `step`:
// swap iff ln u < (beta_{t-1} - beta_t) (lnp_hot - lnp_cold), u from Philox counter (step, row_hot, 3) -- word 3
// is used by no other draw.  lnp is untempered; a NaN (both -inf) rejects.
MP_RNG_HD bool pt_swap_accept(uint64_t seed, uint64_t step, uint32_t row_hot, double beta_cold, double beta_hot,
                              double lnp_hot, double lnp_cold) {
  const Philox r = philox4x32_10((uint32_t)step, (uint32_t)(step >> 32), row_hot, 3u, (uint32_t)seed, (uint32_t)(seed >> 32));
  return log(u01(r.c[0], r.c[1])) < (beta_cold - beta_hot) * (lnp_hot - lnp_cold);
}

// ---- the differential-evolution moves (mp_ensemble_moves_half_step) -------------------------------------
// The partner rule of every move: position min(floor(u m), m-1) of m.
MP_RNG_HD uint32_t pick_index(double u, uint32_t m) {
  const uint32_t i = (uint32_t)(u * m);
  return i < m ? i : m - 1u;
}
// The four uniforms of a DE or snooker mover: Philox blocks A = counter (hs, me, 4) and B = (hs, me, 5); u[0] from
// A0,A1, u[1] from A2,A3, u[2] from B0,B1, u[3] from B2,B3 (the accept draw).  Words 0-3 stay the stretch move's.
struct MoveDraws {
  double u[4];
};
MP_RNG_HD MoveDraws move_draws(uint64_t seed, uint64_t hs, uint32_t me) {
  const Philox a = philox4x32_10((uint32_t)hs, (uint32_t)(hs >> 32), me, 4u, (uint32_t)seed, (uint32_t)(seed >> 32));
  const Philox b = philox4x32_10((uint32_t)hs, (uint32_t)(hs >> 32), me, 5u, (uint32_t)seed, (uint32_t)(seed >> 32));
  MoveDraws d;
  d.u[0] = u01(a.c[0], a.c[1]);
  d.u[1] = u01(a.c[2], a.c[3]);
  d.u[2] = u01(b.c[0], b.c[1]);
  d.u[3] = u01(b.c[2], b.c[3]);
  return d;
}
// The accept draw u of mover `me` (row) at half-step hs, ln u compared with ln f + lp(q) - lp(s): the stretch move's
// (kind 0) from Philox counter (hs, me, 1), words 0-1; DE's and snooker's from block B of move_draws, = u[3]; the KDE
// move's (kind 4, MP_MOVE_KDE) from words 2-3 of counter (hs, me, 8).
MP_RNG_HD double accept_uniform(int kind, uint64_t seed, uint64_t hs, uint32_t me) {
  const Philox r = philox4x32_10((uint32_t)hs, (uint32_t)(hs >> 32), me, kind == 0 ? 1u : (kind == 4 ? 8u : 5u),
                                 (uint32_t)seed, (uint32_t)(seed >> 32));
  return kind == 0 ? u01(r.c[0], r.c[1]) : u01(r.c[2], r.c[3]);
}
// DE: an ordered pair of distinct positions of the complement (nc >= 2).
MP_RNG_HD void de_pair(double uj, double uk, uint32_t nc, uint32_t* j, uint32_t* k) {
  *j = pick_index(uj, nc);
  *k = pick_index(uk, nc - 1u);
  if (*k >= *j) *k += 1u;
}
// Snooker: three distinct positions z, r1, r2 of the complement (nc >= 3), each uniform over the positions left.
MP_RNG_HD void snooker_triple(double uz, double u1, double u2, uint32_t nc, uint32_t* z, uint32_t* r1, uint32_t* r2) {
  *z = pick_index(uz, nc);
  *r1 = pick_index(u1, nc - 1u);
  if (*r1 >= *z) *r1 += 1u;
  const uint32_t lo = *z < *r1 ? *z : *r1, hi = *z < *r1 ? *r1 : *z;
  *r2 = pick_index(u2, nc - 2u);
  if (*r2 >= lo) *r2 += 1u;
  if (*r2 >= hi) *r2 += 1u;
}
// Which of n moves MCMC step `step` runs (one move per step, as emcee picks one per iteration): u from Philox counter
// (step, 0, word 6); the first k with u W < cum_k, W and cum_k the sequential sums of the weights.  (Should rounding
// leave no such k, the last move of positive weight.)
MP_RNG_HD int choose_move(uint64_t seed, uint64_t step, const double* weights, int n) {
  const Philox r = philox4x32_10((uint32_t)step, (uint32_t)(step >> 32), 0u, 6u, (uint32_t)seed, (uint32_t)(seed >> 32));
  const double u = u01(r.c[0], r.c[1]);
  double W = 0.0;
  for (int k = 0; k < n; ++k) W += weights[k];
  const double uw = u * W;
  double cum = 0.0;
  int last = 0;
  for (int k = 0; k < n; ++k) {
    cum += weights[k];
    if (weights[k] > 0.0) last = k;
    if (uw < cum) return k;
  }
  return last;
}

// ---- the kernel-density move: Gaussians that the host reproduces bit for bit -----------------------------------
// libdevice's log / sincos and libm's differ in the last bit, so the KDE proposal uses its own, built from exact IEEE
// operations only (the library is compiled with -fmad=false; a host build needs -ffp-contract=off).
// ln x for a positive normal x: x = 2^e m with m in [sqrt(1/2), sqrt(2)] (bit manipulation), s = (m - 1)/(m + 1),
// ln m = 2 atanh s by its series to s^23 (|s| <= 0.172), ln x = e ln2_hi + (e ln2_lo + ln m); ln2_hi has 32 bits, so
// e ln2_hi is exact.
MP_RNG_HD double kde_log(double x) {
  uint64_t b;
  memcpy(&b, &x, sizeof(b));
  int e = (int)((b >> 52) & 0x7ffu) - 1023;
  b = (b & 0x000FFFFFFFFFFFFFull) | 0x3FF0000000000000ull;
  double m;
  memcpy(&m, &b, sizeof(m));
  if (m > 1.4142135623730951) {
    m = m * 0.5;
    e += 1;
  }
  const double s = (m - 1.0) / (m + 1.0);
  const double s2 = s * s;
  double p = 1.0 / 23.0;
  p = p * s2 + 1.0 / 21.0;
  p = p * s2 + 1.0 / 19.0;
  p = p * s2 + 1.0 / 17.0;
  p = p * s2 + 1.0 / 15.0;
  p = p * s2 + 1.0 / 13.0;
  p = p * s2 + 1.0 / 11.0;
  p = p * s2 + 1.0 / 9.0;
  p = p * s2 + 1.0 / 7.0;
  p = p * s2 + 1.0 / 5.0;
  p = p * s2 + 1.0 / 3.0;
  p = p * s2 + 1.0;
  const double ln2_hi = 6.93147180369123816490e-01, ln2_lo = 1.90821492927058770002e-10;
  return (double)e * ln2_hi + ((double)e * ln2_lo + (2.0 * s) * p);
}
// sin and cos of x in [0, pi/4]: Taylor polynomials to x^19 and x^20 in Horner form.
MP_RNG_HD void kde_sincos_poly(double x, double* s, double* c) {
  const double x2 = x * x;
  double p = -8.22063524662433e-18;
  p = p * x2 + 2.8114572543455206e-15;
  p = p * x2 + -7.647163731819816e-13;
  p = p * x2 + 1.6059043836821613e-10;
  p = p * x2 + -2.505210838544172e-08;
  p = p * x2 + 2.7557319223985893e-06;
  p = p * x2 + -0.0001984126984126984;
  p = p * x2 + 0.008333333333333333;
  p = p * x2 + -0.16666666666666666;
  *s = x + x * (x2 * p);
  double q = 4.110317623312165e-19;
  q = q * x2 + -1.5619206968586225e-16;
  q = q * x2 + 4.779477332387385e-14;
  q = q * x2 + -1.1470745597729725e-11;
  q = q * x2 + 2.08767569878681e-09;
  q = q * x2 + -2.755731922398589e-07;
  q = q * x2 + 2.48015873015873e-05;
  q = q * x2 + -0.001388888888888889;
  q = q * x2 + 0.041666666666666664;
  q = q * x2 + -0.5;
  *c = 1.0 + x2 * q;
}
// One Box-Muller pair: z = sqrt(-2 ln u1) (cos 2 pi u2, sin 2 pi u2), u1, u2 in (0, 1).  The quadrant is the integer
// part of 4 u2 (exact), f its fraction (exact); the angle f pi/2 is reflected to (1 - f) pi/2 (exact) when f > 1/2,
// so the polynomials see [0, pi/4] only.
MP_RNG_HD void gauss_pair(double u1, double u2, double* z0, double* z1) {
  const double r = sqrt(-2.0 * kde_log(u1));
  const double t = 4.0 * u2;
  const int quad = (int)t;
  const double f = t - (double)quad;
  const bool refl = f > 0.5;
  double s, c;
  kde_sincos_poly((refl ? 1.0 - f : f) * 1.5707963267948966, &s, &c);
  if (refl) {
    const double tmp = s;
    s = c;
    c = tmp;
  }
  // (c, s) = (cos, sin) of f pi/2; turn by quad quarter turns
  double C = c, S = s;
  if (quad == 1) { C = -s; S = c; }
  else if (quad == 2) { C = -c; S = -s; }
  else if (quad == 3) { C = s; S = -c; }
  *z0 = r * C;
  *z1 = r * S;
}
// The KDE mover's draws: u_c (which centre) from words 0,1 of Philox counter (hs, me, 8) -- words 2,3 are its accept
// uniform -- and ndim standard normals, pair k from counter (hs, me, 9 + k), u1 = u01(words 0,1), u2 = u01(words 2,3).
// Words 8 to 13 are used by no other draw.
MP_RNG_HD double kde_centre_uniform(uint64_t seed, uint64_t hs, uint32_t me) {
  const Philox r = philox4x32_10((uint32_t)hs, (uint32_t)(hs >> 32), me, 8u, (uint32_t)seed, (uint32_t)(seed >> 32));
  return u01(r.c[0], r.c[1]);
}
MP_RNG_HD void kde_gaussians(uint64_t seed, uint64_t hs, uint32_t me, int ndim, double* z) {
  for (int k = 0; 2 * k < ndim; ++k) {
    const Philox r = philox4x32_10((uint32_t)hs, (uint32_t)(hs >> 32), me, 9u + (uint32_t)k, (uint32_t)seed,
                                   (uint32_t)(seed >> 32));
    double a, b;
    gauss_pair(u01(r.c[0], r.c[1]), u01(r.c[2], r.c[3]), &a, &b);
    z[2 * k] = a;
    if (2 * k + 1 < ndim) z[2 * k + 1] = b;
  }
}

// ---- sequential Monte Carlo (mp_smc_resample) ---------------------------------------------------------------
// The one uniform of SMC stage `stage`'s systematic resampling: u01 of words 0,1 of Philox counter (stage, 0, 7).
// Word 7 is used by no other draw (stretch 0/1, permutation key 2, swap 3, DE/snooker 4/5, move choice 6).
MP_RNG_HD double smc_stage_uniform(uint64_t seed, uint64_t stage) {
  const Philox r = philox4x32_10((uint32_t)stage, (uint32_t)(stage >> 32), 0u, 7u, (uint32_t)seed, (uint32_t)(seed >> 32));
  return u01(r.c[0], r.c[1]);
}

}  // namespace mp
