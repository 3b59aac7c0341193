// magprop_rng.cuh -- counter-based random numbers of the ensemble move: Philox4x32-10 draws, the keyed
// permutation that defines the per-step random halves, and parallel tempering's mover -> row mapping and swap
// decision.  Plain C++ apart from the qualifiers, so the CPU tests can compile it for the host and pin it against
// their NumPy restatement.
#pragma once
#include <math.h>
#include <stdint.h>

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
// (kind 0) from Philox counter (hs, me, 1), words 0-1; DE's and snooker's from block B of move_draws, = u[3].
MP_RNG_HD double accept_uniform(int kind, uint64_t seed, uint64_t hs, uint32_t me) {
  const Philox r = philox4x32_10((uint32_t)hs, (uint32_t)(hs >> 32), me, kind == 0 ? 1u : 5u, (uint32_t)seed,
                                 (uint32_t)(seed >> 32));
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

// ---- sequential Monte Carlo (mp_smc_resample) ---------------------------------------------------------------
// The one uniform of SMC stage `stage`'s systematic resampling: u01 of words 0,1 of Philox counter (stage, 0, 7).
// Word 7 is used by no other draw (stretch 0/1, permutation key 2, swap 3, DE/snooker 4/5, move choice 6).
MP_RNG_HD double smc_stage_uniform(uint64_t seed, uint64_t stage) {
  const Philox r = philox4x32_10((uint32_t)stage, (uint32_t)(stage >> 32), 0u, 7u, (uint32_t)seed, (uint32_t)(seed >> 32));
  return u01(r.c[0], r.c[1]);
}

}  // namespace mp
