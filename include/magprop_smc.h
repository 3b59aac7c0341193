/* magprop_smc.h -- C ABI of sequential Monte Carlo on the device (adaptive tempering from the prior to the posterior,
 * with the evidence).  An extension of magprop_b200.h: same conventions, same library (libmagprop_b200.so), same
 * return codes; MP_ABI_VERSION covers both headers.
 *
 * One SMC stage of N particles (coords [N][ndim], lnp [N] = lnlike + lnprior, untempered) at inverse temperature beta:
 *   1. mp_smc_weights   incremental weights w_i = exp(dbeta (lnp_i - max lnp)) of a step beta -> beta + dbeta; the
 *                       driver bisects dbeta on the host with d_w = NULL until the ESS S1^2 / S2 meets its target,
 *                       then calls once more with d_w to keep the weights.  ln Z grows by dbeta m + ln(S1 / N).
 *   2. mp_smc_resample  systematic resampling of the particles by those weights, into separate buffers.
 *   3. mp_annealed_moves_half_step, split 0 and 1, a few MCMC steps at the new beta.
 */
#ifndef MAGPROP_SMC_H
#define MAGPROP_SMC_H

#include "magprop_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- sequential Monte Carlo: weights, resampling, a half-step at one beta ------------------------------------
 * mp_smc_weights: d_lnp [n] on `device`.  m = the largest finite lnp; w_i = exp(dbeta * (lnp_i - m)) for a finite
 *   lnp_i and 0 for -inf or any other non-finite entry; out (HOST [3]) = {m, S1 = sum w_i, S2 = sum w_i^2}.  d_w [n]
 *   (may be NULL) receives the weights.  Two passes: the max, then the sums; every block of the sum pass writes its
 *   partial sums and one block adds them in block order -- no floating-point atomics, so repeated calls return
 *   identical bits on any stream.  No finite entry: m = -inf, S1 = S2 = 0 and MP_OK (the caller decides).  n >= 1 and
 *   dbeta finite and >= 0, else MP_ERR_BAD_ARG before any device work.  Runs on `stream` and synchronises it.
 * mp_smc_resample: systematic resampling of n particles by the weights d_w [n] (finite, >= 0: mp_smc_weights').
 *   cum is the inclusive prefix sum of w in this order: w is cut into consecutive tiles of MP_SMC_TILE elements
 *   (the last one may be shorter); p_j is the running sum of w within j's tile, left to right from the tile's first
 *   element; base_0 = 0 and base_{k+1} = base_k + (tile k's last p), left to right over the tiles; cum_j = base_k + p_j
 *   for j in tile k, and total = cum_{n-1} (= base of the tile past the last).  u = u01 of words 0,1 of Philox4x32-10
 *   counter (stage, 0, 7) keyed by the seed (word 7 is used by no move).  Particle i takes ancestor a_i = the smallest
 *   j with cum_j > (i + u) * (total / n), and the last j with w_j > 0 if that is larger or no j qualifies (a rounded
 *   target can reach total): a particle of weight 0 is never chosen.  coords_out[i] = coords_in[a_i],
 *   lnp_out[i] = lnp_in[a_i], d_ancestors[i] = a_i (d_ancestors may be NULL).  total == 0, which the host cannot see,
 *   gives a_i = i.  Checked before any device work (MP_ERR_BAD_ARG): null pointers, n < 1, ndim outside
 *   1..MP_MAX_NDIM, and an output range that overlaps an input range or another output.  Stream-ordered (its work
 *   space is allocated on `stream`); does not synchronise.
 * mp_annealed_moves_half_step: mp_tempered_moves_half_step with the one-entry ladder {beta}, 0 < beta <= 1 (so beta
 *   need not be 1): the movers accept on beta * lnp.  The ensemble runs on one rank (world 1, no peers, no pack_out),
 *   ndim in 1..MP_MAX_NDIM, moves as for mp_ensemble_moves_half_step; every argument is checked on the host before any
 *   device work (MP_ERR_BAD_ARG; a NaN beta fails).  At beta == 1 it equals mp_ensemble_moves_half_step bit for bit.  */
#define MP_SMC_TILE 64
int mp_smc_weights(const double* d_lnp, int64_t n, double dbeta, double* d_w, double* out, int32_t device, void* stream);
int mp_smc_resample(const double* d_w, int64_t n, int32_t ndim, uint64_t seed, uint64_t stage,
                    const double* d_coords_in, const double* d_lnp_in, double* d_coords_out, double* d_lnp_out,
                    int64_t* d_ancestors, int32_t device, void* stream);
int mp_annealed_moves_half_step(mp_handle* h, const mp_ensemble* e, double beta, const mp_move* moves, int32_t n_moves,
                                uint64_t step, int32_t split, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MAGPROP_SMC_H */
