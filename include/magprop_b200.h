/* magprop_b200.h -- C ABI of the B200-native magprop likelihood hot path.
 *
 * The reference (sgibson91/magprop) is pure Python and has NO FFI boundary; the
 * path it runs per walker is
 *     lnprob  -> lnprior -> lnlike -> model_lum/model_lc -> odeint(ODEs/odes)
 *             -> luminosity stage -> interp1d -> chi-square
 * (code/synthetic_datasets/mcmc_eqns.py:52-81, funcs.py:146-236 and
 *  magnetar/mcmc_eqns.py:87-119, magnetar/funcs.py:105-220).
 * This header is the boundary a maintainer binds with ctypes (INTEGRATION.md
 * shows the stub); every entry point cites the reference interface it replaces.
 *
 * Conventions: plain pointers and sizes, no C++/torch types; all reals are
 * IEEE binary64; row-major; every function returns an mp_status code except
 * where noted; the library never falls back to a CPU implementation -- with no
 * usable CUDA device every compute call returns MP_ERR_CUDA.
 */
#ifndef MAGPROP_B200_H
#define MAGPROP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MP_ABI_VERSION 2
#define MP_MAX_NDIM 9

/* ---- return codes ------------------------------------------------------- */
enum mp_status {
  MP_OK = 0,
  MP_ERR_BAD_ARG = 1,        /* null pointer, negative size, ndim not in 6..9            */
  MP_ERR_DATA_RANGE = 2,     /* a data time lies outside the grid: interp1d raises        */
                             /*   ValueError (funcs.py:233-234, magnetar/funcs.py:214)    */
  MP_ERR_CUDA = 3,           /* CUDA runtime error / no device; mp_last_error() has text  */
  MP_ERR_BAD_GRID = 4,       /* grid not strictly increasing or shorter than 2 nodes      */
  MP_ERR_NO_DATA = 5         /* handle was created without data but a data call was made  */
};

/* ---- per-walker status word (bit field) ---------------------------------- */
#define MP_WALKER_OK 0
#define MP_WALKER_PRIOR_REJECT 1   /* lnprior == -inf (mcmc_eqns.py:43-49)                 */
#define MP_WALKER_INTEGRATOR_FAIL 2 /* step budget / step underflow: the analogue of the   */
                                   /*   reference's 'flag' (funcs.py:172-173) -> -inf      */
#define MP_WALKER_NONFINITE_STATE 4 /* parameters outside the physical domain (NaN state): */
                                   /*   luminosity is 0 as the reference's isfinite clamps */
                                   /*   make it (funcs.py:216-227)                         */
#define MP_WALKER_NONFINITE_LNLIKE 8 /* lnlike was NaN/inf -> -inf (mcmc_eqns.py:72-79)    */

/* ---- model description ----------------------------------------------------
 * One POD covers the reference's divergent copies of the model (script variant
 * code/synthetic_datasets/funcs.py, packaged variant magnetar/funcs.py, figure
 * scripts).  "rhs_*" are the knobs the ODE right-hand side sees, "lum_*" the
 * ones the luminosity stage sees: the packaged model_lc does not forward its
 * kwargs to odeint (magnetar/funcs.py:150-151), so they can differ.          */
typedef struct mp_model_spec {
  double inertia_factor;   /* I = f*M*R^2 : 0.35 (funcs.py:17) | 0.8 (magnetar/funcs.py:12)  */
  double mdot_factor;      /* Rm ~ (f*Mdisc/tvisc)^(-2/7): 3 (funcs.py:105) | 1 (magnetar/funcs.py:64) */
  double rhs_n, rhs_alpha, rhs_cs7, rhs_k;
  double lum_n, lum_alpha, lum_cs7, lum_k;
  double dipeff, propeff, f_beam;  /* defaults; theta[6..8] override per mp_model_spec.ndim rule */
  double breakup_rhs;      /* rot_param > x => Nacc = 0 in the RHS (0.27: funcs.py:131)      */
  double breakup_lum;      /* same test in the luminosity stage: 0.27 (funcs.py:206) | 0.0 (magnetar/funcs.py:193) */
  int32_t lprop_binding_term; /* 1: Lprop = propeff*(-Nacc*w - GM/Rm*eta2*Mdot) (funcs.py:222-223); 0: propeff*(-Nacc*w) (magnetar/funcs.py:206) */
  int32_t unlog_mask;      /* bit i set: theta[i] is log10 and is un-logged before the model (mcmc_eqns.py:17: bits 2..5) */
  double rtol;             /* relative tolerance of the spin integrator (0 => default 1e-10) */
  int32_t max_steps;       /* step budget per walker (0 => default 50000)                   */
  int32_t dipole_torque;   /* RHS dipole torque: 0 classical -mu^2 w^3/(6c^3) (funcs.py:119) | 1 Bucciantini et al. (2006),
                              (-2/3)(mu^2 w^3/c^3)(Rlc/Rm)^3 (figure_3.py:142-143); the luminosity stage keeps the classical Ldip */
} mp_model_spec;

/* Top-hat prior: inclusive bounds, NaN rejects (mcmc_eqns.py:40-49,
 * magnetar/mcmc_eqns.py:62-84 incl. the 7-parameter special case, which the
 * caller resolves when filling lower/upper).  ndim entries are used.         */
typedef struct mp_prior_spec {
  int32_t ndim;
  int32_t enabled;         /* 0: no prior test (model_lum / model_lc calls)                 */
  double lower[MP_MAX_NDIM];
  double upper[MP_MAX_NDIM];
} mp_prior_spec;

typedef struct mp_handle mp_handle;

/* ---- lifetime ------------------------------------------------------------- */
int mp_abi_version(void);
int mp_device_count(void);                 /* number of CUDA devices (0 if none)            */
const char* mp_last_error(void);           /* text of the last error on this thread          */

/* Create a likelihood handle on `device`.
 *   grid[G]          : the model time grid, np.logspace(0|-3, 6, 10001)
 *                      (funcs.py:19, magnetar/funcs.py:132-141) -- passed in so its
 *                      bits are the caller's NumPy bits
 *   t,y,yerr[D]      : the burst data (x,y,yerr of generate_data.py:70 or
 *                      t,Lum50,Lum50err of magnetar/mcmc_eqns.py:17-19); D may be 0
 *                      (t=y=yerr=NULL) for a curves-only handle
 * The handle owns device copies of everything it is given.                      */
int mp_create(const mp_model_spec* spec, const mp_prior_spec* prior,
              const double* grid, int32_t G,
              const double* t, const double* y, const double* yerr, int32_t D,
              int32_t device, mp_handle** out);
void mp_destroy(mp_handle* h);
int mp_set_prior(mp_handle* h, const mp_prior_spec* prior);
/* ---- the hot path ----------------------------------------------------------
 * lnprob for W walkers in one launch: replaces  [lnprob(theta_i, x, y, yerr, fbad)
 * for i in walkers]  (mcmc_eqns.py:52-81; emcee's compute_log_prob with
 * vectorize=True).  theta is [W][ndim] row-major.  lnp[W] receives lnprior+lnlike
 * or -inf (never NaN).  status[W] (may be NULL) receives the MP_WALKER_* bits,
 * n_rhs[W] (may be NULL) the number of right-hand-side evaluations spent.
 * Host-pointer form: copies in, launches, copies out, synchronises.            */
int mp_lnprob_batch(mp_handle* h, const double* theta, int32_t W, int32_t ndim,
                    double* lnp, int32_t* status, int32_t* n_rhs);

/* Device-pointer form: all pointers are device addresses on the handle's device
 * (e.g. torch.Tensor.data_ptr()); enqueues on `stream` (a cudaStream_t, NULL =
 * default stream) and returns without synchronising.                           */
/* The same without the final wait: the copies and launches are queued on the handle's two streams and the
 * call returns; the outputs are valid after mp_synchronize(h).  Lets one host thread keep several handles
 * (independent datasets / bursts, BASELINE configs[2]) in flight at once; the caller's buffers must stay alive
 * and, for the copies to overlap, be pinned.  mp_lnprob_batch == mp_lnprob_batch_async + mp_synchronize.   */
int mp_lnprob_batch_async(mp_handle* h, const double* theta, int32_t W, int32_t ndim,
                          double* lnp, int32_t* status, int32_t* n_rhs);
int mp_synchronize(mp_handle* h);
int mp_lnprob_batch_device(mp_handle* h, const double* d_theta, int32_t W, int32_t ndim,
                           double* d_lnp, int32_t* d_status, int32_t* d_n_rhs,
                           void* stream);

/* Model luminosity at the data times, /1e50: replaces model_lum(pars, xdata=x)
 * (funcs.py:233-236) / model_lc(pars, xdata=x, ...) (magnetar/funcs.py:213-217).
 * pars is [W][ndim] PHYSICAL parameters (no un-logging, no prior); out is [W][D];
 * status[W] may be NULL (MP_WALKER_INTEGRATOR_FAIL <=> the 'flag' return).      */
int mp_model_at_data(mp_handle* h, const double* pars, int32_t W, int32_t ndim,
                     double* out, int32_t* status);

/* Full light curves: replaces model_lum(pars) / model_lc(pars) with xdata=None
 * (funcs.py:230-231, magnetar/funcs.py:219-220).  Every node_stride-th grid node
 * is produced (0, s, 2s, ...; the last grid node is appended if not hit):
 * Gs = mp_curve_nodes(h, node_stride).  out is [W][3][Gs] = Ltot, Lprop, Ldip
 * (/1e50).  state (may be NULL) is [W][2][Gs] = Mdisc, omega at those nodes
 * (the odeint solution of tests/test_funcs.py:28-48).                           */
int32_t mp_curve_nodes(const mp_handle* h, int32_t node_stride);
int mp_model_curves(mp_handle* h, const double* pars, int32_t W, int32_t ndim,
                    int32_t node_stride, double* out, double* state, int32_t* status);
int mp_model_curves_device(mp_handle* h, const double* d_pars, int32_t W, int32_t ndim,
                           int32_t node_stride, double* d_out, double* d_state,
                           int32_t* d_status, void* stream);

/* Right-hand side of the coupled ODEs for a batch of states, computed on the
 * device: replaces ODEs(y,t,B,MdiscI,RdiscI,epsilon,delta,n,alpha,cs7,k)
 * (funcs.py:75-142) / odes(...) (magnetar/funcs.py:33-101).
 * y [W][2], t [W], pars [W][5] = B,MdiscI,RdiscI,epsilon,delta; knobs [4] =
 * n,alpha,cs7,k; dydt [W][2].  Host pointers.                                   */
int mp_rhs_batch(const mp_model_spec* spec, const double* y, const double* t,
                 const double* pars, const double* knobs, int32_t W, double* dydt,
                 int32_t device);

/* One emcee-style stretch-move half-step on the device (synth_mcmc.py:180-185
 * configures emcee's default StretchMove(a=2)): proposes for the Ns walkers of
 * `d_active` (indices into the ensemble) from the complementary set, evaluates
 * lnprob, accepts/rejects in place -- one fused launch.  Counter-based RNG
 * (Philox4x32-10) keyed by seed with counter (step, walker), so any rank can
 * reproduce any walker's draws.  d_accepted[nwalkers] (may be NULL) counts
 * acceptances, d_n_rhs[nwalkers] (may be NULL) receives the RHS evaluations.
 * All pointers are device pointers.                                             */
int mp_stretch_half_step(mp_handle* h, double* d_coords, double* d_lnp, int32_t nwalkers,
                         int32_t ndim, const int32_t* d_active, int32_t n_active,
                         const int32_t* d_complement, int32_t n_complement,
                         double a, uint64_t seed, uint64_t step, int32_t* d_accepted,
                         int32_t* d_n_rhs, void* stream);

/* ---- device-resident ensemble (emcee's RedBlueMove, synth_mcmc.py:180-185) -------------------
 * The ensemble a sampler keeps: positions and log-probabilities on the device, replicated on every
 * rank of a multi-GPU run.  One MCMC step is two half-steps (split = 0, 1).  In half-step `split` the
 * walkers of half `split` are moved against the other half -- which includes the updates the first
 * half-step of the same step made, as in emcee.
 *
 * Which walkers form the halves: position g of the ensemble order holds walker P(g); half 0 is
 * g in [0, n/2), half 1 is g in [n/2, n).  randomize_split = 1 makes P a pseudo-random permutation
 * keyed by (seed, step) -- emcee's `inds = arange(n) % 2; random.shuffle(inds)` re-drawn every step --
 * computed on the fly inside the kernel (a cycle-walking Feistel network), so every rank of a sharded run
 * derives the same split without communication.  randomize_split = 0: P = identity (fixed halves).
 *
 * Sharding: rank r of `world` moves positions [r*m, (r+1)*m) of the active half, m = n/2/world.  A rank's
 * next half-step needs other ranks' moves -- the partners it draws, the current positions of the walkers it
 * is about to move.  Two ways to get them there:
 *   peer reads    peer_coords/peer_lnp hold the other ranks' replicas mapped into this process (mp_peer_open,
 *                 NVLink).  A rank writes the rows it moves into its own replica only; the kernels READ a row
 *                 from the replica of the rank that moved that walker last -- which every rank can work out,
 *                 the ensemble order being a keyed permutation -- so only the ~2m rows a rank actually needs
 *                 cross NVLink per half-step, not the (world-1)*m an all-gather delivers, and no collective is
 *                 launched: the caller runs mp_peer_barrier after each half-step.  A replica is then complete
 *                 only for the rows its rank moved last; mp_ensemble_sync completes it (for reading the chain
 *                 out), and synced_step tells the kernels from which step on the replicas have diverged.
 *   packed rows   pack_out [m][ndim+1] receives every moved walker's (row, lnp) in position order; the
 *                 caller all-gathers the ranks' packs and scatters them with mp_ensemble_unpack (one
 *                 collective per half-step; this is also what the gloo CPU tests drive).
 *
 * status[n] (may be NULL) receives the MP_WALKER_* bits of each walker's latest proposal.  bad_rows /
 * bad_count (may be NULL) log the proposals whose likelihood was not finite -- the rows the reference
 * appends to {GRB}_bad.csv (mcmc_eqns.py:72-79); at most bad_capacity rows are kept, bad_count keeps
 * counting.                                                                                        */
#define MP_MAX_PEERS 15
typedef struct mp_ensemble {
  double* coords;            /* [nwalkers][ndim] */
  double* lnp;               /* [nwalkers]        */
  int32_t nwalkers, ndim;
  double a;                  /* stretch scale (emcee default 2.0) */
  uint64_t seed;
  int32_t randomize_split;
  int32_t rank, world;
  int32_t* accepted;         /* [nwalkers] acceptance counters, or NULL */
  int32_t* status;           /* [nwalkers] or NULL */
  int32_t* n_rhs;            /* [nwalkers] or NULL */
  int32_t n_peers;           /* 0, or world-1: the other ranks' replicas, in rank order without this rank */
  double* peer_coords[MP_MAX_PEERS];
  double* peer_lnp[MP_MAX_PEERS];
  uint64_t synced_step;      /* all replicas held every row when this step began (set_state / mp_ensemble_sync) */
  double* pack_out;          /* [nwalkers/2/world][ndim+1] or NULL */
  double* bad_rows;          /* [bad_capacity][ndim] or NULL */
  int32_t* bad_count;        /* [1] or NULL */
  int32_t bad_capacity;
} mp_ensemble;

/* One half-step for this rank's share of half `split` at MCMC step `step`: proposal, lnprob, accept, in one
 * fused launch (plus the stiff-bucket launch).  Counter-based RNG (Philox4x32-10) keyed by seed with counter
 * (2*step + split, walker): any rank reproduces any walker's draws.  Enqueues on `stream`.             */
int mp_ensemble_half_step(mp_handle* h, const mp_ensemble* ens, uint64_t step, int32_t split, void* stream);
/* Peer-read ensembles: fetch every row another rank moved last into this replica (all ranks call it between two
 * mp_peer_barrier calls, with `step` = the next step to run; afterwards synced_step = step).                  */
int mp_ensemble_sync(const mp_ensemble* ens, uint64_t step, void* stream);
/* Scatter all-gathered packs ([nwalkers/2][ndim+1], position order) of half `split` into coords / lnp.  */
int mp_ensemble_unpack(const mp_ensemble* ens, uint64_t step, int32_t split, const double* d_packed, void* stream);
/* The ensemble order itself: d_order[g] = P(g) for g in [0, nwalkers) (tests, host-side bookkeeping).   */
int mp_ensemble_order(int32_t nwalkers, uint64_t seed, uint64_t step, int32_t randomize_split,
                      int32_t* d_order, void* stream);

/* ---- parallel-tempered ensembles (emcee 2's PTSampler / ptemcee) -------------------------------------
 * ntemps temperatures x n = e->nwalkers walkers per temperature: coords [ntemps][n][ndim], lnp [ntemps][n] and
 * accepted / status / n_rhs [ntemps][n]; row r = t*n + w.  lnp is UNTEMPERED (lnlike + lnprior).  betas is a HOST
 * array of ntemps inverse temperatures: betas[0] == 1, strictly decreasing, all > 0; ntemps <= MP_MAX_TEMPS and
 * ntemps*n < 2^31.  world must be 1, n_peers 0 and pack_out NULL.  Every argument is checked on the host before
 * any device work (MP_ERR_BAD_ARG).
 *
 * mp_tempered_half_step: half-step `split` of every temperature in ONE fused launch.  Each temperature moves as
 *   mp_ensemble_half_step moves one ensemble -- shared split P of (seed, step), partners from the complementary half
 *   of the same temperature, Philox counter (2*step + split, r) -- except that the accept test is
 *   (ndim-1) ln z + beta_t lnp(q) - beta_t lnp(x) > ln u'.  With ntemps = 1 it is mp_ensemble_half_step bit for bit.
 * mp_tempered_swap: once per MCMC step, after half-step 1.  For t = ntemps-1 down to 1 and every column j, walker j
 *   of temperature t swaps its row and lnp with walker j of t-1 iff
 *   ln u < (betas[t-1] - betas[t]) (lnp[t][j] - lnp[t-1][j]),  u from Philox counter (step, t*n + j, word 3).
 *   d_swap_accepted[ntemps-1] (may be NULL) counts the accepted swaps of each adjacent pair (t-1, t).
 *   Runs on the current device.                                                                               */
#define MP_MAX_TEMPS 256
int mp_tempered_half_step(mp_handle* h, const mp_ensemble* e, int32_t ntemps, const double* betas, uint64_t step,
                          int32_t split, void* stream);
int mp_tempered_swap(const mp_ensemble* e, int32_t ntemps, const double* betas, uint64_t step,
                     int32_t* d_swap_accepted, void* stream);

/* ---- emcee 3's moves= (StretchMove, DEMove, DESnookerMove) --------------------------------------------------
 * The half-steps above with a weighted mix of moves; mp_ensemble_half_step and mp_tempered_half_step are these with
 * the one move MP_MOVE_STRETCH of e->a.  Per half-step, with the existing split: mover x is moved against the
 * complement half C, |C| = Nc (in a tempered ensemble, the complement within the mover's own temperature).
 * hs = 2*step + split is the half-step counter, me the mover's row, and idx(u, m) = min((int)(u*m), m-1) the partner
 * rule.  Every move proposes q with the log of its Hastings factor, ln f, and draws its accept uniform ua from
 * Philox4x32-10 blocks keyed by the seed: the stretch move from counter (hs, me, 0) and (hs, me, 1), the others from
 * A = counter (hs, me, 4) and B = counter (hs, me, 5).
 *   MP_MOVE_STRETCH (a; Goodman & Weare 2010): uz = u01(S0,S1), up = u01(S2,S3) of block S = (hs, me, 0),
 *     ua = u01 of words 0,1 of (hs, me, 1).  z = ((a-1)*uz + 1)^2 / a, partner c = C[idx(up, Nc)],
 *     q_c = c_c - (c_c - x_c)*z, ln f = (ndim-1) * log(z).
 *   MP_MOVE_DE (gamma0, sigma; Nelson et al. 2014): uj = u01(A0,A1), uk = u01(A2,A3), ug = u01(B0,B1),
 *     ua = u01(B2,B3).  Partners are an ordered pair of distinct positions: j = idx(uj, Nc), then k = idx(uk, Nc-1),
 *     and k += 1 if k >= j.  g = gamma0 * (1 + s3*(2*ug - 1)) with s3 = sigma*sqrt(3) (host); gamma0 = 0 means
 *     2.38/sqrt(2*ndim).  q_c = x_c + g*(c_j,c - c_k,c), every operation rounded on its own.  ln f = 0.  Unlike
 *     emcee the jitter on gamma is uniform with standard deviation sigma, not Gaussian (no log/cos: positions stay
 *     reproducible bit for bit on the host).
 *   MP_MOVE_DE_SNOOKER (gammas; ter Braak & Vrugt 2008): uz = u01(A0,A1), u1 = u01(A2,A3), u2 = u01(B0,B1),
 *     ua = u01(B2,B3).  Three distinct positions: z = idx(uz, Nc); r1 = idx(u1, Nc-1), moved up past z;
 *     r2 = idx(u2, Nc-2), moved up past z and r1 in ascending order.  e = x - z, ee = sum_c e_c^2,
 *     dd = sum_c (r1_c - r2_c)*e_c (ascending c, rounded term by term); q = x + (gammas*dd/ee)*e;
 *     ln f = (0.5*(ndim-1)) * log(sum_c (q_c - z_c)^2 / ee).  ee == 0: q = x and ln f = 0; a zero numerator gives
 *     ln f = -inf (rejected).
 *   Accept: ((ln f + lq) - lx) > log(ua), lq and lx weighted by beta_t in a tempered ensemble.  Status, bad_rows,
 *     counters and pack_out as described for mp_ensemble.
 *   Which move runs: one per MCMC step, for both half-steps and every temperature.  u = u01 of Philox counter
 *     (step, 0, 6); the move is the first k with u*W < cum_k, W and cum_k the sequential sums of the weights.
 *   MP_MOVE_KDE (gamma0; emcee's KDEMove): a Gaussian kernel-density estimate of the complement, sampled.  Centres:
 *     the complement positions cpos0 + [0, M) in the ensemble order, M = min(Nc, MP_KDE_MAX_CENTRES) -- with a
 *     randomised split a fresh uniform subset every half-step, fixed during it and independent of any mover (emcee
 *     uses every complement walker; the cap bounds the density sums).  mu and Sigma: their mean and covariance
 *     (ddof = 1), every sum in tiles of 64 centres, each tile left to right, then the tile sums left to right;
 *     mu = S / M, Sigma = S2 / (M-1).  Sigma = L L^T by Cholesky in one thread in row order; a pivot <= 0 or not
 *     finite makes every mover of that temperature propose q = x with ln f = -inf (rejected).  Bandwidth h = gamma0,
 *     or Scott's M^(-1/(ndim+4)) (host pow) when gamma0 = 0.  Draws: u_c = u01 of words 0,1 of (hs, me, 8), ua of
 *     its words 2,3; z from Box-Muller pairs of blocks (hs, me, 9 .. 8 + ceil(ndim/2)) with the library's own
 *     ln / sincos (gauss_pair, magprop_rng.cuh), reproducible on the host.  Centre j = idx(u_c, M),
 *     q = c_j + h L z (row r: c_r + h * sum_{k<=r} L_rk z_k, ascending k).  y(p) = L^-1 (p - mu) / h by forward
 *     substitution in ascending rows, r2_j(p) = sum_c (y_c(p) - y_c(c_j))^2 (ascending c),
 *     lk(p) = -0.5 min_j r2_j + log(sum_j exp(-0.5 (r2_j - min_j r2_j))) (ascending j), ln f = lk(x) - lk(q).
 *     One rank only: world 1, no peers, no pack_out.
 * Checked on the host before any device work (MP_ERR_BAD_ARG): moves non-null, 1 <= n_moves <= MP_MAX_MOVES, known
 * kinds, weights finite and >= 0 with a positive sum, stretch a > 1, DE 0 <= sigma < 1 and gamma0 >= 0, snooker
 * gammas > 0, KDE gamma0 finite and >= 0, a half (per temperature) of at least 2 walkers for DE, 3 for snooker and
 * ndim + 1 for KDE when they have weight, and a weighted KDE move on one rank.  Kind 3 is not assigned.            */
#define MP_MOVE_STRETCH 0
#define MP_MOVE_DE 1
#define MP_MOVE_DE_SNOOKER 2
#define MP_MOVE_KDE 4
#define MP_MAX_MOVES 8
#define MP_KDE_MAX_CENTRES 4096
typedef struct mp_move {
  int32_t kind;
  int32_t pad;
  double weight, a, gamma0, sigma, gammas;
} mp_move;
int mp_ensemble_moves_half_step(mp_handle* h, const mp_ensemble* e, const mp_move* moves, int32_t n_moves,
                                uint64_t step, int32_t split, void* stream);
int mp_tempered_moves_half_step(mp_handle* h, const mp_ensemble* e, int32_t ntemps, const double* betas,
                                const mp_move* moves, int32_t n_moves, uint64_t step, int32_t split, void* stream);
/* Sequential Monte Carlo (a half-step at one inverse temperature, the weights and their ESS, systematic resampling)
 * is declared in magprop_smc.h, which includes this header.                                                          */

/* Peer-mappable device memory for the replicas (CUDA IPC; one process per GPU on one node).
 * mp_peer_alloc: cudaMalloc + export a 64-byte handle other processes pass to mp_peer_open, which maps the
 * block into the caller's address space on `device` (NVLink peer access).  mp_peer_barrier: every rank calls
 * it with the same `epoch` after a half-step; it raises flag[rank] = epoch in every peer's flag array and
 * waits until every peer has raised its own in `my_flags` -- after which every rank's writes of the half-step
 * are visible to every other rank's reads.  A peer that does not arrive within ~10 s sets *d_error = 1 instead of hanging.          */
int mp_peer_alloc(int32_t device, uint64_t bytes, void** d_ptr, unsigned char handle[64]);
int mp_peer_open(int32_t device, const unsigned char handle[64], void** d_ptr);
int mp_peer_close(int32_t device, void* d_ptr);
int mp_peer_free(int32_t device, void* d_ptr);
int mp_peer_barrier(int32_t device, uint64_t* d_my_flags, uint64_t* const* peer_flags, int32_t rank,
                    int32_t world, uint64_t epoch, int32_t* d_error, void* stream);

/* ---- posterior summaries of a device-resident chain ---------------------------------------------
 * What the reference's plot_synth.py computes from the chain file (plot_synth.py:150-166) -- pairwise
 * correlation coefficients and the 2.5 / 50 / 97.5 percentiles of every parameter -- as reductions over the chain
 * where the sampler left it.  d_chain is [n][ndim] row-major on `device` (the stored chain, flattened).
 *   mp_chain_moments            column means and the covariance matrix (n-1 normalisation, as np.cov /
 *                               np.corrcoef use); host outputs mean[ndim], cov[ndim][ndim]
 *   mp_chain_order_statistics   the ranks[r]-th smallest value (0-based) of column `col`, exactly (radix select
 *                               on the IEEE bit patterns, 64-bit counts): -0.0 before +0.0, every NaN last (a
 *                               NaN comes back with its sign bit cleared); np.percentile's linear interpolation
 *                               between two neighbouring order statistics is the caller's (it is done AFTER
 *                               un-logging, plot_synth.py:160-166).  Ranks outside [0, n) are MP_ERR_BAD_ARG.
 * Both run on `stream` with stream-ordered allocations and synchronise it before returning.  No floating-point
 * atomics: the blocks' partial sums are added in a fixed order, so two calls on one chain return identical bits on
 * any stream.                                                                                                */
int mp_chain_moments(const double* d_chain, int64_t n, int32_t ndim, double* mean, double* cov,
                     int32_t device, void* stream);
int mp_chain_order_statistics(const double* d_chain, int64_t n, int32_t ndim, int32_t col,
                              const int64_t* ranks, int32_t n_ranks, double* values, int32_t device, void* stream);
/* The order statistics of many columns at once, for credible bands of light curves, are declared in magprop_band.h. */
/* Walker-averaged normalised autocorrelation function of a device-resident chain [n_steps][nwalkers][ndim]
 * (emcee's integrated_time before the window): rows first, first+thin, ...; lags [lag_begin, lag_end) of the
 * n = ceil((n_steps-first)/thin) retained rows; acf is a HOST array [ndim][lag_end-lag_begin].  Synchronises.
 *   acf[d][k-lag_begin] = (1/nwalkers) sum_w C_wd(k) / C_wd(0),   C_wd(k) = sum_{t<n-k} s_t s_{t+k},
 * s_t the series of walker w, dimension d minus its mean, computed directly (no FFT).  The mean is taken after
 * shifting the series by its first retained sample, so an exactly constant series (a stuck walker, or n = 1)
 * has C(0) = 0 and makes acf[d] NaN -- what emcee's formula gives in exact arithmetic.  The sums run in a fixed
 * order (no atomics): two calls on one chain return identical bits on any stream.                           */
int mp_chain_autocorr(const double* d_chain, int64_t n_steps, int32_t nwalkers, int32_t ndim,
                      int64_t first, int64_t thin, int64_t lag_begin, int64_t lag_end,
                      double* acf, int32_t device, void* stream);

/* The comparison model of the reference's figure 5 (code/figure_5.py:222-363, "Ben's model": an accreting-mass
 * magnetar with an exponentially draining disc, explicit Euler steps of 1 s in a Python loop over 1e6 elements).
 * pars [W][6] physical (B, P, MdiscI, RdiscI, epsilon, delta; the last two are not used by this model);
 * knobs [6] = alpha, cs7, k, omass, dipeff, propeff (figure_5.py:12,17-21); step i is at t = 1 + i s; every
 * stride-th step is stored: out [W][3][ceil(n_steps/stride)] = Ltot, Lprop, Ldip (/1e50).  Host pointers.        */
int mp_gompertz_curves(const double* pars, int32_t W, const double* knobs, int64_t n_steps, int32_t stride,
                       double* out, int32_t device);

/* Diagnostic: how many walkers of the most recent launch on this handle were bucketed as stiff
 * and re-run by the implicit (Radau IIA) launch.  Synchronises the device.               */
int mp_last_stiff_count(mp_handle* h, int32_t* count);

/* Diagnostic: how many kernels of the evaluation pipeline (work-list ordering, setup, the two integrator launches,
 * reduce) this handle has launched so far -- what bench.py reports as gpu_launches for its timed region.        */
int64_t mp_kernels_launched(const mp_handle* h);

/* FP64 FMA peak micro-benchmark (roofline denominator; MEASURED_PEAKS.json has
 * no FP64 entry): returns achieved TFLOP/s of dependent-chain-free DFMA.        */
int mp_fp64_peak_tflops(int32_t device, double* tflops);

#ifdef __cplusplus
}
#endif
#endif /* MAGPROP_B200_H */
