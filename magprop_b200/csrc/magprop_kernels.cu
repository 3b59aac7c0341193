// magprop_kernels.cu -- the evaluation pipeline: its sm_100a kernels, the likelihood handle and every entry point of
// include/magprop_b200.h that launches the pipeline.
//
// FP64 throughout, no tensor cores -- the path is a scalar ODE solve per walker, not a contraction.
// One likelihood evaluation runs as a short pipeline of launches on one stream (DESIGN.md section 3):
//   setup_kernel      prior -> parameters -> per-walker constants -> initial step      one thread per walker
//   advance_kernel    the spin integration (Dormand-Prince 5(4), dense output at the   persistent warps; every lane
//                     nodes the data need); stiff walkers are queued for ...            pulls its next walker off a
//   advance_kernel<STIFF>  ... the implicit (Radau IIA) integrator                      queue when its own is done
//   reduce_*_kernel   luminosity -> interpolation -> chi-square -> lnprob (or model /  thread per walker, or a warp
//                     light-curve output; or the stretch move's accept step)           per walker with a shuffle-
//                                                                                       reduced chi-square
// plus the ensemble-order helpers of the device-resident sampler and pt_swap_kernel (replica exchange of a
// parallel-tempered ensemble).  The rest of the library lives beside this file: magprop_chain.cu (posterior
// summaries of a chain), magprop_models.cu (reference restatements of the model) and magprop_device.cu (IPC, the
// peer barrier, the FP64 peak, version and errors).  Only this file includes magprop_core.cuh, so the disc tables
// are compiled into the library once.
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "magprop_host.hpp"
#include "magprop_rng.cuh"
#include "magprop_abi.hpp"
#include "magprop_kde.hpp"

namespace mp {

constexpr unsigned kFull = 0xffffffffu;

// Warp-aggregated append: the lanes with `want` get consecutive slots of a list whose length is *count.
__device__ __forceinline__ int warp_append(bool want, int* count) {
  const unsigned m = __ballot_sync(kFull, want);
  if (!m) return -1;
  const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
  int base = 0;
  if (lane == leader) base = atomicAdd(count, __popc(m));
  base = __shfl_sync(kFull, base, leader);
  return want ? base + __popc(m & ((1u << lane) - 1u)) : -1;
}


// What every stage of a launch needs to know (passed by value in the kernel parameters).
struct Problem {
  Spec sp;
  DataView dv;          // nodes (+ the dataset for lnprob / model-at-data)
  const int* dat_orig;  // sorted datum -> caller's index (kModeModelAtData)
  double lower[MP_MAX_NDIM], upper[MP_MAX_NDIM];
  int prior_enabled;
  int ndim;
};

// Device work space of one launch (a slab of walkers), owned by the handle's lane.  Layouts follow the readers:
//   recs   the stage-1 records as a structure of arrays -- 8-byte word k of walker i at recs[k*stride + i] -- so
//          that the one-thread-per-walker kernels read and write them coalesced
//   ybuf   node j of walker i at ybuf[i*ws + j*ns]: walker-minor (ws = 1, ns = the launch's slab size S) when stage 3
//          runs one thread per walker (small datasets), node-minor (ws = Nn, ns = 1) when it runs one warp per walker;
//          either way it spans S * Nn values (recs' stride is the lane's capacity, which may exceed S)
struct Work {
  int W;               // walkers in the slab
  int stride;          // slab capacity
  size_t ws, ns;
  unsigned long long* recs;
  double* ybuf;        // stage 2 -> stage 3: y = omega^-2 at the nodes
  int* status;         // [W]
  int* n_rhs;          // [W]
  int* work;           // [W] walkers for the explicit integrator
  StiffRec* squeue;    // [W] walkers for the implicit integrator
  int* counters;       // [0] walkers in `work`, [1] next to hand out, [2] walkers in `squeue`, [3] next to hand out,
                       // [4..7] extent of the ensemble in the ordering's bins: max(im + 1), max(256 - im), max(ie + 1), max(32 - ie),
                       // [8..11] the extent the host has been told
  int track;           // 1: the setup kernel measures [4..7] (launches large enough to be ordered)
  int* hint;           // (track) where the host reads [4..7] later: mapped pinned memory, written by the implicit launch's first thread
  // ordering of `work` (large launches): per-walker bucket key and the bucket histogram / cursors
  int* key;            // [W] bucket key of every walker
  int* hist;           // [kOrderBuckets + 3]: bucket counts / offsets, "tight" flag, tight cursor, block ticket
  int* slot_wid;       // [W] or null: the stages index their work space by SLOT; slot s holds walker slot_wid[s]
};                     //          (null: slot = walker, launches too small to be worth ordering)

// The order in which the integrator takes the walkers of a large launch.  Lanes that start together run through
// the same phases of the integration together only if their walkers are alike, so the walkers of a large launch are
// given SLOTS -- the index under which all three stages keep a walker's record, node values and status, so that
// neighbouring lanes also touch neighbouring memory -- in the order of a key of
// the two parameter combinations that set a walker's timeline: the mass that flows through the disc, M_disc * delta
// (1/24-decade bins, DESCENDING: the number of steps grows with it -- correlation 0.83..0.94 with log(steps) on
// posterior-like ensembles of the four synthetic datasets -- and a launch whose long integrations start last ends
// with a tail as long as one of them, `tools/sched_sim.py`) and, within a bin, the fallback time scale epsilon
// (quarter-decade bins).  A counting sort: histogram in order_key_kernel, one scan, one scatter.
// Measured on 2^18 walkers against the unordered list: prior-uniform +13 %, posterior-like spreads +10..30 %,
// a 1e-4 ball unchanged; results do not depend on the order (tested).
constexpr int kOrderBuckets = 32 * 256;
#ifndef MP_ORDER_MIN_WALKERS
#define MP_ORDER_MIN_WALKERS 8192
#endif
constexpr int kOrderMinWalkers = MP_ORDER_MIN_WALKERS;
constexpr int kCoopSmallWalkers = 2048;   // launches up to this size run stage 3 with a warp per walker (see reduce_coop_kernel)
constexpr int kOrderTightBuckets = 8;
__device__ __forceinline__ void order_bins(const Spec& sp, const double* th, int& ie, int& im) {
  const float le = ((sp.unlog_mask >> 4) & 1) ? (float)th[4] : __log10f((float)th[4]);
  const float lm = ((sp.unlog_mask >> 2) & 1) ? (float)th[2] : __log10f((float)th[2]);
  const float ld = ((sp.unlog_mask >> 5) & 1) ? (float)th[5] : __log10f((float)th[5]);
  const float eb = fminf(fmaxf((le + 4.0f) * 4.0f, 0.0f), 31.0f);
  const float mb = fminf(fmaxf((lm + ld + 10.0f) * 24.0f, 0.0f), 255.0f);
  ie = (eb == eb) ? (int)eb : 0;
  im = (mb == mb) ? (int)mb : 0;
}
__device__ __forceinline__ int order_key_of(const Spec& sp, const double* th) {
  int ie, im;
  order_bins(sp, th, ie, im);
  // descending in M*delta (the long integrations first), zig-zag in epsilon: neighbouring buckets across an M*delta boundary are alike
  return (255 - im) * 32 + ((im & 1) ? 31 - ie : ie);
}
// An ensemble inside a few neighbouring buckets gains nothing from the ordering (launch_eval skips it).
constexpr int kTightMdBins = 2, kTightEpsBins = 1;
// The threads of a block claim slots of their keys' counters: lanes with the same key share one atomic, and when
// the whole block holds one key (a tight ensemble: every walker in the same bucket) so do its warps -- otherwise
// thousands of warps would queue on one address.  Every thread of the block must call (it synchronises).
__device__ __forceinline__ int block_claim_by_key(bool want, int key, int* counters) {
  __shared__ int s_key[32], s_cnt[32], s_base;
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  const unsigned wanting = __ballot_sync(kFull, want);
  const unsigned peers = __match_any_sync(kFull, want ? key : -1);
  // this warp's key, from its first wanting lane: -1 nothing to claim, -2 mixed keys
  const int first = wanting ? __ffs(wanting) - 1 : 0;
  const int fkey = __shfl_sync(kFull, key, first);
  const unsigned fpeers = __shfl_sync(kFull, peers, first);
  if (lane == 0) {
    s_cnt[wrp] = __popc(wanting);
    s_key[wrp] = !wanting ? -1 : ((fpeers == wanting) ? fkey : -2);
  }
  __syncthreads();
  int common = -1, before = 0, total = 0;
  bool uniform = true;
  for (int w = 0; w < nw; ++w) {
    const int kw = s_key[w];
    if (kw == -1) continue;
    if (kw == -2 || (common >= 0 && kw != common)) uniform = false;
    if (common < 0) common = kw;
    if (w < wrp) before += s_cnt[w];
    total += s_cnt[w];
  }
  int pos = -1;
  if (uniform && common >= 0) {
    if (threadIdx.x == 0) s_base = atomicAdd(counters + common, total);
    __syncthreads();
    if (want) pos = s_base + before + __popc(wanting & ((1u << lane) - 1u));
  } else {
    __syncthreads();
    if (want) {
      const int leader = __ffs(peers) - 1;
      int base = 0;
      if (lane == leader) base = atomicAdd(counters + key, __popc(peers));
      base = __shfl_sync(peers, base, leader);
      pos = base + __popc(peers & ((1u << lane) - 1u));
    }
  }
  return pos;
}
// Exclusive scan of the bucket histogram in place (hist[b] becomes the first slot of bucket b), by the NT threads of
// one block.  An ensemble that occupies only a handful of buckets is tight enough to be taken as it comes:
// hist[kOrderBuckets] tells the scatter so, which then hands out the slots in index order (cursor: hist[kOrderBuckets + 1]).
template <int NT>
__device__ __forceinline__ void scan_buckets(int* __restrict__ hist) {
  __shared__ int part[NT];
  __shared__ int occupied;
  constexpr int per = kOrderBuckets / NT;
  const int base = threadIdx.x * per;
  int sum = 0, nz = 0;
  if (threadIdx.x == 0) occupied = 0;
  for (int c = 0; c < per; ++c) { const int v = __ldcg(hist + base + c); sum += v; nz += v != 0; }   // (written by other blocks' atomics: read at L2)
  part[threadIdx.x] = sum;
  __syncthreads();
  if (nz) atomicAdd(&occupied, nz);
  __syncthreads();
  if (occupied <= kOrderTightBuckets) {
    if (threadIdx.x == 0) hist[kOrderBuckets] = 1;
    return;
  }
  for (int off = 1; off < NT; off <<= 1) {
    const int v = (threadIdx.x >= off) ? part[threadIdx.x - off] : 0;
    __syncthreads();
    part[threadIdx.x] += v;
    __syncthreads();
  }
  int run = part[threadIdx.x] - sum;
  for (int c = 0; c < per; ++c) { const int v = __ldcg(hist + base + c); hist[base + c] = run; run += v; }
}
__global__ void order_scatter_kernel(int W, const int* __restrict__ key, int* __restrict__ cursor, int* __restrict__ slot_wid) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int kk = (i < W) ? key[i] : -1;
  if (cursor[kOrderBuckets]) {                       // tight ensemble: as it comes
    const int we = warp_append(kk >= 0, cursor + kOrderBuckets + 1);
    if (kk >= 0) slot_wid[we] = i;
    return;
  }
  const int pos = block_claim_by_key(kk >= 0, kk, cursor);
  if (kk >= 0) slot_wid[pos] = i;
}

// The ensemble move wrapped around an evaluation (mp_stretch_half_step / mp_ensemble_half_step / the *_moves_ entry
// points).  `kind` is the stretch move (Goodman & Weare 2010; emcee's RedBlueMove), differential evolution or its
// snooker update (include/magprop_b200.h, mp_move); one kind per launch.  Every kind has one contract: the proposal
// (setup_kernel, or order_key_kernel on an ordered launch) leaves q in `prop` and ln f, the log of its Hastings
// factor, in `lnf`; the accept step (the reduce kernels, deliver) takes
//   accept iff ln f + lp(q) - lp(s) > ln u,  u = accept_uniform(kind, ...)
// tempered: beta_t lp(q) - beta_t lp(s).
struct Move {
  double* coords;        // [nwalkers][ndim], updated in place
  double* lnp;           // [nwalkers]
  // who moves against whom: explicit index lists (mp_stretch_half_step) ...
  const int* active;     // [n_active] walkers to move (disjoint from complement), or null
  const int* complement; // [n_complement]
  // ... or positions of the ensemble order, with T temperatures of n walkers (T = 1 without a ladder): mover
  // mover0 + i is the tempered_mover of positions pos0 + [0, n/2), its partner is drawn from its own temperature's
  // P(cpos0 + [0, n_complement))
  SplitPerm perm;
  int pos0, cpos0;
  int n_complement;
  const double* betas;   // [T] the accept test weighs the log-probabilities by betas[t] (null: untempered)
  int mover0;
  double a;
  uint64_t seed, step;   // step: the half-step counter (RNG counter word)
  double* prop;          // [n_active][ndim] the proposals (work space)
  int* accepted;         // [nwalkers] counters (may be null)
  int* status;           // [nwalkers] MP_WALKER_* bits of the latest proposal (may be null)
  int* n_rhs;            // [nwalkers] (may be null)
  // Sharded ensembles with peer-mapped replicas (NVLink): a rank writes the rows it moves into its OWN replica
  // only, and reads a row it needs -- its movers' current positions, their partners -- from the replica of the
  // rank that moved that walker last, which every rank can work out (the ensemble order is a keyed permutation):
  //   moved earlier in this step (the partners of half-step 1)  ->  rank (position within the half) / n_mine
  //   otherwise                                                 ->  the same rule with LAST step's order, unless the
  //                                                                 replicas were synchronised since (`synced`)
  // No collective, no remote stores; one flag barrier per half-step (mp_peer_barrier) orders the reads after the writes.
  int n_peers;
  const double* peer_coords[MP_MAX_PEERS];   // the other ranks' replicas, in rank order without this rank
  const double* peer_lnp[MP_MAX_PEERS];
  SplitPerm prev_perm;   // last step's ensemble order
  int rank, n_mine, half, split, synced;
  double* pack_out;      // [n_active][ndim+1]: every mover's (row, lnp) after the move, or null
  double* bad_rows;      // proposals whose likelihood was not finite ({GRB}_bad.csv, mcmc_eqns.py:72-79)
  int* bad_count;
  int bad_capacity;
  int kind;              // MP_MOVE_STRETCH (a above), MP_MOVE_DE (g0 = gamma0, s3 = sigma sqrt 3), MP_MOVE_DE_SNOOKER (gammas)
  double g0, s3, gammas;
  double* lnf;           // [n_active] ln of each proposal's Hastings factor (work space next to prop)
};

// Which rank's replica holds walker w's current row (see Move).
__device__ __forceinline__ int home_before_this_step(const Move& m, int w) {
  if (m.synced) return m.rank;
  return (int)(perm_inv(m.prev_perm, (uint32_t)w) % (uint32_t)m.half) / m.n_mine;
}
__device__ __forceinline__ const double* replica_coords(const Move& m, int home) {
  return home == m.rank ? m.coords : m.peer_coords[home < m.rank ? home : home - 1];
}
__device__ __forceinline__ const double* replica_lnp(const Move& m, int home) {
  return home == m.rank ? m.lnp : m.peer_lnp[home < m.rank ? home : home - 1];
}
// The row mover i moves, and its temperature (0 without a ladder).
__device__ __forceinline__ int mover_row(const Move& m, int i, int& t) {
  t = 0;
  if (m.active) return m.active[i];
  const TemperedMover tm = tempered_mover(m.perm, (uint32_t)m.pos0, (uint32_t)(m.mover0 + i));
  t = (int)tm.t;
  return (int)tm.row;
}
// The row at position pj of the complement of a mover of temperature t.
__device__ __forceinline__ int partner_row(const Move& m, int t, int pj) {
  if (m.complement) return m.complement[pj];
  return (int)tempered_partner(m.perm, (uint32_t)m.cpos0, (uint32_t)t, (uint32_t)pj);
}

constexpr int kRecWords = (int)(sizeof(WalkerRec) / 8);
static_assert(sizeof(WalkerRec) % 8 == 0, "WalkerRec is moved as 8-byte words");
__device__ __forceinline__ void rec_store(const Work& k, int i, const WalkerRec& r) {
  unsigned long long tmp[kRecWords];
  memcpy(tmp, &r, sizeof(r));
#pragma unroll
  for (int c = 0; c < kRecWords; ++c) k.recs[(size_t)c * k.stride + i] = tmp[c];
}
__device__ __forceinline__ void rec_load(const Work& k, int i, WalkerRec& r) {
  unsigned long long tmp[kRecWords];
#pragma unroll
  for (int c = 0; c < kRecWords; ++c) tmp[c] = k.recs[(size_t)c * k.stride + i];
  memcpy(&r, tmp, sizeof(r));
}

// Only what a stage reads of a record: stage 3 needs disc_mass and the luminosity stage (19 of the 55 words),
// the integrators the disc-mass and torque constants (16) -- a lane taking a walker loads them one lane at a time.
#define MP_WFIELD(name) \
  w.name = __longlong_as_double((long long)k.recs[((offsetof(WalkerRec, w) + offsetof(Walker, name)) / 8) * (size_t)k.stride + i])
#define MP_RWORD(member) k.recs[(offsetof(WalkerRec, member) / 8) * (size_t)k.stride + i]
__device__ __forceinline__ void rec_load_step(const Work& k, int i, Walker& w) {
  MP_WFIELD(inv_tv); MP_WFIELD(eps); MP_WFIELD(u0); MP_WFIELD(K); MP_WFIELD(C); MP_WFIELD(u_late); MP_WFIELD(Kq);
  MP_WFIELD(sqrtA); MP_WFIELD(KqA); MP_WFIELD(tvI); MP_WFIELD(g_sqrtA); MP_WFIELD(g_tvI); MP_WFIELD(Cdip_I); MP_WFIELD(Cdip_I2);
  MP_WFIELD(KtvI); MP_WFIELD(M_init);
  w.bad = 0;
}
__device__ __forceinline__ void rec_load_lum(const Work& k, int i, Walker& w) {
  MP_WFIELD(inv_tv); MP_WFIELD(eps); MP_WFIELD(u0); MP_WFIELD(K); MP_WFIELD(C); MP_WFIELD(M_init); MP_WFIELD(u_late);
  MP_WFIELD(l_inv_tv); MP_WFIELD(l_Ccap); MP_WFIELD(l_kc); MP_WFIELD(l_sqrtA); MP_WFIELD(l_sGMkc); MP_WFIELD(l_GM_kc);
  MP_WFIELD(Ldip_coef); MP_WFIELD(dipeff); MP_WFIELD(propeff); MP_WFIELD(f_beam); MP_WFIELD(omega0);
  w.bad = (int)k.recs[((offsetof(WalkerRec, w) + offsetof(Walker, bad)) / 8) * (size_t)k.stride + i];
}

// ---- stage 1: setup ---------------------------------------------------------------------------------
// The stretch proposal of mover i (see Move): q = c - (c - s) z, kept in m.prop[i] for the accept step.  With
// peer-mapped replicas the mover's current row is first brought into the local replica (it is about to be moved
// here) and the partner's row is read from its home.
__device__ __forceinline__ void fetch_mover(const Move& m, int me, int ndim) {
  const int hm = home_before_this_step(m, me);
  if (hm != m.rank) {
    const double* src = replica_coords(m, hm);
    for (int c = 0; c < ndim; ++c) m.coords[(size_t)me * ndim + c] = src[(size_t)me * ndim + c];
    m.lnp[me] = replica_lnp(m, hm)[me];
  }
}
// The replica that holds the current row of the walker at complement position pj (row `row`).
__device__ __forceinline__ const double* partner_replica(const Move& m, int pj, int row) {
  if (m.n_peers == 0) return m.coords;
  return replica_coords(m, m.split == 1 ? pj / m.n_mine : home_before_this_step(m, row));
}
// The differential-evolution proposals of mover i (Move::kind MP_MOVE_DE or MP_MOVE_DE_SNOOKER; the formulas are those
// of include/magprop_b200.h, mp_move): q in th and m.prop[i], ln f in m.lnf[i].  No FMA contraction, as in propose().
__device__ __noinline__ void propose_de(const Move& m, int i, int ndim, double* th) {
  int t;
  const int me = mover_row(m, i, t);
  const MoveDraws u = move_draws(m.seed, m.step, (uint32_t)me);
  if (m.n_peers > 0) fetch_mover(m, me, ndim);
  const double* x = m.coords + (size_t)me * ndim;
  const uint32_t nc = (uint32_t)m.n_complement;
  double lnf = 0.0;
  if (m.kind == MP_MOVE_DE) {
    uint32_t j, k;
    de_pair(u.u[0], u.u[1], nc, &j, &k);
    const int rj = partner_row(m, t, (int)j), rk = partner_row(m, t, (int)k);
    const double* cj = partner_replica(m, (int)j, rj) + (size_t)rj * ndim;
    const double* ck = partner_replica(m, (int)k, rk) + (size_t)rk * ndim;
    const double g = __dmul_rn(m.g0, __dadd_rn(1.0, __dmul_rn(m.s3, __dadd_rn(__dmul_rn(2.0, u.u[2]), -1.0))));
    for (int c = 0; c < ndim; ++c) th[c] = __dadd_rn(x[c], __dmul_rn(g, __dadd_rn(cj[c], -ck[c])));
  } else {
    uint32_t jz, j1, j2;
    snooker_triple(u.u[0], u.u[1], u.u[2], nc, &jz, &j1, &j2);
    const int rz = partner_row(m, t, (int)jz), r1 = partner_row(m, t, (int)j1), r2 = partner_row(m, t, (int)j2);
    const double* z = partner_replica(m, (int)jz, rz) + (size_t)rz * ndim;
    const double* c1 = partner_replica(m, (int)j1, r1) + (size_t)r1 * ndim;
    const double* c2 = partner_replica(m, (int)j2, r2) + (size_t)r2 * ndim;
    double ee = 0.0, dd = 0.0;
    for (int c = 0; c < ndim; ++c) {
      const double e = __dadd_rn(x[c], -z[c]);
      ee = __dadd_rn(ee, __dmul_rn(e, e));
      dd = __dadd_rn(dd, __dmul_rn(__dadd_rn(c1[c], -c2[c]), e));
    }
    if (ee == 0.0) {
      for (int c = 0; c < ndim; ++c) th[c] = x[c];
    } else {
      const double f = __ddiv_rn(__dmul_rn(m.gammas, dd), ee);
      double nq = 0.0;
      for (int c = 0; c < ndim; ++c) {
        th[c] = __dadd_rn(x[c], __dmul_rn(f, __dadd_rn(x[c], -z[c])));
        const double w = __dadd_rn(th[c], -z[c]);
        nq = __dadd_rn(nq, __dmul_rn(w, w));
      }
      lnf = nq == 0.0 ? -INFINITY : __dmul_rn(0.5 * (ndim - 1.0), log(__ddiv_rn(nq, ee)));
    }
  }
  for (int c = 0; c < ndim; ++c) m.prop[(size_t)i * ndim + c] = th[c];
  m.lnf[i] = lnf;
}

// The proposal of mover i: q in th and m.prop[i], ln f in m.lnf[i].  The stretch move draws u_z and u_partner from
// Philox counter (half-step, row, 0):  z = ((a-1) u_z + 1)^2 / a,  q = c - (c - s) z,  ln f = (ndim-1) ln z.
__device__ __forceinline__ void propose(const Move& m, int i, int ndim, double* th) {
  if (m.kind == MP_MOVE_KDE) {    // formed by kde_propose (magprop_kde.cu) ahead of this launch
    for (int c = 0; c < ndim; ++c) th[c] = m.prop[(size_t)i * ndim + c];
    return;
  }
  if (m.kind != MP_MOVE_STRETCH) {
    propose_de(m, i, ndim, th);
    return;
  }
  int t;
  const int me = mover_row(m, i, t);
  const Philox r = philox4x32_10((uint32_t)m.step, (uint32_t)(m.step >> 32), (uint32_t)me, 0u,
                                 (uint32_t)m.seed, (uint32_t)(m.seed >> 32));
  const double zr = __dadd_rn(__dmul_rn(m.a - 1.0, u01(r.c[0], r.c[1])), 1.0);
  const double z = __ddiv_rn(__dmul_rn(zr, zr), m.a);
  const int pj = (int)pick_index(u01(r.c[2], r.c[3]), (uint32_t)m.n_complement);
  const int partner = partner_row(m, t, pj);
  const double* pc = m.coords;
  if (m.n_peers > 0) {
    fetch_mover(m, me, ndim);
    pc = partner_replica(m, pj, partner);
  }
  for (int c = 0; c < ndim; ++c) {
    const double cc = pc[(size_t)partner * ndim + c];
    const double x = m.coords[(size_t)me * ndim + c];
    th[c] = __dadd_rn(cc, -__dmul_rn(__dadd_rn(cc, -x), z));   // no FMA contraction: reproducible on the host
    m.prop[(size_t)i * ndim + c] = th[c];
  }
  m.lnf[i] = __dmul_rn(ndim - 1.0, log(z));
}

// Large launches, before the setup: every walker's bucket key and the bucket histogram (MOVE: the proposals are
// formed here, the setup then reads them from m.prop).
template <bool MOVE>
__global__ void __launch_bounds__(128) order_key_kernel(const __grid_constant__ Problem p, const __grid_constant__ Work k,
                                                        const double* __restrict__ theta, const __grid_constant__ Move m) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const bool have = i < k.W;
  double th[MP_MAX_NDIM];
  int kk = -1;
  if (have) {
    if (MOVE) propose(m, i, p.ndim, th);
    else
      for (int c = 0; c < p.ndim; ++c) th[c] = theta[(size_t)i * p.ndim + c];
    kk = order_key_of(p.sp, th);
    k.key[i] = kk;
  }
  block_claim_by_key(have, kk, k.hist);
  // the last block to get here turns the histogram into bucket offsets (saves a launch)
  __shared__ int last;
  __threadfence();
  if (threadIdx.x == 0) last = atomicAdd(k.hist + kOrderBuckets + 2, 1) == (int)gridDim.x - 1;
  __syncthreads();
  if (last) {
    __threadfence();
    scan_buckets<128>(k.hist);
  }
}

// MOVE = false: walker i's parameters are theta[i][:].  MOVE = true: walker i is mover i of an ensemble-move
// half-step and its parameters are the proposal q.  One thread per SLOT (= walker unless the launch is ordered).
template <bool MOVE>
__global__ void __launch_bounds__(128, 4) setup_kernel(const __grid_constant__ Problem p, const __grid_constant__ Work k,
                                                    const double* __restrict__ theta, const __grid_constant__ Move m) {
  const int sl = blockIdx.x * blockDim.x + threadIdx.x;
  const bool have = sl < k.W;
  const int ndim = p.ndim;
  double th[MP_MAX_NDIM];
  if (have) {
    const int i = k.slot_wid ? k.slot_wid[sl] : sl;
    if (MOVE && !k.slot_wid) {
      propose(m, i, ndim, th);
    } else {
      const double* src = MOVE ? m.prop : theta;
      for (int c = 0; c < ndim; ++c) th[c] = src[(size_t)i * ndim + c];
    }
  }
  bool to_explicit = false, to_implicit = false;
  double y0 = 0.0, h0 = 0.0;
  int n_rhs0 = 0;
  if (have) {
    WalkerRec r;
    const double t_end = p.dv.n_nodes > 0 ? p.dv.node_t[p.dv.n_nodes - 1] : p.dv.t_start;
    prepare_walker(p.sp, th, ndim, p.prior_enabled != 0, p.lower, p.upper, p.dv.t_start, t_end, r);
    if (!(r.status & kWalkerPriorReject)) rec_store(k, sl, r);
    y0 = r.y0; h0 = r.h0; n_rhs0 = r.n_rhs;
    k.status[sl] = r.status;
    k.n_rhs[sl] = r.n_rhs;
    // (a walker whose initialisation failed still goes to the integrator, which marks its nodes)
    const bool go = (r.status == kWalkerOk || r.status == kWalkerIntegratorFail) && p.dv.n_nodes > 0;
    to_implicit = go && p.sp.bucciantini && r.status == kWalkerOk;
    to_explicit = go && !to_implicit;
  }
  if (k.track && (blockIdx.x & 15) == 0) {
    // how far the ensemble reaches in the ordering's bins (the host decides from it whether the NEXT launch is
    // ordered); every 16th block looks -- a sample of >= 512 walkers is ample for the purpose
    const bool in = to_explicit || to_implicit;
    int ie = 0, im = 0;
    if (in) order_bins(p.sp, th, ie, im);
    const int v[4] = {in ? im + 1 : 0, in ? 256 - im : 0, in ? ie + 1 : 0, in ? 32 - ie : 0};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int m = __reduce_max_sync(kFull, v[q]);
      if ((threadIdx.x & 31) == 0 && m > __ldcg(k.counters + 4 + q)) atomicMax(k.counters + 4 + q, m);
    }
  }
  const int we = warp_append(to_explicit, k.counters + 0);      // (threads run in slot order: so does the work list)
  if (to_explicit) k.work[we] = sl;
  const int wi = warp_append(to_implicit, k.counters + 2);
  if (to_implicit) {
    StiffRec q;
    q.t = p.dv.t_start; q.y = y0; q.h = h0; q.wid = sl; q.jn = 0; q.n_rhs = n_rhs0; q.n_steps = 0;
    k.squeue[wi] = q;
  }
}

// ---- stage 2: advance -------------------------------------------------------------------------------
// Persistent warps.  Every trip of the loop is ONE integrator step for every lane that holds a walker; a lane
// whose walker is finished (all nodes delivered), failed or -- explicit variant -- turned stiff hands it on
// and takes the next walker off the queue at the top of the next trip, so the lanes of a warp stay busy
// whatever the spread of step counts in the ensemble (40 .. 10^3 over the prior box).  The cheap, divergent
// parts (delivering nodes, hand-over, taking a walker) sit between the steps.
// Resident blocks per SM the explicit integrator is compiled for: 10 x 64 threads = 20 warps at 96 registers.
// (With the luminosity stage out of this kernel the spills at 96 registers are 86 bytes; measured against 8 blocks /
// 128 registers: +7 % on 2^18-walker launches, +5 % through the host-pointer path; 12 and 14 blocks no better.)
#ifndef MP_MIN_BLOCKS_32
#define MP_MIN_BLOCKS_32 20
#endif
#ifndef MP_MIN_BLOCKS_64
#define MP_MIN_BLOCKS_64 10
#endif
// Resident warps per SM the implicit variant is compiled for: 12 (166 registers, no spills), and 16 (128 registers)
// for launches large enough that its queue is longer than one wave of the 12-warp build -- 75 904 stiff walkers of
// 2^18 prior-uniform ones on 56 832 lanes are 1.34 waves, on 75 776 lanes one: 7.13 -> 6.71 ms per launch, 10^6
// walkers 22.2 -> 21.5; a single wave (2^16 walkers) is faster on the 12-warp build, 4.78 against 5.19 ms.
#ifndef MP_STIFF_MIN_WARPS
#define MP_STIFF_MIN_WARPS 12
#endif
constexpr int kStiffWarpsWide = 16;
constexpr int kStiffWideMinWalkers = 196608;
constexpr int kNodeSmemDoubles = 512;      // node times staged per block when they fit (4 KB)

template <bool STIFF, int BLOCK, int STIFF_WARPS = MP_STIFF_MIN_WARPS>
__global__ void __launch_bounds__(BLOCK, STIFF ? (STIFF_WARPS * 32 / BLOCK) : (BLOCK == 32 ? MP_MIN_BLOCKS_32 : MP_MIN_BLOCKS_64))
advance_kernel(const __grid_constant__ Problem p, const __grid_constant__ Work k) {
  __shared__ double s_nodes[kNodeSmemDoubles];
  const int Nn = p.dv.n_nodes;
  const double* node_t = p.dv.node_t;
  if (Nn <= kNodeSmemDoubles) {
    for (int j = threadIdx.x; j < Nn; j += BLOCK) s_nodes[j] = node_t[j];
    node_t = s_nodes;
    __syncthreads();
  }
  const int lane = threadIdx.x & 31;
  if (STIFF && k.track && blockIdx.x == 0 && threadIdx.x == 0)        // (see launch_eval: the next launch's hint;
    for (int q = 0; q < 4; ++q) {                                     // written over PCIe only when it changes)
      const int v = k.counters[4 + q];
      if (v != k.counters[8 + q]) { k.counters[8 + q] = v; k.hint[q] = v; }
    }
  const int n_items = k.counters[STIFF ? 2 : 0];
  int* next = k.counters + (STIFF ? 3 : 1);
  const double t_end = ldd(node_t + (Nn - 1));
  Walker w;
  Integrator in;
  in.status = kWalkerOk; in.stiff = 0; in.n_rhs = 0; in.t = p.dv.t_start;
  int wid = 0, jn = 0;
  double* row = k.ybuf;
  bool have = false, empty = false;
  int waited = 0;
  for (;;) {
    // ---- take walkers
    // A lane that is done waits a few trips for the other lanes of its warp before it takes a new walker:
    // lanes that start together run through the same phases of the integration together (capped / uncapped
    // Alfven radius, saturated / unsaturated tanh, kinks on the same trips), which is worth more than the idle
    // trips when the ensemble is tight (+10 % at a posterior-like spread of 0.01..0.05, measured), and when it
    // is not -- prior-uniform, where the step counts differ tenfold -- the wait is over after MP_REFILL_PATIENCE trips.
    const unsigned idle = __ballot_sync(kFull, !have);
#ifndef MP_REFILL_PATIENCE
#define MP_REFILL_PATIENCE 32
#endif
    waited = idle ? waited + 1 : 0;
    // (one warp-wide vote per trip: whether any lane holds a walker follows from `idle` unless lanes were just refilled)
    if (!(idle && !empty && (idle == kFull || waited > MP_REFILL_PATIENCE))) {
      if (idle == kFull) break;
    } else {
      waited = 0;
      const int leader = __ffs(idle) - 1;
      int base = 0;
      if (lane == leader) base = atomicAdd(next, __popc(idle));
      base = __shfl_sync(kFull, base, leader);
      if (base + __popc(idle) >= n_items) empty = true;          // (uniform across the warp)
      const int my = base + __popc(idle & ((1u << lane) - 1u));
      if (!have && my < n_items) {
        have = true;
        if (STIFF) {
          const StiffRec q = k.squeue[my];
          wid = q.wid;
          rec_load_step(k, wid, w);
          integrator_load_stiff(q, in);
          jn = q.jn;
        } else {
          wid = k.work[my];
          rec_load_step(k, wid, w);
          const int i = wid;
          WalkerRec r;                                             // (its Walker part stays unset: see rec_load_step)
          r.y0 = __longlong_as_double((long long)MP_RWORD(y0));
          r.h0 = __longlong_as_double((long long)MP_RWORD(h0));
          r.k1 = __longlong_as_double((long long)MP_RWORD(k1));
          const unsigned long long rs = MP_RWORD(regime0);         // regime0 | status << 32
          r.regime0 = (unsigned)rs;
          r.status = (int)(rs >> 32);
          r.n_rhs = (int)(unsigned)MP_RWORD(n_rhs);
          integrator_load(r, w.C, p.dv.t_start, in);
          if (r.status != kWalkerOk) in.status = kWalkerIntegratorFail;
          jn = 0;
        }
        row = k.ybuf + (size_t)wid * k.ws;
        jn = drain_nodes<STIFF>(in, jn, Nn, node_t, row, k.ns);      // a node at the starting time
      }
      if (!__any_sync(kFull, have)) break;
    }
    // ---- one step for every lane that holds a walker (a fresh walker whose nodes are all delivered
    // already, or whose initialisation failed, skips it)
    if (have && jn < Nn && in.status == kWalkerOk) {
      if (STIFF) radau_step(p.sp, w, t_end, in);
      else integrator_step(p.sp, w, t_end, in);
      jn = drain_nodes<STIFF>(in, jn, Nn, node_t, row, k.ns);
    }
    // ---- hand finished walkers on
    if (have) {
      const bool failed = in.status != kWalkerOk;
      const bool stiff = !STIFF && in.stiff && !failed && jn < Nn;
      if (jn >= Nn || failed || stiff) {
        if (failed)
          for (; jn < Nn; ++jn) row[jn * k.ns] = NAN;            // stage 3 sees no solution there
        if (stiff) {
          // (explicit variant) the implicit integrator picks the walker up where this one stopped
          StiffRec q;
          q.t = in.t; q.y = in.omega; q.h = in.h; q.wid = wid; q.jn = jn; q.n_rhs = in.n_rhs; q.n_steps = in.n_steps;
          k.squeue[atomicAdd(k.counters + 2, 1)] = q;
        } else {
          k.status[wid] |= in.status;
          k.n_rhs[wid] = in.n_rhs;
        }
        have = false;
      }
    }
  }
}

// ---- stage 3: reduce ----------------------------------------------------------------------------------
// The dataset a block works against -- node times and, per datum, y/yerr, 1e-50/yerr, x - t_lo, the
// interpolation weight and the lower-node index -- staged in shared memory when it fits the budget below
// (the synthetic datasets take 2.2 KB).
constexpr int kDataSmemDoubles = 768;      // 6 KB per block
__device__ __forceinline__ bool stage_data(const DataView& g, DataView& s, double* buf, int nthreads) {
  const int Nn = g.n_nodes, D = g.n_data;
  const int need = Nn + 4 * D + (D + 1) / 2;
  if (need > kDataSmemDoubles) return false;
  double* q = buf;
  double* nt = q; q += Nn;
  double* ys = q; q += D;
  double* c = q; q += D;
  double* dx = q; q += D;
  double* w = q; q += D;
  int* lo = reinterpret_cast<int*>(q);
  for (int i = threadIdx.x; i < Nn; i += nthreads) nt[i] = g.node_t[i];
  for (int i = threadIdx.x; i < D; i += nthreads) {
    ys[i] = g.dat_ys[i]; c[i] = g.dat_c[i]; dx[i] = g.dat_dx[i]; w[i] = g.dat_w[i]; lo[i] = g.dat_lo[i];
  }
  s = g;
  s.node_t = nt; s.dat_ys = ys; s.dat_c = c; s.dat_dx = dx; s.dat_w = w; s.dat_lo = lo;
  __syncthreads();
  return true;
}

// Where a finished evaluation goes: the caller's arrays, or the accept step of the ensemble move.
struct Sink {
  double* lnp;     // [W]
  int* status;     // [W] or null
  int* n_rhs;      // [W] or null
};

template <bool MOVE>
__device__ __forceinline__ void deliver(const Problem& p, const Work& k, const Sink& s, const Move& m, int sl, double lp_new,
                                        int st) {
  const int nr = k.n_rhs[sl];
  const int i = k.slot_wid ? k.slot_wid[sl] : sl;              // the walker this slot holds
  if (!MOVE) {
    s.lnp[i] = lp_new;
    if (s.status) s.status[i] = st;
    if (s.n_rhs) s.n_rhs[i] = nr;
    return;
  }
  const int ndim = p.ndim;
  int t;
  const int me = mover_row(m, i, t);
  const double ua = accept_uniform(m.kind, m.seed, m.step, (uint32_t)me);
  const double* q = m.prop + (size_t)i * ndim;
  const double lp_old = m.lnp[me];
  double lq = lp_new, lx = lp_old;           // tempered: beta_t lp (lnp stays untempered)
  if (m.betas) {
    const double b = m.betas[t];
    lq = __dmul_rn(b, lp_new);
    lx = __dmul_rn(b, lp_old);
  }
  const double lnpdiff = __dadd_rn(__dadd_rn(m.lnf[i], lq), -lx);
  const bool accept = lnpdiff > log(ua);
  if (accept) {
    for (int c = 0; c < ndim; ++c) m.coords[(size_t)me * ndim + c] = q[c];
    m.lnp[me] = lp_new;
    if (m.accepted) m.accepted[me] += 1;
  }
  if (m.pack_out) {
    double* rowp = m.pack_out + (size_t)i * (ndim + 1);
    for (int c = 0; c < ndim; ++c) rowp[c] = accept ? q[c] : m.coords[(size_t)me * ndim + c];
    rowp[ndim] = accept ? lp_new : lp_old;
  }
  if (m.status) m.status[me] = st;
  if (m.bad_count && (st & (kWalkerIntegratorFail | kWalkerNonfiniteLnlike))) {
    const int slot = atomicAdd(m.bad_count, 1);
    if (slot < m.bad_capacity)
      for (int c = 0; c < ndim; ++c) m.bad_rows[(size_t)slot * ndim + c] = q[c];
  }
  if (m.n_rhs) m.n_rhs[me] = nr;
}

// One thread per walker, nodes one after the other: every lane of a warp walks the same node and datum
// indices (the dataset is shared), so the loop is converged.  Used when the dataset is small (synthetic
// light curves: 50 points) -- there a warp per walker would leave half its lanes without a node.
template <int MODE, bool MOVE>
__global__ void __launch_bounds__(64, 12) reduce_rows_kernel(const __grid_constant__ Problem p, const __grid_constant__ Work k,
                                                         const __grid_constant__ Sink s, double* __restrict__ out,
                                                         const __grid_constant__ Move m) {
  __shared__ double s_data[kDataSmemDoubles];
  DataView dv = p.dv;
  stage_data(p.dv, dv, s_data, 64);
  const int sl = blockIdx.x * 64 + threadIdx.x;
  if (sl >= k.W) return;
  int st = k.status[sl];
  double result = -INFINITY;
  if (!(st & kWalkerPriorReject)) {
    Walker w;
    rec_load_lum(k, sl, w);
    double* o = (MODE == kModeModelAtData) ? out + (size_t)(k.slot_wid ? k.slot_wid[sl] : sl) * dv.n_data : nullptr;
    const double chi2 = reduce_rows<MODE>(p.sp, dv, w, k.ybuf + (size_t)sl * k.ws, o, nullptr, 1, p.dat_orig, k.ns);
    if (MODE == kModeLnprob) result = lnlike_of(chi2, st);                       // + lnprior == 0.0
  }
  if (MODE == kModeLnprob) deliver<MOVE>(p, k, s, m, sl, result, st);
  else if (s.status) s.status[k.slot_wid ? k.slot_wid[sl] : sl] = st;
}

// One warp per walker, one DATUM per lane: the lane evaluates the luminosity stage at its datum's two
// bracketing nodes (one if the datum sits on a node), interpolates, forms its residual -- and the chi-square
// is a warp-shuffle reduction over the data.  Used for the large datasets (the short-GRB sample: up to 1944
// points, ~2 nodes per datum), and it is what makes a small ensemble on such a burst run at the speed of the
// integration alone instead of one thread walking thousands of nodes.
// ORDERED = true: the residuals are summed in datum order (passed round the warp by shuffles) instead of by a tree,
// which reproduces reduce_rows_kernel's chi-square bit for bit: small launches on SMALL datasets use this form --
// a 128-walker half-step then spends 5 us here instead of 80 -- while large ones keep one thread per walker, and a
// walker's lnprob still does not depend on the size of the batch it is in.
template <int MODE, bool MOVE, bool ORDERED>
__global__ void __launch_bounds__(128) reduce_coop_kernel(const __grid_constant__ Problem p, const __grid_constant__ Work k,
                                                          const __grid_constant__ Sink s, double* __restrict__ out,
                                                          const __grid_constant__ Move m) {
  const int lane = threadIdx.x & 31;
  const int sl = (blockIdx.x * 128 + threadIdx.x) >> 5;
  if (sl >= k.W) return;
  const int i = k.slot_wid ? k.slot_wid[sl] : sl;              // the walker this slot holds
  int st = k.status[sl];
  double chi2 = 0.0;
  if (!(st & kWalkerPriorReject)) {
    Walker w;
    rec_load_lum(k, sl, w);                                    // (every lane the same words: broadcast loads)
    const double* row = k.ybuf + (size_t)sl * k.ws;
    const DataView& dv = p.dv;
    for (int d0 = 0; d0 < dv.n_data; d0 += 32) {
      const int d = d0 + lane;
      double r = 0.0;
      if (d < dv.n_data) {
        const int lo = dv.dat_lo[d];
        const double dx = dv.dat_dx[d];
        double M, om;
        const double L_lo = node_luminosity(p.sp, w, dv.node_t[lo], dv.t_start, row[lo * k.ns], false, M, om).tot;
        double mod = L_lo;                                     // datum sits on a grid node
        if (dx != 0.0) {
          const double L_hi = node_luminosity(p.sp, w, dv.node_t[lo + 1], dv.t_start, row[(lo + 1) * k.ns], false, M, om).tot;
          mod = fma(L_hi - L_lo, dv.dat_w[d], L_lo);           // np.interp: slope*(x-x_lo)+y_lo
        }
        if (MODE == kModeLnprob) r = fma(-mod, dv.dat_c[d], dv.dat_ys[d]);   // (y - mod/1e50)/yerr
        else out[(size_t)i * dv.n_data + (p.dat_orig ? p.dat_orig[d] : d)] = mod * 1.0e-50;
      }
      if (MODE == kModeLnprob) {
        if (ORDERED) {
          const int cnt = min(32, dv.n_data - d0);
          for (int l = 0; l < cnt; ++l) {
            const double rl = __shfl_sync(kFull, r, l);
            chi2 = fma(rl, rl, chi2);
          }
        } else {
          chi2 = fma(r, r, chi2);
        }
      }
    }
    if (MODE == kModeLnprob && !ORDERED)
      for (int off = 16; off > 0; off >>= 1) chi2 += __shfl_xor_sync(kFull, chi2, off);   // same value on every lane
  }
  if (lane != 0) return;
  if (MODE == kModeLnprob) {
    double result = -INFINITY;
    if (!(st & kWalkerPriorReject)) result = lnlike_of(chi2, st);
    deliver<MOVE>(p, k, s, m, sl, result, st);
  } else if (s.status) {
    s.status[i] = st;
  }
}

// Light curves: one warp per walker, one NODE per lane, so the three output rows (and the state rows) are
// written as 256-byte runs along the node axis.  out [W][3][Nn] = Ltot, Lprop, Ldip (/1e50); state [W][2][Nn].
__global__ void __launch_bounds__(128) reduce_curves_kernel(const __grid_constant__ Problem p, const __grid_constant__ Work k,
                                                            double* __restrict__ out, double* __restrict__ state,
                                                            int* __restrict__ status) {
  const int lane = threadIdx.x & 31;
  const int sl = (blockIdx.x * 128 + threadIdx.x) >> 5;
  if (sl >= k.W) return;
  const int i = k.slot_wid ? k.slot_wid[sl] : sl;              // the walker this slot holds
  Walker w;
  rec_load_lum(k, sl, w);
  const int Nn = p.dv.n_nodes;
  const double* row = k.ybuf + (size_t)sl * k.ws;              // node-minor: k.ns == 1
  double* o = out + (size_t)i * 3 * Nn;
  double* so = state ? state + (size_t)i * 2 * Nn : nullptr;
  for (int j = lane; j < Nn; j += 32) {
    double M, om;
    const Lum L = node_luminosity(p.sp, w, p.dv.node_t[j], p.dv.t_start, row[j], so != nullptr, M, om);
    o[j] = L.tot * 1.0e-50;            // (/1e50, funcs.py:231,236, as one multiplication: <= 1 ulp)
    o[Nn + j] = L.prop * 1.0e-50;
    o[2 * Nn + j] = L.dip * 1.0e-50;
    if (so) {
      so[j] = M;
      so[Nn + j] = om;
    }
  }
  if (lane == 0 && status) status[i] = k.status[sl];
}

// Scatter of all-gathered packs (the collective exchange): packed row i of the half -> walker P(pos0 + i).
__global__ void unpack_kernel(SplitPerm perm, int pos0, int n, int ndim, const double* __restrict__ packed,
                              double* __restrict__ coords, double* __restrict__ lnp) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const size_t w = perm_at(perm, (uint32_t)(pos0 + i));
  const double* row = packed + (size_t)i * (ndim + 1);
  for (int d = 0; d < ndim; ++d) coords[w * ndim + d] = row[d];
  lnp[w] = row[ndim];
}

// Bring this rank's replica up to date (peer-mapped ensembles): every row whose last mover was another rank is
// fetched from that rank's replica.  `m.prev_perm` is the order of the last completed step.
__global__ void sync_replica_kernel(const __grid_constant__ Move m, int n, int ndim) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n) return;
  const int home = home_before_this_step(m, w);
  if (home == m.rank) return;
  const double* src = replica_coords(m, home);
  for (int c = 0; c < ndim; ++c) m.coords[(size_t)w * ndim + c] = src[(size_t)w * ndim + c];
  m.lnp[w] = replica_lnp(m, home)[w];
}

__global__ void order_kernel(SplitPerm perm, int n, int* __restrict__ order) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < n) order[g] = (int)perm_at(perm, (uint32_t)g);
}

// Replica exchange of a tempered ensemble (mp_tempered_swap): thread j owns column j and walks the adjacent pairs
// from the hottest down, so a row can travel more than one temperature in one step, as in ptemcee.  Columns are
// independent: no thread reads another's rows.  Accepted swaps are counted per pair, one atomic per warp.
struct PtLadder {
  double beta[MP_MAX_TEMPS];
};
__global__ void pt_swap_kernel(double* __restrict__ coords, double* __restrict__ lnp, int n, int ndim, int ntemps,
                               const __grid_constant__ PtLadder lad, uint64_t seed, uint64_t step, int* __restrict__ accepted) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const bool have = j < n;
  for (int t = ntemps - 1; t >= 1; --t) {
    bool sw = false;
    if (have) {
      const size_t hot = (size_t)t * n + j, cold = hot - n;
      const double lh = lnp[hot], lc = lnp[cold];
      sw = pt_swap_accept(seed, step, (uint32_t)hot, lad.beta[t - 1], lad.beta[t], lh, lc);
      if (sw) {
        for (int c = 0; c < ndim; ++c) {
          const double x = coords[hot * ndim + c];
          coords[hot * ndim + c] = coords[cold * ndim + c];
          coords[cold * ndim + c] = x;
        }
        lnp[hot] = lc;
        lnp[cold] = lh;
      }
    }
    if (accepted) {
      const unsigned b = __ballot_sync(kFull, sw);
      if ((threadIdx.x & 31) == 0 && b) atomicAdd(accepted + t - 1, __popc(b));
    }
  }
}

}  // namespace mp

// =====================================================================================
//                                     C ABI
// =====================================================================================
using namespace mp;

struct DeviceNodes {
  DevBuf<double> node_t;
  int n_nodes = 0;
};

struct mp_handle {
  int device = 0;
  mp_model_spec model;
  Spec spec;
  mp_prior_spec prior;
  std::vector<double> grid;
  // data
  int D = 0;
  NodeProgram np;
  DeviceNodes data_nodes;
  DevBuf<double> d_y, d_yerr, d_dx, d_Dx;   // y/yerr, 1e-50/yerr, dx, dx/Dx (DataView)
  DevBuf<int> d_lo, d_orig;
  // curve node sets per stride
  std::map<int, DeviceNodes> curve_nodes;
  // staging for the host-pointer entry points
  DevBuf<double> s_theta, s_out, s_state, s_lnp;
  DevBuf<int> s_status, s_nrhs, s_cstatus;
  // A lane = a stream plus the work space the stages of a launch hand to one another.  The handle owns two
  // pipeline lanes so that the host-pointer entry points can overlap the H2D copy of one chunk with the
  // kernels of the previous one.  Device-pointer entry points run on the caller's stream, and every such
  // stream gets a lane of its own (work space only): calls on one handle from different streams -- several
  // ensembles on one dataset, a device call next to an mp_lnprob_batch_async in flight -- never share work
  // space; calls on ONE stream are ordered by the stream.
  struct Lane {
    cudaStream_t stream = nullptr;   // the handle's own lanes only (a caller's stream is never kept here, nor destroyed)
    DevBuf<unsigned long long> recs;   // kRecWords rows, each as long as the lane's capacity in walkers
    DevBuf<double> ybuf, prop, lnf;  // lnf: ln of each proposal's Hastings factor (the DE moves), indexed as prop
    DevBuf<double> kde_stats, kde_white;   // the KDE move's per-temperature factors and whitened centres (KdeMove)
    DevBuf<int> status, n_rhs, work, counters, key, hist, slot_wid;
    DevBuf<StiffRec> squeue;
    DevBuf<double> betas;        // the ladder of the tempered half-steps on this lane, and its host copy
    std::vector<double> betas_host;
    int* hint_host = nullptr;    // mapped pinned int[4]: counters[4..7] of the last large launch on this lane (see launch_eval)
    int* hint_dev = nullptr;     // the device's pointer to it
    ~Lane() {
      if (hint_host) cudaFreeHost(hint_host);
      if (stream) cudaStreamDestroy(stream);
    }
  } lanes[2];
  std::map<cudaStream_t, Lane> user_lanes;
  std::mutex user_lanes_mu;
  int sm_count = 148;
  cudaStream_t stream = nullptr;   // == lanes[0].stream
  Lane* last_lane = nullptr;       // work space of the most recent launch (mp_last_stiff_count)
  int64_t kernels_launched = 0;    // evaluation-pipeline kernels launched through this handle so far (mp_kernels_launched)
};

extern "C" int mp_create(const mp_model_spec* spec, const mp_prior_spec* prior, const double* grid,
                         int32_t G, const double* t, const double* y, const double* yerr, int32_t D,
                         int32_t device, mp_handle** out) {
  if (!spec || !grid || !out || D < 0 || (D > 0 && (!t || !y || !yerr)))
    return fail(MP_ERR_BAD_ARG, "mp_create: null pointer or negative size");
  *out = nullptr;
  NodeProgram np;
  int rc = build_node_program(grid, G, t, y, yerr, D, np);
  if (rc == MP_ERR_BAD_GRID) return fail(rc, "mp_create: grid must be strictly increasing with >= 2 nodes");
  if (rc == MP_ERR_DATA_RANGE)
    return fail(rc, "A value in x_new is outside the interpolation range.");
  if ((rc = select_device(device, "mp_create"))) return rc;
  std::unique_ptr<mp_handle> h(new mp_handle());
  h->device = device;
  h->model = *spec;
  h->spec = make_spec(*spec);
  if (prior) h->prior = *prior;
  else std::memset(&h->prior, 0, sizeof(h->prior));
  h->grid.assign(grid, grid + G);
  {
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) h->sm_count = prop.multiProcessorCount;
  }
  for (auto& L : h->lanes)
    if (cudaStreamCreateWithFlags(&L.stream, cudaStreamNonBlocking) != cudaSuccess)
      return fail(MP_ERR_CUDA, "mp_create: stream creation failed");
  h->stream = h->lanes[0].stream;
  h->D = D;
  h->np = np;
  h->data_nodes.n_nodes = (int)np.node_t.size();
  MP_CUDA(h->data_nodes.node_t.upload(np.node_t));
  MP_CUDA(h->d_y.upload(np.ys));
  MP_CUDA(h->d_yerr.upload(np.c));
  MP_CUDA(h->d_dx.upload(np.dx));
  MP_CUDA(h->d_Dx.upload(np.w));
  MP_CUDA(h->d_lo.upload(np.lo));
  MP_CUDA(h->d_orig.upload(np.order));
  *out = h.release();
  return MP_OK;
}

extern "C" void mp_destroy(mp_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  delete h;
}

extern "C" int mp_set_prior(mp_handle* h, const mp_prior_spec* prior) {
  if (!h || !prior) return fail(MP_ERR_BAD_ARG, "mp_set_prior: null pointer");
  h->prior = *prior;
  return MP_OK;
}

static int fill_problem(mp_handle* h, Problem& p, const DeviceNodes& nodes, bool with_data, int ndim, int W,
                        bool use_prior) {
  if (ndim < 6 || ndim > MP_MAX_NDIM) return fail(MP_ERR_BAD_ARG, "ndim must be 6, 7, 8 or 9");
  if (W < 0) return fail(MP_ERR_BAD_ARG, "negative walker count");
  if (use_prior && h->prior.enabled && h->prior.ndim != ndim)
    return fail(MP_ERR_BAD_ARG, "prior dimension does not match ndim");
  std::memset(&p, 0, sizeof(p));
  p.sp = h->spec;
  p.dv.n_nodes = nodes.n_nodes;
  p.dv.node_t = nodes.node_t.get();
  p.dv.t_start = h->grid[0];
  if (with_data) {
    p.dv.n_data = h->D;
    p.dv.dat_ys = h->d_y.get();
    p.dv.dat_c = h->d_yerr.get();
    p.dv.dat_dx = h->d_dx.get();
    p.dv.dat_w = h->d_Dx.get();
    p.dv.dat_lo = h->d_lo.get();
    p.dat_orig = h->d_orig.get();
  }
  p.prior_enabled = use_prior ? h->prior.enabled : 0;
  for (int i = 0; i < MP_MAX_NDIM; ++i) {
    p.lower[i] = h->prior.lower[i];
    p.upper[i] = h->prior.upper[i];
  }
  p.ndim = ndim;
  return MP_OK;
}

// lane >= 0: one of the handle's own pipeline lanes; lane < 0: the lane of the caller's stream
static int lane_for(mp_handle* h, cudaStream_t stream, int lane, mp_handle::Lane** out) {
  if (lane >= 0) {
    *out = &h->lanes[lane];
  } else {
    std::lock_guard<std::mutex> g(h->user_lanes_mu);
    *out = &h->user_lanes[stream];
  }
  h->last_lane = *out;
  return MP_OK;
}

// Walkers per slab: a launch of more walkers than this runs as several slabs one after the other, so the work
// space stays below ~1.5 GiB whatever the ensemble (10^7 walkers) or the node count (10 001 for full curves).
static int slab_walkers(int Nn) {
  const size_t per_walker = sizeof(WalkerRec) + sizeof(StiffRec) + 8 * (size_t)Nn + 16;
  const size_t n = ((size_t)3 << 29) / per_walker;
  return (int)std::min<size_t>(std::max<size_t>(n, 4096), (size_t)1 << 22);
}

// The lane's work space for a slab of S walkers.  Every array grows only, so the stride of recs is the lane's
// capacity in walkers, which an earlier launch of more walkers may have made larger than S (see Work).
static int ensure_work(mp_handle::Lane& L, int S, int Nn, int ndim_prop, Work& k) {
  MP_CUDA(L.recs.ensure((size_t)S * kRecWords));
  MP_CUDA(L.status.ensure(S));
  MP_CUDA(L.n_rhs.ensure(S));
  MP_CUDA(L.work.ensure(S));
  MP_CUDA(L.key.ensure(S));
  MP_CUDA(L.slot_wid.ensure(S));
  MP_CUDA(L.squeue.ensure(S));
  if (!L.counters.get()) {             // [8..11]: what the host was told last (never reset)
    MP_CUDA(L.counters.ensure(12));
    MP_CUDA(cudaMemset(L.counters.get(), 0, 12 * sizeof(int)));
  }
  MP_CUDA(L.hist.ensure(kOrderBuckets + 3));
  if (!L.hint_host && cudaHostAlloc((void**)&L.hint_host, 4 * sizeof(int), cudaHostAllocMapped) == cudaSuccess) {
    std::memset(L.hint_host, 0, 4 * sizeof(int));
    if (cudaHostGetDevicePointer((void**)&L.hint_dev, L.hint_host, 0) != cudaSuccess) L.hint_dev = nullptr;
  }
  MP_CUDA(L.ybuf.ensure((size_t)S * Nn));
  if (ndim_prop > 0) {
    MP_CUDA(L.prop.ensure((size_t)S * ndim_prop));
    MP_CUDA(L.lnf.ensure(S));
  }
  k.stride = (int)(L.recs.size() / kRecWords);
  k.recs = L.recs.get(); k.ybuf = L.ybuf.get(); k.status = L.status.get(); k.n_rhs = L.n_rhs.get(); k.work = L.work.get();
  k.squeue = L.squeue.get(); k.counters = L.counters.get();
  return MP_OK;
}

// One evaluation of W walkers: setup -> advance (explicit, then the stiff queue) -> reduce, slab by slab.
//   MOVE = false: parameters from d_theta [W][ndim]; results to `sink` (lnprob), `out` (model at data
//                 [W][D], or curves [W][3][Nn]) and `state` (curves, optional)
//   MOVE = true : the W movers of an ensemble-move half-step described by `mv`
//   kde         : with MOVE and the KDE move, its launches (prepared here, then run ahead of each slab)
template <int MODE, bool MOVE>
static int launch_eval(mp_handle* h, const Problem& p, const double* d_theta, int W, Sink sink, double* out, double* state,
                       const Move* mv, cudaStream_t stream, int lane = -1, const KdeMove* kde = nullptr) {
  if (W == 0) return MP_OK;
  mp_handle::Lane* Lp = nullptr;
  lane_for(h, stream, lane, &Lp);
  const int Nn = p.dv.n_nodes, D = p.dv.n_data, ndim = p.ndim;
  const int S = std::min(W, slab_walkers(Nn));
  Work k;
  std::memset(&k, 0, sizeof(k));
  int rc = ensure_work(*Lp, S, Nn, MOVE ? ndim : 0, k);
  if (rc) return rc;
  Move m;
  if (MOVE) m = *mv;
  else std::memset(&m, 0, sizeof(m));
  const bool coop = Nn > 64 || MODE == kModeCurves;   // by the DATASET only: a walker's lnprob never depends on the batch it is in
  // (ybuf holds S * Nn values: its walker-minor stride is this launch's slab, not the lane's record capacity, which an
  // earlier launch of more walkers on fewer nodes may have made larger)
  k.ws = coop ? (size_t)Nn : 1;
  k.ns = coop ? 1 : (size_t)S;
  KdeMove km;
  if (MOVE && kde) {
    km = *kde;
    MP_CUDA(Lp->kde_stats.ensure((size_t)km.T * kKdeStats));
    MP_CUDA(Lp->kde_white.ensure((size_t)km.T * km.M * km.ndim));
    km.stats = Lp->kde_stats.get();
    km.white = Lp->kde_white.get();
    if ((rc = kde_prepare(km, stream))) return rc;
    h->kernels_launched += 1;
  }
  for (int i0 = 0; i0 < W; i0 += S) {
    const int n = std::min(S, W - i0);
    k.W = n;
    Move ms = m;
    if (MOVE) {
      if (ms.active) ms.active += i0;
      else ms.mover0 += i0;     // (a tempered slab may span temperatures: offset the mover, not the position)
      ms.prop = Lp->prop.get();
      ms.lnf = Lp->lnf.get();
      if (ms.pack_out) ms.pack_out += (size_t)i0 * (ndim + 1);
    }
    Sink sk = sink;
    if (sk.lnp) sk.lnp += i0;
    if (sk.status) sk.status += i0;
    if (sk.n_rhs) sk.n_rhs += i0;
    MP_CUDA(cudaMemsetAsync(k.counters, 0, 8 * sizeof(int), stream));
    // (a sharded move that reads its rows from peer replicas forms its proposals inside the setup kernel, where the
    // remote reads hide behind the other threads' arithmetic: in a kernel of their own they cost 0.07 ms per half-step)
    // A tight ensemble gains nothing from the ordering and pays two launches for it.  How far an ensemble reaches in the
    // ordering's bins is measured by every large launch's setup kernel; the four numbers travel to pinned host memory
    // behind the launch and are read HERE, unsynchronised, by the next launch on the same lane (a chain's ensemble moves
    // slowly): inside kTightMdBins x kTightEpsBins the walkers are taken as they come.  Results do not depend on it (a
    // walker's arithmetic is the same in any slot).
    bool ordered = n >= kOrderMinWalkers && Nn > 0 && !(MOVE && m.n_peers > 0);
    k.track = (ordered && Lp->hint_dev) ? 1 : 0;
    k.hint = Lp->hint_dev;
    if (ordered && Lp->hint_host) {
      const volatile int* e = Lp->hint_host;
      const int e0 = e[0], e1 = e[1], e2 = e[2], e3 = e[3];
      if (e0 > 0 && e0 + e1 - 257 <= kTightMdBins && e2 + e3 - 33 <= kTightEpsBins) ordered = false;
    }
    if (MOVE && kde) {
      if ((rc = kde_propose(km, ms.mover0, n, ms.prop, ms.lnf, stream))) return rc;
      h->kernels_launched += 1;
    }
    const double* th0 = MOVE ? nullptr : d_theta + (size_t)i0 * ndim;
    k.key = Lp->key.get();
    k.hist = Lp->hist.get();
    k.slot_wid = ordered ? Lp->slot_wid.get() : nullptr;
    if (ordered) {
      // slots in key order: keys + histogram (MOVE: and the proposals), scan, scatter -- then the setup runs per slot
      MP_CUDA(cudaMemsetAsync(k.hist, 0, (kOrderBuckets + 3) * sizeof(int), stream));
      order_key_kernel<MOVE><<<(n + 127) / 128, 128, 0, stream>>>(p, k, th0, ms);
      order_scatter_kernel<<<(n + 1023) / 1024, 1024, 0, stream>>>(n, k.key, k.hist, k.slot_wid);
      h->kernels_launched += 2;
    }
    setup_kernel<MOVE><<<(n + 127) / 128, 128, 0, stream>>>(p, k, th0, ms);
    // small launches: 32-thread blocks spread the warps over more SMs
    if (Nn == 0) {
      // (a handle without data -- lnprior-only callers: nothing to integrate, lnlike = -0.5 * 0)
    } else if (n <= h->sm_count * 64 * 4) {
      advance_kernel<false, 32><<<std::min((n + 31) / 32, h->sm_count * MP_MIN_BLOCKS_32), 32, 0, stream>>>(p, k);
      advance_kernel<true, 32><<<std::min((n + 31) / 32, h->sm_count * MP_STIFF_MIN_WARPS), 32, 0, stream>>>(p, k);
    } else {
      advance_kernel<false, 64><<<std::min((n + 63) / 64, h->sm_count * MP_MIN_BLOCKS_64), 64, 0, stream>>>(p, k);
      if (n >= kStiffWideMinWalkers)
        advance_kernel<true, 64, kStiffWarpsWide><<<std::min((n + 63) / 64, h->sm_count * kStiffWarpsWide / 2), 64, 0, stream>>>(p, k);
      else
        advance_kernel<true, 64><<<std::min((n + 63) / 64, h->sm_count * MP_STIFF_MIN_WARPS / 2), 64, 0, stream>>>(p, k);
    }
    if (MODE == kModeCurves) {
      reduce_curves_kernel<<<(n + 3) / 4, 128, 0, stream>>>(p, k, out + (size_t)i0 * 3 * Nn,
                                                            state ? state + (size_t)i0 * 2 * Nn : nullptr, sk.status);
    } else {
      double* o = out ? out + (size_t)i0 * D : nullptr;
      if (coop) reduce_coop_kernel<MODE, MOVE, false><<<(n + 3) / 4, 128, 0, stream>>>(p, k, sk, o, ms);
      else if (n <= kCoopSmallWalkers) reduce_coop_kernel<MODE, MOVE, true><<<(n + 3) / 4, 128, 0, stream>>>(p, k, sk, o, ms);
      else reduce_rows_kernel<MODE, MOVE><<<(n + 63) / 64, 64, 0, stream>>>(p, k, sk, o, ms);
    }
    h->kernels_launched += (Nn == 0) ? 2 : 4;      // setup, advance (explicit), advance (implicit), reduce
    MP_CUDA(cudaGetLastError());
  }
  return MP_OK;
}

extern "C" int64_t mp_kernels_launched(const mp_handle* h) { return h ? h->kernels_launched : 0; }

extern "C" int mp_lnprob_batch_device(mp_handle* h, const double* d_theta, int32_t W, int32_t ndim,
                                      double* d_lnp, int32_t* d_status, int32_t* d_n_rhs, void* stream) {
  if (!h || (W > 0 && (!d_theta || !d_lnp))) return fail(MP_ERR_BAD_ARG, "mp_lnprob_batch_device: null pointer");
  MP_CUDA(cudaSetDevice(h->device));
  Problem p;
  int rc = fill_problem(h, p, h->data_nodes, true, ndim, W, true);
  if (rc) return rc;
  return launch_eval<kModeLnprob, false>(h, p, d_theta, W, Sink{d_lnp, d_status, d_n_rhs}, nullptr, nullptr, nullptr,
                                         (cudaStream_t)stream);
}

// One full wave of the explicit integrator: its resident 64-thread blocks on every SM.
static int wave_walkers(const mp_handle* h) { return h->sm_count * MP_MIN_BLOCKS_64 * 64; }

extern "C" int mp_lnprob_batch_async(mp_handle* h, const double* theta, int32_t W, int32_t ndim, double* lnp,
                                     int32_t* status, int32_t* n_rhs) {
  if (!h || (W > 0 && (!theta || !lnp))) return fail(MP_ERR_BAD_ARG, "mp_lnprob_batch: null pointer");
  if (ndim < 6 || ndim > MP_MAX_NDIM) return fail(MP_ERR_BAD_ARG, "ndim must be 6, 7, 8 or 9");
  if (W == 0) return MP_OK;
  MP_CUDA(cudaSetDevice(h->device));
  MP_CUDA(h->s_theta.ensure((size_t)W * MP_MAX_NDIM));
  MP_CUDA(h->s_lnp.ensure(W));
  MP_CUDA(h->s_status.ensure(W));
  MP_CUDA(h->s_nrhs.ensure(W));
  double* const s_theta = h->s_theta.get();
  double* const s_lnp = h->s_lnp.get();
  int* const s_status = h->s_status.get();
  int* const s_nrhs = h->s_nrhs.get();
  // Large batches go through in chunks of a few waves on two alternating lanes: the H2D copy of chunk
  // k+1 and the D2H copy of chunk k-1 overlap the kernels of chunk k (when the caller's buffers are
  // pinned; pageable buffers still work, the copies just serialise).
  const int wave = 4 * wave_walkers(h);
  const int chunk = (W <= wave + wave / 2) ? W : wave;
  Problem p;
  int rc = fill_problem(h, p, h->data_nodes, true, ndim, W, true);
  if (rc) return rc;
  int k = 0;
  for (int c0 = 0; c0 < W; c0 += chunk, ++k) {
    const int lane = k & 1;
    cudaStream_t st = h->lanes[lane].stream;
    int n = W - c0;
    if (n > chunk + chunk / 2) n = chunk;          // the last chunk absorbs a remainder below half a chunk
    MP_CUDA(cudaMemcpyAsync(s_theta + (size_t)c0 * ndim, theta + (size_t)c0 * ndim, (size_t)n * ndim * sizeof(double),
                            cudaMemcpyHostToDevice, st));
    if ((rc = launch_eval<kModeLnprob, false>(h, p, s_theta + (size_t)c0 * ndim, n,
                                              Sink{s_lnp + c0, s_status + c0, s_nrhs + c0}, nullptr, nullptr, nullptr,
                                              st, lane)))
      return rc;
    MP_CUDA(cudaMemcpyAsync(lnp + c0, s_lnp + c0, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (status) MP_CUDA(cudaMemcpyAsync(status + c0, s_status + c0, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, st));
    if (n_rhs) MP_CUDA(cudaMemcpyAsync(n_rhs + c0, s_nrhs + c0, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, st));
    if (n != chunk) break;
  }
  return MP_OK;
}

extern "C" int mp_synchronize(mp_handle* h) {
  if (!h) return fail(MP_ERR_BAD_ARG, "mp_synchronize: null handle");
  MP_CUDA(cudaSetDevice(h->device));
  MP_CUDA(cudaStreamSynchronize(h->lanes[0].stream));
  MP_CUDA(cudaStreamSynchronize(h->lanes[1].stream));
  return MP_OK;
}

extern "C" int mp_lnprob_batch(mp_handle* h, const double* theta, int32_t W, int32_t ndim, double* lnp,
                               int32_t* status, int32_t* n_rhs) {
  const int rc = mp_lnprob_batch_async(h, theta, W, ndim, lnp, status, n_rhs);
  if (rc) return rc;
  return (W > 0) ? mp_synchronize(h) : MP_OK;
}

extern "C" int mp_model_at_data(mp_handle* h, const double* pars, int32_t W, int32_t ndim, double* out,
                                int32_t* status) {
  if (!h || (W > 0 && (!pars || !out))) return fail(MP_ERR_BAD_ARG, "mp_model_at_data: null pointer");
  if (h->D == 0) return fail(MP_ERR_NO_DATA, "mp_model_at_data: handle has no data times");
  if (W == 0) return MP_OK;
  MP_CUDA(cudaSetDevice(h->device));
  Problem p;
  int rc = fill_problem(h, p, h->data_nodes, true, ndim, W, false);
  if (rc) return rc;
  p.sp.unlog_mask = 0;  // model_lum takes physical parameters
  MP_CUDA(h->s_theta.ensure((size_t)W * MP_MAX_NDIM));
  MP_CUDA(h->s_out.ensure((size_t)W * h->D));
  MP_CUDA(h->s_cstatus.ensure(W));
  MP_CUDA(cudaMemcpyAsync(h->s_theta.get(), pars, (size_t)W * ndim * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  if ((rc = launch_eval<kModeModelAtData, false>(h, p, h->s_theta.get(), W, Sink{nullptr, h->s_cstatus.get(), nullptr},
                                                 h->s_out.get(), nullptr, nullptr, h->stream, 0)))
    return rc;
  MP_CUDA(cudaMemcpyAsync(out, h->s_out.get(), (size_t)W * h->D * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (status) MP_CUDA(cudaMemcpyAsync(status, h->s_cstatus.get(), (size_t)W * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  MP_CUDA(cudaStreamSynchronize(h->stream));
  return MP_OK;
}

static int curve_node_set(mp_handle* h, int stride, DeviceNodes** out) {
  if (stride < 1) stride = 1;
  auto it = h->curve_nodes.find(stride);
  if (it == h->curve_nodes.end()) {
    std::vector<double> nt;
    std::vector<int> gi;
    build_curve_nodes(h->grid.data(), (int)h->grid.size(), stride, nt, gi);
    DeviceNodes dn;
    dn.n_nodes = (int)nt.size();
    MP_CUDA(dn.node_t.upload(nt));
    it = h->curve_nodes.emplace(stride, std::move(dn)).first;
  }
  *out = &it->second;
  return MP_OK;
}

extern "C" int32_t mp_curve_nodes(const mp_handle* h, int32_t node_stride) {
  if (!h) return 0;
  if (node_stride < 1) node_stride = 1;
  const int G = (int)h->grid.size();
  int n = (G + node_stride - 1) / node_stride;
  if ((n - 1) * node_stride != G - 1) ++n;
  return n;
}

static int curves_on(mp_handle* h, const double* d_pars, int32_t W, int32_t ndim, int32_t node_stride, double* d_out,
                     double* d_state, int32_t* d_status, cudaStream_t stream, int lane) {
  DeviceNodes* dn = nullptr;
  int rc = curve_node_set(h, node_stride, &dn);
  if (rc) return rc;
  Problem p;
  if ((rc = fill_problem(h, p, *dn, false, ndim, W, false))) return rc;
  p.sp.unlog_mask = 0;
  return launch_eval<kModeCurves, false>(h, p, d_pars, W, Sink{nullptr, d_status, nullptr}, d_out, d_state, nullptr, stream, lane);
}

extern "C" int mp_model_curves_device(mp_handle* h, const double* d_pars, int32_t W, int32_t ndim,
                                      int32_t node_stride, double* d_out, double* d_state,
                                      int32_t* d_status, void* stream) {
  if (!h || (W > 0 && (!d_pars || !d_out))) return fail(MP_ERR_BAD_ARG, "mp_model_curves_device: null pointer");
  MP_CUDA(cudaSetDevice(h->device));
  return curves_on(h, d_pars, W, ndim, node_stride, d_out, d_state, d_status, (cudaStream_t)stream, -1);
}

extern "C" int mp_model_curves(mp_handle* h, const double* pars, int32_t W, int32_t ndim, int32_t node_stride,
                               double* out, double* state, int32_t* status) {
  if (!h || (W > 0 && (!pars || !out))) return fail(MP_ERR_BAD_ARG, "mp_model_curves: null pointer");
  if (ndim < 6 || ndim > MP_MAX_NDIM) return fail(MP_ERR_BAD_ARG, "ndim must be 6, 7, 8 or 9");
  if (W == 0) return MP_OK;
  MP_CUDA(cudaSetDevice(h->device));
  const size_t Gs = (size_t)mp_curve_nodes(h, node_stride);
  MP_CUDA(h->s_theta.ensure((size_t)W * MP_MAX_NDIM));
  MP_CUDA(h->s_out.ensure((size_t)W * 3 * Gs));
  if (state) MP_CUDA(h->s_state.ensure((size_t)W * 2 * Gs));
  int* d_status = nullptr;
  if (status) {
    MP_CUDA(h->s_cstatus.ensure(W));
    d_status = h->s_cstatus.get();
  }
  MP_CUDA(cudaMemcpyAsync(h->s_theta.get(), pars, (size_t)W * ndim * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  int rc = curves_on(h, h->s_theta.get(), W, ndim, node_stride, h->s_out.get(), state ? h->s_state.get() : nullptr, d_status,
                     h->stream, 0);
  if (!rc) {
    cudaMemcpyAsync(out, h->s_out.get(), (size_t)W * 3 * Gs * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
    if (state) cudaMemcpyAsync(state, h->s_state.get(), (size_t)W * 2 * Gs * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
    if (status) cudaMemcpyAsync(status, d_status, (size_t)W * sizeof(int), cudaMemcpyDeviceToHost, h->stream);
    cudaError_t e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) rc = fail(MP_ERR_CUDA, std::string("mp_model_curves: ") + cudaGetErrorString(e));
  }
  return rc;
}

static int fill_move_problem(mp_handle* h, Problem& p, int ndim, int n_active) {
  return fill_problem(h, p, h->data_nodes, true, ndim, n_active, true);
}

extern "C" int mp_stretch_half_step(mp_handle* h, double* d_coords, double* d_lnp, int32_t nwalkers,
                                    int32_t ndim, const int32_t* d_active, int32_t n_active,
                                    const int32_t* d_complement, int32_t n_complement, double a,
                                    uint64_t seed, uint64_t step, int32_t* d_accepted, int32_t* d_n_rhs,
                                    void* stream) {
  if (!h || !d_coords || !d_lnp || !d_active || !d_complement || n_active < 0 || n_complement <= 0 ||
      nwalkers <= 0)
    return fail(MP_ERR_BAD_ARG, "mp_stretch_half_step: null pointer or empty set");
  MP_CUDA(cudaSetDevice(h->device));
  Problem p;
  int rc = fill_move_problem(h, p, ndim, n_active);
  if (rc) return rc;
  Move m;
  std::memset(&m, 0, sizeof(m));
  m.coords = d_coords;
  m.lnp = d_lnp;
  m.active = d_active;
  m.complement = d_complement;
  m.n_complement = n_complement;
  m.a = a;
  m.seed = seed;
  m.step = step;
  m.accepted = d_accepted;
  m.n_rhs = d_n_rhs;
  return launch_eval<kModeLnprob, true>(h, p, nullptr, n_active, Sink{nullptr, nullptr, nullptr}, nullptr, nullptr, &m,
                                        (cudaStream_t)stream);
}

static int check_ensemble(const mp_ensemble* e, const char* who) {
  if (!e || !e->coords || !e->lnp) return fail(MP_ERR_BAD_ARG, std::string(who) + ": null ensemble / coords / lnp");
  if (e->nwalkers < 2 || (e->nwalkers & 1)) return fail(MP_ERR_BAD_ARG, std::string(who) + ": nwalkers must be even");
  if (e->world < 1 || e->rank < 0 || e->rank >= e->world || (e->nwalkers / 2) % e->world)
    return fail(MP_ERR_BAD_ARG, std::string(who) + ": half-ensemble does not split evenly over the ranks");
  if (e->n_peers < 0 || e->n_peers > MP_MAX_PEERS) return fail(MP_ERR_BAD_ARG, std::string(who) + ": bad n_peers");
  return MP_OK;
}

// The pull side of a peer-mapped ensemble: replicas, last step's order, whether the replicas are in sync.
static int fill_pull(const mp_ensemble* e, uint64_t step, Move& m, const char* who) {
  m.n_peers = e->n_peers;
  m.rank = e->rank;
  m.half = e->nwalkers / 2;
  m.n_mine = m.half / e->world;
  if (e->n_peers == 0) return MP_OK;
  if (e->n_peers != e->world - 1) return fail(MP_ERR_BAD_ARG, std::string(who) + ": n_peers must be 0 or world - 1");
  if (step < e->synced_step) return fail(MP_ERR_BAD_ARG, std::string(who) + ": step lies before synced_step");
  for (int r = 0; r < e->n_peers; ++r) {
    if (!e->peer_coords[r] || !e->peer_lnp[r]) return fail(MP_ERR_BAD_ARG, std::string(who) + ": null peer replica");
    m.peer_coords[r] = e->peer_coords[r];
    m.peer_lnp[r] = e->peer_lnp[r];
  }
  m.synced = step == e->synced_step;
  if (!m.synced) m.prev_perm = make_split_perm(e->nwalkers, e->seed, step - 1, e->randomize_split);
  return MP_OK;
}

extern "C" int mp_ensemble_sync(const mp_ensemble* e, uint64_t step, void* stream) {
  int rc = check_ensemble(e, "mp_ensemble_sync");
  if (rc) return rc;
  Move m;
  std::memset(&m, 0, sizeof(m));
  m.coords = e->coords;
  m.lnp = e->lnp;
  if ((rc = fill_pull(e, step, m, "mp_ensemble_sync"))) return rc;
  if (e->n_peers == 0 || m.synced) return MP_OK;
  sync_replica_kernel<<<(e->nwalkers + 255) / 256, 256, 0, (cudaStream_t)stream>>>(m, e->nwalkers, e->ndim);
  MP_CUDA(cudaGetLastError());
  return MP_OK;
}

// The stretch move of scale a as an mp_move (the move of mp_ensemble_half_step / mp_tempered_half_step).
static mp_move stretch_move(double a) {
  mp_move mv;
  std::memset(&mv, 0, sizeof(mv));
  mv.kind = MP_MOVE_STRETCH;
  mv.weight = 1.0;
  mv.a = a;
  return mv;
}

// The host-side checks of a list of moves for the (checked) ensemble e, halves per temperature of nwalkers/2 (see mp_move).
static int check_moves(const mp_move* moves, int32_t n_moves, const mp_ensemble* e, const char* who) {
  const int half = e->nwalkers / 2;
  const std::string w(who);
  if (!moves || n_moves < 1 || n_moves > MP_MAX_MOVES)
    return fail(MP_ERR_BAD_ARG, w + ": moves must be non-null and n_moves in [1, MP_MAX_MOVES]");
  double total = 0.0;
  for (int k = 0; k < n_moves; ++k) {
    const mp_move& mv = moves[k];
    if (!(mv.weight >= 0.0 && std::isfinite(mv.weight))) return fail(MP_ERR_BAD_ARG, w + ": move weights must be finite and >= 0");
    total += mv.weight;
    int need = 1;
    if (mv.kind == MP_MOVE_STRETCH) {
      if (!(mv.a > 1.0 && std::isfinite(mv.a))) return fail(MP_ERR_BAD_ARG, w + ": stretch move needs a > 1");
    } else if (mv.kind == MP_MOVE_DE) {
      if (!(mv.sigma >= 0.0 && mv.sigma < 1.0)) return fail(MP_ERR_BAD_ARG, w + ": DE move needs 0 <= sigma < 1");
      if (!(mv.gamma0 >= 0.0 && std::isfinite(mv.gamma0))) return fail(MP_ERR_BAD_ARG, w + ": DE move needs gamma0 >= 0");
      need = 2;
    } else if (mv.kind == MP_MOVE_DE_SNOOKER) {
      if (!(mv.gammas > 0.0 && std::isfinite(mv.gammas))) return fail(MP_ERR_BAD_ARG, w + ": snooker move needs gammas > 0");
      need = 3;
    } else if (mv.kind == MP_MOVE_KDE) {
      if (!(mv.gamma0 >= 0.0 && std::isfinite(mv.gamma0)))
        return fail(MP_ERR_BAD_ARG, w + ": KDE move needs a bandwidth factor gamma0 >= 0 (0: Scott's rule)");
      if (mv.weight > 0.0 && (e->world != 1 || e->n_peers != 0 || e->pack_out))
        return fail(MP_ERR_BAD_ARG, w + ": the KDE move runs on one rank (world 1, no peers, no pack_out)");
      need = e->ndim + 1;
    } else {
      return fail(MP_ERR_BAD_ARG, w + ": unknown move kind");
    }
    if (mv.weight > 0.0 && half < need)
      return fail(MP_ERR_BAD_ARG, w + ": a half of the ensemble holds fewer walkers than the move's partners");
  }
  if (!(total > 0.0 && std::isfinite(total))) return fail(MP_ERR_BAD_ARG, w + ": move weights must have a positive, finite sum");
  return MP_OK;
}

// The move MCMC step `step` runs (choose_move: one per step, the same for both half-steps and every temperature).
static const mp_move& pick_move(const mp_move* moves, int32_t n_moves, uint64_t seed, uint64_t step) {
  double w[MP_MAX_MOVES];
  for (int k = 0; k < n_moves; ++k) w[k] = moves[k].weight;
  return moves[choose_move(seed, step, w, n_moves)];
}

// The move of this rank's share of half `split` at MCMC step `step` (everything but the pull side).
static void fill_ensemble_move(const mp_ensemble* e, uint64_t step, int split, const mp_move& mv, Move& m) {
  const int half = e->nwalkers / 2, n_mine = half / e->world;
  std::memset(&m, 0, sizeof(m));
  m.coords = e->coords;
  m.lnp = e->lnp;
  m.perm = make_split_perm(e->nwalkers, e->seed, step, e->randomize_split);
  m.pos0 = split * half + e->rank * n_mine;
  m.cpos0 = (1 - split) * half;
  m.n_complement = half;
  m.kind = mv.kind;
  m.a = mv.a;
  m.g0 = mv.gamma0 > 0.0 ? mv.gamma0 : 2.38 / std::sqrt(2.0 * e->ndim);
  m.s3 = mv.sigma * std::sqrt(3.0);
  m.gammas = mv.gammas;
  m.seed = e->seed;
  m.step = 2 * step + (uint64_t)split;
  m.accepted = e->accepted;
  m.status = e->status;
  m.n_rhs = e->n_rhs;
  m.split = split;
  m.pack_out = e->pack_out;
  if (e->bad_rows && e->bad_count && e->bad_capacity > 0) {
    m.bad_rows = e->bad_rows;
    m.bad_count = e->bad_count;
    m.bad_capacity = e->bad_capacity;
  }
}

// The KDE launches of half `split` at MCMC step `step` over ntemps temperatures of the ensemble e (see KdeMove).
static KdeMove kde_move(const mp_ensemble* e, int ntemps, const mp_move& mv, const Move& m) {
  KdeMove k;
  std::memset(&k, 0, sizeof(k));
  k.coords = e->coords;
  k.perm = m.perm;
  k.pos0 = m.pos0;
  k.cpos0 = m.cpos0;
  k.T = ntemps;
  k.n = e->nwalkers;
  k.ndim = e->ndim;
  k.M = std::min(m.n_complement, MP_KDE_MAX_CENTRES);
  k.h = mv.gamma0 > 0.0 ? mv.gamma0 : std::pow((double)k.M, -1.0 / (e->ndim + 4));
  k.seed = m.seed;
  k.hs = m.step;
  return k;
}

// One half-step of a (checked) ensemble with move `mv`: mp_ensemble_half_step and mp_ensemble_moves_half_step.
static int ensemble_half_step(mp_handle* h, const mp_ensemble* e, const mp_move& mv, uint64_t step, int32_t split,
                              void* stream, const char* who) {
  MP_CUDA(cudaSetDevice(h->device));
  const int n_mine = e->nwalkers / 2 / e->world;
  Problem p;
  int rc = fill_move_problem(h, p, e->ndim, n_mine);
  if (rc) return rc;
  Move m;
  fill_ensemble_move(e, step, split, mv, m);
  if ((rc = fill_pull(e, step, m, who))) return rc;
  const KdeMove km = kde_move(e, 1, mv, m);
  return launch_eval<kModeLnprob, true>(h, p, nullptr, n_mine, Sink{nullptr, nullptr, nullptr}, nullptr, nullptr, &m,
                                        (cudaStream_t)stream, -1, mv.kind == MP_MOVE_KDE ? &km : nullptr);
}

extern "C" int mp_ensemble_half_step(mp_handle* h, const mp_ensemble* e, uint64_t step, int32_t split, void* stream) {
  if (!h) return fail(MP_ERR_BAD_ARG, "mp_ensemble_half_step: null handle");
  int rc = check_ensemble(e, "mp_ensemble_half_step");
  if (rc) return rc;
  if (split != 0 && split != 1) return fail(MP_ERR_BAD_ARG, "mp_ensemble_half_step: split must be 0 or 1");
  return ensemble_half_step(h, e, stretch_move(e->a), step, split, stream, "mp_ensemble_half_step");
}

extern "C" int mp_ensemble_moves_half_step(mp_handle* h, const mp_ensemble* e, const mp_move* moves, int32_t n_moves,
                                           uint64_t step, int32_t split, void* stream) {
  const char* who = "mp_ensemble_moves_half_step";
  int rc = check_ensemble(e, who);
  if (rc) return rc;
  if (split != 0 && split != 1) return fail(MP_ERR_BAD_ARG, std::string(who) + ": split must be 0 or 1");
  if ((rc = check_moves(moves, n_moves, e, who))) return rc;
  if (!h) return fail(MP_ERR_BAD_ARG, std::string(who) + ": null handle");
  return ensemble_half_step(h, e, pick_move(moves, n_moves, e->seed, step), step, split, stream, who);
}

// ---- parallel tempering ----------------------------------------------------------------------------
// Both tempered entry points check everything on the host, before any device work: a bad ladder is
// MP_ERR_BAD_ARG on a machine without a GPU too.
static int check_tempered(const mp_ensemble* e, int32_t ntemps, const double* betas, const char* who) {
  int rc = check_ensemble(e, who);
  if (rc) return rc;
  const std::string w(who);
  if (e->world != 1 || e->n_peers != 0 || e->pack_out)
    return fail(MP_ERR_BAD_ARG, w + ": a tempered ensemble runs on one rank (world 1, no peers, no pack_out)");
  if (e->ndim < 1 || e->ndim > MP_MAX_NDIM) return fail(MP_ERR_BAD_ARG, w + ": bad ndim");
  if (ntemps < 1 || ntemps > MP_MAX_TEMPS || !betas)
    return fail(MP_ERR_BAD_ARG, w + ": ntemps must be in [1, MP_MAX_TEMPS] and betas non-null");
  if ((int64_t)ntemps * e->nwalkers >= ((int64_t)1 << 31))
    return fail(MP_ERR_BAD_ARG, w + ": ntemps * nwalkers must be below 2^31");
  if (betas[0] != 1.0) return fail(MP_ERR_BAD_ARG, w + ": betas[0] must be 1");
  for (int t = 1; t < ntemps; ++t)
    if (!(betas[t] > 0.0 && betas[t] < betas[t - 1]))     // (NaN fails too)
      return fail(MP_ERR_BAD_ARG, w + ": betas must be strictly decreasing and positive");
  return MP_OK;
}

// The ladder a lane's tempered half-steps read: copied in stream order, and only when it differs from the last one.
static int upload_ladder(mp_handle::Lane& L, int ntemps, const double* betas, cudaStream_t stream) {
  if (L.betas_host.size() == (size_t)ntemps && std::equal(betas, betas + ntemps, L.betas_host.begin())) return MP_OK;
  MP_CUDA(L.betas.ensure(MP_MAX_TEMPS));
  L.betas_host.clear();
  MP_CUDA(cudaMemcpyAsync(L.betas.get(), betas, (size_t)ntemps * sizeof(double), cudaMemcpyHostToDevice, stream));
  L.betas_host.assign(betas, betas + ntemps);
  return MP_OK;
}

// One half-step of every temperature of a (checked) tempered ensemble with move `mv`: mp_tempered_half_step and
// mp_tempered_moves_half_step.
static int tempered_half_step(mp_handle* h, const mp_ensemble* e, int32_t ntemps, const double* betas, const mp_move& mv,
                              uint64_t step, int32_t split, void* stream) {
  int rc;
  MP_CUDA(cudaSetDevice(h->device));
  const cudaStream_t s = (cudaStream_t)stream;
  const int half = e->nwalkers / 2, n_movers = ntemps * half;
  Problem p;
  if ((rc = fill_move_problem(h, p, e->ndim, n_movers))) return rc;
  mp_handle::Lane* L = nullptr;
  lane_for(h, s, -1, &L);
  if ((rc = upload_ladder(*L, ntemps, betas, s))) return rc;
  Move m;
  fill_ensemble_move(e, step, split, mv, m);
  m.rank = 0;
  m.half = m.n_mine = half;
  m.betas = L->betas.get();
  const KdeMove km = kde_move(e, ntemps, mv, m);
  return launch_eval<kModeLnprob, true>(h, p, nullptr, n_movers, Sink{nullptr, nullptr, nullptr}, nullptr, nullptr, &m, s, -1,
                                        mv.kind == MP_MOVE_KDE ? &km : nullptr);
}

extern "C" int mp_tempered_half_step(mp_handle* h, const mp_ensemble* e, int32_t ntemps, const double* betas, uint64_t step,
                                     int32_t split, void* stream) {
  int rc = check_tempered(e, ntemps, betas, "mp_tempered_half_step");
  if (rc) return rc;
  if (!h) return fail(MP_ERR_BAD_ARG, "mp_tempered_half_step: null handle");
  if (split != 0 && split != 1) return fail(MP_ERR_BAD_ARG, "mp_tempered_half_step: split must be 0 or 1");
  return tempered_half_step(h, e, ntemps, betas, stretch_move(e->a), step, split, stream);
}

extern "C" int mp_tempered_moves_half_step(mp_handle* h, const mp_ensemble* e, int32_t ntemps, const double* betas,
                                           const mp_move* moves, int32_t n_moves, uint64_t step, int32_t split, void* stream) {
  const char* who = "mp_tempered_moves_half_step";
  int rc = check_tempered(e, ntemps, betas, who);
  if (rc) return rc;
  if (split != 0 && split != 1) return fail(MP_ERR_BAD_ARG, std::string(who) + ": split must be 0 or 1");
  if ((rc = check_moves(moves, n_moves, e, who))) return rc;
  if (!h) return fail(MP_ERR_BAD_ARG, std::string(who) + ": null handle");
  return tempered_half_step(h, e, ntemps, betas, pick_move(moves, n_moves, e->seed, step), step, split, stream);
}

// ---- sequential Monte Carlo: one ensemble at one inverse temperature --------------------------------------------
// The tempered half-step with the ladder {beta}; unlike a tempered ensemble's, that one beta need not be 1.
extern "C" int mp_annealed_moves_half_step(mp_handle* h, const mp_ensemble* e, double beta, const mp_move* moves,
                                           int32_t n_moves, uint64_t step, int32_t split, void* stream) {
  const char* who = "mp_annealed_moves_half_step";
  int rc = check_ensemble(e, who);
  if (rc) return rc;
  const std::string w(who);
  if (e->world != 1 || e->n_peers != 0 || e->pack_out)
    return fail(MP_ERR_BAD_ARG, w + ": an annealed ensemble runs on one rank (world 1, no peers, no pack_out)");
  if (e->ndim < 1 || e->ndim > MP_MAX_NDIM) return fail(MP_ERR_BAD_ARG, w + ": bad ndim");
  if (!(beta > 0.0 && beta <= 1.0)) return fail(MP_ERR_BAD_ARG, w + ": beta must lie in (0, 1]");   // (NaN fails too)
  if (split != 0 && split != 1) return fail(MP_ERR_BAD_ARG, w + ": split must be 0 or 1");
  if ((rc = check_moves(moves, n_moves, e, who))) return rc;
  if (!h) return fail(MP_ERR_BAD_ARG, w + ": null handle");
  return tempered_half_step(h, e, 1, &beta, pick_move(moves, n_moves, e->seed, step), step, split, stream);
}

extern "C" int mp_tempered_swap(const mp_ensemble* e, int32_t ntemps, const double* betas, uint64_t step,
                                int32_t* d_swap_accepted, void* stream) {
  int rc = check_tempered(e, ntemps, betas, "mp_tempered_swap");
  if (rc) return rc;
  if (ntemps == 1) return MP_OK;
  PtLadder lad;
  std::memset(&lad, 0, sizeof(lad));
  std::memcpy(lad.beta, betas, (size_t)ntemps * sizeof(double));
  pt_swap_kernel<<<(e->nwalkers + 127) / 128, 128, 0, (cudaStream_t)stream>>>(e->coords, e->lnp, e->nwalkers, e->ndim, ntemps,
                                                                              lad, e->seed, step, d_swap_accepted);
  MP_CUDA(cudaGetLastError());
  return MP_OK;
}

extern "C" int mp_ensemble_unpack(const mp_ensemble* e, uint64_t step, int32_t split, const double* d_packed, void* stream) {
  int rc = check_ensemble(e, "mp_ensemble_unpack");
  if (rc) return rc;
  if (!d_packed || (split != 0 && split != 1)) return fail(MP_ERR_BAD_ARG, "mp_ensemble_unpack: bad argument");
  const int half = e->nwalkers / 2;
  const SplitPerm perm = make_split_perm(e->nwalkers, e->seed, step, e->randomize_split);
  unpack_kernel<<<(half + 255) / 256, 256, 0, (cudaStream_t)stream>>>(perm, split * half, half, e->ndim, d_packed, e->coords, e->lnp);
  MP_CUDA(cudaGetLastError());
  return MP_OK;
}

extern "C" int mp_ensemble_order(int32_t nwalkers, uint64_t seed, uint64_t step, int32_t randomize_split,
                                 int32_t* d_order, void* stream) {
  if (nwalkers <= 0 || !d_order) return fail(MP_ERR_BAD_ARG, "mp_ensemble_order: bad argument");
  const SplitPerm perm = make_split_perm(nwalkers, seed, step, randomize_split);
  order_kernel<<<(nwalkers + 255) / 256, 256, 0, (cudaStream_t)stream>>>(perm, nwalkers, d_order);
  MP_CUDA(cudaGetLastError());
  return MP_OK;
}

extern "C" int mp_last_stiff_count(mp_handle* h, int32_t* count) {
  if (!h || !count) return fail(MP_ERR_BAD_ARG, "mp_last_stiff_count: null pointer");
  MP_CUDA(cudaSetDevice(h->device));
  MP_CUDA(cudaDeviceSynchronize());
  *count = 0;
  if (h->last_lane && h->last_lane->counters.get())
    MP_CUDA(cudaMemcpy(count, h->last_lane->counters.get() + 2, sizeof(int), cudaMemcpyDeviceToHost));
  return MP_OK;
}
