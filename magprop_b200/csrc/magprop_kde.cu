// magprop_kde.cu -- emcee 3's KDEMove on the device ensembles: the proposal q and ln f of every mover, formed ahead of
// the evaluation pipeline, which then takes q from `prop` and ln f from `lnf` as it does for every move kind
// (magprop_kernels.cu, Move).  The formulas and the order of every sum are those of MP_MOVE_KDE in
// include/magprop_b200.h; the library is compiled with -fmad=false, so no operation here is contracted and the NumPy
// restatement (tests/kde_ref.py) reproduces q bit for bit.  No atomics: nothing depends on the launch shape.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>

#include "magprop_kde.hpp"

namespace mp {

constexpr int kKdeTile = 64;            // centres per tile of the mean and covariance sums
constexpr int kKdeTiles = MP_KDE_MAX_CENTRES / kKdeTile;   // one prepare thread per tile
constexpr int kKdePairs = MP_MAX_NDIM * (MP_MAX_NDIM + 1) / 2;
constexpr int kKdeThreads = 128;        // movers per block of the proposal kernel
static_assert(MP_KDE_MAX_CENTRES % kKdeTile == 0, "whole tiles");
static_assert(kKdeStats >= 12 + MP_MAX_NDIM * MP_MAX_NDIM, "stats hold mu, ok and L");

__device__ __forceinline__ const double* centre(const KdeMove& k, int t, int j) {
  return k.coords + (size_t)tempered_partner(k.perm, (uint32_t)k.cpos0, (uint32_t)t, (uint32_t)j) * k.ndim;
}

// y = L^-1 (p - mu) / h: forward substitution, rows ascending.
__device__ __forceinline__ void whiten(const double* mu, const double* L, double h, int d, const double* p, double* y) {
  double w[MP_MAX_NDIM];
#pragma unroll
  for (int r = 0; r < MP_MAX_NDIM; ++r) {
    if (r < d) {
      double s = p[r] - mu[r];
#pragma unroll
      for (int c = 0; c < r; ++c) s = s - L[r * MP_MAX_NDIM + c] * w[c];
      w[r] = s / L[r * MP_MAX_NDIM + r];
      y[r] = w[r] / h;
    }
  }
}

// One block per temperature, one thread per tile of 64 centres.
__global__ void __launch_bounds__(kKdeTiles) kde_prepare_kernel(const __grid_constant__ KdeMove k) {
  __shared__ double part[kKdeTiles][kKdePairs];
  __shared__ double mu[MP_MAX_NDIM], L[MP_MAX_NDIM * MP_MAX_NDIM];
  __shared__ int ok;
  const int t = blockIdx.x, d = k.ndim, M = k.M, tile = threadIdx.x;
  const int ntiles = (M + kKdeTile - 1) / kKdeTile;
  const int j0 = tile * kKdeTile, j1 = min(j0 + kKdeTile, M);
  // the tile's coordinate sums, left to right; then thread 0 adds the tiles left to right
  double s[MP_MAX_NDIM];
#pragma unroll
  for (int c = 0; c < MP_MAX_NDIM; ++c) s[c] = 0.0;
  for (int j = j0; j < j1; ++j) {
    const double* x = centre(k, t, j);
#pragma unroll
    for (int c = 0; c < MP_MAX_NDIM; ++c)
      if (c < d) s[c] = s[c] + x[c];
  }
#pragma unroll
  for (int c = 0; c < MP_MAX_NDIM; ++c) part[tile][c] = s[c];
  __syncthreads();
  if (tile == 0)
    for (int c = 0; c < d; ++c) {
      double S = 0.0;
      for (int q = 0; q < ntiles; ++q) S = S + part[q][c];
      mu[c] = S / (double)M;
    }
  __syncthreads();
  // the tile's sums of (x_a - mu_a)(x_b - mu_b), b <= a, pair index a(a+1)/2 + b
  double s2[kKdePairs];
#pragma unroll
  for (int p = 0; p < kKdePairs; ++p) s2[p] = 0.0;
  for (int j = j0; j < j1; ++j) {
    const double* x = centre(k, t, j);
    double e[MP_MAX_NDIM];
#pragma unroll
    for (int c = 0; c < MP_MAX_NDIM; ++c) e[c] = c < d ? x[c] - mu[c] : 0.0;
#pragma unroll
    for (int a = 0; a < MP_MAX_NDIM; ++a)
#pragma unroll
      for (int b = 0; b <= a; ++b)
        if (a < d) s2[a * (a + 1) / 2 + b] = s2[a * (a + 1) / 2 + b] + e[a] * e[b];
  }
  __syncthreads();   // (every thread has read mu; part is reused)
#pragma unroll
  for (int p = 0; p < kKdePairs; ++p) part[tile][p] = s2[p];
  __syncthreads();
  if (tile == 0) {
    // Sigma = S2 / (M - 1); Cholesky in row order
    double Ls[MP_MAX_NDIM * MP_MAX_NDIM];
    for (int p = 0; p < MP_MAX_NDIM * MP_MAX_NDIM; ++p) Ls[p] = 0.0;
    int good = 1;
    for (int i = 0; i < d && good; ++i)
      for (int j = 0; j <= i; ++j) {
        double S = 0.0;
        for (int q = 0; q < ntiles; ++q) S = S + part[q][i * (i + 1) / 2 + j];
        double v = S / (double)(M - 1);
        for (int c = 0; c < j; ++c) v = v - Ls[i * MP_MAX_NDIM + c] * Ls[j * MP_MAX_NDIM + c];
        if (i == j) {
          if (!(v > 0.0 && isfinite(v))) {
            good = 0;
            break;
          }
          Ls[i * MP_MAX_NDIM + i] = sqrt(v);
        } else {
          Ls[i * MP_MAX_NDIM + j] = v / Ls[j * MP_MAX_NDIM + j];
        }
      }
    double* st = k.stats + (size_t)t * kKdeStats;
    for (int c = 0; c < MP_MAX_NDIM; ++c) st[c] = c < d ? mu[c] : 0.0;
    st[9] = good ? 1.0 : 0.0;
    for (int p = 0; p < MP_MAX_NDIM * MP_MAX_NDIM; ++p) {
      L[p] = Ls[p];
      st[12 + p] = Ls[p];
    }
    ok = good;
  }
  __syncthreads();
  if (!ok) return;
  for (int j = tile; j < M; j += kKdeTiles) {
    double y[MP_MAX_NDIM];
    whiten(mu, L, k.h, d, centre(k, t, j), y);
    double* w = k.white + ((size_t)t * M + j) * d;
#pragma unroll
    for (int c = 0; c < MP_MAX_NDIM; ++c)
      if (c < d) w[c] = y[c];
  }
}

// -0.5 min_j r2_j and sum_j exp(-0.5 (r2_j - min)), j ascending, for the two points x and q at once.
__global__ void __launch_bounds__(kKdeThreads) kde_propose_kernel(const __grid_constant__ KdeMove k, int mover0, int count,
                                                                 double* __restrict__ prop, double* __restrict__ lnf) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const int d = k.ndim, M = k.M;
  const TemperedMover tm = tempered_mover(k.perm, (uint32_t)k.pos0, (uint32_t)(mover0 + i));
  const int t = (int)tm.t;
  const double* st = k.stats + (size_t)t * kKdeStats;
  const double* mu = st;
  const double* L = st + 12;
  const double* x = k.coords + (size_t)tm.row * d;
  double* out = prop + (size_t)i * d;
  if (st[9] == 0.0) {          // no Cholesky factor: stay, rejected
    for (int c = 0; c < d; ++c) out[c] = x[c];
    lnf[i] = -INFINITY;
    return;
  }
  const uint32_t me = tm.row;
  double z[MP_MAX_NDIM + 1];
  kde_gaussians(k.seed, k.hs, me, d, z);
  const double* cj = centre(k, t, (int)pick_index(kde_centre_uniform(k.seed, k.hs, me), (uint32_t)M));
  double q[MP_MAX_NDIM], xx[MP_MAX_NDIM];
#pragma unroll
  for (int r = 0; r < MP_MAX_NDIM; ++r) {
    if (r < d) {
      double s = 0.0;
#pragma unroll
      for (int c = 0; c <= r; ++c) s = s + L[r * MP_MAX_NDIM + c] * z[c];
      q[r] = cj[r] + k.h * s;
      out[r] = q[r];
      xx[r] = x[r];
    }
  }
  double yx[MP_MAX_NDIM], yq[MP_MAX_NDIM];
  whiten(mu, L, k.h, d, xx, yx);
  whiten(mu, L, k.h, d, q, yq);
  const double* w = k.white + (size_t)t * M * d;
  double mx = INFINITY, mq = INFINITY;
  for (int j = 0; j < M; ++j) {
    double rx = 0.0, rq = 0.0;
#pragma unroll
    for (int c = 0; c < MP_MAX_NDIM; ++c) {
      if (c < d) {
        const double wc = w[(size_t)j * d + c];
        const double ex = yx[c] - wc, eq = yq[c] - wc;
        rx = rx + ex * ex;
        rq = rq + eq * eq;
      }
    }
    mx = fmin(mx, rx);
    mq = fmin(mq, rq);
  }
  double sx = 0.0, sq = 0.0;
  for (int j = 0; j < M; ++j) {
    double rx = 0.0, rq = 0.0;
#pragma unroll
    for (int c = 0; c < MP_MAX_NDIM; ++c) {
      if (c < d) {
        const double wc = w[(size_t)j * d + c];
        const double ex = yx[c] - wc, eq = yq[c] - wc;
        rx = rx + ex * ex;
        rq = rq + eq * eq;
      }
    }
    sx = sx + exp(-0.5 * (rx - mx));
    sq = sq + exp(-0.5 * (rq - mq));
  }
  lnf[i] = (-0.5 * mx + log(sx)) - (-0.5 * mq + log(sq));
}

int kde_prepare(const KdeMove& k, cudaStream_t stream) {
  kde_prepare_kernel<<<k.T, kKdeTiles, 0, stream>>>(k);
  MP_CUDA(cudaGetLastError());
  return MP_OK;
}

int kde_propose(const KdeMove& k, int mover0, int count, double* prop, double* lnf, cudaStream_t stream) {
  kde_propose_kernel<<<(count + kKdeThreads - 1) / kKdeThreads, kKdeThreads, 0, stream>>>(k, mover0, count, prop, lnf);
  MP_CUDA(cudaGetLastError());
  return MP_OK;
}

}  // namespace mp
