// magprop_chain.cu -- posterior summaries of a device-resident chain: column means and covariances
// (mp_chain_moments), exact order statistics (mp_chain_order_statistics) and the walker-averaged autocorrelation
// function (mp_chain_autocorr).  They read a chain the caller keeps on the device and return a few numbers to the
// host; none of them uses a likelihood handle.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include <vector>

#include "magprop_abi.hpp"

namespace mp {

constexpr unsigned kFull = 0xffffffffu;

// ---- posterior summaries of a device-resident chain (plot_synth.py:150-166) -------------------------------
// Column means and the centred cross-products (for np.corrcoef), and exact order statistics by radix select
// (for np.percentile): the chain never leaves the device, the host receives a few dozen numbers.
// No floating-point atomics: every block writes its partial sums to part[block][q], and a one-block finish kernel adds
// them in block order -- the result depends only on n and ndim, so two calls on one chain agree bit for bit.
constexpr int kMomBlocks = 1184, kMomThreads = 256;

__global__ void chain_mean_kernel(const double* __restrict__ x, long long n, int ndim, double* __restrict__ part) {
  __shared__ double sh[MP_MAX_NDIM][8];
  double acc[MP_MAX_NDIM];
  for (int d = 0; d < MP_MAX_NDIM; ++d) acc[d] = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    for (int d = 0; d < ndim; ++d) acc[d] += x[i * ndim + d];
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  for (int d = 0; d < ndim; ++d) {
    double v = acc[d];
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(kFull, v, off);
    if (lane == 0) sh[d][wrp] = v;
  }
  __syncthreads();
  if (threadIdx.x < ndim) {
    double v = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) v += sh[threadIdx.x][w];
    part[blockIdx.x * ndim + threadIdx.x] = v;
  }
}

// mean[d] = (sum of the blocks' partials in block order) / n
__global__ void chain_mean_finish_kernel(const double* __restrict__ part, int blocks, long long n, int ndim,
                                         double* __restrict__ mean) {
  const int d = threadIdx.x;
  if (d >= ndim) return;
  double v = 0.0;
  for (int b = 0; b < blocks; ++b) v += part[b * ndim + d];
  mean[d] = v / (double)n;
}

__global__ void chain_cov_kernel(const double* __restrict__ x, long long n, int ndim, const double* __restrict__ mean,
                                 double* __restrict__ part /*[block][npair], pairs (a <= b) row by row*/) {
  __shared__ double sh[MP_MAX_NDIM * MP_MAX_NDIM][8];
  double acc[MP_MAX_NDIM * (MP_MAX_NDIM + 1) / 2];
  const int npair = ndim * (ndim + 1) / 2;
  for (int q = 0; q < npair; ++q) acc[q] = 0.0;
  double mu[MP_MAX_NDIM];
  for (int d = 0; d < ndim; ++d) mu[d] = mean[d];
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    double c[MP_MAX_NDIM];
    for (int d = 0; d < ndim; ++d) c[d] = x[i * ndim + d] - mu[d];
    int q = 0;
    for (int a = 0; a < ndim; ++a)
      for (int b = a; b < ndim; ++b, ++q) acc[q] = fma(c[a], c[b], acc[q]);
  }
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  for (int q = 0; q < npair; ++q) {
    double v = acc[q];
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(kFull, v, off);
    if (lane == 0) sh[q][wrp] = v;
  }
  __syncthreads();
  if (threadIdx.x < npair) {
    double v = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) v += sh[threadIdx.x][w];
    part[blockIdx.x * npair + threadIdx.x] = v;
  }
}

// cov[a][b] = cov[b][a] = (sum of the blocks' partials of pair (a, b) in block order) / max(n - 1, 1)
__global__ void chain_cov_finish_kernel(const double* __restrict__ part, int blocks, long long n, int ndim,
                                        double* __restrict__ cov) {
  const int npair = ndim * (ndim + 1) / 2, q = threadIdx.x;
  if (q >= npair) return;
  int a = 0, r = q;
  while (r >= ndim - a) {   // row a of the upper triangle holds pairs (a, a..ndim-1)
    r -= ndim - a;
    ++a;
  }
  const int b = a + r;
  double v = 0.0;
  for (int k = 0; k < blocks; ++k) v += part[k * npair + q];
  v /= (double)(n > 1 ? n - 1 : 1);
  cov[a * ndim + b] = v;
  cov[b * ndim + a] = v;
}

// IEEE doubles as unsigned keys in ascending order: -inf < ... < -0 < +0 < ... < +inf < every NaN.  A NaN's sign bit
// is dropped, so a NaN made with the sign bit set (0/0 on x86) sorts last too, as np.sort puts it.
__device__ __forceinline__ unsigned long long order_key(double v) {
  unsigned long long b = (unsigned long long)__double_as_longlong(v);
  if ((b & 0x7fffffffffffffffull) > 0x7ff0000000000000ull) b &= 0x7fffffffffffffffull;
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
constexpr int kSelectBins = 1 << 16;   // one per value of the 16-bit digit a radix-select pass sorts on
// One pass of the radix select on column `col`: histogram of the 16-bit digit at `shift` over the elements whose
// higher digits equal those of `prefix`.  64-bit bins, so a column of 2^32 or more equal digits cannot wrap one.  The
// lanes of a warp that fall in the same bin add to it once (match + popc): a chain's ties (stuck walkers, a long
// constant column) otherwise serialise on one address.
__global__ void select_hist_kernel(const double* __restrict__ x, long long n, int ndim, int col, unsigned long long prefix,
                                   int shift, unsigned long long* __restrict__ hist) {
  const unsigned long long himask = (shift >= 48) ? 0ull : (~0ull << (shift + 16));
  const int lane = threadIdx.x & 31;
  const long long stride = (long long)gridDim.x * blockDim.x;
  // base is the warp's first row: the loop condition is uniform over the warp, so every lane reaches the match
  for (long long base = blockIdx.x * (long long)blockDim.x + (threadIdx.x & ~31); base < n; base += stride) {
    const long long i = base + lane;
    unsigned bin = 0xffffffffu;                          // no bin: past the end, or another prefix
    if (i < n) {
      const unsigned long long key = order_key(x[i * ndim + col]);
      if ((key & himask) == (prefix & himask)) bin = (unsigned)((key >> shift) & 0xffffull);
    }
    const unsigned peers = __match_any_sync(kFull, bin);
    if (bin != 0xffffffffu && lane == __ffs(peers) - 1) atomicAdd(hist + bin, (unsigned long long)__popc(peers));
  }
}

// ---- walker-averaged autocorrelation function of a device-resident chain (emcee's integrated_time) ---------------
// The chain [n_steps][nwalkers][ndim] is read as [n_steps][J], J = nwalkers*ndim: series j = w*ndim + d is column j,
// retained rows first + t*thin, t in [0, n).  Three launches, no floating-point atomics -- the result depends only on
// the shapes and the SM count, so two calls on one chain agree bit for bit:
//   acf_center_kernel  one thread per series: shift x0 = first retained sample, mean m of (x - x0), and
//                      C(0) = sum_t s_t^2 of the centred series s_t = (x_t - x0) - m
//   acf_lag_kernel     a block owns kAcfKB lags (kAcfKR per warp) of 32 consecutive series (one per lane) for a group
//                      of such series tiles and a range of time chunks.  Per chunk of kAcfT anchor rows it stages the
//                      centred rows [t0, t0+T) and [t0+kbase, t0+kbase+T+KB) in shared memory (row reads coalesced
//                      along the walker axis); every thread accumulates C(k) of its series for its kAcfKR lags in
//                      registers through a sliding window of 2*kAcfKR lagged samples (2 shared loads per kAcfKR FMAs).
//                      C(k)/C(0) is then summed per dimension in lane order, and over the group's tiles in tile order.
//   acf_finish_kernel  one thread per (d, k): the blocks' partials in a fixed order, / nwalkers
constexpr int kAcfKR = 16, kAcfWarps = 8, kAcfKB = kAcfKR * kAcfWarps, kAcfT = 128;
constexpr int kAcfNQ = (MP_MAX_NDIM * kAcfKB + 32 * kAcfWarps - 1) / (32 * kAcfWarps);
constexpr size_t kAcfSmem = (size_t)(2 * kAcfT + kAcfKB) * 32 * sizeof(double);

struct AcfShape {
  const double* x;
  long long J;                  // nwalkers * ndim
  long long first, thin, n;     // retained rows first + t*thin, t < n
  long long lag_begin, nl;      // lags [lag_begin, lag_begin + nl)
  long long n_tiles, n_groups;  // 32-series tiles; block group g takes tiles g, g + n_groups, ...
  int ndim, n_lb;               // lag blocks of kAcfKB
  int cps, nsplit;              // time chunks per split, splits
};

__global__ void acf_center_kernel(const AcfShape a, double* __restrict__ x0, double* __restrict__ mu,
                                  double* __restrict__ c0) {
  const long long stride = a.thin * a.J;
  for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j < a.J; j += (long long)gridDim.x * blockDim.x) {
    const double* col = a.x + a.first * a.J + j;
    const double s0 = col[0];
    double sum = 0.0;
    for (long long t = 0; t < a.n; ++t) sum += col[t * stride] - s0;
    const double m = sum / (double)a.n;
    double ss = 0.0;
    for (long long t = 0; t < a.n; ++t) {
      const double s = (col[t * stride] - s0) - m;
      ss = fma(s, s, ss);
    }
    x0[j] = s0;
    mu[j] = m;
    c0[j] = ss;
  }
}

__global__ void __launch_bounds__(32 * kAcfWarps, 2) acf_lag_kernel(const AcfShape a, const double* __restrict__ x0,
                                                                    const double* __restrict__ mu,
                                                                    const double* __restrict__ c0,
                                                                    double* __restrict__ part /*[item][ndim][kAcfKB]*/) {
  extern __shared__ double acf_sm[];
  double* sa = acf_sm;                    // [kAcfT][32]          anchor rows
  double* sb = acf_sm + kAcfT * 32;       // [kAcfT + kAcfKB][32] lagged rows
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  long long item = blockIdx.x;            // = (g * n_lb + lb) * nsplit + split
  const int split = (int)(item % a.nsplit);
  item /= a.nsplit;
  const int lb = (int)(item % a.n_lb);
  const long long g = item / a.n_lb;
  const long long kbase = a.lag_begin + (long long)lb * kAcfKB;
  const long long n_chunks = (a.n + kAcfT - 1) / kAcfT;
  const long long c_lo = (long long)split * a.cps, c_hi = min(c_lo + a.cps, n_chunks);
  const long long rstride = a.thin * a.J;
  const double* rows = a.x + a.first * a.J;
  double racc[kAcfNQ];
#pragma unroll
  for (int q = 0; q < kAcfNQ; ++q) racc[q] = 0.0;

  for (long long tile = g; tile < a.n_tiles; tile += a.n_groups) {
    const long long j = tile * 32 + lane;
    const bool live = j < a.J;
    const double sx0 = live ? x0[j] : 0.0, smu = live ? mu[j] : 0.0;
    double acc[kAcfKR];
#pragma unroll
    for (int r = 0; r < kAcfKR; ++r) acc[r] = 0.0;
    for (long long c = c_lo; c < c_hi; ++c) {
      const long long t0 = c * kAcfT;
      if (t0 + kbase >= a.n) break;       // every pair of this and later chunks reaches past the last row
      __syncthreads();
      // centred samples; zero past the last retained row, so pairs (t, t+k) with t+k >= n add nothing
      for (int r = warp; r < kAcfT; r += kAcfWarps) {
        const long long t = t0 + r;
        sa[r * 32 + lane] = (live && t < a.n) ? (rows[t * rstride + j] - sx0) - smu : 0.0;
      }
      for (int r = warp; r < kAcfT + kAcfKB; r += kAcfWarps) {
        const long long t = t0 + kbase + r;
        sb[r * 32 + lane] = (live && t < a.n) ? (rows[t * rstride + j] - sx0) - smu : 0.0;
      }
      __syncthreads();
      // lag kbase + warp*kAcfKR + r of anchor tb + i is sb row tb + warp*kAcfKR + i + r
      const double* bw = sb + warp * kAcfKR * 32 + lane;
      double b[2 * kAcfKR];
#pragma unroll
      for (int q = 0; q < kAcfKR; ++q) b[q] = bw[q * 32];
#pragma unroll 1
      for (int tb = 0; tb < kAcfT; tb += kAcfKR) {
#pragma unroll
        for (int q = 0; q < kAcfKR; ++q) b[kAcfKR + q] = bw[(tb + kAcfKR + q) * 32];
#pragma unroll
        for (int i = 0; i < kAcfKR; ++i) {
          const double av = sa[(tb + i) * 32 + lane];
#pragma unroll
          for (int r = 0; r < kAcfKR; ++r) acc[r] = fma(av, b[i + r], acc[r]);
        }
#pragma unroll
        for (int q = 0; q < kAcfKR; ++q) b[q] = b[kAcfKR + q];
      }
    }
    // C(k)/C(0) of the tile's series, summed per dimension: lanes l with (tile*32 + l) % ndim == d, in lane order.
    // A constant series has C(0) = 0 and gives NaN, as emcee's formula does.
    const double cz = live ? c0[j] : 1.0;
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kAcfKR; ++r) sa[(warp * kAcfKR + r) * 32 + lane] = live ? acc[r] / cz : 0.0;
    __syncthreads();
    const int d0 = (int)((tile * 32) % a.ndim);
#pragma unroll
    for (int qi = 0; qi < kAcfNQ; ++qi) {
      const int q = threadIdx.x + qi * 32 * kAcfWarps;
      if (q < a.ndim * kAcfKB) {
        const int d = q / kAcfKB, kk = q % kAcfKB;
        double v = 0.0;
        for (int l = (d - d0 + a.ndim) % a.ndim; l < 32; l += a.ndim) v += sa[kk * 32 + l];
        racc[qi] += v;
      }
    }
  }
#pragma unroll
  for (int qi = 0; qi < kAcfNQ; ++qi) {
    const int q = threadIdx.x + qi * 32 * kAcfWarps;
    if (q < a.ndim * kAcfKB) part[blockIdx.x * (long long)(a.ndim * kAcfKB) + q] = racc[qi];
  }
}

__global__ void acf_finish_kernel(const AcfShape a, const double* __restrict__ part, int nwalkers, double* __restrict__ out) {
  const long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (q >= a.ndim * a.nl) return;
  const int d = (int)(q / a.nl);
  const long long kl = q % a.nl;
  const int lb = (int)(kl / kAcfKB), kk = (int)(kl % kAcfKB);
  double v = 0.0;
  for (long long g = 0; g < a.n_groups; ++g)
    for (int s = 0; s < a.nsplit; ++s)
      v += part[((g * a.n_lb + lb) * a.nsplit + s) * (a.ndim * kAcfKB) + d * kAcfKB + kk];
  out[q] = v / (double)nwalkers;
}

}  // namespace mp

using namespace mp;

extern "C" int mp_chain_moments(const double* d_chain, int64_t n, int32_t ndim, double* mean, double* cov, int32_t device,
                                void* stream) {
  if (!d_chain || !mean || !cov || n < 1 || ndim < 1 || ndim > MP_MAX_NDIM) return fail(MP_ERR_BAD_ARG, "mp_chain_moments: bad argument");
  int rc = select_device(device, "mp_chain_moments");
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = (int)std::min<int64_t>((n + kMomThreads - 1) / kMomThreads, kMomBlocks);
  const int npair = ndim * (ndim + 1) / 2;
  const size_t n_out = (size_t)ndim + (size_t)ndim * ndim;
  double* d_buf = nullptr;
  MP_CUDA(cudaMallocAsync((void**)&d_buf, (n_out + (size_t)blocks * npair) * sizeof(double), st));
  double *d_mean = d_buf, *d_cov = d_mean + ndim, *d_part = d_cov + (size_t)ndim * ndim;   // part: [blocks][ndim or npair]
  chain_mean_kernel<<<blocks, kMomThreads, 0, st>>>(d_chain, n, ndim, d_part);
  chain_mean_finish_kernel<<<1, 32, 0, st>>>(d_part, blocks, n, ndim, d_mean);
  chain_cov_kernel<<<blocks, kMomThreads, 0, st>>>(d_chain, n, ndim, d_mean, d_part);
  chain_cov_finish_kernel<<<1, 64, 0, st>>>(d_part, blocks, n, ndim, d_cov);
  std::vector<double> h(n_out);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(h.data(), d_buf, n_out * sizeof(double), cudaMemcpyDeviceToHost, st);
  const cudaError_t ef = cudaFreeAsync(d_buf, st);
  if (e == cudaSuccess) e = ef;
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return fail(MP_ERR_CUDA, std::string("mp_chain_moments: ") + cudaGetErrorString(e));
  std::memcpy(mean, h.data(), ndim * sizeof(double));
  std::memcpy(cov, h.data() + ndim, (size_t)ndim * ndim * sizeof(double));
  return MP_OK;
}

extern "C" int mp_chain_order_statistics(const double* d_chain, int64_t n, int32_t ndim, int32_t col, const int64_t* ranks,
                                         int32_t n_ranks, double* values, int32_t device, void* stream) {
  if (!d_chain || !ranks || !values || n < 1 || ndim < 1 || col < 0 || col >= ndim || n_ranks < 0)
    return fail(MP_ERR_BAD_ARG, "mp_chain_order_statistics: bad argument");
  for (int r = 0; r < n_ranks; ++r)
    if (ranks[r] < 0 || ranks[r] >= n) return fail(MP_ERR_BAD_ARG, "mp_chain_order_statistics: rank outside [0, n)");
  int rc = select_device(device, "mp_chain_order_statistics");
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long* d_hist = nullptr;
  MP_CUDA(cudaMallocAsync((void**)&d_hist, kSelectBins * sizeof(unsigned long long), st));
  std::vector<unsigned long long> hist(kSelectBins);
  const int blocks = (int)std::min<int64_t>((n + kMomThreads - 1) / kMomThreads, kMomBlocks);   // the moments' grid
  cudaError_t e = cudaSuccess;
  for (int r = 0; r < n_ranks && e == cudaSuccess; ++r) {
    unsigned long long k = (unsigned long long)ranks[r];
    unsigned long long prefix = 0ull;
    for (int shift = 48; shift >= 0; shift -= 16) {
      e = cudaMemsetAsync(d_hist, 0, kSelectBins * sizeof(unsigned long long), st);
      if (e == cudaSuccess) {
        select_hist_kernel<<<blocks, kMomThreads, 0, st>>>(d_chain, n, ndim, col, prefix, shift, d_hist);
        e = cudaGetLastError();
      }
      if (e == cudaSuccess)
        e = cudaMemcpyAsync(hist.data(), d_hist, kSelectBins * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st);
      if (e == cudaSuccess) e = cudaStreamSynchronize(st);
      if (e != cudaSuccess) break;
      unsigned digit = 0;
      for (; digit < kSelectBins - 1u && k >= hist[digit]; ++digit) k -= hist[digit];
      prefix |= (unsigned long long)digit << shift;
    }
    // key -> double
    const unsigned long long b = (prefix >> 63) ? (prefix & 0x7fffffffffffffffull) : ~prefix;
    std::memcpy(values + r, &b, sizeof(double));
  }
  const cudaError_t ef = cudaFreeAsync(d_hist, st);
  if (e == cudaSuccess) e = ef;
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return fail(MP_ERR_CUDA, std::string("mp_chain_order_statistics: ") + cudaGetErrorString(e));
  return MP_OK;
}

extern "C" int mp_chain_autocorr(const double* d_chain, int64_t n_steps, int32_t nwalkers, int32_t ndim, int64_t first,
                                 int64_t thin, int64_t lag_begin, int64_t lag_end, double* acf, int32_t device, void* stream) {
  if (!d_chain || !acf || nwalkers < 1 || ndim < 1 || ndim > MP_MAX_NDIM || thin < 1 || first < 0 || first >= n_steps ||
      lag_begin < 0 || lag_end <= lag_begin)
    return fail(MP_ERR_BAD_ARG, "mp_chain_autocorr: bad argument");
  const int64_t n = (n_steps - first + thin - 1) / thin;
  if (lag_end > n) return fail(MP_ERR_BAD_ARG, "mp_chain_autocorr: lag_end exceeds the number of retained rows");
  int rc = select_device(device, "mp_chain_autocorr");
  if (rc) return rc;
  int sms = 0;
  MP_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  MP_CUDA(cudaFuncSetAttribute(acf_lag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kAcfSmem));
  cudaStream_t st = (cudaStream_t)stream;

  AcfShape a;
  a.x = d_chain;
  a.J = (long long)nwalkers * ndim;
  a.first = first, a.thin = thin, a.n = n;
  a.lag_begin = lag_begin, a.nl = lag_end - lag_begin;
  a.ndim = ndim;
  a.n_lb = (int)((a.nl + kAcfKB - 1) / kAcfKB);
  a.n_tiles = (a.J + 31) / 32;
  // One wave of acf_lag_kernel (two blocks per SM): tiles are dealt out over the blocks; when there are fewer tiles x lag
  // blocks than that (few walkers), the time axis is split as well and the splits' partials are summed by the last pass.
  const long long wave = 2LL * sms;
  const long long n_chunks = (n + kAcfT - 1) / kAcfT;
  a.n_groups = std::min<long long>(a.n_tiles, std::max<long long>(1, wave / a.n_lb));
  long long nsplit = 1;
  if (a.n_groups == a.n_tiles) nsplit = std::min<long long>(n_chunks, std::max<long long>(1, wave / (a.n_tiles * a.n_lb)));
  a.cps = (int)((n_chunks + nsplit - 1) / nsplit);
  a.nsplit = (int)((n_chunks + a.cps - 1) / a.cps);
  const long long items = a.n_groups * a.n_lb * a.nsplit;

  const size_t n_part = (size_t)items * ndim * kAcfKB, n_out = (size_t)ndim * a.nl;
  double* d_buf = nullptr;
  MP_CUDA(cudaMallocAsync((void**)&d_buf, (3 * (size_t)a.J + n_part + n_out) * sizeof(double), st));
  double *d_x0 = d_buf, *d_mu = d_x0 + a.J, *d_c0 = d_mu + a.J, *d_part = d_c0 + a.J, *d_out = d_part + n_part;
  acf_center_kernel<<<(int)std::min<long long>((a.J + 255) / 256, 8LL * sms), 256, 0, st>>>(a, d_x0, d_mu, d_c0);
  acf_lag_kernel<<<(unsigned)items, 32 * kAcfWarps, kAcfSmem, st>>>(a, d_x0, d_mu, d_c0, d_part);
  acf_finish_kernel<<<(unsigned)((n_out + 255) / 256), 256, 0, st>>>(a, d_part, nwalkers, d_out);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(acf, d_out, n_out * sizeof(double), cudaMemcpyDeviceToHost, st);
  const cudaError_t ef = cudaFreeAsync(d_buf, st);
  if (e == cudaSuccess) e = ef;
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return fail(MP_ERR_CUDA, std::string("mp_chain_autocorr: ") + cudaGetErrorString(e));
  return MP_OK;
}
