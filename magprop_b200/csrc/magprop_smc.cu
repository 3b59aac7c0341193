// magprop_smc.cu -- the population primitives of sequential Monte Carlo (include/magprop_smc.h): the incremental
// weights of a tempering step with their sums (mp_smc_weights) and systematic resampling (mp_smc_resample).  They read
// and write particle arrays the caller keeps on the device and use no likelihood handle; the MCMC moves between the
// stages are the ensemble's (mp_annealed_moves_half_step, magprop_kernels.cu).
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>

#include "magprop_abi.hpp"
#include "magprop_rng.cuh"

namespace mp {

constexpr unsigned kFull = 0xffffffffu;
// The weights' grid: a fixed number of blocks for a given n, so the order the partial sums are added in depends on n
// alone -- never on the stream or on what else runs.
constexpr int kSmcBlocks = 1184, kSmcThreads = 256;
constexpr int kTile = MP_SMC_TILE;

// Largest finite lnp of each block's grid-stride share (-inf if it has none).  A max is exact, so no order matters.
__global__ void smc_max_kernel(const double* __restrict__ lnp, long long n, double* __restrict__ part) {
  __shared__ double sh[kSmcThreads / 32];
  double m = -INFINITY;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double v = lnp[i];
    if (isfinite(v)) m = fmax(m, v);
  }
  for (int off = 16; off > 0; off >>= 1) m = fmax(m, __shfl_xor_sync(kFull, m, off));
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 1; k < (int)(blockDim.x >> 5); ++k) m = fmax(m, sh[k]);
    part[blockIdx.x] = m;
  }
}

__global__ void smc_max_finish_kernel(const double* __restrict__ part, int blocks, double* __restrict__ m_out) {
  double m = -INFINITY;
  for (int b = threadIdx.x; b < blocks; b += 32) m = fmax(m, part[b]);
  for (int off = 16; off > 0; off >>= 1) m = fmax(m, __shfl_xor_sync(kFull, m, off));
  if (threadIdx.x == 0) *m_out = m;
}

// w_i = exp(dbeta (lnp_i - m)) (0 for a non-finite lnp_i), and each block's S1 and S2: lanes in shuffle order, warps in
// order -- part[block][2].
__global__ void smc_sum_kernel(const double* __restrict__ lnp, long long n, double dbeta, const double* __restrict__ m_in,
                               double* __restrict__ w, double* __restrict__ part) {
  __shared__ double sh[2][kSmcThreads / 32];
  const double m = *m_in;
  double s1 = 0.0, s2 = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double v = lnp[i];
    const double wi = isfinite(v) ? exp(dbeta * (v - m)) : 0.0;
    if (w) w[i] = wi;
    s1 += wi;
    s2 += wi * wi;
  }
  for (int off = 16; off > 0; off >>= 1) {
    s1 += __shfl_xor_sync(kFull, s1, off);
    s2 += __shfl_xor_sync(kFull, s2, off);
  }
  if ((threadIdx.x & 31) == 0) {
    sh[0][threadIdx.x >> 5] = s1;
    sh[1][threadIdx.x >> 5] = s2;
  }
  __syncthreads();
  if (threadIdx.x < 2) {
    double v = 0.0;
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) v += sh[threadIdx.x][k];
    part[blockIdx.x * 2 + threadIdx.x] = v;
  }
}

// out = {m, S1, S2}: the blocks' partials added in block order.
__global__ void smc_sum_finish_kernel(const double* __restrict__ part, int blocks, const double* __restrict__ m_in,
                                      double* __restrict__ out) {
  const int q = threadIdx.x;
  if (q >= 2) return;
  double v = 0.0;
  for (int b = 0; b < blocks; ++b) v += part[b * 2 + q];
  out[1 + q] = v;
  if (q == 0) out[0] = *m_in;
}

// ---- systematic resampling -------------------------------------------------------------------------------------
// Tile k = [k*kTile, min((k+1)*kTile, n)): its total (left to right from 0) and its last index of positive weight.
__global__ void smc_tile_kernel(const double* __restrict__ w, long long n, long long ntiles, double* __restrict__ tile_sum,
                                long long* __restrict__ tile_last) {
  for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < ntiles; k += (long long)gridDim.x * blockDim.x) {
    const long long lo = k * kTile, hi = min(lo + kTile, n);
    double p = 0.0;
    long long last = -1;
    for (long long j = lo; j < hi; ++j) {
      const double v = w[j];
      p += v;
      if (v > 0.0) last = j;
    }
    tile_sum[k] = p;
    tile_last[k] = last;
  }
}

// One thread: base[k+1] = base[k] + tile_sum[k] left to right, and the last index of positive weight overall.  The
// loads of a batch are issued before its dependent adds.
constexpr int kScanBatch = 32;
__global__ void smc_scan_kernel(const double* __restrict__ tile_sum, const long long* __restrict__ tile_last, long long ntiles,
                                double* __restrict__ base, long long* __restrict__ jlast) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double b = 0.0;
  long long last = -1;
  base[0] = 0.0;
  for (long long k0 = 0; k0 < ntiles; k0 += kScanBatch) {
    double v[kScanBatch];
    long long l[kScanBatch];
#pragma unroll
    for (int q = 0; q < kScanBatch; ++q) {
      v[q] = k0 + q < ntiles ? tile_sum[k0 + q] : 0.0;
      l[q] = k0 + q < ntiles ? tile_last[k0 + q] : -1;
    }
#pragma unroll
    for (int q = 0; q < kScanBatch; ++q) {
      if (k0 + q < ntiles) {
        b += v[q];
        base[k0 + q + 1] = b;
        if (l[q] >= 0) last = l[q];
      }
    }
  }
  *jlast = last;
}

// a_i: the smallest j with cum_j > (i + u)(total / n), clamped to the last j of positive weight; a_i = i if total == 0.
// The tile holding a_i is the first k with base[k+1] > target (binary search); within it cum_j = base[k] + p_j is
// recomputed in the tile kernel's order, so cum at the tile's last element is base[k+1] bit for bit.
__global__ void smc_ancestor_kernel(const double* __restrict__ w, long long n, int ndim, long long ntiles,
                                    const double* __restrict__ base, const long long* __restrict__ jlast_p, double u,
                                    const double* __restrict__ coords_in, const double* __restrict__ lnp_in,
                                    double* __restrict__ coords_out, double* __restrict__ lnp_out,
                                    long long* __restrict__ ancestors) {
  const double total = base[ntiles];
  const long long jlast = *jlast_p;
  const double stride = total / (double)n;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    long long a = i;
    if (total > 0.0 && jlast >= 0) {
      const double target = ((double)i + u) * stride;
      long long lo = 0, hi = ntiles;
      while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (base[mid + 1] > target) hi = mid;
        else lo = mid + 1;
      }
      a = jlast;
      if (lo < ntiles) {
        const long long j0 = lo * kTile, j1 = min(j0 + kTile, n);
        const double bk = base[lo];
        double p = 0.0;
        for (long long j = j0; j < j1; ++j) {
          p += w[j];
          if (bk + p > target) {
            a = j;
            break;
          }
        }
        if (a > jlast) a = jlast;
      }
    }
    for (int d = 0; d < ndim; ++d) coords_out[i * ndim + d] = coords_in[a * ndim + d];
    lnp_out[i] = lnp_in[a];
    if (ancestors) ancestors[i] = a;
  }
}

// [p, p + bytes) and [q, q + qbytes) share a byte (a null range shares none).
static bool overlaps(const void* p, __int128 bytes, const void* q, __int128 qbytes) {
  if (!p || !q) return false;
  const __int128 a = (__int128)(uintptr_t)p, b = (__int128)(uintptr_t)q;
  return a < b + qbytes && b < a + bytes;
}

static int grid_for(long long items) { return (int)std::min<long long>((items + 255) / 256, 1LL << 20); }

}  // namespace mp

using namespace mp;

extern "C" int mp_smc_weights(const double* d_lnp, int64_t n, double dbeta, double* d_w, double* out, int32_t device,
                              void* stream) {
  if (!d_lnp || !out) return fail(MP_ERR_BAD_ARG, "mp_smc_weights: null lnp or out");
  if (n < 1) return fail(MP_ERR_BAD_ARG, "mp_smc_weights: n must be >= 1");
  if (!(dbeta >= 0.0 && std::isfinite(dbeta))) return fail(MP_ERR_BAD_ARG, "mp_smc_weights: dbeta must be finite and >= 0");
  int rc = select_device(device, "mp_smc_weights");
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = (int)std::min<int64_t>((n + kSmcThreads - 1) / kSmcThreads, kSmcBlocks);
  double* d_buf = nullptr;
  MP_CUDA(cudaMallocAsync((void**)&d_buf, (size_t)(3 * blocks + 4) * sizeof(double), st));
  double *d_out = d_buf, *d_m = d_out + 3, *d_maxp = d_m + 1, *d_sump = d_maxp + blocks;   // sump: [blocks][2]
  smc_max_kernel<<<blocks, kSmcThreads, 0, st>>>(d_lnp, n, d_maxp);
  smc_max_finish_kernel<<<1, 32, 0, st>>>(d_maxp, blocks, d_m);
  smc_sum_kernel<<<blocks, kSmcThreads, 0, st>>>(d_lnp, n, dbeta, d_m, d_w, d_sump);
  smc_sum_finish_kernel<<<1, 32, 0, st>>>(d_sump, blocks, d_m, d_out);
  double h[3];
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(h, d_out, sizeof(h), cudaMemcpyDeviceToHost, st);
  const cudaError_t ef = cudaFreeAsync(d_buf, st);
  if (e == cudaSuccess) e = ef;
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return fail(MP_ERR_CUDA, std::string("mp_smc_weights: ") + cudaGetErrorString(e));
  std::memcpy(out, h, sizeof(h));
  return MP_OK;
}

extern "C" int mp_smc_resample(const double* d_w, int64_t n, int32_t ndim, uint64_t seed, uint64_t stage,
                               const double* d_coords_in, const double* d_lnp_in, double* d_coords_out, double* d_lnp_out,
                               int64_t* d_ancestors, int32_t device, void* stream) {
  if (!d_w || !d_coords_in || !d_lnp_in || !d_coords_out || !d_lnp_out)
    return fail(MP_ERR_BAD_ARG, "mp_smc_resample: null weights, coords or lnp");
  if (n < 1) return fail(MP_ERR_BAD_ARG, "mp_smc_resample: n must be >= 1");
  if (ndim < 1 || ndim > MP_MAX_NDIM) return fail(MP_ERR_BAD_ARG, "mp_smc_resample: ndim must lie in 1..MP_MAX_NDIM");
  const __int128 nb = (__int128)n * 8, cb = nb * ndim;
  const void* ins[3] = {d_w, d_coords_in, d_lnp_in};
  const __int128 in_bytes[3] = {nb, cb, nb};
  const void* outs[3] = {d_coords_out, d_lnp_out, d_ancestors};
  const __int128 out_bytes[3] = {cb, nb, nb};
  for (int o = 0; o < 3; ++o) {
    for (int i = 0; i < 3; ++i)
      if (overlaps(outs[o], out_bytes[o], ins[i], in_bytes[i]))
        return fail(MP_ERR_BAD_ARG, "mp_smc_resample: an output overlaps an input");
    for (int p = o + 1; p < 3; ++p)
      if (overlaps(outs[o], out_bytes[o], outs[p], out_bytes[p]))
        return fail(MP_ERR_BAD_ARG, "mp_smc_resample: two outputs overlap");
  }
  int rc = select_device(device, "mp_smc_resample");
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const long long ntiles = (n + kTile - 1) / kTile;
  const double u = smc_stage_uniform(seed, stage);
  void* d_buf = nullptr;
  MP_CUDA(cudaMallocAsync(&d_buf, (size_t)(3 * ntiles + 2) * 8, st));
  double* d_tsum = (double*)d_buf;                        // [ntiles]
  double* d_base = d_tsum + ntiles;                       // [ntiles + 1]
  long long* d_tlast = (long long*)(d_base + ntiles + 1); // [ntiles]
  long long* d_jlast = d_tlast + ntiles;                  // [1]
  smc_tile_kernel<<<grid_for(ntiles), 256, 0, st>>>(d_w, n, ntiles, d_tsum, d_tlast);
  smc_scan_kernel<<<1, 1, 0, st>>>(d_tsum, d_tlast, ntiles, d_base, d_jlast);
  smc_ancestor_kernel<<<grid_for(n), 256, 0, st>>>(d_w, n, ndim, ntiles, d_base, d_jlast, u, d_coords_in, d_lnp_in,
                                                   d_coords_out, d_lnp_out, (long long*)d_ancestors);
  cudaError_t e = cudaGetLastError();
  const cudaError_t ef = cudaFreeAsync(d_buf, st);
  if (e == cudaSuccess) e = ef;
  if (e != cudaSuccess) return fail(MP_ERR_CUDA, std::string("mp_smc_resample: ") + cudaGetErrorString(e));
  return MP_OK;
}
