// magprop_device.cu -- device plumbing of the C ABI: version, device count and the last error message; CUDA IPC
// allocations for peer-mapped ensemble replicas and the cross-GPU flag barrier; the FP64 FMA peak.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>

#include "magprop_abi.hpp"

namespace mp {

thread_local std::string g_err;

int fail_cuda(const char* func, const char* call, cudaError_t e) {
  return fail(MP_ERR_CUDA, std::string(func) + ": " + call + ": " + cudaGetErrorString(e));
}

// ---- cross-GPU flag barrier over peer-mapped memory ---------------------------------------------
// Thread p of the one block: raise flag[rank] = epoch in peer p's array (a system-scope release, after the
// preceding kernel's peer stores -- stream order plus the fence make them visible first), then spin on
// this rank's own array until peer p has raised its flag (system-scope acquire).  The spin is on LOCAL
// memory; the only NVLink traffic is one 8-byte store per peer.
struct PeerFlags {
  uint64_t* p[MP_MAX_PEERS + 1];
};
__global__ void peer_barrier_kernel(uint64_t* my_flags, PeerFlags pf, int rank, int world, uint64_t epoch, int* error) {
  const int p = threadIdx.x;
  if (p >= world || p == rank) return;
  __threadfence_system();
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(pf.p[p] + rank), "l"(epoch) : "memory");
  unsigned long long t0, t1;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  for (;;) {
    uint64_t v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(my_flags + p) : "memory");
    if (v >= epoch) break;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    if (t1 - t0 > 10000000000ull) {   // 10 s: a peer died -- report instead of hanging the GPU
      if (error) *error = 1;
      break;
    }
    __nanosleep(200);
  }
}

// ---- FP64 FMA peak: 8 independent chains per thread, 2 flop per DFMA ---------------
__global__ void __launch_bounds__(256) dfma_peak_kernel(double* out, int iters, double seed) {
  double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6,
         a7 = a0 + 7;
  const double m = 0.9999999, c = 1e-9;
#pragma unroll 1
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
      a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
  }
  const double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
  if (s == 12345.678) out[0] = s;  // keep the chains alive
}

}  // namespace mp

using namespace mp;

extern "C" int mp_abi_version(void) { return MP_ABI_VERSION; }

extern "C" int mp_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

extern "C" const char* mp_last_error(void) { return g_err.c_str(); }

// ---- peer-mapped replicas (CUDA IPC) -------------------------------------------------------------
static_assert(sizeof(cudaIpcMemHandle_t) == 64, "the C ABI carries IPC handles as 64 bytes");

extern "C" int mp_peer_alloc(int32_t device, uint64_t bytes, void** d_ptr, unsigned char handle[64]) {
  if (!d_ptr || !handle || bytes == 0) return fail(MP_ERR_BAD_ARG, "mp_peer_alloc: bad argument");
  const int rc = select_device(device, "mp_peer_alloc");
  if (rc) return rc;
  void* p = nullptr;
  MP_CUDA(cudaMalloc(&p, bytes));
  cudaError_t e = cudaMemset(p, 0, bytes);
  cudaIpcMemHandle_t hd;
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&hd, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    return fail(MP_ERR_CUDA, std::string("mp_peer_alloc: ") + cudaGetErrorString(e));
  }
  std::memcpy(handle, &hd, 64);
  *d_ptr = p;
  return MP_OK;
}

extern "C" int mp_peer_open(int32_t device, const unsigned char handle[64], void** d_ptr) {
  if (!d_ptr || !handle) return fail(MP_ERR_BAD_ARG, "mp_peer_open: null pointer");
  MP_CUDA(cudaSetDevice(device));
  cudaIpcMemHandle_t hd;
  std::memcpy(&hd, handle, 64);
  MP_CUDA(cudaIpcOpenMemHandle(d_ptr, hd, cudaIpcMemLazyEnablePeerAccess));
  return MP_OK;
}

extern "C" int mp_peer_close(int32_t device, void* d_ptr) {
  if (!d_ptr) return MP_OK;
  MP_CUDA(cudaSetDevice(device));
  MP_CUDA(cudaIpcCloseMemHandle(d_ptr));
  return MP_OK;
}

extern "C" int mp_peer_free(int32_t device, void* d_ptr) {
  if (!d_ptr) return MP_OK;
  MP_CUDA(cudaSetDevice(device));
  MP_CUDA(cudaFree(d_ptr));
  return MP_OK;
}

extern "C" int mp_peer_barrier(int32_t device, uint64_t* d_my_flags, uint64_t* const* peer_flags, int32_t rank,
                               int32_t world, uint64_t epoch, int32_t* d_error, void* stream) {
  if (!d_my_flags || !peer_flags || world < 1 || world > MP_MAX_PEERS + 1 || rank < 0 || rank >= world)
    return fail(MP_ERR_BAD_ARG, "mp_peer_barrier: bad argument");
  if (world == 1) return MP_OK;
  MP_CUDA(cudaSetDevice(device));
  PeerFlags pf;
  std::memset(&pf, 0, sizeof(pf));
  for (int p = 0; p < world; ++p) {
    if (p != rank && !peer_flags[p]) return fail(MP_ERR_BAD_ARG, "mp_peer_barrier: null peer flag array");
    pf.p[p] = peer_flags[p];
  }
  peer_barrier_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(d_my_flags, pf, rank, world, epoch, d_error);
  MP_CUDA(cudaGetLastError());
  return MP_OK;
}

extern "C" int mp_fp64_peak_tflops(int32_t device, double* tflops) {
  if (!tflops) return fail(MP_ERR_BAD_ARG, "mp_fp64_peak_tflops: null pointer");
  const int rc = select_device(device, "mp_fp64_peak_tflops");
  if (rc) return rc;
  cudaDeviceProp prop;
  MP_CUDA(cudaGetDeviceProperties(&prop, device));
  DevBuf<double> d;
  MP_CUDA(d.ensure(1));
  const int blocks = prop.multiProcessorCount * 8, iters = 4096;
  struct Events {   // destroyed on every path
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    ~Events() {
      if (e0) cudaEventDestroy(e0);
      if (e1) cudaEventDestroy(e1);
    }
  } ev;
  MP_CUDA(cudaEventCreate(&ev.e0));
  MP_CUDA(cudaEventCreate(&ev.e1));
  double best = 0.0;
  for (int rep = 0; rep < 6; ++rep) {
    MP_CUDA(cudaEventRecord(ev.e0));
    dfma_peak_kernel<<<blocks, 256>>>(d.get(), iters, 1.0 + rep);
    MP_CUDA(cudaEventRecord(ev.e1));
    MP_CUDA(cudaEventSynchronize(ev.e1));
    float ms = 0;
    MP_CUDA(cudaEventElapsedTime(&ms, ev.e0, ev.e1));
    const double flops = 2.0 * 64.0 * iters * 256.0 * blocks;
    if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
  }
  *tflops = best;
  return MP_OK;
}
