// magprop_abi.hpp -- what the host code of every translation unit of the library shares (host only, internal):
// the thread's last error message behind mp_last_error, the CUDA-call check, device selection, and DevBuf, the
// device buffer that frees itself.  It includes only the public headers: the per-walker core and its disc tables
// are compiled into magprop_kernels.cu alone.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <string>
#include <vector>

#include "../../include/magprop_b200.h"
#include "../../include/magprop_band.h"
#include "../../include/magprop_smc.h"

namespace mp {

extern thread_local std::string g_err;   // defined in magprop_device.cu

inline int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

// MP_ERR_CUDA, with the message "func: call: CUDA's reason" (out of line: MP_CUDA expands at every call site).
int fail_cuda(const char* func, const char* call, cudaError_t e);

}  // namespace mp

// Returns MP_ERR_CUDA from the calling function when `call` does not return cudaSuccess.
#define MP_CUDA(call)                                                      \
  do {                                                                     \
    cudaError_t e_ = (call);                                               \
    if (e_ != cudaSuccess) return mp::fail_cuda(__func__, #call, e_);      \
  } while (0)

namespace mp {

// Makes `device` current for the entry point `who`; a device that does not exist is an error (there is no CPU path).
inline int select_device(int device, const char* who) {
  if (device < 0 || device >= mp_device_count())
    return fail(MP_ERR_CUDA, std::string(who) + ": no such CUDA device (magprop_b200 has no CPU path)");
  const cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) return fail(MP_ERR_CUDA, std::string(who) + ": cudaSetDevice: " + cudaGetErrorString(e));
  return MP_OK;
}

// [p, p + bytes) and [q, q + qbytes) share a byte (a null range shares none).
inline bool overlaps(const void* p, __int128 bytes, const void* q, __int128 qbytes) {
  if (!p || !q) return false;
  const __int128 a = (__int128)(uintptr_t)p, b = (__int128)(uintptr_t)q;
  return a < b + qbytes && b < a + bytes;
}

// A device array that owns its memory: moved, never copied, and freed by its destructor.  Its size is the capacity in elements.
// cudaFree waits for the device, so memory that a launch still reads is released only after that launch.
template <typename T>
class DevBuf {
 public:
  DevBuf() = default;
  DevBuf(DevBuf&& o) noexcept : p_(o.p_), n_(o.n_) {
    o.p_ = nullptr;
    o.n_ = 0;
  }
  ~DevBuf() { cudaFree(p_); }

  T* get() const { return p_; }
  size_t size() const { return n_; }

  // Grow-only: room for at least n elements, contents not kept.  Frees before it allocates; after a failed
  // allocation the buffer is empty.
  cudaError_t ensure(size_t n) {
    if (n <= n_) return cudaSuccess;
    cudaFree(p_);
    p_ = nullptr;
    n_ = 0;
    const cudaError_t e = cudaMalloc((void**)&p_, n * sizeof(T));
    if (e != cudaSuccess) p_ = nullptr;
    else n_ = n;
    return e;
  }

  // A device copy of v (an empty v leaves the buffer as it is).
  cudaError_t upload(const std::vector<T>& v) {
    if (v.empty()) return cudaSuccess;
    cudaError_t e = ensure(v.size());
    if (e == cudaSuccess) e = cudaMemcpy(p_, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
    return e;
  }

 private:
  T* p_ = nullptr;
  size_t n_ = 0;
};

}  // namespace mp
