// Host-side helpers shared by the launchers: error reporting, TMA tensor-map encoding.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/adp_b200.h"

namespace adp {

int set_error(const char* fmt, ...);  // returns non-zero, records the message (thread-local)

#define ADP_CHECK(cond, ...)                         \
  do {                                               \
    if (!(cond)) return ::adp::set_error(__VA_ARGS__); \
  } while (0)

#define ADP_CUDA(expr)                                                                   \
  do {                                                                                   \
    cudaError_t e_ = (expr);                                                             \
    if (e_ != cudaSuccess)                                                               \
      return ::adp::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_),    \
                              __FILE__, __LINE__);                                       \
  } while (0)

#define ADP_LAUNCH_CHECK() ADP_CUDA(cudaGetLastError())

// bf16 tensor map, up to 4 dims.  dims[0] is the contiguous dimension; strides_bytes[i] is
// the byte stride of dims[i+1].  swizzle_bytes in {0, 32, 64, 128}.
int make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                   const uint64_t* strides_bytes, const uint32_t* box, int swizzle_bytes);

inline cudaStream_t as_stream(adp_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device attribute: remember the largest
// value set so far for each device (one static cache per kernel instantiation at the call site).
struct SmemAttrCache { size_t set[64] = {}; };
template <typename Kern>
inline cudaError_t ensure_dyn_smem(Kern kernel, size_t bytes, SmemAttrCache& cache) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  size_t& cur = cache.set[dev & 63];
  // always opt in on first use: static + dynamic shared memory together may exceed the 48 KB
  // default even when the dynamic part alone does not
  if (bytes <= cur) return cudaSuccess;
  e = cudaFuncSetAttribute((const void*)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess) cur = bytes;
  return e;
}

// Every kernel is launched with the programmatic-dependent-launch attribute: kernel N+1 may
// start (set up smem / mbarriers / TMEM, prefetch tensor maps) while kernel N drains; it calls
// griddepcontrol.wait before its first global-memory access.  adp_debug_set(6, 0) disables.
extern int g_pdl;
template <typename Kern, typename... Args>
inline cudaError_t launch_k(Kern kernel, dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                            Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = g_pdl ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  void* ptrs[] = {(void*)&args...};
  return cudaLaunchKernelExC(&cfg, (const void*)kernel, ptrs);
}

}  // namespace adp
