// common.cuh -- shared helpers for the sm_100a kernels of libgpt4roi_b200.so
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/gpt4roi_b200.h"

namespace g4r {

// ---- error plumbing ---------------------------------------------------------
void set_error(const char* fmt, ...);  // defined in api_common.cu
int cuda_fail(cudaError_t e, const char* what);

#define G4R_REQUIRE(cond, ...)        \
  do {                                \
    if (!(cond)) {                    \
      g4r::set_error(__VA_ARGS__);    \
      return G4R_EINVAL;              \
    }                                 \
  } while (0)

#define G4R_CUDA(call)                                        \
  do {                                                        \
    cudaError_t e__ = (call);                                 \
    if (e__ != cudaSuccess) return g4r::cuda_fail(e__, #call); \
  } while (0)

#define G4R_LAUNCH_CHECK(name)                                   \
  do {                                                           \
    cudaError_t e__ = cudaGetLastError();                        \
    if (e__ != cudaSuccess) return g4r::cuda_fail(e__, name);    \
  } while (0)

inline size_t dtype_size(int dt) {
  switch (dt) {
    case G4R_F32: return 4;
    case G4R_F16: return 2;
    case G4R_BF16: return 2;
    case G4R_F64: return 8;
  }
  return 0;
}

int num_sms();  // cached cudaDevAttrMultiProcessorCount of the current device
int sm_budget();  // num_sms() minus the reserve of g4r_set_sm_reserve (grid size of the persistent GEMM kernels)

// ---- programmatic dependent launch (the decode step's kernel chain) -----------------------------------------
// The decode step behind generate() is ~230 short, HBM-bound kernels in one CUDA graph; what separates it from the
// weight-streaming floor is each kernel's ramp-up and tail.  Kernels launched through launch_pdl() may start while
// their predecessor in the stream is still running: they fetch what does not depend on it (their first weight
// block) and then execute pdl_wait(), which returns once the predecessor grid has completed and its writes are
// visible.  Everything read BEFORE pdl_wait() must be constant for the step (weights); everything the predecessor
// produced is read after it, through ordinary (coherent) loads.  Every kernel launched this way must execute
// pdl_wait() before it exits, so completion stays transitive along the chain.
//   pdl_on(): false unless the caller has switched the chain on with g4r_set_pdl(1) (the decode step does; nothing
//   else may -- see api_common.cu).  Off, the kernels launch in plain stream order and pdl_sync() is a no-op.
bool pdl_on();
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_release() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
// prologue of a PDL-aware kernel, after the loads that do not depend on the predecessor have been issued: dependents
// are released once this kernel's own inputs are ready (one kernel of look-ahead; releasing them at kernel start
// measured 3.36 vs 3.34 ms per decode step, profiles/r2_decode_pdl_depth.md)
__device__ __forceinline__ void pdl_sync() {
  pdl_wait();
  pdl_release();
}

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                     dim3 cluster, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int n = 0;
  attr[n].id = cudaLaunchAttributeClusterDimension;
  attr[n].val.clusterDim.x = cluster.x; attr[n].val.clusterDim.y = cluster.y; attr[n].val.clusterDim.z = cluster.z;
  n++;
  if (pdl_on()) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    n++;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// ---- element conversion -----------------------------------------------------
template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// 16-byte vector of N = 16/sizeof(T) elements, widened to fp32 on load.
template <typename T> struct Vec16 {
  static constexpr int N = 16 / sizeof(T);
};

template <typename T>
__device__ __forceinline__ void load16(const T* p, float (&out)[16 / sizeof(T)]) {
  uint4 raw = *reinterpret_cast<const uint4*>(p);
  const T* e = reinterpret_cast<const T*>(&raw);
#pragma unroll
  for (int i = 0; i < 16 / (int)sizeof(T); i++) out[i] = to_f32<T>(e[i]);
}

template <typename T>
__device__ __forceinline__ void store16(T* p, const float (&v)[16 / sizeof(T)]) {
  uint4 raw;
  T* e = reinterpret_cast<T*>(&raw);
#pragma unroll
  for (int i = 0; i < 16 / (int)sizeof(T); i++) e[i] = from_f32<T>(v[i]);
  *reinterpret_cast<uint4*>(p) = raw;
}

// i / d and i % d for a grid-stride element index: 32-bit unsigned arithmetic whenever the index fits (always, for the
// tensors of this path) -- a 64-bit div/mod pair by a run-time divisor costs more instructions than the element's math.
__device__ __forceinline__ void divmod_idx(long long i, int d, long long& q, int& r) {
  if (i >= 0 && i <= 0xffffffffLL) {
    const unsigned ii = (unsigned)i, qq = ii / (unsigned)d;
    q = qq;
    r = (int)(ii - qq * (unsigned)d);
  } else {
    q = i / d;
    r = (int)(i - q * d);
  }
}

}  // namespace g4r
