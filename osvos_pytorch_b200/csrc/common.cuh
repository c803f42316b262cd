// Shared host/device helpers for libosvos_b200: status codes, environment switches, the driver entry
// point for cuTensorMapEncodeTiled (resolved at run time so the library loads on
// a box without libcuda), the persistent-kernel launch, split-bf16 arithmetic.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/osvos_b200.h"

namespace osvos {

#define OSVOS_CHECK_ARG(cond)                                                              \
  do {                                                                                     \
    if (!(cond)) {                                                                         \
      set_last_error("%s:%d: invalid argument: %s", __FILE__, __LINE__, #cond);            \
      return OSVOS_ERR_INVALID_ARGUMENT;                                                   \
    }                                                                                      \
  } while (0)

#define OSVOS_CHECK_CUDA(expr)                                                             \
  do {                                                                                     \
    cudaError_t e__ = (expr);                                                              \
    if (e__ != cudaSuccess) {                                                              \
      set_last_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__)); \
      return OSVOS_ERR_CUDA;                                                               \
    }                                                                                      \
  } while (0)

void set_last_error(const char* fmt, ...);

// Library switches (environment variables; the list, the defaults and the caching rule are in runtime.cu).
// env_int: atoi of the value, `dflt` when unset.  env_is: the variable is set to exactly `value`.
int env_int(const char* name, int dflt);
bool env_is(const char* name, const char* value);

// Encodes a tiled tensor map over a bf16 / fp32 tensor. dims/strides innermost first;
// strides[0] is implied by the element size. Returns an OSVOS_* status.
int encode_tensor_map(CUtensorMap* map, CUtensorMapDataType dtype, int elem_bytes, int rank, const void* base,
                      const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box,
                      CUtensorMapSwizzle swizzle);
// Split-bf16 NHWC activation [n, h, w, c]: the hi and lo maps, box {64 channels, box_w, box_h, 1}, SWIZZLE_128B.
// A NULL `lo` (one-plane fast mode) encodes the hi plane twice, so that both maps are valid.
int encode_act_maps(CUtensorMap* hi, CUtensorMap* lo, const void* base_hi, const void* base_lo, int n, int h, int w, int c,
                    int box_w, int box_h);
// Packed weights [plane][tap][rows][cin] (two planes, hi then lo): the hi and lo maps, box {64, box_rows, box_taps},
// SWIZZLE_128B.
int encode_weight_maps(CUtensorMap* hi, CUtensorMap* lo, const void* w_packed, int rows, int cin, int box_rows,
                       int box_taps);

int device_sm_count();

// Programmatic dependent launch: OSVOS_PDL, overridden by osvos_set_pdl(); otherwise plain stream-ordered launches.
bool pdl_enabled();

// Launches `kern` on `stream`; with PDL enabled the launch carries the programmatic-stream-serialization attribute,
// so the kernel's prologue (barrier init, TMEM allocation, descriptor prefetch) overlaps the previous kernel's tail.
// ONLY for kernels that execute pdl_wait() (ptx.cuh) before their first dependent global access.
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                     Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// Opt-in to > 48 KiB of dynamic shared memory, once per (kernel, DEVICE): the attribute is per device, and the engine
// supports modules on any GPU of the process.  Every instantiation of this template keeps its own bit mask of devices.
template <auto Kern>
static inline cudaError_t ensure_dynamic_smem(int bytes) {
  static uint64_t done_mask = 0;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev < 64 && ((done_mask >> dev) & 1ull)) return cudaSuccess;
  e = cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess && dev < 64) done_mask |= 1ull << dev;
  return e;
}

// Persistent CTAs: one per work item up to one per SM; CTA b takes items b, b + grid, b + 2 grid, ...
static inline int persistent_grid(int items, int sms) { return items < sms ? items : sms; }

// Launches the persistent kernel `Kern` over `items` work items: shared-memory opt-in, persistent_grid on this device's
// SMs, launch_pdl (so, like launch_pdl, only for kernels that execute pdl_wait()).
template <auto Kern, typename... Args>
static inline cudaError_t launch_persistent(int items, int threads, int smem, cudaStream_t stream, Args&&... args) {
  const cudaError_t e = ensure_dynamic_smem<Kern>(smem);
  if (e != cudaSuccess) return e;
  return launch_pdl(Kern, dim3(persistent_grid(items, device_sm_count())), dim3(threads), smem, stream,
                    static_cast<Args&&>(args)...);
}

// ---- split-bf16 ("bf16x2") representation of an fp32 value: v ~= hi + lo ------
__device__ __forceinline__ void split_bf16(float v, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(v);
  lo = __float2bfloat16_rn(v - __bfloat162float(hi));
}
__device__ __forceinline__ uint32_t pack_bf16x2(__nv_bfloat16 a, __nv_bfloat16 b) {
  return static_cast<uint32_t>(__bfloat16_as_ushort(a)) | (static_cast<uint32_t>(__bfloat16_as_ushort(b)) << 16);
}
// Grid-wide "last block finalizes" pattern: true in exactly one block, the last one to arrive, after every other
// block's prior global writes / atomics have become visible.  `counter` must be zero at launch.
__device__ __forceinline__ bool last_block_arrives(unsigned int* counter) {
  __shared__ bool is_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = atomicAdd(counter, 1u) == gridDim.x * gridDim.y - 1;
  __syncthreads();
  if (is_last) __threadfence();
  return is_last;
}

__device__ __forceinline__ float bf16_lo_to_float(uint32_t packed) { return __uint_as_float(packed << 16); }
__device__ __forceinline__ float bf16_hi_to_float(uint32_t packed) { return __uint_as_float(packed & 0xFFFF0000u); }

}  // namespace osvos
