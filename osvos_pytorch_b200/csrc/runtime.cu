// Library-level plumbing: version, thread-local error text, environment switches, tensor-map encoding
// through a run-time resolved driver entry point (no link-time libcuda
// dependency, so the .so loads on a CPU-only box for the symbol tests).
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <mutex>
#include <optional>
#include <string>

#include "common.cuh"

namespace osvos {

static thread_local char g_err[512] = "";

void set_last_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess) {
      fn = reinterpret_cast<EncodeTiledFn>(p);
    }
  });
  return fn;
}

int encode_tensor_map(CUtensorMap* map, CUtensorMapDataType dtype, int elem_bytes, int rank, const void* base,
                      const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box,
                      CUtensorMapSwizzle swizzle) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) {
    set_last_error("cuTensorMapEncodeTiled is not available (no CUDA driver?)");
    return OSVOS_ERR_CUDA;
  }
  cuuint64_t gdims[5];
  cuuint64_t gstrides[4];
  cuuint32_t gbox[5];
  cuuint32_t estr[5];
  for (int i = 0; i < rank; ++i) {
    gdims[i] = dims[i];
    gbox[i] = box[i];
    estr[i] = 1;
    if (i > 0) gstrides[i - 1] = strides_bytes[i - 1];
  }
  (void)elem_bytes;
  CUresult r = fn(map, dtype, static_cast<cuuint32_t>(rank), const_cast<void*>(base), gdims, gstrides, gbox, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_last_error("cuTensorMapEncodeTiled failed with CUresult %d (rank %d, dims %llu %llu %llu %llu, box %u %u %u %u)",
                   (int)r, rank, (unsigned long long)dims[0], (unsigned long long)dims[1],
                   (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 3 ? dims[3] : 0), box[0],
                   box[1], rank > 2 ? box[2] : 0, rank > 3 ? box[3] : 0);
    return OSVOS_ERR_CUDA;
  }
  return OSVOS_OK;
}

int encode_act_maps(CUtensorMap* hi, CUtensorMap* lo, const void* base_hi, const void* base_lo, int n, int h, int w, int c,
                    int box_w, int box_h) {
  const uint64_t dims[4] = {(uint64_t)c, (uint64_t)w, (uint64_t)h, (uint64_t)n};
  const uint64_t strides[3] = {(uint64_t)c * 2, (uint64_t)w * c * 2, (uint64_t)h * w * c * 2};
  const uint32_t box[4] = {64, (uint32_t)box_w, (uint32_t)box_h, 1};
  const int rc = encode_tensor_map(hi, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, 4, base_hi, dims, strides, box,
                                   CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  return encode_tensor_map(lo, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, 4, base_lo ? base_lo : base_hi, dims, strides, box,
                           CU_TENSOR_MAP_SWIZZLE_128B);
}

int encode_weight_maps(CUtensorMap* hi, CUtensorMap* lo, const void* w_packed, int rows, int cin, int box_rows,
                       int box_taps) {
  const size_t plane = static_cast<size_t>(9) * rows * cin;  // elements
  const uint64_t dims[3] = {(uint64_t)cin, (uint64_t)rows, 9};
  const uint64_t strides[2] = {(uint64_t)cin * 2, (uint64_t)rows * cin * 2};
  const uint32_t box[3] = {64, (uint32_t)box_rows, (uint32_t)box_taps};
  const __nv_bfloat16* wp = static_cast<const __nv_bfloat16*>(w_packed);
  const int rc = encode_tensor_map(hi, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, 3, wp, dims, strides, box,
                                   CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  return encode_tensor_map(lo, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, 3, wp + plane, dims, strides, box,
                           CU_TENSOR_MAP_SWIZZLE_128B);
}

int device_sm_count() {
  static int sms[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (sms[dev] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    sms[dev] = v;
  }
  return sms[dev];
}

// ---- environment switches -----------------------------------------------------------------------------------------
// Every switch of the library is read here, by the same rule: once per process (the first read of a name is kept), or on
// every call when OSVOS_ENV_RELOAD=1 was set at the first read - tests and scripts/ab_env.py flip switches inside one
// process.  The defaults are the measured winners; the other values select A/B arms, cross-checks and diagnosis.
//   OSVOS_HALO_LEAN=1      lean epilogue for plain forward halo launches (conv_common.cuh); 0: the general epilogue
//   OSVOS_CONV_N256=1      256-wide halo tiles where they save a wave; 0: never
//   OSVOS_SPLITACC128=1    N-concatenated split accumulator for 128-wide exact halo tiles; 0: three plain passes
//   OSVOS_S1_SW64=1        fused stage-1 kernel with SWIZZLE_64B conv1_1 operands and a 5-stage weight ring;
//                          0: 128-byte operand rows and 3 stages
//   OSVOS_WGRAD_ROWS=1     weight gradient of Cin = Cout = 64 layers by tap rows; 0: by tap pairs
//   OSVOS_WGRAD_SPLITS     unset: weight-gradient pixel splits chosen by cost; legacy: the first rule, ceil(2 SMs / tiles)
//   OSVOS_SIDE_IMPL        unset: 16-output side convolutions on side_conv.cu; generic: the halo kernel's N = 16 tiles
//   OSVOS_FIRST_IMPL       unset: conv1_1 on the tensor cores (conv_first_tc.cu); simt: the CUDA-core kernel
//   OSVOS_ABLATE=0         timing ablation bit mask of the conv kernels (ConvParams::ablate; results are garbage)
//   OSVOS_PDL=0            programmatic dependent launch; osvos_set_pdl() overrides it
// (The engine's own switches - OSVOS_FUSE_STAGE1, OSVOS_FOLD_SIDE, ... - are read by engine.py on every call.)
static const char* env_str(const char* name) {
  static const bool reload = [] {
    const char* e = getenv("OSVOS_ENV_RELOAD");
    return e != nullptr && atoi(e) != 0;
  }();
  if (reload) return getenv(name);
  static std::mutex mu;
  static std::map<std::string, std::optional<std::string>> first_read;
  std::lock_guard<std::mutex> lock(mu);
  auto it = first_read.find(name);
  if (it == first_read.end()) {
    const char* e = getenv(name);
    it = first_read.emplace(name, e ? std::optional<std::string>(e) : std::nullopt).first;
  }
  return it->second ? it->second->c_str() : nullptr;
}

int env_int(const char* name, int dflt) {
  const char* e = env_str(name);
  return e == nullptr ? dflt : atoi(e);
}

bool env_is(const char* name, const char* value) {
  const char* e = env_str(name);
  return e != nullptr && strcmp(e, value) == 0;
}

// Programmatic dependent launch: process default from OSVOS_PDL, overridden per call sequence by
// osvos_set_pdl() - the engine switches it on around the inference pass (measured +1.4 % there, -1.7 % on the fwd+bwd
// graph: profiles/r01f_pdl_ab.txt).  A captured graph keeps the attribute its launches were captured with.
static int g_pdl_override = -1;   // -1: environment default
bool pdl_enabled() {
  if (g_pdl_override >= 0) return g_pdl_override == 1;
  return env_int("OSVOS_PDL", 0) != 0;
}

}  // namespace osvos

extern "C" int osvos_version(void) { return OSVOS_B200_VERSION; }
extern "C" int osvos_set_pdl(int mode) {
  const int prev = osvos::g_pdl_override;
  osvos::g_pdl_override = mode < 0 ? -1 : (mode != 0 ? 1 : 0);
  return prev;
}
extern "C" const char* osvos_last_error(void) { return osvos::g_err; }
