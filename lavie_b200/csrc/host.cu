// Host-side plumbing of the C ABI: thread-local error string, launch checking, TMA tensor-map encoding.
#include <stdarg.h>
#include <stdio.h>

#include <mutex>

#include "common.cuh"

namespace {
thread_local char g_error[512] = "";

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;

typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t,
                                   const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeIm2colFn g_encode_im2col = nullptr;

EncodeIm2colFn get_encode_im2col() {
  if (g_encode_im2col) return g_encode_im2col;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || fn == nullptr) {
    cudaGetLastError();
    return nullptr;
  }
  g_encode_im2col = reinterpret_cast<EncodeIm2colFn>(fn);
  return g_encode_im2col;
}

EncodeTiledFn get_encode() {
  if (g_encode) return g_encode;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || fn == nullptr) {
    cudaGetLastError();
    return nullptr;
  }
  g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  return g_encode;
}
}  // namespace

void lavie_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}

int lavie_check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    lavie_set_error("%s: %s (%d)", what, cudaGetErrorString(e), static_cast<int>(e));
    return LAVIE_ERR_CUDA;
  }
  return LAVIE_OK;
}

int lavie_make_tmap(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                    const uint64_t* strides_bytes, const uint32_t* box, CUtensorMapSwizzle swizzle) {
  EncodeTiledFn enc = get_encode();
  LAVIE_REQUIRE(enc != nullptr, LAVIE_ERR_DRIVER, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t gdim[5];
  cuuint64_t gstr[4];
  cuuint32_t bx[5];
  cuuint32_t es[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
  }
  for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i];
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, static_cast<cuuint32_t>(rank), const_cast<void*>(base), gdim,
                   gstr, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    lavie_set_error("cuTensorMapEncodeTiled failed: CUresult %d (rank %d, dims %llu x %llu, box %u x %u)",
                    static_cast<int>(r), rank, static_cast<unsigned long long>(dims[0]),
                    static_cast<unsigned long long>(rank > 1 ? dims[1] : 1), box[0], rank > 1 ? box[1] : 1);
    return LAVIE_ERR_DRIVER;
  }
  return LAVIE_OK;
}

// im2col-mode tensor map over a channels-last feature map [N, H, W, C] for a 3x3 convolution: one TMA request
// fetches `pixels` consecutive OUTPUT pixels x `channels` input channels for one filter tap, walking the (W, H, N)
// bounding box and zero-filling the halo (PTX ISA "im2col mode"; same corner convention as CUTLASS:
// lower = -pad_before, upper = pad_after - (filter - 1)).  The box spans the filter windows' first input pixel, from
// `lower` to (extent - 1 + upper), and is walked in steps of `stride`.
int lavie_make_tmap_im2col(CUtensorMap* map, const void* base, int N, int H, int W, int C, int channels, int pixels,
                           int stride, int lower_w, int lower_h, int upper_w, int upper_h) {
  EncodeIm2colFn enc = get_encode_im2col();
  LAVIE_REQUIRE(enc != nullptr, LAVIE_ERR_DRIVER, "cuTensorMapEncodeIm2col is not available from the driver");
  const cuuint64_t gdim[4] = {static_cast<cuuint64_t>(C), static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H),
                              static_cast<cuuint64_t>(N)};
  const cuuint64_t gstr[3] = {static_cast<cuuint64_t>(C) * 2, static_cast<cuuint64_t>(W) * C * 2,
                              static_cast<cuuint64_t>(H) * W * C * 2};
  // 3x3 pad (1, 1): lower = upper = -1; Downsample2D's pad (0, 1): lower = 0, upper = -1.  The 2x2 phase convs of the
  // fused upsample (gemm.cu conv == 3) pad one pixel before (phase 0) or one pixel after (phase 1): lower = upper =
  // phase - 1 per axis.
  const int lower[2] = {lower_w, lower_h};
  const int upper[2] = {upper_w, upper_h};
  const cuuint32_t es[4] = {1, static_cast<cuuint32_t>(stride), static_cast<cuuint32_t>(stride), 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), gdim, gstr, lower, upper,
                   static_cast<cuuint32_t>(channels), static_cast<cuuint32_t>(pixels), es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    lavie_set_error("cuTensorMapEncodeIm2col failed: CUresult %d (N=%d H=%d W=%d C=%d)", static_cast<int>(r), N, H, W, C);
    return LAVIE_ERR_DRIVER;
  }
  return LAVIE_OK;
}

int lavie_current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    cudaGetLastError();
    dev = 0;
  }
  return (dev >= 0 && dev < LAVIE_MAX_DEVICES) ? dev : 0;
}

namespace {
std::mutex g_config_mutex;
int g_sm_count[LAVIE_MAX_DEVICES];
}  // namespace

int lavie_num_sms() {
  const int dev = lavie_current_device();
  int n = g_sm_count[dev];
  if (n > 0) return n;
  std::lock_guard<std::mutex> lock(g_config_mutex);
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) {
    cudaGetLastError();
    n = 148;                          // no device (host-only planning queries): a B200
  }
  g_sm_count[dev] = n;
  return n;
}

int lavie_config_smem_impl(const void* func, int bytes, LavieSmemConfig* st, const char* what) {
  const int dev = lavie_current_device();
  if (st->bytes[dev] >= bytes) return LAVIE_OK;
  std::lock_guard<std::mutex> lock(g_config_mutex);
  if (st->bytes[dev] >= bytes) return LAVIE_OK;
  cudaError_t e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  LAVIE_REQUIRE(e == cudaSuccess, LAVIE_ERR_CUDA, "cudaFuncSetAttribute(%s, %d bytes) on device %d: %s", what, bytes, dev,
                cudaGetErrorString(e));
  st->bytes[dev] = bytes;
  return LAVIE_OK;
}

int g_lavie_pdl = 1;
int g_lavie_xattn = 0;         // lavie_debug_set(8, 1): short key sequences (Sk <= 80) run on the single-pass mma.sync kernel.
                               // Correct, but bound by the legacy HMMA issue rate (~150 TFLOP/s on B200): 85 vs 64 us at the
                               // 40x64 level, 30.5 vs 33 us at 20x32 -> off by default (profiles/r2_notes.md)
int g_lavie_attn_poly = -1;    // -1: per-shape default, 0: all exponentials on the MUFU, 4: every 4th on the FMA pipe
void* g_lavie_debug_buf = nullptr;

extern "C" int lavie_debug_buffer(void* device_ptr) {
  g_lavie_debug_buf = device_ptr;
  return 0;
}

extern "C" const char* lavie_last_error(void) { return g_error; }
extern "C" int lavie_abi_version(void) { return 1; }
