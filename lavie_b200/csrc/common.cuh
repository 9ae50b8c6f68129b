// Shared device/host helpers for the lavie_b200 kernels (sm_100a only).
// Thin inline-PTX wrappers: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld),
// UMMA shared-memory + instruction descriptors.  Bit layouts follow the PTX ISA tcgen05 chapter.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/lavie_b200.h"

// ---------------------------------------------------------------------------------------------
// Host-side error plumbing (C ABI: never throw, never exit)
// ---------------------------------------------------------------------------------------------
void lavie_set_error(const char* fmt, ...);
int lavie_check_launch(const char* what);

#define LAVIE_REQUIRE(cond, code, ...)      \
  do {                                      \
    if (!(cond)) {                          \
      lavie_set_error(__VA_ARGS__);         \
      return (code);                        \
    }                                       \
  } while (0)

// Tensor-map creation (driver entry point resolved at run time; see tma_host.cu)
int lavie_make_tmap(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                    const uint64_t* strides_bytes /* rank-1 entries */, const uint32_t* box,
                    CUtensorMapSwizzle swizzle);

int lavie_make_tmap_im2col(CUtensorMap* map, const void* base, int N, int H, int W, int C, int channels, int pixels,
                           int stride, int lower_w, int lower_h, int upper_w, int upper_h);

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch (PDL): every kernel of the library is launched with
// cudaLaunchAttributeProgrammaticStreamSerialization, calls griddepcontrol.launch_dependents at its very start and
// griddepcontrol.wait before it touches memory a predecessor may have written.  The next kernel's CTAs can therefore
// be scheduled, set up barriers / TMEM / descriptors and park at the wait while the current kernel drains, instead of
// paying launch latency + prologue after it (~2-4 us per launch x ~550 launches per step).
// ---------------------------------------------------------------------------------------------
extern int g_lavie_pdl;       // 1 = on (default); lavie_debug_set(3, 0) turns it off for A/B timing
extern void* g_lavie_debug_buf; // device scratch for the clock64 timelines (lavie_debug_buffer), nullptr = off
extern int g_lavie_xattn;     // attention: single-pass kernel for Sk <= 80 on/off; lavie_debug_set(8, v)
extern int g_lavie_attn_poly; // attention: every n-th exp2 on the FMA pipe (0 = none); lavie_debug_set(4, n)

// Per-DEVICE lazily configured kernel attributes.  cudaFuncSetAttribute(MaxDynamicSharedMemorySize) applies to the
// current device only, and one process may drive several GPUs (one host thread per device), so the "already
// configured" state is an array indexed by cudaGetDevice(); the slow path is serialised by a mutex (host.cu).
constexpr int LAVIE_MAX_DEVICES = 64;
struct LavieSmemConfig {
  int bytes[LAVIE_MAX_DEVICES];     // static storage: zero-initialised
};
int lavie_current_device();
int lavie_num_sms();                // SM count of the current device (cached per device)
int lavie_config_smem_impl(const void* func, int bytes, LavieSmemConfig* st, const char* what);

#ifdef __CUDACC__
template <typename K>
inline int lavie_config_smem(K kernel, int bytes, LavieSmemConfig* st, const char* what) {
  return lavie_config_smem_impl(reinterpret_cast<const void*>(kernel), bytes, st, what);
}

template <typename... KArgs, typename... Args>
inline void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = g_lavie_pdl;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
// start of every kernel: let the dependent grid begin its prologue, then wait for our own predecessors
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_prologue() {
  pdl_launch_dependents();
  pdl_wait();
}

// ---------------------------------------------------------------------------------------------
// Small device utilities
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float2 unpack_bf16(uint32_t w) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&w);
  return __bfloat1622float2(v);
}
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// 2^x on the FMA/ALU pipes (no MUFU): round-to-nearest split x = n + f, f in [-0.5, 0.5], degree-3 polynomial for
// 2^f, exponent n added into the float's exponent field.  Relative error <= 2.3e-4 -- an order of magnitude under the
// bf16 rounding the attention probabilities get anyway.  The softmax loop is bound by the 16-lane/clk MUFU unit;
// evaluating a fraction of the exponentials here balances the two pipes (the trick FlashAttention-4 uses on Blackwell).
__device__ __forceinline__ float exp2_poly(float x) {
  x = fmaxf(x, -125.0f);
  const float t = x + 12582912.0f;            // 1.5 * 2^23: the integer part lands in the low mantissa bits
  const float f = x - (t - 12582912.0f);
  float p = fmaf(f, 0.05485820025205612f, 0.24183107912540436f);
  p = fmaf(p, f, 0.6932342052459717f);
  p = fmaf(p, f, 0.9999654293060303f);
  return __int_as_float(__float_as_int(p) + (__float_as_int(t) << 23));
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
__device__ __forceinline__ float silu_f(float x) { return __fdividef(x, 1.0f + __expf(-x)); }
__device__ __forceinline__ float gelu_erf_f(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }
// Exact-form (erf) GELU at 7 FMA-pipe instructions + 1 MUFU, for epilogues that run it on every accumulator element:
//   Phi(-t) = erfc(t / sqrt 2) / 2 = 2^-q(t),  q(t) = 1 + t * Q(t),  Q = degree-4 minimax fit on t in [0, 6]
//   (leading coefficient > 0, so q keeps growing and 2^-q -> 0 for any larger t);
//   gelu(x) = x * Phi(x) = max(x, 0) - |x| * Phi(-|x|).
// |gelu_fast - gelu_erf| <= 1.6e-6 over the whole real line (fit + fp32 evaluation, tools/fit_gelu.py), i.e. three
// orders of magnitude below the bf16 rounding of the result.
__device__ __forceinline__ float gelu_fast_f(float x) {
  const float t = fabsf(x);
  float q = fmaf(t, 0.0005355844041332603f, -0.007474260404706001f);
  q = fmaf(q, t, 0.052688680589199066f);
  q = fmaf(q, t, 0.4591757357120514f);
  q = fmaf(q, t, 1.1511057615280151f);
  q = fmaf(q, t, 1.0f);
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-q));
  return fmaf(-t, e, fmaxf(x, 0.0f));
}

// ---------------------------------------------------------------------------------------------
// mbarrier
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Suspend-time hint: the waiting thread sleeps in hardware until the phase completes (or the hint elapses) instead of
// re-issuing the probe every few cycles -- in the attention kernel the probe loops were ~15 % of all issued instructions.
constexpr uint32_t kMbarSuspendHintNs = 20000;
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2, %3;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(kMbarSuspendHintNs)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must trap (visible CUDA error) instead of hanging the GPU box.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 22)) __trap();
  }
}

// ---------------------------------------------------------------------------------------------
// TMA tiled loads (global -> shared, completion on an mbarrier)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, "
      "%6}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
// generic-proxy smem writes -> visible to the async proxy (TMA / tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---------------------------------------------------------------------------------------------
// tcgen05: TMEM allocation, MMA, commit, loads
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* slot_in_smem, uint32_t ncols) {   // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_in_smem)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {          // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]; one thread issues for the CTA.
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// same with the A operand in tensor memory (lane = row, one 32-bit column = two consecutive K elements)
__device__ __forceinline__ void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier once every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread t of the warp gets TMEM lane (lane_base + t).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_wait_st() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// ---------------------------------------------------------------------------------------------
// UMMA descriptors
// ---------------------------------------------------------------------------------------------
// Shared-memory matrix descriptor, 128-byte swizzle.  Fields (PTX ISA "shared memory descriptor"):
//   [0,14)  start address >> 4      [16,30) leading byte offset >> 4     [32,46) stride byte offset >> 4
//   [46,48) version = 1 (sm_100)    [49,52) base offset = 0              [61,64) layout: 2 = SWIZZLE_128B
// K-major operand (rows of 64 bf16 = 128 B): SBO = 1024 (8 rows), LBO unused (1).
// MN-major operand (64 MN-elements contiguous per 128-B row, rows run along K): SBO = 1024 (8 K-rows),
//   LBO = byte distance between consecutive 64-wide MN chunks.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// Instruction descriptor for kind::f16, BF16 x BF16 -> FP32 (PTX ISA "instruction descriptor"):
//   [4,6) D fmt (1 = f32)  [7,10) A fmt (1 = bf16)  [10,13) B fmt (1 = bf16)  [15] A major (0 = K)  [16] B major
//   [17,23) N >> 3         [24,29) M >> 4
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int m, int n, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(a_mn_major) << 15) |
         (static_cast<uint32_t>(b_mn_major) << 16) | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>(m >> 4) << 24);
}
#endif  // __CUDACC__
