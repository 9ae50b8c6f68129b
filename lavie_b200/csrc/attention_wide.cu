// Single-head wide attention of the x4-upscaler VAE decoder's mid block (sm_100a).
//
//  lavie_attention_wide_bf16   O = softmax(Q K^T) V for one head of d = 512 channels, batched over frames, on tcgen05 /
//                              TMEM with TMA-staged tiles.  The 512^-1/2 scale is folded into the query projection by
//                              the caller (lavie_b200/vae.py), so the scores leave the MMA already scaled.
//
// Why not attn_fwd_kernel<512>: its Q tile alone would be 128 KB of shared memory (Q + K + V: 256 KB), and a 128 x 512
// fp32 O accumulator fills all 512 TMEM columns, leaving none for S.
//
// Layout: two CTAs per 128-query tile of one frame.  CTA "half" h owns the output columns O[:, 256h : 256h + 256]; both
// compute the full S = Q K^T of every key tile (that product is executed twice: 1.5x the algorithmic 4 S^2 d FLOPs),
// and nothing is exchanged between CTAs.  128 threads of softmax (thread t = query row t = TMEM lane t) + one control
// warp (TMA + MMA issue), as attn_fwd_kernel.  Per 64-key tile j:
//   S(j) = Q K(j)^T  (32 MMAs of K = 16, fp32 into TMEM buffer j & 1)
//   softmax warps: S(j) -> registers -> p = exp2(s log2e - m_used) -> bf16 P(j) over the first 32 columns of S(j)
//   O_h += P(j) V(j)[:, half]  (A operand from TMEM, V MN-major from shared memory)
// S is double-buffered, so the softmax of tile j + 1 runs while the tensor core executes P(j) V(j) and Q K(j+2)^T.
// The running maximum moves lazily (only when it grows by more than 2^8), and the O rescale that follows waits for the
// previous P V to retire.
//
// Budget per CTA (one CTA per SM):
//   shared memory  Q 128 x 512 bf16 (8 swizzled 64-column slabs)   131072 B
//                  K  64 x 512 bf16 (8 slabs)                         65536 B
//                  V  64 x 256 bf16 (this half's 4 slabs)             32768 B
//                  1024-B alignment pad + 10 barriers + TMEM slot      1152 B   -> 230528 B <= 227 KB (232448 B)
//   TMEM           S buffers 2 x 64 columns + O 256 columns = 384 -> one 512-column allocation
// Keys and queries past S are zero-filled by the TMA (3-D tensor maps: column, token, frame) and masked in the softmax;
// query rows past S are not stored.  Frame and row offsets are 64-bit: N * S * 512 may pass 2^31 elements.
// Deterministic: every output element is written once by one thread, no atomics.
#include "common.cuh"

namespace {

constexpr int WA_M = 128;                    // queries per CTA
constexpr int WA_N = 64;                     // keys per tile
constexpr int WA_D = 512;                    // head width (Q K^T contraction)
constexpr int WA_DV = 256;                   // output columns per CTA
constexpr int WA_QC = WA_D / 64;             // 64-column slabs of Q / K
constexpr int WA_VC = WA_DV / 64;            // 64-column slabs of this CTA's V half
constexpr int WA_Q_SLAB = WA_M * 128;        // bytes of one slab of a 128-row tile
constexpr int WA_KV_SLAB = WA_N * 128;       // bytes of one slab of a 64-row tile
constexpr int WA_SMEM = WA_QC * WA_Q_SLAB + WA_QC * WA_KV_SLAB + WA_VC * WA_KV_SLAB + 1024 + 128;
constexpr uint32_t WA_TMEM_COLS = 512;
constexpr int WA_THREADS = 160;              // warps 0-3: softmax, warp 4: TMA + MMA issue
static_assert(WA_SMEM <= 227 * 1024, "wide attention: shared memory over budget");
static_assert(2 * WA_N + WA_DV <= (int)WA_TMEM_COLS, "wide attention: TMEM over budget");

struct WideParams {
  int S;
  long long ldo;
  __nv_bfloat16* o;
};

__global__ void __launch_bounds__(WA_THREADS, 1)
attn_wide_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                 const __grid_constant__ CUtensorMap tmap_v, const WideParams p) {
  pdl_launch_dependents();
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + WA_QC * WA_Q_SLAB;
  uint8_t* sV = sK + WA_QC * WA_KV_SLAB;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + WA_VC * WA_KV_SLAB);
  uint64_t* bar_q = bars + 0;        // Q landed
  uint64_t* bar_k = bars + 1;        // K(j) landed, phase j
  uint64_t* bar_v = bars + 2;        // V(j) landed, phase j
  uint64_t* bar_s = bars + 3;        // [2]: S(j) complete in buffer j & 1, phase j >> 1
  // [2]: the 4 softmax warps stored P(j) into buffer j & 1, phase j >> 1.  One barrier per buffer: S(j+1) is complete
  // before every warp has finished tile j, so a fast warp may arrive for tile j + 1 while a slow one still works on tile
  // j; on a single barrier that arrival would count towards tile j.  A warp is never two tiles ahead (S(j+2) is issued
  // only after all four arrived for tile j), so each buffer's barrier sees the arrivals of one tile at a time.
  uint64_t* bar_p_full = bars + 5;
  uint64_t* bar_pv = bars + 7;       // O += P(j) V(j) retired, phase j
  // The last P V retired: one phase only.  A parity wait on bar_pv cannot tell the softmax warps this, because S(j) is
  // issued ahead of P(j-1) V(j-1): when the last S has completed, the last two P V phases may still be open.
  uint64_t* bar_o = bars + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int lane = tid & 31;
  const int q_tile = blockIdx.x >> 1, half = blockIdx.x & 1, frame = blockIdx.z;
  const int n_kv = (p.S + WA_N - 1) / WA_N;

  if (tid == 0) {
    tma_prefetch_desc(&tmap_q);
    tma_prefetch_desc(&tmap_k);
    tma_prefetch_desc(&tmap_v);
    mbar_init(bar_q, 1);
    mbar_init(bar_k, 1);
    mbar_init(bar_v, 1);
    mbar_init(bar_s + 0, 1);
    mbar_init(bar_s + 1, 1);
    mbar_init(bar_p_full + 0, 4);
    mbar_init(bar_p_full + 1, 4);
    mbar_init(bar_pv, 1);
    mbar_init(bar_o, 1);
    mbar_fence_init();
  }
  if (warp == 4) {
    tmem_alloc(tmem_slot, WA_TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_o = tmem_base + 2 * WA_N;  // columns [128, 384)

  if (warp == 4) {
    // =============================== control warp: TMA loads + MMA issue ===============================
    constexpr uint32_t idesc_qk = umma_idesc_bf16(WA_M, WA_N, 0, 0);
    constexpr uint32_t idesc_pv = umma_idesc_bf16(WA_M, WA_DV, 0, 1);
    const uint64_t desc_q = umma_desc_sw128(smem_u32(sQ), 16, 1024);
    const uint64_t desc_k = umma_desc_sw128(smem_u32(sK), 16, 1024);
    const uint64_t desc_v = umma_desc_sw128(smem_u32(sV), WA_KV_SLAB, 1024);
    auto issue_qk = [&](int buf) {
#pragma unroll
      for (int kk = 0; kk < WA_D / 16; ++kk) {
        const uint32_t qoff = (kk >> 2) * WA_Q_SLAB + (kk & 3) * 32;
        const uint32_t koff = (kk >> 2) * WA_KV_SLAB + (kk & 3) * 32;
        umma_bf16(tmem_base + buf * WA_N, desc_q + (qoff >> 4), desc_k + (koff >> 4), idesc_qk, kk != 0);
      }
      umma_commit(bar_s + buf);
    };
    auto load_k = [&](int j) {
      mbar_expect_tx(bar_k, WA_QC * WA_KV_SLAB);
      for (int c = 0; c < WA_QC; ++c) tma_load_3d(sK + c * WA_KV_SLAB, &tmap_k, bar_k, c * 64, j * WA_N, frame);
    };
    auto load_v = [&](int j) {
      mbar_expect_tx(bar_v, WA_VC * WA_KV_SLAB);
      for (int c = 0; c < WA_VC; ++c)
        tma_load_3d(sV + c * WA_KV_SLAB, &tmap_v, bar_v, half * WA_DV + c * 64, j * WA_N, frame);
    };
    if (elect_one()) {
      mbar_expect_tx(bar_q, WA_QC * WA_Q_SLAB);
      for (int c = 0; c < WA_QC; ++c) tma_load_3d(sQ + c * WA_Q_SLAB, &tmap_q, bar_q, c * 64, q_tile * WA_M, frame);
      load_k(0);
      load_v(0);
    }
    __syncwarp();
    mbar_wait(bar_q, 0);
    mbar_wait(bar_k, 0);
    tc_fence_after();
    if (elect_one()) issue_qk(0);
    __syncwarp();
    if (n_kv > 1) {
      mbar_wait(bar_s + 0, 0);                   // Q K(0)^T retired: the K buffer is free
      if (elect_one()) load_k(1);
      __syncwarp();
      mbar_wait(bar_k, 1);
      tc_fence_after();
      if (elect_one()) issue_qk(1);
      __syncwarp();
    }
    for (int j = 0; j < n_kv; ++j) {
      const int buf = j & 1;
      const int kv_len = min(WA_N, p.S - j * WA_N);
      if (j + 2 < n_kv) {                        // K(j+2) streams in as soon as Q K(j+1)^T has read K(j+1)
        mbar_wait(bar_s + ((j + 1) & 1), ((j + 1) >> 1) & 1);
        if (elect_one()) load_k(j + 2);
        __syncwarp();
      }
      mbar_wait(bar_v, j & 1);                   // V(j) landed
      mbar_wait(bar_p_full + buf, (j >> 1) & 1); // P(j) in tensor memory, O rescaled where needed
      tc_fence_after();
      if (elect_one()) {
        const uint32_t tmem_p = tmem_base + buf * WA_N;
        const int nk = (kv_len + 15) >> 4;       // 16 keys = 8 packed columns of P per MMA
        for (int kk = 0; kk < nk; ++kk)
          umma_bf16_ts(tmem_o, tmem_p + kk * 8, desc_v + ((kk * 2048) >> 4), idesc_pv, (j > 0 || kk != 0));
        umma_commit(bar_pv);
        if (j == n_kv - 1) umma_commit(bar_o);
      }
      __syncwarp();
      if (j + 2 < n_kv) {                        // behind P(j) V(j) in issue order: S(j+2) overwrites P(j) only after
        mbar_wait(bar_k, (j + 2) & 1);
        tc_fence_after();
        if (elect_one()) issue_qk(buf);
        __syncwarp();
      }
      if (j + 1 < n_kv) {
        mbar_wait(bar_pv, j & 1);                // P(j) V(j) retired: the V buffer is free
        if (elect_one()) load_v(j + 1);
        __syncwarp();
      }
    }
  } else {
    // =============================== softmax warps: one query row per thread ===========================
    const uint32_t lane_base = static_cast<uint32_t>(warp * 32) << 16;
    constexpr float sc = 1.4426950408889634f;    // log2(e): the 512^-1/2 scale is already in Q
    float m_used = -INFINITY, l_run = 0.f;
    for (int j = 0; j < n_kv; ++j) {
      const int buf = j & 1;
      const uint32_t tmem_s = tmem_base + buf * WA_N;
      const int kv_len = min(WA_N, p.S - j * WA_N);
      mbar_wait(bar_s + buf, (j >> 1) & 1);
      tc_fence_after();
      uint32_t s0[32], s1[32];
      tmem_ld_32x32(tmem_s + lane_base, s0);
      tmem_ld_32x32(tmem_s + lane_base + 32, s1);
      tmem_wait_ld();
      const bool full = (kv_len == WA_N);        // CTA-uniform
      float mx0 = -INFINITY, mx1 = -INFINITY;
      if (full) {
        float mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
        for (int e = 0; e < 32; e += 4) {
          mx0 = fmax3(mx0, __uint_as_float(s0[e]), __uint_as_float(s0[e + 1]));
          mx1 = fmax3(mx1, __uint_as_float(s1[e]), __uint_as_float(s1[e + 1]));
          mx2 = fmax3(mx2, __uint_as_float(s0[e + 2]), __uint_as_float(s0[e + 3]));
          mx3 = fmax3(mx3, __uint_as_float(s1[e + 2]), __uint_as_float(s1[e + 3]));
        }
        mx0 = fmaxf(mx0, mx2);
        mx1 = fmaxf(mx1, mx3);
      } else {
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          if (e < kv_len) mx0 = fmaxf(mx0, __uint_as_float(s0[e]));
          if (32 + e < kv_len) mx1 = fmaxf(mx1, __uint_as_float(s1[e]));
        }
      }
      const float m_tile = fmaxf(mx0, mx1) * sc;
      const bool grow = m_tile > m_used + 8.0f;  // always true for j == 0
      if (j > 0 && __any_sync(0xffffffffu, grow)) {
        // S(j) may have been issued before P(j-1) V(j-1): O is stable only once that product has retired.  S(j) was
        // issued behind P(j-2) V(j-2) and P(j) V(j) waits for this warp, so only phase j - 1 can be open: the parity
        // wait is exact.
        mbar_wait(bar_pv, (j - 1) & 1);
        tc_fence_after();
        const float alpha = grow ? fast_exp2(m_used - m_tile) : 1.0f;
#pragma unroll 4
        for (int c = 0; c < WA_DV / 16; ++c) {
          uint32_t v[16];
          tmem_ld_32x16(tmem_o + lane_base + c * 16, v);
          tmem_wait_ld();
#pragma unroll
          for (int e = 0; e < 16; ++e) v[e] = __float_as_uint(__uint_as_float(v[e]) * alpha);
          tmem_st_32x16(tmem_o + lane_base + c * 16, v);
        }
        tmem_wait_st();
        l_run *= alpha;
      }
      if (grow) m_used = m_tile;
      const float neg_m = -m_used;
      float rs0 = 0.f, rs1 = 0.f;
      auto soft_half = [&](uint32_t (&sv)[32], int c) {
        if (full) {
#pragma unroll
          for (int e = 0; e < 32; e += 2) {
            const float p0 = fast_exp2(fmaf(__uint_as_float(sv[e]), sc, neg_m));
            const float p1 = fast_exp2(fmaf(__uint_as_float(sv[e + 1]), sc, neg_m));
            rs0 += p0;
            rs1 += p1;
            sv[e >> 1] = pack_bf16(p0, p1);
          }
        } else {
#pragma unroll
          for (int e = 0; e < 32; e += 2) {
            const float p0 = (c * 32 + e < kv_len) ? fast_exp2(fmaf(__uint_as_float(sv[e]), sc, neg_m)) : 0.f;
            const float p1 = (c * 32 + e + 1 < kv_len) ? fast_exp2(fmaf(__uint_as_float(sv[e + 1]), sc, neg_m)) : 0.f;
            rs0 += p0;
            rs1 += p1;
            sv[e >> 1] = pack_bf16(p0, p1);
          }
        }
      };
      soft_half(s0, 0);
      soft_half(s1, 1);
      l_run += rs0 + rs1;
      {
        uint32_t pk[32];
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          pk[e] = s0[e];
          pk[16 + e] = s1[e];
        }
        tmem_st_32x32(tmem_s + lane_base, pk);
        tmem_wait_st();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_p_full + buf);
    }
    // ---- O complete ----
    mbar_wait(bar_o, 0);
    tc_fence_after();
    const float inv = 1.f / l_run;
    const int qrow = q_tile * WA_M + tid;
    __nv_bfloat16* dst = p.o + (static_cast<long long>(frame) * p.S + qrow) * p.ldo + half * WA_DV;
#pragma unroll 2
    for (int c = 0; c < WA_DV / 16; ++c) {
      uint32_t v[16];
      tmem_ld_32x16(tmem_o + lane_base + c * 16, v);
      tmem_wait_ld();
      if (qrow < p.S) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          uint4 o;
          o.x = pack_bf16(__uint_as_float(v[8 * h]) * inv, __uint_as_float(v[8 * h + 1]) * inv);
          o.y = pack_bf16(__uint_as_float(v[8 * h + 2]) * inv, __uint_as_float(v[8 * h + 3]) * inv);
          o.z = pack_bf16(__uint_as_float(v[8 * h + 4]) * inv, __uint_as_float(v[8 * h + 5]) * inv);
          o.w = pack_bf16(__uint_as_float(v[8 * h + 6]) * inv, __uint_as_float(v[8 * h + 7]) * inv);
          *reinterpret_cast<uint4*>(dst + c * 16 + h * 8) = o;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    tmem_dealloc(tmem_base, WA_TMEM_COLS);
  }
}

// (512 columns, S tokens, frames) view of a row-major [frames * S, 512] matrix with row stride ld
int make_wide_map(CUtensorMap* map, const void* base, long long ld, int S, int frames, int box_rows) {
  const uint64_t dims[3] = {static_cast<uint64_t>(WA_D), static_cast<uint64_t>(S), static_cast<uint64_t>(frames)};
  const uint64_t strides[2] = {static_cast<uint64_t>(ld) * 2, static_cast<uint64_t>(ld) * 2 * static_cast<uint64_t>(S)};
  const uint32_t box[3] = {64, static_cast<uint32_t>(box_rows), 1};
  return lavie_make_tmap(map, base, 3, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

bool wide_al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace

extern "C" int lavie_attention_wide_bf16(const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, void* o,
                                         int ldo, int frames, int S, cudaStream_t stream) {
  LAVIE_REQUIRE(q && k && v && o && frames >= 1 && S >= 1, LAVIE_ERR_SHAPE,
                "attention_wide: bad sizes frames=%d S=%d", frames, S);
  LAVIE_REQUIRE(frames <= 65535 && S <= 0x7FFFFFFF - WA_M, LAVIE_ERR_SHAPE,
                "attention_wide: grid too large (frames=%d S=%d)", frames, S);
  LAVIE_REQUIRE(ldq >= WA_D && ldk >= WA_D && ldv >= WA_D && ldo >= WA_D, LAVIE_ERR_SHAPE,
                "attention_wide: row strides must be >= 512 (ldq=%d ldk=%d ldv=%d ldo=%d)", ldq, ldk, ldv, ldo);
  LAVIE_REQUIRE(wide_al16(q) && wide_al16(k) && wide_al16(v) && wide_al16(o) && ldq % 8 == 0 && ldk % 8 == 0 &&
                    ldv % 8 == 0 && ldo % 8 == 0,
                LAVIE_ERR_ALIGN, "attention_wide: 16-byte aligned pointers and row strides required");
  // TMA global strides must stay below 2^40 bytes
  const long long max_ld = ldq > ldk ? (ldq > ldv ? ldq : ldv) : (ldk > ldv ? ldk : ldv);
  LAVIE_REQUIRE(static_cast<long long>(S) * max_ld * 2 < (1LL << 40), LAVIE_ERR_SHAPE,
                "attention_wide: frame stride S*ld=%lld elements too large for a tensor map",
                static_cast<long long>(S) * max_ld);
  CUtensorMap mq, mk, mv;
  int rc = make_wide_map(&mq, q, ldq, S, frames, WA_M);
  if (rc) return rc;
  rc = make_wide_map(&mk, k, ldk, S, frames, WA_N);
  if (rc) return rc;
  rc = make_wide_map(&mv, v, ldv, S, frames, WA_N);
  if (rc) return rc;
  static LavieSmemConfig configured;
  rc = lavie_config_smem(attn_wide_kernel, WA_SMEM, &configured, "attn_wide_kernel");
  if (rc) return rc;
  WideParams p;
  p.S = S;
  p.ldo = ldo;
  p.o = static_cast<__nv_bfloat16*>(o);
  const dim3 grid(2 * ((S + WA_M - 1) / WA_M), 1, frames);
  launch_pdl(attn_wide_kernel, grid, WA_THREADS, WA_SMEM, stream, mq, mk, mv, p);
  return lavie_check_launch("attn_wide_kernel");
}
