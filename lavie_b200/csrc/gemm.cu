// tcgen05 GEMM / implicit-GEMM 3x3 convolution for the LaVie denoiser (sm_100a), CTA-pair (cta_group::2) version.
//
//   D[M,N] = epilogue( A[M,K] * W[N,K]^T )        bf16 operands, fp32 accumulation in TMEM, bf16 out
//
// Replaces every nn.Linear / 1x1 conv / 3x3 InflatedConv3d call of the reference hot path
// (base/models/attention.py:95-104,328,356 ; resnet.py:13-21,146,162,171-175 ; diffusers FeedForward).
//
// Why CTA pairs: the kernel is fed from L2, and its throughput follows the L2->SM bytes per flop of the tile shape
// (tools/bench_feedtheory.py).  A pair of SMs computes a 256 x BN tile with ONE tcgen05.mma.cta_group::2 stream: each
// CTA stages its own 128 rows of A and HALF of the W tile.  BN = 320 (two 160-wide MMAs per K step sharing the A
// stage) is the widest tile and the one the N = 320 / 640 layers use.
//
// Structure: persistent clusters of 2 CTAs (one pair per two SMs), 320 threads per CTA:
//   warp 0      : TMA producer   (A 128x64 slab + this CTA's W rows per stage, 128-byte swizzle, ring of STAGES;
//                                 both CTAs' loads complete on the LEADER CTA's full barrier)
//   warp 1      : MMA issuer     (leader CTA only: tcgen05.mma.cta_group::2 M=256, N<=256, K=16; commits are multicast
//                                 to both CTAs' barriers) + TMEM owner (both CTAs)
//   warps 2..9  : epilogue       (each CTA drains its own 128 accumulator rows: tcgen05.ld -> bias / time-bias /
//                                 GEGLU / TMA-prefetched residual -> bf16 staged in smem -> TMA store, or fp32
//                                 split-K partials)
// Two TMEM accumulator stages (one for BN = 320) let the epilogue of item i overlap the main loop of item i+1.
//
// Work item = (m_tile, n_tile, k_split).  Split-K (deterministic: fp32 partials + ordered reduction kernel) keeps the
// 74 pairs busy on the 5x8 / 10x16 levels where M is only 1280..5120 rows but K reaches 23040; a launch whose last
// wave would be nearly empty is issued as full waves over the leading tile rows plus a split-K "tail window"
// (make_plan).
//
// A-operand modes
//   plain : A is [M, K] row-major (row stride lda); optionally split along K over two sources
//           (the folded torch.cat([h, skip], dim=1) in front of a 1x1 shortcut, unet_blocks.py:538,630).
//   conv  : A is the channels-last feature map [NF, H, W, C]; K = 9*C ordered (kh, kw, c); every K block is one
//           (tap, 64-channel) slab of 128 consecutive OUTPUT pixels fetched by ONE im2col-mode TMA request (the
//           hardware walks the pixels, applies the stride and zero-fills the halo = the conv's zero padding).
//   frame : nn.Conv3d with a (k,1,1) kernel (vsr/models/resnet.py:253-254,269) on a map whose frame axis is padded
//           with k/2 zero frames on both sides: K = k*C ordered (tap, c), tap t of output row m is input row
//           m + t * (pixels per frame) -- the same 2-D TMA box, shifted by whole frames.
#include "common.cuh"

namespace {

constexpr int BLOCK_M = 128;          // rows per CTA; a pair covers 256
constexpr int PAIR_M = 256;
constexpr int BLOCK_K = 64;
constexpr int UMMA_K = 16;
constexpr int A_STAGE_BYTES = BLOCK_M * BLOCK_K * 2;   // 16 KiB
constexpr int NUM_EPI_WARPS = 8;                  // 2 per TMEM lane quarter (16 measured: no faster, GEGLU slower)
constexpr int EPI_SPLIT = NUM_EPI_WARPS / 4;      // warps sharing one 32-row slab take every EPI_SPLIT-th 32-column chunk
constexpr int NUM_THREADS = 64 + 32 * NUM_EPI_WARPS;   // 320
constexpr int EPI_BAR_ID = 1;
constexpr int EPI_CHUNK_BYTES = 32 * 32 * 2;      // one 32-row x 32-column bf16 chunk (TMA box, 64-byte swizzle)

struct GemmParams {
  int M, N, K;
  int num_k_blocks;
  int k_split_blocks;        // plain mode: K blocks [0, k_split) come from A0, the rest from A1
  int m_tiles, n_tiles;      // m_tiles counts 256-row pair tiles of THIS launch's window
  int m_tile0;               // first pair tile of the window (a GEMM may be issued as main window + split-K tail window)
  int rows_window;           // rows covered by the window (stride of the split-K partial planes)
  int splits, kb_per_split;  // split-K
  // conv3 mode
  int conv;                  // 0 plain GEMM, 1 implicit-GEMM 3x3 conv (im2col-mode TMA), 2 frame conv (k,1,1)
  int c_blocks;              // Cin / 64
  int out_h, out_w, conv_stride;   // im2col-mode conv (conv == 1): output geometry and stride
  int pad_before;            // conv == 1: zero rows / columns before the image (1: pad (1, 1); 0: Downsample2D's (0, 1))
  int tap_rows;              // frame conv (conv == 2): rows between consecutive taps = pixels per frame
  int phases;                // 4: nearest-2x upsample + 3x3 conv as four 2x2 "phase" convs on the LOW-resolution map
                             // (conv == 3; item = (m, n, phase); output pixel (2y + py, 2x + px)); else 1
  int lowres_w;              // conv == 3: W of the low-resolution map (5-D output box coordinates)
  int slabs_total;           // conv == 3: 32-row slabs per phase (stride of the phase segments of colstats)
  // epilogue
  const float* bias;         // [N] or null
  const float* row_bias;     // [M / rows_per_batch, ld_row_bias] or null  (time embedding add, resnet.py:187-190)
  int rows_per_batch;
  int ld_row_bias;
  const __nv_bfloat16* residual;   // [M, ldr] or null
  int ldr;
  int geglu;                 // 1: tile columns [0,BN/2) = value, [BN/2,BN) = gate -> out = value * gelu(gate)
  __nv_bfloat16* out;
  int ldo;
  float* partial;            // split-K workspace [splits, M, N] fp32 (splits > 1)
  int* tickets;              // in-kernel split-K reduction: one zeroed counter per (128-row block, n tile); the CTA whose
                             // partial arrives LAST sums all planes in split order and runs the fused epilogue (no
                             // reduction launch).  nullptr: the separate reduction kernel does it.
  float* colstats;           // [M / 32, N / 32, 4, 2] or null: per 32-row slab and 10-channel micro-group (stored per
                             // 32-column chunk and decade piece), (sum, sum of squares) of the bf16-rounded outputs: the
                             // GroupNorm statistics of the NEXT layer, emitted by the producer
  int mg8;                   // micro-group width of colstats: 0 = 10 channels (N % 10 == 0), 1 = 8 channels (otherwise)
  int check;                 // fp32-accumulate check mode: accumulators ALWAYS leave as fp32 partials (even with
                             // splits == 1); bias / residual / GEGLU run in fp32 on split-bf16 triples (check reduce)
  int k_rot;                 // K-sweep rotation stride per M tile (0 = off)
  int debug;                 // tuning only: 1 = skip TMA (pure MMA issue rate), 2 = skip MMA (pure TMA feed rate)
};

template <int BLOCK_N>
struct SmemLayout {
  // One tcgen05.mma covers at most N = 256.  A 320-wide tile is two 160-wide MMAs per K step that share the A stage:
  // the activation operand is fetched from L2 once per 320 output columns instead of once per 160, which is what
  // bounds the N = 320 / 640 layers (tools/bench_feedtheory.py: throughput follows L2->SM bytes per flop).
  static constexpr int N_MMA = BLOCK_N > 256 ? 2 : 1;
  static constexpr int UMMA_N = BLOCK_N / N_MMA;
  static constexpr int ACC_STAGES = 2 * BLOCK_N <= 512 ? 2 : 1;     // TMEM has 512 columns
  static constexpr int B_HALF_BYTES = (UMMA_N / 2) * BLOCK_K * 2;   // this CTA's rows of one MMA's B operand
  static constexpr int B_STAGE_BYTES = N_MMA * B_HALF_BYTES;
  static constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
  static constexpr int BIAS_BYTES = 0;
  static constexpr int EPI_CHUNKS = (BLOCK_N / 32 + EPI_SPLIT - 1) / EPI_SPLIT;   // 32-column chunks per epilogue warp
  static constexpr int EPI_BYTES = NUM_EPI_WARPS * EPI_CHUNKS * EPI_CHUNK_BYTES;  // per-warp bf16 staging chunks
  static constexpr int MAX_SMEM = 227 * 1024 - 2048 - BIAS_BYTES - EPI_BYTES;
  static constexpr int STAGES_RAW = MAX_SMEM / STAGE_BYTES;
  static constexpr int STAGES = STAGES_RAW > 8 ? 8 : STAGES_RAW;
  static constexpr int TOTAL = STAGES * STAGE_BYTES + BIAS_BYTES + EPI_BYTES + 1024 /*align*/ + 512 /*barriers*/;
};

// ---- cluster / cta_group::2 PTX ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t local_smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  // .relaxed: the only thing this arrive publishes is "my tcgen05.ld's have completed", which tcgen05.wait::ld +
  // tcgen05.fence::before_thread_sync already order.  The default .release.cluster compiles to MEMBAR.ALL.GPU +
  // CCTL.IVALL and cost 3000-4000 cycles per tile while TMA stores were in flight (tools/gemm_timeline.py).
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish2() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the barrier at this smem offset in BOTH CTAs of the pair once all prior MMAs of this thread retired
__device__ __forceinline__ void umma2_commit_mc(uint64_t* bar) {
  const uint16_t mask = 3;
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(smem_u32(bar)), "h"(mask)
      : "memory");
}
// TMA loads whose completion bytes are credited to a barrier given by its shared::cluster address (the leader's)
__device__ __forceinline__ void tma2_load_2d(void* dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0,
                                             int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
// im2col-mode TMA (conv halo handled by the hardware): coordinates = first output pixel of the tile in the bounding box
// (w = x - pad, h = y - pad, n), offsets = filter tap (s, r)
__device__ __forceinline__ void tma2_load_im2col(void* dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c,
                                                 int w, int h, int n, uint16_t off_w, uint16_t off_h) {
  asm volatile(
      "cp.async.bulk.tensor.4d.im2col.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4, %5, %6}], [%2], {%7, %8};" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c), "r"(w), "r"(h), "r"(n), "h"(off_w), "h"(off_h)
      : "memory");
}
__device__ __forceinline__ void epi_bar_sync() {
  asm volatile("bar.sync %0, %1;" ::"n"(EPI_BAR_ID), "n"(32 * NUM_EPI_WARPS) : "memory");
}

struct Item {
  int m_blk, n_blk, kb_begin, kb_end, phase;
};
__device__ __forceinline__ Item decode_item(const GemmParams& p, int item) {
  Item it;
  const int split = item % p.splits;
  int rest = item / p.splits;
  it.phase = 0;
  if (p.phases > 1) {                        // the four phases of one tile run back to back: they read the same pixels
    it.phase = rest % p.phases;
    rest /= p.phases;
  }
  it.n_blk = rest % p.n_tiles;
  it.m_blk = rest / p.n_tiles + p.m_tile0;
  it.kb_begin = split * p.kb_per_split;
  it.kb_end = min(p.num_k_blocks, it.kb_begin + p.kb_per_split);
  return it;
}

template <int BLOCK_N>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
gemm_bf16_tcgen05(const __grid_constant__ CUtensorMap tmap_a0, const __grid_constant__ CUtensorMap tmap_a1,
                  const __grid_constant__ CUtensorMap tmap_a2, const __grid_constant__ CUtensorMap tmap_a3,
                  const __grid_constant__ CUtensorMap tmap_b, const __grid_constant__ CUtensorMap tmap_out,
                  const __grid_constant__ CUtensorMap tmap_res, const GemmParams p) {
  pdl_launch_dependents();
  using L = SmemLayout<BLOCK_N>;
  constexpr int STAGES = L::STAGES;
  constexpr int ACC_STAGES = L::ACC_STAGES;
  constexpr int ACC_COLS = ACC_STAGES * BLOCK_N;
  constexpr uint32_t TMEM_COLS = (ACC_COLS <= 32) ? 32 : (ACC_COLS <= 64) ? 64 : (ACC_COLS <= 128) ? 128
                                 : (ACC_COLS <= 256) ? 256 : 512;
  static_assert(BLOCK_N % 32 == 0 && BLOCK_N >= 32 && ACC_COLS <= 512 && L::UMMA_N % 16 == 0 && L::UMMA_N <= 256,
                "BLOCK_N");

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* s_epi = smem + STAGES * L::STAGE_BYTES + L::BIAS_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * L::STAGE_BYTES + L::BIAS_BYTES + L::EPI_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;     // [2]
  uint64_t* tmem_empty = tmem_full + 2;         // [2]  (only the leader's are waited on)
  uint64_t* res_bar = tmem_empty + 2;           // [NUM_EPI_WARPS] residual-prefetch barriers
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_bar + NUM_EPI_WARPS);
  volatile uint32_t* s_last = tmem_slot + 1;          // in-kernel split-K: "this CTA finishes the tile" flag

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1;
  const int num_pairs = gridDim.x >> 1;
  const int num_items = p.m_tiles * p.n_tiles * p.splits * p.phases;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a0);
    tma_prefetch_desc(&tmap_a1);
    if (p.phases > 1) {
      tma_prefetch_desc(&tmap_a2);
      tma_prefetch_desc(&tmap_a3);
    }
    tma_prefetch_desc(&tmap_b);
    tma_prefetch_desc(&tmap_out);
    tma_prefetch_desc(&tmap_res);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], 2 * NUM_EPI_WARPS);   // one arrive per epilogue warp of BOTH CTAs
    }
    for (int w = 0; w < NUM_EPI_WARPS; ++w) mbar_init(&res_bar[w], 1);
    mbar_fence_init();
  }
  if (warp == 1) {
    tmem_alloc2(tmem_slot, TMEM_COLS);
    tmem_relinquish2();
  }
  tc_fence_before();
  cluster_sync_all();            // barriers of both CTAs initialised before any remote arrive / multicast commit
  tc_fence_after();
  pdl_wait();                    // everything above overlapped the previous kernel's tail; its data is visible from here
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================================== TMA producer (both CTAs) =====================================
    // The whole warp runs the loop (warp-uniform control flow keeps addresses / coordinates in uniform registers);
    // one elected lane issues.
    int stage = 0;
    uint32_t phase = 0;
    for (int item = pair; item < num_items; item += num_pairs) {
      const Item it = decode_item(p, item);
      const int m_cta = it.m_blk * 2 + static_cast<int>(rank);        // this CTA's 128-row block
      // K-sweep rotation: pairs working on different M tiles start at different K blocks, so the ~37 CTAs that share
      // a weight slab do not request the same L2 lines in lockstep (fp32 accumulation order changes per tile, but
      // the tile -> rotation mapping is fixed, so results stay bit-reproducible).
      const int klen = it.kb_end - it.kb_begin;
      const int rot = (it.m_blk * p.k_rot) % klen;
      for (int i = 0; i < klen; ++i) {
        int kb = it.kb_begin + i + rot;
        if (kb >= it.kb_end) kb -= klen;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        if (elect_one()) {
          uint8_t* a_dst = smem + stage * L::STAGE_BYTES;
          uint8_t* b_dst = a_dst + A_STAGE_BYTES;
          const uint32_t full_leader = mapa_u32(smem_u32(&full_bar[stage]), 0);
          if (p.debug & 1) {
            if (rank == 0) mbar_arrive(&full_bar[stage]);
          } else {
            if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * L::STAGE_BYTES);   // bytes landing in both CTAs
            if (p.conv == 3) {
              // nearest-2x upsample + 3x3 conv == four 2x2 convs on the low-resolution map, one per output-pixel parity
              // (py, px): taps (a, b) read source pixel (y + py - 1 + a, x + px - 1 + b); the tap weights were summed on
              // the host.  One im2col request per (tap, 64 channels) like the 3x3 mode; the bounding-box corners differ
              // per phase, hence one tensor map per phase.
              const int tap = kb / p.c_blocks;
              const int c0 = (kb - tap * p.c_blocks) * BLOCK_K;
              const int m0 = m_cta * BLOCK_M;
              const int img = m0 / (p.out_h * p.out_w);
              const int rem = m0 - img * (p.out_h * p.out_w);
              const int oy = rem / p.out_w, ox = rem - oy * p.out_w;
              const int px = it.phase & 1, py = it.phase >> 1;
              const CUtensorMap* am = it.phase == 0 ? &tmap_a0 : it.phase == 1 ? &tmap_a1 : it.phase == 2 ? &tmap_a2 : &tmap_a3;
              tma2_load_im2col(a_dst, am, full_leader, c0, ox + px - 1, oy + py - 1, img, static_cast<uint16_t>(tap & 1),
                               static_cast<uint16_t>(tap >> 1));
            } else if (p.conv == 2) {
              // (k,1,1) conv over frames on a frame-padded map: tap t of output row m is input row m + t * tap_rows
              const int tap = kb / p.c_blocks;
              tma2_load_2d(a_dst, &tmap_a0, full_leader, (kb - tap * p.c_blocks) * BLOCK_K,
                           m_cta * BLOCK_M + tap * p.tap_rows);
            } else if (p.conv) {
              // one request: 128 consecutive output pixels x 64 channels of filter tap (r, s)
              const int tap = kb / p.c_blocks;
              const int c0 = (kb - tap * p.c_blocks) * BLOCK_K;
              const int m0 = m_cta * BLOCK_M;
              const int img = m0 / (p.out_h * p.out_w);
              const int rem = m0 - img * (p.out_h * p.out_w);
              const int oy = rem / p.out_w, ox = rem - oy * p.out_w;
              tma2_load_im2col(a_dst, &tmap_a0, full_leader, c0, ox * p.conv_stride - p.pad_before,
                               oy * p.conv_stride - p.pad_before, img,
                               static_cast<uint16_t>(tap % 3), static_cast<uint16_t>(tap / 3));
            } else if (kb < p.k_split_blocks) {
              tma2_load_2d(a_dst, &tmap_a0, full_leader, kb * BLOCK_K, m_cta * BLOCK_M);
            } else {
              tma2_load_2d(a_dst, &tmap_a1, full_leader, (kb - p.k_split_blocks) * BLOCK_K, m_cta * BLOCK_M);
            }
#pragma unroll
            for (int h = 0; h < L::N_MMA; ++h)       // this CTA's half of each MMA's weight rows
              tma2_load_2d(b_dst + h * L::B_HALF_BYTES, &tmap_b, full_leader, kb * BLOCK_K,
                           it.phase * p.N + it.n_blk * BLOCK_N + h * L::UMMA_N + static_cast<int>(rank) * (L::UMMA_N / 2));
          }
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================================== MMA issuer (leader CTA only) =================================
    if (rank == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(PAIR_M, L::UMMA_N, 0, 0);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int item = pair; item < num_items; item += num_pairs) {
        const Item it = decode_item(p, item);
        const bool tl = (p.debug & 512) && blockIdx.x == 0 && lane == 0;    // debug timeline (tools/gemm_timeline.py)
        long long* tl_row = reinterpret_cast<long long*>(p.partial) + 8192 + ((item - pair) / num_pairs) * 8;
        if (tl) tl_row[0] = clock64();
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        if (tl) tl_row[1] = clock64();
        const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
        for (int kb = it.kb_begin; kb < it.kb_end; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          if (tl && kb == it.kb_begin) tl_row[2] = clock64();
          if (tl && kb == it.kb_end - 1) tl_row[3] = clock64();
          const uint32_t a_addr = smem_u32(smem + stage * L::STAGE_BYTES);
          const uint32_t b_addr = a_addr + A_STAGE_BYTES;
          const uint64_t a_desc = umma_desc_sw128(a_addr, 16, 1024);
          const uint64_t b_desc = umma_desc_sw128(b_addr, 16, 1024);
          if (elect_one()) {
            if (!(p.debug & 2)) {
#pragma unroll
              for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
                // advancing 16 bf16 = 32 bytes along K inside the 128-byte swizzle atom: +2 in the >>4 address field
#pragma unroll
                for (int h = 0; h < L::N_MMA; ++h)
                  umma2_bf16(d_tmem + h * L::UMMA_N, a_desc + 2 * k, b_desc + h * (L::B_HALF_BYTES >> 4) + 2 * k, idesc,
                             (kb > it.kb_begin || k > 0) ? 1u : 0u);
              }
            }
            umma2_commit_mc(&empty_bar[stage]);    // frees this smem stage in both CTAs once the MMAs retire
            if (kb == it.kb_end - 1) umma2_commit_mc(&tmem_full[acc]);   // accumulator complete -> both epilogues
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        if (tl) tl_row[4] = clock64();
        if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    // ===================================== epilogue (both CTAs) =========================================
    // tcgen05.ld hands every lane one accumulator ROW; writing rows straight to global memory would touch 32
    // different 128-byte lines per instruction.  Each warp instead stages its 32x32 bf16 chunks in shared memory
    // (64-byte-swizzled, conflict-free) and lets the TMA move them: the residual tile is PREFETCHED into the same
    // buffers with TMA loads while the MMAs of the tile are still running, the sum is written back in place and
    // leaves with a TMA store (which also clips the M / N tails).
    const int ew = warp - 2;                       // 0..NUM_EPI_WARPS-1
    const int q = warp & 3;                        // TMEM lane quarter this warp may access
    const int chalf = ew >> 2;                     // which share of the 32-column chunks this warp drains
    const uint32_t tmem_empty_leader = mapa_u32(smem_u32(&tmem_empty[0]), 0);
    uint8_t* my_stage = s_epi + ew * (L::EPI_CHUNKS * EPI_CHUNK_BYTES);
    uint64_t* my_res_bar = &res_bar[ew];
    uint32_t res_phase = 0;
    const int swz = (lane >> 1) & 3;               // 64-byte swizzle: 16-byte unit j of row r lives at unit j ^ ((r>>1)&3)
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int item = pair; item < num_items; item += num_pairs) {
      const Item it = decode_item(p, item);
      const int split = item % p.splits;
      const int row0 = (it.m_blk * 2 + static_cast<int>(rank)) * BLOCK_M;
      const int wrow0 = row0 + q * 32;             // first row of this warp's 32-row slab
      const int row = wrow0 + lane;
      const bool row_ok = row < p.M;
      const int n0 = it.n_blk * BLOCK_N;
      const bool staged = p.splits == 1 && !p.check;
      const bool fixup = p.splits > 1 && !p.check && p.tickets != nullptr;     // in-kernel split-K reduction
      const bool has_res = staged && p.residual != nullptr;
      const bool tl = (p.debug & 512) && blockIdx.x == 0 && ew == 0 && lane == 0;
      long long* tl_row = reinterpret_cast<long long*>(p.partial) + ((item - pair) / num_pairs) * 8;
      if (tl) tl_row[0] = clock64();
      if (staged || fixup) {
        // buffers are free once the previous tile's stores have finished READING them
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        __syncwarp();
      }
      if (staged) {
        if (has_res && lane == 0 && !(p.debug & 64)) {
          int nch = 0;
          for (int c = chalf; c < BLOCK_N / 32; c += EPI_SPLIT) ++nch;
          mbar_expect_tx(my_res_bar, nch * EPI_CHUNK_BYTES);
          int k = 0;
          for (int c = chalf; c < BLOCK_N / 32; c += EPI_SPLIT, ++k)
            tma_load_2d(my_stage + k * EPI_CHUNK_BYTES, &tmap_res, my_res_bar, n0 + c * 32, wrow0);
        }
      }

      if (tl) tl_row[1] = clock64();
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      if (tl) tl_row[2] = clock64();
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BLOCK_N;
      if (has_res && !(p.debug & 64)) {
        mbar_wait(my_res_bar, res_phase);
        res_phase ^= 1;
      }
      const float* rb_row = (p.row_bias && row_ok) ? p.row_bias + static_cast<size_t>(row / p.rows_per_batch) * p.ld_row_bias
                                                    : nullptr;

      // packs f[32] (+ residual already in the buffer) into the warp's chunk buffer k and hands it to the TMA
      auto stage_and_store = [&](float (&f)[32], int k, int col_out0, bool add_res) {
        uint8_t* buf = my_stage + k * EPI_CHUNK_BYTES + lane * 64;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint4* slot = reinterpret_cast<uint4*>(buf + ((j ^ swz) << 4));
          if (add_res) {
            const uint4 r = *slot;
            const float2 r0 = unpack_bf16(r.x), r1 = unpack_bf16(r.y), r2 = unpack_bf16(r.z), r3 = unpack_bf16(r.w);
            f[8 * j] += r0.x; f[8 * j + 1] += r0.y; f[8 * j + 2] += r1.x; f[8 * j + 3] += r1.y;
            f[8 * j + 4] += r2.x; f[8 * j + 5] += r2.y; f[8 * j + 6] += r3.x; f[8 * j + 7] += r3.y;
          }
          uint4 o;
          o.x = pack_bf16(f[8 * j], f[8 * j + 1]);
          o.y = pack_bf16(f[8 * j + 2], f[8 * j + 3]);
          o.z = pack_bf16(f[8 * j + 4], f[8 * j + 5]);
          o.w = pack_bf16(f[8 * j + 6], f[8 * j + 7]);
          *slot = o;
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0 && !(p.debug & 16)) {
          if (p.phases > 1) {
            // output pixel (2y + py, 2x + px) of the high-resolution map: 5-D box (c, px, x, py, n*H + y)
            const int ny0 = wrow0 / p.lowres_w, x0 = wrow0 - ny0 * p.lowres_w;
            asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];" ::"l"(
                             reinterpret_cast<uint64_t>(&tmap_out)),
                         "r"(smem_u32(my_stage + k * EPI_CHUNK_BYTES)), "r"(col_out0), "r"(it.phase & 1), "r"(x0),
                         "r"(it.phase >> 1), "r"(ny0)
                         : "memory");
          } else {
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                             reinterpret_cast<uint64_t>(&tmap_out)),
                         "r"(smem_u32(my_stage + k * EPI_CHUNK_BYTES)), "r"(col_out0), "r"(wrow0)
                         : "memory");
          }
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
      };

      // GroupNorm statistics of the consumer from the staged bf16 chunks.  Runs AFTER the accumulator has been handed back
      // to the MMA warp (it only needs the staging buffers, which stay valid until this warp's next tile), so it overlaps
      // the next tile's main loop even for the single-accumulator 320-wide tiles.
      auto chunk_stats = [&](int k, int col_out0) {
        if (col_out0 < p.N && wrow0 < p.M) {
          // GroupNorm statistics of the consumer, from the staged bf16 chunk (exactly the values that reach memory).
          // lane = (row parity, column pair): 16 conflict-free LDS.32 walk the 32 rows and one shuffle folds the parities;
          // a segmented scan over the 16 column pairs then folds them into 10-channel MICRO-GROUPS (every GroupNorm of
          // the model has C / 32 = a multiple of 10 channels per group, so any consumer -- also a later concat with
          // another group size -- can assemble its groups from them).  A 32-column chunk overlaps at most 4 decades:
          // colstats[slab][chunk][piece 0..3] = (sum, sumsq), piece = decade - first decade of the chunk.  Rows >= M skip.
          const int par = lane >> 4, c2 = lane & 15;
          const uint8_t* chunk = my_stage + k * EPI_CHUNK_BYTES;
          float s0 = 0.f, q0 = 0.f;
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const int r = 2 * i + par;
            const uint32_t w = *reinterpret_cast<const uint32_t*>(chunk + r * 64 + (((c2 >> 2) ^ ((r >> 1) & 3)) << 4) +
                                                                   (c2 & 3) * 4);
            float2 v2 = unpack_bf16(w);
            if (wrow0 + r >= p.M) v2 = make_float2(0.f, 0.f);
            s0 += v2.x + v2.y;
            q0 = fmaf(v2.x, v2.x, fmaf(v2.y, v2.y, q0));
          }
          s0 += __shfl_xor_sync(0xffffffffu, s0, 16);
          q0 += __shfl_xor_sync(0xffffffffu, q0, 16);
          const int col = col_out0 + 2 * c2;                         // even; a pair never straddles a decade
          // micro-group index: col / 10 (col < 16384), or col / 8 for models whose groups are multiples of 8 only (VSR)
          const int dec = p.mg8 ? (col >> 3) : ((col * 6554) >> 16);
          const int dec0 = p.mg8 ? (col_out0 >> 3) : ((col_out0 * 6554) >> 16);
          // segmented inclusive scan over lanes 0..15 of each half (segments = equal decade, contiguous lanes)
#pragma unroll
          for (int o = 1; o < 16; o <<= 1) {
            const float ts = __shfl_up_sync(0xffffffffu, s0, o);
            const float tq = __shfl_up_sync(0xffffffffu, q0, o);
            const int td = __shfl_up_sync(0xffffffffu, dec, o);
            if (c2 >= o && td == dec) {
              s0 += ts;
              q0 += tq;
            }
          }
          const int dec_next = __shfl_down_sync(0xffffffffu, dec, 1);
          const bool last_of_piece = (c2 == 15) || (dec_next != dec) || (col + 2 >= p.N);
          if (par == 0 && last_of_piece && col < p.N)
            *reinterpret_cast<float2*>(p.colstats + ((static_cast<size_t>(it.phase * p.slabs_total + (wrow0 >> 5)) * (p.N >> 5) +
                                                      (col_out0 >> 5)) * 4 + (dec - dec0)) * 2) = make_float2(s0, q0);
        }
      };

      if (p.splits > 1 || p.check) {
        // fp32 partials for the ordered split-K reduction
        float* dst_row = p.partial + (static_cast<size_t>(split) * p.rows_window + (row - p.m_tile0 * PAIR_M)) * p.N;
#pragma unroll 1
        for (int c = chalf; c < BLOCK_N / 32; c += EPI_SPLIT) {
          uint32_t v[32];
          tmem_ld_32x32(t_row + c * 32, v);
          tmem_wait_ld();
          const int col0 = n0 + c * 32;
          if (row_ok) {
#pragma unroll
            for (int j = 0; j < 32; j += 4)
              if (col0 + j < p.N)
                *reinterpret_cast<uint4*>(dst_row + col0 + j) = make_uint4(v[j], v[j + 1], v[j + 2], v[j + 3]);
          }
        }
      } else if (!p.geglu) {
        int k = 0;
#pragma unroll 1
        for (int c = chalf; c < BLOCK_N / 32; c += EPI_SPLIT, ++k) {
          uint32_t v[32];
          tmem_ld_32x32(t_row + c * 32, v);
          tmem_wait_ld();
          if (tl && k == 0) tl_row[3] = clock64();
          const int col0 = n0 + c * 32;
          float f[32];
#pragma unroll
          for (int e = 0; e < 32; ++e) f[e] = __uint_as_float(v[e]);
          if (col0 + 32 <= p.N) {
            if (p.bias) {                          // warp-uniform addresses: broadcast loads
#pragma unroll
              for (int e = 0; e < 32; e += 4) {
                const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + e));
                f[e] += b4.x; f[e + 1] += b4.y; f[e + 2] += b4.z; f[e + 3] += b4.w;
              }
            }
            if (rb_row) {
#pragma unroll
              for (int e = 0; e < 32; e += 4) {
                const float4 b4 = __ldg(reinterpret_cast<const float4*>(rb_row + col0 + e));
                f[e] += b4.x; f[e + 1] += b4.y; f[e + 2] += b4.z; f[e + 3] += b4.w;
              }
            }
          } else if (col0 < p.N) {
            // the last chunk of an N % 32 != 0 output: its columns past N are clipped by the TMA store, and their bias
            // loads must not read past the caller's [N] rows (N % 8 == 0: whole float4s).  A separate branch so that
            // the full chunks keep their unpredicated loads (the guard in every chunk measured ~2% slower per step)
#pragma unroll
            for (int e = 0; e < 32; e += 4) {
              if (col0 + e < p.N) {
                if (p.bias) {
                  const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + e));
                  f[e] += b4.x; f[e + 1] += b4.y; f[e + 2] += b4.z; f[e + 3] += b4.w;
                }
                if (rb_row) {
                  const float4 b4 = __ldg(reinterpret_cast<const float4*>(rb_row + col0 + e));
                  f[e] += b4.x; f[e + 1] += b4.y; f[e + 2] += b4.z; f[e + 3] += b4.w;
                }
              }
            }
          }
          stage_and_store(f, k, col0, has_res && !(p.debug & 64));
        }
      } else {
        // GEGLU: value columns [0, BN/2), gate columns [BN/2, BN) of the same tile (weights interleaved on the
        // host); out[:, n_blk*BN/2 + j] = (value + b) * gelu_erf(gate + b')   (diffusers GEGLU, mirror at
        // vsr/models/diffusers_attention.py:811-822)
        constexpr int HALF = BLOCK_N / 2;
        int k = 0;
#pragma unroll 1
        for (int c = chalf; c < HALF / 32; c += EPI_SPLIT, ++k) {
          uint32_t v[32], g[32];
          tmem_ld_32x32(t_row + c * 32, v);
          tmem_ld_32x32(t_row + HALF + c * 32, g);
          tmem_wait_ld();
          float f[32];
#pragma unroll
          for (int e = 0; e < 32; e += 4) {
            float4 bv = make_float4(0.f, 0.f, 0.f, 0.f), bg = bv;
            if (p.bias) {                                   // warp-uniform addresses: one broadcast transaction each
              bv = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + c * 32 + e));
              bg = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + HALF + c * 32 + e));
            }
            f[e] = (__uint_as_float(v[e]) + bv.x) * gelu_fast_f(__uint_as_float(g[e]) + bg.x);
            f[e + 1] = (__uint_as_float(v[e + 1]) + bv.y) * gelu_fast_f(__uint_as_float(g[e + 1]) + bg.y);
            f[e + 2] = (__uint_as_float(v[e + 2]) + bv.z) * gelu_fast_f(__uint_as_float(g[e + 2]) + bg.z);
            f[e + 3] = (__uint_as_float(v[e + 3]) + bv.w) * gelu_fast_f(__uint_as_float(g[e + 3]) + bg.w);
          }
          stage_and_store(f, k, it.n_blk * HALF + c * 32, false);
        }
      }
      if (tl) tl_row[4] = clock64();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tmem_empty_leader + acc * 8);
      bool finished_here = staged;
      if (fixup) {
        // In-kernel split-K reduction.  Every epilogue thread has stored its share of this CTA's partial block; publish
        // it (fence), count this CTA's arrival on the block's ticket, and let the LAST arrival finish the block: it sums
        // the planes in split order 0..S-1 (so the result does not depend on who is last), then runs the same epilogue
        // as an unsplit tile.  The ticket is left at zero for the next launch.
        // (one device-scope fence by the ticket thread, cumulative over the CTA barrier -- the grid-sync pattern; a fence
        // in every thread cost tens of microseconds with the strided partial stores in flight)
        epi_bar_sync();
        if (ew == 0 && lane == 0) {
          __threadfence();
          int* tk = p.tickets + (it.m_blk * 2 + static_cast<int>(rank)) * p.n_tiles + it.n_blk;
          const int last = atomicAdd(tk, 1) == p.splits - 1;
          if (last) {
            *tk = 0;
            __threadfence();
          }
          *s_last = static_cast<uint32_t>(last);
        }
        epi_bar_sync();
        if (*s_last) {
          finished_here = true;
          // Coalesced sweep: for this part of the epilogue a lane owns a COLUMN, so every load instruction reads 128
          // consecutive bytes of one partial row; the bf16 results go straight into the (swizzled) staging chunk the TMA
          // store and the statistics read.  Same summation order as the reduction kernel: planes 0..S-1, bias, time bias,
          // residual.
          const size_t plane = static_cast<size_t>(p.rows_window) * p.N;
          int k = 0;
#pragma unroll 1
          for (int c = chalf; c < BLOCK_N / 32; c += EPI_SPLIT, ++k) {
            const int col0 = n0 + c * 32;
            const int col = col0 + lane;
            const bool col_ok = col < p.N;
            uint8_t* chunk = my_stage + k * EPI_CHUNK_BYTES;
            const float bias_c = (p.bias && col_ok) ? __ldg(p.bias + col) : 0.f;
            // 32 independent loads in flight per lane and plane (one per row of the slab)
            float a[32];
#pragma unroll
            for (int r = 0; r < 32; ++r) a[r] = 0.f;
            const int rows_here = min(32, p.M - wrow0);                 // <= 0: slab entirely beyond M
            const float* src0 = p.partial + static_cast<size_t>(wrow0 - p.m_tile0 * PAIR_M) * p.N + col;
            if (col_ok) {
              for (int sp = 0; sp < p.splits; ++sp) {
                const float* src = src0 + sp * plane;
#pragma unroll
                for (int r = 0; r < 32; ++r)
                  if (r < rows_here) a[r] += __ldcg(src + static_cast<size_t>(r) * p.N);
              }
            }
#pragma unroll
            for (int r = 0; r < 32; ++r) {
              const int grow = wrow0 + r;
              float v = a[r];
              if (r < rows_here && col_ok) {
                v += bias_c;
                if (p.row_bias) v += __ldg(p.row_bias + static_cast<size_t>(grow / p.rows_per_batch) * p.ld_row_bias + col);
                if (p.residual) v += __bfloat162float(p.residual[static_cast<size_t>(grow) * p.ldr + col]);
              } else {
                v = 0.f;
              }
              *reinterpret_cast<__nv_bfloat16*>(chunk + r * 64 + ((((lane >> 3) ^ ((r >> 1) & 3)) << 4) + (lane & 7) * 2)) =
                  __float2bfloat16_rn(v);
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                               reinterpret_cast<uint64_t>(&tmap_out)),
                           "r"(smem_u32(chunk)), "r"(col0), "r"(wrow0)
                           : "memory");
              asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
          }
        }
      }
      if (p.colstats != nullptr && finished_here && !p.check && !p.geglu) {
        int k = 0;
        for (int c = chalf; c < BLOCK_N / 32; c += EPI_SPLIT, ++k) chunk_stats(k, n0 + c * 32);
      }
      if (tl) tl_row[5] = clock64();
      if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1; }
    }
  }

  if (warp >= 2 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // output stores complete
  tc_fence_before();
  cluster_sync_all();            // the peer may still be reading smem / TMEM that a cta_group::2 MMA touches
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc2(tmem_base, TMEM_COLS);
  }
}

// Ordered split-K reduction + the same fused epilogue (bias / time-bias / residual) -> bf16
__global__ void __launch_bounds__(256)
splitk_reduce_kernel(const float* __restrict__ partial, int splits, int M, int N, const float* __restrict__ bias,
                     const float* __restrict__ row_bias, int rows_per_batch, int ld_row_bias,
                     const __nv_bfloat16* __restrict__ residual, int ldr, __nv_bfloat16* __restrict__ out, int ldo,
                     int row0) {
  // M rows of a window that starts at absolute row row0; partial / residual / out already point at the window
  pdl_prologue();
  const int nvec = N >> 2;
  const long long total = static_cast<long long>(M) * nvec;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int row = static_cast<int>(i / nvec);
    const int col = static_cast<int>(i % nvec) * 4;
    float4 a = *reinterpret_cast<const float4*>(partial + static_cast<size_t>(row) * N + col);
    for (int s = 1; s < splits; ++s) {
      const float4 b = *reinterpret_cast<const float4*>(partial + (static_cast<size_t>(s) * M + row) * N + col);
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    if (bias) {
      const float4 b = *reinterpret_cast<const float4*>(bias + col);
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    if (row_bias) {
      const float4 b = *reinterpret_cast<const float4*>(row_bias + static_cast<size_t>((row + row0) / rows_per_batch) * ld_row_bias + col);
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    if (residual) {
      const uint2 r = *reinterpret_cast<const uint2*>(residual + static_cast<size_t>(row) * ldr + col);
      const float2 r0 = unpack_bf16(r.x), r1 = unpack_bf16(r.y);
      a.x += r0.x; a.y += r0.y; a.z += r1.x; a.w += r1.y;
    }
    *reinterpret_cast<uint2*>(out + static_cast<size_t>(row) * ldo + col) = make_uint2(pack_bf16(a.x, a.y), pack_bf16(a.z, a.w));
  }
}

// Split-K reduction that also emits the consumer's GroupNorm micro-group statistics (same layout as the epilogue's):
// block = one 32-row slab x 128 columns; thread = (4 columns, 4 rows) with all its loads independent.
__global__ void __launch_bounds__(256)
splitk_reduce_stats_kernel(const float* __restrict__ partial, int splits, int M, int N, int M_total,
                           const float* __restrict__ bias, const float* __restrict__ row_bias, int rows_per_batch,
                           int ld_row_bias, const __nv_bfloat16* __restrict__ residual, int ldr,
                           __nv_bfloat16* __restrict__ out, int ldo, int row0, float* __restrict__ colstats, int mg) {
  pdl_prologue();
  constexpr int R = 4;                                 // rows per thread
  __shared__ float s_cs[8][128][2];                    // [row group][column][sum, sumsq]
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int cbase = blockIdx.y * 128;
  const int col = cbase + tx * 4;
  const int r_begin = blockIdx.x * 32 + ty * R;        // window-relative; row0 is a multiple of 256
  float s[4] = {0.f, 0.f, 0.f, 0.f}, q[4] = {0.f, 0.f, 0.f, 0.f};
  if (col < N) {
    float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (bias) b4 = *reinterpret_cast<const float4*>(bias + col);
    float4 acc[R];
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const int row = r_begin + i;
      acc[i] = row < M ? *reinterpret_cast<const float4*>(partial + static_cast<size_t>(row) * N + col) : b4;
    }
    for (int sp = 1; sp < splits; ++sp) {
#pragma unroll
      for (int i = 0; i < R; ++i) {
        const int row = r_begin + i;
        if (row < M) {
          const float4 b = *reinterpret_cast<const float4*>(partial + (static_cast<size_t>(sp) * M + row) * N + col);
          acc[i].x += b.x; acc[i].y += b.y; acc[i].z += b.z; acc[i].w += b.w;
        }
      }
    }
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const int row = r_begin + i;
      if (row >= M) continue;
      float4 a = acc[i];
      a.x += b4.x; a.y += b4.y; a.z += b4.z; a.w += b4.w;
      if (row_bias) {
        const float4 b = *reinterpret_cast<const float4*>(row_bias + static_cast<size_t>((row + row0) / rows_per_batch) * ld_row_bias + col);
        a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
      }
      if (residual) {
        const uint2 r = *reinterpret_cast<const uint2*>(residual + static_cast<size_t>(row) * ldr + col);
        const float2 r0 = unpack_bf16(r.x), r1 = unpack_bf16(r.y);
        a.x += r0.x; a.y += r0.y; a.z += r1.x; a.w += r1.y;
      }
      const uint2 o = make_uint2(pack_bf16(a.x, a.y), pack_bf16(a.z, a.w));
      *reinterpret_cast<uint2*>(out + static_cast<size_t>(row) * ldo + col) = o;
      if (row + row0 < M_total) {
        const float2 v0 = unpack_bf16(o.x), v1 = unpack_bf16(o.y);
        s[0] += v0.x; q[0] = fmaf(v0.x, v0.x, q[0]);
        s[1] += v0.y; q[1] = fmaf(v0.y, v0.y, q[1]);
        s[2] += v1.x; q[2] = fmaf(v1.x, v1.x, q[2]);
        s[3] += v1.y; q[3] = fmaf(v1.y, v1.y, q[3]);
      }
    }
  }
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    s_cs[ty][tx * 4 + e][0] = s[e];
    s_cs[ty][tx * 4 + e][1] = q[e];
  }
  __syncthreads();
  // 4 chunks x 4 pieces: thread t < 16 folds the columns of one (chunk, decade) piece, row groups in a fixed order
  if (threadIdx.x < 16) {
    const int cl = threadIdx.x >> 2, piece = threadIdx.x & 3;
    const int c0 = cbase + cl * 32;
    if (c0 < N) {
      const int dec = c0 / mg + piece;
      const int lo = max(c0, dec * mg), hi = min(min(c0 + 32, dec * mg + mg), N);
      if (lo < hi) {
        float a = 0.f, b = 0.f;
        for (int c = lo; c < hi; ++c)
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            a += s_cs[g][c - cbase][0];
            b += s_cs[g][c - cbase][1];
          }
        const size_t slab = static_cast<size_t>((blockIdx.x * 32 + row0) >> 5);
        *reinterpret_cast<float2*>(colstats + ((slab * (N >> 5) + (c0 >> 5)) * 4 + piece) * 2) = make_float2(a, b);
      }
    }
  }
}

// Check-mode epilogue: ordered sum of the fp32 partials, then bias / time bias / residual / GEGLU in fp32 (exact erf
// GELU) on split-bf16 triples: residual row = [hi | lo | hi] of width N each, output row = [hi | lo | hi] of width n_out.
__global__ void __launch_bounds__(256)
splitk_reduce_check_kernel(const float* __restrict__ partial, int splits, int M, int N, const float* __restrict__ bias,
                           const float* __restrict__ row_bias, int rows_per_batch, int ld_row_bias,
                           const __nv_bfloat16* __restrict__ residual, int ldr, int geglu,
                           __nv_bfloat16* __restrict__ out, int ldo, int row0) {
  pdl_prologue();
  const int n_out = geglu ? N / 2 : N;
  const long long total = static_cast<long long>(M) * n_out;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int row = static_cast<int>(i / n_out);
    const int col = static_cast<int>(i - static_cast<long long>(row) * n_out);
    auto acc_at = [&](int c) {
      float a = partial[static_cast<size_t>(row) * N + c];
      for (int s = 1; s < splits; ++s) a += partial[(static_cast<size_t>(s) * M + row) * N + c];
      if (bias) a += bias[c];
      return a;
    };
    float v;
    if (geglu) {                                   // 256-column tiles: 128 value columns, then their 128 gate columns
      const int t = col >> 7, j = col & 127;
      const float val = acc_at(t * 256 + j), gate = acc_at(t * 256 + 128 + j);
      v = val * (0.5f * gate * (1.0f + erff(gate * 0.70710678118654752440f)));
    } else {
      v = acc_at(col);
      if (row_bias) v += row_bias[static_cast<size_t>((row + row0) / rows_per_batch) * ld_row_bias + col];
      if (residual) {
        const __nv_bfloat16* r = residual + static_cast<size_t>(row) * ldr + col;
        v += __bfloat162float(r[0]) + __bfloat162float(r[N]);
      }
    }
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    const __nv_bfloat16 lo = __float2bfloat16_rn(v - __bfloat162float(hi));
    __nv_bfloat16* o = out + static_cast<size_t>(row) * ldo + col;
    o[0] = hi;
    o[n_out] = lo;
    o[2 * n_out] = hi;
  }
}

template <int BLOCK_N>
int launch_gemm(const CUtensorMap& a0, const CUtensorMap& a1, const CUtensorMap& a2, const CUtensorMap& a3,
                const CUtensorMap& b, const CUtensorMap& mo, const CUtensorMap& mr, const GemmParams& p,
                int num_sms, cudaStream_t stream) {
  using L = SmemLayout<BLOCK_N>;
  static LavieSmemConfig configured;
  int rc = lavie_config_smem(gemm_bf16_tcgen05<BLOCK_N>, L::TOTAL, &configured, "gemm_bf16_tcgen05");
  if (rc) return rc;
  const int items = p.m_tiles * p.n_tiles * p.splits * p.phases;
  int pairs = num_sms / 2;
  if (items < pairs) pairs = items;
  launch_pdl(gemm_bf16_tcgen05<BLOCK_N>, 2 * pairs, NUM_THREADS, L::TOTAL, stream, a0, a1, a2, a3, b, mo, mr, p);
  rc = lavie_check_launch("gemm_bf16_tcgen05");
  if (rc) return rc;
  if (p.check) {
    const int row0 = p.m_tile0 * PAIR_M;
    const long long total = static_cast<long long>(p.rows_window) * (p.geglu ? p.N / 2 : p.N);
    long long blocks = (total + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    launch_pdl(splitk_reduce_check_kernel, static_cast<int>(blocks), 256, 0, stream, p.partial, p.splits, p.rows_window,
               p.N, p.bias, p.row_bias, p.rows_per_batch, p.ld_row_bias,
               p.residual ? p.residual + static_cast<size_t>(row0) * p.ldr : nullptr, p.ldr, p.geglu,
               p.out + static_cast<size_t>(row0) * p.ldo, p.ldo, row0);
    rc = lavie_check_launch("splitk_reduce_check_kernel");
  } else if (p.splits > 1 && p.tickets != nullptr) {
    // the last-arriving CTA of every block already reduced and stored it (and emitted the statistics)
  } else if (p.splits > 1 && p.colstats != nullptr) {
    const int row0 = p.m_tile0 * PAIR_M;
    dim3 grid((p.rows_window + 31) / 32, (p.N + 127) / 128);
    launch_pdl(splitk_reduce_stats_kernel, grid, 256, 0, stream, p.partial, p.splits, p.rows_window, p.N, p.M, p.bias,
               p.row_bias, p.rows_per_batch, p.ld_row_bias,
               p.residual ? p.residual + static_cast<size_t>(row0) * p.ldr : nullptr, p.ldr,
               p.out + static_cast<size_t>(row0) * p.ldo, p.ldo, row0, p.colstats, p.mg8 ? 8 : 10);
    rc = lavie_check_launch("splitk_reduce_stats_kernel");
  } else if (p.splits > 1) {
    const int row0 = p.m_tile0 * PAIR_M;
    const long long total = static_cast<long long>(p.rows_window) * (p.N >> 2);
    long long blocks = (total + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    launch_pdl(splitk_reduce_kernel, static_cast<int>(blocks), 256, 0, stream, p.partial, p.splits, p.rows_window, p.N,
               p.bias, p.row_bias, p.rows_per_batch, p.ld_row_bias,
               p.residual ? p.residual + static_cast<size_t>(row0) * p.ldr : nullptr, p.ldr,
               p.out + static_cast<size_t>(row0) * p.ldo, p.ldo, row0);
    rc = lavie_check_launch("splitk_reduce_kernel");
  }
  return rc;
}

int g_force_splits = 0;
int g_debug = 0;
int g_k_rot = 0;   // measured: no effect on B200 (profiles/r1_notes.md), kept as a tuning hook only
int g_no_tail = 0; // lavie_debug_set(5, 1): never split a GEMM into main + tail launches (A/B timing)
int g_inkernel_reduce = 0;   // lavie_debug_set(7, 1): the last-arriving CTA of a block sums the split-K planes in the kernel
                             // instead of the separate reduction kernel.  Correct (same output bits; the column statistics
                             // are summed in the epilogue's order, so they differ in the last fp32 bits), but measured
                             // SLOWER on the full step (profiles/r2_ab_inkernel_splitk.txt): off by default, kept for A/B.
constexpr size_t TICKET_BYTES = 64 * 1024;   // tail of the caller's workspace: zero before first use, left zero
int num_sms() { return lavie_num_sms(); }

// Tile-shape / split-K choice: minimise  waves x (K blocks per item x per-block time + per-item overhead), where the
// per-block time is the larger of the MMA time (2*BN cycles per SM) and the L2 feed time of the stage bytes.
struct Plan {
  int bn;
  int splits, kb_per_split;            // main window: pair tiles [0, m_tiles - tail_tiles)
  int tail_tiles;                      // > 0: the last tail_tiles pair-tile rows run as a second, split-K launch
  int tail_splits, tail_kb_per_split;
};

// modelled cycles of one launch over `m_tiles` pair-tile rows with `s` K splits (s must divide evenly into k blocks)
double window_cost(int m_tiles, int n_tiles, int bn, int s, int kbps, double t_kb, double t_epi, int pairs, int N) {
  const long items = static_cast<long>(m_tiles) * n_tiles * s;
  const long waves = (items + pairs - 1) / pairs;
  double cost = static_cast<double>(waves) * (kbps * t_kb + 1500.0 + 6.0 * bn + t_epi);
  if (s > 1) cost += 4000.0 + 0.0013 * (s + 0.5) * static_cast<double>(m_tiles) * PAIR_M * N;   // reduction pass (HBM)
  return cost;
}

// best split-K factor for a window; returns cost, writes s / kbps
double best_split(int m_tiles, int n_tiles, int bn, int num_k_blocks, int max_splits, double t_kb, double t_epi,
                  int pairs, int N, size_t ws_bytes, int forced, int* s_out, int* kbps_out) {
  double best = 1e30;
  const long tiles = static_cast<long>(m_tiles) * n_tiles;
  for (int s = 1; s <= max_splits; ++s) {
    if (s > 1) {
      if (static_cast<size_t>(s) * m_tiles * PAIR_M * N * 4 > ws_bytes) break;
      if (num_k_blocks / s < 8) break;
      if (tiles * (s - 1) >= pairs) break;           // no point splitting once the machine is full
    }
    if (forced && s != forced) continue;
    const int kbps = (num_k_blocks + s - 1) / s;
    if ((num_k_blocks + kbps - 1) / kbps != s) continue;
    const double c = window_cost(m_tiles, n_tiles, bn, s, kbps, t_kb, t_epi, pairs, N);
    if (c < best) {
      best = c;
      *s_out = s;
      *kbps_out = kbps;
    }
  }
  return best;
}

// Tile shape / split-K / tail choice.  Per K block a CTA pays the larger of the MMA time (2*bn cycles) and the L2
// feed time of its stage bytes.  A launch whose last wave is mostly empty can instead run as two launches: full waves
// over the leading tile rows, then the remaining rows split along K so that they fill the machine once more.
Plan make_plan(int M, int N, int num_k_blocks, int forced_bn, bool geglu, bool conv, size_t ws_bytes,
               bool no_split = false) {
  const int pairs = num_sms() / 2;
  const int m_tiles = (M + PAIR_M - 1) / PAIR_M;
  const int cands[6] = {320, 256, 192, 160, 128, 64};
  Plan best{128, 1, num_k_blocks, 0, 1, num_k_blocks};
  double best_cost = 1e30;
  const int max_splits = (geglu || no_split) ? 1 : 16;
  const int forced_s = (geglu || no_split) ? 0 : g_force_splits;
  for (int i = 0; i < 6; ++i) {
    const int bn = cands[i];
    if (forced_bn && bn != forced_bn) continue;
    if (geglu && bn != 256) continue;
    const int n_tiles = (N + bn - 1) / bn;
    // measured L2->SM feed per SM and clock with all SMs pulling (tools/bench_feedtheory.py): ~47 B dense, ~38 B through
    // the im2col-mode TMA; a 64-deep K block needs 16 KiB of A plus 64*bn bytes of B per CTA
    const double t_kb = fmax(2.0 * bn, (16384.0 + 64.0 * bn) / (conv ? 38.0 : 47.0));
    const double t_epi = bn > 256 ? 5000.0 : 0.0;      // single accumulator stage: the epilogue is not overlapped
    int s = 1, kbps = num_k_blocks;
    const double c1 = best_split(m_tiles, n_tiles, bn, num_k_blocks, max_splits, t_kb, t_epi, pairs, N, ws_bytes,
                                 forced_s, &s, &kbps);
    if (c1 < best_cost) {
      best_cost = c1;
      best = Plan{bn, s, kbps, 0, 1, num_k_blocks};
    }
    // main window (no split) + split-K tail; only when the single launch needs more than one wave
    const long tiles = static_cast<long>(m_tiles) * n_tiles;
    if (geglu || no_split || forced_s || g_no_tail || tiles <= pairs || num_k_blocks < 16) continue;
    for (int tail = 1; tail < m_tiles && tail <= 16; ++tail) {
      const int main_tiles = m_tiles - tail;
      const long main_items = static_cast<long>(main_tiles) * n_tiles;
      if (main_items % pairs != 0 && main_items % pairs < pairs * 3 / 4) continue;   // the main window must end on a full wave
      int ts = 1, tk = num_k_blocks;
      const double ct = best_split(tail, n_tiles, bn, num_k_blocks, 16, t_kb, t_epi, pairs, N, ws_bytes, 0, &ts, &tk);
      const double cm = window_cost(main_tiles, n_tiles, bn, 1, num_k_blocks, t_kb, t_epi, pairs, N);
      const double c2 = cm + ct + 6000.0;              // second launch: prologue + drain
      if (c2 < 0.93 * best_cost) {
        best_cost = c2;
        best = Plan{bn, 1, num_k_blocks, tail, ts, tk};
      }
    }
  }
  return best;
}

// TMA maps of the epilogue: 32x32 bf16 boxes, 64-byte swizzle, over the output and (optionally) the residual
int make_epilogue_maps(const GemmParams& p, CUtensorMap* mo, CUtensorMap* mr) {
  const uint32_t box[2] = {32, 32};
  const uint64_t odims[2] = {static_cast<uint64_t>(p.geglu ? p.N / 2 : p.N), static_cast<uint64_t>(p.M)};
  const uint64_t ostr[1] = {static_cast<uint64_t>(p.ldo) * 2};
  int rc = lavie_make_tmap(mo, p.out, 2, odims, ostr, box, CU_TENSOR_MAP_SWIZZLE_64B);
  if (rc) return rc;
  if (p.residual) {
    const uint64_t rdims[2] = {static_cast<uint64_t>(p.N), static_cast<uint64_t>(p.M)};
    const uint64_t rstr[1] = {static_cast<uint64_t>(p.ldr) * 2};
    return lavie_make_tmap(mr, p.residual, 2, rdims, rstr, box, CU_TENSOR_MAP_SWIZZLE_64B);
  }
  *mr = *mo;
  return LAVIE_OK;
}

int launch_window(int bn, const CUtensorMap* a, const CUtensorMap& b, const CUtensorMap& mo, const CUtensorMap& mr,
                  const GemmParams& p, cudaStream_t stream) {
  switch (bn) {
    case 64: return launch_gemm<64>(a[0], a[1], a[2], a[3], b, mo, mr, p, num_sms(), stream);
    case 128: return launch_gemm<128>(a[0], a[1], a[2], a[3], b, mo, mr, p, num_sms(), stream);
    case 160: return launch_gemm<160>(a[0], a[1], a[2], a[3], b, mo, mr, p, num_sms(), stream);
    case 192: return launch_gemm<192>(a[0], a[1], a[2], a[3], b, mo, mr, p, num_sms(), stream);
    case 256: return launch_gemm<256>(a[0], a[1], a[2], a[3], b, mo, mr, p, num_sms(), stream);
    case 320: return launch_gemm<320>(a[0], a[1], a[2], a[3], b, mo, mr, p, num_sms(), stream);
    default: lavie_set_error("unsupported BLOCK_N %d", bn); return LAVIE_ERR_SHAPE;
  }
}

void set_window(GemmParams& p, int m_tile0, int m_tiles, int splits, int kbps);

int make_phase_output_map(const GemmParams& p, CUtensorMap* mo);

int dispatch_maps(const Plan& plan, const CUtensorMap* a, const CUtensorMap& b, GemmParams& p, cudaStream_t stream) {
  CUtensorMap mo, mr;
  int rc;
  if (p.phases > 1) {
    rc = make_phase_output_map(p, &mo);
    mr = mo;
  } else {
    rc = make_epilogue_maps(p, &mo, &mr);
  }
  if (rc) return rc;
  const int m_tiles = (p.M + PAIR_M - 1) / PAIR_M;
  set_window(p, 0, m_tiles - plan.tail_tiles, plan.splits, plan.kb_per_split);
  rc = launch_window(plan.bn, a, b, mo, mr, p, stream);
  if (rc || plan.tail_tiles == 0) return rc;
  set_window(p, m_tiles - plan.tail_tiles, plan.tail_tiles, plan.tail_splits, plan.tail_kb_per_split);
  return launch_window(plan.bn, a, b, mo, mr, p, stream);
}

int dispatch(const Plan& plan, const CUtensorMap& a0, const CUtensorMap& a1, const CUtensorMap& b, GemmParams& p,
             cudaStream_t stream) {
  const CUtensorMap a[4] = {a0, a1, a0, a0};
  return dispatch_maps(plan, a, b, p, stream);
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

int make_weight_map(CUtensorMap* map, const void* w, int N, int K, int bn) {
  const uint64_t dims[2] = {static_cast<uint64_t>(K), static_cast<uint64_t>(N)};
  const uint64_t strides[1] = {static_cast<uint64_t>(K) * 2};
  // each CTA of the pair stages half of the weight rows of one MMA (a 320-wide tile is two 160-wide MMAs)
  const uint32_t box[2] = {BLOCK_K, static_cast<uint32_t>((bn > 256 ? bn / 2 : bn) / 2)};
  return lavie_make_tmap(map, w, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

int fill_epilogue(GemmParams& p, const lavie_epilogue* ep, int N, void* out, int ldo) {
  p.bias = nullptr; p.row_bias = nullptr; p.rows_per_batch = 1; p.ld_row_bias = N; p.residual = nullptr; p.ldr = 0;
  p.geglu = 0;
  p.colstats = nullptr;
  p.mg8 = (N % 10 != 0) ? 1 : 0;
  if (ep) {
    p.colstats = ep->col_stats;
    LAVIE_REQUIRE(!p.colstats || (aligned16(p.colstats) && !ep->geglu && N % 32 == 0 && N <= 8192), LAVIE_ERR_SHAPE,
                  "gemm: col_stats needs a 16-byte aligned buffer, N %% 32 == 0 (<= 8192) and no GEGLU");
    p.bias = ep->bias;
    p.row_bias = ep->row_bias;
    p.rows_per_batch = ep->rows_per_batch > 0 ? ep->rows_per_batch : 1;
    p.ld_row_bias = ep->ld_row_bias > 0 ? ep->ld_row_bias : N;
    p.residual = static_cast<const __nv_bfloat16*>(ep->residual);
    p.ldr = ep->ld_residual;
    p.geglu = ep->geglu;
    LAVIE_REQUIRE(!p.residual || (aligned16(p.residual) && p.ldr % 8 == 0), LAVIE_ERR_ALIGN,
                  "gemm: residual must be 16-byte aligned with ld %% 8 == 0");
    LAVIE_REQUIRE(!p.bias || aligned16(p.bias), LAVIE_ERR_ALIGN, "gemm: bias must be 16-byte aligned");
    LAVIE_REQUIRE(!p.row_bias || (aligned16(p.row_bias) && p.ld_row_bias % 4 == 0), LAVIE_ERR_ALIGN,
                  "gemm: row_bias must be 16-byte aligned with ld %% 4 == 0");
    LAVIE_REQUIRE(!(p.geglu && (p.residual || p.row_bias)), LAVIE_ERR_SHAPE,
                  "gemm: GEGLU epilogue cannot be combined with residual/row_bias");
  }
  p.out = static_cast<__nv_bfloat16*>(out);
  p.ldo = ldo;
  LAVIE_REQUIRE(aligned16(out) && ldo % 8 == 0, LAVIE_ERR_ALIGN, "gemm: out must be 16-byte aligned, ldo %% 8 == 0");
  return LAVIE_OK;
}

// bytes of the caller's workspace the planner may use for partial planes: the tail holds the split-K tickets
size_t plan_ws_bytes(const void* workspace, size_t workspace_bytes, int check) {
  if (workspace == nullptr) return 0;
  if (g_inkernel_reduce && !check && workspace_bytes > 4 * TICKET_BYTES) return workspace_bytes - TICKET_BYTES;
  return workspace_bytes;
}

void apply_plan(GemmParams& p, const Plan& plan, void* workspace, size_t workspace_bytes = 0) {
  if (p.phases < 1) p.phases = 1;
  p.n_tiles = (p.N + plan.bn - 1) / plan.bn;
  p.tickets = nullptr;
  if (workspace != nullptr && plan_ws_bytes(workspace, workspace_bytes, p.check) != workspace_bytes) {
    const size_t blocks = static_cast<size_t>((p.M + PAIR_M - 1) / PAIR_M) * 2 * p.n_tiles;
    if (blocks * sizeof(int) <= TICKET_BYTES)
      p.tickets = reinterpret_cast<int*>(static_cast<char*>(workspace) + workspace_bytes - TICKET_BYTES);
  }
  p.partial = static_cast<float*>(workspace);
  p.debug = g_debug;
  p.k_rot = g_k_rot;
}

void set_window(GemmParams& p, int m_tile0, int m_tiles, int splits, int kbps) {
  p.m_tile0 = m_tile0;
  p.m_tiles = m_tiles;
  const int rows_left = p.M - m_tile0 * PAIR_M;
  p.rows_window = rows_left < m_tiles * PAIR_M ? rows_left : m_tiles * PAIR_M;
  p.splits = splits;
  p.kb_per_split = kbps;
}

}  // namespace

extern int g_lavie_gn_target_ctas;

extern "C" int lavie_debug_set(int what, int value) {
  if (what == 1) g_force_splits = value;
  if (what == 2) g_debug = value;
  if (what == 0) g_k_rot = value;
  if (what == 3) g_lavie_pdl = value ? 1 : 0;
  if (what == 4) g_lavie_attn_poly = value;
  if (what == 5) g_no_tail = value;
  if (what == 6 && value > 0) g_lavie_gn_target_ctas = value;
  if (what == 7) g_inkernel_reduce = value ? 1 : 0;
  if (what == 8) g_lavie_xattn = value ? 1 : 0;
  return 0;
}

extern "C" int lavie_gemm_plan(int M, int N, int K, int conv, int geglu, size_t workspace_bytes, int* block_n,
                               int* splits, int* tail_tiles, int* tail_splits) {
  LAVIE_REQUIRE(M > 0 && N > 0 && K > 0, LAVIE_ERR_SHAPE, "gemm_plan: empty problem M=%d N=%d K=%d", M, N, K);
  const Plan plan = make_plan(M, N, (K + BLOCK_K - 1) / BLOCK_K, 0, geglu != 0, conv != 0, workspace_bytes);
  if (block_n) *block_n = plan.bn;
  if (splits) *splits = plan.splits;
  if (tail_tiles) *tail_tiles = plan.tail_tiles;
  if (tail_splits) *tail_splits = plan.tail_tiles ? plan.tail_splits : 1;
  return LAVIE_OK;
}

namespace {
// check-mode launches need room for one fp32 plane of the (256-row padded) output in the workspace
int check_workspace(int check, int M, int N, const void* workspace, size_t workspace_bytes) {
  if (!check) return LAVIE_OK;
  const size_t need = static_cast<size_t>((M + PAIR_M - 1) / PAIR_M) * PAIR_M * N * sizeof(float);
  LAVIE_REQUIRE(workspace != nullptr && workspace_bytes >= need, LAVIE_ERR_WORKSPACE,
                "check mode: workspace of %zu bytes needed (fp32 accumulator plane), got %zu", need, workspace_bytes);
  return LAVIE_OK;
}

int gemm_impl(const void* a0, int lda0, int k0, const void* a1, int lda1, int k1, const void* w, void* out, int ldo,
              int M, int N, const lavie_epilogue* ep, int block_n, void* workspace, size_t workspace_bytes, int check,
              cudaStream_t stream) {
  const int K = k0 + k1;
  LAVIE_REQUIRE(M > 0 && N > 0 && K > 0, LAVIE_ERR_SHAPE, "gemm: empty problem M=%d N=%d K=%d", M, N, K);
  LAVIE_REQUIRE(N % 8 == 0 && k0 % 8 == 0 && k1 % 8 == 0, LAVIE_ERR_SHAPE, "gemm: N, K must be multiples of 8");
  LAVIE_REQUIRE(k1 == 0 || k0 % BLOCK_K == 0, LAVIE_ERR_SHAPE, "gemm: split-K source boundary must be a multiple of 64");
  LAVIE_REQUIRE(aligned16(a0) && aligned16(w) && lda0 % 8 == 0 && (k1 == 0 || (aligned16(a1) && lda1 % 8 == 0)),
                LAVIE_ERR_ALIGN, "gemm: operands must be 16-byte aligned with ld %% 8 == 0");
  LAVIE_REQUIRE(workspace == nullptr || aligned16(workspace), LAVIE_ERR_ALIGN, "gemm: workspace alignment");
  GemmParams p{};
  const bool geglu = ep && ep->geglu;
  LAVIE_REQUIRE(!geglu || N % 256 == 0, LAVIE_ERR_SHAPE, "gemm: GEGLU needs N %% 256 == 0");
  p.M = M; p.N = N; p.K = K;
  p.num_k_blocks = (K + BLOCK_K - 1) / BLOCK_K;
  p.k_split_blocks = k1 ? k0 / BLOCK_K : p.num_k_blocks;
  p.conv = 0;
  p.check = check;
  int rc = check_workspace(check, M, N, workspace, workspace_bytes);
  if (rc) return rc;
  const Plan plan = make_plan(M, N, p.num_k_blocks, block_n, geglu, false, plan_ws_bytes(workspace, workspace_bytes, check));
  apply_plan(p, plan, workspace, workspace_bytes);
  rc = fill_epilogue(p, ep, N, out, ldo);
  if (rc) return rc;
  CUtensorMap ma0, ma1, mb;
  {
    const uint64_t dims[2] = {static_cast<uint64_t>(k0), static_cast<uint64_t>(M)};
    const uint64_t strides[1] = {static_cast<uint64_t>(lda0) * 2};
    const uint32_t box[2] = {BLOCK_K, BLOCK_M};
    rc = lavie_make_tmap(&ma0, a0, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  }
  if (k1) {
    const uint64_t dims[2] = {static_cast<uint64_t>(k1), static_cast<uint64_t>(M)};
    const uint64_t strides[1] = {static_cast<uint64_t>(lda1) * 2};
    const uint32_t box[2] = {BLOCK_K, BLOCK_M};
    rc = lavie_make_tmap(&ma1, a1, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  } else {
    ma1 = ma0;
  }
  rc = make_weight_map(&mb, w, N, K, plan.bn);
  if (rc) return rc;
  return dispatch(plan, ma0, ma1, mb, p, stream);
}
}  // namespace

extern "C" int lavie_gemm_bf16(const void* a0, int lda0, int k0, const void* a1, int lda1, int k1, const void* w,
                               void* out, int ldo, int M, int N, const lavie_epilogue* ep, int block_n,
                               void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  return gemm_impl(a0, lda0, k0, a1, lda1, k1, w, out, ldo, M, N, ep, block_n, workspace, workspace_bytes, 0, stream);
}

extern "C" int lavie_check_gemm(const void* a0, int lda0, int k0, const void* a1, int lda1, int k1, const void* w,
                                void* out, int ldo, int M, int N, const lavie_epilogue* ep, void* workspace,
                                size_t workspace_bytes, cudaStream_t stream) {
  return gemm_impl(a0, lda0, k0, a1, lda1, k1, w, out, ldo, M, N, ep, 0, workspace, workspace_bytes, 1, stream);
}

namespace {
int frame_conv_impl(const void* x, int ldx, long long rows_in, int C, int taps, int tap_rows, const void* w, void* out,
                    int ldo, int M, int N, const lavie_epilogue* ep, int block_n, void* workspace,
                    size_t workspace_bytes, cudaStream_t stream) {
  LAVIE_REQUIRE(M > 0 && N > 0 && taps >= 1 && taps <= 9 && tap_rows > 0, LAVIE_ERR_SHAPE,
                "frame_conv: empty problem M=%d N=%d taps=%d tap_rows=%d", M, N, taps, tap_rows);
  LAVIE_REQUIRE(C % BLOCK_K == 0 && N % 8 == 0 && ldx % 8 == 0, LAVIE_ERR_SHAPE,
                "frame_conv: C=%d must be a multiple of 64, N and ldx multiples of 8", C);
  LAVIE_REQUIRE(rows_in >= static_cast<long long>(M) + static_cast<long long>(taps - 1) * tap_rows, LAVIE_ERR_SHAPE,
                "frame_conv: the padded input holds %lld rows, M + (taps-1)*tap_rows = %lld needed", rows_in,
                static_cast<long long>(M) + static_cast<long long>(taps - 1) * tap_rows);
  LAVIE_REQUIRE(aligned16(x) && aligned16(w), LAVIE_ERR_ALIGN, "frame_conv: alignment");
  LAVIE_REQUIRE(workspace == nullptr || aligned16(workspace), LAVIE_ERR_ALIGN, "frame_conv: workspace alignment");
  LAVIE_REQUIRE(!(ep && ep->geglu), LAVIE_ERR_SHAPE, "frame_conv: GEGLU epilogue not supported");
  GemmParams p{};
  p.M = M; p.N = N; p.K = taps * C;
  p.num_k_blocks = taps * (C / BLOCK_K);
  p.k_split_blocks = p.num_k_blocks;
  p.c_blocks = C / BLOCK_K;
  p.tap_rows = tap_rows;
  p.conv = 2;
  p.check = 0;
  const Plan plan = make_plan(M, N, p.num_k_blocks, block_n, false, false, plan_ws_bytes(workspace, workspace_bytes, 0));
  apply_plan(p, plan, workspace, workspace_bytes);
  int rc = fill_epilogue(p, ep, N, out, ldo);
  if (rc) return rc;
  CUtensorMap ma, mb;
  const uint64_t dims[2] = {static_cast<uint64_t>(C), static_cast<uint64_t>(rows_in)};
  const uint64_t strides[1] = {static_cast<uint64_t>(ldx) * 2};
  const uint32_t box[2] = {BLOCK_K, BLOCK_M};
  rc = lavie_make_tmap(&ma, x, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  rc = make_weight_map(&mb, w, N, taps * C, plan.bn);
  if (rc) return rc;
  return dispatch(plan, ma, ma, mb, p, stream);
}
}  // namespace

extern "C" int lavie_frame_conv_bf16(const void* x, int ldx, long long rows_in, int C, int taps, int tap_rows,
                                     const void* w, void* out, int ldo, int M, int N, const lavie_epilogue* ep,
                                     int block_n, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  return frame_conv_impl(x, ldx, rows_in, C, taps, tap_rows, w, out, ldo, M, N, ep, block_n, workspace, workspace_bytes,
                         stream);
}

namespace {
// 5-D view of the contiguous high-resolution output [NF, 2H, 2W, N]: (c, px, x, py, n*H + y); one epilogue chunk = 32
// consecutive low-resolution pixels x 32 channels = a box of (32 / by) x by pixels of one phase.
int make_phase_output_map(const GemmParams& p, CUtensorMap* mo) {
  const int W = p.lowres_w;
  const uint32_t bx = W >= 32 ? 32u : static_cast<uint32_t>(W);
  const uint32_t by = 32u / bx;
  const uint64_t N = static_cast<uint64_t>(p.N);
  const uint64_t dims[5] = {N, 2, static_cast<uint64_t>(W), 2, static_cast<uint64_t>(p.M / W)};
  const uint64_t strides[4] = {N * 2, 2 * N * 2, 2 * static_cast<uint64_t>(W) * N * 2, 4 * static_cast<uint64_t>(W) * N * 2};
  const uint32_t box[5] = {32, 1, bx, 1, by};
  return lavie_make_tmap(mo, p.out, 5, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B);
}
}  // namespace

extern "C" int lavie_upsample_conv3x3_supported(int H, int W, int C) {
  (void)H;
  return (C % BLOCK_K == 0 && W > 0 && (W % 32 == 0 || 32 % W == 0)) ? 1 : 0;
}

extern "C" int lavie_upsample_conv3x3_bf16(const void* x, int NF, int H, int W, int C, const void* w_phases, void* out,
                                           int N, const lavie_epilogue* ep, int block_n, cudaStream_t stream) {
  LAVIE_REQUIRE(lavie_upsample_conv3x3_supported(H, W, C), LAVIE_ERR_SHAPE,
                "upsample_conv3x3: C=%d must be a multiple of 64 and W=%d a divisor or a multiple of 32", C, W);
  LAVIE_REQUIRE(N % 8 == 0 && aligned16(x) && aligned16(w_phases) && aligned16(out), LAVIE_ERR_ALIGN,
                "upsample_conv3x3: alignment");
  LAVIE_REQUIRE(!(ep && (ep->geglu || ep->residual || ep->row_bias)), LAVIE_ERR_SHAPE,
                "upsample_conv3x3: only bias and col_stats are supported in the epilogue");
  const int M = NF * H * W;                       // low-resolution pixels; every one produces 2 x 2 output pixels
  GemmParams p{};
  p.M = M; p.N = N; p.K = 4 * C;
  p.num_k_blocks = 4 * (C / BLOCK_K);
  p.k_split_blocks = p.num_k_blocks;
  p.c_blocks = C / BLOCK_K;
  p.out_h = H; p.out_w = W; p.conv_stride = 1;
  p.conv = 3;
  p.phases = 4;
  p.lowres_w = W;
  p.slabs_total = (M + 31) / 32;
  p.check = 0;
  // the four phases multiply the work items: plan as if M were 4x as tall; no split-K (the partial planes are per phase)
  const Plan plan = make_plan(4 * M, N, p.num_k_blocks, block_n, false, true, 0, true);
  apply_plan(p, plan, nullptr);
  int rc = fill_epilogue(p, ep, N, out, N);
  if (rc) return rc;
  CUtensorMap ma[4], mb;
  for (int ph = 0; ph < 4; ++ph) {
    rc = lavie_make_tmap_im2col(&ma[ph], x, NF, H, W, C, BLOCK_K, BLOCK_M, 1, (ph & 1) - 1, (ph >> 1) - 1, (ph & 1) - 1,
                                (ph >> 1) - 1);
    if (rc) return rc;
  }
  // weights [4 phases * N, 4 * C]: phase-major rows, K ordered (a, b, c)
  {
    const uint64_t dims[2] = {static_cast<uint64_t>(4 * C), static_cast<uint64_t>(4) * N};
    const uint64_t strides[1] = {static_cast<uint64_t>(4 * C) * 2};
    const uint32_t box[2] = {BLOCK_K, static_cast<uint32_t>((plan.bn > 256 ? plan.bn / 2 : plan.bn) / 2)};
    rc = lavie_make_tmap(&mb, w_phases, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  }
  Plan single = plan;
  single.splits = 1; single.kb_per_split = p.num_k_blocks; single.tail_tiles = 0;
  return dispatch_maps(single, ma, mb, p, stream);
}

extern "C" int lavie_conv3x3_supported(int H, int W, int C) {
  (void)H; (void)W;
  return C % BLOCK_K == 0 ? 1 : 0;      // im2col-mode TMA handles any image geometry; channels come in 64-wide slabs
}

extern "C" int lavie_conv3x3_out_size(int n, int stride, int pad_before, int pad_after) {
  const int padded = n + pad_before + pad_after;
  return padded < 3 || stride < 1 ? 0 : (padded - 3) / stride + 1;
}

namespace {
int conv3x3_impl(const void* x, int NF, int H, int W, int C, int stride, int pad_before, int pad_after, const void* w,
                 void* out, int ldo, int N, const lavie_epilogue* ep, int block_n, void* workspace,
                 size_t workspace_bytes, int check, cudaStream_t stream) {
  LAVIE_REQUIRE(lavie_conv3x3_supported(H, W, C), LAVIE_ERR_SHAPE, "conv3x3: C=%d must be a multiple of 64", C);
  LAVIE_REQUIRE(stride == 1 || stride == 2, LAVIE_ERR_SHAPE, "conv3x3: stride must be 1 or 2");
  LAVIE_REQUIRE((pad_before == 0 || pad_before == 1) && (pad_after == 0 || pad_after == 1), LAVIE_ERR_SHAPE,
                "conv3x3: padding (%d, %d) must be 0 or 1 on each side", pad_before, pad_after);
  const int Ho = lavie_conv3x3_out_size(H, stride, pad_before, pad_after);
  const int Wo = lavie_conv3x3_out_size(W, stride, pad_before, pad_after);
  LAVIE_REQUIRE(Ho > 0 && Wo > 0, LAVIE_ERR_SHAPE, "conv3x3: H=%d W=%d too small for padding (%d, %d)", H, W, pad_before,
                pad_after);
  LAVIE_REQUIRE(N % 8 == 0 && aligned16(x) && aligned16(w), LAVIE_ERR_ALIGN, "conv3x3: alignment");
  LAVIE_REQUIRE(workspace == nullptr || aligned16(workspace), LAVIE_ERR_ALIGN, "conv3x3: workspace alignment");
  LAVIE_REQUIRE(!(ep && ep->geglu), LAVIE_ERR_SHAPE, "conv3x3: GEGLU epilogue not supported");
  const int M = NF * Ho * Wo;
  GemmParams p{};
  p.M = M; p.N = N; p.K = 9 * C;
  p.num_k_blocks = 9 * (C / BLOCK_K);
  p.k_split_blocks = p.num_k_blocks;
  p.c_blocks = C / BLOCK_K;
  p.out_h = Ho; p.out_w = Wo; p.conv_stride = stride; p.pad_before = pad_before;
  p.conv = 1;
  p.check = check;
  int rc = check_workspace(check, M, N, workspace, workspace_bytes);
  if (rc) return rc;
  const Plan plan = make_plan(M, N, p.num_k_blocks, block_n, false, true, plan_ws_bytes(workspace, workspace_bytes, check));
  apply_plan(p, plan, workspace, workspace_bytes);
  rc = fill_epilogue(p, ep, N, out, ldo);
  if (rc) return rc;
  CUtensorMap ma, mb;
  rc = lavie_make_tmap_im2col(&ma, x, NF, H, W, C, BLOCK_K, BLOCK_M, stride, -pad_before, -pad_before, pad_after - 2,
                              pad_after - 2);
  if (rc) return rc;
  rc = make_weight_map(&mb, w, N, 9 * C, plan.bn);
  if (rc) return rc;
  return dispatch(plan, ma, ma, mb, p, stream);
}
}  // namespace

extern "C" int lavie_conv3x3_bf16(const void* x, int NF, int H, int W, int C, int stride, const void* w, void* out,
                                  int ldo, int N, const lavie_epilogue* ep, int block_n, void* workspace,
                                  size_t workspace_bytes, cudaStream_t stream) {
  return conv3x3_impl(x, NF, H, W, C, stride, 1, 1, w, out, ldo, N, ep, block_n, workspace, workspace_bytes, 0, stream);
}

extern "C" int lavie_conv3x3_pad_bf16(const void* x, int NF, int H, int W, int C, int stride, int pad_before,
                                      int pad_after, const void* w, void* out, int ldo, int N, const lavie_epilogue* ep,
                                      int block_n, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  return conv3x3_impl(x, NF, H, W, C, stride, pad_before, pad_after, w, out, ldo, N, ep, block_n, workspace,
                      workspace_bytes, 0, stream);
}

extern "C" int lavie_check_conv3x3(const void* x, int NF, int H, int W, int C3, int stride, const void* w, void* out,
                                   int ldo, int N, const lavie_epilogue* ep, void* workspace, size_t workspace_bytes,
                                   cudaStream_t stream) {
  return conv3x3_impl(x, NF, H, W, C3, stride, 1, 1, w, out, ldo, N, ep, 0, workspace, workspace_bytes, 1, stream);
}
