/* lavie_b200 -- C ABI of the sm_100a kernels behind LaVie's per-step denoiser.
 *
 * One shared object (liblavie_b200.so), plain pointers and sizes, no torch types.  The reference is pure
 * PyTorch and has no FFI of its own; every entry point below names the reference call it replaces
 * (paths relative to the reference root, e.g. base/models/attention.py:209-239).  INTEGRATION.md shows the
 * ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *  - All activation tensors are bf16, channels-last: a feature map [B,C,F,H,W] of the reference is stored as
 *    rows = (b, f, y, x) pixels, columns = channels, with an explicit row stride ("ld", in ELEMENTS).
 *  - Weights are bf16 [out_features, in_features] row-major (nn.Linear layout); 3x3 conv weights are repacked by
 *    the caller to [Cout, kh, kw, Cin].  Biases / statistics / time-embedding vectors are fp32.
 *  - Ownership: the caller allocates every buffer (inputs, outputs, workspaces).  The library never allocates or
 *    frees device memory and keeps no global state besides lazily configured kernel attributes.
 *  - Every function enqueues work on `stream` and returns immediately: no host synchronisation, safe under CUDA
 *    graph capture, re-entrant from one host thread per device.
 *  - Return value: LAVIE_OK (0) or a negative lavie_status; lavie_last_error() gives a thread-local message.
 *    Nothing throws, nothing calls exit().
 */
#ifndef LAVIE_B200_H_
#define LAVIE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* lavie_stream_t; /* == cudaStream_t */

typedef enum {
  LAVIE_OK = 0,
  LAVIE_ERR_SHAPE = -1,     /* unsupported / inconsistent dimensions */
  LAVIE_ERR_ALIGN = -2,     /* pointer or leading dimension not 16-byte aligned */
  LAVIE_ERR_WORKSPACE = -3, /* caller workspace too small */
  LAVIE_ERR_CUDA = -4,      /* CUDA runtime / driver error (message has the code) */
  LAVIE_ERR_DRIVER = -5     /* cuTensorMapEncodeTiled unavailable */
} lavie_status;

const char* lavie_last_error(void);
int lavie_abi_version(void);
/* Tuning hooks for tests/benchmarks (never needed for correct results): what = 1 forces the split-K factor of the
 * GEMM (0 = automatic); 2 = debug bit mask (512: GEMM per-tile clock64 timeline into the workspace); 3 = programmatic
 * dependent launch on/off; 4 = attention: every n-th exp2 on the FMA pipe (0 = all on the MUFU); 5 = no split-K tail
 * windows; 7 = in-kernel split-K reduction on/off (default off); 8 = single-pass mma.sync attention kernel for short key
 * sequences (Sk <= 80: the text cross-attentions) on/off (default off: bound by the legacy HMMA rate, not faster). */
int lavie_debug_set(int what, int value);
/* Device scratch (>= 64 KB) that the attention kernel fills with a per-tile clock64 timeline of one CTA; NULL = off. */
int lavie_debug_buffer(void* device_ptr);

/* Fused GEMM epilogue: out = bf16( acc + bias[n] + row_bias[row / rows_per_batch][n] + residual[row][n] ), or with
 * geglu != 0: out[:, j] = (acc[:, j] + bias) * gelu_erf(acc[:, j + 128] + bias') per 256-column tile. */
typedef struct {
  const float* bias;     /* [N] or NULL */
  const float* row_bias; /* [M / rows_per_batch, ld_row_bias] or NULL */
  int ld_row_bias;       /* elements; 0 = N */
  int rows_per_batch;
  const void* residual;  /* bf16 [M, ld_residual] or NULL */
  int ld_residual;
  int geglu;
  float* col_stats;      /* NULL or fp32 [ceil(M / 32), N / 32, 4, 2] (N % 32 == 0): per 32-row slab and micro-group of
                            mg channels, (sum, sum of squares) of the bf16-rounded outputs; mg = 10 when N % 10 == 0 (base /
                            interpolation model: every GroupNorm group is a whole number of decades), else 8 (VSR model:
                            groups of 8..64 channels).  Entry [slab][chunk][piece] covers the part of micro-group
                            (chunk * 32) / mg + piece that lies inside columns [chunk * 32, chunk * 32 + 32).  This is the
                            statistics pass of the GroupNorm that consumes the output (resnet.py:180,191; attention.py:369),
                            emitted by the producer's epilogue instead of a second read of the tensor; fold with
                            lavie_groupnorm_finalize_colsums.  Not in check mode. */
} lavie_epilogue;

/* nn.Linear / 1x1 InflatedConv3d: out[M,N] = [a0 | a1][M, k0+k1] * w[N, k0+k1]^T (+ epilogue).
 * a1/k1 = 0 for a single source; two sources fold torch.cat([h, skip], 1) (unet_blocks.py:538,630) in front of
 * resnet.py:202-203 conv_shortcut.  Replaces attention.py:95-104 (to_q/k/v/out), :328,356 (proj_in/out),
 * diffusers FeedForward (mirror vsr/models/diffusers_attention.py:734-822).  block_n = 0 lets the library choose.
 * workspace (optional, caller-owned, fp32) enables deterministic split-K on small-M / large-K problems: the library
 * uses at most workspace_bytes and picks splits <= workspace_bytes / (4*M*N).  Only with lavie_debug_set(7, 1) (in-kernel
 * reduction: the CTA whose partial block arrives last sums the planes in split order and runs the fused epilogue; same
 * bits, no reduction launch, measured slower and therefore off by default) and workspace_bytes > 256 KiB, the LAST 64 KiB
 * hold its tickets: that tail must be ZERO before the first call and the library leaves it zero. */
/* Host-only query: the launch plan the library would choose for a GEMM (conv = 0) or a 3x3 conv (conv = 1, K = 9*Cin)
 * on the current device (148 SMs assumed when no device is present): tile width, split-K factor of the main window,
 * number of 256-row tile rows issued as a second split-K "tail window" launch (0 = single launch) and its split-K
 * factor.  Lets callers and tests see wave quantisation decisions without running anything. */
int lavie_gemm_plan(int M, int N, int K, int conv, int geglu, size_t workspace_bytes, int* block_n, int* splits,
                    int* tail_tiles, int* tail_splits);
int lavie_gemm_bf16(const void* a0, int lda0, int k0, const void* a1, int lda1, int k1, const void* w, void* out,
                    int ldo, int M, int N, const lavie_epilogue* ep, int block_n, void* workspace,
                    size_t workspace_bytes, lavie_stream_t stream);

/* Upsample3D (resnet.py:44-76: F.interpolate(scale_factor=(1,2,2), mode="nearest") then the 3x3 conv) WITHOUT the 4x map:
 * a 3x3 conv on a nearest-2x upsampled image equals, for each output-pixel parity (py, px), a 2x2 conv on the
 * low-resolution image whose taps are sums of the original ones -- 16 tap-GEMMs of M = NF*H*W rows instead of 36 (2.25x
 * fewer FLOPs) and no upsampled copy in HBM.  x bf16 [NF, H, W, C] contiguous (C % 64 == 0, W a divisor or a multiple of
 * 32: lavie_upsample_conv3x3_supported); w_phases bf16 [4, N, 2, 2, C] = phase (py*2+px)-major rows, tap (a, b) reads
 * source pixel (y + py - 1 + a, x + px - 1 + b), weights: py = 0 -> a = 0: kh 0, a = 1: kh 1 + kh 2; py = 1 -> a = 0: kh 0 +
 * kh 1, a = 1: kh 2 (same along x).  out bf16 [NF, 2H, 2W, N] contiguous.  Epilogue: bias and col_stats only (the
 * statistics come in 4 phase segments, see lavie_groupnorm_finalize_colsums_seg). */
int lavie_upsample_conv3x3_supported(int H, int W, int C);
int lavie_upsample_conv3x3_bf16(const void* x, int NF, int H, int W, int C, const void* w_phases, void* out, int N,
                                const lavie_epilogue* ep, int block_n, lavie_stream_t stream);

/* nn.Conv3d with a (taps,1,1) kernel over FRAMES (vsr/models/resnet.py:253-254,269: ResnetBlock3DCNN conv1 / conv2) as
 * an implicit GEMM with K = taps*C.  x points at a channels-last map of ONE batch item whose frame axis the caller has
 * padded with taps/2 zero frames on both sides: rows_in = (F + taps - 1) * tap_rows rows of C channels (row stride ldx),
 * tap_rows = H*W.  Output row m (M = F*H*W rows) = sum_t x[m + t*tap_rows, :] . w[:, t, :]; w is bf16 [N, taps, C]. */
int lavie_frame_conv_bf16(const void* x, int ldx, long long rows_in, int C, int taps, int tap_rows, const void* w,
                          void* out, int ldo, int M, int N, const lavie_epilogue* ep, int block_n, void* workspace,
                          size_t workspace_bytes, lavie_stream_t stream);

/* 3x3 pad-1 InflatedConv3d, stride 1 or 2 (resnet.py:13-21; Downsample3D :102-110) as implicit GEMM over a CONTIGUOUS
 * channels-last map x[NF, H, W, C]; w is [N, 3, 3, C]; out has NF*Ho*Wo rows.  The A operand is fetched with
 * im2col-mode TMA (the hardware walks the output pixels and zero-fills the halo), so any H, W works;
 * lavie_conv3x3_supported() only asks for C % 64 == 0 (otherwise: lavie_im2col3x3_bf16 + lavie_gemm_bf16). */
int lavie_conv3x3_supported(int H, int W, int C);
int lavie_conv3x3_bf16(const void* x, int NF, int H, int W, int C, int stride, const void* w, void* out, int ldo, int N,
                       const lavie_epilogue* ep, int block_n, void* workspace, size_t workspace_bytes,
                       lavie_stream_t stream);
/* The same conv with explicit zero padding: pad_before rows / columns before the image and pad_after after it, each 0
 * or 1, on both axes.  (1, 1) is lavie_conv3x3_bf16; (0, 1) with stride 2 is diffusers' Downsample2D(padding=0), which
 * pads (0, 1, 0, 1) and then runs a pad-0 conv: output pixel i reads input rows 2i, 2i+1, 2i+2.  The output has
 * lavie_conv3x3_out_size(H, ...) x lavie_conv3x3_out_size(W, ...) pixels per image; the epilogue is unchanged. */
int lavie_conv3x3_pad_bf16(const void* x, int NF, int H, int W, int C, int stride, int pad_before, int pad_after,
                           const void* w, void* out, int ldo, int N, const lavie_epilogue* ep, int block_n,
                           void* workspace, size_t workspace_bytes, lavie_stream_t stream);
/* Output extent of a 3x3 conv along one axis of n pixels: (n + pad_before + pad_after - 3) / stride + 1, 0 when the
 * padded extent is shorter than the filter.  Pure host query. */
int lavie_conv3x3_out_size(int n, int stride, int pad_before, int pad_after);

/* Patch matrix for the general / strided conv (Downsample3D stride 2, resnet.py:102-110):
 * col[NF*Ho*Wo, 9*C] with K ordered (kh, kw, c), pad 1. */
int lavie_im2col3x3_bf16(const void* x, int NF, int H, int W, int C, int stride, void* col, lavie_stream_t stream);

/* GroupNorm over channels-last rows, 32-style groups of C/groups contiguous channels.
 * Sample s = rows [s*rows_per_sample, (s+1)*rows_per_sample): rows_per_sample = F*H*W reproduces nn.GroupNorm on the
 * 5-D tensor (statistics across frames, resnet.py:180,191; unet.py:504), = H*W the per-frame norm of
 * Transformer3DModel (attention.py:363-369).  The input may be the channel concat of two sources.
 *   stats    : partial[samples, chunks, groups, 2] (sum, sum of squares), chunks = lavie_groupnorm_chunks()
 *   finalize : scale_shift[samples, C, 2] with y = x*scale + shift  (folds gamma/beta, mean, rstd)
 *   apply    : y = act(x*scale + shift), act = SiLU when silu != 0; writes a contiguous [rows, C] bf16 tensor */
int lavie_groupnorm_chunks(int samples, int rows_per_sample);
int lavie_groupnorm_stats(const void* x0, int ld0, int c0, const void* x1, int ld1, int c1, int samples,
                          int rows_per_sample, int groups, float* partial, lavie_stream_t stream);
int lavie_groupnorm_finalize(const float* partial, int samples, int chunks, int groups, int C,
                             long long count_per_group, const float* gamma, const float* beta, float eps,
                             float* scale_shift, lavie_stream_t stream);
/* stats + finalize in ONE launch: the last block of each sample to publish its partials (atomic ticket) folds them
 * into scale_shift with the arithmetic of lavie_groupnorm_finalize.  tickets: int[samples], zero on entry, left zero. */
int lavie_groupnorm_scale_shift(const void* x0, int ld0, int c0, const void* x1, int ld1, int c1, int samples,
                                int rows_per_sample, int groups, const float* gamma, const float* beta, float eps,
                                float* partial, int* tickets, float* scale_shift, lavie_stream_t stream);
int lavie_groupnorm_apply(const void* x0, int ld0, int c0, const void* x1, int ld1, int c1, int samples,
                          int rows_per_sample, const float* scale_shift, int silu, void* y, int ldy,
                          lavie_stream_t stream);

/* GroupNorm statistics from the PRODUCERS' micro-group sums (lavie_epilogue.col_stats) instead of lavie_groupnorm_stats:
 * cs0 / cs1 = [rows / 32, c / 32, 4, 2] of the one or two concatenated sources (c0, c1 multiples of 32; C / groups a
 * multiple of 10); rows_per_sample must be a multiple of 32 (a slab never straddles two samples).  Same (scale, shift)
 * output and fp64 combination as lavie_groupnorm_finalize.
 * lavie_groupnorm_reduce_colsums stops at sums[samples, groups, 2] (fp64), the quantity frame shards exchange. */
int lavie_groupnorm_finalize_colsums(const float* cs0, int c0, const float* cs1, int c1, int samples,
                                     int rows_per_sample, int groups, const float* gamma, const float* beta, float eps,
                                     float* scale_shift, lavie_stream_t stream);
/* The same with sources whose statistics were written by lavie_upsample_conv3x3_bf16: their slabs sit in segs = 4 phase
 * segments (one per output-pixel parity), each holding a quarter of every sample's slabs; segs = 1 for ordinary sources. */
int lavie_groupnorm_finalize_colsums_seg(const float* cs0, int c0, int segs0, const float* cs1, int c1, int segs1,
                                         int samples, int rows_per_sample, int groups, const float* gamma,
                                         const float* beta, float eps, float* scale_shift, lavie_stream_t stream);
int lavie_groupnorm_reduce_colsums(const float* cs0, int c0, const float* cs1, int c1, int samples, int rows_per_sample,
                                   int groups, double* sums, lavie_stream_t stream);

/* nn.LayerNorm over the channel dimension of every row (attention.py:444-477 norm1/norm2/norm_temp/norm3). */
int lavie_layernorm_bf16(const void* x, int ldx, const float* gamma, const float* beta, float eps, void* y, int ldy,
                         int rows, int C, lavie_stream_t stream);

/* Frame sharding (SURVEY.md 8e; one CFG half spread over P GPUs, F/P frames each).
 *  - lavie_groupnorm_reduce: ordered sum of the stats partials -> sums[samples, groups, 2] (fp64); the caller
 *    all-reduces `sums` across the frame shards (NCCL) and calls lavie_groupnorm_finalize_sums with the GLOBAL count.
 *  - lavie_layernorm_scatter_bf16: LayerNorm whose output row (f, pixel) lands at (pixel / hwp, f, pixel % hwp):
 *    the send buffer of the all-to-all that switches from frame sharding to pixel sharding before the temporal
 *    attention (replaces the in-memory transpose attention.py:549-550).
 *  - lavie_add_gathered_bf16: out[(f, pixel)] = res[(f, pixel)] + z[(pixel / hwp, f, pixel % hwp)]: residual add over
 *    the receive buffer of the all-to-all back (attention.py:554-555). */
int lavie_groupnorm_reduce(const float* partial, int samples, int chunks, int groups, double* sums,
                           lavie_stream_t stream);
int lavie_groupnorm_finalize_sums(const double* sums, int samples, int groups, int C, long long count_per_group,
                                  const float* gamma, const float* beta, float eps, float* scale_shift,
                                  lavie_stream_t stream);
int lavie_layernorm_scatter_bf16(const void* x, int ldx, const float* gamma, const float* beta, float eps, void* y,
                                 int ldy, int rows, int C, int hw, int hwp, lavie_stream_t stream);
int lavie_add_gathered_bf16(const void* res, int ldr, const void* z, int ldz, void* out, int ldo, int rows, int C,
                            int hw, int hwp, lavie_stream_t stream);

/* The same three exchanges fused into the compute kernels over NVLink PEER MEMORY (no NCCL on the data path).
 * `*_ptrs` are HOST arrays of P device pointers, entry r = rank r's buffer as mapped into this process (CUDA IPC /
 * symmetric memory, set up by the caller); flag_ptrs[r] -> uint32[P] (zero-initialised), slot_ptrs[r] ->
 * double[2][P][samples*groups*2]; epoch_counter is a device uint32 owned by this rank (zero-initialised).  All ranks of
 * the frame group must issue the same sequence of these calls.
 *  - lavie_gn_exchange_finalize: local reduce -> store my sums into every peer -> flag barrier -> ordered sum ->
 *    (scale, shift).  Replaces lavie_groupnorm_reduce + all-reduce + lavie_groupnorm_finalize_sums.
 *  - lavie_layernorm_scatter_p2p: LayerNorm whose rows are stored into the peers' receive buffers
 *    (recv_ptrs[r] -> bf16 [F, hw/P, C] on rank r); follow with lavie_rank_barrier before reading the local one.
 *  - lavie_add_gathered_p2p: out = res + rows loaded from the peers' y buffers (y_ptrs[r] -> bf16 [F, hw/P, C]);
 *    precede with lavie_rank_barrier (every rank's y complete).
 *  - lavie_rank_barrier: "everything I launched before this is done and visible" handshake among the P ranks. */
/* Bounded waits: a rank whose peer does not signal within `timeout_seconds` of wall time (default 30; <= 0 keeps the
 * current value) writes uint32 {0x4C564945, my rank, missing peer, epoch wanted, epoch seen} into `host_mapped_words`
 * (pinned, device-accessible HOST memory of >= 8 words owned by the caller, or NULL for no report) and traps.  The trap
 * is a sticky CUDA error on that rank; its peers, never signalled, time out the same way: one rank's failure aborts the
 * whole frame group. */
int lavie_p2p_fault_buffer(void* host_mapped_words, int timeout_seconds);
int lavie_rank_barrier(void* const* flag_ptrs, unsigned int* epoch_counter, int P, int my_rank, lavie_stream_t stream);
int lavie_gn_exchange_finalize(const float* partial, int samples, int chunks, int groups, int C,
                               long long count_per_group_global, const float* gamma, const float* beta, float eps,
                               float* scale_shift, void* const* slot_ptrs, void* const* flag_ptrs,
                               unsigned int* epoch_counter, int P, int my_rank, lavie_stream_t stream);
/* the same exchange starting from this rank's fp64 sums[samples, groups, 2] (lavie_groupnorm_reduce_colsums) */
int lavie_gn_exchange_finalize_sums(const double* local_sums, int samples, int groups, int C,
                                    long long count_per_group_global, const float* gamma, const float* beta, float eps,
                                    float* scale_shift, void* const* slot_ptrs, void* const* flag_ptrs,
                                    unsigned int* epoch_counter, int P, int my_rank, lavie_stream_t stream);
/* frame_off = global index of this rank's first frame (shards may be uneven: 61 interpolation frames = 16/15/15/15);
 * negative = my_rank * rows / hw (equal shards).
 * Fused barriers (flag_ptrs != NULL, with the rank's epoch counter and a zero-initialised device int `ticket` that the
 * kernel leaves zero): the flag barrier runs INSIDE the kernel instead of a separate lavie_rank_barrier launch --
 * scatter / halo push: the last block to finish signals the peers and waits for theirs (kernel completion == every
 * rank's rows have landed); add_gathered: block 0 signals "my y buffer is complete", every block waits for all peers
 * before its first peer load. */
int lavie_layernorm_scatter_p2p(const void* x, int ldx, const float* gamma, const float* beta, float eps,
                                void* const* recv_ptrs, int rows, int C, int hw, int hwp, int P, int my_rank,
                                int frame_off, void* const* flag_ptrs, unsigned int* epoch_counter, int* ticket,
                                lavie_stream_t stream);
int lavie_add_gathered_p2p(const void* res, int ldr, void* const* y_ptrs, void* out, int ldo, int rows, int C, int hw,
                           int hwp, int P, int my_rank, int frame_off, void* const* flag_ptrs,
                           unsigned int* epoch_counter, int* ticket, lavie_stream_t stream);
/* lavie_gn_exchange_finalize starting from the producers' micro-group statistics of this rank (lavie_epilogue.col_stats):
 * local reduction, peer exchange and finalize in ONE single-block launch. */
int lavie_gn_exchange_finalize_colsums(const float* cs0, int c0, const float* cs1, int c1, int samples, int rows_local,
                                       int groups, long long count_per_group_global, const float* gamma,
                                       const float* beta, float eps, float* scale_shift, void* const* slot_ptrs,
                                       void* const* flag_ptrs, unsigned int* epoch_counter, int P, int my_rank,
                                       lavie_stream_t stream);
/* Halo exchange of SparseCausalAttention under frame sharding (interpolation/models/attention.py:629-638): ext_ptrs[r] ->
 * rank r's buffer [2 halo frames | its local frames] of frame_bytes each.  Rank 0 stores first_frame (frame 0 of the
 * video) into block 0 of EVERY rank, every rank but the last stores last_frame (its last local frame) into block 1 of its
 * right neighbour.  Follow with lavie_rank_barrier (or pass flag_ptrs for the fused barrier), then
 * lavie_attention_strided_bf16(sc_halo = 1, or 2 on rank 0). */
int lavie_halo_push_p2p(const void* first_frame, const void* last_frame, long long frame_bytes, void* const* ext_ptrs,
                        int P, int my_rank, void* const* flag_ptrs, unsigned int* epoch_counter, int* ticket,
                        lavie_stream_t stream);

/* softmax(q k^T * scale) v per (batch, head)  (CrossAttention._attention, attention.py:209-239).
 * q rows = batch*Sq, k/v rows = (batch / kv_batch_div)*Sk (kv_batch_div = F shares the text keys across frames,
 * attention.py:364).  Head h occupies columns [h*head_pitch, h*head_pitch + d) of q/k/v (pitch >= d rounded up to 16,
 * padding columns must be zero) and [h*d, (h+1)*d) of o. */
int lavie_attention_bf16(const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, void* o, int ldo,
                         int batch, int heads, int Sq, int Sk, int d, int head_pitch, int kv_batch_div, float scale,
                         lavie_stream_t stream);

/* The same kernel with explicit strides (in ELEMENTS) and the interpolation model's attention variants:
 *  - row of (batch b, token s) = base + b * batch_stride + s * seq_stride, so a sequence need not be contiguous rows:
 *    the frames of one pixel (seq_stride = H*W*ld, batch_stride = ld) give the PLAIN temporal attention of the
 *    interpolation UNet (interpolation/models/attention.py:536-545,598-606: CrossAttention over frames, no RoPE, no
 *    bias) without the two (b f) d c <-> (b d) f c transposes, for any number of frames (61 in LaVie);
 *  - sparse_causal_frames = F > 0: SparseCausalAttention (interpolation/models/attention.py:611-664): batch = (video,
 *    frame) and the keys / values of frame f are [the Sk keys of frame 0 | the Sk keys of frame max(f-1, 0)] of the
 *    same video (2*Sk keys per query, never materialised: the kernel walks two key segments).  sc_halo != 0 (frame
 *    sharding, one video): k / v start with two halo frames [frame 0 of the video | the frame before this rank's first]
 *    followed by the `batch` local frames (lavie_halo_push_p2p); sc_halo = 2 on the rank that owns frame 0. */
int lavie_attention_strided_bf16(const void* q, long long q_seq_stride, long long q_batch_stride, const void* k,
                                 const void* v, long long kv_seq_stride, long long kv_batch_stride, void* o,
                                 long long o_seq_stride, long long o_batch_stride, int batch, int heads, int Sq, int Sk,
                                 int d, int head_pitch, int kv_batch_div, int sparse_causal_frames, int sc_halo,
                                 float scale, lavie_stream_t stream);

/* TemporalAttention._attention (attention.py:634-667): per (b, pixel, head) attention over the F frames, with
 * q scaled before RoPE, rotary embedding on the first 2*rot_pairs dims, + rel-pos bias[heads,F,F].
 * qkv rows = (b, f, pixel); q at column 0, k at k_off, v at v_off (+ h*head_pitch).  rope = [F, rot_pairs, 2]
 * (cos, sin) fp32.  o[(b,f,pixel), h*d + c]. */
int lavie_temporal_attention_bf16(const void* qkv, int ld, int k_off, int v_off, void* o, int ldo, int B, int F,
                                  int HW, int heads, int d, int head_pitch, float scale, const float* rope,
                                  int rot_pairs, const float* bias, lavie_stream_t stream);

/* Small-M linear for the time-embedding path (unet.py:428-434, resnet.py:187): out[m, n] = act_in(x[m,:]) . w[n,:] +
 * bias[n], x/out fp32, w bf16 [N,K]; silu_in applies SiLU to x on load, silu_out to the result. m <= 8. */
int lavie_linear_smallm(const float* x, int M, int K, const void* w, const float* bias, float* out, int N,
                        int silu_in, int silu_out, lavie_stream_t stream);
/* Timesteps(dim, flip_sin_to_cos=True, freq_shift=0): out[b] = [cos(t w_i) | sin(t w_i)], w_i = 10000^(-i/(dim/2)). */
int lavie_timestep_embedding(const float* t, int B, int dim, float* out, lavie_stream_t stream);

/* conv_in (unet.py:454): x fp32 [B, Cin, F, H, W] -> bf16 channels-last [B*F*H*W, Cout]; w fp32 [Cout, Cin, 3, 3]. */
int lavie_conv_in(const float* x, int B, int Cin, int F, int H, int W, const float* w, const float* bias, int Cout,
                  void* out, int ldo, lavie_stream_t stream);
/* The same with the scheduler's scale_model_input folded in (EulerDiscreteScheduler: x / sqrt(sigma^2 + 1),
 * pipeline_videogen.py:667): conv_in(s * x) = (s * W) * x + bias, so no separate elementwise pass over the latents.
 * input_scale is a DEVICE scalar (NULL = 1): a captured CUDA graph of the step serves every sigma of the schedule. */
int lavie_conv_in_scaled(const float* x, const float* input_scale, int B, int Cin, int F, int H, int W, const float* w,
                         const float* bias, int Cout, void* out, int ldo, lavie_stream_t stream);
/* conv_norm_out + SiLU + conv_out (unet.py:504-506): x bf16 [B*F*H*W, C] (raw), scale_shift from
 * lavie_groupnorm_finalize, w fp32 [Cout, 3, 3, C]; writes fp32 [B, Cout, F, H, W]. */
int lavie_conv_out(const void* x, int ldx, const float* scale_shift, int B, int F, int H, int W, int C,
                   const float* w, const float* bias, int Cout, float* out, lavie_stream_t stream);

/* emb[b, :] += table[labels[b], :]: the noise-level class embedding the VSR UNet adds to the time embedding
 * (vsr/models/unet.py:180, 494-507).  emb fp32 [B, dim], table fp32 [rows, dim], labels int64 [B] (clamped to the table). */
int lavie_embedding_add(float* emb, const float* table, const long long* labels, int B, int dim, int rows,
                        lavie_stream_t stream);

/* conv_in (unet.py:454) on the tensor cores: explicit im2col of the fp32 [B, Cin, F, H, W] input (scaled by
 * *input_scale when given) into bf16 rows col[B*F*H*W, kpad], K index = c*9 + kh*3 + kw, zeros beyond 9*Cin and outside
 * the image; the conv is then lavie_gemm_bf16 against the [Cout, kpad] zero-padded filters. */
int lavie_im2col_input_bf16(const float* x, const float* input_scale, int B, int Cin, int F, int H, int W, int kpad,
                            void* col, lavie_stream_t stream);

/* Last step of conv_out when the 3x3 conv itself ran on the tensor cores (lavie_conv3x3_bf16 with the Cout filters
 * zero-padded to a 32-row weight matrix): y bf16 [B*F*H*W, ldy] channels-last -> fp32 [B, Cout, F, H, W], the layout
 * base/models/unet.py:506 returns. */
int lavie_unpack_nchw_f32(const void* y, int ldy, int B, int Cout, int F, int H, int W, float* out,
                          lavie_stream_t stream);

/* F.interpolate(scale_factor=(1,2,2), mode="nearest") of Upsample3D (resnet.py:59-62), channels-last. */
int lavie_upsample_nearest2x(const void* x, int NF, int H, int W, int C, void* y, lavie_stream_t stream);

/* Caller-side step (pipeline_videogen.py:678-683): noise = u + g (t - u); DDIM (eta 0) latent update with the two
 * cumulative alphas; fp32 [n] each. */
int lavie_cfg_ddim_step(const float* noise_uncond, const float* noise_text, float guidance, float alpha_t,
                        float alpha_prev, const float* latents, float* latents_out, long long n,
                        lavie_stream_t stream);

/* Guidance + scheduler.step for every epsilon-prediction scheduler the reference wires up (predict.py:74-96: DDIM,
 * DDPM, EulerDiscrete): eps = u + g (t - u); latents_out = a * latents + b * eps + c_noise * noise (noise may be NULL).
 * The host computes (a, b, c_noise) per step (lavie_b200/pipeline.py; DDIM mirror vsr/diffusion/scheduling_ddim.py:345-394). */
int lavie_cfg_linear_step(const float* noise_uncond, const float* noise_text, float guidance, float a, float b,
                          float c_noise, const float* latents, const float* noise, float* latents_out, long long n,
                          lavie_stream_t stream);
/* forward_with_cfg (base/models/unet.py:514-538, interpolation/models/unet.py:453-474): out0 = out1 = uncond +
 * scale * (cond - uncond); out1 may be NULL. */
int lavie_cfg_combine(const float* cond, const float* uncond, float scale, float* out0, float* out1, long long n,
                      lavie_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Once-per-video encoders / decoders around the denoiser (SURVEY 8f row N4).  The heavy parts reuse lavie_gemm_bf16,
 * lavie_conv3x3_bf16, the GroupNorm and LayerNorm entries above; these are the pieces only they need.
 * ------------------------------------------------------------------------------------------------------------- */
/* CLIPTextEmbeddings.forward (transformers CLIPTextModel, called at base/pipelines/pipeline_videogen.py:337-348):
 * out[row, :] = bf16(token_embedding[ids[row], :] + position_embedding[row % L, :]); tables fp32, ids int64 [rows]. */
int lavie_clip_embed(const long long* ids, const float* token_embedding, const float* position_embedding, int rows, int L,
                     int C, int vocab, void* out, lavie_stream_t stream);
/* CLIPAttention core under the causal mask of CLIPTextTransformer: qkv bf16 [B*L, ld] = (q | k | v) x heads x d,
 * out bf16 [B*L, heads*d]; L <= 128, d = 64 or 128; softmax(scale * q k^T + causal mask) v per (batch item, head). */
int lavie_causal_attention_small(const void* qkv, int ld, int B, int L, int heads, int d, float scale, void* out, int ldo,
                                 lavie_stream_t stream);
/* in place on n bf16 values: kind 0 = quick_gelu x * sigmoid(1.702 x) (CLIP ViT-L text MLP), 1 = erf GELU. */
int lavie_activation_bf16(void* x, long long n, int kind, lavie_stream_t stream);
/* in place: every row of s (bf16 [rows, ld], n <= 4096 columns used) becomes softmax(scale * row) -- the attention
 * probabilities of the VAE decoder's single-head mid-block attention (diffusers AttentionBlock), whose Q K^T and P V
 * products are plain GEMMs. */
int lavie_softmax_rows_bf16(void* s, int ld, long long rows, int n, float scale, lavie_stream_t stream);
/* One-head attention with d = 512, per frame: o = softmax(q k^T) v, the single-head mid-block attention of the
 * x4-upscaler VAE decoder (diffusers AttentionBlock, 512 channels) at any token count S >= 1.  q, k, v, o are bf16
 * row-major [frames * S, 512] views with row strides ld* (multiples of 8, >= 512) and 16-byte aligned bases; frame f
 * occupies rows [f * S, (f + 1) * S).  The 512^-1/2 scale must already be folded into q.  fp32 accumulation,
 * deterministic, writes only the 512 columns of each o row.  frames <= 65535. */
int lavie_attention_wide_bf16(const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, void* o, int ldo,
                              int frames, int S, lavie_stream_t stream);
/* AutoencoderKL.post_quant_conv (1x1, 4 -> 4; mirror vsr/models/autoencoder_kl.py:183) on an fp32 [N, Cin, pixels] map,
 * with decode_latents' 1/0.18215 folded in: out[n, co, p] = bias[co] + sum_ci w[co, ci] * scale * x[n, ci, p]. */
int lavie_pointwise_conv_nchw_f32(const float* x, const float* w, const float* bias, float scale, int N, int Cin, int Cout,
                                  long long pixels, float* out, lavie_stream_t stream);
/* decode_latents post-processing (pipeline_videogen.py:426-428): out[pixel, 0..2] = uint8(clamp((y[pixel, 0..2] / 2 + 0.5)
 * * 255 + 0.5, 0, 255)); y bf16 channels-last rows of >= 4 columns. */
int lavie_image_to_uint8(const void* y, int ld, long long pixels, unsigned char* out, lavie_stream_t stream);
/* VAE encoder conv_in on uint8 video frames (the layout decode_latents returns): frames [N, H, W, 3] channels-last ->
 * col bf16 [N*H*W, kpad], the rows lavie_im2col_input_bf16 writes for Cin = 3 from the normalised image
 * (x / 255 - 0.5) / 0.5 (fp32, IEEE division); the conv is then lavie_gemm_bf16 against the [Cout, kpad] filters. */
int lavie_im2col_frames_bf16(const unsigned char* frames, int N, int H, int W, int kpad, void* col,
                             lavie_stream_t stream);
/* AutoencoderKL.encode's DiagonalGaussianDistribution, sampled and scaled as the interpolation stage does
 * (vae.encode(frames).latent_dist.sample().mul_(0.18215)): moments fp32 [B*F, 8, pixels] (mean | logvar, the quant_conv
 * output), noise fp32 [B*F, 4, pixels] or NULL (then the mode, the mean, is taken) ->
 * out fp32 [B, 4, F, pixels] = scale * (mean + exp(0.5 * clamp(logvar, -30, 20)) * noise), frame n = b * F + f. */
int lavie_posterior_sample_f32(const float* moments, const float* noise, int B, int F, long long pixels, float scale,
                               float* out, lavie_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------
 * fp32-accumulate CHECK MODE (BASELINE north star: noise-prediction rel-L2 <= 1e-3 against the reference fp32 forward).
 * Activations are "split-bf16 triples": a row of C channels is stored as [hi | lo | hi] (3C bf16, hi = bf16(x),
 * lo = bf16(x - hi), ~16 mantissa bits).  With weights repacked by the caller as W' = [Wh | Wh | Wl] along K the
 * product's own tcgen05 mainloop computes Ah Wh + Al Wh + Ah Wl in fp32; lavie_check_gemm / lavie_check_conv3x3 are
 * lavie_gemm_bf16 / lavie_conv3x3_bf16 with k0 / k1 / C counting the TRIPLED widths, the accumulators leaving as fp32
 * through the workspace (>= 4 * M rounded up to 256 * N bytes) and the epilogue (bias, row_bias, residual triple of width
 * N, GEGLU with the exact erf GELU) evaluated in fp32; out is the triple [M, 3 * n_out].  The remaining entry points are
 * the fp32 twins of the normalisation / attention / small kernels reading hi + lo.  Same reference calls as their bf16
 * counterparts above. */
int lavie_check_split3(const float* x, long long rows, int C, void* y_triple, lavie_stream_t stream);
int lavie_check_gemm(const void* a0, int lda0, int k0, const void* a1, int lda1, int k1, const void* w, void* out,
                     int ldo, int M, int N, const lavie_epilogue* ep, void* workspace, size_t workspace_bytes,
                     lavie_stream_t stream);
int lavie_check_conv3x3(const void* x, int NF, int H, int W, int C3, int stride, const void* w, void* out, int ldo,
                        int N, const lavie_epilogue* ep, void* workspace, size_t workspace_bytes, lavie_stream_t stream);
int lavie_check_groupnorm_stats(const void* x0, int ld0, int c0, const void* x1, int ld1, int c1, int samples,
                                int rows_per_sample, int groups, float* partial, lavie_stream_t stream);
int lavie_check_groupnorm_apply(const void* x0, int ld0, int c0, const void* x1, int ld1, int c1, int samples,
                                int rows_per_sample, const float* scale_shift, int silu, void* y, int ldy,
                                lavie_stream_t stream);
int lavie_check_layernorm(const void* x, int ldx, const float* gamma, const float* beta, float eps, void* y, int ldy,
                          int rows, int C, lavie_stream_t stream);
/* One fp32 attention core for every attention of both models: strides as lavie_attention_strided_bf16, *_lo_offset =
 * column distance from a hi block to its lo block (o_lo_offset = heads * d), optional q pre-scale + rotary table
 * [S, rot_pairs, 2] + bias [heads, Sq, Sk] (the base model's temporal attention), optional sparse-causal key segments. */
int lavie_check_attention(const void* q, long long q_seq_stride, long long q_batch_stride, int q_lo_offset,
                          const void* k, const void* v, long long kv_seq_stride, long long kv_batch_stride,
                          int kv_lo_offset, void* o, long long o_seq_stride, long long o_batch_stride, int o_lo_offset,
                          int batch, int heads, int Sq, int Sk, int d, int head_pitch, int kv_batch_div,
                          int sparse_causal_frames, float scale, const float* rope, int rot_pairs, const float* bias,
                          lavie_stream_t stream);
int lavie_check_linear_smallm(const float* x, int M, int K, const float* w_fp32, const float* bias, float* out, int N,
                              int silu_in, int silu_out, lavie_stream_t stream);
int lavie_check_conv_in(const float* x, const float* input_scale, int B, int Cin, int F, int H, int W, const float* w,
                        const float* bias, int Cout, void* out_triple, int ldo, lavie_stream_t stream);
int lavie_check_conv_out(const void* x_triple, int ldx, const float* scale_shift, int B, int F, int H, int W, int C,
                         const float* w, const float* bias, int Cout, float* out, lavie_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* LAVIE_B200_H_ */
