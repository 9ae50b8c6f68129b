// Small kernels of the once-per-video encoders / decoders around the denoiser (SURVEY 8f row N4):
//   * CLIP text encoder (transformers CLIPTextModel, called at base/pipelines/pipeline_videogen.py:337-348, 395-406):
//     token + position embedding, causal self-attention over <= 128 tokens, quick-GELU / GELU activation;
//   * VAE decoder (diffusers AutoencoderKL.decode, called at pipeline_videogen.py:422-429): row softmax of the single-head
//     2560 x 2560 mid-block attention (its Q K^T and P V products run on the tcgen05 GEMM), image post-processing.
// Everything heavy (projections, MLPs, 3x3 convs, GroupNorm, LayerNorm) reuses the denoiser's kernels.
#include "common.cuh"

namespace {

bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// out[row, :] = bf16(tok[ids[row], :] + pos[row % L, :])     (CLIPTextEmbeddings.forward)
__global__ void __launch_bounds__(256)
clip_embed_kernel(const long long* __restrict__ ids, const float* __restrict__ tok, const float* __restrict__ pos, int rows,
                  int L, int C, int vocab, __nv_bfloat16* __restrict__ out) {
  pdl_prologue();
  const int nvec = C >> 2;
  const long long total = static_cast<long long>(rows) * nvec;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int row = static_cast<int>(i / nvec), v = static_cast<int>(i % nvec);
    long long id = ids[row];
    id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
    const float4 a = __ldg(reinterpret_cast<const float4*>(tok + id * C) + v);
    const float4 b = __ldg(reinterpret_cast<const float4*>(pos + static_cast<size_t>(row % L) * C) + v);
    *reinterpret_cast<uint2*>(out + static_cast<size_t>(row) * C + v * 4) =
        make_uint2(pack_bf16(a.x + b.x, a.y + b.y), pack_bf16(a.z + b.z, a.w + b.w));
  }
}

// Causal self-attention over a short sequence (CLIPAttention with the causal mask of CLIPTextTransformer): one block per
// (batch item, head); K and V of the head live in shared memory as fp32; a warp owns a query row at a time: lanes split
// the keys for the scores and the softmax, then the head dimensions for P V.
template <int D>
__global__ void __launch_bounds__(128)
causal_attention_small_kernel(const __nv_bfloat16* __restrict__ qkv, int ld, int L, int heads, float scale,
                              __nv_bfloat16* __restrict__ out, int ldo) {
  pdl_prologue();
  extern __shared__ float sm[];
  float* sk = sm;                          // [L][D + 1]  (padded: lanes read different keys, same dimension)
  float* sv = sk + L * (D + 1);            // [L][D]
  float* sp = sv + L * D;                  // [4 warps][L] probabilities of the row in flight
  float* sq = sp + 4 * L;                  // [4 warps][D]
  const int b = blockIdx.x / heads, h = blockIdx.x % heads;
  const int hd = heads * D;
  const __nv_bfloat16* base = qkv + static_cast<size_t>(b) * L * ld + h * D;
  for (int i = threadIdx.x; i < L * D; i += blockDim.x) {
    const int j = i / D, c = i % D;
    sk[j * (D + 1) + c] = __bfloat162float(base[static_cast<size_t>(j) * ld + hd + c]);
    sv[j * D + c] = __bfloat162float(base[static_cast<size_t>(j) * ld + 2 * hd + c]);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* myp = sp + warp * L;
  float* myq = sq + warp * D;
  for (int i = warp; i < L; i += 4) {
    for (int c = lane; c < D; c += 32) myq[c] = __bfloat162float(base[static_cast<size_t>(i) * ld + c]) * scale;
    __syncwarp();
    float mx = -INFINITY;
    for (int j = lane; j <= i; j += 32) {
      float s = 0.f;
#pragma unroll 8
      for (int c = 0; c < D; ++c) s = fmaf(myq[c], sk[j * (D + 1) + c], s);
      myp[j] = s;
      mx = fmaxf(mx, s);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j <= i; j += 32) {
      const float p = __expf(myp[j] - mx);
      myp[j] = p;
      sum += p;
    }
    sum = warp_sum(sum);
    __syncwarp();
    const float inv = 1.0f / sum;
    for (int c = lane; c < D; c += 32) {
      float o = 0.f;
      for (int j = 0; j <= i; ++j) o = fmaf(myp[j], sv[j * D + c], o);
      out[(static_cast<size_t>(b) * L + i) * ldo + h * D + c] = __float2bfloat16_rn(o * inv);
    }
    __syncwarp();
  }
}

// in-place activation on a bf16 matrix: kind 0 = quick_gelu x * sigmoid(1.702 x) (CLIP ViT-L), 1 = erf GELU (OpenCLIP ViT-H)
__global__ void __launch_bounds__(256)
activation_kernel(__nv_bfloat16* __restrict__ x, long long n8, int kind) {
  pdl_prologue();
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n8;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    uint4 v = reinterpret_cast<uint4*>(x)[i];
    uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float2 f = unpack_bf16(w[e]);
      if (kind == 0) {
        f.x = f.x / (1.0f + __expf(-1.702f * f.x));
        f.y = f.y / (1.0f + __expf(-1.702f * f.y));
      } else {
        f.x = 0.5f * f.x * (1.0f + erff(f.x * 0.70710678118654752440f));
        f.y = 0.5f * f.y * (1.0f + erff(f.y * 0.70710678118654752440f));
      }
      w[e] = pack_bf16(f.x, f.y);
    }
    reinterpret_cast<uint4*>(x)[i] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// Row softmax of a bf16 score matrix, in place: p = softmax(scale * s) over n columns; one warp per row, the row is read
// once into registers (n <= 32 * 8 * PER_LANE), statistics in fp32.
template <int VECS>                       // 16-byte vectors per lane
__global__ void __launch_bounds__(256)
softmax_rows_kernel(__nv_bfloat16* __restrict__ s, int ld, long long rows, int n, float scale) {
  pdl_prologue();
  const int lane = threadIdx.x & 31;
  const long long warps_total = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
  const float k = scale * 1.4426950408889634f;
  for (long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); row < rows;
       row += warps_total) {
    __nv_bfloat16* p = s + row * ld;
    float f[VECS][8];
    float mx = -INFINITY;
#pragma unroll
    for (int u = 0; u < VECS; ++u) {
      const int c = (u * 32 + lane) * 8;
      if (c < n) {
        const uint4 v = *reinterpret_cast<const uint4*>(p + c);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 t = unpack_bf16(w[e]);
          f[u][2 * e] = t.x;
          f[u][2 * e + 1] = t.y;
          mx = fmaxf(mx, fmaxf(t.x, t.y));
        }
      }
    }
    mx = warp_max(mx);
    float sum = 0.f;
#pragma unroll
    for (int u = 0; u < VECS; ++u) {
      const int c = (u * 32 + lane) * 8;
      if (c < n) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          f[u][e] = exp2f((f[u][e] - mx) * k);
          sum += f[u][e];
        }
      }
    }
    sum = warp_sum(sum);
    const float inv = 1.0f / sum;
#pragma unroll
    for (int u = 0; u < VECS; ++u) {
      const int c = (u * 32 + lane) * 8;
      if (c < n)
        *reinterpret_cast<uint4*>(p + c) =
            make_uint4(pack_bf16(f[u][0] * inv, f[u][1] * inv), pack_bf16(f[u][2] * inv, f[u][3] * inv),
                       pack_bf16(f[u][4] * inv, f[u][5] * inv), pack_bf16(f[u][6] * inv, f[u][7] * inv));
    }
  }
}

// decode_latents post-processing (pipeline_videogen.py:426-428): uint8 = clamp((x / 2 + 0.5) * 255 + 0.5, 0, 255),
// channels-last bf16 rows [pixels, ld] (first 3 columns = RGB) -> uint8 [pixels, 3] (the layout the pipeline returns)
__global__ void __launch_bounds__(256)
image_to_uint8_kernel(const __nv_bfloat16* __restrict__ y, int ld, long long pixels, unsigned char* __restrict__ out) {
  pdl_prologue();
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < pixels;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const uint2 v = __ldg(reinterpret_cast<const uint2*>(y + i * ld));
    const float2 a = unpack_bf16(v.x), b = unpack_bf16(v.y);
    const float c[3] = {a.x, a.y, b.x};
#pragma unroll
    for (int e = 0; e < 3; ++e) {
      const float u = fminf(fmaxf((c[e] * 0.5f + 0.5f) * 255.0f + 0.5f, 0.0f), 255.0f);
      out[i * 3 + e] = static_cast<unsigned char>(u);          // truncation, like torch's .to(torch.uint8)
    }
  }
}

// 1x1 conv on an fp32 NCHW map with a handful of channels (AutoencoderKL.post_quant_conv, 4 -> 4), input scaled first:
// out[n, co, p] = bias[co] + sum_ci w[co, ci] * (scale * x[n, ci, p])
__global__ void __launch_bounds__(256)
pointwise_conv_nchw_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                           float scale, int N, int Cin, int Cout, long long pix, float* __restrict__ out) {
  pdl_prologue();
  const long long total = static_cast<long long>(N) * pix;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long n = i / pix, p = i - n * pix;
    for (int co = 0; co < Cout; ++co) {
      float a = bias[co];
      for (int ci = 0; ci < Cin; ++ci) a = fmaf(w[co * Cin + ci], scale * x[(n * Cin + ci) * pix + p], a);
      out[(n * Cout + co) * pix + p] = a;
    }
  }
}

// AutoencoderKL.encode's DiagonalGaussianDistribution and the interpolation stage's scaling
// (interpolation/sample.py: vae.encode(frames).latent_dist.sample().mul_(0.18215)): moments fp32 [N, 8, pix] (mean |
// logvar, as quant_conv leaves them) -> out[b, c, f, p] = scale * (mean + exp(0.5 * clamp(logvar, -30, 20)) * noise)
// for frame n = b * F + f, i.e. the [B, 4, F, h, w] latents the interpolation UNet reads.  No noise: scale * mean.
__global__ void __launch_bounds__(256)
posterior_sample_kernel(const float* __restrict__ moments, const float* __restrict__ noise, int F, long long pix,
                        long long total, float scale, float* __restrict__ out) {
  pdl_prologue();
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long p = i % pix;
    const long long nc = i / pix;                  // n * 4 + c
    const int c = static_cast<int>(nc % 4);
    const long long n = nc / 4;
    const long long b = n / F;
    const int f = static_cast<int>(n - b * F);
    float z = moments[(n * 8 + c) * pix + p];
    if (noise) {
      const float lv = fminf(fmaxf(moments[(n * 8 + 4 + c) * pix + p], -30.0f), 20.0f);
      z = z + expf(0.5f * lv) * noise[i];
    }
    out[((b * 4 + c) * F + f) * pix + p] = scale * z;
  }
}

int grid_for_n(long long total, int threads) {
  long long b = (total + threads - 1) / threads;
  const long long cap = static_cast<long long>(lavie_num_sms()) * 16;
  return static_cast<int>(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace

extern "C" int lavie_clip_embed(const long long* ids, const float* token_embedding, const float* position_embedding,
                                int rows, int L, int C, int vocab, void* out, cudaStream_t stream) {
  LAVIE_REQUIRE(ids && token_embedding && position_embedding && out && rows > 0 && L > 0 && vocab > 0, LAVIE_ERR_SHAPE,
                "clip_embed: bad arguments");
  LAVIE_REQUIRE(C % 8 == 0 && al16(token_embedding) && al16(position_embedding) && al16(out), LAVIE_ERR_ALIGN,
                "clip_embed: C %% 8 == 0 and 16-byte aligned tables");
  launch_pdl(clip_embed_kernel, grid_for_n(static_cast<long long>(rows) * (C / 4), 256), 256, 0, stream, ids,
             token_embedding, position_embedding, rows, L, C, vocab, static_cast<__nv_bfloat16*>(out));
  return lavie_check_launch("clip_embed_kernel");
}

extern "C" int lavie_causal_attention_small(const void* qkv, int ld, int B, int L, int heads, int d, float scale, void* out,
                                            int ldo, cudaStream_t stream) {
  LAVIE_REQUIRE(qkv && out && B > 0 && L > 0 && L <= 128 && heads > 0 && (d == 64 || d == 128), LAVIE_ERR_SHAPE,
                "causal_attention_small: L=%d must be <= 128, head dim %d must be 64 or 128", L, d);
  LAVIE_REQUIRE(ld >= 3 * heads * d && ldo >= heads * d, LAVIE_ERR_SHAPE, "causal_attention_small: row strides");
  const size_t smem = (static_cast<size_t>(L) * (2 * d + 1) + 4 * L + 4 * d) * sizeof(float);
  static LavieSmemConfig c64, c128;
  int rc = d == 64 ? lavie_config_smem(causal_attention_small_kernel<64>, static_cast<int>(smem), &c64, "causal_attention<64>")
                   : lavie_config_smem(causal_attention_small_kernel<128>, static_cast<int>(smem), &c128, "causal_attention<128>");
  if (rc) return rc;
  if (d == 64)
    launch_pdl(causal_attention_small_kernel<64>, B * heads, 128, smem, stream, static_cast<const __nv_bfloat16*>(qkv), ld,
               L, heads, scale, static_cast<__nv_bfloat16*>(out), ldo);
  else
    launch_pdl(causal_attention_small_kernel<128>, B * heads, 128, smem, stream, static_cast<const __nv_bfloat16*>(qkv), ld,
               L, heads, scale, static_cast<__nv_bfloat16*>(out), ldo);
  return lavie_check_launch("causal_attention_small_kernel");
}

extern "C" int lavie_activation_bf16(void* x, long long n, int kind, cudaStream_t stream) {
  LAVIE_REQUIRE(x && n > 0 && n % 8 == 0 && al16(x) && (kind == 0 || kind == 1), LAVIE_ERR_SHAPE,
                "activation: n %% 8 == 0, kind 0 (quick_gelu) or 1 (gelu)");
  launch_pdl(activation_kernel, grid_for_n(n / 8, 256), 256, 0, stream, static_cast<__nv_bfloat16*>(x), n / 8, kind);
  return lavie_check_launch("activation_kernel");
}

extern "C" int lavie_softmax_rows_bf16(void* s, int ld, long long rows, int n, float scale, cudaStream_t stream) {
  LAVIE_REQUIRE(s && rows > 0 && n > 0 && n % 8 == 0 && ld % 8 == 0 && ld >= n && al16(s) && n <= 32 * 8 * 16,
                LAVIE_ERR_SHAPE, "softmax_rows: n=%d must be a multiple of 8 and <= 4096", n);
  const int blocks = grid_for_n(rows * 32, 256);
  __nv_bfloat16* p = static_cast<__nv_bfloat16*>(s);
  const int vecs = (n + 255) / 256;
  if (vecs <= 4) launch_pdl(softmax_rows_kernel<4>, blocks, 256, 0, stream, p, ld, rows, n, scale);
  else if (vecs <= 10) launch_pdl(softmax_rows_kernel<10>, blocks, 256, 0, stream, p, ld, rows, n, scale);
  else launch_pdl(softmax_rows_kernel<16>, blocks, 256, 0, stream, p, ld, rows, n, scale);
  return lavie_check_launch("softmax_rows_kernel");
}

extern "C" int lavie_image_to_uint8(const void* y, int ld, long long pixels, unsigned char* out, cudaStream_t stream) {
  LAVIE_REQUIRE(y && out && pixels > 0 && ld >= 4 && ld % 4 == 0 && (reinterpret_cast<uintptr_t>(y) & 7) == 0,
                LAVIE_ERR_SHAPE, "image_to_uint8: rows of >= 4 bf16, 8-byte aligned");
  launch_pdl(image_to_uint8_kernel, grid_for_n(pixels, 256), 256, 0, stream, static_cast<const __nv_bfloat16*>(y), ld,
             pixels, out);
  return lavie_check_launch("image_to_uint8_kernel");
}

extern "C" int lavie_pointwise_conv_nchw_f32(const float* x, const float* w, const float* bias, float scale, int N, int Cin,
                                             int Cout, long long pixels, float* out, cudaStream_t stream) {
  LAVIE_REQUIRE(x && w && bias && out && N > 0 && Cin > 0 && Cin <= 16 && Cout > 0 && Cout <= 16 && pixels > 0,
                LAVIE_ERR_SHAPE, "pointwise_conv_nchw: up to 16 channels");
  launch_pdl(pointwise_conv_nchw_kernel, grid_for_n(static_cast<long long>(N) * pixels, 256), 256, 0, stream, x, w, bias,
             scale, N, Cin, Cout, pixels, out);
  return lavie_check_launch("pointwise_conv_nchw_kernel");
}

extern "C" int lavie_posterior_sample_f32(const float* moments, const float* noise, int B, int F, long long pixels,
                                          float scale, float* out, cudaStream_t stream) {
  LAVIE_REQUIRE(moments && out && B > 0 && F > 0 && pixels > 0, LAVIE_ERR_SHAPE, "posterior_sample: bad arguments");
  const long long total = static_cast<long long>(B) * F * 4 * pixels;
  launch_pdl(posterior_sample_kernel, grid_for_n(total, 256), 256, 0, stream, moments, noise, F, pixels, total, scale,
             out);
  return lavie_check_launch("posterior_sample_kernel");
}
