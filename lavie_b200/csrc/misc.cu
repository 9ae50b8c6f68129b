// Small / bandwidth-bound helpers of the denoiser step: time-embedding path, first and last convolution,
// patch matrix for strided convs, nearest upsampling, and the caller-side CFG + DDIM update.
#include "common.cuh"

namespace {

bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// ---------------------------------------------------------------------------------------------------------
// Timesteps(dim, flip_sin_to_cos=True, freq_shift=0): [cos | sin]   (unet.py:153,428; diffusers 0.16)
// ---------------------------------------------------------------------------------------------------------
__global__ void timestep_embedding_kernel(const float* __restrict__ t, int B, int dim, float* __restrict__ out) {
  pdl_prologue();
  const int half = dim >> 1;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * half) return;
  const int b = i / half, k = i - b * half;
  const float freq = expf(-logf(10000.0f) * static_cast<float>(k) / static_cast<float>(half));
  const float arg = t[b] * freq;
  out[b * dim + k] = cosf(arg);
  out[b * dim + half + k] = sinf(arg);
}

// ---------------------------------------------------------------------------------------------------------
// out[m, n] = act_out( sum_k act_in(x[m,k]) * w[n,k] + bias[n] ),  m <= 8.  One warp per output feature.
// ---------------------------------------------------------------------------------------------------------
template <int MAXM>
__global__ void __launch_bounds__(256)
linear_smallm_kernel(const float* __restrict__ x, int M, int K, const __nv_bfloat16* __restrict__ w,
                     const float* __restrict__ bias, float* __restrict__ out, int N, int silu_in, int silu_out) {
  pdl_prologue();
  const int n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (n >= N) return;
  float acc[MAXM];
#pragma unroll
  for (int m = 0; m < MAXM; ++m) acc[m] = 0.f;
  const __nv_bfloat16* wr = w + static_cast<size_t>(n) * K;
  for (int k = lane * 8; k < K; k += 256) {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(wr + k));
    const uint32_t ww[4] = {u.x, u.y, u.z, u.w};
    float wf[8];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = unpack_bf16(ww[e]);
      wf[2 * e] = f.x;
      wf[2 * e + 1] = f.y;
    }
#pragma unroll
    for (int m = 0; m < MAXM; ++m) {
      if (m < M) {
        const float4 a = *reinterpret_cast<const float4*>(x + static_cast<size_t>(m) * K + k);
        const float4 b = *reinterpret_cast<const float4*>(x + static_cast<size_t>(m) * K + k + 4);
        float xv[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float v = silu_in ? silu_f(xv[e]) : xv[e];
          acc[m] += v * wf[e];
        }
      }
    }
  }
#pragma unroll
  for (int m = 0; m < MAXM; ++m) {
    const float s = warp_sum(acc[m]);
    if (lane == 0 && m < M) {
      float r = s + (bias ? bias[n] : 0.f);
      if (silu_out) r = silu_f(r);
      out[static_cast<size_t>(m) * N + n] = r;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// conv_in: fp32 [B,Cin,F,H,W] -> bf16 channels-last [B*F*H*W, Cout].
// thread = (strip of 4 pixels along x, 8 output channels): every weight vector fetched from shared memory feeds
// 4 pixels (32 FMAs per 2 LDS.128), the 6 input values of a filter row are loaded once per (channel, dy).
// ---------------------------------------------------------------------------------------------------------
constexpr int CIN_P = 4;
__global__ void __launch_bounds__(256)
conv_in_kernel(const float* __restrict__ x, int B, int Cin, int F, int H, int W, const float* __restrict__ w,
               const float* __restrict__ bias, int Cout, __nv_bfloat16* __restrict__ out, int ldo,
               const float* __restrict__ input_scale_ptr, int triple) {
  pdl_prologue();
  const float input_scale = input_scale_ptr ? __ldg(input_scale_ptr) : 1.0f;
  extern __shared__ float s_w[];     // transposed to [Cin*9][Cout]: a warp reads 1 KiB contiguous per tap
  const int kk = Cin * 9;
  for (int i = threadIdx.x; i < Cout * kk; i += blockDim.x) {
    const int o = i / kk, r = i - o * kk;
    s_w[r * Cout + o] = w[i] * input_scale;      // conv(s * x) = (s * W) * x: the scheduler's scale_model_input, folded
  }
  __syncthreads();
  const int groups = Cout >> 3;
  const int strips = (W + CIN_P - 1) / CIN_P;
  const long long total = static_cast<long long>(B) * F * H * strips * groups;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int g = static_cast<int>(i % groups);
    const long long sidx = i / groups;
    const int xs = static_cast<int>(sidx % strips) * CIN_P;
    const int yh = static_cast<int>((sidx / strips) % H);
    const int f = static_cast<int>((sidx / (static_cast<long long>(strips) * H)) % F);
    const int b = static_cast<int>(sidx / (static_cast<long long>(strips) * H * F));
    float acc[CIN_P][8];
    {
      const float4 b0 = *reinterpret_cast<const float4*>(bias + g * 8);
      const float4 b1 = *reinterpret_cast<const float4*>(bias + g * 8 + 4);
#pragma unroll
      for (int pp = 0; pp < CIN_P; ++pp) {
        acc[pp][0] = b0.x; acc[pp][1] = b0.y; acc[pp][2] = b0.z; acc[pp][3] = b0.w;
        acc[pp][4] = b1.x; acc[pp][5] = b1.y; acc[pp][6] = b1.z; acc[pp][7] = b1.w;
      }
    }
    for (int c = 0; c < Cin; ++c) {
      const float* plane = x + ((static_cast<size_t>(b) * Cin + c) * F + f) * H * W;
#pragma unroll
      for (int dy = 0; dy < 3; ++dy) {
        const int yy = yh + dy - 1;
        if (yy < 0 || yy >= H) continue;
        float xv[CIN_P + 2];
#pragma unroll
        for (int j = 0; j < CIN_P + 2; ++j) {
          const int xx = xs - 1 + j;
          xv[j] = (xx >= 0 && xx < W) ? __ldg(plane + yy * W + xx) : 0.f;
        }
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
          const float4* wp = reinterpret_cast<const float4*>(s_w + (c * 9 + dy * 3 + dx) * Cout + g * 8);
          const float4 w0 = wp[0], w1 = wp[1];
#pragma unroll
          for (int pp = 0; pp < CIN_P; ++pp) {
            const float v = xv[pp + dx];
            acc[pp][0] += v * w0.x; acc[pp][1] += v * w0.y; acc[pp][2] += v * w0.z; acc[pp][3] += v * w0.w;
            acc[pp][4] += v * w1.x; acc[pp][5] += v * w1.y; acc[pp][6] += v * w1.z; acc[pp][7] += v * w1.w;
          }
        }
      }
    }
    const size_t pix0 = ((static_cast<size_t>(b) * F + f) * H + yh) * W + xs;
#pragma unroll
    for (int pp = 0; pp < CIN_P; ++pp) {
      if (xs + pp < W) {
        uint4 o;
        o.x = pack_bf16(acc[pp][0], acc[pp][1]);
        o.y = pack_bf16(acc[pp][2], acc[pp][3]);
        o.z = pack_bf16(acc[pp][4], acc[pp][5]);
        o.w = pack_bf16(acc[pp][6], acc[pp][7]);
        *reinterpret_cast<uint4*>(out + (pix0 + pp) * ldo + g * 8) = o;
        if (triple) {      // check mode: [hi | lo | hi]
          const float2 h0 = unpack_bf16(o.x), h1 = unpack_bf16(o.y), h2 = unpack_bf16(o.z), h3 = unpack_bf16(o.w);
          uint4 l;
          l.x = pack_bf16(acc[pp][0] - h0.x, acc[pp][1] - h0.y);
          l.y = pack_bf16(acc[pp][2] - h1.x, acc[pp][3] - h1.y);
          l.z = pack_bf16(acc[pp][4] - h2.x, acc[pp][5] - h2.y);
          l.w = pack_bf16(acc[pp][6] - h3.x, acc[pp][7] - h3.y);
          *reinterpret_cast<uint4*>(out + (pix0 + pp) * ldo + Cout + g * 8) = l;
          *reinterpret_cast<uint4*>(out + (pix0 + pp) * ldo + 2 * Cout + g * 8) = o;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// conv_norm_out -> SiLU -> conv_out, fused.  One warp per strip of 4 output pixels; lane l owns the channel pairs
// {l, l+32, ...} (coalesced 128-byte reads of the activation rows).  For each pair and filter row the 6 input pixels
// are normalised + activated once and feed 3 taps x 4 pixels x COUT outputs; every weight pair read from shared
// memory feeds 8 FMAs.  Zero padding applies to the ACTIVATED map, so out-of-image taps contribute 0.
// ---------------------------------------------------------------------------------------------------------
constexpr int COUT_P = 4;
template <int COUT, bool TRIPLE>      // TRIPLE: check mode, x = hi + lo of a split-bf16 triple (lo lo_off columns further)
__global__ void __launch_bounds__(256)
conv_out_kernel(const __nv_bfloat16* __restrict__ x, int ldx, const float* __restrict__ scale_shift, int B, int F,
                int H, int W, int C, const float* __restrict__ w, const float* __restrict__ bias,
                float* __restrict__ out, int lo_off) {
  pdl_prologue();
  extern __shared__ float s_w[];     // [9][COUT][C]   (source layout [COUT][9][C])
  for (int i = threadIdx.x; i < COUT * 9 * C; i += blockDim.x) {
    const int c = i % C, ot = i / C;
    const int o = ot / 9, t = ot - o * 9;
    s_w[(t * COUT + o) * C + c] = w[i];
  }
  __syncthreads();
  const float2* s_w2 = reinterpret_cast<const float2*>(s_w);
  const int lane = threadIdx.x & 31;
  const int npairs = C >> 1;
  const int strips = (W + COUT_P - 1) / COUT_P;
  const long long total = static_cast<long long>(B) * F * H * strips;
  const long long warps_total = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
  for (long long task = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); task < total;
       task += warps_total) {
    const int xs = static_cast<int>(task % strips) * COUT_P;
    const int yh = static_cast<int>((task / strips) % H);
    const long long bf = task / (static_cast<long long>(strips) * H);
    const int b = static_cast<int>(bf / F);
    const int f = static_cast<int>(bf % F);
    float acc[COUT_P][COUT];
#pragma unroll
    for (int pp = 0; pp < COUT_P; ++pp)
#pragma unroll
      for (int o = 0; o < COUT; ++o) acc[pp][o] = 0.f;
    for (int p = lane; p < npairs; p += 32) {
      const float4 ss = __ldg(reinterpret_cast<const float4*>(scale_shift + (static_cast<size_t>(b) * C + 2 * p) * 2));
#pragma unroll
      for (int dy = 0; dy < 3; ++dy) {
        const int yy = yh + dy - 1;
        const bool row_ok = yy >= 0 && yy < H;       // out-of-image rows contribute zeros (no divergent control flow)
        // first tap column of the strip (may be x = -1: only dereferenced when inside the image)
        const __nv_bfloat16* xp = x + (((static_cast<long long>(bf) * H + yy) * W) + xs - 1) * ldx + 2 * p;
        float a0[COUT_P + 2], a1[COUT_P + 2];
#pragma unroll
        for (int i = 0; i < COUT_P + 2; ++i) {
          const int xx = xs - 1 + i;
          if (row_ok && xx >= 0 && xx < W) {
            float2 t2 = unpack_bf16(__ldg(reinterpret_cast<const uint32_t*>(xp + i * ldx)));
            if (TRIPLE) {            // check mode: x = hi + lo of the split-bf16 triple
              const float2 tl = unpack_bf16(__ldg(reinterpret_cast<const uint32_t*>(xp + i * ldx + lo_off)));
              t2.x += tl.x;
              t2.y += tl.y;
            }
            a0[i] = silu_f(t2.x * ss.x + ss.y);
            a1[i] = silu_f(t2.y * ss.z + ss.w);
          } else {
            a0[i] = 0.f;
            a1[i] = 0.f;
          }
        }
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
#pragma unroll
          for (int o = 0; o < COUT; ++o) {
            const float2 wv = s_w2[((dy * 3 + dx) * COUT + o) * npairs + p];
#pragma unroll
            for (int pp = 0; pp < COUT_P; ++pp) acc[pp][o] = fmaf(a1[pp + dx], wv.y, fmaf(a0[pp + dx], wv.x, acc[pp][o]));
          }
        }
      }
    }
#pragma unroll
    for (int pp = 0; pp < COUT_P; ++pp) {
#pragma unroll
      for (int o = 0; o < COUT; ++o) {
        const float s = warp_sum(acc[pp][o]);
        if (lane == 0 && xs + pp < W)
          out[(((static_cast<size_t>(b) * COUT + o) * F + f) * H + yh) * W + xs + pp] = s + bias[o];
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// im2col for 3x3 pad-1 convs with stride (Downsample3D) or geometries the TMA path does not take.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
im2col3x3_kernel(const __nv_bfloat16* __restrict__ x, int NF, int H, int W, int C, int stride, int Ho, int Wo,
                 __nv_bfloat16* __restrict__ col) {
  pdl_prologue();
  const int nvec = C >> 3;
  const long long total = static_cast<long long>(NF) * Ho * Wo * 9 * nvec;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int v = static_cast<int>(i % nvec);
    const int t = static_cast<int>((i / nvec) % 9);
    const long long opix = i / (9LL * nvec);
    const int xo = static_cast<int>(opix % Wo);
    const int yo = static_cast<int>((opix / Wo) % Ho);
    const int n = static_cast<int>(opix / (static_cast<long long>(Wo) * Ho));
    const int yy = yo * stride + t / 3 - 1, xx = xo * stride + t % 3 - 1;
    uint4 val = make_uint4(0, 0, 0, 0);
    if (yy >= 0 && yy < H && xx >= 0 && xx < W)
      val = __ldg(reinterpret_cast<const uint4*>(x + ((static_cast<size_t>(n) * H + yy) * W + xx) * C + v * 8));
    *reinterpret_cast<uint4*>(col + (static_cast<size_t>(opix) * 9 + t) * C + v * 8) = val;
  }
}

__global__ void __launch_bounds__(256)
upsample2x_kernel(const __nv_bfloat16* __restrict__ x, int NF, int H, int W, int C, __nv_bfloat16* __restrict__ y) {
  pdl_prologue();
  const int nvec = C >> 3;
  const int Ho = 2 * H, Wo = 2 * W;
  const long long total = static_cast<long long>(NF) * Ho * Wo * nvec;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int v = static_cast<int>(i % nvec);
    const long long opix = i / nvec;
    const int xo = static_cast<int>(opix % Wo);
    const int yo = static_cast<int>((opix / Wo) % Ho);
    const int n = static_cast<int>(opix / (static_cast<long long>(Wo) * Ho));
    const uint4 val =
        __ldg(reinterpret_cast<const uint4*>(x + ((static_cast<size_t>(n) * H + (yo >> 1)) * W + (xo >> 1)) * C + v * 8));
    *reinterpret_cast<uint4*>(y + static_cast<size_t>(opix) * C + v * 8) = val;
  }
}

// conv_out on the tensor cores: the 3x3 conv runs as an implicit GEMM with the Cout = 4 filters zero-padded to a
// 32-column weight tile (gemm.cu, conv mode); this kernel picks the real channels out of the channels-last bf16 rows and
// writes the reference's fp32 [B, Cout, F, H, W] layout (base/models/unet.py:506).  One thread per pixel: 8-byte read,
// Cout coalesced 4-byte writes.
__global__ void __launch_bounds__(256)
unpack_nchw_kernel(const __nv_bfloat16* __restrict__ y, int ldy, int B, int Cout, long long pix_per_sample,
                   float* __restrict__ out) {
  pdl_prologue();
  const long long total = static_cast<long long>(B) * pix_per_sample;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long b = i / pix_per_sample, pix = i - b * pix_per_sample;
    const __nv_bfloat16* row = y + i * ldy;
    for (int c0 = 0; c0 < Cout; c0 += 4) {
      const uint2 v = __ldg(reinterpret_cast<const uint2*>(row + c0));
      const float2 v0 = unpack_bf16(v.x), v1 = unpack_bf16(v.y);
      const float f[4] = {v0.x, v0.y, v1.x, v1.y};
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (c0 + e < Cout) out[(b * Cout + c0 + e) * pix_per_sample + pix] = f[e];
    }
  }
}

// emb[b, :] += table[labels[b], :]   (the VSR UNet's noise-level class embedding, vsr/models/unet.py:494-507)
__global__ void embedding_add_kernel(float* __restrict__ emb, const float* __restrict__ table,
                                     const long long* __restrict__ labels, int B, int dim, int rows) {
  pdl_prologue();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * dim) return;
  const int b = i / dim, c = i - b * dim;
  long long l = labels[b];
  l = l < 0 ? 0 : (l >= rows ? rows - 1 : l);         // the reference raises on out-of-range levels; clamp, never fault
  emb[i] += table[l * dim + c];
}

// conv_in on the tensor cores: explicit im2col of the few-channel fp32 input (4 latent channels; 8 with the interpolation
// model's conditioning, 7 with the VSR model's low-resolution frames) into bf16 rows [pixels, Kpad], K index =
// c * 9 + kh * 3 + kw, zero beyond 9 * Cin and outside the image; the conv itself is then one GEMM with N = Cout.
// (The CUDA-core conv_in kernel costs 1.3 ns per pixel: 0.12 ms for the base model, 6.9 ms at the VSR model's 320x512.)
__global__ void __launch_bounds__(256)
im2col_input_kernel(const float* __restrict__ x, const float* __restrict__ input_scale, int B, int Cin, int F, int H, int W,
                    int kpad, __nv_bfloat16* __restrict__ col) {
  pdl_prologue();
  const float sc = input_scale ? __ldg(input_scale) : 1.0f;
  const int nvec = kpad >> 3;
  const long long total = static_cast<long long>(B) * F * H * W * nvec;
  const long long plane = static_cast<long long>(H) * W;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int v = static_cast<int>(i % nvec);
    const long long pix = i / nvec;
    const int xo = static_cast<int>(pix % W);
    const int yo = static_cast<int>((pix / W) % H);
    const long long bf = pix / plane;
    const int f = static_cast<int>(bf % F);
    const long long b = bf / F;
    float e[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = v * 8 + j;
      const int c = k / 9, tap = k - c * 9;
      const int yy = yo + tap / 3 - 1, xx = xo + tap % 3 - 1;
      e[j] = 0.f;
      if (c < Cin && yy >= 0 && yy < H && xx >= 0 && xx < W)
        e[j] = sc * __ldg(x + ((b * Cin + c) * F + f) * plane + static_cast<long long>(yy) * W + xx);
    }
    *reinterpret_cast<uint4*>(col + pix * kpad + v * 8) =
        make_uint4(pack_bf16(e[0], e[1]), pack_bf16(e[2], e[3]), pack_bf16(e[4], e[5]), pack_bf16(e[6], e[7]));
  }
}

// The VAE encoder's conv_in on uint8 video frames (the layout decode_latents returns): channels-last [N, H, W, 3] ->
// the same bf16 rows im2col_input_kernel writes for Cin = 3, with the interpolation stage's normalisation
// (x / 255 - 0.5) / 0.5 evaluated in fp32 exactly as written (IEEE division: the library is built without fast-math).
__global__ void __launch_bounds__(256)
im2col_frames_kernel(const unsigned char* __restrict__ frames, int N, int H, int W, int kpad,
                     __nv_bfloat16* __restrict__ col) {
  pdl_prologue();
  const int nvec = kpad >> 3;
  const long long total = static_cast<long long>(N) * H * W * nvec;
  const long long plane = static_cast<long long>(H) * W;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int v = static_cast<int>(i % nvec);
    const long long pix = i / nvec;
    const int xo = static_cast<int>(pix % W);
    const int yo = static_cast<int>((pix / W) % H);
    const long long n = pix / plane;
    float e[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = v * 8 + j;
      const int c = k / 9, tap = k - c * 9;
      const int yy = yo + tap / 3 - 1, xx = xo + tap % 3 - 1;
      e[j] = 0.f;
      if (c < 3 && yy >= 0 && yy < H && xx >= 0 && xx < W) {
        const float u = static_cast<float>(__ldg(frames + ((n * H + yy) * W + xx) * 3 + c));
        e[j] = (u / 255.0f - 0.5f) / 0.5f;
      }
    }
    *reinterpret_cast<uint4*>(col + pix * kpad + v * 8) =
        make_uint4(pack_bf16(e[0], e[1]), pack_bf16(e[2], e[3]), pack_bf16(e[4], e[5]), pack_bf16(e[6], e[7]));
  }
}

__global__ void cfg_ddim_kernel(const float* __restrict__ nu, const float* __restrict__ nt, float g, float sa_t,
                                float s1a_t, float sa_p, float s1a_p, const float* __restrict__ lat,
                                float* __restrict__ out, long long n) {
  pdl_prologue();
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float eps = nu[i] + g * (nt[i] - nu[i]);
    const float x0 = (lat[i] - s1a_t * eps) / sa_t;
    out[i] = sa_p * x0 + s1a_p * eps;
  }
}

// eps = u + g (c - u); out = a * latents + b * eps (+ c_noise * noise): every epsilon-prediction scheduler update of
// the reference pipelines is this linear form (DDIM eta 0, DDPM ancestral, EulerDiscrete), coefficients from the host.
__global__ void cfg_linear_step_kernel(const float* __restrict__ nu, const float* __restrict__ nt, float g, float a,
                                       float b, float c_noise, const float* __restrict__ lat,
                                       const float* __restrict__ noise, float* __restrict__ out, long long n) {
  pdl_prologue();
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float eps = nu[i] + g * (nt[i] - nu[i]);
    float v = fmaf(a, lat[i], b * eps);
    if (noise) v = fmaf(c_noise, noise[i], v);
    out[i] = v;
  }
}

// forward_with_cfg (base/models/unet.py:514-538): half_eps = uncond + s (cond - uncond), returned for both halves
__global__ void cfg_combine_kernel(const float* __restrict__ cond, const float* __restrict__ uncond, float s,
                                   float* __restrict__ out0, float* __restrict__ out1, long long n) {
  pdl_prologue();
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float u = uncond[i];
    const float v = u + s * (cond[i] - u);
    out0[i] = v;
    if (out1) out1[i] = v;
  }
}

int grid_for(long long total, int threads) {
  long long b = (total + threads - 1) / threads;
  if (b > 148LL * 32) b = 148LL * 32;
  if (b < 1) b = 1;
  return static_cast<int>(b);
}

}  // namespace

extern "C" int lavie_timestep_embedding(const float* t, int B, int dim, float* out, cudaStream_t stream) {
  LAVIE_REQUIRE(B > 0 && dim > 0 && dim % 2 == 0, LAVIE_ERR_SHAPE, "timestep_embedding: dim must be even");
  const int total = B * (dim / 2);
  launch_pdl(timestep_embedding_kernel, (total + 127) / 128, 128, 0, stream, t, B, dim, out);
  return lavie_check_launch("timestep_embedding_kernel");
}

extern "C" int lavie_linear_smallm(const float* x, int M, int K, const void* w, const float* bias, float* out, int N,
                                   int silu_in, int silu_out, cudaStream_t stream) {
  LAVIE_REQUIRE(M >= 1 && M <= 8 && K % 8 == 0 && N > 0, LAVIE_ERR_SHAPE, "linear_smallm: M=%d (<=8) K=%d N=%d", M, K, N);
  LAVIE_REQUIRE(al16(x) && al16(w), LAVIE_ERR_ALIGN, "linear_smallm: alignment");
  const int blocks = (N + 7) / 8;
  const __nv_bfloat16* wp = static_cast<const __nv_bfloat16*>(w);
  if (M <= 2) launch_pdl(linear_smallm_kernel<2>, blocks, 256, 0, stream, x, M, K, wp, bias, out, N, silu_in, silu_out);
  else launch_pdl(linear_smallm_kernel<8>, blocks, 256, 0, stream, x, M, K, wp, bias, out, N, silu_in, silu_out);
  return lavie_check_launch("linear_smallm_kernel");
}

namespace {
int conv_in_impl(const float* x, int B, int Cin, int F, int H, int W, const float* w, const float* bias, int Cout,
                 void* out, int ldo, const float* input_scale, int triple, cudaStream_t stream) {
  LAVIE_REQUIRE(Cout % 8 == 0 && ldo % 8 == 0 && al16(out), LAVIE_ERR_SHAPE, "conv_in: Cout/ldo must be multiples of 8");
  const int smem = Cout * Cin * 9 * static_cast<int>(sizeof(float));
  LAVIE_REQUIRE(smem <= 200 * 1024, LAVIE_ERR_SHAPE, "conv_in: weights do not fit shared memory");
  static LavieSmemConfig configured;
  const int rc_cfg = lavie_config_smem(conv_in_kernel, smem, &configured, "conv_in_kernel");
  if (rc_cfg) return rc_cfg;
  LAVIE_REQUIRE(al16(bias), LAVIE_ERR_ALIGN, "conv_in: bias must be 16-byte aligned");
  const long long total = static_cast<long long>(B) * F * H * ((W + CIN_P - 1) / CIN_P) * (Cout / 8);
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 4) blocks = 148 * 4;
  launch_pdl(conv_in_kernel, static_cast<int>(blocks), 256, smem, stream, x, B, Cin, F, H, W, w, bias, Cout,
             static_cast<__nv_bfloat16*>(out), ldo, input_scale, triple);
  return lavie_check_launch("conv_in_kernel");
}
}  // namespace

extern "C" int lavie_conv_in(const float* x, int B, int Cin, int F, int H, int W, const float* w, const float* bias,
                             int Cout, void* out, int ldo, cudaStream_t stream) {
  return conv_in_impl(x, B, Cin, F, H, W, w, bias, Cout, out, ldo, nullptr, 0, stream);
}

extern "C" int lavie_conv_in_scaled(const float* x, const float* input_scale, int B, int Cin, int F, int H, int W,
                                    const float* w, const float* bias, int Cout, void* out, int ldo,
                                    cudaStream_t stream) {
  return conv_in_impl(x, B, Cin, F, H, W, w, bias, Cout, out, ldo, input_scale, 0, stream);
}

/* check mode: fp32 conv_in (already fp32 arithmetic) writing the split-bf16 triple [rows, 3*Cout] (ldo >= 3*Cout) */
extern "C" int lavie_check_conv_in(const float* x, const float* input_scale, int B, int Cin, int F, int H, int W,
                                   const float* w, const float* bias, int Cout, void* out, int ldo,
                                   cudaStream_t stream) {
  LAVIE_REQUIRE(ldo >= 3 * Cout, LAVIE_ERR_SHAPE, "check_conv_in: ldo must cover the triple");
  return conv_in_impl(x, B, Cin, F, H, W, w, bias, Cout, out, ldo, input_scale, 1, stream);
}

namespace {
int conv_out_impl(const void* x, int ldx, const float* scale_shift, int B, int F, int H, int W, int C, const float* w,
                  const float* bias, int Cout, float* out, int lo_off, cudaStream_t stream) {
  LAVIE_REQUIRE(Cout == 4 && C % 8 == 0 && ldx % 8 == 0, LAVIE_ERR_SHAPE, "conv_out: Cout must be 4, C %% 8 == 0");
  LAVIE_REQUIRE(al16(x) && al16(scale_shift), LAVIE_ERR_ALIGN, "conv_out: alignment");
  const int smem = Cout * 9 * C * static_cast<int>(sizeof(float));
  LAVIE_REQUIRE(smem <= 200 * 1024, LAVIE_ERR_SHAPE, "conv_out: weights do not fit shared memory");
  static LavieSmemConfig configured, configured_t;
  const int rc_cfg = lo_off ? lavie_config_smem(conv_out_kernel<4, true>, smem, &configured_t, "conv_out_kernel<check>")
                            : lavie_config_smem(conv_out_kernel<4, false>, smem, &configured, "conv_out_kernel");
  if (rc_cfg) return rc_cfg;
  const long long total = static_cast<long long>(B) * F * H * ((W + COUT_P - 1) / COUT_P);
  long long blocks = (total + 7) / 8;
  if (blocks > 148 * 2) blocks = 148 * 2;        // 2 resident blocks per SM (registers): one wave, one weight fill each
  if (lo_off)
    launch_pdl(conv_out_kernel<4, true>, static_cast<int>(blocks), 256, smem, stream,
               static_cast<const __nv_bfloat16*>(x), ldx, scale_shift, B, F, H, W, C, w, bias, out, lo_off);
  else
    launch_pdl(conv_out_kernel<4, false>, static_cast<int>(blocks), 256, smem, stream,
               static_cast<const __nv_bfloat16*>(x), ldx, scale_shift, B, F, H, W, C, w, bias, out, lo_off);
  return lavie_check_launch("conv_out_kernel");
}
}  // namespace

extern "C" int lavie_conv_out(const void* x, int ldx, const float* scale_shift, int B, int F, int H, int W, int C,
                              const float* w, const float* bias, int Cout, float* out, cudaStream_t stream) {
  return conv_out_impl(x, ldx, scale_shift, B, F, H, W, C, w, bias, Cout, out, 0, stream);
}

/* check mode: x is the split-bf16 triple [rows, 3C] (ldx >= 2C) */
extern "C" int lavie_check_conv_out(const void* x, int ldx, const float* scale_shift, int B, int F, int H, int W, int C,
                                    const float* w, const float* bias, int Cout, float* out, cudaStream_t stream) {
  LAVIE_REQUIRE(ldx >= 2 * C, LAVIE_ERR_SHAPE, "check_conv_out: ldx must cover hi and lo");
  return conv_out_impl(x, ldx, scale_shift, B, F, H, W, C, w, bias, Cout, out, C, stream);
}

extern "C" int lavie_im2col3x3_bf16(const void* x, int NF, int H, int W, int C, int stride, void* col,
                                    cudaStream_t stream) {
  LAVIE_REQUIRE(C % 8 == 0 && (stride == 1 || stride == 2), LAVIE_ERR_SHAPE, "im2col: C %% 8 == 0, stride 1 or 2");
  LAVIE_REQUIRE(al16(x) && al16(col), LAVIE_ERR_ALIGN, "im2col: alignment");
  const int Ho = (H + 2 - 3) / stride + 1, Wo = (W + 2 - 3) / stride + 1;
  const long long total = static_cast<long long>(NF) * Ho * Wo * 9 * (C / 8);
  launch_pdl(im2col3x3_kernel, grid_for(total, 256), 256, 0, stream, static_cast<const __nv_bfloat16*>(x), NF, H, W, C, stride,
                                                             Ho, Wo, static_cast<__nv_bfloat16*>(col));
  return lavie_check_launch("im2col3x3_kernel");
}

extern "C" int lavie_upsample_nearest2x(const void* x, int NF, int H, int W, int C, void* y, cudaStream_t stream) {
  LAVIE_REQUIRE(C % 8 == 0, LAVIE_ERR_SHAPE, "upsample: C %% 8 == 0");
  LAVIE_REQUIRE(al16(x) && al16(y), LAVIE_ERR_ALIGN, "upsample: alignment");
  const long long total = static_cast<long long>(NF) * 4 * H * W * (C / 8);
  launch_pdl(upsample2x_kernel, grid_for(total, 256), 256, 0, stream, static_cast<const __nv_bfloat16*>(x), NF, H, W, C,
                                                              static_cast<__nv_bfloat16*>(y));
  return lavie_check_launch("upsample2x_kernel");
}

extern "C" int lavie_unpack_nchw_f32(const void* y, int ldy, int B, int Cout, int F, int H, int W, float* out,
                                     cudaStream_t stream) {
  LAVIE_REQUIRE(B > 0 && Cout > 0 && F > 0 && H > 0 && W > 0, LAVIE_ERR_SHAPE, "unpack_nchw: empty problem");
  LAVIE_REQUIRE(ldy % 4 == 0 && ldy >= ((Cout + 3) & ~3) && (reinterpret_cast<uintptr_t>(y) & 7) == 0, LAVIE_ERR_ALIGN,
                "unpack_nchw: rows must be 8-byte aligned and hold Cout rounded up to 4 columns");
  const long long pps = static_cast<long long>(F) * H * W;
  launch_pdl(unpack_nchw_kernel, grid_for(B * pps, 256), 256, 0, stream, static_cast<const __nv_bfloat16*>(y), ldy, B,
             Cout, pps, out);
  return lavie_check_launch("unpack_nchw_kernel");
}

extern "C" int lavie_embedding_add(float* emb, const float* table, const long long* labels, int B, int dim, int rows,
                                   cudaStream_t stream) {
  LAVIE_REQUIRE(emb && table && labels && B > 0 && dim > 0 && rows > 0, LAVIE_ERR_SHAPE, "embedding_add: bad arguments");
  launch_pdl(embedding_add_kernel, (B * dim + 255) / 256, 256, 0, stream, emb, table, labels, B, dim, rows);
  return lavie_check_launch("embedding_add_kernel");
}

extern "C" int lavie_im2col_input_bf16(const float* x, const float* input_scale, int B, int Cin, int F, int H, int W,
                                       int kpad, void* col, cudaStream_t stream) {
  LAVIE_REQUIRE(x && col && B > 0 && Cin > 0 && F > 0 && H > 0 && W > 0, LAVIE_ERR_SHAPE, "im2col_input: bad arguments");
  LAVIE_REQUIRE(kpad % 8 == 0 && kpad >= 9 * Cin && al16(col), LAVIE_ERR_SHAPE,
                "im2col_input: kpad=%d must be a multiple of 8 and >= 9 * Cin = %d", kpad, 9 * Cin);
  const long long total = static_cast<long long>(B) * F * H * W * (kpad / 8);
  launch_pdl(im2col_input_kernel, grid_for(total, 256), 256, 0, stream, x, input_scale, B, Cin, F, H, W, kpad,
             static_cast<__nv_bfloat16*>(col));
  return lavie_check_launch("im2col_input_kernel");
}

extern "C" int lavie_im2col_frames_bf16(const unsigned char* frames, int N, int H, int W, int kpad, void* col,
                                        cudaStream_t stream) {
  LAVIE_REQUIRE(frames && col && N > 0 && H > 0 && W > 0, LAVIE_ERR_SHAPE, "im2col_frames: bad arguments");
  LAVIE_REQUIRE(kpad % 8 == 0 && kpad >= 27 && al16(col), LAVIE_ERR_SHAPE,
                "im2col_frames: kpad=%d must be a multiple of 8 and >= 27, col 16-byte aligned", kpad);
  const long long total = static_cast<long long>(N) * H * W * (kpad / 8);
  launch_pdl(im2col_frames_kernel, grid_for(total, 256), 256, 0, stream, frames, N, H, W, kpad,
             static_cast<__nv_bfloat16*>(col));
  return lavie_check_launch("im2col_frames_kernel");
}

extern "C" int lavie_cfg_ddim_step(const float* noise_uncond, const float* noise_text, float guidance, float alpha_t,
                                   float alpha_prev, const float* latents, float* latents_out, long long n,
                                   cudaStream_t stream) {
  LAVIE_REQUIRE(n > 0 && alpha_t > 0.f && alpha_t <= 1.f && alpha_prev > 0.f && alpha_prev <= 1.f, LAVIE_ERR_SHAPE,
                "cfg_ddim_step: bad arguments");
  launch_pdl(cfg_ddim_kernel, grid_for(n, 256), 256, 0, stream, noise_uncond, noise_text, guidance, sqrtf(alpha_t),
                                                        sqrtf(1.f - alpha_t), sqrtf(alpha_prev),
                                                        sqrtf(1.f - alpha_prev), latents, latents_out, n);
  return lavie_check_launch("cfg_ddim_kernel");
}


extern "C" int lavie_cfg_linear_step(const float* noise_uncond, const float* noise_text, float guidance, float a,
                                     float b, float c_noise, const float* latents, const float* noise,
                                     float* latents_out, long long n, cudaStream_t stream) {
  LAVIE_REQUIRE(n > 0 && noise_uncond && noise_text && latents && latents_out, LAVIE_ERR_SHAPE,
                "cfg_linear_step: bad arguments");
  launch_pdl(cfg_linear_step_kernel, grid_for(n, 256), 256, 0, stream, noise_uncond, noise_text, guidance, a, b, c_noise,
             latents, noise, latents_out, n);
  return lavie_check_launch("cfg_linear_step_kernel");
}

extern "C" int lavie_cfg_combine(const float* cond, const float* uncond, float scale, float* out0, float* out1,
                                 long long n, cudaStream_t stream) {
  LAVIE_REQUIRE(n > 0 && cond && uncond && out0, LAVIE_ERR_SHAPE, "cfg_combine: bad arguments");
  launch_pdl(cfg_combine_kernel, grid_for(n, 256), 256, 0, stream, cond, uncond, scale, out0, out1, n);
  return lavie_check_launch("cfg_combine_kernel");
}
