// AutoencoderKL (VAE) support kernels — SURVEY.md §8 (f)4 tail. The reference pipelines VAE-encode the condition image before
// the denoise loop (src/UniGenPipeline.py:306-308, src/condition.py:90-99) and VAE-decode the final latents after it
// (:430-433, :1120-1124); the network itself is diffusers 0.32.2 `AutoencoderKL` (ResnetBlock2D / Downsample2D / Upsample2D /
// the single-head mid-block attention). Every convolution runs on the tcgen05 GEMM (ug_gemm.cu: implicit 3x3, or a patch gather
// from here + the plain GEMM); this file holds the HBM-bound rest, all over NHWC bf16 activations with 16-byte accesses.
#include "ug_host.h"
#include "ug_ptx.cuh"

namespace ug {

namespace {

__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
  const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 p = unpack_bf16x2(u[i]);
    f[2 * i] = p.x;
    f[2 * i + 1] = p.y;
  }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  return make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
}

// ---------------------------------------------------------------------------------------------------------------------
// GroupNorm statistics, deterministic (no floating-point atomics: the same input gives the same bits on every run, eager or graph
// replay). Every sum is taken of x - P, P = the group's first channel at the image's first pixel (a bf16 value, so x - P is exact
// in fp32): a one-pass E[x^2] - mean^2 cancels all its digits once the group's mean is ~1e3 x its spread, the shifted sums only
// lose the digits of (mean - P)^2 / var, which is O(1) for a pivot drawn from the data.
// Pass 1: grid (chunks, batch); a block walks its share of the pixels, thread t owns the channel octet t % (c / 8) of every
// (t / (c / 8))-th pixel; the per-thread shifted sums are folded over the pixel lanes, then over each group's channels, in a fixed
// order, and the block writes one (mean - P, M2) pair per group (its element count follows from the block index).
// Pass 2: one warp per (image, group) merges the blocks' pairs with Chan's formula in a fixed order and stores (mean, var).
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float groupnorm_pivot(const __nv_bfloat16* x, long long b, int pixels, int c, int cpg, int ch) {
  return __bfloat162float(x[b * pixels * c + (ch / cpg) * cpg]);
}

__global__ void __launch_bounds__(256) groupnorm_partial_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ partial,
                                                                int pixels, int c, int groups) {
  __shared__ float part[256][17];  // [thread][8 sums | 8 sums of squares] (+1: no bank conflicts on the column walk)
  __shared__ float chs[2048], chq[2048];
  const int b = blockIdx.y;
  const int octets = c >> 3;
  const int cpg = c / groups;
  const int lanes_px = blockDim.x / octets;  // pixels a block covers per sweep (host guarantees octets <= blockDim.x)
  const int o = threadIdx.x % octets, sub = threadIdx.x / octets;
  const int per_block = (pixels + gridDim.x - 1) / gridDim.x;
  const int p0 = min(pixels, blockIdx.x * per_block), p1 = min(pixels, p0 + per_block);
  float s[8] = {0, 0, 0, 0, 0, 0, 0, 0}, q[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (sub < lanes_px) {
    float pv[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) pv[i] = groupnorm_pivot(x, b, pixels, c, cpg, o * 8 + i);
    const __nv_bfloat16* base = x + ((long long)b * pixels) * c + o * 8;
    int p = p0 + sub;
    // four pixels per trip: four independent 16-byte loads in flight per thread (the pass is a pure HBM stream)
    for (; p + 3 * lanes_px < p1; p += 4 * lanes_px) {
      uint4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = *reinterpret_cast<const uint4*>(base + (long long)(p + u * lanes_px) * c);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float f[8];
        unpack8(v[u], f);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float t = f[i] - pv[i];
          s[i] += t;
          q[i] = fmaf(t, t, q[i]);
        }
      }
    }
    for (; p < p1; p += lanes_px) {
      const uint4 v = *reinterpret_cast<const uint4*>(base + (long long)p * c);
      float f[8];
      unpack8(v, f);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float t = f[i] - pv[i];
        s[i] += t;
        q[i] = fmaf(t, t, q[i]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    part[threadIdx.x][i] = s[i];
    part[threadIdx.x][8 + i] = q[i];
  }
  __syncthreads();
  for (int ch = threadIdx.x; ch < c; ch += blockDim.x) {
    const int oo = ch >> 3, i = ch & 7;
    float ss = 0.0f, qq = 0.0f;
    for (int l = 0; l < lanes_px; ++l) {
      ss += part[l * octets + oo][i];
      qq += part[l * octets + oo][8 + i];
    }
    chs[ch] = ss;
    chq[ch] = qq;
  }
  __syncthreads();
  const float n = (float)(p1 - p0) * (float)cpg;
  for (int g = threadIdx.x; g < groups; g += blockDim.x) {
    float ss = 0.0f, qq = 0.0f;
    for (int j = 0; j < cpg; ++j) {
      ss += chs[g * cpg + j];
      qq += chq[g * cpg + j];
    }
    const float m = n > 0.0f ? ss / n : 0.0f;
    float* dst = partial + (((long long)b * gridDim.x + blockIdx.x) * groups + g) * 2;
    dst[0] = m;
    dst[1] = fmaxf(fmaf(-ss, m, qq), 0.0f);
  }
}

// Chan et al.: (n_a, m_a, M2_a) += (n_b, m_b, M2_b); an empty side leaves the other unchanged
__device__ __forceinline__ void chan_merge(float& n, float& m, float& m2, float nb, float mb, float m2b) {
  const float nt = n + nb;
  if (nb == 0.0f || nt == 0.0f) return;
  const float d = mb - m, f = nb / nt;
  m = fmaf(d, f, m);
  m2 = m2 + m2b + d * d * n * f;
  n = nt;
}

__global__ void __launch_bounds__(32) groupnorm_finalize_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ partial,
                                                                float* __restrict__ stats, int chunks, int pixels, int c, int groups) {
  const int b = blockIdx.x / groups, g = blockIdx.x % groups;
  const int cpg = c / groups;
  const int per_block = (pixels + chunks - 1) / chunks;
  float n = 0.0f, m = 0.0f, m2 = 0.0f;
  for (int k = threadIdx.x; k < chunks; k += 32) {
    const float* src = partial + (((long long)b * chunks + k) * groups + g) * 2;
    const int p0 = min(pixels, k * per_block), p1 = min(pixels, p0 + per_block);
    chan_merge(n, m, m2, (float)(p1 - p0) * (float)cpg, src[0], src[1]);
  }
  for (int off = 1; off < 32; off <<= 1) {
    const float nb = __shfl_xor_sync(0xffffffffu, n, off), mb = __shfl_xor_sync(0xffffffffu, m, off),
                m2b = __shfl_xor_sync(0xffffffffu, m2, off);
    chan_merge(n, m, m2, nb, mb, m2b);
  }
  if (threadIdx.x == 0) {
    stats[((long long)b * groups + g) * 2] = groupnorm_pivot(x, b, pixels, c, cpg, g * cpg) + m;
    stats[((long long)b * groups + g) * 2 + 1] = m2 / n;
  }
}

// Normalise + affine (+ SiLU). The grid stride is a multiple of c / 8, so a thread keeps ONE channel octet for its whole walk:
// its eight (mean, a = rstd * gamma) pairs are rebuilt only when the walk crosses into the next image. y = (x - mean) * a + beta:
// x - mean is exact when x is near the mean, where the folded form x * a + (beta - mean * a) would round beta - mean * a at the
// scale of mean * a.
template <bool kSilu>
__global__ void __launch_bounds__(256, 3) groupnorm_apply_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y,
                                                              const __nv_bfloat16* __restrict__ gamma,
                                                              const __nv_bfloat16* __restrict__ beta, const float* __restrict__ stats,
                                                              int pixels, int c, int groups, float eps, long long total_octets) {
  const int octets = c >> 3;
  const int cpg = c / groups;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long per_image = (long long)pixels * octets;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int o = (int)(i % octets);
  float bt[8], a[8], mn[8];
  unpack8(*reinterpret_cast<const uint4*>(beta + o * 8), bt);
  long long img_end = 0;  // the walk only moves forward: coefficients are rebuilt when it passes the end of the current image
  auto coeffs = [&](long long idx) {
    if (idx < img_end) return;
    const long long b = idx / per_image;
    img_end = (b + 1) * per_image;
    const float* st = stats + b * 2 * groups;
    float gm[8];  // re-read per image (L1 / L2 hits) rather than held in registers through the walk
    unpack8(*reinterpret_cast<const uint4*>(gamma + o * 8), gm);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int g = (o * 8 + j) / cpg;
      mn[j] = st[2 * g];
      a[j] = rsqrtf(st[2 * g + 1] + eps) * gm[j];
    }
  };
  auto one = [&](long long idx, const uint4& v) {
    float f[8];
    unpack8(v, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float r = fmaf(f[j] - mn[j], a[j], bt[j]);
      if (kSilu) r = __fdividef(r, 1.0f + __expf(-r));  // one ex2 + one rcp on the MUFU unit (a full-precision divide costs ~10 more)
      f[j] = r;
    }
    *reinterpret_cast<uint4*>(y + idx * 8) = pack8(f);
  };
  // four octets per trip (four independent 16-byte loads in flight per thread); they usually belong to the same image
  for (; i + 3 * stride < total_octets; i += 4 * stride) {
    uint4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = *reinterpret_cast<const uint4*>(x + (i + u * stride) * 8);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      coeffs(i + u * stride);
      one(i + u * stride, v[u]);
    }
  }
  for (; i + stride < total_octets; i += 2 * stride) {
    const uint4 v0 = *reinterpret_cast<const uint4*>(x + i * 8);
    const uint4 v1 = *reinterpret_cast<const uint4*>(x + (i + stride) * 8);
    coeffs(i);
    one(i, v0);
    coeffs(i + stride);
    one(i + stride, v1);
  }
  if (i < total_octets) {
    const uint4 v0 = *reinterpret_cast<const uint4*>(x + i * 8);
    coeffs(i);
    one(i, v0);
  }
}

// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) upsample2x_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, int h, int w, int octets,
                                                         long long total) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    // i indexes the OUTPUT (b, yo, xo, octet): coalesced stores, the four readers of an input pixel hit L1 / L2
    const int o = (int)(i % octets);
    long long t = i / octets;
    const int xo = (int)(t % (2 * w));
    t /= 2 * w;
    const int yo = (int)(t % (2 * h));
    const long long b = t / (2 * h);
    y[i] = x[((b * h + (yo >> 1)) * w + (xo >> 1)) * octets + o];
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Patch gather. Vector flavour: NHWC bf16 with c % 8 == 0 (one 16-byte load / store per thread and octet); scalar flavour: any
// strides / fp32 input (the 3-channel image, the 16-channel latents: tiny).
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) im2col_vec_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ cols, int h,
                                                         int w, int c, int kh, int kw, int stride, int pad_top, int pad_left, int h_out,
                                                         int w_out, int k_pad, long long total) {
  const int koct = k_pad >> 3, octets = c >> 3;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int ko = (int)(i % koct);
    long long m = i / koct;
    const int xo = (int)(m % w_out);
    long long t = m / w_out;
    const int yo = (int)(t % h_out);
    const long long b = t / h_out;
    uint4 v = make_uint4(0, 0, 0, 0);
    const int tap = ko / octets, o = ko - tap * octets;
    if (tap < kh * kw) {
      const int ky = tap / kw, kx = tap - ky * kw;
      const int yi = yo * stride + ky - pad_top, xi = xo * stride + kx - pad_left;
      if (yi >= 0 && yi < h && xi >= 0 && xi < w) v = *reinterpret_cast<const uint4*>(x + (((b * h + yi) * w + xi) * c + o * 8));
    }
    *reinterpret_cast<uint4*>(cols + i * 8) = v;
  }
}

template <typename T>
__global__ void __launch_bounds__(256) im2col_scalar_kernel(const T* __restrict__ x, long long sb, long long sy, long long sx,
                                                            long long sc, __nv_bfloat16* __restrict__ cols, int h, int w, int c, int kh,
                                                            int kw, int stride, int pad_top, int pad_left, int h_out, int w_out,
                                                            int k_pad, float alpha, float beta, long long total) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(i % k_pad);
    long long m = i / k_pad;
    const int xo = (int)(m % w_out);
    long long t = m / w_out;
    const int yo = (int)(t % h_out);
    const long long b = t / h_out;
    float v = 0.0f;
    if (k < kh * kw * c) {
      const int tap = k / c, ch = k - tap * c;
      const int ky = tap / kw, kx = tap - ky * kw;
      const int yi = yo * stride + ky - pad_top, xi = xo * stride + kx - pad_left;
      if (yi >= 0 && yi < h && xi >= 0 && xi < w) v = fmaf(alpha, (float)x[b * sb + yi * sy + xi * sx + ch * sc], beta);
    }
    cols[i] = __float2bfloat16(v);
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Row softmax in place: one block per row, three passes over the row at every length (max, sum of exponentials, normalise and
// store) read the row from memory three times; rows of the VAE attention are 4096-65536 long.
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float block_reduce(float v, float* red, bool is_max) {
  for (int off = 16; off > 0; off >>= 1) {
    const float o = __shfl_xor_sync(0xffffffffu, v, off);
    v = is_max ? fmaxf(v, o) : v + o;
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();  // red may still be read from the previous reduction
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float r = red[0];
  for (int i = 1; i < nw; ++i) r = is_max ? fmaxf(r, red[i]) : r + red[i];
  return r;
}

__global__ void __launch_bounds__(256) softmax_rows_kernel(__nv_bfloat16* __restrict__ x, long long row_stride, int cols) {
  __shared__ float red[8];
  __nv_bfloat16* row = x + (long long)blockIdx.x * row_stride;
  const int octets = cols >> 3;
  constexpr float kLog2e = 1.4426950408889634f;
  float m = -INFINITY;
  for (int o = threadIdx.x; o < octets; o += blockDim.x) {
    float f[8];
    unpack8(*reinterpret_cast<const uint4*>(row + o * 8), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) m = fmaxf(m, f[j]);
  }
  m = block_reduce(m, red, true);
  float sum = 0.0f;
  for (int o = threadIdx.x; o < octets; o += blockDim.x) {
    float f[8];
    unpack8(*reinterpret_cast<const uint4*>(row + o * 8), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) sum += exp2f((f[j] - m) * kLog2e);
  }
  sum = block_reduce(sum, red, false);
  const float inv = 1.0f / sum;
  for (int o = threadIdx.x; o < octets; o += blockDim.x) {
    float f[8];
    unpack8(*reinterpret_cast<const uint4*>(row + o * 8), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = exp2f((f[j] - m) * kLog2e) * inv;
    *reinterpret_cast<uint4*>(row + o * 8) = pack8(f);
  }
}

// ---------------------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) nhwc_to_nchw_kernel(const __nv_bfloat16* __restrict__ x, long long pixel_stride, T* __restrict__ y,
                                                           int c, long long pixels, long long total) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    // i indexes the OUTPUT (b, ch, pixel)
    const long long px = i % pixels;
    long long t = i / pixels;
    const int ch = (int)(t % c);
    const long long b = t / c;
    const __nv_bfloat16 v = x[(b * pixels + px) * pixel_stride + ch];
    if constexpr (sizeof(T) == 4) y[i] = __bfloat162float(v); else y[i] = v;
  }
}

__global__ void __launch_bounds__(256) vae_sample_kernel(const __nv_bfloat16* __restrict__ moments, long long pixel_stride,
                                                         const float* __restrict__ noise, __nv_bfloat16* __restrict__ latents, int c,
                                                         long long pixels, float shift, float scale, long long total) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long px = i % pixels;
    long long t = i / pixels;
    const int ch = (int)(t % c);
    const long long b = t / c;
    const __nv_bfloat16* mrow = moments + (b * pixels + px) * pixel_stride;
    float z = __bfloat162float(mrow[ch]);
    if (noise) {
      const float logvar = fminf(fmaxf(__bfloat162float(mrow[c + ch]), -30.0f), 20.0f);
      z = fmaf(__expf(0.5f * logvar), noise[i], z);
    }
    latents[i] = __float2bfloat16((z - shift) * scale);
  }
}

inline int grid_for(long long work_items, int threads = 256) {
  const long long blocks = (work_items + threads - 1) / threads;
  const long long cap = (long long)num_sms() * 16;
  return (int)(blocks < 1 ? 1 : (blocks > cap ? cap : blocks));
}

}  // namespace
}  // namespace ug

using namespace ug;

extern "C" int ug_groupnorm_bf16(const void* x, void* y, const void* gamma, const void* beta, float* stats, int32_t batch,
                                 int32_t pixels, int32_t c, int32_t groups, float eps, int32_t silu_act, void* stream) {
  UG_CHECK_ARG(x && y && gamma && beta && stats, "groupnorm: null pointer");
  UG_CHECK_ARG(batch >= 1 && pixels >= 1 && c >= 8 && c % 8 == 0 && c <= 2048, "groupnorm: c (%d) must be a multiple of 8, <= 2048", c);
  UG_CHECK_ARG(groups >= 1 && groups <= 256 && c % groups == 0, "groupnorm: groups (%d) must divide c (%d)", groups, c);
  UG_CHECK_ARG(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(gamma) |
                 reinterpret_cast<uintptr_t>(beta)) & 15) == 0, "groupnorm: operands must be 16-byte aligned");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  // enough blocks per image to fill the machine, at least ~64 pixels each
  int chunks = (num_sms() * 4 + batch - 1) / batch;
  if (chunks > (pixels + 63) / 64) chunks = (pixels + 63) / 64;
  if (chunks > UG_GROUPNORM_MAX_CHUNKS) chunks = UG_GROUPNORM_MAX_CHUNKS;
  if (chunks < 1) chunks = 1;
  float* partial = stats + (long long)batch * groups * 2;
  groupnorm_partial_kernel<<<dim3(chunks, batch), 256, 0, s>>>((const __nv_bfloat16*)x, partial, pixels, c, groups);
  UG_CHECK_LAUNCH("groupnorm_partial");
  groupnorm_finalize_kernel<<<batch * groups, 32, 0, s>>>((const __nv_bfloat16*)x, partial, stats, chunks, pixels, c, groups);
  UG_CHECK_LAUNCH("groupnorm_finalize");
  const long long total = (long long)batch * pixels * (c / 8);
  // grid stride (blocks x 256 threads) must be a multiple of c / 8: a thread then keeps one channel octet for its whole walk
  int mult = c / 8, g256 = 256;
  while (g256 % 2 == 0 && mult % 2 == 0) { g256 /= 2; mult /= 2; }  // mult = (c / 8) / gcd(c / 8, 256)
  int grid = grid_for((total + 3) / 4);
  grid = (grid + mult - 1) / mult * mult;
  if (silu_act)
    groupnorm_apply_kernel<true><<<grid, 256, 0, s>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)y, (const __nv_bfloat16*)gamma,
                                                      (const __nv_bfloat16*)beta, stats, pixels, c, groups, eps, total);
  else
    groupnorm_apply_kernel<false><<<grid, 256, 0, s>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)y, (const __nv_bfloat16*)gamma,
                                                       (const __nv_bfloat16*)beta, stats, pixels, c, groups, eps, total);
  UG_CHECK_LAUNCH("groupnorm_apply");
  return UG_OK;
}

extern "C" int ug_upsample2x_nhwc_bf16(const void* x, void* y, int32_t batch, int32_t h, int32_t w, int32_t c, void* stream) {
  UG_CHECK_ARG(x && y && batch >= 1 && h >= 1 && w >= 1 && c >= 8 && c % 8 == 0, "upsample2x: bad arguments (c must be a multiple of 8)");
  UG_CHECK_ARG(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) == 0, "upsample2x: 16-byte alignment");
  const long long total = (long long)batch * 4 * h * w * (c / 8);
  upsample2x_kernel<<<grid_for(total), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>((const uint4*)x, (uint4*)y, h, w, c / 8, total);
  UG_CHECK_LAUNCH("upsample2x");
  return UG_OK;
}

extern "C" int ug_im2col_bf16(const void* x, int32_t x_is_f32, int64_t sb, int64_t sy, int64_t sx, int64_t sc, void* cols,
                              int32_t batch, int32_t h, int32_t w, int32_t c, int32_t kh, int32_t kw, int32_t stride,
                              int32_t pad_top, int32_t pad_left, int32_t h_out, int32_t w_out, int32_t k_pad, float alpha, float beta,
                              void* stream) {
  UG_CHECK_ARG(x && cols && batch >= 1 && h >= 1 && w >= 1 && c >= 1 && kh >= 1 && kw >= 1 && stride >= 1 && h_out >= 1 && w_out >= 1,
               "im2col: bad arguments");
  UG_CHECK_ARG(k_pad >= kh * kw * c && k_pad % 8 == 0, "im2col: k_pad (%d) must be a multiple of 8 and cover kh * kw * c (%d)", k_pad,
               kh * kw * c);
  UG_CHECK_ARG((reinterpret_cast<uintptr_t>(cols) & 15) == 0, "im2col: cols must be 16-byte aligned");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const long long rows = (long long)batch * h_out * w_out;
  const bool nhwc = sc == 1 && sx == c && sy == (int64_t)w * c && sb == (int64_t)h * w * c;
  if (!x_is_f32 && nhwc && c % 8 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 && alpha == 1.0f && beta == 0.0f) {
    const long long total = rows * (k_pad / 8);
    im2col_vec_kernel<<<grid_for(total), 256, 0, s>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)cols, h, w, c, kh, kw, stride, pad_top,
                                                      pad_left, h_out, w_out, k_pad, total);
  } else {
    const long long total = rows * k_pad;
    if (x_is_f32)
      im2col_scalar_kernel<float><<<grid_for(total), 256, 0, s>>>((const float*)x, sb, sy, sx, sc, (__nv_bfloat16*)cols, h, w, c, kh, kw,
                                                                  stride, pad_top, pad_left, h_out, w_out, k_pad, alpha, beta, total);
    else
      im2col_scalar_kernel<__nv_bfloat16><<<grid_for(total), 256, 0, s>>>((const __nv_bfloat16*)x, sb, sy, sx, sc, (__nv_bfloat16*)cols, h,
                                                                          w, c, kh, kw, stride, pad_top, pad_left, h_out, w_out, k_pad,
                                                                          alpha, beta, total);
  }
  UG_CHECK_LAUNCH("im2col");
  return UG_OK;
}

extern "C" int ug_softmax_rows_bf16(void* x, int64_t row_stride, int32_t rows, int32_t cols, void* stream) {
  UG_CHECK_ARG(x && rows >= 1 && cols >= 8 && cols % 8 == 0 && row_stride >= cols && row_stride % 8 == 0,
               "softmax_rows: cols (%d) and the row stride must be multiples of 8", cols);
  UG_CHECK_ARG((reinterpret_cast<uintptr_t>(x) & 15) == 0, "softmax_rows: 16-byte alignment");
  softmax_rows_kernel<<<rows, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>((__nv_bfloat16*)x, row_stride, cols);
  UG_CHECK_LAUNCH("softmax_rows");
  return UG_OK;
}

extern "C" int ug_nhwc_to_nchw(const void* x, int64_t pixel_stride, void* y, int32_t y_is_f32, int32_t batch, int32_t c, int32_t h,
                               int32_t w, void* stream) {
  UG_CHECK_ARG(x && y && batch >= 1 && c >= 1 && h >= 1 && w >= 1 && pixel_stride >= c, "nhwc_to_nchw: bad arguments");
  const long long pixels = (long long)h * w, total = (long long)batch * c * pixels;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (y_is_f32)
    nhwc_to_nchw_kernel<float><<<grid_for(total), 256, 0, s>>>((const __nv_bfloat16*)x, pixel_stride, (float*)y, c, pixels, total);
  else
    nhwc_to_nchw_kernel<__nv_bfloat16><<<grid_for(total), 256, 0, s>>>((const __nv_bfloat16*)x, pixel_stride, (__nv_bfloat16*)y, c, pixels,
                                                                       total);
  UG_CHECK_LAUNCH("nhwc_to_nchw");
  return UG_OK;
}

extern "C" int ug_vae_sample(const void* moments, int64_t pixel_stride, const float* noise, void* latents, int32_t batch, int32_t c,
                             int32_t pixels, float shift, float scale, void* stream) {
  UG_CHECK_ARG(moments && latents && batch >= 1 && c >= 1 && pixels >= 1 && pixel_stride >= 2 * c, "vae_sample: bad arguments");
  const long long total = (long long)batch * c * pixels;
  vae_sample_kernel<<<grid_for(total), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>((const __nv_bfloat16*)moments, pixel_stride, noise,
                                                                                         (__nv_bfloat16*)latents, c, pixels, shift, scale,
                                                                                         total);
  UG_CHECK_LAUNCH("vae_sample");
  return UG_OK;
}
