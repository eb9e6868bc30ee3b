// Fused elementwise family of the UniGen hot path (HBM-bound): LayerNorm+modulate, per-head RMSNorm+RoPE,
// RoPE table, small-M linears (AdaLN / timestep / expert-modulation GEMVs), adds / copies / casts.
// All kernels use 16-byte vector accesses and fp32 math; bf16 is storage only.
#include <cstdlib>
#include <cstring>

#include <cuda_fp8.h>

#include <algorithm>

#include "ug_host.h"
#include "ug_ptx.cuh"

namespace ug {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 u;
  u.x = pack_bf16x2(f[0], f[1]); u.y = pack_bf16x2(f[2], f[3]);
  u.z = pack_bf16x2(f[4], f[5]); u.w = pack_bf16x2(f[6], f[7]);
  return u;
}

// ---------------------------------------------------------------------------------------------------
// Row-wise e4m3 quantisation (the activation side of the fp8 GEMM): amax = max |x| of the row; amax == 0 -> scale 1, q = 0;
// else inv = 448 / amax, scale = amax / 448 (IEEE round-to-nearest divisions) and q = cvt.rn.satfinite.e4m3(x * inv).
// ---------------------------------------------------------------------------------------------------
struct Fp8Out {  // e4m3 rows + one fp32 scale per row; q == nullptr: plain bf16 output
  uint8_t* q;
  long long q_rs, q_bs;
  float* scale;
  long long s_bs;
};

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float fp8_inv_scale(float amax) { return amax == 0.f ? 0.f : __fdiv_rn(448.0f, amax); }
__device__ __forceinline__ float fp8_row_scale(float amax) { return amax == 0.f ? 1.f : __fdiv_rn(amax, 448.0f); }
// the values a bf16 store of f would hold (the fused LN kernels quantise exactly what ug_ln_modulate writes)
__device__ __forceinline__ void round_bf16x8(float (&f)[8]) {
#pragma unroll
  for (int j = 0; j < 8; ++j) f[j] = __bfloat162float(__float2bfloat16_rn(f[j]));
}
__device__ __forceinline__ float absmax8(const float (&f)[8], float m) {
#pragma unroll
  for (int j = 0; j < 8; ++j) m = fmaxf(m, fabsf(f[j]));
  return m;
}
// 8 values -> 8 e4m3 bytes (x * inv, saturating round-to-nearest); inv == 0 (all-zero row) stores +0 everywhere
__device__ __forceinline__ uint2 e4m3x8(const float (&f)[8], float inv) {
  if (inv == 0.f) return make_uint2(0u, 0u);
  uint32_t h[4];
#pragma unroll
  for (int j = 0; j < 4; ++j)
    h[j] = (uint32_t)__nv_cvt_float2_to_fp8x2(make_float2(f[2 * j] * inv, f[2 * j + 1] * inv), __NV_SATFINITE, __NV_E4M3);
  return make_uint2(h[0] | (h[1] << 16), h[2] | (h[3] << 16));
}

// one block per row, the row resident in registers (k <= 8 * kThreads * kMaxV)
template <int kThreads, int kMaxV>
__global__ void __launch_bounds__(kThreads) quant_rows_fp8_kernel(const __nv_bfloat16* __restrict__ x, long long x_rs, long long x_bs,
                                                                  Fp8Out o, int k) {
  constexpr int kWarps = kThreads / 32;
  __shared__ float red[kWarps];
  const int t = threadIdx.x, r = blockIdx.x, b = blockIdx.y;
  const uint4* xp = reinterpret_cast<const uint4*>(x + (long long)b * x_bs + (long long)r * x_rs);
  const int nvec = k >> 3;
  uint4 buf[kMaxV];
  float amax = 0.f;
#pragma unroll
  for (int i = 0; i < kMaxV; ++i) {
    const int v = t + kThreads * i;
    if (v < nvec) {
      buf[i] = xp[v];
      float f[8];
      unpack8(buf[i], f);
      amax = absmax8(f, amax);
    }
  }
  amax = warp_max(amax);
  if ((t & 31) == 0) red[t >> 5] = amax;
  __syncthreads();
#pragma unroll
  for (int w = 0; w < kWarps; ++w) amax = fmaxf(amax, red[w]);
  const float inv = fp8_inv_scale(amax);
  uint2* qp = reinterpret_cast<uint2*>(o.q + (long long)b * o.q_bs + (long long)r * o.q_rs);
#pragma unroll
  for (int i = 0; i < kMaxV; ++i) {
    const int v = t + kThreads * i;
    if (v < nvec) {
      float f[8];
      unpack8(buf[i], f);
      qp[v] = e4m3x8(f, inv);
    }
  }
  if (t == 0) o.scale[(long long)b * o.s_bs + r] = fp8_row_scale(amax);
}

// ---------------------------------------------------------------------------------------------------
// LayerNorm (no affine) + (1 + scale) * x + shift.  One warp per row, row kept in registers (d <= 8*32*kMaxV).
// Algorithmic HBM bytes per row: 2*d (read) + 2*d (write).
// ---------------------------------------------------------------------------------------------------
struct RowSegs {
  int nseg;
  int bounds[UG_MAX_SEGMENTS + 1];
};

// kFp8 (every kernel below): the row is written as e4m3 + one fp32 scale (Fp8Out) instead of bf16 — the same values, rounded to
// bf16 first, then quantised like quant_rows_fp8_kernel (a first pass over the row finds the amax, a second one stores).
template <int kMaxV, bool kFp8 = false>
__global__ void __launch_bounds__(256) ln_modulate_kernel(const __nv_bfloat16* __restrict__ x, long long x_rs,
                                                          long long x_bs, __nv_bfloat16* __restrict__ out,
                                                          long long o_rs, long long o_bs,
                                                          const float* __restrict__ shift,
                                                          const float* __restrict__ scale, long long mod_bs, int batch,
                                                          int rows, int d, float eps,
                                                          const int* __restrict__ slot_token = nullptr, int capacity = 1,
                                                          int tokens_per_batch = 1, int empty_index = 0,
                                                          long long mod_es = 0, RowSegs segs = RowSegs{0, {0}},
                                                          long long mod_seg_stride = 0, Fp8Out fo = Fp8Out{}) {
  const int warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp_global >= batch * rows) return;
  const int b = warp_global / rows, r = warp_global % rows;
  // modulation row: the sample index b, or (slot mode) expert e = r / capacity and the sample the slot's token came from
  long long mod_off = (long long)b * mod_bs;
  if (segs.nseg > 0) {  // per-row-segment modulation vectors (the P-variant's text / image / condition streams in one launch)
    int si = 0;
    for (int s = 0; s < segs.nseg; ++s)
      if (r >= segs.bounds[s] && r < segs.bounds[s + 1]) si = s;
    mod_off += (long long)si * mod_seg_stride;
  }
  if (slot_token) {
    const int token = slot_token[r];
    mod_off = (long long)(r / capacity) * mod_es + (long long)(token < 0 ? empty_index : token / tokens_per_batch) * mod_bs;
  }
  const uint4* xp = reinterpret_cast<const uint4*>(x + (long long)b * x_bs + (long long)r * x_rs);
  const int nvec = d >> 3;
  uint4 buf[kMaxV];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < kMaxV; ++i) {
    const int v = lane + 32 * i;
    if (v < nvec) {
      buf[i] = xp[v];
      float f[8];
      unpack8(buf[i], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) sum += f[j];
    }
  }
  const float mean = warp_sum(sum) / (float)d;
  float var = 0.f;
#pragma unroll
  for (int i = 0; i < kMaxV; ++i) {
    const int v = lane + 32 * i;
    if (v < nvec) {
      float f[8];
      unpack8(buf[i], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) { float t = f[j] - mean; var += t * t; }
    }
  }
  const float rstd = rsqrtf(warp_sum(var) / (float)d + eps);
  uint4* op = reinterpret_cast<uint4*>(out + (long long)b * o_bs + (long long)r * o_rs);
  uint2* qp = kFp8 ? reinterpret_cast<uint2*>(fo.q + (long long)b * fo.q_bs + (long long)r * fo.q_rs) : nullptr;
  const float* sh = shift + mod_off;
  const float* sc = scale + mod_off;
  float amax = 0.f, inv = 0.f;
#pragma unroll 1
  for (int pass = kFp8 ? 0 : 1; pass < 2; ++pass) {
    if (kFp8 && pass == 1) {
      amax = warp_max(amax);
      inv = fp8_inv_scale(amax);
    }
#pragma unroll
    for (int i = 0; i < kMaxV; ++i) {
      const int v = lane + 32 * i;
      if (v < nvec) {
        float f[8];
        unpack8(buf[i], f);
        const float4 s0 = *reinterpret_cast<const float4*>(sc + 8 * v), s1 = *reinterpret_cast<const float4*>(sc + 8 * v + 4);
        const float4 h0 = *reinterpret_cast<const float4*>(sh + 8 * v), h1 = *reinterpret_cast<const float4*>(sh + 8 * v + 4);
        const float s[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
        const float h[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = (f[j] - mean) * rstd * (1.f + s[j]) + h[j];
        if constexpr (kFp8) {
          round_bf16x8(f);
          if (pass == 0) amax = absmax8(f, amax);
          else qp[v] = e4m3x8(f, inv);
        } else {
          op[v] = pack8(f);
        }
      }
    }
  }
  if (kFp8 && lane == 0) fo.scale[(long long)b * fo.s_bs + r] = fp8_row_scale(amax);
}

// Same op, TWO warps per row (adjacent warps 2i, 2i+1 of a block; partial sums meet in shared memory). With one warp per
// row and the row in registers a 3072-wide pass needs ~80 registers per thread -> 24 resident warps per SM -> 4608 rows take
// 1.3 waves and the HBM pipe idles through the partial second wave; half the row per warp halves the registers, doubles the
// resident rows' worth of loads in flight and shortens the tail.
template <int kMaxV, bool kFp8 = false>
__global__ void __launch_bounds__(256, 4) ln_modulate2_kernel(const __nv_bfloat16* __restrict__ x, long long x_rs,
                                                           long long x_bs, __nv_bfloat16* __restrict__ out,
                                                           long long o_rs, long long o_bs,
                                                           const float* __restrict__ shift,
                                                           const float* __restrict__ scale, long long mod_bs, int batch,
                                                           int rows, int d, float eps, const int* __restrict__ slot_token,
                                                           int capacity, int tokens_per_batch, int empty_index,
                                                           long long mod_es, RowSegs segs, long long mod_seg_stride,
                                                           Fp8Out fo = Fp8Out{}) {
  __shared__ float red_sum[8], red_var[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row_global = (long long)blockIdx.x * 4 + (warp >> 1);
  const bool valid = row_global < (long long)batch * rows;
  const int b = valid ? (int)(row_global / rows) : 0, r = valid ? (int)(row_global % rows) : 0;
  const int l64 = (warp & 1) * 32 + lane;
  long long mod_off = (long long)b * mod_bs;
  if (segs.nseg > 0) {
    int si = 0;
    for (int s = 0; s < segs.nseg; ++s)
      if (r >= segs.bounds[s] && r < segs.bounds[s + 1]) si = s;
    mod_off += (long long)si * mod_seg_stride;
  }
  if (slot_token && valid) {
    const int token = slot_token[r];
    mod_off = (long long)(r / capacity) * mod_es + (long long)(token < 0 ? empty_index : token / tokens_per_batch) * mod_bs;
  }
  const uint4* xp = reinterpret_cast<const uint4*>(x + (long long)b * x_bs + (long long)r * x_rs);
  const int nvec = d >> 3;
  uint4 buf[kMaxV];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < kMaxV; ++i) {
    const int v = l64 + 64 * i;
    if (valid && v < nvec) {
      buf[i] = xp[v];
      float f[8];
      unpack8(buf[i], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) sum += f[j];
    }
  }
  sum = warp_sum(sum);
  if (lane == 0) red_sum[warp] = sum;
  __syncthreads();
  const float mean = (red_sum[warp] + red_sum[warp ^ 1]) / (float)d;
  float var = 0.f;
#pragma unroll
  for (int i = 0; i < kMaxV; ++i) {
    const int v = l64 + 64 * i;
    if (valid && v < nvec) {
      float f[8];
      unpack8(buf[i], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) { float t = f[j] - mean; var += t * t; }
    }
  }
  var = warp_sum(var);
  if (lane == 0) red_var[warp] = var;
  __syncthreads();
  const float rstd = rsqrtf((red_var[warp] + red_var[warp ^ 1]) / (float)d + eps);
  if (!kFp8 && !valid) return;  // (fp8: every thread reaches the amax barrier below)
  uint4* op = reinterpret_cast<uint4*>(out + (long long)b * o_bs + (long long)r * o_rs);
  uint2* qp = kFp8 ? reinterpret_cast<uint2*>(fo.q + (long long)b * fo.q_bs + (long long)r * fo.q_rs) : nullptr;
  const float* sh = shift + mod_off;
  const float* sc = scale + mod_off;
  float amax = 0.f, inv = 0.f;
#pragma unroll 1
  for (int pass = kFp8 ? 0 : 1; pass < 2; ++pass) {
    if (kFp8 && pass == 1) {  // red_sum is free again: every thread read it before the variance barrier
      amax = warp_max(amax);
      if (lane == 0) red_sum[warp] = amax;
      __syncthreads();
      amax = fmaxf(red_sum[warp], red_sum[warp ^ 1]);
      inv = fp8_inv_scale(amax);
    }
#pragma unroll
    for (int i = 0; i < kMaxV; ++i) {
      const int v = l64 + 64 * i;
      if (valid && v < nvec) {
        float f[8];
        unpack8(buf[i], f);
        const float4 s0 = *reinterpret_cast<const float4*>(sc + 8 * v), s1 = *reinterpret_cast<const float4*>(sc + 8 * v + 4);
        const float4 h0 = *reinterpret_cast<const float4*>(sh + 8 * v), h1 = *reinterpret_cast<const float4*>(sh + 8 * v + 4);
        const float s[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
        const float h[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = (f[j] - mean) * rstd * (1.f + s[j]) + h[j];
        if constexpr (kFp8) {
          round_bf16x8(f);
          if (pass == 0) amax = absmax8(f, amax);
          else qp[v] = e4m3x8(f, inv);
        } else {
          op[v] = pack8(f);
        }
      }
    }
  }
  if (kFp8 && valid && l64 == 0) fo.scale[(long long)b * fo.s_bs + r] = fp8_row_scale(amax);
}

// Same op for the plain per-sample form (no slots / row segments), kR rows per block: thread t owns the 16-byte column chunks
// t, t + kThreads, ... of ALL kR rows, so the fp32 shift / scale vectors — 4 x the bytes of a bf16 row, and the same for every
// row of a sample — are loaded ONCE per kR rows, and they are requested together with the rows (one memory latency per block
// instead of two: in the two-warp kernel the modulation loads only issue after both reductions, ncu: 50 % of its stall samples
// are long-scoreboard waits on `1 + scale`). kR * kChunks + 4 * kChunks 16-byte loads in flight per thread.
template <int kThreads, int kChunks, int kR, bool kFp8 = false>
__global__ void __launch_bounds__(kThreads) ln_modulate_rows_kernel(const __nv_bfloat16* __restrict__ x, long long x_rs, long long x_bs,
                                                                    __nv_bfloat16* __restrict__ out, long long o_rs, long long o_bs,
                                                                    const float* __restrict__ shift, const float* __restrict__ scale,
                                                                    long long mod_bs, int rows, int d, float eps, Fp8Out fo = Fp8Out{}) {
  constexpr int kWarps = kThreads / 32;
  __shared__ float red[2][kR][kWarps];
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int b = blockIdx.y;
  const int r0 = blockIdx.x * kR;
  const __nv_bfloat16* xb = x + (long long)b * x_bs;
  uint4 buf[kR][kChunks];
#pragma unroll
  for (int r = 0; r < kR; ++r) {
    const int row = min(r0 + r, rows - 1);  // a ragged last block re-reads the last row; only rows < `rows` are stored
    const uint4* xp = reinterpret_cast<const uint4*>(xb + (long long)row * x_rs);
#pragma unroll
    for (int i = 0; i < kChunks; ++i) buf[r][i] = xp[t + kThreads * i];
  }
  float4 sc[kChunks][2], sh[kChunks][2];
  const float* scp = scale + (long long)b * mod_bs;
  const float* shp = shift + (long long)b * mod_bs;
#pragma unroll
  for (int i = 0; i < kChunks; ++i) {
    const int c = 8 * (t + kThreads * i);
    sc[i][0] = *reinterpret_cast<const float4*>(scp + c); sc[i][1] = *reinterpret_cast<const float4*>(scp + c + 4);
    sh[i][0] = *reinterpret_cast<const float4*>(shp + c); sh[i][1] = *reinterpret_cast<const float4*>(shp + c + 4);
  }
  float mean[kR], rstd[kR];
#pragma unroll
  for (int r = 0; r < kR; ++r) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < kChunks; ++i) {
      float f[8];
      unpack8(buf[r][i], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) s += f[j];
    }
    s = warp_sum(s);
    if (lane == 0) red[0][r][warp] = s;
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < kR; ++r) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) s += red[0][r][w];
    mean[r] = s / (float)d;
    float v = 0.f;
#pragma unroll
    for (int i = 0; i < kChunks; ++i) {
      float f[8];
      unpack8(buf[r][i], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) { const float u = f[j] - mean[r]; v += u * u; }
    }
    v = warp_sum(v);
    if (lane == 0) red[1][r][warp] = v;
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < kR; ++r) {
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) v += red[1][r][w];
    rstd[r] = rsqrtf(v / (float)d + eps);
  }
  __nv_bfloat16* ob = out + (long long)b * o_bs;
  float amax[kR], inv[kR];
#pragma unroll
  for (int r = 0; r < kR; ++r) amax[r] = inv[r] = 0.f;
#pragma unroll 1
  for (int pass = kFp8 ? 0 : 1; pass < 2; ++pass) {
    if (kFp8 && pass == 1) {  // red[0] is free again: every thread read it before the variance barrier
#pragma unroll
      for (int r = 0; r < kR; ++r) {
        const float m = warp_max(amax[r]);
        if (lane == 0) red[0][r][warp] = m;
      }
      __syncthreads();
#pragma unroll
      for (int r = 0; r < kR; ++r) {
        float m = 0.f;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) m = fmaxf(m, red[0][r][w]);
        amax[r] = m;
        inv[r] = fp8_inv_scale(m);
      }
    }
#pragma unroll
    for (int r = 0; r < kR; ++r) {
      if (r0 + r >= rows) break;
      uint4* op = reinterpret_cast<uint4*>(ob + (long long)(r0 + r) * o_rs);
#pragma unroll
      for (int i = 0; i < kChunks; ++i) {
        float f[8];
        unpack8(buf[r][i], f);
        const float s[8] = {sc[i][0].x, sc[i][0].y, sc[i][0].z, sc[i][0].w, sc[i][1].x, sc[i][1].y, sc[i][1].z, sc[i][1].w};
        const float h[8] = {sh[i][0].x, sh[i][0].y, sh[i][0].z, sh[i][0].w, sh[i][1].x, sh[i][1].y, sh[i][1].z, sh[i][1].w};
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = (f[j] - mean[r]) * rstd[r] * (1.f + s[j]) + h[j];
        if constexpr (kFp8) {
          round_bf16x8(f);
          if (pass == 0) {
            amax[r] = absmax8(f, amax[r]);
          } else {
            uint2* qp = reinterpret_cast<uint2*>(fo.q + (long long)b * fo.q_bs + (long long)(r0 + r) * fo.q_rs);
            qp[t + kThreads * i] = e4m3x8(f, inv[r]);
          }
        } else {
          op[t + kThreads * i] = pack8(f);
        }
      }
    }
  }
  if constexpr (kFp8) {
    if (t == 0) {
#pragma unroll
      for (int r = 0; r < kR; ++r)
        if (r0 + r < rows) fo.scale[(long long)b * fo.s_bs + r0 + r] = fp8_row_scale(amax[r]);
    }
  }
}

// Persistent form of the same kernel (same thread -> column mapping and reduction order: bit-identical results). A block keeps
// its (1 + scale, shift) column chunks in registers and walks the row groups g = blockIdx.x, + gridDim.x, ...; the rows of group
// g + gridDim.x are requested BEFORE group g is reduced, so after the first group the load latency hides behind the two
// reductions and the stores, and the modulation vectors (as many bytes as the kR rows of a group) are fetched once per block
// instead of once per group. The one-group-per-block kernel was wave-latency-bound: 2.6 waves of (load -> 2 syncs -> store).
template <int kThreads, int kChunks, int kR>
__global__ void __launch_bounds__(kThreads) ln_modulate_stream_kernel(const __nv_bfloat16* __restrict__ x, long long x_rs, long long x_bs,
                                                                      __nv_bfloat16* __restrict__ out, long long o_rs, long long o_bs,
                                                                      const float* __restrict__ shift, const float* __restrict__ scale,
                                                                      long long mod_bs, int rows, int d, float eps) {
  constexpr int kWarps = kThreads / 32;
  __shared__ float red[2][kR][kWarps];
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int b = blockIdx.y;
  const int groups = (rows + kR - 1) / kR;
  const __nv_bfloat16* xb = x + (long long)b * x_bs;
  __nv_bfloat16* ob = out + (long long)b * o_bs;
  auto load_group = [&](int g, uint4 (&dst)[kR][kChunks]) {
#pragma unroll
    for (int r = 0; r < kR; ++r) {
      const int row = min(g * kR + r, rows - 1);  // a ragged last group re-reads the last row; only rows < `rows` are stored
      const uint4* xp = reinterpret_cast<const uint4*>(xb + (long long)row * x_rs);
#pragma unroll
      for (int i = 0; i < kChunks; ++i) dst[r][i] = xp[t + kThreads * i];
    }
  };
  int g = blockIdx.x;
  if (g >= groups) return;
  uint4 buf[kR][kChunks];
  load_group(g, buf);
  // this thread's column chunks of (scale, shift), parked in shared memory (each thread reads back only what it wrote: no
  // barrier, conflict-free) — in registers they would not fit next to two groups of rows
  __shared__ float4 smod[2][kChunks * 2][kThreads];
  const float* scp = scale + (long long)b * mod_bs;
  const float* shp = shift + (long long)b * mod_bs;
#pragma unroll
  for (int i = 0; i < kChunks; ++i) {
    const int c = 8 * (t + kThreads * i);
    smod[0][2 * i][t] = *reinterpret_cast<const float4*>(scp + c); smod[0][2 * i + 1][t] = *reinterpret_cast<const float4*>(scp + c + 4);
    smod[1][2 * i][t] = *reinterpret_cast<const float4*>(shp + c); smod[1][2 * i + 1][t] = *reinterpret_cast<const float4*>(shp + c + 4);
  }
  for (; g < groups; g += gridDim.x) {
    const int gn = g + gridDim.x;
    uint4 nxt[kR][kChunks];
    if (gn < groups) load_group(gn, nxt);
    float mean[kR], rstd[kR];
#pragma unroll
    for (int r = 0; r < kR; ++r) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < kChunks; ++i) {
        float f[8];
        unpack8(buf[r][i], f);
#pragma unroll
        for (int j = 0; j < 8; ++j) s += f[j];
      }
      s = warp_sum(s);
      if (lane == 0) red[0][r][warp] = s;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kR; ++r) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) s += red[0][r][w];
      mean[r] = s / (float)d;
      float v = 0.f;
#pragma unroll
      for (int i = 0; i < kChunks; ++i) {
        float f[8];
        unpack8(buf[r][i], f);
#pragma unroll
        for (int j = 0; j < 8; ++j) { const float u = f[j] - mean[r]; v += u * u; }
      }
      v = warp_sum(v);
      if (lane == 0) red[1][r][warp] = v;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kR; ++r) {
      float v = 0.f;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) v += red[1][r][w];
      rstd[r] = rsqrtf(v / (float)d + eps);
    }
#pragma unroll
    for (int r = 0; r < kR; ++r) {
      if (g * kR + r >= rows) break;
      uint4* op = reinterpret_cast<uint4*>(ob + (long long)(g * kR + r) * o_rs);
#pragma unroll
      for (int i = 0; i < kChunks; ++i) {
        float f[8];
        unpack8(buf[r][i], f);
        const float4 c0 = smod[0][2 * i][t], c1 = smod[0][2 * i + 1][t], h0 = smod[1][2 * i][t], h1 = smod[1][2 * i + 1][t];
        const float s8[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
        const float h8[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = (f[j] - mean[r]) * rstd[r] * (1.f + s8[j]) + h8[j];
        op[t + kThreads * i] = pack8(f);
      }
    }
    if (gn < groups) {
#pragma unroll
      for (int r = 0; r < kR; ++r)
#pragma unroll
        for (int i = 0; i < kChunks; ++i) buf[r][i] = nxt[r][i];
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Per-head RMSNorm (learned weight) + interleaved-pair RoPE, in place. One warp per token row, looping heads.
// ---------------------------------------------------------------------------------------------------
template <int kDh>
__global__ void __launch_bounds__(256) qk_rmsnorm_rope_kernel(__nv_bfloat16* __restrict__ x, long long rs, long long bs,
                                                              int batch, int rows, int heads,
                                                              const __nv_bfloat16* __restrict__ w, int heads_per_weight,
                                                              float eps, const float* __restrict__ cos_sin) {
  // 16 bytes (8 elements) per lane: a head spans LPH lanes, a warp covers HPW heads per pass; kUnroll passes are
  // loaded before any is reduced so that enough bytes are in flight to approach HBM bandwidth.
  constexpr int LPH = kDh / 8, HPW = 32 / LPH, kUnroll = 4;
  // one warp per (row, chunk of HPW * kUnroll heads): more warps (and 16-byte accesses) in flight than one warp per row
  const int chunks = (heads + HPW * kUnroll - 1) / (HPW * kUnroll);
  const long long wg = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (wg >= (long long)batch * rows * chunks) return;
  const int chunk = (int)(wg % chunks);
  const int warp_global = (int)(wg / chunks);
  const int b = warp_global / rows, r = warp_global % rows;
  __nv_bfloat16* row = x + (long long)b * bs + (long long)r * rs;
  const int sub = lane / LPH, e0 = (lane % LPH) * 8;  // head slot inside the pass, first element inside the head
  float cs[4], sn[4];
  if (cos_sin) {
    const float* t = cos_sin + (long long)r * kDh + e0;  // [rows, dh/2, 2]: (cos, sin) of pair
    const float4 t0 = *reinterpret_cast<const float4*>(t), t1 = *reinterpret_cast<const float4*>(t + 4);
    cs[0] = t0.x; sn[0] = t0.y; cs[1] = t0.z; sn[1] = t0.w; cs[2] = t1.x; sn[2] = t1.y; cs[3] = t1.z; sn[3] = t1.w;
  }
  {
    const int h0 = chunk * HPW * kUnroll;
    uint4 u[kUnroll];
#pragma unroll
    for (int k = 0; k < kUnroll; ++k) {
      const int h = h0 + k * HPW + sub;
      if (h < heads) u[k] = *reinterpret_cast<const uint4*>(row + h * kDh + e0);
    }
#pragma unroll
    for (int k = 0; k < kUnroll; ++k) {
      const int h = h0 + k * HPW + sub;
      const bool on = h < heads;
      float f[8];
      if (on) unpack8(u[k], f);
      else {
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] = 0.f;
      }
      float ss = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) ss += f[i] * f[i];
#pragma unroll
      for (int o = LPH / 2; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
      if (on) {
        const float rstd = rsqrtf(ss / (float)kDh + eps);
        float wf[8];
        unpack8(*reinterpret_cast<const uint4*>(w + (h / heads_per_weight) * kDh + e0), wf);
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] = f[i] * rstd * wf[i];
        if (cos_sin) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float x0 = f[2 * q], x1 = f[2 * q + 1];
            f[2 * q] = x0 * cs[q] - x1 * sn[q];
            f[2 * q + 1] = x1 * cs[q] + x0 * sn[q];
          }
        }
        *reinterpret_cast<uint4*>(row + h * kDh + e0) = pack8(f);
      }
    }
  }
}

// FluxPosEmbed: per axis a, pair j: angle = ids[r,a] / theta^(2j/d_a) in float64; table holds (cos, sin) per pair.
__global__ void rope_table_kernel(const float* __restrict__ ids, int rows, int d0, int d1, int d2, float theta,
                                  float* __restrict__ cos_sin) {
  const int half = (d0 + d1 + d2) / 2;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * half) return;
  const int r = idx / half;
  int j = idx % half;
  int axis, da;
  if (j < d0 / 2) { axis = 0; da = d0; }
  else if (j < (d0 + d1) / 2) { axis = 1; da = d1; j -= d0 / 2; }
  else { axis = 2; da = d2; j -= (d0 + d1) / 2; }
  const double pos = (double)ids[r * 3 + axis];
  const double freq = 1.0 / pow((double)theta, (double)(2 * j) / (double)da);
  const double ang = pos * freq;
  cos_sin[2 * idx] = (float)cos(ang);
  cos_sin[2 * idx + 1] = (float)sin(ang);
}

// ---------------------------------------------------------------------------------------------------
// Small-M linear: one warp computes kRowsPerWarp output features for up to kB batch rows, streaming W once.
// Algorithmic HBM bytes: 2*n*k (weights) — x and out are negligible.
// ---------------------------------------------------------------------------------------------------
template <int kB>
__global__ void __launch_bounds__(256) gemv_kernel(const float* __restrict__ x, long long x_stride,
                                                   const __nv_bfloat16* __restrict__ w,
                                                   const __nv_bfloat16* __restrict__ bias, float* __restrict__ out,
                                                   long long out_stride, int batch0, int batch, int n, int k,
                                                   int silu_in, int silu_out, int accumulate) {
  constexpr int kRows = 4;
  const int warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int n0 = warp_global * kRows;
  if (n0 >= n) return;
  float acc[kRows][kB];
#pragma unroll
  for (int i = 0; i < kRows; ++i)
#pragma unroll
    for (int b = 0; b < kB; ++b) acc[i][b] = 0.f;
  const int nb = min(kB, batch - batch0);
  for (int kk = lane * 8; kk < k; kk += 256) {
    float xv[kB][8];
#pragma unroll
    for (int b = 0; b < kB; ++b) {
      if (b < nb) {
        const float* xp = x + (long long)(batch0 + b) * x_stride + kk;
        const float4 a = *reinterpret_cast<const float4*>(xp), c = *reinterpret_cast<const float4*>(xp + 4);
        xv[b][0] = a.x; xv[b][1] = a.y; xv[b][2] = a.z; xv[b][3] = a.w;
        xv[b][4] = c.x; xv[b][5] = c.y; xv[b][6] = c.z; xv[b][7] = c.w;
        if (silu_in) {
#pragma unroll
          for (int j = 0; j < 8; ++j) xv[b][j] = xv[b][j] / (1.f + expf(-xv[b][j]));
        }
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) xv[b][j] = 0.f;
      }
    }
#pragma unroll
    for (int i = 0; i < kRows; ++i) {
      if (n0 + i < n) {
        const uint4 wv = *reinterpret_cast<const uint4*>(w + (long long)(n0 + i) * k + kk);
        float wf[8];
        unpack8(wv, wf);
#pragma unroll
        for (int b = 0; b < kB; ++b)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[i][b] += wf[j] * xv[b][j];
      }
    }
  }
#pragma unroll
  for (int i = 0; i < kRows; ++i)
#pragma unroll
    for (int b = 0; b < kB; ++b) acc[i][b] = warp_sum(acc[i][b]);
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < kRows; ++i) {
      if (n0 + i >= n) continue;
      const float bv = bias ? __bfloat162float(bias[n0 + i]) : 0.f;
#pragma unroll
      for (int b = 0; b < kB; ++b) {
        if (b >= nb) continue;
        float v = acc[i][b] + bv;
        if (silu_out) v = v / (1.f + expf(-v));
        float* o = out + (long long)(batch0 + b) * out_stride + n0 + i;
        *o = accumulate ? (*o + v) : v;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Grouped small-M linear: ONE launch streams the weights of MANY independent linears (every AdaLN `linear(silu(temb))` of a
// denoise step: 117 matrices, ~10 GB of bf16 at cfg3) at HBM speed. The per-linear launches of gemv_kernel covered 4608
// warps each (< 1 wave of a B200) and paid a launch + tail per 57-113 MB; here a grid that fills every SM walks the
// concatenated list of 4-row groups of all jobs, 16 independent 16-byte weight loads in flight per lane (batch 1).
// With a peer table the output rows are stored into EVERY rank's pool (job.out = byte offset): the sequence-parallel ranks
// each compute 1/P of the groups and the table is all-gathered by the stores themselves.
// ---------------------------------------------------------------------------------------------------
struct GemvPeers {
  int world, rank;
  uint8_t* base[UG_MAX_PEERS];
};

// U consecutive 256-element K chunks of 4 weight rows: all 4 * U 16-byte loads are issued before the first FMA.
template <int kB, int U>
__device__ __forceinline__ void gemv_chunks(const __nv_bfloat16* __restrict__ w0, const __nv_bfloat16* __restrict__ w1,
                                            const __nv_bfloat16* __restrict__ w2, const __nv_bfloat16* __restrict__ w3,
                                            const float* __restrict__ x, long long x_stride, int kk, int batch, bool silu_in,
                                            float (&acc)[4][kB]) {
  uint4 wv[U][4];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    wv[u][0] = *reinterpret_cast<const uint4*>(w0 + kk + 256 * u);
    wv[u][1] = *reinterpret_cast<const uint4*>(w1 + kk + 256 * u);
    wv[u][2] = *reinterpret_cast<const uint4*>(w2 + kk + 256 * u);
    wv[u][3] = *reinterpret_cast<const uint4*>(w3 + kk + 256 * u);
  }
#pragma unroll
  for (int u = 0; u < U; ++u) {
#pragma unroll
    for (int b = 0; b < kB; ++b) {
      if (b < batch) {
        const float* xp = x + (long long)b * x_stride + kk + 256 * u;
        const float4 a = *reinterpret_cast<const float4*>(xp), c = *reinterpret_cast<const float4*>(xp + 4);
        float xv[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
        if (silu_in) {
#pragma unroll
          for (int j = 0; j < 8; ++j) xv[j] = xv[j] / (1.f + expf(-xv[j]));
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float2 p0 = unpack_bf16x2(wv[u][i].x), p1 = unpack_bf16x2(wv[u][i].y), p2 = unpack_bf16x2(wv[u][i].z),
                       p3 = unpack_bf16x2(wv[u][i].w);
          acc[i][b] += p0.x * xv[0] + p0.y * xv[1] + p1.x * xv[2] + p1.y * xv[3] + p2.x * xv[4] + p2.y * xv[5] + p3.x * xv[6] +
                       p3.y * xv[7];
        }
      }
    }
  }
}

template <int kB, int kUnroll>
__global__ void __launch_bounds__(256, 2) gemv_grouped_kernel(const ug_gemv_job* __restrict__ jobs, int n_jobs, int g_begin,
                                                              int g_end, int batch, GemvPeers peers) {
  constexpr int kRows = 4;
  __shared__ int first_group[UG_MAX_GEMV_JOBS + 1];
  for (int i = threadIdx.x; i <= n_jobs; i += blockDim.x)
    first_group[i] = i < n_jobs ? jobs[i].first_group : 0x7fffffff;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int warps_total = (gridDim.x * blockDim.x) >> 5;
  for (int g = g_begin + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5); g < g_end; g += warps_total) {
    int lo = 0, hi = n_jobs - 1;  // last job whose first_group <= g
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (first_group[mid] <= g) lo = mid; else hi = mid - 1;
    }
    const ug_gemv_job* J = jobs + lo;
    const int n = J->n, k = J->k;
    const int n0 = (g - first_group[lo]) * kRows;
    // a ragged last group re-reads row n - 1 instead of predicating the loads; only rows < n are stored
    const __nv_bfloat16* wbase = reinterpret_cast<const __nv_bfloat16*>(J->w);
    const __nv_bfloat16* w0 = wbase + (long long)min(n0, n - 1) * k;
    const __nv_bfloat16* w1 = wbase + (long long)min(n0 + 1, n - 1) * k;
    const __nv_bfloat16* w2 = wbase + (long long)min(n0 + 2, n - 1) * k;
    const __nv_bfloat16* w3 = wbase + (long long)min(n0 + 3, n - 1) * k;
    const float* x = J->x;
    const long long x_stride = J->x_stride;
    const bool silu_in = (J->flags & 1) != 0;
    const bool accumulate = (J->flags & 2) != 0;
    float acc[kRows][kB];
#pragma unroll
    for (int i = 0; i < kRows; ++i)
#pragma unroll
      for (int b = 0; b < kB; ++b) acc[i][b] = 0.f;
    int kk = lane * 8;
    for (; kk + 256 * (kUnroll - 1) < k; kk += 256 * kUnroll) gemv_chunks<kB, kUnroll>(w0, w1, w2, w3, x, x_stride, kk, batch, silu_in, acc);
    for (; kk < k; kk += 256) gemv_chunks<kB, 1>(w0, w1, w2, w3, x, x_stride, kk, batch, silu_in, acc);
#pragma unroll
    for (int i = 0; i < kRows; ++i)
#pragma unroll
      for (int b = 0; b < kB; ++b) acc[i][b] = warp_sum(acc[i][b]);
    if (lane == 0) {
      const __nv_bfloat16* bias = reinterpret_cast<const __nv_bfloat16*>(J->bias);
      const long long out_stride = J->out_stride;
#pragma unroll
      for (int i = 0; i < kRows; ++i) {
        if (n0 + i >= n) continue;
        const float bv = bias ? __bfloat162float(bias[n0 + i]) : 0.f;
#pragma unroll
        for (int b = 0; b < kB; ++b) {
          if (b >= batch) continue;
          float v = acc[i][b] + bv;
          const long long off = (long long)b * out_stride + n0 + i;
          if (peers.world == 0) {
            if (accumulate) v += J->out[off];
            J->out[off] = v;
          } else {
            const long long byte_off = (long long)reinterpret_cast<uintptr_t>(J->out);
            // accumulate: the running value is this rank's OWN copy (every copy is identical after the preceding barrier)
            if (accumulate) v += reinterpret_cast<const float*>(peers.base[peers.rank] + byte_off)[off];
#pragma unroll
            for (int r = 0; r < UG_MAX_PEERS; ++r)  // constant indices: the table stays in the parameter bank
              if (r < peers.world) reinterpret_cast<float*>(peers.base[r] + byte_off)[off] = v;
          }
        }
      }
    }
  }
}

__global__ void __launch_bounds__(256) silu_f32_kernel(const float* __restrict__ x, float* __restrict__ out, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float v = x[i];
    out[i] = v / (1.f + expf(-v));
  }
}

__global__ void timestep_embedding_kernel(const float* __restrict__ t, long long t_stride, int batch, int dim, float scale,
                                          float* __restrict__ out) {
  const int half = dim / 2;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= batch * half) return;
  const int b = idx / half, j = idx % half;
  // exponent = -ln(10000) * j / (half - downscale_freq_shift), downscale_freq_shift = 0
  const float freq = expf(-logf(10000.f) * (float)j / (float)half);
  const float a = (t[(long long)b * t_stride] * scale) * freq;
  // flip_sin_to_cos=True -> [cos | sin]
  out[b * dim + j] = cosf(a);
  out[b * dim + half + j] = sinf(a);
}

template <bool kAdd>
__global__ void __launch_bounds__(256) rows_kernel(const __nv_bfloat16* __restrict__ a, long long a_rs, long long a_bs,
                                                   const __nv_bfloat16* __restrict__ b2, long long b_rs, long long b_bs,
                                                   __nv_bfloat16* __restrict__ out, long long o_rs, long long o_bs,
                                                   int batch, int rows, int d) {
  const int nvec = d >> 3;
  const long long total = (long long)batch * rows * nvec;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % nvec);
    const long long rr = i / nvec;
    const int r = (int)(rr % rows), b = (int)(rr / rows);
    uint4 u = *reinterpret_cast<const uint4*>(a + b * a_bs + r * a_rs + 8 * v);
    if constexpr (kAdd) {
      const uint4 w = *reinterpret_cast<const uint4*>(b2 + b * b_bs + r * b_rs + 8 * v);
      float f[8], g[8];
      unpack8(u, f);
      unpack8(w, g);
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] += g[j];
      u = pack8(f);
    }
    *reinterpret_cast<uint4*>(out + b * o_bs + r * o_rs + 8 * v) = u;
  }
}

__global__ void cast_f32_bf16_kernel(const float* __restrict__ s, __nv_bfloat16* __restrict__ d, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    d[i] = __float2bfloat16(s[i]);
}
__global__ void cast_bf16_f32_kernel(const __nv_bfloat16* __restrict__ s, float* __restrict__ d, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    d[i] = __bfloat162float(s[i]);
}

// x[r,:] += gate[e(r), idx(r), :] * y[r,:] on capacity-slot buffers (per-token AdaLN gates of the SD3 experts)
__global__ void __launch_bounds__(256) gated_add_slots_kernel(__nv_bfloat16* __restrict__ x, long long x_rs,
                                                              const __nv_bfloat16* __restrict__ y, long long y_rs,
                                                              const float* __restrict__ gate, long long mod_es, long long mod_bs,
                                                              const int* __restrict__ slot_token, int rows, int capacity,
                                                              int tokens_per_batch, int empty_index, int d) {
  const int nvec = d >> 3;
  const long long total = (long long)rows * nvec;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % nvec);
    const int r = (int)(i / nvec);
    const int token = slot_token[r];
    const float* g = gate + (long long)(r / capacity) * mod_es +
                     (long long)(token < 0 ? empty_index : token / tokens_per_batch) * mod_bs + 8 * v;
    const float4 g0 = *reinterpret_cast<const float4*>(g), g1 = *reinterpret_cast<const float4*>(g + 4);
    const float gv[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
    float xf[8], yf[8];
    unpack8(*reinterpret_cast<const uint4*>(x + (long long)r * x_rs + 8 * v), xf);
    unpack8(*reinterpret_cast<const uint4*>(y + (long long)r * y_rs + 8 * v), yf);
#pragma unroll
    for (int j = 0; j < 8; ++j) xf[j] += gv[j] * yf[j];
    *reinterpret_cast<uint4*>(x + (long long)r * x_rs + 8 * v) = pack8(xf);
  }
}

// UG_LN_KERNEL=stream|rows|warp: A/B switch between the persistent prefetching kernel (default), the one-group-per-block kernel
// (bit-identical to it) and the one / two-warps-per-row kernels
static inline int ln_kernel_choice() {
  static int cached = -1;
  if (cached < 0) {
    const char* e = getenv("UG_LN_KERNEL");
    cached = (e && strcmp(e, "warp") == 0) ? 0 : (e && strcmp(e, "rows") == 0) ? 1 : 2;
  }
  return cached;
}
static inline bool ln_rows_kernel_enabled() { return ln_kernel_choice() >= 1; }

static inline int grid_for(long long threads, int block) {
  long long g = (threads + block - 1) / block;
  const long long cap = (long long)num_sms() * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}
static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace ug

using namespace ug;

static int launch_ln_modulate(const void* x, int64_t x_rs, int64_t x_bs, void* out, int64_t o_rs, int64_t o_bs,
                              const float* shift, const float* scale, int64_t mod_bs, int32_t batch, int32_t rows, int32_t d,
                              float eps, const int32_t* slot_token, int32_t capacity, int32_t tokens_per_batch,
                              int32_t empty_index, int64_t mod_es, void* stream, const char* name,
                              ug::RowSegs segs = ug::RowSegs{0, {0}}, int64_t mod_seg_stride = 0,
                              ug::Fp8Out fo = ug::Fp8Out{nullptr, 0, 0, nullptr, 0}) {
  const bool fp8 = fo.q != nullptr;  // ln_modulate_fp8: e4m3 rows + scales instead of `out` (same kernel choice, same bits)
  UG_CHECK_ARG(x && out && shift && scale, "%s: null pointer", name);
  UG_CHECK_ARG(batch >= 1 && rows >= 1 && d >= 8 && d % 8 == 0, "%s: bad shape batch %d rows %d d %d", name, batch, rows, d);
  UG_CHECK_ARG(x_rs % 8 == 0 && o_rs % 8 == 0 && x_bs % 8 == 0 && o_bs % 8 == 0 && mod_bs % 4 == 0 && mod_es % 4 == 0 &&
                   aligned16(x) && aligned16(out) && aligned16(shift) && aligned16(scale),
               "%s: operands must be 16-byte aligned", name);
  if (d > 8 * 32 * 16) {
    set_error("%s: d = %d exceeds the register-resident row limit (4096)", name, d);
    return UG_ERR_UNSUPPORTED;
  }
  const long long warps = (long long)batch * rows;
  const int block = 256;
  const int grid = (int)((warps * 32 + block - 1) / block);
  auto s = reinterpret_cast<cudaStream_t>(stream);
  auto xp = (const __nv_bfloat16*)x;
  auto op = (__nv_bfloat16*)out;
  if (!slot_token && segs.nseg == 0 && ln_rows_kernel_enabled() && batch <= 65535) {
    // plain per-sample form: kR rows per block share one load of the modulation vectors
    constexpr int kR = 4;
    const dim3 g((unsigned)((rows + kR - 1) / kR), (unsigned)batch);
    const int nvec = d >> 3;
    bool done = true;
    // (the persistent kernel is bit-identical to the one-group-per-block kernel: the fp8 form uses the latter)
    if (!fp8 && ln_kernel_choice() == 2 && nvec == 3 * 128 && (long long)g.x * batch > 2LL * num_sms()) {
      // persistent: two blocks per SM over all samples, each walking its row groups with the next group's rows in flight
      const dim3 gp((unsigned)std::max(1, std::min((int)g.x, (2 * num_sms() + batch - 1) / batch)), (unsigned)batch);
      ln_modulate_stream_kernel<128, 3, kR><<<gp, 128, 0, s>>>(xp, x_rs, x_bs, op, o_rs, o_bs, shift, scale, mod_bs, rows, d, eps);
    } else
#define UG_LN_ROWS(T, C)                                                                                                 \
  do {                                                                                                                   \
    if (fp8) ln_modulate_rows_kernel<T, C, kR, true><<<g, T, 0, s>>>(xp, x_rs, x_bs, op, o_rs, o_bs, shift, scale, mod_bs, rows, d, eps, fo); \
    else ln_modulate_rows_kernel<T, C, kR><<<g, T, 0, s>>>(xp, x_rs, x_bs, op, o_rs, o_bs, shift, scale, mod_bs, rows, d, eps);            \
  } while (0)
    if (nvec == 3 * 128) UG_LN_ROWS(128, 3);
    else if (nvec == 3 * 64) UG_LN_ROWS(64, 3);
    else if (nvec == 2 * 128) UG_LN_ROWS(128, 2);
    else done = false;
#undef UG_LN_ROWS
    if (done) {
      UG_CHECK_LAUNCH(name);
      return UG_OK;
    }
  }
#define UG_LN_LAUNCH(V)                                                                                                           \
  do {                                                                                                                            \
    if (fp8) ln_modulate_kernel<V, true><<<grid, block, 0, s>>>(xp, x_rs, x_bs, op, o_rs, o_bs, shift, scale, mod_bs, batch, rows, d, eps, slot_token, capacity, tokens_per_batch, empty_index, mod_es, segs, mod_seg_stride, fo); \
    else ln_modulate_kernel<V><<<grid, block, 0, s>>>(xp, x_rs, x_bs, op, o_rs, o_bs, shift, scale, mod_bs, batch, rows, d, eps, slot_token, capacity, tokens_per_batch, empty_index, mod_es, segs, mod_seg_stride); \
  } while (0)
  const int grid2 = (int)((warps + 3) / 4);  // two warps per row, four rows per 256-thread block
#define UG_LN2_LAUNCH(V)                                                                                                          \
  do {                                                                                                                            \
    if (fp8) ln_modulate2_kernel<V, true><<<grid2, block, 0, s>>>(xp, x_rs, x_bs, op, o_rs, o_bs, shift, scale, mod_bs, batch, rows, d, eps, slot_token, capacity, tokens_per_batch, empty_index, mod_es, segs, mod_seg_stride, fo); \
    else ln_modulate2_kernel<V><<<grid2, block, 0, s>>>(xp, x_rs, x_bs, op, o_rs, o_bs, shift, scale, mod_bs, batch, rows, d, eps, slot_token, capacity, tokens_per_batch, empty_index, mod_es, segs, mod_seg_stride); \
  } while (0)
  if (d <= 8 * 32 * 2) UG_LN_LAUNCH(2);
  else if (d <= 8 * 64 * 3) UG_LN2_LAUNCH(3);
  else if (d <= 8 * 64 * 6) UG_LN2_LAUNCH(6);
  else if (d <= 8 * 32 * 12) UG_LN_LAUNCH(12);
  else UG_LN_LAUNCH(16);
#undef UG_LN2_LAUNCH
#undef UG_LN_LAUNCH
  UG_CHECK_LAUNCH(name);
  return UG_OK;
}

extern "C" int ug_ln_modulate(const void* x, int64_t x_rs, int64_t x_bs, void* out, int64_t o_rs, int64_t o_bs,
                              const float* shift, const float* scale, int64_t mod_bs, int32_t batch, int32_t rows,
                              int32_t d, float eps, void* stream) {
  return launch_ln_modulate(x, x_rs, x_bs, out, o_rs, o_bs, shift, scale, mod_bs, batch, rows, d, eps, nullptr, 1, 1, 0, 0, stream,
                            "ln_modulate");
}

extern "C" int ug_ln_modulate_fp8(const void* x, int64_t x_rs, int64_t x_bs, void* q, int64_t q_rs, int64_t q_bs, float* q_scale,
                                  int64_t q_scale_bs, const float* shift, const float* scale, int64_t mod_bs, int32_t batch,
                                  int32_t rows, int32_t d, float eps, void* stream) {
  UG_CHECK_ARG(q && q_scale, "ln_modulate_fp8: null output pointer");
  UG_CHECK_ARG((reinterpret_cast<uintptr_t>(q) & 7) == 0 && q_rs % 8 == 0 && q_bs % 8 == 0 && (reinterpret_cast<uintptr_t>(q_scale) & 3) == 0,
               "ln_modulate_fp8: e4m3 rows must be 8-byte aligned");
  UG_CHECK_ARG(batch == 1 || q_bs >= (int64_t)rows * q_rs, "ln_modulate_fp8: overlapping output batches");
  // `out` is never written in the fp8 form: the input pointer stands in for it in the shared argument checks
  return launch_ln_modulate(x, x_rs, x_bs, const_cast<void*>(x), x_rs, x_bs, shift, scale, mod_bs, batch, rows, d, eps, nullptr, 1, 1,
                            0, 0, stream, "ln_modulate_fp8", ug::RowSegs{0, {0}}, 0,
                            ug::Fp8Out{static_cast<uint8_t*>(q), q_rs, q_bs, q_scale, q_scale_bs});
}

extern "C" int ug_quant_rows_fp8(const void* x, int64_t x_rs, int64_t x_bs, void* q, int64_t q_rs, int64_t q_bs, float* scale,
                                 int64_t scale_bs, int32_t batch, int32_t rows, int32_t k, void* stream) {
  UG_CHECK_ARG(x && q && scale, "quant_rows_fp8: null pointer");
  UG_CHECK_ARG(batch >= 1 && batch <= 65535 && rows >= 1 && k >= 8 && k % 8 == 0, "quant_rows_fp8: bad shape batch %d rows %d k %d",
               batch, rows, k);
  UG_CHECK_ARG(aligned16(x) && x_rs % 8 == 0 && x_bs % 8 == 0 && (reinterpret_cast<uintptr_t>(q) & 7) == 0 && q_rs % 8 == 0 &&
                   q_bs % 8 == 0 && (reinterpret_cast<uintptr_t>(scale) & 3) == 0,
               "quant_rows_fp8: bf16 rows must be 16-byte, e4m3 rows 8-byte aligned");
  if (k > 8 * 256 * 8) {
    set_error("quant_rows_fp8: k = %d exceeds the register-resident row limit (16384)", k);
    return UG_ERR_UNSUPPORTED;
  }
  auto s = reinterpret_cast<cudaStream_t>(stream);
  const ug::Fp8Out o{static_cast<uint8_t*>(q), q_rs, q_bs, scale, scale_bs};
  const dim3 g((unsigned)rows, (unsigned)batch);
  auto xp = (const __nv_bfloat16*)x;
  if (k <= 8 * 128 * 4) quant_rows_fp8_kernel<128, 4><<<g, 128, 0, s>>>(xp, x_rs, x_bs, o, k);
  else quant_rows_fp8_kernel<256, 8><<<g, 256, 0, s>>>(xp, x_rs, x_bs, o, k);
  UG_CHECK_LAUNCH("quant_rows_fp8");
  return UG_OK;
}

extern "C" int ug_ln_modulate_segs(const void* x, int64_t x_rs, int64_t x_bs, void* out, int64_t o_rs, int64_t o_bs,
                                   const float* shift, const float* scale, int64_t mod_bs, int64_t mod_seg_stride, int32_t nseg,
                                   const int32_t* seg_bounds, int32_t batch, int32_t rows, int32_t d, float eps, void* stream) {
  UG_CHECK_ARG(seg_bounds && nseg >= 1 && nseg <= UG_MAX_SEGMENTS && mod_seg_stride % 4 == 0, "ln_modulate_segs: bad segment table");
  ug::RowSegs segs;
  segs.nseg = nseg;
  for (int i = 0; i <= UG_MAX_SEGMENTS; ++i) segs.bounds[i] = i <= nseg ? seg_bounds[i] : rows;
  return launch_ln_modulate(x, x_rs, x_bs, out, o_rs, o_bs, shift, scale, mod_bs, batch, rows, d, eps, nullptr, 1, 1, 0, 0, stream,
                            "ln_modulate_segs", segs, mod_seg_stride);
}

extern "C" int ug_ln_modulate_segs_fp8(const void* x, int64_t x_rs, int64_t x_bs, void* q, int64_t q_rs, int64_t q_bs, float* q_scale,
                                       int64_t q_scale_bs, const float* shift, const float* scale, int64_t mod_bs,
                                       int64_t mod_seg_stride, int32_t nseg, const int32_t* seg_bounds, int32_t batch, int32_t rows,
                                       int32_t d, float eps, void* stream) {
  UG_CHECK_ARG(seg_bounds && nseg >= 1 && nseg <= UG_MAX_SEGMENTS && mod_seg_stride % 4 == 0, "ln_modulate_segs_fp8: bad segment table");
  UG_CHECK_ARG(q && q_scale, "ln_modulate_segs_fp8: null output pointer");
  UG_CHECK_ARG((reinterpret_cast<uintptr_t>(q) & 7) == 0 && q_rs % 8 == 0 && q_bs % 8 == 0 && (reinterpret_cast<uintptr_t>(q_scale) & 3) == 0,
               "ln_modulate_segs_fp8: e4m3 rows must be 8-byte aligned");
  UG_CHECK_ARG(batch == 1 || q_bs >= (int64_t)rows * q_rs, "ln_modulate_segs_fp8: overlapping output batches");
  ug::RowSegs segs;
  segs.nseg = nseg;
  for (int i = 0; i <= UG_MAX_SEGMENTS; ++i) segs.bounds[i] = i <= nseg ? seg_bounds[i] : rows;
  // `out` is never written in the fp8 form: the input pointer stands in for it in the shared argument checks
  return launch_ln_modulate(x, x_rs, x_bs, const_cast<void*>(x), x_rs, x_bs, shift, scale, mod_bs, batch, rows, d, eps, nullptr, 1, 1,
                            0, 0, stream, "ln_modulate_segs_fp8", segs, mod_seg_stride,
                            ug::Fp8Out{static_cast<uint8_t*>(q), q_rs, q_bs, q_scale, q_scale_bs});
}

extern "C" int ug_ln_modulate_slots(const void* x, int64_t x_rs, void* out, int64_t o_rs, const float* shift, const float* scale,
                                    int64_t mod_expert_stride, int64_t mod_index_stride, const int32_t* slot_token,
                                    int32_t experts, int32_t capacity, int32_t tokens_per_batch, int32_t empty_index, int32_t d,
                                    float eps, void* stream) {
  UG_CHECK_ARG(slot_token && experts >= 1 && capacity >= 1 && tokens_per_batch >= 1 && empty_index >= 0,
               "ln_modulate_slots: bad slot arguments");
  return launch_ln_modulate(x, x_rs, 0, out, o_rs, 0, shift, scale, mod_index_stride, 1, experts * capacity, d, eps, slot_token,
                            capacity, tokens_per_batch, empty_index, mod_expert_stride, stream, "ln_modulate_slots");
}

extern "C" int ug_gated_add_slots(void* x, int64_t x_rs, const void* y, int64_t y_rs, const float* gate, int64_t mod_expert_stride,
                                  int64_t mod_index_stride, const int32_t* slot_token, int32_t experts, int32_t capacity,
                                  int32_t tokens_per_batch, int32_t empty_index, int32_t d, void* stream) {
  UG_CHECK_ARG(x && y && gate && slot_token, "gated_add_slots: null pointer");
  UG_CHECK_ARG(experts >= 1 && capacity >= 1 && tokens_per_batch >= 1 && empty_index >= 0 && d >= 8 && d % 8 == 0,
               "gated_add_slots: bad shape");
  UG_CHECK_ARG(x_rs % 8 == 0 && y_rs % 8 == 0 && mod_expert_stride % 4 == 0 && mod_index_stride % 4 == 0 && aligned16(x) &&
                   aligned16(y) && aligned16(gate), "gated_add_slots: operands must be 16-byte aligned");
  const int rows = experts * capacity;
  const long long total = (long long)rows * (d >> 3);
  gated_add_slots_kernel<<<grid_for(total, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      (__nv_bfloat16*)x, x_rs, (const __nv_bfloat16*)y, y_rs, gate, mod_expert_stride, mod_index_stride, slot_token, rows, capacity,
      tokens_per_batch, empty_index, d);
  UG_CHECK_LAUNCH("gated_add_slots");
  return UG_OK;
}

extern "C" int ug_qk_rmsnorm_rope(void* x, int64_t rs, int64_t bs, int32_t batch, int32_t rows, int32_t heads,
                                  int32_t head_dim, const void* w, int32_t heads_per_weight, float eps,
                                  const float* cos_sin, void* stream) {
  UG_CHECK_ARG(x && w, "qk_rmsnorm_rope: null pointer");
  UG_CHECK_ARG(batch >= 1 && rows >= 1 && heads >= 1, "qk_rmsnorm_rope: bad shape");
  if (heads_per_weight <= 0) heads_per_weight = heads;
  UG_CHECK_ARG(rs % 8 == 0 && bs % 8 == 0 && aligned16(x) && aligned16(w) && (!cos_sin || aligned16(cos_sin)), "qk_rmsnorm_rope: alignment");
  const int heads_per_warp = (32 / (head_dim >= 8 ? head_dim / 8 : 1)) * 4;
  const long long warps = (long long)batch * rows * ((heads + heads_per_warp - 1) / heads_per_warp);
  const int block = 256;
  const int grid = (int)((warps * 32 + block - 1) / block);
  auto s = reinterpret_cast<cudaStream_t>(stream);
  if (head_dim == 128)
    qk_rmsnorm_rope_kernel<128><<<grid, block, 0, s>>>((__nv_bfloat16*)x, rs, bs, batch, rows, heads, (const __nv_bfloat16*)w, heads_per_weight, eps, cos_sin);
  else if (head_dim == 64)
    qk_rmsnorm_rope_kernel<64><<<grid, block, 0, s>>>((__nv_bfloat16*)x, rs, bs, batch, rows, heads, (const __nv_bfloat16*)w, heads_per_weight, eps, cos_sin);
  else {
    set_error("qk_rmsnorm_rope: head_dim %d not supported (64 or 128)", head_dim);
    return UG_ERR_UNSUPPORTED;
  }
  UG_CHECK_LAUNCH("qk_rmsnorm_rope");
  return UG_OK;
}

extern "C" int ug_rope_table(const float* ids, int32_t rows, const int32_t* axes, float theta, float* cos_sin, void* stream) {
  UG_CHECK_ARG(ids && axes && cos_sin && rows >= 1, "rope_table: bad arguments");
  UG_CHECK_ARG(axes[0] % 2 == 0 && axes[1] % 2 == 0 && axes[2] % 2 == 0, "rope_table: axes dims must be even");
  const int half = (axes[0] + axes[1] + axes[2]) / 2;
  const long long total = (long long)rows * half;
  rope_table_kernel<<<(int)((total + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(ids, rows, axes[0], axes[1], axes[2], theta, cos_sin);
  UG_CHECK_LAUNCH("rope_table");
  return UG_OK;
}

extern "C" int ug_gemv(const float* x, int64_t x_stride, const void* w, const void* bias, float* out, int64_t out_stride,
                       int32_t batch, int32_t n, int32_t k, int32_t silu_in, int32_t silu_out, int32_t accumulate,
                       void* stream) {
  UG_CHECK_ARG(x && w && out, "gemv: null pointer");
  UG_CHECK_ARG(batch >= 1 && n >= 1 && k >= 8 && k % 8 == 0, "gemv: bad shape batch %d n %d k %d", batch, n, k);
  UG_CHECK_ARG(x_stride % 4 == 0 && aligned16(x) && aligned16(w), "gemv: x / w must be 16-byte aligned");
  auto s = reinterpret_cast<cudaStream_t>(stream);
  const int warps = (n + 3) / 4;
  const int block = 256;
  const int grid = (warps * 32 + block - 1) / block;
  auto wp = (const __nv_bfloat16*)w;
  auto bp = (const __nv_bfloat16*)bias;
  for (int b0 = 0; b0 < batch; b0 += 8) {
    const int nb = batch - b0;
    if (nb == 1) gemv_kernel<1><<<grid, block, 0, s>>>(x, x_stride, wp, bp, out, out_stride, b0, batch, n, k, silu_in, silu_out, accumulate);
    else if (nb == 2) gemv_kernel<2><<<grid, block, 0, s>>>(x, x_stride, wp, bp, out, out_stride, b0, batch, n, k, silu_in, silu_out, accumulate);
    else if (nb <= 4) gemv_kernel<4><<<grid, block, 0, s>>>(x, x_stride, wp, bp, out, out_stride, b0, batch, n, k, silu_in, silu_out, accumulate);
    else gemv_kernel<8><<<grid, block, 0, s>>>(x, x_stride, wp, bp, out, out_stride, b0, batch, n, k, silu_in, silu_out, accumulate);
    UG_CHECK_LAUNCH("gemv");
  }
  return UG_OK;
}

extern "C" int ug_gemv_grouped(const ug_gemv_job* jobs_dev, int32_t n_jobs, int32_t total_groups, int32_t batch, int32_t group_begin,
                               int32_t group_end, const ug_peer_table* peers, void* stream) {
  UG_CHECK_ARG(jobs_dev && n_jobs >= 1 && n_jobs <= UG_MAX_GEMV_JOBS, "gemv_grouped: need 1..%d jobs (got %d)", UG_MAX_GEMV_JOBS, n_jobs);
  UG_CHECK_ARG(batch >= 1 && batch <= 8, "gemv_grouped: batch %d outside [1, 8]", batch);
  UG_CHECK_ARG(group_begin >= 0 && group_begin <= group_end && group_end <= total_groups, "gemv_grouped: group range [%d, %d) outside [0, %d)",
               group_begin, group_end, total_groups);
  UG_CHECK_ARG((reinterpret_cast<uintptr_t>(jobs_dev) & 7) == 0, "gemv_grouped: job table must be 8-byte aligned");
  if (group_begin == group_end) return UG_OK;
  ug::GemvPeers pp;
  pp.world = 0;
  pp.rank = 0;
  for (int i = 0; i < UG_MAX_PEERS; ++i) pp.base[i] = nullptr;
  if (peers) {
    UG_CHECK_ARG(peers->world >= 1 && peers->world <= UG_MAX_PEERS, "gemv_grouped: bad peer world %d", peers->world);
    UG_CHECK_ARG(peers->rank >= 0 && peers->rank < peers->world, "gemv_grouped: bad peer rank %d", peers->rank);
    pp.world = peers->world;
    pp.rank = peers->rank;
    for (int i = 0; i < peers->world; ++i) {
      UG_CHECK_ARG(peers->base[i], "gemv_grouped: null peer base %d", i);
      pp.base[i] = reinterpret_cast<uint8_t*>(peers->base[i]);
    }
  }
  const int groups = group_end - group_begin;
  const int warps_per_block = 8;
  int grid = (groups + warps_per_block - 1) / warps_per_block;
  const int cap = num_sms() * 2;  // 2 resident blocks of 256 threads per SM (launch bounds of the kernel: up to 128 registers)
  if (grid > cap) grid = cap;
  auto s = reinterpret_cast<cudaStream_t>(stream);
  if (batch == 1) gemv_grouped_kernel<1, 4><<<grid, 256, 0, s>>>(jobs_dev, n_jobs, group_begin, group_end, batch, pp);
  else if (batch == 2) gemv_grouped_kernel<2, 2><<<grid, 256, 0, s>>>(jobs_dev, n_jobs, group_begin, group_end, batch, pp);
  else if (batch <= 4) gemv_grouped_kernel<4, 1><<<grid, 256, 0, s>>>(jobs_dev, n_jobs, group_begin, group_end, batch, pp);
  else gemv_grouped_kernel<8, 1><<<grid, 256, 0, s>>>(jobs_dev, n_jobs, group_begin, group_end, batch, pp);
  UG_CHECK_LAUNCH("gemv_grouped");
  return UG_OK;
}

extern "C" int ug_silu_f32(const float* x, float* out, int64_t n, void* stream) {
  UG_CHECK_ARG(x && out && n >= 1, "silu_f32: bad arguments");
  silu_f32_kernel<<<grid_for(n, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(x, out, n);
  UG_CHECK_LAUNCH("silu_f32");
  return UG_OK;
}

extern "C" int ug_timestep_embedding(const float* t, int64_t t_stride, int32_t batch, int32_t dim, float scale, float* out,
                                     void* stream) {
  UG_CHECK_ARG(t && out && batch >= 1 && dim >= 2 && dim % 2 == 0 && t_stride >= 0, "timestep_embedding: bad arguments");
  const int total = batch * dim / 2;
  timestep_embedding_kernel<<<(total + 127) / 128, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(t, t_stride, batch, dim, scale, out);
  UG_CHECK_LAUNCH("timestep_embedding");
  return UG_OK;
}

static int rows_op(bool add, const void* a, int64_t a_rs, int64_t a_bs, const void* b, int64_t b_rs, int64_t b_bs, void* out,
                   int64_t o_rs, int64_t o_bs, int32_t batch, int32_t rows, int32_t d, void* stream, const char* name) {
  UG_CHECK_ARG(a && out && (!add || b), "%s: null pointer", name);
  UG_CHECK_ARG(batch >= 1 && rows >= 1 && d >= 8 && d % 8 == 0, "%s: bad shape", name);
  UG_CHECK_ARG(a_rs % 8 == 0 && a_bs % 8 == 0 && o_rs % 8 == 0 && o_bs % 8 == 0 && aligned16(a) && aligned16(out), "%s: alignment", name);
  if (add) UG_CHECK_ARG(b_rs % 8 == 0 && b_bs % 8 == 0 && aligned16(b), "%s: alignment", name);
  const long long total = (long long)batch * rows * (d >> 3);
  const int grid = grid_for(total, 256);
  auto s = reinterpret_cast<cudaStream_t>(stream);
  if (add)
    rows_kernel<true><<<grid, 256, 0, s>>>((const __nv_bfloat16*)a, a_rs, a_bs, (const __nv_bfloat16*)b, b_rs, b_bs, (__nv_bfloat16*)out, o_rs, o_bs, batch, rows, d);
  else
    rows_kernel<false><<<grid, 256, 0, s>>>((const __nv_bfloat16*)a, a_rs, a_bs, nullptr, 0, 0, (__nv_bfloat16*)out, o_rs, o_bs, batch, rows, d);
  UG_CHECK_LAUNCH(name);
  return UG_OK;
}

extern "C" int ug_add_bf16(const void* a, int64_t a_rs, int64_t a_bs, const void* b, int64_t b_rs, int64_t b_bs, void* out,
                           int64_t o_rs, int64_t o_bs, int32_t batch, int32_t rows, int32_t d, void* stream) {
  return rows_op(true, a, a_rs, a_bs, b, b_rs, b_bs, out, o_rs, o_bs, batch, rows, d, stream, "add_bf16");
}
extern "C" int ug_copy_bf16(const void* src, int64_t s_rs, int64_t s_bs, void* dst, int64_t d_rs, int64_t d_bs, int32_t batch,
                            int32_t rows, int32_t d, void* stream) {
  return rows_op(false, src, s_rs, s_bs, nullptr, 0, 0, dst, d_rs, d_bs, batch, rows, d, stream, "copy_bf16");
}
extern "C" int ug_cast_f32_to_bf16(const float* src, void* dst, int64_t n, void* stream) {
  UG_CHECK_ARG(src && dst && n >= 1, "cast_f32_to_bf16: bad arguments");
  cast_f32_bf16_kernel<<<grid_for(n, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(src, (__nv_bfloat16*)dst, n);
  UG_CHECK_LAUNCH("cast_f32_to_bf16");
  return UG_OK;
}
extern "C" int ug_cast_bf16_to_f32(const void* src, float* dst, int64_t n, void* stream) {
  UG_CHECK_ARG(src && dst && n >= 1, "cast_bf16_to_f32: bad arguments");
  cast_bf16_f32_kernel<<<grid_for(n, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>((const __nv_bfloat16*)src, dst, n);
  UG_CHECK_LAUNCH("cast_bf16_to_f32");
  return UG_OK;
}

// ---------------------------------------------------------------------------------------------------
// LoRA down-projection t[b, r, :] = x[b, r, :] @ A[g(r)]^T (fp32), the skinny half of the switched low-rank update
// whose up-projection is fused into the GEMM epilogue.  One warp per row, 4 outputs per pass.
// ---------------------------------------------------------------------------------------------------
namespace ug {
struct LoraSegs {
  int nseg;
  int bounds[UG_MAX_SEGMENTS + 1];
  int group[UG_MAX_SEGMENTS];
};
__global__ void __launch_bounds__(256) lora_down_kernel(const __nv_bfloat16* __restrict__ x, long long x_rs, long long x_bs,
                                                        const __nv_bfloat16* __restrict__ a, float* __restrict__ t,
                                                        long long t_rs, long long t_bs, int batch, int rows, int k,
                                                        int rtot, LoraSegs segs) {
  const int warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp_global >= batch * rows) return;
  const int b = warp_global / rows, r = warp_global % rows;
  int g = -1;
  for (int s = 0; s < segs.nseg; ++s)
    if (r >= segs.bounds[s] && r < segs.bounds[s + 1]) g = segs.group[s];
  float* tp = t + (long long)b * t_bs + (long long)r * t_rs;
  if (g < 0) {
    for (int j = lane; j < rtot; j += 32) tp[j] = 0.f;
    return;
  }
  const __nv_bfloat16* xr = x + (long long)b * x_bs + (long long)r * x_rs;
  const __nv_bfloat16* ag = a + (long long)g * rtot * k;
  for (int j0 = 0; j0 < rtot; j0 += 4) {
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int kk = lane * 8; kk < k; kk += 256) {
      float xf[8];
      unpack8(*reinterpret_cast<const uint4*>(xr + kk), xf);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (j0 + j < rtot) {
          float af[8];
          unpack8(*reinterpret_cast<const uint4*>(ag + (long long)(j0 + j) * k + kk), af);
#pragma unroll
          for (int i = 0; i < 8; ++i) acc[j] += xf[i] * af[i];
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[j] = warp_sum(acc[j]);
    if (lane == 0) {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (j0 + j < rtot) tp[j0 + j] = acc[j];
    }
  }
}
// Same projection, written as bf16 in the K-extension layout of ug_gemm_args.a2: [rows, groups * block], the row's own
// group block holds x @ A_g^T (first rtot columns), everything else is zero.
__global__ void __launch_bounds__(256) lora_down_wide_kernel(const __nv_bfloat16* __restrict__ x, long long x_rs, long long x_bs,
                                                             const __nv_bfloat16* __restrict__ a, __nv_bfloat16* __restrict__ t,
                                                             long long t_rs, long long t_bs, int batch, int rows, int k, int rtot,
                                                             int groups, int block, LoraSegs segs) {
  __shared__ float res_s[8][64];
  const int warp_in_block = threadIdx.x >> 5;
  const int warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp_global >= batch * rows) return;
  const int b = warp_global / rows, r = warp_global % rows;
  int g = -1;
  for (int s = 0; s < segs.nseg; ++s)
    if (r >= segs.bounds[s] && r < segs.bounds[s + 1]) g = segs.group[s];
  float* res = res_s[warp_in_block];
  if (g >= 0) {
    const __nv_bfloat16* xr = x + (long long)b * x_bs + (long long)r * x_rs;
    const __nv_bfloat16* ag = a + (long long)g * rtot * k;
    for (int j0 = 0; j0 < rtot; j0 += 4) {
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
      for (int kk = lane * 8; kk < k; kk += 256) {
        float xf[8];
        unpack8(*reinterpret_cast<const uint4*>(xr + kk), xf);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (j0 + j < rtot) {
            float af[8];
            unpack8(*reinterpret_cast<const uint4*>(ag + (long long)(j0 + j) * k + kk), af);
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[j] += xf[i] * af[i];
          }
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[j] = warp_sum(acc[j]);
      if (lane == 0) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (j0 + j < rtot) res[j0 + j] = acc[j];
      }
    }
  }
  __syncwarp();
  __nv_bfloat16* tp = t + (long long)b * t_bs + (long long)r * t_rs;
  const int width = groups * block;
  for (int c0 = lane * 8; c0 < width; c0 += 256) {
    float f[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int c = c0 + i, j = c % block;
      f[i] = (g >= 0 && c / block == g && j < rtot) ? res[j] : 0.f;
    }
    *reinterpret_cast<uint4*>(tp + c0) = pack8(f);
  }
}
}  // namespace ug

extern "C" int ug_lora_down_wide(const void* x, int64_t x_rs, int64_t x_bs, const void* a_stack, void* t_wide, int64_t t_rs,
                                 int64_t t_bs, int32_t batch, int32_t rows, int32_t k, int32_t rank_total, int32_t groups,
                                 int32_t block, int32_t nseg, const int32_t* seg_bounds, const int32_t* seg_group, void* stream) {
  UG_CHECK_ARG(x && a_stack && t_wide && seg_bounds && seg_group, "lora_down_wide: null pointer");
  UG_CHECK_ARG(batch >= 1 && rows >= 1 && k >= 8 && k % 8 == 0 && rank_total >= 1 && rank_total <= 64, "lora_down_wide: bad shape");
  UG_CHECK_ARG(groups >= 1 && block >= rank_total && block % 64 == 0, "lora_down_wide: block (%d) must be a multiple of 64 >= rank_total (%d)",
               block, rank_total);
  UG_CHECK_ARG(nseg >= 1 && nseg <= UG_MAX_SEGMENTS, "lora_down_wide: nseg %d out of range", nseg);
  UG_CHECK_ARG(x_rs % 8 == 0 && x_bs % 8 == 0 && t_rs % 8 == 0 && t_bs % 8 == 0 && aligned16(x) && aligned16(a_stack) && aligned16(t_wide),
               "lora_down_wide: alignment");
  ug::LoraSegs segs;
  segs.nseg = nseg;
  for (int i = 0; i <= UG_MAX_SEGMENTS; ++i) segs.bounds[i] = i <= nseg ? seg_bounds[i] : rows;
  for (int i = 0; i < UG_MAX_SEGMENTS; ++i) segs.group[i] = i < nseg ? seg_group[i] : -1;
  const long long warps = (long long)batch * rows;
  const int grid = (int)((warps * 32 + 255) / 256);
  ug::lora_down_wide_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      (const __nv_bfloat16*)x, x_rs, x_bs, (const __nv_bfloat16*)a_stack, (__nv_bfloat16*)t_wide, t_rs, t_bs, batch, rows, k, rank_total,
      groups, block, segs);
  UG_CHECK_LAUNCH("lora_down_wide");
  return UG_OK;
}

extern "C" int ug_lora_down(const void* x, int64_t x_rs, int64_t x_bs, const void* a_stack, float* t, int64_t t_rs,
                            int64_t t_bs, int32_t batch, int32_t rows, int32_t k, int32_t rank_total, int32_t nseg,
                            const int32_t* seg_bounds, const int32_t* seg_group, void* stream) {
  UG_CHECK_ARG(x && a_stack && t && seg_bounds && seg_group, "lora_down: null pointer");
  UG_CHECK_ARG(batch >= 1 && rows >= 1 && k >= 8 && k % 8 == 0 && rank_total >= 1, "lora_down: bad shape");
  UG_CHECK_ARG(nseg >= 1 && nseg <= UG_MAX_SEGMENTS, "lora_down: nseg %d out of range", nseg);
  UG_CHECK_ARG(x_rs % 8 == 0 && x_bs % 8 == 0 && aligned16(x) && aligned16(a_stack), "lora_down: alignment");
  ug::LoraSegs segs;
  segs.nseg = nseg;
  for (int i = 0; i <= UG_MAX_SEGMENTS; ++i) segs.bounds[i] = i <= nseg ? seg_bounds[i] : rows;
  for (int i = 0; i < UG_MAX_SEGMENTS; ++i) segs.group[i] = i < nseg ? seg_group[i] : -1;
  const long long warps = (long long)batch * rows;
  const int grid = (int)((warps * 32 + 255) / 256);
  ug::lora_down_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      (const __nv_bfloat16*)x, x_rs, x_bs, (const __nv_bfloat16*)a_stack, t, t_rs, t_bs, batch, rows, k, rank_total, segs);
  UG_CHECK_LAUNCH("lora_down");
  return UG_OK;
}
