// Dense bf16 GEMM for sm_100a: TMA -> 128B-swizzled smem ring -> tcgen05.mma (accumulators in TMEM,
// double-buffered) -> fused epilogue from TMEM (bias / GELU-tanh / gate * alpha / residual) -> HBM.
// kFp8 instances read e4m3 operands (kind::f8f6f4, one 128-byte swizzle row = 128 elements, so stage bytes, TMA boxes and
// smem descriptors keep their sizes) and dequantise the accumulator with per-row / per-channel scales before the epilogue.
// kExt16 (fp8 only): the second operand pair (K extension) stays bf16 — its K blocks are 64 bf16 = the same 128-byte swizzle
// row, issued as kind::f16 MMAs into the accumulator the kind::f8f6f4 MMAs of the first pair started.
//
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = MMA issuer (+ TMEM owner), warps 2..9 = epilogue
// (warp w reads TMEM lanes 32*(w%4)..+31, the hardware lane-quarter rule of tcgen05.ld; the two warps that share a lane
// quarter split the tile's columns, which halves the epilogue latency per tile — it matters when the K loop is short).
// Persistent: grid = min(tiles, SMs); tiles are walked m-fastest so concurrently running CTAs share W tiles in L2.
// kCta == 2 pairs two SMs on a 256 x BN tile (cta_group::2): each CTA loads its own 128 A rows and HALF of the
// W tile; the leader CTA issues the MMAs, commits are multicast to both CTAs.
//
// Replaces every nn.Linear call on the reference path (SURVEY.md §8 A3-A6, A10).
#include <cstdlib>
#include <cstring>

#include "ug_host.h"
#include "ug_ptx.cuh"

namespace ug {

constexpr int kEpiWarps = 8;                     // 4 or 8
constexpr int kGemmThreads = 64 + 32 * kEpiWarps;

struct GemmParams {
  int rows, n, k, batch;
  int m_tiles, n_tiles, k_blocks, total_tiles;
  int group_m;    // tile walk: m-tiles (x batch) are swept in bands of group_m, n-tiles inside a band (L2 reuse for tall A)
  int k1_blocks;  // K blocks of the first operand pair (A, W); blocks [k1_blocks, k_blocks) come from the second pair (A2, W2)
  __nv_bfloat16* c;
  long long c_rs, c_bs;
  const __nv_bfloat16* bias;
  long long bias_bs;
  const float* gate;
  long long gate_bs;
  int colmask_block;           // != 0: output columns outside block lora_group(row) (blocks of colmask_block columns) are zeroed
  long long gate_seg_stride;  // != 0: rows of segment i (lora_bounds) use gate + i * gate_seg_stride
  float alpha;
  int act;
  const __nv_bfloat16* res;
  long long res_rs, res_bs;
  int w_batched;
  // grouped low-rank (LoRA) update, switched per row segment:  acc[r, c] += sum_j t[r, blk(c)*R + j] * Bl[g(r)][c][j]
  const float* lora_t;
  long long lora_t_rs, lora_t_bs;
  const __nv_bfloat16* lora_b;
  int lora_r, lora_block_n, lora_nseg;
  int lora_bounds[UG_MAX_SEGMENTS + 1];
  int lora_group[UG_MAX_SEGMENTS];
  // fused QK-RMSNorm + RoPE (QKV projections): columns [0, qk_d) = q heads, [qk_d, 2 qk_d) = k heads, rest = v
  const __nv_bfloat16* qk_w;  // [2, qk_dh]: norm_q, norm_k weights (NULL = plain epilogue)
  const float* qk_cos_sin;    // fp32 [rows, qk_dh]: (cos, sin) per rotation pair, row = row of the C view (NULL = no RoPE)
  int qk_dh, qk_d;
  float qk_eps;
  // implicit-GEMM 3x3 convolution (stride 1, zero padding 1) over an NHWC image: the A operand is a 4-D tensor map
  // (channel, x, y, image); K block kb = filter tap kb / conv_cblocks, channel block kb % conv_cblocks, and the A tile of that
  // block is the box of the tile's 128 output pixels shifted by the tap offset (out-of-image pixels arrive as zeros from the
  // TMA unit: the padding costs nothing). conv_cblocks == 0: plain GEMM.
  int conv_cblocks, conv_w;
  // row-wise fp8 dequantisation (kFp8 instances): acc[r, c] * a_scale[b, r] * w_scale[wb, c]
  const float* a_scale;
  long long a_scale_bs;
  const float* w_scale;
  long long w_scale_bs;
};

// host-side description of the convolution a GEMM launch computes (ug_conv3x3_bf16)
struct ConvDesc {
  const void* x;
  int batch, h, w, c_in;
};

template <int kCta, int BN, int kStages, bool kTmaEpi = false, bool kFp8 = false>
struct GemmCfg {
  static constexpr int BM = 128;  // rows per CTA
  static constexpr int ESIZE = kFp8 ? 1 : 2;
  static constexpr int BK = 128 / ESIZE;  // 64 bf16 / 128 e4m3 = one 128-byte swizzle row
  static constexpr int BN_LOAD = BN / kCta;
  static constexpr int A_BYTES = BM * BK * ESIZE;
  static constexpr int B_BYTES = BN_LOAD * BK * ESIZE;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int TMEM_COLS = 2 * BN;
  // smem-staged epilogue: every epilogue warp owns EPI_SLABS staging slabs of 32 rows x 64 bf16 columns (4 KB, 128B-swizzled:
  // the box of one TMA store / one TMA residual load), one per 64-column slab of its share of the tile
  static constexpr int EPI_SLABS = BN / (64 * (kEpiWarps / 4));
  static constexpr int EPI_SLAB_BYTES = 32 * 128;
  static constexpr int EPI_WARP_BYTES = EPI_SLABS * EPI_SLAB_BYTES;
  static constexpr int EPI_BYTES = kTmaEpi ? kEpiWarps * EPI_WARP_BYTES : 0;
  static constexpr int EPI_BARS = kTmaEpi ? kEpiWarps * EPI_SLABS : 0;
  static constexpr int BAR_BYTES = (2 * kStages + 4 + EPI_BARS) * 8 + 16;
  static constexpr int SMEM_BYTES = kStages * STAGE_BYTES + EPI_BYTES + BAR_BYTES + 1024;
  static_assert(TMEM_COLS == 256 || TMEM_COLS == 512, "TMEM allocation must be a power of two");
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
};

// LoRA group of row r (-1: no adapter on this row segment)
__device__ __forceinline__ int lora_group_of(const GemmParams& p, int r) {
  int g = -1;
  for (int s = 0; s < p.lora_nseg; ++s)
    if (r >= p.lora_bounds[s] && r < p.lora_bounds[s + 1]) g = p.lora_group[s];
  return g;
}

__device__ __forceinline__ int seg_index_of(const GemmParams& p, int r) {
  int g = 0;
  for (int s = 0; s < p.lora_nseg; ++s)
    if (r >= p.lora_bounds[s] && r < p.lora_bounds[s + 1]) g = s;
  return g;
}

// fp8: dequantise the 32 accumulator columns [col0, col0 + 32) of one row in place, acc * a_scale(row) * w_scale[c]; this comes
// before every other epilogue op. Columns past n (partial last tile) read no scale and are never stored.
__device__ __forceinline__ void dequant32(const GemmParams& p, uint32_t (&v)[32], int b, float a_s, int col0) {
  const float* ws = p.w_scale + (p.w_batched ? (long long)b * p.w_scale_bs : 0LL);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = col0 + 8 * j;
    float4 w0 = make_float4(0.f, 0.f, 0.f, 0.f), w1 = w0;
    if (c < p.n) {
      w0 = __ldg(reinterpret_cast<const float4*>(ws + c));
      w1 = __ldg(reinterpret_cast<const float4*>(ws + c + 4));
    }
    const float w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
    for (int i = 0; i < 8; ++i) v[8 * j + i] = __float_as_uint(__uint_as_float(v[8 * j + i]) * a_s * w[i]);
  }
}

__device__ __forceinline__ void epilogue_chunk(const GemmParams& p, const uint32_t (&v)[32], int b, int r, int col0,
                                               int lora_g, const float* gate_row) {
  const long long c_off = (long long)b * p.c_bs + (long long)r * p.c_rs;
  const long long r_off = (long long)b * p.res_bs + (long long)r * p.res_rs;
  // residual operand of the whole 32-column chunk up front: the residual may alias C (in-place update), so the compiler
  // cannot hoist these loads above the stores of the previous 8 columns itself and every one of them would expose a full
  // memory latency; a thread only ever writes the locations it reads here, so loading early is safe. (+1.3 % per cfg3 step;
  // a deeper variant that also keeps the NEXT chunk's TMEM + residual loads in flight needs 255 registers and measured
  // 3 % slower.)
  uint4 rv4[4];
  if (p.res) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      rv4[j] = (col0 + 8 * j < p.n) ? *reinterpret_cast<const uint4*>(p.res + r_off + col0 + 8 * j) : make_uint4(0, 0, 0, 0);
  }
  // low-rank down-projection of this row for the sub-linear (fused q|k|v ...) the 32-column chunk belongs to
  float lt[16];
  const __nv_bfloat16* lb = nullptr;
  if (lora_g >= 0) {
    const float* tp = p.lora_t + (long long)b * p.lora_t_bs + (long long)r * p.lora_t_rs + (col0 / p.lora_block_n) * p.lora_r;
#pragma unroll
    for (int i = 0; i < 16; i += 4) {
      if (i < p.lora_r) {
        const float4 t4 = *reinterpret_cast<const float4*>(tp + i);
        lt[i] = t4.x; lt[i + 1] = t4.y; lt[i + 2] = t4.z; lt[i + 3] = t4.w;
      }
    }
    lb = p.lora_b + ((long long)lora_g * p.n) * p.lora_r;
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = col0 + 8 * j;
    if (c >= p.n) break;
    float x[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = __uint_as_float(v[8 * j + i]);
    if (lb) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const __nv_bfloat16* bp = lb + (long long)(c + i) * p.lora_r;
        float acc = 0.f;
#pragma unroll
        for (int q = 0; q < 16; q += 4) {
          if (q < p.lora_r) {
            const uint2 u = *reinterpret_cast<const uint2*>(bp + q);
            const float2 b0 = unpack_bf16x2(u.x), b1 = unpack_bf16x2(u.y);
            acc += lt[q] * b0.x + lt[q + 1] * b0.y + lt[q + 2] * b1.x + lt[q + 3] * b1.y;
          }
        }
        x[i] += acc;
      }
    }
    if (p.bias) {
      uint4 bv = *reinterpret_cast<const uint4*>(p.bias + (long long)b * p.bias_bs + c);
      float2 f0 = unpack_bf16x2(bv.x), f1 = unpack_bf16x2(bv.y), f2 = unpack_bf16x2(bv.z), f3 = unpack_bf16x2(bv.w);
      x[0] += f0.x; x[1] += f0.y; x[2] += f1.x; x[3] += f1.y;
      x[4] += f2.x; x[5] += f2.y; x[6] += f3.x; x[7] += f3.y;
    }
    if (p.act == UG_ACT_GELU_TANH) {
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = gelu_tanh(x[i]);
    }
    if (gate_row) {
      const float* g = gate_row + c;
      float4 g0 = *reinterpret_cast<const float4*>(g), g1 = *reinterpret_cast<const float4*>(g + 4);
      x[0] *= g0.x * p.alpha; x[1] *= g0.y * p.alpha; x[2] *= g0.z * p.alpha; x[3] *= g0.w * p.alpha;
      x[4] *= g1.x * p.alpha; x[5] *= g1.y * p.alpha; x[6] *= g1.z * p.alpha; x[7] *= g1.w * p.alpha;
    } else if (p.alpha != 1.0f) {
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] *= p.alpha;
    }
    if (p.res) {
      const uint4 rv = rv4[j];
      float2 f0 = unpack_bf16x2(rv.x), f1 = unpack_bf16x2(rv.y), f2 = unpack_bf16x2(rv.z), f3 = unpack_bf16x2(rv.w);
      x[0] += f0.x; x[1] += f0.y; x[2] += f1.x; x[3] += f1.y;
      x[4] += f2.x; x[5] += f2.y; x[6] += f3.x; x[7] += f3.y;
    }
    uint4 o;
    o.x = pack_bf16x2(x[0], x[1]);
    o.y = pack_bf16x2(x[2], x[3]);
    o.z = pack_bf16x2(x[4], x[5]);
    o.w = pack_bf16x2(x[6], x[7]);
    *reinterpret_cast<uint4*>(p.c + c_off + c) = o;
  }
}

// bias / GELU-tanh / gate * alpha / residual of 8 consecutive columns starting at c (c < p.n, c % 8 == 0) -> 8 bf16.
// The residual arrives as the 16 bytes the staged epilogue read from its (TMA-loaded) shared-memory slab.
__device__ __forceinline__ uint4 epilogue_group8(const GemmParams& p, const uint32_t* v8, int b, int c, const float* gate_row,
                                                 const uint4& rv) {
  float x[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) x[i] = __uint_as_float(v8[i]);
  if (p.bias) {
    const uint4 bv = *reinterpret_cast<const uint4*>(p.bias + (long long)b * p.bias_bs + c);
    const float2 f0 = unpack_bf16x2(bv.x), f1 = unpack_bf16x2(bv.y), f2 = unpack_bf16x2(bv.z), f3 = unpack_bf16x2(bv.w);
    x[0] += f0.x; x[1] += f0.y; x[2] += f1.x; x[3] += f1.y;
    x[4] += f2.x; x[5] += f2.y; x[6] += f3.x; x[7] += f3.y;
  }
  if (p.act == UG_ACT_GELU_TANH) {
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = gelu_tanh(x[i]);
  }
  if (gate_row) {
    const float* g = gate_row + c;
    const float4 g0 = *reinterpret_cast<const float4*>(g), g1 = *reinterpret_cast<const float4*>(g + 4);
    x[0] *= g0.x * p.alpha; x[1] *= g0.y * p.alpha; x[2] *= g0.z * p.alpha; x[3] *= g0.w * p.alpha;
    x[4] *= g1.x * p.alpha; x[5] *= g1.y * p.alpha; x[6] *= g1.z * p.alpha; x[7] *= g1.w * p.alpha;
  } else if (p.alpha != 1.0f) {
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] *= p.alpha;
  }
  if (p.res) {
    const float2 f0 = unpack_bf16x2(rv.x), f1 = unpack_bf16x2(rv.y), f2 = unpack_bf16x2(rv.z), f3 = unpack_bf16x2(rv.w);
    x[0] += f0.x; x[1] += f0.y; x[2] += f1.x; x[3] += f1.y;
    x[4] += f2.x; x[5] += f2.y; x[6] += f3.x; x[7] += f3.y;
  }
  uint4 o;
  o.x = pack_bf16x2(x[0], x[1]);
  o.y = pack_bf16x2(x[2], x[3]);
  o.z = pack_bf16x2(x[4], x[5]);
  o.w = pack_bf16x2(x[6], x[7]);
  return o;
}

// Fused QK-RMSNorm + RoPE of 8 consecutive q / k columns starting at c: (acc + bias) * rstd * norm_weight, then the interleaved-
// pair rotation with the (cos, sin) table row of token row r. `which` 0 / 1 = q / k head (selects norm_q / norm_k).
__device__ __forceinline__ uint4 epilogue_qk_group8(const GemmParams& p, const uint32_t* v8, int b, int r, int c, int which, float rstd) {
  const int c_in_head = c % p.qk_dh;
  float x[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) x[i] = __uint_as_float(v8[i]);
  if (p.bias) {
    const uint4 bv = *reinterpret_cast<const uint4*>(p.bias + (long long)b * p.bias_bs + c);
    const float2 f0 = unpack_bf16x2(bv.x), f1 = unpack_bf16x2(bv.y), f2 = unpack_bf16x2(bv.z), f3 = unpack_bf16x2(bv.w);
    x[0] += f0.x; x[1] += f0.y; x[2] += f1.x; x[3] += f1.y;
    x[4] += f2.x; x[5] += f2.y; x[6] += f3.x; x[7] += f3.y;
  }
  const uint4 wv = *reinterpret_cast<const uint4*>(p.qk_w + which * p.qk_dh + c_in_head);
  const float2 w0 = unpack_bf16x2(wv.x), w1 = unpack_bf16x2(wv.y), w2 = unpack_bf16x2(wv.z), w3 = unpack_bf16x2(wv.w);
  x[0] *= rstd * w0.x; x[1] *= rstd * w0.y; x[2] *= rstd * w1.x; x[3] *= rstd * w1.y;
  x[4] *= rstd * w2.x; x[5] *= rstd * w2.y; x[6] *= rstd * w3.x; x[7] *= rstd * w3.y;
  if (p.qk_cos_sin) {
    // rows past the matrix edge are computed (and clipped by the TMA store): keep their table reads inside the table
    const float* cs = p.qk_cos_sin + (long long)min(r, p.rows - 1) * p.qk_dh + c_in_head;
    const float4 t0 = __ldg(reinterpret_cast<const float4*>(cs)), t1 = __ldg(reinterpret_cast<const float4*>(cs + 4));
    const float co[4] = {t0.x, t0.z, t1.x, t1.z}, si[4] = {t0.y, t0.w, t1.y, t1.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float a0 = x[2 * q], a1 = x[2 * q + 1];
      x[2 * q] = a0 * co[q] - a1 * si[q];
      x[2 * q + 1] = a1 * co[q] + a0 * si[q];
    }
  }
  uint4 o;
  o.x = pack_bf16x2(x[0], x[1]);
  o.y = pack_bf16x2(x[2], x[3]);
  o.z = pack_bf16x2(x[4], x[5]);
  o.w = pack_bf16x2(x[6], x[7]);
  return o;
}

// bias (+ per-head RMSNorm weight * rstd + interleaved-pair RoPE for q / k columns) -> bf16.  c_in_head = column of the
// first element of this 32-column chunk inside its head; `which` 0/1 = q/k head (normalised), 2 = v head (plain).
__device__ __forceinline__ void epilogue_qkv_chunk(const GemmParams& p, const uint32_t (&v)[32], int b, int r, int col0,
                                                   int c_in_head, int which, float rstd) {
  const long long c_off = (long long)b * p.c_bs + (long long)r * p.c_rs;
  const float* cs = (which < 2 && p.qk_cos_sin) ? p.qk_cos_sin + (long long)r * p.qk_dh + c_in_head : nullptr;
  const __nv_bfloat16* wq = p.qk_w + which * p.qk_dh + c_in_head;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = col0 + 8 * j;
    float x[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = __uint_as_float(v[8 * j + i]);
    if (p.bias) {
      uint4 bv = *reinterpret_cast<const uint4*>(p.bias + (long long)b * p.bias_bs + c);
      float2 f0 = unpack_bf16x2(bv.x), f1 = unpack_bf16x2(bv.y), f2 = unpack_bf16x2(bv.z), f3 = unpack_bf16x2(bv.w);
      x[0] += f0.x; x[1] += f0.y; x[2] += f1.x; x[3] += f1.y;
      x[4] += f2.x; x[5] += f2.y; x[6] += f3.x; x[7] += f3.y;
    }
    if (which < 2) {
      uint4 wv = *reinterpret_cast<const uint4*>(wq + 8 * j);
      float2 w0 = unpack_bf16x2(wv.x), w1 = unpack_bf16x2(wv.y), w2 = unpack_bf16x2(wv.z), w3 = unpack_bf16x2(wv.w);
      x[0] *= rstd * w0.x; x[1] *= rstd * w0.y; x[2] *= rstd * w1.x; x[3] *= rstd * w1.y;
      x[4] *= rstd * w2.x; x[5] *= rstd * w2.y; x[6] *= rstd * w3.x; x[7] *= rstd * w3.y;
      if (cs) {
        const float4 t0 = *reinterpret_cast<const float4*>(cs + 8 * j), t1 = *reinterpret_cast<const float4*>(cs + 8 * j + 4);
        const float co[4] = {t0.x, t0.z, t1.x, t1.z}, si[4] = {t0.y, t0.w, t1.y, t1.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float a0 = x[2 * q], a1 = x[2 * q + 1];
          x[2 * q] = a0 * co[q] - a1 * si[q];
          x[2 * q + 1] = a1 * co[q] + a0 * si[q];
        }
      }
    }
    uint4 o;
    o.x = pack_bf16x2(x[0], x[1]);
    o.y = pack_bf16x2(x[2], x[3]);
    o.z = pack_bf16x2(x[4], x[5]);
    o.w = pack_bf16x2(x[6], x[7]);
    *reinterpret_cast<uint4*>(p.c + c_off + c) = o;
  }
}

// sum over the chunk of (acc + bias)^2 — first pass of the fused per-head RMSNorm
__device__ __forceinline__ float chunk_sumsq(const GemmParams& p, const uint32_t (&v)[32], int b, int col0) {
  float ss = 0.f;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float x[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = __uint_as_float(v[8 * j + i]);
    if (p.bias) {
      uint4 bv = *reinterpret_cast<const uint4*>(p.bias + (long long)b * p.bias_bs + col0 + 8 * j);
      float2 f0 = unpack_bf16x2(bv.x), f1 = unpack_bf16x2(bv.y), f2 = unpack_bf16x2(bv.z), f3 = unpack_bf16x2(bv.w);
      x[0] += f0.x; x[1] += f0.y; x[2] += f1.x; x[3] += f1.y;
      x[4] += f2.x; x[5] += f2.y; x[6] += f3.x; x[7] += f3.y;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) ss += x[i] * x[i];
  }
  return ss;
}

// Persistent tile walk. Band b covers m-indices [b * group_m, ...): inside a band the m index runs fastest, then n, so the
// CTAs running at the same time share group_m A row-tiles and a handful of W column-tiles. group_m = all m-tiles gives the
// plain m-fastest order (best when A fits in L2); a small band keeps tall-A problems (M = 16 k rows: A alone exceeds what L2
// can hold next to the streaming C writes, and every n-wave re-read it from HBM: 4.7 GB per launch) inside L2.
__device__ __forceinline__ void tile_coords(const GemmParams& p, int tile, int mb_count, int& mb, int& nt) {
  const int band = p.group_m * p.n_tiles;
  const int g = tile / band, in_band = tile - g * band;
  const int first = g * p.group_m;
  const int size = min(mb_count - first, p.group_m);
  mb = first + in_band % size;
  nt = in_band / size;
}

template <int kCta, int BN, int kStages, bool kTmaEpi, bool kFp8, bool kExt16>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_w,
                 const __grid_constant__ CUtensorMap tma_a2, const __grid_constant__ CUtensorMap tma_w2,
                 const __grid_constant__ CUtensorMap tma_c, const __grid_constant__ CUtensorMap tma_r, const GemmParams p) {
  using Cfg = GemmCfg<kCta, BN, kStages, kTmaEpi, kFp8>;
  extern __shared__ uint8_t smem_raw[];
  // 128B swizzle atoms need 1024-byte alignment; the offset is identical in both CTAs of a pair.
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + kStages * Cfg::A_BYTES;
  uint8_t* smem_epi = smem + kStages * Cfg::STAGE_BYTES;  // 1024-byte aligned (every stage is a multiple of 1 KB)
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + kStages * Cfg::STAGE_BYTES + Cfg::EPI_BYTES);
  uint64_t* empty = full + kStages;
  uint64_t* tmem_full = empty + kStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* res_bars = tmem_empty + 2;  // [kEpiWarps][EPI_SLABS] (staged epilogue only)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_bars + Cfg::EPI_BARS);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = (kCta == 2) ? cluster_ctarank() : 0u;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_w);
    if (p.k1_blocks < p.k_blocks) {
      tma_prefetch_desc(&tma_a2);
      tma_prefetch_desc(&tma_w2);
    }
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], kEpiWarps * kCta);  // one arrive per epilogue warp per CTA
    }
    for (int s = 0; s < Cfg::EPI_BARS; ++s) mbar_init(&res_bars[s], 1);
    if constexpr (kTmaEpi) {
      tma_prefetch_desc(&tma_c);
      if (p.res) tma_prefetch_desc(&tma_r);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<kCta>(tmem_slot, Cfg::TMEM_COLS);
  tc_fence_before();
  if constexpr (kCta == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int unit = (kCta == 2) ? (blockIdx.x >> 1) : blockIdx.x;
  const int num_units = (kCta == 2) ? (gridDim.x >> 1) : gridDim.x;
  const int mb_count = p.m_tiles * p.batch;

  if (warp == 0) {
    // ------------------------------ TMA producer ------------------------------
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = unit; tile < p.total_tiles; tile += num_units) {
      int mb, nt;
      tile_coords(p, tile, mb_count, mb, nt);
      const int b = mb / p.m_tiles, mt = mb % p.m_tiles;
      const int row0 = mt * (Cfg::BM * kCta) + (int)cta_rank * Cfg::BM;
      const int wrow0 = nt * BN + (int)cta_rank * Cfg::BN_LOAD;
      const int wb = p.w_batched ? b : 0;
      int conv_y0 = 0, conv_x0 = 0, conv_tap = 0, conv_cb = 0;
      if (p.conv_cblocks) {
        conv_y0 = row0 / p.conv_w;
        conv_x0 = row0 - conv_y0 * p.conv_w;
      }
      for (int kb = 0; kb < p.k_blocks; ++kb) {
        mbar_wait(&empty[stage], phase ^ 1);
        if (elect_one_sync()) {
          void* sa = smem_a + stage * Cfg::A_BYTES;
          void* sb = smem_b + stage * Cfg::B_BYTES;
          if (p.conv_cblocks) {
            const int dy = conv_tap / 3, dx = conv_tap - 3 * dy;
            if constexpr (kCta == 1) {
              mbar_arrive_expect_tx(&full[stage], Cfg::STAGE_BYTES);
              tma_load_4d(sa, &tma_a, &full[stage], conv_cb * Cfg::BK, conv_x0 + dx - 1, conv_y0 + dy - 1, b);
              tma_load_3d(sb, &tma_w, &full[stage], kb * Cfg::BK, wrow0, 0);
            } else {
              if (cta_rank == 0) mbar_arrive_expect_tx(&full[stage], 2 * Cfg::STAGE_BYTES);
              tma_load_4d_2sm(sa, &tma_a, &full[stage], conv_cb * Cfg::BK, conv_x0 + dx - 1, conv_y0 + dy - 1, b);
              tma_load_3d_2sm(sb, &tma_w, &full[stage], kb * Cfg::BK, wrow0, 0);
            }
          } else {
            // second operand pair (K extension: C += A2 @ W2^T accumulates into the same TMEM tile)
            const bool second = kb >= p.k1_blocks;
            const CUtensorMap* ma = second ? &tma_a2 : &tma_a;
            const CUtensorMap* mw = second ? &tma_w2 : &tma_w;
            const int kc = second ? (kb - p.k1_blocks) * (kExt16 ? 64 : Cfg::BK) : kb * Cfg::BK;
            if constexpr (kCta == 1) {
              mbar_arrive_expect_tx(&full[stage], Cfg::STAGE_BYTES);
              tma_load_3d(sa, ma, &full[stage], kc, row0, b);
              tma_load_3d(sb, mw, &full[stage], kc, wrow0, second ? 0 : wb);
            } else {
              if (cta_rank == 0) mbar_arrive_expect_tx(&full[stage], 2 * Cfg::STAGE_BYTES);
              tma_load_3d_2sm(sa, ma, &full[stage], kc, row0, b);
              tma_load_3d_2sm(sb, mw, &full[stage], kc, wrow0, second ? 0 : wb);
            }
          }
        }
        if (p.conv_cblocks && ++conv_cb == p.conv_cblocks) { conv_cb = 0; ++conv_tap; }
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------ MMA issuer (leader CTA only) ------------------------------
    if (cta_rank == 0) {
      constexpr uint32_t idesc = kFp8 ? make_idesc_e4m3(Cfg::BM * kCta, BN) : make_idesc_bf16(Cfg::BM * kCta, BN, false, false);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = unit; tile < p.total_tiles; tile += num_units, ++it) {
        const int as = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        mbar_wait(&tmem_empty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          // elect.sync, not `lane == 0`: ptxas then knows the block is single-threaded and keeps the descriptors in uniform
          // registers; with a lane test every tcgen05.mma was wrapped in an R2UR + ELECT / BRA.U.ANY loop
          if (elect_one_sync()) {
            const uint64_t a_desc = make_sdesc_sw128(smem_u32(smem_a + stage * Cfg::A_BYTES), 16, 1024);
            const uint64_t b_desc = make_sdesc_sw128(smem_u32(smem_b + stage * Cfg::B_BYTES), 16, 1024);
            if (kExt16 && kb >= p.k1_blocks) {
              // bf16 K-extension block (kb >= 1: always accumulates onto the fp8 partial sums)
              constexpr uint32_t idesc16 = make_idesc_bf16(Cfg::BM * kCta, BN, false, false);
#pragma unroll
              for (int k = 0; k < 4; ++k) umma_ss<kCta, false>(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc16, 1u);
            } else {
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                // +32 bytes per K step (16 bf16 / 32 e4m3) inside the 128-byte swizzle row (start-address field is in 16 B units)
                umma_ss<kCta, kFp8>(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
              }
            }
            if constexpr (kCta == 1) {
              umma_commit(&empty[stage]);
              if (kb == p.k_blocks - 1) umma_commit(&tmem_full[as]);
            } else {
              umma_commit_2sm(&empty[stage], 0b11);
              if (kb == p.k_blocks - 1) umma_commit_2sm(&tmem_full[as], 0b11);
            }
          }
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ------------------------------ epilogue (warps 2..) ------------------------------
    const int q = warp & 3;
    const int col_half = (warp - 2) >> 2;  // 0 / 1 with 8 epilogue warps: which half of the tile's columns this warp converts
    const int row_local = q * 32 + lane;
    uint32_t res_phase = 0;  // staged epilogue: parity bit per residual-slab barrier of this warp
    (void)res_phase;
    int it = 0;
    for (int tile = unit; tile < p.total_tiles; tile += num_units, ++it) {
      int mb, nt;
      tile_coords(p, tile, mb_count, mb, nt);
      const int b = mb / p.m_tiles, mt = mb % p.m_tiles;
      const int r = mt * (Cfg::BM * kCta) + (int)cta_rank * Cfg::BM + row_local;
      const int n0 = nt * BN;
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      if constexpr (!kTmaEpi) {  // (the staged epilogue first issues its residual prefetch, then waits)
        mbar_wait(&tmem_full[as], aphase);
        tc_fence_after();
      }
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + as * BN;
      const int lora_g = (p.lora_t || p.colmask_block) ? lora_group_of(p, r) : -1;
      // fp8: this row's activation scale (rows past the matrix edge are computed, never stored: read a valid entry)
      // (kExt16: a NULL a_scale means unit scales — the masked down-projection of the LoRA operand A2)
      const float a_s = !kFp8 || (kExt16 && !p.a_scale) ? 1.f : __ldg(p.a_scale + (long long)b * p.a_scale_bs + min(r, p.rows - 1));
      (void)a_s;
      // gate vector of this row: per sample, and per row segment when gate_seg_stride is set (once per tile, not per chunk)
      const float* gate_row = p.gate ? p.gate + (long long)b * p.gate_bs + (p.gate_seg_stride ? seg_index_of(p, r) * p.gate_seg_stride : 0)
                                     : nullptr;
      auto release_acc = [&]() {
        // accumulator stage fully read: hand it back to the MMA warp before doing the last stores
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (kCta == 1 || cta_rank == 0) mbar_arrive(&tmem_empty[as]);
          else mbar_arrive_cluster(&tmem_empty[as], 0);
        }
      };
      if constexpr (kTmaEpi) {
        // ---- smem-staged epilogue: TMEM -> registers -> (bias / GELU / gate / residual) -> this warp's 128B-swizzled slab ->
        // ONE TMA store per 32 x 64 slab (full 128-byte lines, rows / columns past the matrix edge clipped by the hardware).
        // The residual slab is TMA-LOADED into the same staging buffer ahead of the accumulator (issued before the wait on
        // tmem_full, so its latency hides behind the MMAs of this tile) instead of 16-byte loads strided over 32 rows. ----
        const int ew = warp - 2;
        uint8_t* slab0 = smem_epi + ew * Cfg::EPI_WARP_BYTES;
        uint64_t* rbar = res_bars + ew * Cfg::EPI_SLABS;
        const int r0 = mt * (Cfg::BM * kCta) + (int)cta_rank * Cfg::BM + q * 32;  // first row of this warp's lane quarter
        const int cw0 = n0 + col_half * (BN / (kEpiWarps / 4));                    // first column of this warp's share
        if (lane == 0) bulk_wait_group_read<0>();  // last tile's stores have drained their staging slabs
        __syncwarp();
        if (p.res && lane == 0) {
#pragma unroll
          for (int sl = 0; sl < Cfg::EPI_SLABS; ++sl) {
            if (cw0 + 64 * sl < p.n) {
              mbar_arrive_expect_tx(&rbar[sl], Cfg::EPI_SLAB_BYTES);
              tma_load_3d(slab0 + sl * Cfg::EPI_SLAB_BYTES, &tma_r, &rbar[sl], cw0 + 64 * sl, r0, b);
            }
          }
        }
        mbar_wait(&tmem_full[as], aphase);
        tc_fence_after();
        constexpr int kChunksPerWarp = (BN / 32) / (kEpiWarps / 4);
        const int ch0 = col_half * kChunksPerWarp;
        // fused QK-RMSNorm + RoPE (q|k|v projections, BN = 256 tiles): this warp's 128 columns are ONE head (dh = 128) or two
        // (dh = 64) of q, k or v; a first pass over the accumulator gives the per-row 1 / rms of each head, the second pass below
        // normalises, rotates and stages — the separate in-place pass over the QKV buffer disappears
        int qk_which = 2;
        float qk_rstd[2] = {1.f, 1.f};
        if constexpr (BN == 256) {
          if (p.qk_w && cw0 < p.n) qk_which = cw0 / p.qk_d;
          if (qk_which < 2) {
            float ss[2] = {0.f, 0.f};
#pragma unroll
            for (int ch = 0; ch < kChunksPerWarp; ++ch) {
              uint32_t v[32];
              tmem_ld_32x32(taddr + (ch0 + ch) * 32, v);
              tmem_ld_wait();
              if constexpr (kFp8) dequant32(p, v, b, a_s, cw0 + 32 * ch);
              if (cw0 + 32 * ch < p.n) ss[(p.qk_dh == 64) ? (ch >> 1) : 0] += chunk_sumsq(p, v, b, cw0 + 32 * ch);
            }
            if (p.qk_dh != 64) ss[1] = ss[0];
            qk_rstd[0] = rsqrtf(ss[0] / (float)p.qk_dh + p.qk_eps);
            qk_rstd[1] = rsqrtf(ss[1] / (float)p.qk_dh + p.qk_eps);
          }
        }
#pragma unroll 1
        for (int sl = 0; sl < Cfg::EPI_SLABS; ++sl) {
          const int cs0 = cw0 + 64 * sl;
          const bool active = cs0 < p.n;  // warp-uniform
          uint8_t* slab = slab0 + sl * Cfg::EPI_SLAB_BYTES;
          if (p.res && active) {
            mbar_wait(&rbar[sl], (res_phase >> sl) & 1u);
            res_phase ^= 1u << sl;
          }
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            uint32_t v[32];
            tmem_ld_32x32(taddr + (ch0 + 2 * sl + h) * 32, v);
            tmem_ld_wait();
            if constexpr (kFp8) dequant32(p, v, b, a_s, cs0 + 32 * h);
            if (sl == Cfg::EPI_SLABS - 1 && h == 1) release_acc();
            if (active) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const int c = cs0 + 32 * h + 8 * j;
                // row `lane` of the slab, 16-byte chunk (4 h + j) XOR-swizzled by the row's position in its 8-row atom
                uint4* cell = reinterpret_cast<uint4*>(slab + lane * 128 + (((4 * h + j) ^ (lane & 7)) << 4));
                if (c < p.n) {
                  if (qk_which < 2) *cell = epilogue_qk_group8(p, &v[8 * j], b, r, c, qk_which, sl == 0 ? qk_rstd[0] : qk_rstd[1]);
                  else *cell = epilogue_group8(p, &v[8 * j], b, c, gate_row, p.res ? *cell : make_uint4(0, 0, 0, 0));
                }
              }
            }
          }
          if (active) {
            fence_proxy_async_smem();  // generic-proxy writes of the slab -> visible to the TMA engine
            __syncwarp();
            if (lane == 0) {
              tma_store_3d(&tma_c, slab, cs0, r0, b);
              bulk_commit_group();
            }
          }
        }
      } else if (p.qk_w) {
        // ---- QKV projection: per-head RMSNorm (two passes over the TMEM columns of a head) + RoPE, fused ----
        const int cph = p.qk_dh >> 5;  // 32-column chunks per head
        // the two warps of a lane quarter split the tile's heads when half a tile holds whole heads; otherwise the first
        // one converts the whole tile and the second only hands its share of the accumulator back
        constexpr int kHalf = BN / (kEpiWarps / 4);
        const bool split = (kHalf % p.qk_dh) == 0;
        const int c_lo = split ? col_half * kHalf : 0;
        const int c_hi = split ? c_lo + kHalf : (col_half == 0 ? BN : 0);
        if (c_hi == 0) release_acc();
#pragma unroll 1
        for (int c_h = c_lo; c_h < c_hi; c_h += p.qk_dh) {
          const int col_h = n0 + c_h;
          const bool active = col_h < p.n;             // warp-uniform
          const int which = active ? col_h / p.qk_d : 2;  // 0 = q head, 1 = k head, 2 = v head
          float rstd = 1.f;
          if (which < 2) {
            float ss = 0.f;
#pragma unroll 1
            for (int ch = 0; ch < cph; ++ch) {
              uint32_t v[32];
              tmem_ld_32x32(taddr + c_h + ch * 32, v);
              tmem_ld_wait();
              if constexpr (kFp8) dequant32(p, v, b, a_s, col_h + ch * 32);
              ss += chunk_sumsq(p, v, b, col_h + ch * 32);
            }
            rstd = rsqrtf(ss / (float)p.qk_dh + p.qk_eps);
          }
#pragma unroll 1
          for (int ch = 0; ch < cph; ++ch) {
            uint32_t v[32];
            tmem_ld_32x32(taddr + c_h + ch * 32, v);
            tmem_ld_wait();
            if constexpr (kFp8) dequant32(p, v, b, a_s, col_h + ch * 32);
            if (c_h + p.qk_dh >= c_hi && ch == cph - 1) release_acc();
            if (r < p.rows && active) epilogue_qkv_chunk(p, v, b, r, col_h + ch * 32, ch * 32, which, rstd);
          }
        }
      } else {
        constexpr int kChunksPerWarp = (BN / 32) / (kEpiWarps / 4);
        const int ch0 = col_half * kChunksPerWarp;
#pragma unroll 1
        for (int ch = ch0; ch < ch0 + kChunksPerWarp; ++ch) {
          uint32_t v[32];
          tmem_ld_32x32(taddr + ch * 32, v);
          tmem_ld_wait();
          if (ch == ch0 + kChunksPerWarp - 1) release_acc();
          const int col0 = n0 + ch * 32;
          if constexpr (kFp8) dequant32(p, v, b, a_s, col0);
          if (p.colmask_block && col0 / p.colmask_block != lora_g) {
            // grouped down-projection: a row keeps only the column block of its own adapter group
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = 0u;
            if (r < p.rows && col0 < p.n) epilogue_chunk(p, v, b, r, col0, -1, nullptr);
          } else if (r < p.rows && col0 < p.n) epilogue_chunk(p, v, b, r, col0, p.lora_t ? lora_g : -1, gate_row);
        }
      }
    }
  }

  if constexpr (kTmaEpi) {
    if (warp >= 2 && lane == 0) bulk_wait_group<0>();  // the last tile's TMA stores have completed before the CTA retires
  }
  tc_fence_before();
  if constexpr (kCta == 2) cluster_sync_all(); else __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<kCta>(tmem_base, Cfg::TMEM_COLS);
  }
}

template <int kCta, int BN, int kStages, bool kTmaEpi = false, bool kFp8 = false, bool kExt16 = false>
static int launch_gemm(const ug_gemm_args& a, cudaStream_t stream, const ConvDesc* conv = nullptr,
                       const ug_gemm_fp8_scales* scales = nullptr) {
  using Cfg = GemmCfg<kCta, BN, kStages, kTmaEpi, kFp8>;
  constexpr uint64_t E = Cfg::ESIZE;
  constexpr int BK2 = kExt16 ? 64 : Cfg::BK;  // K block of the second operand pair (always bf16: 64 = one swizzle row)
  static_assert(!kExt16 || kFp8, "kExt16 is the bf16 K extension of an fp8 GEMM");
  // A / W operand maps: bf16, or one e4m3 per byte (UINT8) for the fp8 instances
  auto encode_op = [](CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides, const uint32_t* box) {
    return kFp8 ? encode_tmap(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, base, rank, dims, strides, box)
                : encode_tmap_bf16(m, base, rank, dims, strides, box);
  };
  auto kern = gemm_bf16_kernel<kCta, BN, kStages, kTmaEpi, kFp8, kExt16>;
  static bool attr_done[64] = {false};
  if (int st = ensure_dynamic_smem(kern, Cfg::SMEM_BYTES, attr_done, "gemm"); st != UG_OK) return st;
  CUtensorMap tma_a, tma_w;
  if (conv) {
    // NHWC image as (channel, x, y, image); box = 64 channels x the 128 output pixels of one CTA's row tile (a run of a row
    // when the width is a multiple of 128, else 128 / width whole rows)
    const uint32_t bw = conv->w % Cfg::BM == 0 ? (uint32_t)Cfg::BM : (uint32_t)conv->w;
    uint64_t dims[4] = {(uint64_t)conv->c_in, (uint64_t)conv->w, (uint64_t)conv->h, (uint64_t)conv->batch};
    uint64_t strides[3] = {(uint64_t)conv->c_in * 2, (uint64_t)conv->w * conv->c_in * 2, (uint64_t)conv->h * conv->w * conv->c_in * 2};
    uint32_t box[4] = {(uint32_t)Cfg::BK, bw, (uint32_t)Cfg::BM / bw, 1};
    int st = encode_tmap_bf16(&tma_a, conv->x, 4, dims, strides, box);
    if (st != UG_OK) return st;
  } else {
    uint64_t dims[3] = {(uint64_t)a.k, (uint64_t)a.rows, (uint64_t)a.batch};
    uint64_t bs = a.batch > 1 ? (uint64_t)a.a_batch_stride : (uint64_t)a.rows * a.a_row_stride;
    uint64_t strides[2] = {(uint64_t)a.a_row_stride * E, bs * E};
    uint32_t box[3] = {(uint32_t)Cfg::BK, (uint32_t)Cfg::BM, 1};
    int st = encode_op(&tma_a, a.a, 3, dims, strides, box);
    if (st != UG_OK) return st;
  }
  const bool w_batched = a.w_batch_stride != 0 && a.batch > 1;
  {
    uint64_t dims[3] = {(uint64_t)a.k, (uint64_t)a.n, (uint64_t)(w_batched ? a.batch : 1)};
    uint64_t bs = w_batched ? (uint64_t)a.w_batch_stride : (uint64_t)a.n * a.w_row_stride;
    uint64_t strides[2] = {(uint64_t)a.w_row_stride * E, bs * E};
    uint32_t box[3] = {(uint32_t)Cfg::BK, (uint32_t)Cfg::BN_LOAD, 1};
    int st = encode_op(&tma_w, a.w, 3, dims, strides, box);
    if (st != UG_OK) return st;
  }
  CUtensorMap tma_a2 = tma_a, tma_w2 = tma_w;
  int k2_blocks = 0;
  if (a.a2) {
    {
      uint64_t dims[3] = {(uint64_t)a.k2, (uint64_t)a.rows, (uint64_t)a.batch};
      uint64_t bs = a.batch > 1 ? (uint64_t)a.a2_batch_stride : (uint64_t)a.rows * a.a2_row_stride;
      uint64_t strides[2] = {(uint64_t)a.a2_row_stride * 2, bs * 2};
      uint32_t box[3] = {(uint32_t)BK2, (uint32_t)Cfg::BM, 1};
      int st = encode_tmap_bf16(&tma_a2, a.a2, 3, dims, strides, box);
      if (st != UG_OK) return st;
    }
    {
      uint64_t dims[3] = {(uint64_t)a.k2, (uint64_t)a.n, 1};
      uint64_t strides[2] = {(uint64_t)a.w2_row_stride * 2, (uint64_t)a.n * a.w2_row_stride * 2};
      uint32_t box[3] = {(uint32_t)BK2, (uint32_t)Cfg::BN_LOAD, 1};
      int st = encode_tmap_bf16(&tma_w2, a.w2, 3, dims, strides, box);
      if (st != UG_OK) return st;
    }
    k2_blocks = (a.k2 + BK2 - 1) / BK2;
  }
  CUtensorMap tma_c = tma_a, tma_r = tma_a;
  if constexpr (kTmaEpi) {
    // output / residual as [n, rows, batch] with a 64-column x 32-row box: one epilogue warp's staging slab
    uint32_t box[3] = {64, 32, 1};
    {
      uint64_t dims[3] = {(uint64_t)a.n, (uint64_t)a.rows, (uint64_t)a.batch};
      uint64_t bs = a.batch > 1 ? (uint64_t)a.c_batch_stride : (uint64_t)a.rows * a.c_row_stride;
      uint64_t strides[2] = {(uint64_t)a.c_row_stride * 2, bs * 2};
      int st = encode_tmap_bf16(&tma_c, a.c, 3, dims, strides, box);
      if (st != UG_OK) return st;
    }
    if (a.residual) {
      uint64_t dims[3] = {(uint64_t)a.n, (uint64_t)a.rows, (uint64_t)a.batch};
      uint64_t bs = a.batch > 1 ? (uint64_t)a.res_batch_stride : (uint64_t)a.rows * a.res_row_stride;
      uint64_t strides[2] = {(uint64_t)a.res_row_stride * 2, bs * 2};
      int st = encode_tmap_bf16(&tma_r, a.residual, 3, dims, strides, box);
      if (st != UG_OK) return st;
    }
  }
  GemmParams p;
  p.rows = a.rows; p.n = a.n; p.k = a.k; p.batch = a.batch;
  p.m_tiles = (a.rows + Cfg::BM * kCta - 1) / (Cfg::BM * kCta);
  p.n_tiles = (a.n + BN - 1) / BN;
  {
    // A bytes one sweep over all m-tiles touches; above ~40 MB it no longer survives in the 126 MB L2 between n-waves
    const long long row_bytes = (long long)a.k * Cfg::ESIZE + (a.a2 ? 2LL * a.k2 : 0LL);  // the second pair is bf16
    const long long a_bytes = (long long)a.batch * a.rows * row_bytes;
    const int mb_all = p.m_tiles * a.batch;
    p.group_m = mb_all;
    if (a_bytes > (40LL << 20) && !(a.w_batch_stride != 0 && a.batch > 1)) {
      // band of A row-tiles worth ~24 MB: it stays in L2 while the band sweeps every n-tile, so A is read from HBM once
      const long long tile_bytes = (long long)Cfg::BM * kCta * row_bytes;
      long long gm = (24LL << 20) / tile_bytes;
      gm = gm < 2 ? 2 : (gm > 16 ? 16 : gm);
      p.group_m = gm < mb_all ? (int)gm : mb_all;
    }
  }
  p.k1_blocks = (a.k + Cfg::BK - 1) / Cfg::BK;
  p.k_blocks = p.k1_blocks + k2_blocks;
  p.total_tiles = p.m_tiles * p.n_tiles * a.batch;
  p.c = (__nv_bfloat16*)a.c; p.c_rs = a.c_row_stride; p.c_bs = a.c_batch_stride;
  p.bias = (const __nv_bfloat16*)a.bias; p.bias_bs = a.bias_batch_stride;
  p.gate = a.gate; p.gate_bs = a.gate_batch_stride; p.gate_seg_stride = a.gate_seg_stride; p.colmask_block = a.colmask_block;
  p.alpha = a.alpha; p.act = a.act;
  p.res = (const __nv_bfloat16*)a.residual; p.res_rs = a.res_row_stride; p.res_bs = a.res_batch_stride;
  p.w_batched = w_batched ? 1 : 0;
  p.qk_w = (const __nv_bfloat16*)a.qk_norm_weight; p.qk_cos_sin = a.qk_cos_sin; p.qk_dh = a.qk_head_dim;
  p.qk_d = a.qk_d; p.qk_eps = a.qk_eps;
  p.conv_cblocks = conv ? conv->c_in / Cfg::BK : 0;
  p.conv_w = conv ? conv->w : 0;
  p.lora_t = a.lora_t; p.lora_t_rs = a.lora_t_row_stride; p.lora_t_bs = a.lora_t_batch_stride;
  p.lora_b = (const __nv_bfloat16*)a.lora_b;
  p.lora_r = a.lora_rank; p.lora_block_n = a.lora_block_n > 0 ? a.lora_block_n : a.n; p.lora_nseg = a.lora_nseg;
  for (int i = 0; i <= UG_MAX_SEGMENTS; ++i) p.lora_bounds[i] = i <= a.lora_nseg ? a.lora_seg_bounds[i] : a.rows;
  for (int i = 0; i < UG_MAX_SEGMENTS; ++i) p.lora_group[i] = i < a.lora_nseg ? a.lora_seg_group[i] : -1;
  p.a_scale = scales ? scales->a_scale : nullptr;
  p.a_scale_bs = scales ? scales->a_scale_batch_stride : 0;
  p.w_scale = scales ? scales->w_scale : nullptr;
  p.w_scale_bs = scales ? scales->w_scale_batch_stride : 0;

  const int sms = num_sms();
  int units = kCta == 2 ? sms / 2 : sms;
  if (units > p.total_tiles) units = p.total_tiles;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(units * kCta);
  cfg.blockDim = dim3(kGemmThreads);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kCta;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, tma_a, tma_w, tma_a2, tma_w2, tma_c, tma_r, p);
  if (e != cudaSuccess) {
    set_error("gemm: launch failed: %s", cudaGetErrorString(e));
    return UG_ERR_CUDA;
  }
  count_launch();
  return UG_OK;
}

// What variant 0 (auto) maps to: the smem-staged TMA-store epilogue (default: -2.4 % per cfg3 step in a same-box A/B,
// profiles/r02_ab_epilogue_ln.txt), or the direct per-thread-store epilogue with UG_GEMM_EPILOGUE=direct (kept as the A/B arm).
static bool staged_epilogue_default() {
  static int cached = -1;
  if (cached < 0) {
    const char* e = getenv("UG_GEMM_EPILOGUE");
    cached = (e && strcmp(e, "direct") == 0) ? 0 : 1;
  }
  return cached == 1;
}

// auto tile choice: estimate each variant's time as  waves x tile area / (SMs per tile x relative tile efficiency)
static int pick_tile_variant(int batch, int rows, int n) {
  const int sms = num_sms();
  struct Cand { int v, tm, tn; double rate; int units; };
  // relative per-SM tile throughput from profiles/r01_probe_gemm_v1.log (large problems: 1371 / 1349 / ~900 TFLOP/s)
  const Cand cands[3] = {{2, 256, 256, 2.0, sms / 2}, {1, 128, 256, 0.98, sms}, {3, 128, 128, 0.67, sms}};
  double best = 0.0;
  int variant = 0;
  for (const Cand& c : cands) {
    const long long tiles = (long long)batch * ((rows + c.tm - 1) / c.tm) * ((n + c.tn - 1) / c.tn);
    const long long waves = (tiles + c.units - 1) / c.units;
    const double t = (double)waves * c.tm * c.tn / c.rate;
    if (variant == 0 || t < best) { best = t; variant = c.v; }
  }
  return variant;
}

template <bool kFp8, bool kExt16 = false>
static int launch_variant(int variant, const ug_gemm_args& a, cudaStream_t s, const ug_gemm_fp8_scales* scales) {
  switch (variant) {
    case 1: return launch_gemm<1, 256, 4, false, kFp8, kExt16>(a, s, nullptr, scales);
    case 2: return launch_gemm<2, 256, 6, false, kFp8, kExt16>(a, s, nullptr, scales);
    case 3: return launch_gemm<1, 128, 6, false, kFp8, kExt16>(a, s, nullptr, scales);
    case 4: return launch_gemm<2, 256, 5, true, kFp8, kExt16>(a, s, nullptr, scales);
    case 5: return launch_gemm<1, 256, 3, true, kFp8, kExt16>(a, s, nullptr, scales);
    case 6: return launch_gemm<1, 128, 6, true, kFp8, kExt16>(a, s, nullptr, scales);
    default:
      set_error("gemm: unknown variant %d", a.variant);
      return UG_ERR_INVALID;
  }
}

// ug_gemm_bf16 (scales == NULL), ug_gemm_fp8 and ug_gemm_fp8_lora (lora: bf16 K extension + column mask allowed, NULL
// a_scale = unit row scales): argument checks, tile / epilogue choice, launch
static int gemm_entry(const ug_gemm_args* args, const ug_gemm_fp8_scales* scales, void* stream, bool lora = false) {
  const bool fp8 = scales != nullptr;
  UG_CHECK_ARG(args != nullptr, "gemm: null args");
  const ug_gemm_args& a = *args;
  UG_CHECK_ARG(a.a && a.w && a.c, "gemm: null operand pointer");
  UG_CHECK_ARG(a.batch >= 1 && a.rows >= 1 && a.n >= 1 && a.k >= 1, "gemm: empty problem (batch %d rows %d n %d k %d)",
               a.batch, a.rows, a.n, a.k);
  UG_CHECK_ARG(a.k % 8 == 0 && a.n % 8 == 0, "gemm: n (%d) and k (%d) must be multiples of 8", a.n, a.k);
  if (fp8) {
    // e4m3 rows: TMA strides must be multiples of 16 bytes = 16 elements
    UG_CHECK_ARG(a.k % 16 == 0, "gemm_fp8: k (%d) must be a multiple of 16", a.k);
    UG_CHECK_ARG(a.a_row_stride % 16 == 0 && a.w_row_stride % 16 == 0 && (a.batch == 1 || a.a_batch_stride % 16 == 0) &&
                     a.w_batch_stride % 16 == 0,
                 "gemm_fp8: e4m3 row / batch strides must be multiples of 16 elements (16 bytes)");
    if (lora) {
      UG_CHECK_ARG(!a.lora_t, "gemm_fp8_lora: lora_t (the update in the epilogue) is bf16-only: pass it as the K extension a2 / w2");
      UG_CHECK_ARG(!a.a2 == !a.w2, "gemm_fp8_lora: a2 and w2 go together");
      UG_CHECK_ARG(scales->w_scale, "gemm_fp8_lora: null w_scale");
    } else {
      UG_CHECK_ARG(!a.lora_t && !a.colmask_block && !a.a2 && !a.w2,
                   "gemm_fp8: lora_t, colmask_block and the second operand pair (a2 / w2) are bf16-only");
      UG_CHECK_ARG(scales->a_scale && scales->w_scale, "gemm_fp8: null a_scale / w_scale");
    }
    UG_CHECK_ARG((reinterpret_cast<uintptr_t>(scales->a_scale) & 3) == 0 && (reinterpret_cast<uintptr_t>(scales->w_scale) & 15) == 0 &&
                     scales->w_scale_batch_stride % 4 == 0,
                 "gemm_fp8: w_scale must be 16-byte aligned (batch stride a multiple of 4), a_scale 4-byte aligned");
  }
  UG_CHECK_ARG(a.a_row_stride % 8 == 0 && a.w_row_stride % 8 == 0 && a.c_row_stride % 8 == 0,
               "gemm: row strides must be multiples of 8 elements (16 bytes)");
  UG_CHECK_ARG(a.a_row_stride >= a.k && a.w_row_stride >= a.k && a.c_row_stride >= a.n, "gemm: row stride smaller than row");
  UG_CHECK_ARG((reinterpret_cast<uintptr_t>(a.c) & 15) == 0, "gemm: C not 16-byte aligned");
  UG_CHECK_ARG(a.batch == 1 || (a.a_batch_stride % 8 == 0 && a.c_batch_stride % 8 == 0), "gemm: batch strides must be multiples of 8");
  if (a.residual) {
    UG_CHECK_ARG(a.res_row_stride % 8 == 0 && (reinterpret_cast<uintptr_t>(a.residual) & 15) == 0, "gemm: residual alignment");
  }
  if (a.bias) UG_CHECK_ARG((reinterpret_cast<uintptr_t>(a.bias) & 15) == 0 && a.bias_batch_stride % 8 == 0, "gemm: bias alignment");
  if (a.gate) UG_CHECK_ARG((reinterpret_cast<uintptr_t>(a.gate) & 15) == 0 && a.gate_batch_stride % 4 == 0, "gemm: gate alignment");
  if (a.gate_seg_stride) {
    UG_CHECK_ARG(a.gate && a.gate_seg_stride % 4 == 0 && a.lora_nseg >= 1 && a.lora_nseg <= UG_MAX_SEGMENTS,
                 "gemm: gate_seg_stride needs a gate and the row-segment table (lora_nseg / lora_seg_bounds)");
  }
  UG_CHECK_ARG(a.act == UG_ACT_NONE || a.act == UG_ACT_GELU_TANH, "gemm: unknown activation %d", a.act);
  if (a.qk_norm_weight) {
    UG_CHECK_ARG(a.qk_head_dim == 64 || a.qk_head_dim == 128, "gemm: fused QK-norm needs head_dim 64 or 128 (got %d)", a.qk_head_dim);
    UG_CHECK_ARG(a.qk_d > 0 && a.qk_d % a.qk_head_dim == 0 && a.n % a.qk_head_dim == 0 && a.n == 3 * a.qk_d,
                 "gemm: fused QK-norm expects n = 3 * qk_d with qk_d a multiple of head_dim (n %d, qk_d %d)", a.n, a.qk_d);
    UG_CHECK_ARG(!a.lora_t && !a.gate && !a.residual && a.act == UG_ACT_NONE && a.alpha == 1.0f,
                 "gemm: the fused QK-norm epilogue composes with bias only");
    UG_CHECK_ARG((reinterpret_cast<uintptr_t>(a.qk_norm_weight) & 15) == 0 &&
                     (!a.qk_cos_sin || (reinterpret_cast<uintptr_t>(a.qk_cos_sin) & 15) == 0), "gemm: QK-norm operand alignment");
  }
  if (a.lora_t) {
    UG_CHECK_ARG(a.lora_b && (a.lora_rank == 4 || a.lora_rank == 8 || a.lora_rank == 12 || a.lora_rank == 16),
                 "gemm: LoRA needs lora_b and a rank in {4, 8, 12, 16} (got %d)", a.lora_rank);
    UG_CHECK_ARG(a.lora_nseg >= 1 && a.lora_nseg <= UG_MAX_SEGMENTS, "gemm: lora_nseg %d out of range", a.lora_nseg);
    UG_CHECK_ARG((a.lora_block_n <= 0 ? a.n : a.lora_block_n) % 32 == 0, "gemm: lora_block_n must be a multiple of 32");
    UG_CHECK_ARG(a.lora_t_row_stride % 4 == 0 && (reinterpret_cast<uintptr_t>(a.lora_t) & 15) == 0 &&
                     (reinterpret_cast<uintptr_t>(a.lora_b) & 7) == 0,
                 "gemm: LoRA operand alignment");
  }
  if (a.colmask_block) {
    UG_CHECK_ARG(a.colmask_block % 32 == 0 && a.lora_nseg >= 1 && a.lora_nseg <= UG_MAX_SEGMENTS && !a.bias && !a.gate && !a.residual &&
                     a.act == UG_ACT_NONE && !a.lora_t,
                 "gemm: colmask_block must be a multiple of 32, needs the row-segment table and composes with no other epilogue op");
  }
  if (a.a2) {
    UG_CHECK_ARG(a.w2 && a.k2 >= 8 && a.k2 % 8 == 0, "gemm: second operand pair needs w2 and k2 (%d) a positive multiple of 8", a.k2);
    UG_CHECK_ARG(a.a2_row_stride % 8 == 0 && a.w2_row_stride % 8 == 0 && a.a2_row_stride >= a.k2 && a.w2_row_stride >= a.k2 &&
                     (a.batch == 1 || a.a2_batch_stride % 8 == 0),
                 "gemm: second operand pair strides must be multiples of 8 elements and cover k2");
  }
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  int variant = a.variant;
  if (variant == 0) {
    // auto: estimate each variant's time as  waves x tile area / (SMs per tile x relative tile efficiency)  and take the
    // smallest — wave quantisation and the padding of a partial last row tile decide for small M (text stream, per-rank
    // shards of sequence parallelism: M = 576 at P = 8), the 2-CTA pair tile (half the per-SM W traffic, measured 2 % faster per
    // cfg3 step under the 1 kW power cap) wins whenever the grid fills the machine
    variant = pick_tile_variant(a.batch, a.rows, a.n);
    if (a.n <= 128) variant = 3;
  }
  // epilogue flavour: variants 4 / 5 / 6 = tiles of 2 / 1 / 3 with the smem-staged TMA-store epilogue. The LoRA-in-epilogue,
  // and column-mask modes keep the direct epilogue (they need per-row state the staged path does not carry).
  const bool special = a.lora_t || a.colmask_block;
  if (a.variant == 0 && !special && staged_epilogue_default() && !(a.qk_norm_weight && a.qk_d % 128 != 0)) {
    if (a.qk_norm_weight && variant == 3) {
      // the fused QK-norm epilogue needs a whole head inside one warp's 128 columns: BN = 256 tiles only
      const int sms = num_sms();
      const long long t2 = (long long)a.batch * ((a.rows + 255) / 256) * ((a.n + 255) / 256);
      const long long t1 = (long long)a.batch * ((a.rows + 127) / 128) * ((a.n + 255) / 256);
      const double c2 = (double)((t2 + sms / 2 - 1) / (sms / 2)) * 256 * 256 / 2.0, c1 = (double)((t1 + sms - 1) / sms) * 128 * 256 / 0.98;
      variant = c2 <= c1 ? 2 : 1;
    }
    variant = variant == 2 ? 4 : (variant == 1 ? 5 : 6);
  }
  if (variant >= 4 && variant <= 6) {
    UG_CHECK_ARG(!special, "gemm: variants 4-6 (staged epilogue) do not compose with lora_t / colmask_block");
    UG_CHECK_ARG(!a.qk_norm_weight || (variant != 6 && a.qk_d % 128 == 0),
                 "gemm: the staged fused QK-norm epilogue needs a 256-column tile (variants 4 / 5) and qk_d a multiple of 128");
    UG_CHECK_ARG(!a.residual || a.res_batch_stride % 8 == 0 || a.batch == 1, "gemm: residual batch stride must be a multiple of 8");
  }
  if (lora) return launch_variant<true, true>(variant, a, s, scales);
  return fp8 ? launch_variant<true>(variant, a, s, scales) : launch_variant<false>(variant, a, s, nullptr);
}

}  // namespace ug

extern "C" int ug_gemm_bf16(const ug_gemm_args* args, void* stream) { return ug::gemm_entry(args, nullptr, stream); }

// Row-wise fp8 GEMM: the persistent kernel above instantiated for e4m3 operands (kind::f8f6f4) with the dequantisation
// multiply in front of every epilogue path. An opt-in path of `UniGenFlux.quantize_fp8()`.
extern "C" int ug_gemm_fp8(const ug_gemm_args* args, const ug_gemm_fp8_scales* scales, void* stream) {
  if (scales == nullptr) {
    ug::set_error("gemm_fp8: null scales");
    return UG_ERR_INVALID;
  }
  return ug::gemm_entry(args, scales, stream);
}

// The fp8 GEMM with the two switched-LoRA features of the P-variant: a bf16 second operand pair (K extension, kind::f16 MMAs
// into the fp8 accumulator: its operands arrive pre-divided by the scales the epilogue multiplies with) and the column mask of
// the grouped down-projection. A NULL a_scale reads as unit row scales. A separate set of kernel instances (kExt16), so the
// instances behind ug_gemm_fp8 keep their code. An opt-in path of `UniCombineFlux.quantize_fp8()`.
extern "C" int ug_gemm_fp8_lora(const ug_gemm_args* args, const ug_gemm_fp8_scales* scales, void* stream) {
  if (scales == nullptr) {
    ug::set_error("gemm_fp8_lora: null scales");
    return UG_ERR_INVALID;
  }
  return ug::gemm_entry(args, scales, stream, true);
}

// 3x3 convolution, stride 1, zero padding 1, over NHWC bf16 images as an implicit GEMM on the tcgen05 path above: no im2col
// buffer exists — the TMA unit assembles every A tile from the image with the filter tap's offset and fills the halo with zeros.
// Replaces the nn.Conv2d(k=3, p=1) calls of the AutoencoderKL the reference pipelines run around the denoiser
// (vae.encode src/UniGenPipeline.py:306-308, vae.decode :430-433, :1120-1124) — SURVEY.md §8 (f)4.
extern "C" int ug_conv3x3_bf16(const ug_conv2d_args* args, void* stream) {
  using namespace ug;
  UG_CHECK_ARG(args != nullptr, "conv3x3: null args");
  const ug_conv2d_args& c = *args;
  UG_CHECK_ARG(c.x && c.w && c.y, "conv3x3: null operand pointer");
  UG_CHECK_ARG(c.batch >= 1 && c.h >= 1 && c.w_px >= 1, "conv3x3: empty image");
  UG_CHECK_ARG(c.c_in >= 64 && c.c_in % 64 == 0, "conv3x3: c_in (%d) must be a multiple of 64 (use ug_im2col_bf16 + ug_gemm_bf16 otherwise)", c.c_in);
  UG_CHECK_ARG(c.c_out >= 8 && c.c_out % 8 == 0 && c.y_pixel_stride >= c.c_out && c.y_pixel_stride % 8 == 0,
               "conv3x3: c_out (%d) and the output pixel stride (%d) must be multiples of 8", c.c_out, (int)c.y_pixel_stride);
  UG_CHECK_ARG(c.w_px % 128 == 0 || (c.w_px <= 128 && 128 % c.w_px == 0),
               "conv3x3: image width %d must be a multiple of 128 or divide 128 (use ug_im2col_bf16 + ug_gemm_bf16 otherwise)", c.w_px);
  UG_CHECK_ARG((reinterpret_cast<uintptr_t>(c.y) & 15) == 0 && (reinterpret_cast<uintptr_t>(c.x) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(c.w) & 15) == 0, "conv3x3: operands must be 16-byte aligned");
  if (c.bias) UG_CHECK_ARG((reinterpret_cast<uintptr_t>(c.bias) & 15) == 0, "conv3x3: bias alignment");
  if (c.residual)
    UG_CHECK_ARG((reinterpret_cast<uintptr_t>(c.residual) & 15) == 0 && c.res_pixel_stride >= c.c_out && c.res_pixel_stride % 8 == 0,
                 "conv3x3: residual alignment / pixel stride");
  ug_gemm_args g;
  memset(&g, 0, sizeof(g));
  const int rows = c.h * c.w_px;
  g.a = c.x; g.a_row_stride = c.c_in; g.a_batch_stride = (int64_t)rows * c.c_in;
  g.w = c.w; g.w_row_stride = 9 * c.c_in;
  g.c = c.y; g.c_row_stride = c.y_pixel_stride; g.c_batch_stride = (int64_t)rows * c.y_pixel_stride;
  g.batch = c.batch; g.rows = rows; g.n = c.c_out; g.k = 9 * c.c_in;
  g.bias = c.bias; g.alpha = c.alpha == 0.0f ? 1.0f : c.alpha; g.act = UG_ACT_NONE;
  g.residual = c.residual; g.res_row_stride = c.res_pixel_stride; g.res_batch_stride = (int64_t)rows * c.res_pixel_stride;
  const ConvDesc cd{c.x, c.batch, c.h, c.w_px, c.c_in};
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  int variant = c.variant;
  if (variant == 0) {
    variant = pick_tile_variant(c.batch, rows, c.c_out);
    variant = variant == 2 ? 4 : (variant == 1 ? 5 : 6);  // smem-staged TMA-store epilogue
    if (c.c_out <= 128) {
      // 128 output channels (the full-resolution level of the VAE): a 2-CTA pair on a 256-pixel x 128-channel tile — each CTA
      // stages its own 128 pixels and HALF of the filter block, 3/4 of the shared-memory operand traffic of a 128 x 128 CTA tile,
      // whose SS MMAs sit on the smem-bandwidth limit (ncu: 52 % tensor-pipe active at 1024^2 x 128)
      const long long pairs = (long long)c.batch * ((rows + 255) / 256);
      variant = pairs >= num_sms() / 2 ? 7 : 6;
    }
  }
  switch (variant) {
    case 1: return launch_gemm<1, 256, 4>(g, s, &cd);
    case 2: return launch_gemm<2, 256, 6>(g, s, &cd);
    case 3: return launch_gemm<1, 128, 6>(g, s, &cd);
    case 4: return launch_gemm<2, 256, 5, true>(g, s, &cd);
    case 5: return launch_gemm<1, 256, 3, true>(g, s, &cd);
    case 6: return launch_gemm<1, 128, 6, true>(g, s, &cd);
    case 7: return launch_gemm<2, 128, 7, true>(g, s, &cd);
    default:
      set_error("conv3x3: unknown variant %d", c.variant);
      return UG_ERR_INVALID;
  }
}
