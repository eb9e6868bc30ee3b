/* unigen_b200 — C ABI of the B200-native UniGen denoiser hot path (libunigen_b200.so).
 *
 * The reference (gavin-gqzhang/UniGen) has NO native boundary: its hot path sits behind a Python
 * torch.nn.Module (`UniGenFlux.forward`, src/UniGenTransformer.py:1182-1271) and calls diffusers /
 * deepspeed / torch library kernels.  This header is therefore the boundary a maintainer would bind
 * (ctypes stub in INTEGRATION.md); every entry point cites the reference call site it replaces.
 *
 * Conventions
 *   - plain C types only; all pointers are DEVICE pointers unless a parameter says "host".
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - every function returns UG_OK (0) or a negative ug_status; the message is in ug_last_error().
 *   - no function allocates device memory (except ug_peer_alloc), synchronises the stream, or falls back to the CPU.
 *   - strides are in ELEMENTS of the tensor's dtype; bf16 rows must be 16-byte aligned.
 *   - "batch" views: a logical [batch, rows, cols] tensor is (ptr, row_stride, batch_stride), which lets the
 *     text / image / condition streams live inside one joint buffer without concat copies.
 */
#ifndef UNIGEN_B200_H_
#define UNIGEN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UG_ABI_VERSION 11

typedef enum {
  UG_OK = 0,
  UG_ERR_INVALID = -1,     /* bad argument (shape / alignment / null) */
  UG_ERR_UNSUPPORTED = -2, /* valid request the sm_100a kernels do not cover (never a CPU fallback) */
  UG_ERR_CUDA = -3,        /* CUDA runtime / driver error; text in ug_last_error() */
  UG_ERR_NO_DEVICE = -4    /* no sm_100 device */
} ug_status;

/* Thread-local message of the last failing call on this thread. */
const char* ug_last_error(void);
int ug_abi_version(void);
/* UG_OK iff the current device is sm_100 (B200) and the TMA driver entry point resolves. */
int ug_device_check(void);
/* Number of kernels this library has launched on this thread since the last reset (bench.py's gpu_launches). */
int64_t ug_launch_count(void);
void ug_reset_launch_count(void);

/* ------------------------------------------------------------------------------------------------------
 * Dense bf16 GEMM on tcgen05 tensor cores with a fused epilogue.
 *   C[b,r,:] = residual[b,r,:] + alpha * gate[b,:] * act( A[b,r,:] @ W[wb]^T + bias[wb,:] )
 * Replaces every nn.Linear on the path (diffusers FluxTransformerBlock / FluxSingleTransformerBlock /
 * FluxAttnProcessor2_0 projections, SURVEY.md §8 A3-A6; zero-linears src/UniGenTransformer.py:755-773,1104;
 * expert linears :956-959) together with the elementwise ops the reference runs after them
 * (bias, GELU-tanh, `gate.unsqueeze(1) * out + residual`, `* conditioning_scale`).
 * A: [batch, rows, k] bf16, W: [n, k] bf16 (row-major, as nn.Linear.weight), C: [batch, rows, n] bf16.
 * ---------------------------------------------------------------------------------------------------- */
#define UG_ACT_NONE 0
#define UG_ACT_GELU_TANH 1
#define UG_MAX_SEGMENTS 8
#define UG_MAX_PEERS 8
#define UG_PEER_HEADER_BYTES 4096
#define UG_PEER_HANDLE_BYTES 64

typedef struct ug_gemm_args {
  const void* a;          /* bf16 */
  int64_t a_row_stride;
  int64_t a_batch_stride;
  const void* w;          /* bf16 [n,k] (or [batch,n,k] when w_batch_stride != 0) */
  int64_t w_row_stride;
  int64_t w_batch_stride; /* 0: weights shared by all batches */
  void* c;                /* bf16 */
  int64_t c_row_stride;
  int64_t c_batch_stride;
  int32_t batch;
  int32_t rows; /* rows per batch */
  int32_t n;
  int32_t k;
  const void* bias;       /* bf16 [n] or NULL */
  int64_t bias_batch_stride;
  const float* gate;      /* fp32 [batch, n] or NULL */
  int64_t gate_batch_stride;
  float alpha;            /* scalar factor (1.0f when unused) */
  int32_t act;            /* UG_ACT_* */
  const void* residual;   /* bf16 or NULL; may alias c (in-place residual update) */
  int64_t res_row_stride;
  int64_t res_batch_stride;
  int32_t variant;        /* 0 = auto; 1 = 1-CTA 128x256; 2 = 2-CTA 256x256 pair; 3 = 1-CTA 128x128 */
  int32_t reserved;
  /* Switched low-rank (LoRA) update fused into the epilogue — the `enable_lora(...)` context of the reference
   * (src/lora_switching_module.py:11-39; call sites UniCombineTransformerBlock.pyc L22,81,121,130,222,229,251,261,283,287)
   * expressed as data: rows [lora_seg_bounds[i], lora_seg_bounds[i+1]) of every batch use adapter group
   * lora_seg_group[i] (-1 = no adapter active on that segment):
   *     acc[r, c] += sum_j lora_t[r, (c / lora_block_n) * lora_rank + j] * lora_b[g(r)][c][j]
   * lora_t = x @ A_g^T from ug_lora_down (fp32); lora_b = B_g pre-multiplied by PEFT `scaling` (bf16 [groups, n, rank]);
   * lora_block_n = width of one sub-linear of a fused projection (D for to_q|to_k|to_v), 0 = n. lora_t NULL = off. */
  const float* lora_t;
  int64_t lora_t_row_stride;
  int64_t lora_t_batch_stride;
  const void* lora_b;
  int32_t lora_rank;      /* 4, 8, 12 or 16 */
  int32_t lora_block_n;
  int32_t lora_nseg;
  int32_t lora_seg_bounds[UG_MAX_SEGMENTS + 1];
  int32_t lora_seg_group[UG_MAX_SEGMENTS];
  /* Fused QK-RMSNorm + RoPE for the q|k|v projection GEMM (n = 3 * qk_d): every q / k head (qk_head_dim columns) is
   * RMS-normalised in fp32 straight from the TMEM accumulator, scaled by norm_q / norm_k, rotated with the (cos, sin)
   * table row of its token, and only then rounded to bf16 — diffusers RMSNorm + apply_rotary_emb after to_q/to_k
   * (SURVEY.md §A.2, §A.4; src/UniGenUtils.py:597-599) without a second pass over HBM. qk_norm_weight NULL = off. */
  const void* qk_norm_weight; /* bf16 [2, qk_head_dim]: norm_q.weight, norm_k.weight */
  const float* qk_cos_sin;    /* fp32 [rows, qk_head_dim] as written by ug_rope_table, row = row of the C view; NULL = no RoPE */
  int32_t qk_head_dim;        /* 64 or 128 */
  int32_t qk_d;               /* heads * head_dim */
  float qk_eps;
  int32_t reserved2;
  /* Per-segment gates: when != 0, rows of segment i of the row-segment table (lora_nseg / lora_seg_bounds, usable without a
   * LoRA update) take their gate vector from gate + i * gate_seg_stride (+ b * gate_batch_stride): the per-stream
   * `gate_msa` / `gate_mlp` of the P-variant's image and condition streams (UniCombineTransformerBlock.pyc L121-132, L222-230)
   * in ONE launch over all streams instead of one under-filled launch per stream. */
  int64_t gate_seg_stride;
  /* Second operand pair (K extension): the accumulator receives  A @ W^T + A2 @ W2^T  before the epilogue, both on the
   * tensor cores. A2: bf16 [batch, rows, k2] (a2_row_stride / a2_batch_stride), W2: bf16 [n, k2] shared by all batches.
   * Used for the switched LoRA update of the P-variant: A2 = the down-projection laid out in one 64-column block per
   * adapter group with zeros outside the row's own group (ug_lora_down_wide), W2 = [B_0 | B_1 | ...] (pre-scaled), so a
   * row only meets its own adapter's B and no tile-alignment of the segments is required. a2 == NULL: off. */
  const void* a2;
  int64_t a2_row_stride, a2_batch_stride;
  const void* w2;
  int64_t w2_row_stride;
  int32_t k2;
  /* Grouped projection mask: when != 0 (a multiple of 32), output columns are blocks of colmask_block columns and row r keeps
   * only block lora_seg_group[segment(r)] (-1: none); every other column is written as zero. With W = the adapter groups'
   * lora_A matrices stacked one block per group this IS ug_lora_down_wide on the tensor cores:
   * t_wide = x @ [A_0; A_1; ...]^T masked to the row's own group. Composes with no other epilogue op. */
  int32_t colmask_block;
} ug_gemm_args;

int ug_gemm_bf16(const ug_gemm_args* args, void* stream);

/* Row-wise FP8 (e4m3) GEMM: the same tiles, tile walk and epilogues as ug_gemm_bf16 with `a` / `w` read as float8_e4m3fn
 * (strides count elements = bytes; a / w row strides and k multiples of 16) and kind::f8f6f4 MMAs accumulating in fp32. The
 * accumulator is dequantised first, then the epilogue of ug_gemm_bf16 runs:
 *   acc[b, r, c] * a_scale[b, r] * w_scale[c]  ->  bias -> GELU-tanh -> gate * alpha -> residual   (or fused QK-norm + RoPE)
 * C, bias, residual and the QK-norm operands stay bf16 / fp32 as in ug_gemm_bf16. lora_t, colmask_block, a2 / w2 are rejected.
 * One fp32 scale per token row of A (dynamic, from ug_quant_rows_fp8 / ug_ln_modulate_fp8) and one per output channel of W
 * (`quantize_fp8()`): the "row-wise" scaling torch._scaled_mm offers. */
typedef struct ug_gemm_fp8_scales {
  const float* a_scale;          /* fp32 [batch, rows]: element (b, r) at a_scale[b * a_scale_batch_stride + r] */
  int64_t a_scale_batch_stride;
  const float* w_scale;          /* fp32 [n] (batched W: [batch, n] at w_scale[b * w_scale_batch_stride + c]) */
  int64_t w_scale_batch_stride;
} ug_gemm_fp8_scales;
int ug_gemm_fp8(const ug_gemm_args* args, const ug_gemm_fp8_scales* scales, void* stream);

/* ug_gemm_fp8 plus the two switched-LoRA features of the P-variant (`UniCombineFlux.quantize_fp8()`), on their own kernel
 * instances (the ones behind ug_gemm_fp8 are unchanged):
 *   - a bf16 second operand pair (a2 / w2 / k2, ug_gemm_args): its K blocks run as kind::f16 MMAs into the SAME fp32 accumulator
 *     as the e4m3 blocks, so the dequantisation multiplies both:  out = a_s[r] w_s[c] (sum_k q[r,k] Wq[c,k] + sum_j A2[r,j] W2[c,j]).
 *     For the LoRA update x A^T B^T pass the pre-divided operands A2 = (x / a_s) A^T and W2 = B / w_s[c] (the scaling is rank-1
 *     separable, so this is exact up to the bf16 rounding of A2 / W2);
 *   - colmask_block with its segment table (the masked grouped down-projection).
 * a_scale == NULL reads as unit row scales: with (q, a_s) = the quantised operand of x and W = the quantised stacked lora_A
 * (per-row scales aw_s) this gives A2 = q @ Aq^T * aw_s = (x / a_s) A^T directly. Tile variants, the auto picker and every
 * epilogue (direct, staged, fused QK-norm + RoPE, gate_seg_stride, bias, GELU, residual) are those of ug_gemm_fp8. Rejected:
 * lora_t, k % 16 != 0, a NULL w_scale. (The implicit-GEMM convolution is bf16-only: ug_conv3x3_bf16 has no fp8 form.) */
int ug_gemm_fp8_lora(const ug_gemm_args* args, const ug_gemm_fp8_scales* scales, void* stream);

/* Dynamic row-wise quantisation of bf16 [batch, rows, k] (strided) to e4m3 [batch, rows, k] plus one fp32 scale per row:
 *   amax = max |x|;  amax == 0: scale = 1, q = 0;  else inv = 448 / amax, scale = amax / 448 (IEEE divisions),
 *   q = cvt.rn.satfinite.e4m3(x * inv)        == torch (x.float() * inv).clamp(-448, 448).to(torch.float8_e4m3fn)
 * scale element (b, r) at scale[b * scale_batch_stride + r]. k a multiple of 8, at most 16384; rows 16-byte aligned. */
int ug_quant_rows_fp8(const void* x, int64_t x_row_stride, int64_t x_batch_stride, void* q, int64_t q_row_stride,
                      int64_t q_batch_stride, float* scale, int64_t scale_batch_stride, int32_t batch, int32_t rows, int32_t k,
                      void* stream);

/* LoRA down-projection for ug_gemm_bf16's fused update: t[b, r, :] = x[b, r, :] @ A[g(r)]^T  (fp32 out).
 * a_stack: bf16 [groups, rank_total, k] (rank_total = n_sub_linears * rank for a fused projection); rows whose
 * segment has group -1 get zeros. peft 0.15 lora.Linear: lora_A (SURVEY.md §A.6). */
int ug_lora_down(const void* x, int64_t x_row_stride, int64_t x_batch_stride, const void* a_stack, float* t,
                 int64_t t_row_stride, int64_t t_batch_stride, int32_t batch, int32_t rows, int32_t k,
                 int32_t rank_total, int32_t nseg, const int32_t* seg_bounds_host, const int32_t* seg_group_host,
                 void* stream);
/* Same down-projection written for the K-extension form of the update (ug_gemm_args.a2): t_wide bf16 [batch, rows,
 * groups * block] with block >= rank_total a multiple of 64; row r holds x[r] @ A[g(r)]^T in columns
 * [g(r) * block, g(r) * block + rank_total) and ZEROS everywhere else (peft computes lora_A's output in the model dtype,
 * so the bf16 rounding of t matches the reference). */
int ug_lora_down_wide(const void* x, int64_t x_row_stride, int64_t x_batch_stride, const void* a_stack, void* t_wide,
                      int64_t t_row_stride, int64_t t_batch_stride, int32_t batch, int32_t rows, int32_t k,
                      int32_t rank_total, int32_t groups, int32_t block, int32_t nseg, const int32_t* seg_bounds_host,
                      const int32_t* seg_group_host, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Joint attention (tcgen05 / TMEM / TMA), softmax(Q K^T * scale + mask) V per head, non-causal.
 * Replaces F.scaled_dot_product_attention in diffusers FluxAttnProcessor2_0 (SURVEY.md §8 A5; same call in
 * src/UniGenUtils.py:601,709) and the per-segment SDPA calls of the predecessor's attn_forward
 * (UniCombineTransformerBlock.pyc L98-110, SURVEY.md §8 A11).
 * q/k/v/o: bf16 [batch, seq, heads, head_dim] views: element (b,s,h,d) at ptr[b*batch_stride + s*row_stride + h*head_dim + d].
 * Segment visibility (optional): tokens [seg_bounds[i], seg_bounds[i+1]) form segment i; a query in segment i
 * attends keys of segment j iff bit j of seg_visible[i] is set. n_seg = 0 means full attention.
 * seg_bounds / seg_visible are HOST pointers (copied into the launch parameters).
 * ---------------------------------------------------------------------------------------------------- */
typedef struct ug_attn_args {
  const void* q;
  const void* k;
  const void* v;
  void* o;
  int64_t q_row_stride, q_batch_stride;
  int64_t k_row_stride, k_batch_stride;
  int64_t v_row_stride, v_batch_stride;
  int64_t o_row_stride, o_batch_stride;
  int32_t batch, heads, seq, head_dim; /* head_dim in {64, 128}; seq_q == seq_k == seq */
  float scale;                         /* 1/sqrt(head_dim) in the reference */
  int32_t n_seg;
  const int32_t* seg_bounds;   /* host, n_seg + 1 entries, seg_bounds[0] = 0, seg_bounds[n_seg] = seq */
  const uint32_t* seg_visible; /* host, n_seg entries */
  int32_t variant;             /* 0 = auto (5 when the 256-row tiles fill the SMs, else 1); 1 = 128-row tile, P in TMEM; 2 = 128-row tile, P
                                * staged in smem; 3 = two 128-row tiles ping-pong; 4 / 6 = as 3 with every 4th / 3rd pair of exponentials
                                * on the FMA pipe (packed polynomial) instead of MUFU.EX2; 5 = as 3 with P published in two 64-key halves;
                                * 7 = 5 as a persistent grid (one CTA per SM walks the (query tile, head) units, next unit's Q / K / V
                                * prefetched, epilogue overlapped with the next unit's first MMAs; bit-identical, measured 2-3 % slower) */
  int32_t reserved;
} ug_attn_args;

int ug_attention_bf16(const ug_attn_args* args, void* stream);
/* Bit-exact expansion of the segment rule into a dense [seq, seq] uint8 mask (1 = visible); parity helper for
 * the "condition attention mask" construction (north_star: bit-exact mask). */
int ug_expand_segment_mask(int32_t seq, int32_t n_seg, const int32_t* seg_bounds_host,
                           const uint32_t* seg_visible_host, uint8_t* mask_dev, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Fused elementwise family (HBM-bound).
 * ---------------------------------------------------------------------------------------------------- */
/* out[b,r,:] = LayerNorm(x[b,r,:], eps, no affine) * (1 + scale[b,:]) + shift[b,:]      (bf16 in/out, fp32 math)
 * diffusers AdaLayerNormZero / AdaLayerNormZeroSingle / AdaLayerNormContinuous and `norm2(h)*(1+scale)+shift`
 * (SURVEY.md §A.2-A.4; reference-owned copies src/UniGenUtils.py:345-351,360-362,370-372). */
int ug_ln_modulate(const void* x, int64_t x_row_stride, int64_t x_batch_stride, void* out, int64_t o_row_stride,
                   int64_t o_batch_stride, const float* shift, const float* scale, int64_t mod_batch_stride,
                   int32_t batch, int32_t rows, int32_t d, float eps, void* stream);

/* ug_ln_modulate followed by the row quantisation of ug_quant_rows_fp8 in one pass: every value is rounded to bf16 first, so
 * (q, q_scale) equal ug_quant_rows_fp8(ug_ln_modulate(x)) bit for bit. The operand of the fp8 GEMMs that read a modulated
 * LayerNorm (q|k|v, ff.net.0, proj_mlp). q: e4m3 [batch, rows, d]; q_scale: fp32, (b, r) at q_scale[b * q_scale_batch_stride + r]. */
int ug_ln_modulate_fp8(const void* x, int64_t x_row_stride, int64_t x_batch_stride, void* q, int64_t q_row_stride,
                       int64_t q_batch_stride, float* q_scale, int64_t q_scale_batch_stride, const float* shift, const float* scale,
                       int64_t mod_batch_stride, int32_t batch, int32_t rows, int32_t d, float eps, void* stream);

/* ug_ln_modulate with one modulation vector per ROW SEGMENT: rows [seg_bounds[i], seg_bounds[i+1]) of every sample use
 * shift/scale + i * mod_seg_stride (+ b * mod_batch_stride) — the text / image / condition streams of a P-variant block
 * (each with its own AdaLN vectors, UniCombineTransformerBlock.pyc L152-170, L207-218) normalised in ONE launch. */
int ug_ln_modulate_segs(const void* x, int64_t x_row_stride, int64_t x_batch_stride, void* out, int64_t o_row_stride,
                        int64_t o_batch_stride, const float* shift, const float* scale, int64_t mod_batch_stride,
                        int64_t mod_seg_stride, int32_t nseg, const int32_t* seg_bounds_host, int32_t batch, int32_t rows,
                        int32_t d, float eps, void* stream);

/* ug_ln_modulate_segs with the e4m3 output of ug_ln_modulate_fp8: (q, q_scale) equal ug_quant_rows_fp8(ug_ln_modulate_segs(x))
 * bit for bit. The shared operand of a quantised P-variant block's text, image / condition and LoRA down-projection GEMMs. */
int ug_ln_modulate_segs_fp8(const void* x, int64_t x_row_stride, int64_t x_batch_stride, void* q, int64_t q_row_stride,
                            int64_t q_batch_stride, float* q_scale, int64_t q_scale_batch_stride, const float* shift,
                            const float* scale, int64_t mod_batch_stride, int64_t mod_seg_stride, int32_t nseg,
                            const int32_t* seg_bounds_host, int32_t batch, int32_t rows, int32_t d, float eps, void* stream);

/* Per-token AdaLN on capacity-slot buffers — the SD3.5 transformer-block experts run `SD3SingleTransformerBlock` on the
 * dispatched (1, C, D) chunks with a PER-TOKEN (1, C, D) temb (src/UniGenUtils.py:354-363,386-414 with a 3-D `emb`;
 * src/UniGenTransformer.py:256-258). A dispatched temb row is the temb of the sample the slot's token came from, or 0 for
 * an empty slot, so its AdaLN vector is one of (samples + 1) distinct rows:
 *   idx(r) = slot_token[r] < 0 ? empty_index : slot_token[r] / tokens_per_batch,   e(r) = r / capacity
 *   out[r,:] = LayerNorm(x[r,:]) * (1 + scale[e, idx, :]) + shift[e, idx, :]         r in [0, experts*capacity)
 * shift/scale: fp32, element (e, idx, c) at ptr[e*mod_expert_stride + idx*mod_index_stride + c]. */
int ug_ln_modulate_slots(const void* x, int64_t x_row_stride, void* out, int64_t o_row_stride, const float* shift,
                         const float* scale, int64_t mod_expert_stride, int64_t mod_index_stride,
                         const int32_t* slot_token, int32_t experts, int32_t capacity, int32_t tokens_per_batch,
                         int32_t empty_index, int32_t d, float eps, void* stream);
/* x[r,:] += gate[e(r), idx(r), :] * y[r,:] — `gate_msa * attn_output` / `gate_mlp * ff_output` + residual of the same
 * per-token AdaLN (src/UniGenUtils.py:399-400,410-412). x, y bf16; gate fp32 with the strides above. */
int ug_gated_add_slots(void* x, int64_t x_row_stride, const void* y, int64_t y_row_stride, const float* gate,
                       int64_t mod_expert_stride, int64_t mod_index_stride, const int32_t* slot_token, int32_t experts,
                       int32_t capacity, int32_t tokens_per_batch, int32_t empty_index, int32_t d, void* stream);

/* In-place per-head RMSNorm (learned weight) followed by interleaved-pair RoPE on rows of a [batch, rows, heads, dh]
 * bf16 view: diffusers RMSNorm(dh, eps) + apply_rotary_emb (SURVEY.md §A.2, §A.4; src/UniGenUtils.py:597-599).
 * norm_weight: bf16 [heads / heads_per_weight, dh] — head h uses row h / heads_per_weight, so the Q and K halves of a
 * fused QKV buffer (heads = 2H, heads_per_weight = H) are normalised with norm_q / norm_k in one launch
 * (heads_per_weight <= 0: one weight row for all heads).
 * cos_sin: fp32 [rows, dh/2, 2] (cos, sin of pair i) shared by all batches/heads, or NULL for no rotation. */
int ug_qk_rmsnorm_rope(void* x, int64_t row_stride, int64_t batch_stride, int32_t batch, int32_t rows,
                       int32_t heads, int32_t head_dim, const void* norm_weight_bf16, int32_t heads_per_weight,
                       float eps, const float* cos_sin, void* stream);

/* RoPE table from position ids: FluxPosEmbed(theta, axes_dim)(ids) (SURVEY.md §A.4), float64 angles -> fp32.
 * ids: fp32 [rows, 3]; axes_dim: host int[3] (sum = head_dim); out: fp32 [rows, head_dim/2, 2]. */
int ug_rope_table(const float* ids, int32_t rows, const int32_t* axes_dim_host, float theta, float* cos_sin,
                  void* stream);

/* Small-M linear (M = batch rows <= 16): out[b,n] (+)= W[n,:] . f(x[b,:]) + bias[n], f = SiLU when silu_in.
 * fp32 x / out, bf16 W / bias. HBM-bound weight streaming. Replaces AdaLN `linear(silu(temb))`, TimestepEmbedding,
 * PixArtAlphaTextProjection and the expert modulation linears `L^e(pooled)` (src/UniGenTransformer.py:956-959). */
int ug_gemv(const float* x, int64_t x_stride, const void* w, const void* bias, float* out, int64_t out_stride,
            int32_t batch, int32_t n, int32_t k, int32_t silu_in, int32_t silu_out, int32_t accumulate,
            void* stream);

/* Grouped small-M linear: every job j is an independent ug_gemv  out_j[b, :] = W_j @ f(x_j[b, :]) + bias_j  and ONE launch
 * streams all of them — the AdaLN `linear(silu(temb))` of every block of a denoise step (temb / condition_temb are step
 * constants, SURVEY.md §7 step 4: "compute ALL blocks' shift / scale / gate vectors in one batched pass at step start").
 * The job table lives in DEVICE memory (built once per workspace; nothing is copied at launch, so the call is graph-capturable).
 * Work unit = a group of 4 consecutive output rows; job j owns groups [first_group_j, first_group_j + ceil(n_j / 4)) of the
 * launch-wide list (first_group ascending, total_groups = their sum). [group_begin, group_end) selects the part THIS call
 * computes: the whole list on one GPU, rank r's 1/world share under sequence parallelism — there `peers` is the pool table and
 * every job's `out` is a BYTE OFFSET into the pools: each result is stored into every rank's pool, which all-gathers the table
 * (follow with ug_peer_barrier). n_j, k_j multiples of 8; x rows 16-byte aligned; batch <= 8. */
#define UG_MAX_GEMV_JOBS 1024
struct ug_peer_table;
typedef struct ug_gemv_job {
  const void* w;      /* bf16 [n, k], contiguous */
  const void* bias;   /* bf16 [n] or NULL */
  const float* x;     /* fp32 [batch, k] */
  float* out;         /* fp32 [batch, n]; with a peer table: byte offset into every rank's pool, cast to a pointer */
  int64_t x_stride, out_stride; /* elements */
  int32_t n, k;
  int32_t first_group;
  int32_t flags;      /* bit 0: f = SiLU; bit 1: out += result (with peers: added to this rank's own copy, so every copy must
                         already hold the same value — issue a ug_peer_barrier after the launch that produced it) */
} ug_gemv_job;
int ug_gemv_grouped(const ug_gemv_job* jobs_dev, int32_t n_jobs, int32_t total_groups, int32_t batch, int32_t group_begin,
                    int32_t group_end, const struct ug_peer_table* peers_or_null, void* stream);
/* out = x * sigmoid(x), fp32, n elements — `silu(temb)` once per step instead of once per AdaLN linear. */
int ug_silu_f32(const float* x, float* out, int64_t n, void* stream);

/* Timesteps(256, flip_sin_to_cos=True, downscale_freq_shift=0): out[b] = [cos(s*f) | sin(s*f)], s = scale * t[b * t_stride]
 * (SURVEY.md §A.4). `scale` folds the `timestep * 1000` / `guidance * 1000` of UniGenFlux.forward
 * (src/UniGenTransformer.py:1217-1220) into the kernel; t_stride = 0 broadcasts one device-resident value (entry i of the
 * sigma table of a graph-captured denoise loop) to every sample. */
int ug_timestep_embedding(const float* t, int64_t t_stride, int32_t batch, int32_t dim, float scale, float* out, void* stream);

/* out = a + b (bf16, same [batch, rows, d] view conventions). `hidden_states+condition_hidden_states`
 * (src/UniGenTransformer.py:979,1089) and the weave add (:1141,1166). */
int ug_add_bf16(const void* a, int64_t a_row_stride, int64_t a_batch_stride, const void* b, int64_t b_row_stride,
                int64_t b_batch_stride, void* out, int64_t o_row_stride, int64_t o_batch_stride, int32_t batch,
                int32_t rows, int32_t d, void* stream);
/* strided 2-D copy of bf16 rows (torch.cat / slicing on the path: src/UniGenTransformer.py:1146,1174). */
int ug_copy_bf16(const void* src, int64_t s_row_stride, int64_t s_batch_stride, void* dst, int64_t d_row_stride,
                 int64_t d_batch_stride, int32_t batch, int32_t rows, int32_t d, void* stream);
/* fp32 -> bf16 and bf16 -> fp32 contiguous casts (pipeline boundary dtype glue). */
int ug_cast_f32_to_bf16(const float* src, void* dst, int64_t n, void* stream);
int ug_cast_bf16_to_f32(const void* src, float* dst, int64_t n, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * CoMoE pre-stage: DeepSpeed top-1 gate with Random-Token-Selection (SURVEY.md §A.5) as sparse index work
 * instead of dense (S,E,C) one-hot einsums (src/UniGenUtils.py:99,140,183).
 *   x            bf16 [tokens, d]    gate input `(hidden+cond).reshape(-1, d)`
 *   wg           fp32 [experts, d]   TopKGate.wg.weight
 *   rts_uniform  fp32 [tokens, experts]  the uniform draw of top1gating (injected for parity)
 * outputs
 *   expert_idx   int32 [tokens]      argmax expert
 *   slot         int32 [tokens]      position inside the expert's capacity buffer, -1 when dropped
 *   prob         fp32  [tokens]      softmax probability of the chosen expert (combine weight)
 *   slot_token   int32 [experts*capacity]  inverse map, -1 for empty slots
 *   exp_counts   int64 [experts]     pre-capacity counts (add_outputs['expert_counts'])
 *   l_aux        fp32  [1]
 * workspace: fp32 [tokens*experts] (softmax gates) ; capacity = max(ceil(tokens/experts), 4) is computed by the caller.
 * ---------------------------------------------------------------------------------------------------- */
int ug_moe_route(const void* x, const float* wg, const float* rts_uniform, int32_t tokens, int32_t d,
                 int32_t experts, int32_t capacity, int32_t* expert_idx, int32_t* slot, float* prob,
                 int32_t* slot_token, int64_t* exp_counts, float* l_aux, float* workspace, void* stream);

/* Gather + modulate: out[e*capacity + s, :] = mod[e, b(token), :] * (x[token, :] (+ addend[e*capacity+s, :]))
 * with token = slot_token[e*capacity+s]; empty slots give zero rows. tokens_per_batch maps token -> b.
 * mod == NULL: plain dispatch (einsum sec,sm->ecm of src/UniGenUtils.py:140) without modulation.
 * `s ⊙ x` prologue of modulated_flatten (src/UniGenUtils.py:204-228) on the dispatched rows. */
int ug_moe_gather_modulate(const void* x, const int32_t* slot_token, const float* mod, int64_t mod_expert_stride,
                           int64_t mod_batch_stride, const void* addend, void* out, int32_t experts,
                           int32_t capacity, int32_t tokens_per_batch, int32_t d, void* stream);
/* Combine: out[token,:] = prob[token] * y[expert_idx*capacity + slot, :] or 0 when dropped (einsum sec,ecm->sm,
 * src/UniGenUtils.py:183-185). */
int ug_moe_combine(const void* y, const int32_t* expert_idx, const int32_t* slot, const float* prob, void* out,
                   int32_t tokens, int32_t capacity, int32_t d, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Denoise-loop glue (callers of the path: src/UniGenPipeline.py:1050-1116), kept on the device between steps.
 * ---------------------------------------------------------------------------------------------------- */
/* FlowMatchEulerDiscreteScheduler.step: latents <- bf16(float(latents) + (sigma_next - sigma) * float(velocity)), n elements. */
int ug_euler_step(void* latents_bf16, const void* velocity_bf16, float sigma, float sigma_next, int64_t n, void* stream);
/* Same update with the schedule resident on the device: sigma = sigmas[step], sigma_next = sigmas[step + 1] (fp32 table of
 * num_steps + 1 entries, src/UniGenPipeline.py:989-1006) are read by the kernel, so a whole sampling loop captured in ONE CUDA
 * graph needs no host value between steps. */
int ug_euler_step_table(void* latents_bf16, const void* velocity_bf16, const float* sigmas_dev, int32_t step, int64_t n,
                        void* stream);
/* classifier-free guidance (src/UniGenPipeline.py:405-412): out = uncond + guidance_scale * (text - uncond). */
int ug_cfg_combine(const void* uncond_bf16, const void* text_bf16, float guidance_scale, void* out_bf16, int64_t n, void* stream);
/* FluxPipeline._pack_latents (unpack = 0): (B, C, H, W) -> (B, (H/2)(W/2), 4C); _unpack_latents (unpack = 1): inverse. */
int ug_pack_latents(const void* src_bf16, void* dst_bf16, int32_t batch, int32_t channels, int32_t height, int32_t width,
                    int32_t unpack, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Ulysses sequence parallelism over peer memory (NVLink 5 / NVSwitch), one process per GPU — north_star subsystem (4).
 * The reference has no sequence parallelism (SURVEY.md §5, §8e); these entry points are the exchange step of the
 * sharded forward, fused into the kernels that produce the data instead of staging copies + NCCL all-to-all.
 * Every rank allocates a pool of the same size; bytes [0, UG_PEER_HEADER_BYTES) are the control block (barrier flags,
 * epoch, error word), payload buffers live at offsets the host chooses identically on all ranks.
 * ---------------------------------------------------------------------------------------------------- */
typedef struct ug_peer_table {
  int32_t world, rank;
  void* base[UG_MAX_PEERS]; /* this process's mapping of rank r's pool; base[rank] = the local pool */
} ug_peer_table;

/* cudaMalloc'd, zero-filled pool / cudaFree. (The only allocating calls of the ABI: IPC export needs a cudaMalloc base.) */
int ug_peer_alloc(size_t bytes, void** dev_ptr);
int ug_peer_free(void* dev_ptr);
/* CUDA IPC handle of a pool (exchange the 64 bytes through any host channel, e.g. torch.distributed.all_gather_object). */
int ug_peer_export(const void* dev_ptr, uint8_t handle[UG_PEER_HANDLE_BYTES]);
int ug_peer_open(const uint8_t handle[UG_PEER_HANDLE_BYTES], void** peer_ptr);
int ug_peer_close(void* peer_ptr);
/* Device-side barrier of all ranks on `stream` (release/acquire flags in the control blocks; no host sync; graph-capturable).
 * Every rank must issue the same sequence of barriers, and the ranks must be host-synchronised (e.g. a process-group
 * barrier) before the first one. A rank that waits longer than the timeout (default 20 s, env UG_PEER_TIMEOUT_MS or
 * ug_peer_set_timeout_ms) sets the STICKY error word to 1 + the rank that did not arrive instead of hanging; later barriers
 * then no longer wait. Everything computed after the word was set is invalid: poll it with ug_peer_error(_async). */
int ug_peer_barrier(const ug_peer_table* table, void* stream);
int ug_peer_set_timeout_ms(int64_t milliseconds);
/* Reads the local error word (synchronous cudaMemcpy): 0 = every barrier so far completed. */
int ug_peer_error(const ug_peer_table* table, int32_t* error_host);
/* Stream-ordered, graph-capturable copy of the error word into PINNED host memory (no host sync). */
int ug_peer_error_async(const ug_peer_table* table, int32_t* error_host_pinned, void* stream);

/* seq-shard x all heads -> all tokens x head-shard, fused with the per-token QK-RMSNorm + RoPE pass:
 * reads `rows` local rows of the fused q|k|v projection ([rows, 3*heads*head_dim] bf16), normalises / rotates the q and k
 * heads exactly like ug_qk_rmsnorm_rope, and stores head h of block `which` (q, k, v) into rank h / (heads/world)'s
 * receive buffer  recv[which][dst_row0 + r][(h % (heads/world)) * head_dim ...],  recv = bf16 [3, seq_total,
 * heads/world*head_dim] at byte `dst_offset` of that rank's pool. */
typedef struct ug_qkv_scatter_args {
  const void* qkv;
  int64_t row_stride;
  int32_t rows, heads, head_dim;
  float eps;
  const void* norm_weight; /* bf16 [2, head_dim] (norm_q, norm_k) or NULL */
  const float* cos_sin;    /* fp32 [rows, head_dim] rows of the LOCAL tokens, or NULL */
  int64_t dst_offset;
  int32_t seq_total, dst_row0;
} ug_qkv_scatter_args;
int ug_qkv_scatter(const ug_peer_table* table, const ug_qkv_scatter_args* args, void* stream);

/* ug_attention_bf16 over this rank's head shard of ALL tokens with the heads -> sequence exchange fused into the epilogue:
 * output row q is stored into rank q / rows_per_rank's buffer (bf16 rows of args->o_row_stride elements at byte `o_offset`
 * of its pool) at row q % rows_per_rank, columns [rank*heads*head_dim, (rank+1)*heads*head_dim). args->o is ignored.
 * rows_per_rank == 0 selects SEGMENT-SHARDED rows (needs args->n_seg >= 1, every bound a multiple of world): each segment
 * [b_s, b_{s+1}) is split evenly over the ranks and a rank keeps its shards in segment order, so row q of segment s goes to
 * rank (q - b_s) / ((b_{s+1} - b_s) / world), local row b_s / world + (q - b_s) % ((b_{s+1} - b_s) / world) — the layout of the
 * sequence-parallel P-variant, where every rank holds 1/world of the text, image and each condition stream. */
int ug_attention_bf16_peer(const ug_attn_args* args, const ug_peer_table* table, int64_t o_offset, int32_t rows_per_rank,
                           void* stream);

/* All-gather by peer stores: rows [dst_row0, dst_row0 + rows) of the bf16 buffer at byte `dst_offset` of EVERY rank's pool
 * <- src rows (the residual stream for the replicated CoMoE pre-stage; the final velocity). */
int ug_peer_bcast_rows(const ug_peer_table* table, const void* src, int64_t src_row_stride, int32_t rows, int32_t d,
                       int64_t dst_offset, int64_t dst_row_stride, int32_t dst_row0, void* stream);

/* SD3 un-patchify (src/UniGenTransformer.py:693-704, `nhwpqc->nchpwq`): tokens bf16 (B, h*w, p*p*C) whose channel index is
 * (py*p + px)*C + c  ->  image bf16 (B, C, h*p, w*p). (The patchify side of diffusers PatchEmbed's Conv2d(k=2, s=2) is
 * ug_pack_latents: channel = c*4 + py*2 + px is exactly the flattened conv-weight layout, so the conv is one ug_gemm_bf16.) */
int ug_unpatchify(const void* tokens_bf16, void* image_bf16, int32_t batch, int32_t h, int32_t w, int32_t p, int32_t channels,
                  void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Whole-step handle: ONE denoise step of UniGenFlux (`UniGenFlux.forward`, src/UniGenTransformer.py:1182-1271, with
 * base_forward :1106-1180, control_forward :1070-1104, preprocess_moe_forward :1028-1068, moe_forward :969-1026) sequenced inside
 * the library, for hosts that are not Python (SURVEY.md §8(b) "what a C-ABI replacement must export"). The handle owns no device
 * memory: weights are BORROWED pointers bound under the reference's state-dict names, the caller supplies one workspace.
 *   ug_flux_create / ug_flux_destroy
 *   ug_flux_bind_weight(handle, "transformer_blocks.0.attn.to_q.weight", ptr, dtype, shape, ndim)   dtype 0 = bf16, 1 = fp32
 *       every key of the reference state dict (diffusers Flux names + control_*, controlnet_add_*, moe.*, shared_expert.*);
 *       bf16 except `moe.moe_layer.gate.wg.weight` (fp32, as DeepSpeed evaluates the gate). Rows that one fused launch reads
 *       must be CONTIGUOUS in memory: to_q|to_k|to_v (and add_q|k|v_proj) weights and biases of a block, norm_q|norm_k
 *       (norm_added_q|k) weights, and the E experts' `.{br}.0` / `.{br}.1` linears stacked in expert order.
 *   ug_flux_workspace_bytes(handle, batch, n_img, n_txt)
 *   ug_flux_forward(handle, inputs, outputs, workspace, bytes, stream)
 *       never allocates, never synchronises — except on the FIRST call with a new (workspace, shape), which uploads the AdaLN
 *       job table and must therefore not run under stream capture; later calls are capturable into a CUDA graph.
 * Numerics: the same kernels in the same order as the Python mirror (unigen_b200/model.py) — bit-identical results.
 * ---------------------------------------------------------------------------------------------------- */
#define UG_FLUX_MAX_CONDITIONS 4
typedef struct ug_flux_desc {
  int32_t num_layers, num_single_layers;     /* 19, 38 */
  int32_t heads, head_dim;                   /* 24, 128 */
  int32_t in_channels, joint_dim, pooled_dim; /* 64, 4096, 768 */
  int32_t guidance_embeds;
  int32_t axes_dims_rope[3];                 /* 16, 56, 56 */
  float theta;                               /* 10000 */
  int32_t n_ctrl_double, n_ctrl_single;      /* num_layers // single_control_dev, num_single_layers // single_control_dev (0: none) */
  int32_t experts, condition_nums;           /* (condition_nums + 1) * expert_num_each_condition, 1 */
  int32_t use_shared_expert, single_add, use_pooled_prompt_embeds; /* control_params (config/unigen.yaml) */
} ug_flux_desc;
typedef struct ug_flux ug_flux;
typedef struct ug_flux_inputs {
  int32_t batch, n_img, n_txt;
  float conditioning_scale;
  const void* hidden_states;         /* bf16 [batch, n_img, in_channels] */
  const void* encoder_hidden_states; /* bf16 [batch, n_txt, joint_dim] */
  const float* pooled_projections;   /* fp32 [batch, pooled_dim] */
  const float* timestep;             /* fp32, already divided by 1000 as the pipeline passes it; element b at timestep[b * timestep_stride] */
  int64_t timestep_stride;           /* 1, or 0 to broadcast one device-resident value (a sigma-table entry) */
  const float* guidance;             /* fp32 [batch] or NULL */
  const float* img_ids;              /* fp32 [n_img, 3] */
  const float* txt_ids;              /* fp32 [n_txt, 3] */
  const void* condition_hidden_states[UG_FLUX_MAX_CONDITIONS];       /* bf16 [batch, n_img, in_channels] per condition */
  const float* condition_pooled_projections[UG_FLUX_MAX_CONDITIONS]; /* fp32 [batch, pooled_dim] */
  const float* condition_ids[UG_FLUX_MAX_CONDITIONS];                /* fp32 [n_img, 3] */
  const float* rts_uniform[UG_FLUX_MAX_CONDITIONS];                  /* fp32 [batch * n_img, experts]: the gate's uniform draw */
} ug_flux_inputs;
typedef struct ug_flux_outputs {
  void* velocity;         /* bf16 [batch, n_img, in_channels] */
  int64_t* expert_counts; /* int64 [experts] (last condition) */
  float* l_aux;           /* fp32 [1]; moe_loss = 0.1 * l_aux */
} ug_flux_outputs;
int ug_flux_create(const ug_flux_desc* desc, ug_flux** handle);
void ug_flux_destroy(ug_flux* handle);
int ug_flux_bind_weight(ug_flux* handle, const char* name, const void* dev_ptr, int32_t dtype, const int64_t* shape, int32_t ndim);
size_t ug_flux_workspace_bytes(const ug_flux* handle, int32_t batch, int32_t n_img, int32_t n_txt);
int ug_flux_forward(ug_flux* handle, const ug_flux_inputs* inputs, const ug_flux_outputs* outputs, void* workspace,
                    size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * AutoencoderKL (VAE) ops — SURVEY.md §8 (f)4 tail: the condition image is VAE-encoded before the denoise loop
 * (`vae.encode(control_image).latent_dist.sample()`, src/UniGenPipeline.py:306-308; Flux: `Condition._encode_image`
 * src/condition.py:90-99) and the final latents are VAE-decoded after it (:430-433, :1120-1124). Activations are NHWC bf16
 * ([batch, h, w, c] contiguous; a "pixel row" is one (b, y, x) with c channels), so every convolution is a GEMM over pixel rows.
 * ---------------------------------------------------------------------------------------------------- */
typedef struct ug_conv2d_args {
  const void* x;            /* bf16 NHWC [batch, h, w_px, c_in], contiguous */
  const void* w;            /* bf16 [c_out, 9 * c_in]: column (ky * 3 + kx) * c_in + c  (nn.Conv2d weight permuted to [co, ky, kx, ci]) */
  const void* bias;         /* bf16 [c_out] or NULL */
  const void* residual;     /* bf16 NHWC [batch, h, w_px, res_pixel_stride] or NULL; may alias y */
  int64_t res_pixel_stride;
  void* y;                  /* bf16 NHWC [batch, h, w_px, y_pixel_stride] */
  int64_t y_pixel_stride;   /* elements between output pixels (>= c_out, multiple of 8) */
  int32_t batch, h, w_px, c_in, c_out;
  float alpha;              /* y = alpha * (conv + bias) + residual; 0 is read as 1 */
  int32_t variant;          /* 0 = auto; 1-6 = the GEMM tile variants of ug_gemm_args; 7 = 2-CTA pair on a 256 x 128 tile (c_out <= 128) */
  int32_t reserved;
} ug_conv2d_args;
/* nn.Conv2d(c_in, c_out, kernel_size=3, stride=1, padding=1) as an IMPLICIT GEMM on the tcgen05 path: the TMA unit assembles
 * each [128 pixels x 64 channels] A tile from the image at the filter tap's offset (zero fill outside the image), no im2col
 * buffer. Needs c_in % 64 == 0 and w_px a multiple of 128 or a divisor of 128; other shapes: ug_im2col_bf16 + ug_gemm_bf16. */
int ug_conv3x3_bf16(const ug_conv2d_args* args, void* stream);

/* Patch gather for the convolutions the implicit path does not take (stride 2 `Downsample2D` with its (0,1,0,1) padding,
 * c_in = 3 / 16 stems): cols[(b, yo, xo), (ky * kw + kx) * c + ch] = x[b, yo * stride + ky - pad_top, xo * stride + kx - pad_left, ch]
 * (0 outside the image, 0 in columns [kh * kw * c, k_pad)). x is addressed through element strides, so NCHW fp32 / bf16 inputs
 * (the pixel-space image, the latents) and NHWC bf16 activations are all accepted. In-image values pass through
 * alpha * x + beta (the `latents / scaling_factor + shift_factor` in front of the decoder's first convolution, whose zero
 * padding must stay zero; alpha = 1, beta = 0 otherwise). cols: bf16 [batch * h_out * w_out, k_pad]. */
int ug_im2col_bf16(const void* x, int32_t x_is_f32, int64_t sb, int64_t sy, int64_t sx, int64_t sc, void* cols, int32_t batch,
                   int32_t h, int32_t w, int32_t c, int32_t kh, int32_t kw, int32_t stride, int32_t pad_top, int32_t pad_left,
                   int32_t h_out, int32_t w_out, int32_t k_pad, float alpha, float beta, void* stream);

/* GroupNorm(groups, c, eps, affine) [+ SiLU] over NHWC bf16 [batch, pixels, c]: statistics in fp32, deterministic (no atomics):
 * per-block sums shifted by a pivot from the image (no cancellation when the mean is large against the spread) -> fixed-order
 * merge of the blocks' (mean, M2) pairs -> normalise / scale / shift / activate (three launches). `stats`: fp32 scratch of
 * batch * groups * 2 * (1 + UG_GROUPNORM_MAX_CHUNKS) elements. y may alias x. */
#define UG_GROUPNORM_MAX_CHUNKS 1024
int ug_groupnorm_bf16(const void* x, void* y, const void* gamma, const void* beta, float* stats, int32_t batch, int32_t pixels,
                      int32_t c, int32_t groups, float eps, int32_t silu, void* stream);

/* F.interpolate(scale_factor=2, mode="nearest") over NHWC bf16: [batch, h, w, c] -> [batch, 2h, 2w, c] (`Upsample2D`). */
int ug_upsample2x_nhwc_bf16(const void* x, void* y, int32_t batch, int32_t h, int32_t w, int32_t c, void* stream);

/* In-place row softmax of bf16 scores (fp32 arithmetic): x[r, :cols] <- softmax(x[r, :cols]); the single-head, 512-wide
 * attention of the VAE mid block runs as GEMM (scaled q k^T) -> this -> GEMM (p v). */
int ug_softmax_rows_bf16(void* x, int64_t row_stride, int32_t rows, int32_t cols, void* stream);

/* NHWC bf16 (pixel stride >= c) -> NCHW (bf16, or fp32 when y_is_f32): the first c channels of every pixel. */
int ug_nhwc_to_nchw(const void* x, int64_t pixel_stride, void* y, int32_t y_is_f32, int32_t batch, int32_t c, int32_t h, int32_t w,
                    void* stream);

/* DiagonalGaussianDistribution over the encoder's moments (NHWC bf16 [batch, pixels, 2 * c]: mean | logvar):
 * z = mean + exp(0.5 * clamp(logvar, -30, 20)) * noise  (noise fp32 NCHW [batch, c, pixels]; NULL = `.mode()`), then
 * latents = (z - shift) * scale — NCHW bf16 [batch, c, pixels]. */
int ug_vae_sample(const void* moments, int64_t pixel_stride, const float* noise, void* latents, int32_t batch, int32_t c,
                  int32_t pixels, float shift, float scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* UNIGEN_B200_H_ */
