"""Host-side operator layer: torch tensors in, C-ABI calls out (include/unigen_b200.h).  torch is used for device
memory and streams only; every arithmetic op below runs in libunigen_b200.so on the current CUDA stream.
There is no fallback: a CPU tensor or a missing library raises."""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional, Sequence

import torch

from . import _lib
from ._lib import UG_ACT_GELU_TANH, UG_ACT_NONE, AttnArgs, GemmArgs, GemmFp8Scales, QkvScatterArgs, UgError, check

__all__ = ["gemm", "gemm_fp8", "quant_rows_fp8", "ln_modulate_fp8", "lora_down", "lora_down_wide", "attention", "attention_peer", "qkv_scatter", "peer_bcast_rows", "peer_barrier", "expand_segment_mask", "ln_modulate", "qk_rmsnorm_rope", "rope_table", "gemv", "GemvPlan", "gemv_grouped", "silu",
           "timestep_embedding", "add", "copy", "to_bf16", "to_f32", "moe_route", "moe_gather_modulate",
           "moe_combine", "ln_modulate_segs", "ln_modulate_segs_fp8", "ln_modulate_slots", "gated_add_slots", "unpatchify", "euler_step", "euler_step_table", "cfg_combine", "pack_latents", "unpack_latents", "conv3x3", "conv3x3_implicit_ok", "im2col", "groupnorm", "upsample2x", "softmax_rows_", "nhwc_to_nchw", "vae_sample", "launch_count", "reset_launch_count", "UG_ACT_NONE", "UG_ACT_GELU_TANH", "UgError"]

BF16 = torch.bfloat16
FP8 = torch.float8_e4m3fn


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dev(t: torch.Tensor, name: str, dtype=None) -> torch.Tensor:
    if not t.is_cuda:
        raise UgError(f"{name}: expected a CUDA tensor — the UniGen hot path has no CPU fallback")
    if dtype is not None and t.dtype != dtype:
        raise UgError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    return t


def _view3(t: torch.Tensor, name: str) -> torch.Tensor:
    """[R, C] -> [1, R, C]; requires a unit inner stride."""
    if t.dim() == 2:
        t = t.unsqueeze(0)
    if t.dim() != 3 or t.stride(2) != 1:
        raise UgError(f"{name}: expected a [batch, rows, cols] view with contiguous cols, got shape {tuple(t.shape)} "
                      f"strides {t.stride()}")
    return t


def launch_count() -> int:
    return int(_lib.load().ug_launch_count()) + _extra_launches


def reset_launch_count() -> None:
    global _extra_launches
    _extra_launches = 0
    _lib.load().ug_reset_launch_count()


_extra_launches = 0
_last_forward_launches = 0


def note_capture_launches(n: int) -> None:
    """Kernels issued by the last forward (so a CUDA-graph replay can account for the launches it re-issues)."""
    global _last_forward_launches
    _last_forward_launches = int(n)


def launch_count_in_last_capture() -> int:
    return _last_forward_launches


def add_launches(n: int) -> None:
    """Graph replays launch the captured kernels without passing through the C ABI: keep the counter truthful."""
    global _extra_launches
    _extra_launches += int(n)


def device_check() -> None:
    check(_lib.load().ug_device_check(), "ug_device_check")


# ------------------------------------------------------------------------------------------------------------------
def gemm(a: torch.Tensor, w: torch.Tensor, out: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None,
         gate: Optional[torch.Tensor] = None, alpha: float = 1.0, act: int = UG_ACT_NONE,
         residual: Optional[torch.Tensor] = None, variant: int = 0, lora: Optional[dict] = None,
         qk_norm: Optional[dict] = None, gate_seg_stride: int = 0, seg_bounds: Optional[Sequence[int]] = None,
         a2: Optional[torch.Tensor] = None, w2: Optional[torch.Tensor] = None, colmask: Optional[dict] = None) -> torch.Tensor:
    """out[b,r,:] = residual + alpha * gate[b,:] * act(a[b,r,:] @ w^T + bias (+ switched LoRA update)).
    a: [B,R,K] view, w: [N,K] or [B,N,K]. lora = dict(t=fp32 [B,R,n_blocks*rank] from lora_down, b=bf16 [groups,N,rank]
    (pre-scaled), rank, block_n, seg_bounds, seg_group) applies adapter group seg_group[i] to rows of segment i."""
    g, out = _gemm_args("gemm", BF16, a, w, out, bias, gate, alpha, act, residual, variant, lora, qk_norm, gate_seg_stride,
                        seg_bounds, a2, w2, colmask)
    check(_lib.load().ug_gemm_bf16(C.byref(g), _stream()), "ug_gemm_bf16")
    return out


def gemm_fp8(a: torch.Tensor, a_scale: Optional[torch.Tensor], w: torch.Tensor, w_scale: torch.Tensor, out: Optional[torch.Tensor] = None,
             bias: Optional[torch.Tensor] = None, gate: Optional[torch.Tensor] = None, alpha: float = 1.0, act: int = UG_ACT_NONE,
             residual: Optional[torch.Tensor] = None, variant: int = 0, qk_norm: Optional[dict] = None, gate_seg_stride: int = 0,
             seg_bounds: Optional[Sequence[int]] = None, a2: Optional[torch.Tensor] = None, w2: Optional[torch.Tensor] = None,
             colmask: Optional[dict] = None) -> torch.Tensor:
    """Row-wise fp8 GEMM: out = residual + alpha * gate * act((a @ w^T) * a_scale[b, r] * w_scale[c] + bias) (or the fused
    QK-norm epilogue), bf16 out. a: e4m3 [B,R,K] view with a_scale fp32 [B,R] (or [R]); w: e4m3 [N,K] with w_scale fp32 [N].
    With a bf16 K extension a2 [B,R,K2] / w2 [N,K2] or a column mask (as in `gemm`) it runs ug_gemm_fp8_lora: the accumulator
    a @ w^T + a2 @ w2^T is dequantised as a whole, so a2 / w2 carry the low-rank update pre-divided by a_scale / w_scale; there
    a_scale=None means unit row scales (the masked down-projection of a quantised operand)."""
    g, out = _gemm_args("gemm_fp8", FP8, a, w, out, bias, gate, alpha, act, residual, variant, None, qk_norm, gate_seg_stride,
                        seg_bounds, a2, w2, colmask)
    lora = a2 is not None or colmask is not None
    B, R = g.batch, g.rows
    _dev(w_scale, "gemm_fp8.w_scale", torch.float32)
    sc = GemmFp8Scales()
    if a_scale is None and not lora:
        raise UgError("gemm_fp8: a_scale is required (None = unit row scales only with a2 / w2 or colmask)")
    if a_scale is not None:
        _dev(a_scale, "gemm_fp8.a_scale", torch.float32)
        s3 = a_scale if a_scale.dim() == 2 else a_scale.unsqueeze(0)
        if tuple(s3.shape) != (B, R) or s3.stride(1) != 1:
            raise UgError(f"gemm_fp8: a_scale must be an fp32 [{B}, {R}] view with unit row stride, got {tuple(a_scale.shape)}")
        sc.a_scale, sc.a_scale_batch_stride = s3.data_ptr(), s3.stride(0)
    if w.dim() != 2 or tuple(w_scale.shape) != (g.n,) or not w_scale.is_contiguous():
        raise UgError(f"gemm_fp8: w must be [N, K] with a contiguous fp32 w_scale [N] (got w {tuple(w.shape)}, w_scale {tuple(w_scale.shape)})")
    sc.w_scale, sc.w_scale_batch_stride = w_scale.data_ptr(), 0
    if lora:
        check(_lib.load().ug_gemm_fp8_lora(C.byref(g), C.byref(sc), _stream()), "ug_gemm_fp8_lora")
    else:
        check(_lib.load().ug_gemm_fp8(C.byref(g), C.byref(sc), _stream()), "ug_gemm_fp8")
    return out


def _gemm_args(name, in_dtype, a, w, out, bias, gate, alpha, act, residual, variant, lora, qk_norm, gate_seg_stride=0,
               seg_bounds=None, a2=None, w2=None, colmask=None):
    """ug_gemm_args of one launch (shared by gemm and gemm_fp8; the operands a / w are `in_dtype`)."""
    a = _view3(_dev(a, f"{name}.a", in_dtype), f"{name}.a")
    _dev(w, f"{name}.w", in_dtype)
    B, R, K = a.shape
    N = w.shape[-2]
    if w.shape[-1] != K:
        raise UgError(f"gemm: K mismatch a {tuple(a.shape)} w {tuple(w.shape)}")
    if out is None:
        out = torch.empty(B, R, N, device=a.device, dtype=BF16)
    o3 = _view3(_dev(out, "gemm.out", BF16), "gemm.out")
    g = GemmArgs()
    g.a, g.a_row_stride, g.a_batch_stride = a.data_ptr(), a.stride(1), a.stride(0)
    g.w, g.w_row_stride = w.data_ptr(), w.stride(-2)
    g.w_batch_stride = w.stride(0) if w.dim() == 3 else 0
    g.c, g.c_row_stride, g.c_batch_stride = o3.data_ptr(), o3.stride(1), o3.stride(0)
    g.batch, g.rows, g.n, g.k = B, R, N, K
    if bias is not None:
        _dev(bias, "gemm.bias", BF16)
        g.bias = bias.data_ptr()
        g.bias_batch_stride = bias.stride(0) if bias.dim() == 2 else 0
    if gate is not None:
        _dev(gate, "gemm.gate", torch.float32)
        if gate.dim() == 1:
            gate = gate.unsqueeze(0)
        g.gate, g.gate_batch_stride = gate.data_ptr(), gate.stride(0)
    g.alpha, g.act = float(alpha), int(act)
    if gate_seg_stride:
        # per-segment gates: segment i of the row-segment table reads gate + i * gate_seg_stride
        g.gate_seg_stride = int(gate_seg_stride)
        sb = seg_bounds if seg_bounds is not None else (lora["seg_bounds"] if lora is not None else None)
        if gate is None or sb is None:
            raise UgError("gemm: gate_seg_stride needs gate and seg_bounds (or a lora segment table)")
        g.lora_nseg = len(sb) - 1
        for i, v in enumerate(sb):
            g.lora_seg_bounds[i] = int(v)
    if residual is not None:
        r3 = _view3(_dev(residual, "gemm.residual", BF16), "gemm.residual")
        g.residual, g.res_row_stride, g.res_batch_stride = r3.data_ptr(), r3.stride(1), r3.stride(0)
    g.variant = variant
    if lora is not None:
        t, lb = lora["t"], lora["b"]
        _dev(t, "gemm.lora_t", torch.float32), _dev(lb, "gemm.lora_b", BF16)
        t3 = t if t.dim() == 3 else t.unsqueeze(0)
        if not lb.is_contiguous() or t3.stride(2) != 1:
            raise UgError("gemm: lora_b must be contiguous [groups, N, rank]; lora_t needs a unit inner stride")
        g.lora_t, g.lora_t_row_stride, g.lora_t_batch_stride = t3.data_ptr(), t3.stride(1), t3.stride(0)
        g.lora_b, g.lora_rank, g.lora_block_n = lb.data_ptr(), int(lora["rank"]), int(lora.get("block_n", 0))
        sb, sg = lora["seg_bounds"], lora["seg_group"]
        g.lora_nseg = len(sg)
        for i, v in enumerate(sb):
            g.lora_seg_bounds[i] = int(v)
        for i, v in enumerate(sg):
            g.lora_seg_group[i] = int(v)
    if colmask is not None:
        # grouped projection: row r keeps only column block seg_group[segment(r)] (dict(block, seg_bounds, seg_group))
        g.colmask_block = int(colmask["block"])
        sb, sg = colmask["seg_bounds"], colmask["seg_group"]
        g.lora_nseg = len(sg)
        for i, v in enumerate(sb):
            g.lora_seg_bounds[i] = int(v)
        for i, v in enumerate(sg):
            g.lora_seg_group[i] = int(v)
    if a2 is not None:
        # second operand pair: accumulator = a @ w^T + a2 @ w2^T (K extension on the tensor cores)
        a23 = _view3(_dev(a2, "gemm.a2", BF16), "gemm.a2")
        _dev(w2, "gemm.w2", BF16)
        if a23.shape[:2] != (B, R) or w2.dim() != 2 or w2.shape[0] != N or w2.shape[1] != a23.shape[2] or w2.stride(1) != 1:
            raise UgError(f"gemm: a2 {tuple(a23.shape)} / w2 {tuple(w2.shape)} do not match a {tuple(a.shape)} / n {N}")
        g.a2, g.a2_row_stride, g.a2_batch_stride = a23.data_ptr(), a23.stride(1), a23.stride(0)
        g.w2, g.w2_row_stride, g.k2 = w2.data_ptr(), w2.stride(0), a23.shape[2]
    if qk_norm is not None:
        # fused per-head RMSNorm + RoPE epilogue of a q|k|v projection: dict(weight=[2,dh] bf16, head_dim, d, cos_sin, eps)
        wq = _dev(qk_norm["weight"], "gemm.qk_norm.weight", BF16)
        g.qk_norm_weight, g.qk_head_dim, g.qk_d = wq.data_ptr(), int(qk_norm["head_dim"]), int(qk_norm["d"])
        g.qk_eps = float(qk_norm.get("eps", 1e-6))
        cs = qk_norm.get("cos_sin")
        if cs is not None:
            _dev(cs, "gemm.qk_norm.cos_sin", torch.float32)
            if cs.shape[0] < R or not cs.is_contiguous():
                raise UgError("gemm: qk_norm cos_sin table too short / not contiguous")
            g.qk_cos_sin = cs.data_ptr()
    return g, out


def lora_down(x: torch.Tensor, a_stack: torch.Tensor, seg_bounds: Sequence[int], seg_group: Sequence[int],
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """t[b,r,:] = x[b,r,:] @ a_stack[g(r)]^T (fp32). a_stack: bf16 [groups, rank_total, K]; rows of a segment whose group
    is -1 get zeros (peft lora_A of the adapters `enable_lora` leaves active on that segment)."""
    x3 = _view3(_dev(x, "lora_down.x", BF16), "lora_down.x")
    _dev(a_stack, "lora_down.a", BF16)
    B, R, K = x3.shape
    G, RT, K2 = a_stack.shape
    if K2 != K or not a_stack.is_contiguous():
        raise UgError("lora_down: a_stack must be contiguous [groups, rank_total, K]")
    if out is None:
        out = torch.empty(B, R, RT, device=x.device, dtype=torch.float32)
    n = len(seg_group)
    sb = (C.c_int32 * (n + 1))(*[int(v) for v in seg_bounds])
    sg = (C.c_int32 * n)(*[int(v) for v in seg_group])
    check(_lib.load().ug_lora_down(x3.data_ptr(), x3.stride(1), x3.stride(0), a_stack.data_ptr(), out.data_ptr(),
                                   out.stride(1), out.stride(0), B, R, K, RT, n, sb, sg, _stream()), "ug_lora_down")
    return out


def _attn_args(q, k, v, heads, head_dim, seg_bounds, seg_visible, scale, variant):
    q, k, v = (_view3(_dev(t, n, BF16), n) for t, n in ((q, "attn.q"), (k, "attn.k"), (v, "attn.v")))
    B, S, HD = q.shape
    if HD != heads * head_dim:
        raise UgError(f"attention: inner dim {HD} != heads {heads} x head_dim {head_dim}")
    a = AttnArgs()
    a.q, a.k, a.v = q.data_ptr(), k.data_ptr(), v.data_ptr()
    a.q_row_stride, a.q_batch_stride = q.stride(1), q.stride(0)
    a.k_row_stride, a.k_batch_stride = k.stride(1), k.stride(0)
    a.v_row_stride, a.v_batch_stride = v.stride(1), v.stride(0)
    a.batch, a.heads, a.seq, a.head_dim = B, heads, S, head_dim
    a.scale = float(scale if scale is not None else 1.0 / math.sqrt(head_dim))
    keep = None
    if seg_bounds is not None:
        n = len(seg_bounds) - 1
        sb = (C.c_int32 * (n + 1))(*seg_bounds)
        sv = (C.c_uint32 * n)(*seg_visible)
        keep = (sb, sv)
        a.n_seg, a.seg_bounds, a.seg_visible = n, sb, sv
    a.variant = variant
    return a, keep


def lora_down_wide(x: torch.Tensor, a_stack: torch.Tensor, seg_bounds: Sequence[int], seg_group: Sequence[int],
                   out: torch.Tensor, block: int = 64) -> torch.Tensor:
    """bf16 out[b, r, g(r)*block : g(r)*block + rank_total] = x[b,r,:] @ a_stack[g(r)]^T, zeros elsewhere
    (out: [B, rows, groups*block]) — the A2 operand of gemm(..., a2=out, w2=[B_0 | B_1 | ...])."""
    x3 = _view3(_dev(x, "lora_down_wide.x", BF16), "lora_down_wide.x")
    o3 = _view3(_dev(out, "lora_down_wide.out", BF16), "lora_down_wide.out")
    _dev(a_stack, "lora_down_wide.a", BF16)
    B, R, K = x3.shape
    G, RT, K2 = a_stack.shape
    if K2 != K or not a_stack.is_contiguous() or o3.shape[2] != G * block or o3.shape[1] != R:
        raise UgError("lora_down_wide: a_stack must be contiguous [groups, rank_total, K] and out [B, rows, groups*block]")
    n = len(seg_group)
    sb = (C.c_int32 * (n + 1))(*[int(v) for v in seg_bounds])
    sg = (C.c_int32 * n)(*[int(v) for v in seg_group])
    check(_lib.load().ug_lora_down_wide(x3.data_ptr(), x3.stride(1), x3.stride(0), a_stack.data_ptr(), o3.data_ptr(), o3.stride(1),
                                        o3.stride(0), B, R, K, RT, G, block, n, sb, sg, _stream()), "ug_lora_down_wide")
    return out


def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, out: torch.Tensor, heads: int, head_dim: int,
              seg_bounds: Optional[Sequence[int]] = None, seg_visible: Optional[Sequence[int]] = None,
              scale: Optional[float] = None, variant: int = 0) -> torch.Tensor:
    """q/k/v/out: [B, S, heads*head_dim] views (any row / batch stride, contiguous inner dim)."""
    a, keep = _attn_args(q, k, v, heads, head_dim, seg_bounds, seg_visible, scale, variant)
    o = _view3(_dev(out, "attn.out", BF16), "attn.out")
    a.o, a.o_row_stride, a.o_batch_stride = o.data_ptr(), o.stride(1), o.stride(0)
    check(_lib.load().ug_attention_bf16(C.byref(a), _stream()), "ug_attention_bf16")
    del keep
    return out


def attention_peer(table, q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, heads: int, head_dim: int, o_offset: int,
                   o_row_stride: int, rows_per_rank: int, seg_bounds: Optional[Sequence[int]] = None,
                   seg_visible: Optional[Sequence[int]] = None, scale: Optional[float] = None, variant: int = 0) -> None:
    """Attention over this rank's head shard of ALL tokens ([1, S, heads*head_dim] views); output row q lands in rank
    q // rows_per_rank's pool at byte o_offset, row q % rows_per_rank (row stride o_row_stride elements), this rank's columns.
    rows_per_rank = 0: segment-sharded rows (every segment of seg_bounds split evenly over the ranks)."""
    a, keep = _attn_args(q, k, v, heads, head_dim, seg_bounds, seg_visible, scale, variant)
    a.o, a.o_row_stride, a.o_batch_stride = 0, int(o_row_stride), 0
    check(_lib.load().ug_attention_bf16_peer(C.byref(a), C.byref(table), int(o_offset), int(rows_per_rank), _stream()),
          "ug_attention_bf16_peer")
    del keep


def qkv_scatter(table, qkv_rows: torch.Tensor, heads: int, head_dim: int, norm_weight: Optional[torch.Tensor],
                cos_sin: Optional[torch.Tensor], dst_offset: int, seq_total: int, dst_row0: int, eps: float = 1e-6) -> None:
    """qkv_rows: local [rows, 3*heads*head_dim] bf16 view of the fused projection -> every head's owner rank (see header)."""
    _dev(qkv_rows, "qkv_scatter.qkv", BF16)
    if qkv_rows.dim() != 2 or qkv_rows.stride(1) != 1 or qkv_rows.shape[1] != 3 * heads * head_dim:
        raise UgError(f"qkv_scatter: expected a [rows, {3 * heads * head_dim}] view, got {tuple(qkv_rows.shape)}")
    a = QkvScatterArgs()
    a.qkv, a.row_stride, a.rows, a.heads, a.head_dim, a.eps = qkv_rows.data_ptr(), qkv_rows.stride(0), qkv_rows.shape[0], heads, head_dim, eps
    if norm_weight is not None:
        a.norm_weight = _dev(norm_weight, "qkv_scatter.norm_weight", BF16).data_ptr()
    if cos_sin is not None:
        _dev(cos_sin, "qkv_scatter.cos_sin", torch.float32)
        if cos_sin.shape[0] < qkv_rows.shape[0] or not cos_sin.is_contiguous():
            raise UgError("qkv_scatter: cos_sin table too short / not contiguous")
        a.cos_sin = cos_sin.data_ptr()
    a.dst_offset, a.seq_total, a.dst_row0 = int(dst_offset), int(seq_total), int(dst_row0)
    check(_lib.load().ug_qkv_scatter(C.byref(table), C.byref(a), _stream()), "ug_qkv_scatter")


def peer_bcast_rows(table, src: torch.Tensor, dst_offset: int, dst_row_stride: int, dst_row0: int) -> None:
    """src: [rows, d] bf16 view -> rows [dst_row0, dst_row0 + rows) of the buffer at byte dst_offset of EVERY rank's pool."""
    _dev(src, "peer_bcast.src", BF16)
    if src.dim() != 2 or src.stride(1) != 1:
        raise UgError("peer_bcast_rows: expected a [rows, d] view with contiguous columns")
    check(_lib.load().ug_peer_bcast_rows(C.byref(table), src.data_ptr(), src.stride(0), src.shape[0], src.shape[1], int(dst_offset),
                                         int(dst_row_stride), int(dst_row0), _stream()), "ug_peer_bcast_rows")


def peer_barrier(table) -> None:
    check(_lib.load().ug_peer_barrier(C.byref(table), _stream()), "ug_peer_barrier")


def expand_segment_mask(seq: int, seg_bounds: Sequence[int], seg_visible: Sequence[int], device) -> torch.Tensor:
    n = len(seg_visible)
    m = torch.empty(seq, seq, dtype=torch.uint8, device=device)
    sb = (C.c_int32 * (n + 1))(*seg_bounds)
    sv = (C.c_uint32 * n)(*seg_visible)
    check(_lib.load().ug_expand_segment_mask(seq, n, sb, sv, m.data_ptr(), _stream()), "ug_expand_segment_mask")
    return m.bool()


def ln_modulate(x: torch.Tensor, out: torch.Tensor, shift: torch.Tensor, scale: torch.Tensor, eps: float = 1e-6) -> torch.Tensor:
    """out = LayerNorm(x) * (1 + scale[b]) + shift[b]; shift/scale: fp32 [B, D] views (same batch stride)."""
    x3, o3 = _view3(_dev(x, "ln.x", BF16), "ln.x"), _view3(_dev(out, "ln.out", BF16), "ln.out")
    _dev(shift, "ln.shift", torch.float32), _dev(scale, "ln.scale", torch.float32)
    B, R, D = x3.shape
    if shift.stride(0) != scale.stride(0) and B > 1:
        raise UgError("ln_modulate: shift and scale need the same batch stride")
    check(_lib.load().ug_ln_modulate(x3.data_ptr(), x3.stride(1), x3.stride(0), o3.data_ptr(), o3.stride(1), o3.stride(0),
                                     shift.data_ptr(), scale.data_ptr(), shift.stride(0), B, R, D, float(eps), _stream()),
          "ug_ln_modulate")
    return out


def quant_rows_fp8(x: torch.Tensor, out: Optional[torch.Tensor] = None, scale: Optional[torch.Tensor] = None):
    """Dynamic row-wise e4m3 quantisation of a bf16 [B, R, K] (or [R, K]) view -> (out e4m3 [B, R, K], scale fp32 [B, R]):
    scale = amax / 448 (1 for an all-zero row), out = satfinite_e4m3(x * 448 / amax). out / scale may be views (unit inner
    strides) into larger buffers; they are allocated contiguous otherwise."""
    x3 = _view3(_dev(x, "quant_rows_fp8.x", BF16), "quant_rows_fp8.x")
    B, R, K = x3.shape
    if out is None:
        out = torch.empty(x.shape, device=x.device, dtype=FP8)
    if scale is None:
        scale = torch.empty(x.shape[:-1], device=x.device, dtype=torch.float32)
    q3 = _view3(_dev(out, "quant_rows_fp8.out", FP8), "quant_rows_fp8.out")
    s3 = _dev(scale, "quant_rows_fp8.scale", torch.float32)
    s3 = s3 if s3.dim() == 2 else s3.unsqueeze(0)
    if tuple(q3.shape) != (B, R, K) or tuple(s3.shape) != (B, R) or s3.stride(1) != 1:
        raise UgError(f"quant_rows_fp8: out {tuple(out.shape)} / scale {tuple(scale.shape)} do not match x {tuple(x.shape)}")
    check(_lib.load().ug_quant_rows_fp8(x3.data_ptr(), x3.stride(1), x3.stride(0), q3.data_ptr(), q3.stride(1), q3.stride(0),
                                        s3.data_ptr(), s3.stride(0), B, R, K, _stream()), "ug_quant_rows_fp8")
    return out, scale


def ln_modulate_fp8(x: torch.Tensor, out: torch.Tensor, out_scale: torch.Tensor, shift: torch.Tensor, scale: torch.Tensor,
                    eps: float = 1e-6):
    """quant_rows_fp8(ln_modulate(x, shift, scale)) in one pass, bit for bit: out e4m3 [B, R, D] view, out_scale fp32 [B, R]."""
    x3, q3 = _view3(_dev(x, "ln_fp8.x", BF16), "ln_fp8.x"), _view3(_dev(out, "ln_fp8.out", FP8), "ln_fp8.out")
    _dev(shift, "ln_fp8.shift", torch.float32), _dev(scale, "ln_fp8.scale", torch.float32), _dev(out_scale, "ln_fp8.out_scale", torch.float32)
    B, R, D = x3.shape
    s3 = out_scale if out_scale.dim() == 2 else out_scale.unsqueeze(0)
    if tuple(q3.shape) != (B, R, D) or tuple(s3.shape) != (B, R) or s3.stride(1) != 1:
        raise UgError(f"ln_modulate_fp8: out {tuple(out.shape)} / out_scale {tuple(out_scale.shape)} do not match x {tuple(x.shape)}")
    if shift.stride(0) != scale.stride(0) and B > 1:
        raise UgError("ln_modulate_fp8: shift and scale need the same batch stride")
    check(_lib.load().ug_ln_modulate_fp8(x3.data_ptr(), x3.stride(1), x3.stride(0), q3.data_ptr(), q3.stride(1), q3.stride(0),
                                         s3.data_ptr(), s3.stride(0), shift.data_ptr(), scale.data_ptr(), shift.stride(0), B, R, D,
                                         float(eps), _stream()), "ug_ln_modulate_fp8")
    return out, out_scale


def ln_modulate_segs(x: torch.Tensor, out: torch.Tensor, shift: torch.Tensor, scale: torch.Tensor, seg_bounds: Sequence[int],
                     mod_seg_stride: int, eps: float = 1e-6) -> torch.Tensor:
    """ln_modulate with per-row-segment vectors: segment i uses shift/scale + i * mod_seg_stride (fp32 [B, D] views of row 0)."""
    x3, o3 = _view3(_dev(x, "ln.x", BF16), "ln.x"), _view3(_dev(out, "ln.out", BF16), "ln.out")
    _dev(shift, "ln.shift", torch.float32), _dev(scale, "ln.scale", torch.float32)
    B, R, D = x3.shape
    n = len(seg_bounds) - 1
    sb = (C.c_int32 * (n + 1))(*[int(v) for v in seg_bounds])
    check(_lib.load().ug_ln_modulate_segs(x3.data_ptr(), x3.stride(1), x3.stride(0), o3.data_ptr(), o3.stride(1), o3.stride(0),
                                          shift.data_ptr(), scale.data_ptr(), shift.stride(0), int(mod_seg_stride), n, sb, B, R, D,
                                          float(eps), _stream()), "ug_ln_modulate_segs")
    return out


def ln_modulate_segs_fp8(x: torch.Tensor, out: torch.Tensor, out_scale: torch.Tensor, shift: torch.Tensor, scale: torch.Tensor,
                         seg_bounds: Sequence[int], mod_seg_stride: int, eps: float = 1e-6):
    """quant_rows_fp8(ln_modulate_segs(x, ...)) in one pass, bit for bit: out e4m3 [B, R, D] view, out_scale fp32 [B, R]."""
    x3, q3 = _view3(_dev(x, "ln_segs_fp8.x", BF16), "ln_segs_fp8.x"), _view3(_dev(out, "ln_segs_fp8.out", FP8), "ln_segs_fp8.out")
    _dev(shift, "ln_segs_fp8.shift", torch.float32), _dev(scale, "ln_segs_fp8.scale", torch.float32)
    _dev(out_scale, "ln_segs_fp8.out_scale", torch.float32)
    B, R, D = x3.shape
    s3 = out_scale if out_scale.dim() == 2 else out_scale.unsqueeze(0)
    if tuple(q3.shape) != (B, R, D) or tuple(s3.shape) != (B, R) or s3.stride(1) != 1:
        raise UgError(f"ln_modulate_segs_fp8: out {tuple(out.shape)} / out_scale {tuple(out_scale.shape)} do not match x {tuple(x.shape)}")
    n = len(seg_bounds) - 1
    sb = (C.c_int32 * (n + 1))(*[int(v) for v in seg_bounds])
    check(_lib.load().ug_ln_modulate_segs_fp8(x3.data_ptr(), x3.stride(1), x3.stride(0), q3.data_ptr(), q3.stride(1), q3.stride(0),
                                              s3.data_ptr(), s3.stride(0), shift.data_ptr(), scale.data_ptr(), shift.stride(0),
                                              int(mod_seg_stride), n, sb, B, R, D, float(eps), _stream()), "ug_ln_modulate_segs_fp8")
    return out, out_scale


def _slot_mod(t: torch.Tensor, name: str):
    """fp32 [E, n_index, D] view of per-expert AdaLN rows -> (ptr, expert stride, index stride)."""
    _dev(t, name, torch.float32)
    if t.dim() != 3 or t.stride(2) != 1:
        raise UgError(f"{name}: expected an fp32 [experts, index, d] view with contiguous d")
    return t.data_ptr(), t.stride(0), t.stride(1)


def ln_modulate_slots(x: torch.Tensor, out: torch.Tensor, shift: torch.Tensor, scale: torch.Tensor, slot_token: torch.Tensor,
                      experts: int, capacity: int, tokens_per_batch: int, empty_index: int, eps: float = 1e-6) -> torch.Tensor:
    """Per-token AdaLN on [experts*capacity, D] slot buffers; shift/scale: fp32 [experts, samples+1, D] views
    (row `empty_index` = the AdaLN vector of an all-zero temb, used by empty slots)."""
    _dev(x, "ln_slots.x", BF16), _dev(out, "ln_slots.out", BF16), _dev(slot_token, "ln_slots.slot_token", torch.int32)
    D = x.shape[-1]
    sp, ses, sis = _slot_mod(shift, "ln_slots.shift")
    cp, ces, cis = _slot_mod(scale, "ln_slots.scale")
    if (ses, sis) != (ces, cis) or x.shape[0] != experts * capacity or slot_token.numel() != experts * capacity:
        raise UgError("ln_modulate_slots: shift / scale strides differ or the slot buffer has the wrong row count")
    check(_lib.load().ug_ln_modulate_slots(x.data_ptr(), x.stride(0), out.data_ptr(), out.stride(0), sp, cp, ses, sis,
                                           slot_token.data_ptr(), experts, capacity, tokens_per_batch, empty_index, D,
                                           float(eps), _stream()), "ug_ln_modulate_slots")
    return out


def gated_add_slots(x: torch.Tensor, y: torch.Tensor, gate: torch.Tensor, slot_token: torch.Tensor, experts: int,
                    capacity: int, tokens_per_batch: int, empty_index: int) -> torch.Tensor:
    """In place: x[r] += gate[e(r), idx(r)] * y[r] on [experts*capacity, D] slot buffers."""
    _dev(x, "gated_add.x", BF16), _dev(y, "gated_add.y", BF16), _dev(slot_token, "gated_add.slot_token", torch.int32)
    gp, ges, gis = _slot_mod(gate, "gated_add.gate")
    if x.shape != y.shape or x.shape[0] != experts * capacity:
        raise UgError("gated_add_slots: x / y shape mismatch")
    check(_lib.load().ug_gated_add_slots(x.data_ptr(), x.stride(0), y.data_ptr(), y.stride(0), gp, ges, gis,
                                         slot_token.data_ptr(), experts, capacity, tokens_per_batch, empty_index,
                                         x.shape[-1], _stream()), "ug_gated_add_slots")
    return x


def qk_rmsnorm_rope(x: torch.Tensor, heads: int, head_dim: int, weight: torch.Tensor,
                    cos_sin: Optional[torch.Tensor] = None, eps: float = 1e-6, heads_per_weight: int = 0) -> torch.Tensor:
    """In-place RMSNorm(weight)+RoPE on a [B, rows, heads*head_dim] view. cos_sin: fp32 [rows, head_dim] table.
    weight: bf16 [heads/heads_per_weight, head_dim] (e.g. [norm_q; norm_k] for the Q|K halves of a fused QKV row)."""
    x3 = _view3(_dev(x, "rms.x", BF16), "rms.x")
    _dev(weight, "rms.weight", BF16)
    B, R, HD = x3.shape
    if HD != heads * head_dim:
        raise UgError("qk_rmsnorm_rope: inner dim mismatch")
    cs = 0
    if cos_sin is not None:
        _dev(cos_sin, "rms.cos_sin", torch.float32)
        if cos_sin.shape[0] < R or not cos_sin.is_contiguous():
            raise UgError("qk_rmsnorm_rope: cos_sin table too short / not contiguous")
        cs = cos_sin.data_ptr()
    check(_lib.load().ug_qk_rmsnorm_rope(x3.data_ptr(), x3.stride(1), x3.stride(0), B, R, heads, head_dim,
                                         weight.data_ptr(), int(heads_per_weight), float(eps), cs, _stream()), "ug_qk_rmsnorm_rope")
    return x


def rope_table(ids: torch.Tensor, axes_dim: Sequence[int], theta: float = 10000.0,
               out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """FluxPosEmbed: ids fp32 [rows, 3] -> fp32 [rows, head_dim] table laid out (cos_i, sin_i) per rotation pair."""
    ids = _dev(ids, "rope.ids").to(torch.float32).contiguous()
    rows, hd = ids.shape[0], sum(axes_dim)
    if out is None:
        out = torch.empty(rows, hd, device=ids.device, dtype=torch.float32)
    ax = (C.c_int32 * 3)(*axes_dim)
    check(_lib.load().ug_rope_table(ids.data_ptr(), rows, ax, float(theta), out.data_ptr(), _stream()), "ug_rope_table")
    return out


def gemv(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], out: Optional[torch.Tensor] = None,
         silu_in: bool = False, silu_out: bool = False, accumulate: bool = False) -> torch.Tensor:
    """out[b,:] (+)= w @ f(x[b,:]) + bias; x/out fp32 [B, K] / [B, N]; w bf16 [N, K]."""
    _dev(x, "gemv.x", torch.float32), _dev(w, "gemv.w", BF16)
    B, K = x.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty(B, N, device=x.device, dtype=torch.float32)
    if not w.is_contiguous() or x.stride(1) != 1 or out.stride(1) != 1:
        raise UgError("gemv: w must be contiguous, x/out need unit inner stride")
    check(_lib.load().ug_gemv(x.data_ptr(), x.stride(0), w.data_ptr(), bias.data_ptr() if bias is not None else 0,
                              out.data_ptr(), out.stride(0), B, N, K, int(silu_in), int(silu_out), int(accumulate),
                              _stream()), "ug_gemv")
    return out


class GemvPlan:
    """Device-resident job table of `gemv_grouped` (ug_gemv_job[]): built once per workspace, launched every step.
    jobs: sequence of (w bf16 [n, k], bias bf16 [n] | None, x fp32 [B, k], out fp32 [B, n] view, silu_in[, accumulate]). With `pool` (a
    parallel.PeerPool) every `out` must be a view INTO that pool: its byte offset is stored instead of the pointer and the
    launch writes each result into every rank's pool."""

    def __init__(self, jobs, device, pool=None):
        if not 1 <= len(jobs) <= _lib.UG_MAX_GEMV_JOBS:
            raise UgError(f"gemv_grouped: 1..{_lib.UG_MAX_GEMV_JOBS} jobs per plan (got {len(jobs)})")
        self.more = None
        B_all = jobs[0][2].shape[0]
        if B_all > 8:  # the kernel holds <= 8 batch rows in registers per weight pass: further rows are a second plan
            self.more = GemvPlan([(j[0], j[1], j[2][8:], j[3][8:]) + tuple(j[4:]) for j in jobs], device, pool)
            jobs = [(j[0], j[1], j[2][:8], j[3][:8]) + tuple(j[4:]) for j in jobs]
        arr = (_lib.GemvJob * len(jobs))()
        self.keep, self.pool, g, self.batch = [], pool, 0, None
        for j, job in enumerate(jobs):
            w, bias, x, out, silu_in = job[:5]
            accumulate = bool(job[5]) if len(job) > 5 else False
            _dev(w, "gemv_grouped.w", BF16), _dev(x, "gemv_grouped.x", torch.float32), _dev(out, "gemv_grouped.out", torch.float32)
            n, k = w.shape
            B = x.shape[0]
            self.batch = B if self.batch is None else self.batch
            if B != self.batch or B > 8:
                raise UgError("gemv_grouped: every job needs the same batch (<= 8)")
            if not w.is_contiguous() or x.shape != (B, k) or out.shape != (B, n) or x.stride(1) != 1 or out.stride(1) != 1 or k % 8 or n % 8:
                raise UgError(f"gemv_grouped: job {j}: w [n,k] contiguous, x [B,k], out [B,n] with unit inner strides, n / k multiples of 8")
            if x.data_ptr() % 16 or (x.stride(0) * 4) % 16 or w.data_ptr() % 16:
                raise UgError(f"gemv_grouped: job {j}: x rows / w must be 16-byte aligned")
            a = arr[j]
            a.w, a.bias, a.x = w.data_ptr(), (_dev(bias, "gemv_grouped.bias", BF16).data_ptr() if bias is not None else None), x.data_ptr()
            if pool is not None:
                off = out.data_ptr() - pool.local.data_ptr()
                if off < 0 or off + ((B - 1) * out.stride(0) + n) * 4 > pool.nbytes:
                    raise UgError(f"gemv_grouped: job {j}: with a peer pool every output must be a view into the pool")
                a.out = off
            else:
                a.out = out.data_ptr()
            a.x_stride, a.out_stride, a.n, a.k, a.first_group, a.flags = x.stride(0), out.stride(0), n, k, g, int(bool(silu_in)) | (2 if accumulate else 0)
            g += (n + 3) // 4
            self.keep.append((w, bias, x, out))
        self.n_jobs, self.total_groups = len(jobs), g
        raw = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8)
        self.table = raw.to(device)
        self.weight_bytes = sum(k_[0].numel() * 2 for k_ in self.keep)


def gemv_grouped(plan: GemvPlan, rank: int = 0, world: int = 1) -> None:
    """One launch over `plan`; (rank, world) selects this rank's contiguous share of the 4-row groups (sequence parallelism:
    the plan was built with the peer pool, results land in every rank's pool — follow with a pool barrier)."""
    G = plan.total_groups
    lo, hi = (G * rank) // world, (G * (rank + 1)) // world
    peers = C.byref(plan.pool.table) if plan.pool is not None else None
    check(_lib.load().ug_gemv_grouped(plan.table.data_ptr(), plan.n_jobs, G, plan.batch, lo, hi, peers, _stream()), "ug_gemv_grouped")
    if plan.more is not None:
        gemv_grouped(plan.more, rank, world)


def silu(x: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """out = x * sigmoid(x) (fp32, contiguous, same numel)."""
    _dev(x, "silu.x", torch.float32), _dev(out, "silu.out", torch.float32)
    if not (x.is_contiguous() and out.is_contiguous()) or x.numel() != out.numel():
        raise UgError("silu: contiguous fp32 tensors of equal size required")
    check(_lib.load().ug_silu_f32(x.data_ptr(), out.data_ptr(), x.numel(), _stream()), "ug_silu_f32")
    return out


def timestep_embedding(t: torch.Tensor, dim: int = 256, scale: float = 1.0, batch: Optional[int] = None,
                       out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Timesteps(dim)(scale * t). t: fp32 [B]; or a ONE-element device view broadcast to `batch` samples (entry i of a
    device-resident sigma table: the whole-loop CUDA graph reads the step's timestep from memory)."""
    t = _dev(t, "timestep").to(torch.float32)
    if t.dim() != 1 or (t.shape[0] > 1 and t.stride(0) != 1):
        t = t.reshape(-1).contiguous()
    B = int(batch) if batch is not None else t.shape[0]
    if t.shape[0] not in (1, B):
        raise UgError(f"timestep_embedding: {t.shape[0]} timesteps for a batch of {B}")
    if out is None:
        out = torch.empty(B, dim, device=t.device, dtype=torch.float32)
    check(_lib.load().ug_timestep_embedding(t.data_ptr(), 0 if t.shape[0] == 1 else 1, B, dim, float(scale), out.data_ptr(),
                                            _stream()), "ug_timestep_embedding")
    return out


def add(a: torch.Tensor, b: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    a3, b3, o3 = (_view3(_dev(t, "add", BF16), "add") for t in (a, b, out))
    B, R, D = a3.shape
    check(_lib.load().ug_add_bf16(a3.data_ptr(), a3.stride(1), a3.stride(0), b3.data_ptr(), b3.stride(1), b3.stride(0),
                                  o3.data_ptr(), o3.stride(1), o3.stride(0), B, R, D, _stream()), "ug_add_bf16")
    return out


def copy(src: torch.Tensor, dst: torch.Tensor) -> torch.Tensor:
    s3, d3 = _view3(_dev(src, "copy", BF16), "copy"), _view3(_dev(dst, "copy", BF16), "copy")
    B, R, D = s3.shape
    check(_lib.load().ug_copy_bf16(s3.data_ptr(), s3.stride(1), s3.stride(0), d3.data_ptr(), d3.stride(1), d3.stride(0),
                                   B, R, D, _stream()), "ug_copy_bf16")
    return dst


def to_bf16(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _dev(x, "to_bf16")
    if x.dtype == BF16:
        return x
    x = x.to(torch.float32).contiguous() if x.dtype != torch.float32 or not x.is_contiguous() else x
    if out is None:
        out = torch.empty(x.shape, device=x.device, dtype=BF16)
    check(_lib.load().ug_cast_f32_to_bf16(x.data_ptr(), out.data_ptr(), x.numel(), _stream()), "ug_cast_f32_to_bf16")
    return out


def to_f32(x: torch.Tensor) -> torch.Tensor:
    _dev(x, "to_f32", BF16)
    x = x.contiguous()
    out = torch.empty(x.shape, device=x.device, dtype=torch.float32)
    check(_lib.load().ug_cast_bf16_to_f32(x.data_ptr(), out.data_ptr(), x.numel(), _stream()), "ug_cast_bf16_to_f32")
    return out


# ------------------------------------------------------------------------------------------------------------------
def moe_capacity(tokens: int, experts: int, capacity_factor: float = 1.0, min_capacity: int = 4) -> int:
    """DeepSpeed `_capacity` (SURVEY.md §A.5): max(ceil(tokens/experts * factor), min_capacity)."""
    return max(int(math.ceil(tokens / experts * capacity_factor)), min_capacity)


def moe_route(x: torch.Tensor, wg: torch.Tensor, rts_uniform: torch.Tensor, capacity: int):
    """x bf16 [tokens, D]; wg fp32 [E, D]; rts_uniform fp32 [tokens, E] ->
    dict(expert_idx, slot, prob, slot_token, exp_counts, l_aux)."""
    _dev(x, "route.x", BF16), _dev(wg, "route.wg", torch.float32), _dev(rts_uniform, "route.uniform", torch.float32)
    tokens, D = x.shape
    E = wg.shape[0]
    if not (x.is_contiguous() and wg.is_contiguous() and rts_uniform.is_contiguous()) or rts_uniform.shape != (tokens, E):
        raise UgError("moe_route: contiguous x [tokens,D], wg [E,D], uniform [tokens,E] required")
    dev = x.device
    r = dict(expert_idx=torch.empty(tokens, dtype=torch.int32, device=dev),
             slot=torch.empty(tokens, dtype=torch.int32, device=dev),
             prob=torch.empty(tokens, dtype=torch.float32, device=dev),
             slot_token=torch.empty(E * capacity, dtype=torch.int32, device=dev),
             exp_counts=torch.empty(E, dtype=torch.int64, device=dev),
             l_aux=torch.empty(1, dtype=torch.float32, device=dev))
    ws = torch.empty(tokens * E + E, dtype=torch.float32, device=dev)
    check(_lib.load().ug_moe_route(x.data_ptr(), wg.data_ptr(), rts_uniform.data_ptr(), tokens, D, E, capacity,
                                   r["expert_idx"].data_ptr(), r["slot"].data_ptr(), r["prob"].data_ptr(),
                                   r["slot_token"].data_ptr(), r["exp_counts"].data_ptr(), r["l_aux"].data_ptr(),
                                   ws.data_ptr(), _stream()), "ug_moe_route")
    r["gates"] = ws[: tokens * E].view(tokens, E)
    return r


def moe_gather_modulate(x: torch.Tensor, slot_token: torch.Tensor, mod: Optional[torch.Tensor], experts: int, capacity: int,
                        tokens_per_batch: int, addend: Optional[torch.Tensor] = None,
                        out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[e*C+s] = mod[b(token), e] * (x[token] (+ addend[e*C+s])); mod: fp32 [B, E, D] (batch-major, as one stacked GEMV
    writes it) or None for a plain dispatch gather."""
    _dev(x, "gather.x", BF16)
    if mod is not None:
        _dev(mod, "gather.mod", torch.float32)
    D = x.shape[-1]
    if out is None:
        out = torch.empty(experts * capacity, D, device=x.device, dtype=BF16)
    check(_lib.load().ug_moe_gather_modulate(x.data_ptr(), slot_token.data_ptr(), mod.data_ptr() if mod is not None else 0,
                                             mod.stride(1) if mod is not None else 0, mod.stride(0) if mod is not None else 0,
                                             addend.data_ptr() if addend is not None else 0, out.data_ptr(), experts,
                                             capacity, tokens_per_batch, D, _stream()), "ug_moe_gather_modulate")
    return out


def moe_combine(y: torch.Tensor, route: dict, capacity: int, out: torch.Tensor) -> torch.Tensor:
    tokens = route["slot"].shape[0]
    D = y.shape[-1]
    check(_lib.load().ug_moe_combine(y.data_ptr(), route["expert_idx"].data_ptr(), route["slot"].data_ptr(),
                                     route["prob"].data_ptr(), out.data_ptr(), tokens, capacity, D, _stream()), "ug_moe_combine")
    return out


# ------------------------------------------------------------------------------------------------------------------
def euler_step(latents: torch.Tensor, velocity: torch.Tensor, sigma: float, sigma_next: float) -> torch.Tensor:
    """In place: latents <- latents + (sigma_next - sigma) * velocity (bf16 storage, fp32 math)."""
    _dev(latents, "euler.latents", BF16), _dev(velocity, "euler.velocity", BF16)
    if not (latents.is_contiguous() and velocity.is_contiguous()) or latents.numel() != velocity.numel():
        raise UgError("euler_step: contiguous tensors of equal size required")
    check(_lib.load().ug_euler_step(latents.data_ptr(), velocity.data_ptr(), float(sigma), float(sigma_next), latents.numel(),
                                    _stream()), "ug_euler_step")
    return latents


def euler_step_table(latents: torch.Tensor, velocity: torch.Tensor, sigmas: torch.Tensor, step: int) -> torch.Tensor:
    """In place: latents <- latents + (sigmas[step + 1] - sigmas[step]) * velocity with the fp32 schedule read on the device."""
    _dev(latents, "euler.latents", BF16), _dev(velocity, "euler.velocity", BF16), _dev(sigmas, "euler.sigmas", torch.float32)
    if not (latents.is_contiguous() and velocity.is_contiguous() and sigmas.is_contiguous()) or latents.numel() != velocity.numel():
        raise UgError("euler_step_table: contiguous tensors of equal size required")
    if not 0 <= step < sigmas.numel() - 1:
        raise UgError(f"euler_step_table: step {step} outside the {sigmas.numel()}-entry schedule")
    check(_lib.load().ug_euler_step_table(latents.data_ptr(), velocity.data_ptr(), sigmas.data_ptr(), int(step), latents.numel(),
                                          _stream()), "ug_euler_step_table")
    return latents


def cfg_combine(uncond: torch.Tensor, text: torch.Tensor, guidance_scale: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _dev(uncond, "cfg.uncond", BF16), _dev(text, "cfg.text", BF16)
    if out is None:
        out = torch.empty_like(text)
    check(_lib.load().ug_cfg_combine(uncond.contiguous().data_ptr(), text.contiguous().data_ptr(), float(guidance_scale),
                                     out.data_ptr(), text.numel(), _stream()), "ug_cfg_combine")
    return out


def pack_latents(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(B, C, H, W) bf16 -> (B, (H/2)(W/2), 4C)."""
    _dev(x, "pack.x", BF16)
    B, Cc, H, W = x.shape
    if out is None:
        out = torch.empty(B, (H // 2) * (W // 2), Cc * 4, device=x.device, dtype=BF16)
    elif not out.is_contiguous() or out.numel() != x.numel():
        raise UgError("pack_latents: out must be a contiguous (B, (H/2)(W/2), 4C) buffer")
    check(_lib.load().ug_pack_latents(x.contiguous().data_ptr(), out.data_ptr(), B, Cc, H, W, 0, _stream()), "ug_pack_latents")
    return out


def unpack_latents(x: torch.Tensor, height: int, width: int) -> torch.Tensor:
    """(B, (H/2)(W/2), 4C) bf16 -> (B, C, H, W) with H, W the latent height / width."""
    _dev(x, "unpack.x", BF16)
    B, _, C4 = x.shape
    out = torch.empty(B, C4 // 4, height, width, device=x.device, dtype=BF16)
    check(_lib.load().ug_pack_latents(x.contiguous().data_ptr(), out.data_ptr(), B, C4 // 4, height, width, 1, _stream()), "ug_pack_latents")
    return out


def unpatchify(tokens: torch.Tensor, h: int, w: int, p: int, channels: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(B, h*w, p*p*C) bf16 tokens with channel order (py, px, c) -> (B, C, h*p, w*p)."""
    _dev(tokens, "unpatchify.tokens", BF16)
    B = tokens.shape[0]
    if not tokens.is_contiguous() or tokens.shape[1] != h * w or tokens.shape[2] != p * p * channels:
        raise UgError(f"unpatchify: expected contiguous (B, {h * w}, {p * p * channels}) tokens, got {tuple(tokens.shape)}")
    if out is None:
        out = torch.empty(B, channels, h * p, w * p, device=tokens.device, dtype=BF16)
    check(_lib.load().ug_unpatchify(tokens.data_ptr(), out.data_ptr(), B, h, w, p, channels, _stream()), "ug_unpatchify")
    return out


# ------------------------------------------------------------------------------------------------------------------
# AutoencoderKL (VAE) ops: NHWC bf16 activations [B, H, W, C] (SURVEY.md §8 (f)4 tail)
# ------------------------------------------------------------------------------------------------------------------
def _nhwc(t: torch.Tensor, name: str) -> torch.Tensor:
    _dev(t, name, BF16)
    if t.dim() != 4 or not t.is_contiguous():
        raise UgError(f"{name}: expected a contiguous NHWC [B, H, W, C] bf16 tensor, got shape {tuple(t.shape)} strides {t.stride()}")
    return t


def conv3x3_implicit_ok(c_in: int, width: int) -> bool:
    """Shapes the implicit-GEMM convolution takes (others go through im2col + gemm)."""
    return c_in % 64 == 0 and (width % 128 == 0 or (width <= 128 and 128 % width == 0))


def conv3x3(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
            out: Optional[torch.Tensor] = None, alpha: float = 1.0, variant: int = 0) -> torch.Tensor:
    """nn.Conv2d(k=3, s=1, p=1) over NHWC: x [B, H, W, Ci], w [Co, 9 * Ci] (column (ky*3+kx)*Ci + c), out [B, H, W, Co'] with
    Co' >= Co (the first Co channels of every pixel are written). Implicit GEMM: no im2col buffer."""
    from ._lib import Conv2dArgs
    _nhwc(x, "conv3x3.x")
    _dev(w, "conv3x3.w", BF16)
    B, H, W, Ci = x.shape
    Co = w.shape[0]
    if w.dim() != 2 or w.shape[1] != 9 * Ci or not w.is_contiguous():
        raise UgError(f"conv3x3: weight must be a contiguous [c_out, 9 * c_in] matrix, got {tuple(w.shape)} for c_in {Ci}")
    if out is None:
        out = torch.empty(B, H, W, Co, device=x.device, dtype=BF16)
    _nhwc(out, "conv3x3.out")
    if out.shape[:3] != x.shape[:3] or out.shape[3] < Co:
        raise UgError(f"conv3x3: out {tuple(out.shape)} does not match x {tuple(x.shape)} / c_out {Co}")
    a = Conv2dArgs()
    a.x, a.w, a.y, a.y_pixel_stride = x.data_ptr(), w.data_ptr(), out.data_ptr(), out.shape[3]
    a.batch, a.h, a.w_px, a.c_in, a.c_out = B, H, W, Ci, Co
    a.alpha, a.variant = float(alpha), int(variant)
    if bias is not None:
        a.bias = _dev(bias, "conv3x3.bias", BF16).data_ptr()
    if residual is not None:
        _nhwc(residual, "conv3x3.residual")
        if residual.shape[:3] != x.shape[:3] or residual.shape[3] < Co:
            raise UgError("conv3x3: residual shape mismatch")
        a.residual, a.res_pixel_stride = residual.data_ptr(), residual.shape[3]
    check(_lib.load().ug_conv3x3_bf16(C.byref(a), _stream()), "ug_conv3x3_bf16")
    return out


def im2col(x: torch.Tensor, layout: str, kh: int, kw: int, stride: int, pad_top: int, pad_left: int, h_out: int, w_out: int,
           k_pad: Optional[int] = None, out: Optional[torch.Tensor] = None, alpha: float = 1.0, beta: float = 0.0) -> torch.Tensor:
    """Patch gather -> bf16 [B * h_out * w_out, k_pad]; layout "nhwc" ([B, H, W, C]) or "nchw" ([B, C, H, W]), bf16 or fp32;
    in-image values pass through alpha * x + beta (padding stays zero)."""
    if not x.is_cuda or x.dim() != 4 or x.dtype not in (BF16, torch.float32):
        raise UgError("im2col: expected a 4-D CUDA bf16 / fp32 tensor — the UniGen hot path has no CPU fallback")
    if layout == "nhwc":
        B, H, W, Cc = x.shape
        sb, sy, sx, sc = x.stride()
    elif layout == "nchw":
        B, Cc, H, W = x.shape
        sb, sc, sy, sx = x.stride()
    else:
        raise UgError(f"im2col: unknown layout {layout!r}")
    k = kh * kw * Cc
    k_pad = k_pad or (k + 7) // 8 * 8
    rows = B * h_out * w_out
    if out is None:
        out = torch.empty(rows, k_pad, device=x.device, dtype=BF16)
    _dev(out, "im2col.out", BF16)
    if out.numel() < rows * k_pad or not out.is_contiguous():
        raise UgError("im2col: out too small / not contiguous")
    check(_lib.load().ug_im2col_bf16(x.data_ptr(), int(x.dtype == torch.float32), sb, sy, sx, sc, out.data_ptr(), B, H, W, Cc, kh, kw,
                                     stride, pad_top, pad_left, h_out, w_out, k_pad, float(alpha), float(beta), _stream()),
          "ug_im2col_bf16")
    return out.view(-1)[:rows * k_pad].view(rows, k_pad)


def groupnorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, groups: int, eps: float = 1e-6, silu_act: bool = False,
              out: Optional[torch.Tensor] = None, stats: Optional[torch.Tensor] = None) -> torch.Tensor:
    """GroupNorm(groups, C, eps) (+ SiLU) over NHWC bf16 [B, H, W, C]; out may be x."""
    _nhwc(x, "groupnorm.x")
    B, H, W, Cc = x.shape
    _dev(gamma, "groupnorm.weight", BF16), _dev(beta, "groupnorm.bias", BF16)
    if out is None:
        out = torch.empty_like(x)
    _nhwc(out, "groupnorm.out")
    need = B * groups * 2 * (1 + _lib.UG_GROUPNORM_MAX_CHUNKS)
    if stats is None:
        stats = torch.empty(need, device=x.device, dtype=torch.float32)
    _dev(stats, "groupnorm.stats", torch.float32)
    if stats.numel() < need:
        raise UgError("groupnorm: stats scratch too small")
    check(_lib.load().ug_groupnorm_bf16(x.data_ptr(), out.data_ptr(), gamma.data_ptr(), beta.data_ptr(), stats.data_ptr(), B, H * W, Cc,
                                        int(groups), float(eps), int(bool(silu_act)), _stream()), "ug_groupnorm_bf16")
    return out


def upsample2x(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _nhwc(x, "upsample2x.x")
    B, H, W, Cc = x.shape
    if out is None:
        out = torch.empty(B, 2 * H, 2 * W, Cc, device=x.device, dtype=BF16)
    _nhwc(out, "upsample2x.out")
    if tuple(out.shape) != (B, 2 * H, 2 * W, Cc):
        raise UgError("upsample2x: out shape mismatch")
    check(_lib.load().ug_upsample2x_nhwc_bf16(x.data_ptr(), out.data_ptr(), B, H, W, Cc, _stream()), "ug_upsample2x_nhwc_bf16")
    return out


def softmax_rows_(x: torch.Tensor) -> torch.Tensor:
    """In-place softmax over the last dim of a bf16 [rows, cols] view (unit inner stride)."""
    _dev(x, "softmax_rows.x", BF16)
    if x.dim() != 2 or x.stride(1) != 1:
        raise UgError("softmax_rows: expected a [rows, cols] view with contiguous cols")
    check(_lib.load().ug_softmax_rows_bf16(x.data_ptr(), x.stride(0), x.shape[0], x.shape[1], _stream()), "ug_softmax_rows_bf16")
    return x


def nhwc_to_nchw(x: torch.Tensor, channels: int, dtype=BF16, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """First `channels` channels of NHWC bf16 [B, H, W, C'] -> NCHW [B, channels, H, W] (bf16 or fp32)."""
    _nhwc(x, "nhwc_to_nchw.x")
    B, H, W, Cs = x.shape
    if dtype not in (BF16, torch.float32) or channels > Cs:
        raise UgError("nhwc_to_nchw: dtype must be bf16 / fp32 and channels <= C")
    if out is None:
        out = torch.empty(B, channels, H, W, device=x.device, dtype=dtype)
    _dev(out, "nhwc_to_nchw.out", dtype)
    if tuple(out.shape) != (B, channels, H, W) or not out.is_contiguous():
        raise UgError("nhwc_to_nchw: out shape mismatch / not contiguous")
    check(_lib.load().ug_nhwc_to_nchw(x.data_ptr(), Cs, out.data_ptr(), int(dtype == torch.float32), B, channels, H, W, _stream()),
          "ug_nhwc_to_nchw")
    return out


def vae_sample(moments: torch.Tensor, latent_channels: int, noise: Optional[torch.Tensor], shift: float = 0.0, scale: float = 1.0,
               out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """moments: NHWC bf16 [B, h, w, >= 2 * c] (mean | logvar) -> NCHW bf16 latents (mean + std * noise - shift) * scale;
    noise: fp32 NCHW [B, c, h, w] or None (the distribution's mode)."""
    _nhwc(moments, "vae_sample.moments")
    B, H, W, Cs = moments.shape
    c = int(latent_channels)
    if Cs < 2 * c:
        raise UgError("vae_sample: moments need 2 * latent_channels channels")
    if noise is not None:
        _dev(noise, "vae_sample.noise", torch.float32)
        if tuple(noise.shape) != (B, c, H, W) or not noise.is_contiguous():
            raise UgError("vae_sample: noise must be a contiguous fp32 [B, c, h, w] tensor")
    if out is None:
        out = torch.empty(B, c, H, W, device=moments.device, dtype=BF16)
    _dev(out, "vae_sample.out", BF16)
    check(_lib.load().ug_vae_sample(moments.data_ptr(), Cs, noise.data_ptr() if noise is not None else None, out.data_ptr(), B, c, H * W,
                                    float(shift), float(scale), _stream()), "ug_vae_sample")
    return out
