"""ctypes binding of libunigen_b200.so (include/unigen_b200.h). The library is mandatory: there is no Python or
CPU fallback for any op — a missing / unloadable extension raises at first use."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "libunigen_b200.so"

UG_ACT_NONE = 0
UG_ACT_GELU_TANH = 1
UG_MAX_SEGMENTS = 8
UG_GROUPNORM_MAX_CHUNKS = 1024
UG_ABI_VERSION = 11  # include/unigen_b200.h; checked against ug_abi_version() of the loaded library


class UgError(RuntimeError):
    pass


class GemmArgs(C.Structure):
    _fields_ = [
        ("a", C.c_void_p), ("a_row_stride", C.c_int64), ("a_batch_stride", C.c_int64),
        ("w", C.c_void_p), ("w_row_stride", C.c_int64), ("w_batch_stride", C.c_int64),
        ("c", C.c_void_p), ("c_row_stride", C.c_int64), ("c_batch_stride", C.c_int64),
        ("batch", C.c_int32), ("rows", C.c_int32), ("n", C.c_int32), ("k", C.c_int32),
        ("bias", C.c_void_p), ("bias_batch_stride", C.c_int64),
        ("gate", C.c_void_p), ("gate_batch_stride", C.c_int64),
        ("alpha", C.c_float), ("act", C.c_int32),
        ("residual", C.c_void_p), ("res_row_stride", C.c_int64), ("res_batch_stride", C.c_int64),
        ("variant", C.c_int32), ("reserved", C.c_int32),
        ("lora_t", C.c_void_p), ("lora_t_row_stride", C.c_int64), ("lora_t_batch_stride", C.c_int64),
        ("lora_b", C.c_void_p), ("lora_rank", C.c_int32), ("lora_block_n", C.c_int32), ("lora_nseg", C.c_int32),
        ("lora_seg_bounds", C.c_int32 * (UG_MAX_SEGMENTS + 1)), ("lora_seg_group", C.c_int32 * UG_MAX_SEGMENTS),
        ("qk_norm_weight", C.c_void_p), ("qk_cos_sin", C.c_void_p), ("qk_head_dim", C.c_int32), ("qk_d", C.c_int32),
        ("qk_eps", C.c_float), ("reserved2", C.c_int32), ("gate_seg_stride", C.c_int64),
        ("a2", C.c_void_p), ("a2_row_stride", C.c_int64), ("a2_batch_stride", C.c_int64),
        ("w2", C.c_void_p), ("w2_row_stride", C.c_int64), ("k2", C.c_int32), ("colmask_block", C.c_int32),
    ]


class GemmFp8Scales(C.Structure):
    _fields_ = [("a_scale", C.c_void_p), ("a_scale_batch_stride", C.c_int64),
                ("w_scale", C.c_void_p), ("w_scale_batch_stride", C.c_int64)]


class Conv2dArgs(C.Structure):
    _fields_ = [("x", C.c_void_p), ("w", C.c_void_p), ("bias", C.c_void_p), ("residual", C.c_void_p), ("res_pixel_stride", C.c_int64),
                ("y", C.c_void_p), ("y_pixel_stride", C.c_int64), ("batch", C.c_int32), ("h", C.c_int32), ("w_px", C.c_int32),
                ("c_in", C.c_int32), ("c_out", C.c_int32), ("alpha", C.c_float), ("variant", C.c_int32), ("reserved", C.c_int32)]


UG_MAX_PEERS = 8
UG_PEER_HEADER_BYTES = 4096
UG_PEER_HANDLE_BYTES = 64


class PeerTable(C.Structure):
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("base", C.c_void_p * UG_MAX_PEERS)]


class QkvScatterArgs(C.Structure):
    _fields_ = [("qkv", C.c_void_p), ("row_stride", C.c_int64), ("rows", C.c_int32), ("heads", C.c_int32),
                ("head_dim", C.c_int32), ("eps", C.c_float), ("norm_weight", C.c_void_p), ("cos_sin", C.c_void_p),
                ("dst_offset", C.c_int64), ("seq_total", C.c_int32), ("dst_row0", C.c_int32)]


UG_MAX_GEMV_JOBS = 1024


class GemvJob(C.Structure):
    _fields_ = [("w", C.c_void_p), ("bias", C.c_void_p), ("x", C.c_void_p), ("out", C.c_void_p),
                ("x_stride", C.c_int64), ("out_stride", C.c_int64), ("n", C.c_int32), ("k", C.c_int32),
                ("first_group", C.c_int32), ("flags", C.c_int32)]


UG_FLUX_MAX_CONDITIONS = 4


class FluxDesc(C.Structure):
    _fields_ = [("num_layers", C.c_int32), ("num_single_layers", C.c_int32), ("heads", C.c_int32), ("head_dim", C.c_int32),
                ("in_channels", C.c_int32), ("joint_dim", C.c_int32), ("pooled_dim", C.c_int32), ("guidance_embeds", C.c_int32),
                ("axes_dims_rope", C.c_int32 * 3), ("theta", C.c_float), ("n_ctrl_double", C.c_int32), ("n_ctrl_single", C.c_int32),
                ("experts", C.c_int32), ("condition_nums", C.c_int32), ("use_shared_expert", C.c_int32), ("single_add", C.c_int32),
                ("use_pooled_prompt_embeds", C.c_int32)]


class FluxInputs(C.Structure):
    _fields_ = [("batch", C.c_int32), ("n_img", C.c_int32), ("n_txt", C.c_int32), ("conditioning_scale", C.c_float),
                ("hidden_states", C.c_void_p), ("encoder_hidden_states", C.c_void_p), ("pooled_projections", C.c_void_p),
                ("timestep", C.c_void_p), ("timestep_stride", C.c_int64), ("guidance", C.c_void_p), ("img_ids", C.c_void_p),
                ("txt_ids", C.c_void_p), ("condition_hidden_states", C.c_void_p * UG_FLUX_MAX_CONDITIONS),
                ("condition_pooled_projections", C.c_void_p * UG_FLUX_MAX_CONDITIONS),
                ("condition_ids", C.c_void_p * UG_FLUX_MAX_CONDITIONS), ("rts_uniform", C.c_void_p * UG_FLUX_MAX_CONDITIONS)]


class FluxOutputs(C.Structure):
    _fields_ = [("velocity", C.c_void_p), ("expert_counts", C.c_void_p), ("l_aux", C.c_void_p)]


class AttnArgs(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p), ("o", C.c_void_p),
        ("q_row_stride", C.c_int64), ("q_batch_stride", C.c_int64),
        ("k_row_stride", C.c_int64), ("k_batch_stride", C.c_int64),
        ("v_row_stride", C.c_int64), ("v_batch_stride", C.c_int64),
        ("o_row_stride", C.c_int64), ("o_batch_stride", C.c_int64),
        ("batch", C.c_int32), ("heads", C.c_int32), ("seq", C.c_int32), ("head_dim", C.c_int32),
        ("scale", C.c_float), ("n_seg", C.c_int32),
        ("seg_bounds", C.POINTER(C.c_int32)), ("seg_visible", C.POINTER(C.c_uint32)),
        ("variant", C.c_int32), ("reserved", C.c_int32),
    ]


# name -> (restype, argtypes); every symbol include/unigen_b200.h declares
_VP, _I32, _I64, _F32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float
SIGNATURES = {
    "ug_last_error": (C.c_char_p, []),
    "ug_abi_version": (C.c_int, []),
    "ug_device_check": (C.c_int, []),
    "ug_launch_count": (C.c_int64, []),
    "ug_reset_launch_count": (None, []),
    "ug_gemm_bf16": (C.c_int, [C.POINTER(GemmArgs), _VP]),
    "ug_gemm_fp8": (C.c_int, [C.POINTER(GemmArgs), C.POINTER(GemmFp8Scales), _VP]),
    "ug_gemm_fp8_lora": (C.c_int, [C.POINTER(GemmArgs), C.POINTER(GemmFp8Scales), _VP]),
    "ug_quant_rows_fp8": (C.c_int, [_VP, _I64, _I64, _VP, _I64, _I64, _VP, _I64, _I32, _I32, _I32, _VP]),
    "ug_ln_modulate_fp8": (C.c_int, [_VP, _I64, _I64, _VP, _I64, _I64, _VP, _I64, _VP, _VP, _I64, _I32, _I32, _I32, _F32, _VP]),
    "ug_lora_down": (C.c_int, [_VP, _I64, _I64, _VP, _VP, _I64, _I64, _I32, _I32, _I32, _I32, _I32,
                               C.POINTER(C.c_int32), C.POINTER(C.c_int32), _VP]),
    "ug_lora_down_wide": (C.c_int, [_VP, _I64, _I64, _VP, _VP, _I64, _I64, _I32, _I32, _I32, _I32, _I32, _I32, _I32,
                                    C.POINTER(C.c_int32), C.POINTER(C.c_int32), _VP]),
    "ug_attention_bf16": (C.c_int, [C.POINTER(AttnArgs), _VP]),
    "ug_expand_segment_mask": (C.c_int, [_I32, _I32, C.POINTER(C.c_int32), C.POINTER(C.c_uint32), _VP, _VP]),
    "ug_ln_modulate": (C.c_int, [_VP, _I64, _I64, _VP, _I64, _I64, _VP, _VP, _I64, _I32, _I32, _I32, _F32, _VP]),
    "ug_ln_modulate_segs": (C.c_int, [_VP, _I64, _I64, _VP, _I64, _I64, _VP, _VP, _I64, _I64, _I32, C.POINTER(C.c_int32), _I32, _I32,
                                      _I32, _F32, _VP]),
    "ug_ln_modulate_segs_fp8": (C.c_int, [_VP, _I64, _I64, _VP, _I64, _I64, _VP, _I64, _VP, _VP, _I64, _I64, _I32, C.POINTER(C.c_int32),
                                          _I32, _I32, _I32, _F32, _VP]),
    "ug_ln_modulate_slots": (C.c_int, [_VP, _I64, _VP, _I64, _VP, _VP, _I64, _I64, _VP, _I32, _I32, _I32, _I32, _I32, _F32, _VP]),
    "ug_gated_add_slots": (C.c_int, [_VP, _I64, _VP, _I64, _VP, _I64, _I64, _VP, _I32, _I32, _I32, _I32, _I32, _VP]),
    "ug_qk_rmsnorm_rope": (C.c_int, [_VP, _I64, _I64, _I32, _I32, _I32, _I32, _VP, _I32, _F32, _VP, _VP]),
    "ug_rope_table": (C.c_int, [_VP, _I32, C.POINTER(C.c_int32), _F32, _VP, _VP]),
    "ug_gemv": (C.c_int, [_VP, _I64, _VP, _VP, _VP, _I64, _I32, _I32, _I32, _I32, _I32, _I32, _VP]),
    "ug_gemv_grouped": (C.c_int, [_VP, _I32, _I32, _I32, _I32, _I32, C.POINTER(PeerTable), _VP]),
    "ug_silu_f32": (C.c_int, [_VP, _VP, _I64, _VP]),
    "ug_flux_create": (C.c_int, [C.POINTER(FluxDesc), C.POINTER(C.c_void_p)]),
    "ug_flux_destroy": (None, [_VP]),
    "ug_flux_bind_weight": (C.c_int, [_VP, C.c_char_p, _VP, _I32, C.POINTER(C.c_int64), _I32]),
    "ug_flux_workspace_bytes": (C.c_size_t, [_VP, _I32, _I32, _I32]),
    "ug_flux_forward": (C.c_int, [_VP, C.POINTER(FluxInputs), C.POINTER(FluxOutputs), _VP, C.c_size_t, _VP]),
    "ug_timestep_embedding": (C.c_int, [_VP, _I64, _I32, _I32, _F32, _VP, _VP]),
    "ug_add_bf16": (C.c_int, [_VP, _I64, _I64, _VP, _I64, _I64, _VP, _I64, _I64, _I32, _I32, _I32, _VP]),
    "ug_copy_bf16": (C.c_int, [_VP, _I64, _I64, _VP, _I64, _I64, _I32, _I32, _I32, _VP]),
    "ug_cast_f32_to_bf16": (C.c_int, [_VP, _VP, _I64, _VP]),
    "ug_cast_bf16_to_f32": (C.c_int, [_VP, _VP, _I64, _VP]),
    "ug_moe_route": (C.c_int, [_VP, _VP, _VP, _I32, _I32, _I32, _I32, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "ug_moe_gather_modulate": (C.c_int, [_VP, _VP, _VP, _I64, _I64, _VP, _VP, _I32, _I32, _I32, _I32, _VP]),
    "ug_moe_combine": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _I32, _I32, _I32, _VP]),
    "ug_euler_step": (C.c_int, [_VP, _VP, _F32, _F32, _I64, _VP]),
    "ug_euler_step_table": (C.c_int, [_VP, _VP, _VP, _I32, _I64, _VP]),
    "ug_cfg_combine": (C.c_int, [_VP, _VP, _F32, _VP, _I64, _VP]),
    "ug_pack_latents": (C.c_int, [_VP, _VP, _I32, _I32, _I32, _I32, _I32, _VP]),
    "ug_peer_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "ug_peer_free": (C.c_int, [_VP]),
    "ug_peer_export": (C.c_int, [_VP, C.POINTER(C.c_uint8)]),
    "ug_peer_open": (C.c_int, [C.POINTER(C.c_uint8), C.POINTER(C.c_void_p)]),
    "ug_peer_close": (C.c_int, [_VP]),
    "ug_peer_barrier": (C.c_int, [C.POINTER(PeerTable), _VP]),
    "ug_peer_error": (C.c_int, [C.POINTER(PeerTable), C.POINTER(C.c_int32)]),
    "ug_peer_set_timeout_ms": (C.c_int, [_I64]),
    "ug_peer_error_async": (C.c_int, [C.POINTER(PeerTable), _VP, _VP]),
    "ug_qkv_scatter": (C.c_int, [C.POINTER(PeerTable), C.POINTER(QkvScatterArgs), _VP]),
    "ug_attention_bf16_peer": (C.c_int, [C.POINTER(AttnArgs), C.POINTER(PeerTable), _I64, _I32, _VP]),
    "ug_peer_bcast_rows": (C.c_int, [C.POINTER(PeerTable), _VP, _I64, _I32, _I32, _I64, _I64, _I32, _VP]),
    "ug_unpatchify": (C.c_int, [_VP, _VP, _I32, _I32, _I32, _I32, _I32, _VP]),
    "ug_conv3x3_bf16": (C.c_int, [C.POINTER(Conv2dArgs), _VP]),
    "ug_im2col_bf16": (C.c_int, [_VP, _I32, _I64, _I64, _I64, _I64, _VP, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _I32,
                                 _I32, _F32, _F32, _VP]),
    "ug_groupnorm_bf16": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _I32, _I32, _I32, _I32, _F32, _I32, _VP]),
    "ug_upsample2x_nhwc_bf16": (C.c_int, [_VP, _VP, _I32, _I32, _I32, _I32, _VP]),
    "ug_softmax_rows_bf16": (C.c_int, [_VP, _I64, _I32, _I32, _VP]),
    "ug_nhwc_to_nchw": (C.c_int, [_VP, _I64, _VP, _I32, _I32, _I32, _I32, _I32, _VP]),
    "ug_vae_sample": (C.c_int, [_VP, _I64, _VP, _VP, _I32, _I32, _I32, _F32, _F32, _VP]),
}

_lib = None


def load() -> C.CDLL:
    """Load the shared library (building it is `__graft_entry__.build()`'s job) and type every entry point."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise UgError(
            f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback for the UniGen hot path)")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library drift apart
        fn.restype = res
        fn.argtypes = args
    got = int(lib.ug_abi_version())
    if got != UG_ABI_VERSION:
        raise UgError(f"{LIB_PATH} reports ABI version {got}, this package binds version {UG_ABI_VERSION}: stale build — "
                      "rebuild with `python -c 'import __graft_entry__ as g; g.build()'`")
    _lib = lib
    return lib


def check(status: int, what: str = "") -> None:
    if status != 0:
        msg = load().ug_last_error().decode(errors="replace")
        raise UgError(f"{what or 'unigen_b200'} failed with status {status}: {msg}")
