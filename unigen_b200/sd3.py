"""Host-side mirror of the reference's SD3.5 denoiser (`UniGenSD3`, reference src/UniGenTransformer.py:490-710 on top of
`UniGenBase` :20-296, block overrides src/UniGenUtils.py:340-522) for the B200-native path — SURVEY.md §8 row A16,
BASELINE cfg5.

Public surface kept: `init_condition_block(condition_nums=..., control_params=...)`, `forward(hidden_states,
condition_hidden_states, conditioning_scale, encoder_hidden_states, pooled_projections, condition_pooled_projections,
timestep, joint_attention_kwargs, skip_layers, **kwargs) -> (velocity (B, C, H, W), {moe_loss}, {expert_counts})`
(:625-710), reference state-dict keys, `.config`, `.dtype`, `.trainable_control_modules`.  Every arithmetic op runs in
libunigen_b200.so; there is no eager / CPU fallback.

Configuration covered = the SHIPPED control_params (config/unigen.yaml): `use_modulate: False`, no `use_rope`,
`use_shared_expert: True`, `use_encoder_hidden_states: True`, `cn2base_method: add` — experts are two
`SD3SingleTransformerBlock`s per expert run on the dispatched capacity buffers with a per-token temb — plus the two
reachable switches around it: `use_modulate: True` (:171-183, :252-255: the experts are the condition-modulated linear
pairs of the Flux class, stacked [E, D, D] and run as two batched GEMMs over the capacity slots) and
`use_shared_expert: False` (:203, :279: the routed experts' outputs alone feed the control stream).
`use_rope: True` stays rejected: the reference's own forward raises NameError there (`prepare_latent_image_ids`, :657,
is defined nowhere in the reference), so there is no behaviour to match.

Data layout in HBM (bf16 unless noted)
  X     [B, N+T, D]  joint residual stream, SAMPLE ROWS FIRST (JointAttnProcessor2_0 concatenates sample | context)
  NX / NX2 / QKV / QKV2 / AO / AO2 / FF   per-block scratch sized for the longest joint sequence (shared_expert[1]: 2N+T)
  PAT   [B, N, C*p*p] patchified latents: PatchEmbed's Conv2d(k=p, s=p) is ONE tcgen05 GEMM with the flattened conv
        weight, the cropped sincos table rides in the epilogue as the residual operand (batch stride 0)
  SL[2] [E*C, D]     capacity-slot buffers of the transformer-block experts; all E experts run as ONE batched GEMM /
        attention launch per op (weights stacked [E, ., .]); per-token AdaLN = a (samples+1)-row table per expert
        indexed through slot_token (row B = the all-zero temb of empty slots, which DO take part in the attention)
  MOD   fp32         AdaLN vectors of all 48 blocks, computed once per step
"""
from __future__ import annotations

import types
from typing import Any, Dict, Optional

import torch

from . import ops
from .model import BF16, FP8, _DenoiserBase, _TimeTextW, _Weights
from .ops import UG_ACT_GELU_TANH


class SD3Arch:
    """diffusers SD3Transformer2DModel config fields read on the path (SD3.5-medium values, SURVEY.md §A.10)."""

    def __init__(self, sample_size=128, patch_size=2, in_channels=16, out_channels=16, num_layers=24, attention_head_dim=64,
                 num_attention_heads=24, joint_attention_dim=4096, pooled_projection_dim=2048, pos_embed_max_size=384,
                 qk_norm="rms_norm", dual_attention_layers=tuple(range(13))):
        self.sample_size, self.patch_size, self.in_channels, self.out_channels = sample_size, patch_size, in_channels, out_channels
        self.num_layers, self.attention_head_dim, self.num_attention_heads = num_layers, attention_head_dim, num_attention_heads
        self.joint_attention_dim, self.pooled_projection_dim = joint_attention_dim, pooled_projection_dim
        self.pos_embed_max_size, self.qk_norm = pos_embed_max_size, qk_norm
        self.dual_attention_layers = tuple(dual_attention_layers)
        self.caption_projection_dim = num_attention_heads * attention_head_dim

    @staticmethod
    def tiny():
        return SD3Arch(sample_size=32, num_layers=4, num_attention_heads=6, pos_embed_max_size=48, dual_attention_layers=(0, 1))


def sincos_pos_embed_2d(embed_dim: int, grid_size: int, base_size: int) -> torch.Tensor:
    """diffusers get_2d_sincos_pos_embed(embed_dim, grid_size, base_size=..., interpolation_scale=1) -> fp32
    [1, grid*grid, embed_dim] (W-first meshgrid, [sin | cos] per axis, float64 angles). A constant of the architecture
    (PatchEmbed registers it as a persistent buffer), computed once at construction — not on the per-step path."""
    g = torch.arange(grid_size, dtype=torch.float32) / (grid_size / base_size)
    gy, gx = torch.meshgrid(g, g, indexing="ij")  # numpy meshgrid(gw, gh)[0] = x coordinate, [1] = y coordinate

    def axis(pos, dim):
        omega = 1.0 / 10000 ** (torch.arange(dim // 2, dtype=torch.float64) / (dim / 2.0))
        out = pos.reshape(-1).double()[:, None] * omega[None, :]
        return torch.cat([out.sin(), out.cos()], dim=1)

    return torch.cat([axis(gx, embed_dim // 2), axis(gy, embed_dim // 2)], dim=1).float().unsqueeze(0)


class _PatchEmbedW:
    """PatchEmbed: Conv2d(C, D, k=p, s=p) weight kept as its [D, C*p*p] GEMM matrix (state-dict view: [D, C, p, p])."""

    def __init__(self, ws: _Weights, p: str, a: SD3Arch, D: int):
        k = a.in_channels * a.patch_size * a.patch_size
        self.w, self.b = ws.alloc(D, k), ws.alloc(D)
        ws.views[p + ".proj.weight"] = self.w.view(D, a.in_channels, a.patch_size, a.patch_size)
        ws.views[p + ".proj.bias"] = self.b
        self.table = ws.alloc(1, a.pos_embed_max_size ** 2, D, dtype=torch.float32)
        self.table.copy_(sincos_pos_embed_2d(D, a.pos_embed_max_size, a.sample_size // a.patch_size))
        ws.views[p + ".pos_embed"] = self.table
        self._crop: Dict[Any, torch.Tensor] = {}
        self.max_size = a.pos_embed_max_size

    def cropped(self, h: int, w: int) -> torch.Tensor:
        """PatchEmbed.cropped_pos_embed as a bf16 [h*w, D] table (cached per latent size; index glue only)."""
        key = (h, w)
        if key not in self._crop:
            m = self.max_size
            if h > m or w > m:
                raise ops.UgError(f"latent grid {h}x{w} exceeds pos_embed_max_size {m}")
            top, left = (m - h) // 2, (m - w) // 2
            t = self.table.view(m, m, -1)[top:top + h, left:left + w].reshape(h * w, -1)
            self._crop[key] = ops.to_bf16(t.contiguous())
        return self._crop[key]


class _AttnW:
    def __init__(self, ws: _Weights, p: str, D: int, dh: int, added: bool, add_out: bool, qk_norm: bool):
        self.qkv = ws.fused([f"{p}.to_q", f"{p}.to_k", f"{p}.to_v"], D, D)
        self.to_out = ws.linear(p + ".to_out.0", D, D)
        self.rms = self.rms_ctx = self.add_qkv = self.to_add_out = None
        if qk_norm:
            self.rms = ws.alloc(2, dh)
            ws.views[p + ".norm_q.weight"], ws.views[p + ".norm_k.weight"] = self.rms[0], self.rms[1]
        if added:
            self.add_qkv = ws.fused([f"{p}.add_q_proj", f"{p}.add_k_proj", f"{p}.add_v_proj"], D, D)
            if add_out:
                self.to_add_out = ws.linear(p + ".to_add_out", D, D)
            if qk_norm:
                self.rms_ctx = ws.alloc(2, dh)
                ws.views[p + ".norm_added_q.weight"], ws.views[p + ".norm_added_k.weight"] = self.rms_ctx[0], self.rms_ctx[1]


class _JointBlockW:
    """JointTransformerBlock(dim, heads, head_dim, context_pre_only, qk_norm, use_dual_attention) parameters."""
    # linears `UniGenSD3.quantize_fp8()` converts (model.quantize_block_linears); the ones a block layout lacks (attn2 without
    # dual attention, to_add_out / ff_context in a context_pre_only block) are None and skipped
    FP8_LINEARS = ("attn.qkv", "attn.add_qkv", "attn.to_out", "attn.to_add_out", "attn2.qkv", "attn2.to_out",
                   "ff1", "ff2", "ffc1", "ffc2")
    fp8 = False

    def __init__(self, ws: _Weights, p: str, D: int, dh: int, dual: bool, context_pre_only: bool, qk_norm: bool):
        self.dual, self.context_pre_only = dual, context_pre_only
        self.n1, self.n1c = (9 if dual else 6), (2 if context_pre_only else 6)
        self.norm1 = ws.linear(p + ".norm1.linear", self.n1 * D, D)
        self.norm1_ctx = ws.linear(p + ".norm1_context.linear", self.n1c * D, D)
        self.attn = _AttnW(ws, p + ".attn", D, dh, True, not context_pre_only, qk_norm)
        self.attn2 = _AttnW(ws, p + ".attn2", D, dh, False, False, qk_norm) if dual else None
        self.ff1 = ws.linear(p + ".ff.net.0.proj", 4 * D, D)
        self.ff2 = ws.linear(p + ".ff.net.2", D, 4 * D)
        self.ffc1 = self.ffc2 = None
        if not context_pre_only:
            self.ffc1 = ws.linear(p + ".ff_context.net.0.proj", 4 * D, D)
            self.ffc2 = ws.linear(p + ".ff_context.net.2", D, 4 * D)


class _ExpertStackW:
    """One branch (0: hidden, 1: condition) of all E transformer-block experts, stacked along a leading expert axis so
    every op of the E `SD3SingleTransformerBlock`s is one batched launch."""

    def __init__(self, ws: _Weights, E: int, br: int, D: int):
        self.norm1_w, self.norm1_b = ws.alloc(E * 6 * D, D), ws.alloc(E * 6 * D)
        self.qkv_w, self.qkv_b = ws.alloc(E, 3 * D, D), ws.alloc(E, 3 * D)
        self.out_w, self.out_b = ws.alloc(E, D, D), ws.alloc(E, D)
        self.ff1_w, self.ff1_b = ws.alloc(E, 4 * D, D), ws.alloc(E, 4 * D)
        self.ff2_w, self.ff2_b = ws.alloc(E, D, 4 * D), ws.alloc(E, D)
        for e in range(E):
            p = f"moe.moe_layer.experts.deepspeed_experts.{e}.{br}"
            ws.views[p + ".norm1.linear.weight"] = self.norm1_w[e * 6 * D:(e + 1) * 6 * D]
            ws.views[p + ".norm1.linear.bias"] = self.norm1_b[e * 6 * D:(e + 1) * 6 * D]
            for i, n in enumerate(("to_q", "to_k", "to_v")):
                ws.views[f"{p}.attn.{n}.weight"] = self.qkv_w[e, i * D:(i + 1) * D]
                ws.views[f"{p}.attn.{n}.bias"] = self.qkv_b[e, i * D:(i + 1) * D]
            ws.views[p + ".attn.to_out.0.weight"], ws.views[p + ".attn.to_out.0.bias"] = self.out_w[e], self.out_b[e]
            ws.views[p + ".ff.net.0.proj.weight"], ws.views[p + ".ff.net.0.proj.bias"] = self.ff1_w[e], self.ff1_b[e]
            ws.views[p + ".ff.net.2.weight"], ws.views[p + ".ff.net.2.bias"] = self.ff2_w[e], self.ff2_b[e]


class UniGenSD3(_DenoiserBase):
    """B200-native drop-in for the reference `UniGenSD3` (SD3.5 MMDiT denoiser + WeaveNet control branch + CoMoE)."""

    def __init__(self, arch: Optional[SD3Arch] = None, device: Any = "cuda", **config):
        super().__init__()
        self.arch = arch or SD3Arch(**config)
        self._init_base(device)
        a = self.arch
        self.config = types.SimpleNamespace(
            sample_size=a.sample_size, patch_size=a.patch_size, in_channels=a.in_channels, out_channels=a.out_channels,
            num_layers=a.num_layers, attention_head_dim=a.attention_head_dim, num_attention_heads=a.num_attention_heads,
            joint_attention_dim=a.joint_attention_dim, caption_projection_dim=a.caption_projection_dim,
            pooled_projection_dim=a.pooled_projection_dim, pos_embed_max_size=a.pos_embed_max_size, qk_norm=a.qk_norm,
            dual_attention_layers=a.dual_attention_layers, guidance_embeds=False)
        self.out_channels = a.out_channels
        self.inner_dim = a.num_attention_heads * a.attention_head_dim
        if a.patch_size != 2:
            raise ops.UgError("PatchEmbed patch_size must be 2 (ug_pack_latents is the patchify kernel)")
        D, dh, ws = self.inner_dim, a.attention_head_dim, self._ws
        qk = a.qk_norm is not None
        self.pos_embed_w = _PatchEmbedW(ws, "pos_embed", a, D)
        self.time_text = _TimeTextW(ws, "time_text_embed", D, a.pooled_projection_dim, False)
        self.context_embedder_w = ws.linear("context_embedder", D, a.joint_attention_dim)
        self.blocks = [_JointBlockW(ws, f"transformer_blocks.{i}", D, dh, i in a.dual_attention_layers, i == a.num_layers - 1, qk)
                       for i in range(a.num_layers)]
        self.norm_out_w = ws.linear("norm_out.linear", 2 * D, D)
        self.proj_out_w = ws.linear("proj_out", a.patch_size * a.patch_size * a.out_channels, D)

    # ---------------------------------------------------------------------------------------------------------
    # reference API: construction (src/UniGenTransformer.py:21-219, 490-496)
    # ---------------------------------------------------------------------------------------------------------
    def init_condition_block(self, condition_nums: int = 1, **kwargs):
        self.condition_nums = condition_nums
        self.init_control_block(kwargs.get("control_params", None))

    def init_control_block(self, control_params=None):
        assert control_params is not None, ValueError("Please provice control net model parameter")
        get = control_params.get
        a, ws, D, dh = self.arch, self._ws, self.inner_dim, self.arch.attention_head_dim
        self.use_pooled_prompt_embeds = get("use_pooled_prompt_embeds", True)
        self.use_encoder_hidden_states = get("use_encoder_hidden_states", True)
        assert self.use_encoder_hidden_states, ValueError("please use joint transformer block to enhance condition hidden states")
        self.use_rope, self.use_modulate = bool(get("use_rope", False)), bool(get("use_modulate", False))
        if self.use_rope:
            raise ops.UgError("UniGenSD3 use_rope=True: the reference forward raises NameError (prepare_latent_image_ids, "
                              "src/UniGenTransformer.py:657, is defined nowhere) — there is no behaviour to reproduce")
        if get("use_pos_embed", False) or get("extra_conditioning_channels", 0):
            raise ops.UgError("use_pos_embed / extra_conditioning_channels are not covered by the B200-native SD3 path")
        self.use_shared_expert = bool(get("use_shared_expert", False))  # :203 (False: the routed experts alone, :279 skipped)
        self.cn_method = get("cn2base_method", "add")
        if self.cn_method != "add":
            raise ops.UgError("cn2base_method='CrossAttn' needs attn.condition_k_proj, which nothing creates (SURVEY.md §2); unsupported")
        self.control_blocks_num = get("num_layers", a.num_layers)
        self.expert_nums = get("expert_num", None) or (self.condition_nums + 1) * get("expert_num_each_condition", 3)
        self.top_k = get("top_num", 1)
        assert self.top_k == 1, "only top-1 gating (the shipped configuration) is implemented"
        self.num_local_experts = self.expert_nums
        qk = get("qk_norm", a.qk_norm) is not None
        dual_layers = tuple(get("dual_attention_layers", a.dual_attention_layers))

        self.control_pos_embed_input_w = _PatchEmbedW(ws, "control_pos_embed_input", a, D)
        self.control_time_text = _TimeTextW(ws, "control_time_text_embed", D, a.pooled_projection_dim, False)
        self.control_condition = _TimeTextW(ws, "control_condition_embed", D, a.pooled_projection_dim, False)
        self.control_context_embedder_w = ws.linear("control_context_embedder", D, D)  # UniGenSD3 re-creates it as (D, D) :493
        self.ctrl_blocks = [_JointBlockW(ws, f"control_transformer_blocks.{j}", D, dh, j in dual_layers, False, qk)
                            for j in range(self.control_blocks_num)]
        self.add_blocks = [ws.linear(f"controlnet_add_blocks.{j}", D, D) for j in range(self.control_blocks_num)]
        E = self.expert_nums
        self.gate_wg = ws.alloc(E, D, dtype=torch.float32)
        ws.views["moe.moe_layer.gate.wg.weight"] = self.gate_wg
        if self.use_modulate:
            # :173-182: expert = [[Linear(D, D), Linear(pooled, D)] (condition), [Linear(D, D), Linear(pooled, D)] (hidden)],
            # stacked over the experts exactly like the Flux class's (model.py)
            P = a.pooled_projection_dim
            self.experts = []
            self.exp_w, self.exp_b = [ws.alloc(E, D, D), ws.alloc(E, D, D)], [ws.alloc(E, D), ws.alloc(E, D)]
            self.exp_mod_w, self.exp_mod_b = [ws.alloc(E * D, P), ws.alloc(E * D, P)], [ws.alloc(E * D), ws.alloc(E * D)]
            for e in range(E):
                for br in (0, 1):
                    p = f"moe.moe_layer.experts.deepspeed_experts.{e}.{br}"
                    ws.views[p + ".0.weight"], ws.views[p + ".0.bias"] = self.exp_w[br][e], self.exp_b[br][e]
                    ws.views[p + ".1.weight"] = self.exp_mod_w[br][e * D:(e + 1) * D]
                    ws.views[p + ".1.bias"] = self.exp_mod_b[br][e * D:(e + 1) * D]
        else:
            self.experts = [_ExpertStackW(ws, E, 0, D), _ExpertStackW(ws, E, 1, D)]
        self.shared = [_JointBlockW(ws, "shared_expert.0", D, dh, False, False, qk),
                       _JointBlockW(ws, "shared_expert.1", D, dh, True, True, qk)] if self.use_shared_expert else []
        self.trainable_control_modules = {k: None for k in (
            "control_pos_embed_input", "control_time_text_embed", "control_condition_embed", "control_context_embedder",
            "control_transformer_blocks", "controlnet_add_blocks", "moe") + (("shared_expert",) if self.use_shared_expert else ())}
        self._control_ready = True
        if get("use_transformer_params", False):
            self.init_control_param()

    @torch.no_grad()
    def init_control_param(self):
        """reference src/UniGenTransformer.py:144-158: the control branch starts from the base model's weights —
        `control_pos_embed_input` <- `pos_embed`, both control time-text embedders <- `time_text_embed`, control block j <-
        base block j (`load_state_dict(..., strict=False)` over the ModuleLists). `control_context_embedder` is re-created
        as a fresh Linear(D, D) right after (:493), so nothing is copied into it. Deviation, on purpose: the LAST base block is
        context_pre_only (`norm1_context.linear` [2D, D], no `to_add_out` / `ff_context`) while its control twin is not
        ([6D, D]) — `strict=False` does not forgive a size mismatch, so the reference call raises RuntimeError with the
        shipped 24 + 24 layout; here keys whose shapes differ are skipped and the call succeeds."""
        if self.linear_dtype != BF16:
            raise ops.UgError("init_control_param on an fp8-quantised model: it copies through the state-dict views, which no longer "
                              "list the quantised block weights — call it (or use_transformer_params) before quantize_fp8()")
        v = self._ws.views

        def copy_prefix(dst: str, src: str):
            for k in [k for k in v if k.startswith(src + ".")]:
                kd = dst + k[len(src):]
                if kd in v and v[kd].shape == v[k].shape:
                    v[kd].copy_(v[k])

        copy_prefix("control_pos_embed_input", "pos_embed")
        copy_prefix("control_time_text_embed", "time_text_embed")
        copy_prefix("control_condition_embed", "time_text_embed")
        for j in range(min(self.control_blocks_num, self.arch.num_layers)):
            copy_prefix(f"control_transformer_blocks.{j}", f"transformer_blocks.{j}")
        self._weights_loaded()

    def quantize_fp8(self):
        """Opt-in fp8 (e4m3) transformer-block linears, in place; returns self (a second call does nothing). Every linear of the
        base and control joint blocks — q|k|v, add_q|k|v, to_out, to_add_out, attn2 q|k|v and attn2.to_out (dual-attention
        layers), ff and ff_context (the context_pre_only last block has neither to_add_out nor ff_context) — gets one fp32 scale
        per output channel and is stored as e4m3; its bf16 copy is released (and leaves `state_dict()`). In every forward their
        operands are quantised per token row on the device and the GEMMs run on the fp8 tensor cores. The patch / context /
        time / text embedders, the AdaLN GEMVs, the control add-linears, norm_out / proj_out, attention and the whole CoMoE
        pre-stage (routed experts, shared experts, gate: routing stays bit-exact) stay bf16. Call after `init_condition_block`
        and any `load_state_dict` / `init_control_param`. Afterwards `state_dict()` / `parameters()` no longer list the quantised
        weights (their biases and every bf16 tensor stay), and `load_state_dict`, `init_random_` and `init_control_param`
        raise `UgError`."""
        return self._quantize_fp8()

    def _fp8_blocks(self):
        return self.blocks + self.ctrl_blocks

    def _weights_loaded(self):
        self.pos_embed_w._crop.clear()
        if self._control_ready:
            self.control_pos_embed_input_w._crop.clear()

    # ---------------------------------------------------------------------------------------------------------
    def _workspace(self, B: int, N: int, T: int):
        return self._cached_workspace((B, N, T), lambda: self._make_workspace(B, N, T))

    def _make_workspace(self, B: int, N: int, T: int):
        a, D, dev = self.arch, self.inner_dim, self.device_
        S, Smax = N + T, 2 * N + T
        E = self.expert_nums
        C = ops.moe_capacity(B * N, E)
        z = lambda *s, dt=BF16: torch.empty(*s, device=dev, dtype=dt)  # noqa: E731
        n_mod = sum(w.n1 + w.n1c for w in self.blocks + self.ctrl_blocks + self.shared) + 2
        kpe = a.in_channels * a.patch_size ** 2
        b = types.SimpleNamespace(
            X=z(B, S, D), NX=z(B, Smax, D), NX2=z(B, 2 * N, D), QKV=z(B, Smax, 3 * D), QKV2=z(B, 2 * N, 3 * D),
            AO=z(B, Smax, D), AO2=z(B, 2 * N, D), FF=z(B, Smax, 4 * D), CH=z(B, N, D), CENC=z(B, T, D), COND=z(B, N, D),
            HC=z(B, 2 * N, D), G=z(B * N, D), CIN=z(B, N, D), EH=z(B * N, D), EC=z(B * N, D),
            SL=[z(E * C, D), z(E * C, D)], SNX=z(E * C, D), SQKV=z(E * C, 3 * D), SAO=z(E * C, D), STMP=z(E * C, D),
            SFF=z(E * C, 4 * D), SMODT=[z(B + 1, E * 6 * D, dt=torch.float32) for _ in (0, 1)],
            TE=[torch.zeros(B + 1, D, device=dev, dtype=torch.float32) for _ in (0, 1)],  # [temb rows | zero row]
            MOD=z(B, n_mod * D, dt=torch.float32), temb=z(B, D, dt=torch.float32), tmp=z(B, D, dt=torch.float32),
            PAT=z(B, N, kpe), NO=z(B, N, D), OUT=z(B, N, a.patch_size ** 2 * a.out_channels), capacity=C)
        if self.use_modulate:  # per-sample, per-expert modulation vectors of the two linear experts
            b.MODC, b.MODH = z(B, E, D, dt=torch.float32), z(B, E, D, dt=torch.float32)
        if self.linear_dtype == FP8:
            # e4m3 operands (+ one fp32 scale per row) of the quantised block linears. Only base and control blocks are
            # quantised, and they run over N + T rows (the 2N + T rows of shared_expert[1] stay bf16). Row layout as in
            # NX / NX2 / AO / FF: sample rows [0, n), context rows [n, n + T).
            f8 = lambda *sh: z(*sh, dt=FP8)  # noqa: E731
            b.NXQ, b.NXS = f8(B, S, D), z(B, S, dt=torch.float32)
            b.NX2Q, b.NX2S = f8(B, N, D), z(B, N, dt=torch.float32)
            b.AOQ, b.AOS = f8(B, S, D), z(B, S, dt=torch.float32)
            b.FFQ, b.FFS = f8(B, S, 4 * D), z(B, S, dt=torch.float32)
        return b

    def _sd3_mod_plans(self, buf, B: int):
        """Job tables (ops.GemvPlan) of every block's AdaLN linear `linear(silu(temb))` for this workspace + the MOD chunk views."""
        mp = getattr(buf, "mod_plans", None)
        if mp is not None:
            return mp
        D = self.inner_dim
        control_temb, condition_temb = buf.TE[0][:B], buf.TE[1][:B]
        slot, early, late = [0], [], []

        def job(w, x, n_chunks, dst):
            s0 = slot[0]
            slot[0] += n_chunks
            region = buf.MOD[:, s0 * D:(s0 + n_chunks) * D]
            dst.append((w[0], w[1], x, region, True))  # SiLU applied on the fly (three distinct temb vectors)
            return [region[:, i * D:(i + 1) * D] for i in range(n_chunks)]

        def pair(w, x, dst):
            return job(w.norm1, x, w.n1, dst), job(w.norm1_ctx, x, w.n1c, dst)

        mp = types.SimpleNamespace()
        mp.m_base = [pair(w, buf.temb, early if i == 0 else late) for i, w in enumerate(self.blocks)]
        mp.m_ctrl = [pair(w, condition_temb, early if j == 0 else late) for j, w in enumerate(self.ctrl_blocks)]
        mp.mods_s0 = mp.mods_s1 = None
        if self.use_shared_expert:
            mp.mods_s0, mp.mods_s1 = pair(self.shared[0], condition_temb, early), pair(self.shared[1], control_temb, early)
        mp.m_out = job(self.norm_out_w, buf.temb, 2, late)  # AdaLayerNormContinuous: (scale, shift)
        mp.early, mp.late = ops.GemvPlan(early, self.device_), ops.GemvPlan(late, self.device_)
        buf.mod_plans = mp
        return mp

    def _patch_embed(self, buf, w: _PatchEmbedW, latents: torch.Tensor, out: torch.Tensor):
        """PatchEmbed.forward: patchify (ug_pack_latents) -> conv-as-GEMM + bias + cropped sincos table (residual operand)."""
        B, C, H, W = latents.shape
        pat = ops.pack_latents(latents, out=buf.PAT)  # channel = c*4 + py*2 + px == the flattened Conv2d weight layout
        table = w.cropped(H // 2, W // 2)
        ops.gemm(pat, w.w, out=out, bias=w.b, residual=table.unsqueeze(0).expand(B, -1, -1), variant=self.gemm_variant)
        return out

    def _attn_qkv(self, x, q, aw_qkv, rms, qkv_rows):
        """q|k|v projection of one stream into its rows of a fused QKV buffer + in-place per-head RMSNorm (no RoPE). For an
        fp8 linear, q = (e4m3 rows, row scales) of x is the GEMM operand."""
        a = self.arch
        if rms is not None and self.fuse_qk_norm and x.dim() == 3 and aw_qkv[0].dim() == 2:
            # per-head RMSNorm of q / k inside the projection GEMM's epilogue (fp32 accumulator, no second pass over the buffer)
            self._linear(aw_qkv, x, q, out=qkv_rows,
                         qk_norm=dict(weight=rms, head_dim=a.attention_head_dim, d=self.inner_dim, cos_sin=None, eps=1e-6))
            return
        self._linear(aw_qkv, x, q, out=qkv_rows)
        if rms is not None:
            ops.qk_rmsnorm_rope(qkv_rows[:, :, :2 * self.inner_dim], 2 * a.num_attention_heads, a.attention_head_dim, rms, None,
                                heads_per_weight=a.num_attention_heads)

    def _joint_block(self, buf, w: _JointBlockW, mod_smp, mod_ctx, smp_in, ctx_in, smp_out, ctx_out):
        """JointTransformerBlock.forward (src/UniGenUtils.py:440-522) + JointAttnProcessor2_0 (sample-first joint attention).
        smp/ctx = sample / context streams ([B, n, D] views); outputs may alias inputs. ctx_out=None skips the context
        stream's post-attention half: exact for context_pre_only blocks and whenever the caller discards the context output
        (control blocks: `encoder_hidden_states` is re-read from moe_output every call, src/UniGenTransformer.py:566).
        An fp8 weight set (`w.fp8`, after quantize_fp8) runs its linears on e4m3 operands: every LayerNorm-modulate writes
        e4m3 rows + row scales directly, AO / AO2 / FF are quantised once per stream before their down-projection. The
        weight set decides, not a model flag: the bf16 shared experts of the pre-stage run through here unchanged."""
        a, D = self.arch, self.inner_dim
        H, dh = a.num_attention_heads, a.attention_head_dim
        B, n_smp, n_ctx = smp_in.shape[0], smp_in.shape[1], ctx_in.shape[1]
        S = n_smp + n_ctx
        qn_s = qn_c = qn2 = qa_s = qa_c = qf_s = qf_c = None
        if w.fp8:
            # Everything below runs on one stream, in program order, and the two streams own disjoint rows of every buffer.
            # Reuses: NXQ's sample / context rows take the second LN of their stream once q|k|v (their first consumer) has
            # run; AOQ's sample rows take AO2 once to_out has read AO; FFQ is written by the GEMM right before its only reader.
            qn_s, qn_c = (buf.NXQ[:, :n_smp], buf.NXS[:, :n_smp]), (buf.NXQ[:, n_smp:S], buf.NXS[:, n_smp:S])
            qn2 = (buf.NX2Q[:, :n_smp], buf.NX2S[:, :n_smp])
            qa_s, qa_c = (buf.AOQ[:, :n_smp], buf.AOS[:, :n_smp]), (buf.AOQ[:, n_smp:S], buf.AOS[:, n_smp:S])
            qf_s, qf_c = (buf.FFQ[:, :n_smp], buf.FFS[:, :n_smp]), (buf.FFQ[:, n_smp:S], buf.FFS[:, n_smp:S])
        if w.dual:
            sh_a, sc_a, g_a, sh_m, sc_m, g_m, sh_a2, sc_a2, g_a2 = mod_smp
        else:
            sh_a, sc_a, g_a, sh_m, sc_m, g_m = mod_smp
        if w.context_pre_only:
            csc_a, csh_a = mod_ctx  # AdaLayerNormContinuous: (scale, shift)
        else:
            csh_a, csc_a, cg_a, csh_m, csc_m, cg_m = mod_ctx
        nx_s, nx_c = buf.NX[:, :n_smp], buf.NX[:, n_smp:S]
        self._ln(w, smp_in, nx_s, qn_s, sh_a, sc_a)
        if w.dual:  # norm_hidden_states2 of the block INPUT (before any residual update, which may be in place)
            self._ln(w, smp_in, buf.NX2[:, :n_smp], qn2, sh_a2, sc_a2)
        self._ln(w, ctx_in, nx_c, qn_c, csh_a, csc_a)
        self._attn_qkv(nx_s, qn_s, w.attn.qkv, w.attn.rms, buf.QKV[:, :n_smp])
        self._attn_qkv(nx_c, qn_c, w.attn.add_qkv, w.attn.rms_ctx, buf.QKV[:, n_smp:S])
        ao = buf.AO[:, :S]
        ops.attention(buf.QKV[:, :S, 0:D], buf.QKV[:, :S, D:2 * D], buf.QKV[:, :S, 2 * D:3 * D], ao, H, dh, variant=self.attn_variant)
        self._linear(w.attn.to_out, ao[:, :n_smp], qa_s, out=smp_out, quantize=True, gate=g_a, residual=smp_in)
        if w.dual:
            self._attn_qkv(buf.NX2[:, :n_smp], qn2, w.attn2.qkv, w.attn2.rms, buf.QKV2[:, :n_smp])
            q2 = buf.QKV2[:, :n_smp]
            ops.attention(q2[:, :, 0:D], q2[:, :, D:2 * D], q2[:, :, 2 * D:3 * D], buf.AO2[:, :n_smp], H, dh, variant=self.attn_variant)
            self._linear(w.attn2.to_out, buf.AO2[:, :n_smp], qa_s, out=smp_out, quantize=True, gate=g_a2, residual=smp_out)
        self._ln(w, smp_out, nx_s, qn_s, sh_m, sc_m)
        self._linear(w.ff1, nx_s, qn_s, out=buf.FF[:, :n_smp], act=UG_ACT_GELU_TANH)
        self._linear(w.ff2, buf.FF[:, :n_smp], qf_s, out=smp_out, quantize=True, gate=g_m, residual=smp_out)
        if ctx_out is not None and not w.context_pre_only:
            self._linear(w.attn.to_add_out, ao[:, n_smp:S], qa_c, out=ctx_out, quantize=True, gate=cg_a, residual=ctx_in)
            self._ln(w, ctx_out, nx_c, qn_c, csh_m, csc_m)
            self._linear(w.ffc1, nx_c, qn_c, out=buf.FF[:, n_smp:S], act=UG_ACT_GELU_TANH)
            self._linear(w.ffc2, buf.FF[:, n_smp:S], qf_c, out=ctx_out, quantize=True, gate=cg_m, residual=ctx_out)

    def _expert_branch(self, buf, br: int, route, B: int, N: int):
        """All E experts of one branch: SD3SingleTransformerBlock (src/UniGenUtils.py:386-414) on the [E*C, D] slot buffer
        `buf.SL[br]` in place, per-token AdaLN through slot_token (reference expert_forward src/UniGenTransformer.py:256-258)."""
        a, D, E, C = self.arch, self.inner_dim, self.expert_nums, buf.capacity
        H, dh = a.num_attention_heads, a.attention_head_dim
        w, x, st = self.experts[br], buf.SL[br], route["slot_token"]
        gv = self.gemm_variant
        # AdaLN rows of every expert for the B sample tembs and the all-zero temb of empty slots: one stacked GEMV
        ops.gemv(buf.TE[br], w.norm1_w, w.norm1_b, out=buf.SMODT[br], silu_in=True)
        m = buf.SMODT[br].view(B + 1, E, 6, D).permute(1, 0, 2, 3)  # [E, B+1, 6, D] view of the [B+1, E*6D] GEMV output
        chunk = lambda i: m[:, :, i]  # noqa: E731  shift_msa, scale_msa, gate_msa, shift_mlp, scale_mlp, gate_mlp
        ops.ln_modulate_slots(x, buf.SNX, chunk(0), chunk(1), st, E, C, N, B)
        ops.gemm(buf.SNX.view(E, C, D), w.qkv_w, out=buf.SQKV.view(E, C, 3 * D), bias=w.qkv_b, variant=gv)
        q = buf.SQKV.view(E, C, 3 * D)
        ops.attention(q[:, :, 0:D], q[:, :, D:2 * D], q[:, :, 2 * D:3 * D], buf.SAO.view(E, C, D), H, dh, variant=self.attn_variant)
        ops.gemm(buf.SAO.view(E, C, D), w.out_w, out=buf.STMP.view(E, C, D), bias=w.out_b, variant=gv)
        ops.gated_add_slots(x, buf.STMP, chunk(2), st, E, C, N, B)
        ops.ln_modulate_slots(x, buf.SNX, chunk(3), chunk(4), st, E, C, N, B)
        ops.gemm(buf.SNX.view(E, C, D), w.ff1_w, out=buf.SFF.view(E, C, 4 * D), bias=w.ff1_b, act=UG_ACT_GELU_TANH, variant=gv)
        ops.gemm(buf.SFF.view(E, C, 4 * D), w.ff2_w, out=buf.STMP.view(E, C, D), bias=w.ff2_b, variant=gv)
        ops.gated_add_slots(x, buf.STMP, chunk(5), st, E, C, N, B)
        return x

    def _prestage(self, buf, B, N, T, x_img, x_txt, cond_latents, mods_s0, mods_s1, rts_uniform, pooled, cpooled):
        """preprocess_moe_forward (src/UniGenTransformer.py:498-540) + moe_forward (:264-296) + MOELayer.forward +
        expert_forward (:222-262): runs once per step after base block 0; leaves the control-stream input in buf.CIN."""
        D, E, C = self.inner_dim, self.expert_nums, buf.capacity
        gv = self.gemm_variant
        self._patch_embed(buf, self.control_pos_embed_input_w, cond_latents, buf.COND)
        ops.gemm(x_txt, self.control_context_embedder_w[0], out=buf.CENC, bias=self.control_context_embedder_w[1], variant=self.gemm_variant)
        self._rec("moe.cond_embed", buf.COND); self._rec("moe.enc_ctrl", buf.CENC)
        ops.add(x_img, buf.COND, buf.G.view(B, N, D))
        route = ops.moe_route(buf.G, self.gate_wg, rts_uniform, C)
        ops.copy(x_img, buf.EH.view(B, N, D))  # contiguous token-major copy of the (strided) image rows for the gather
        if self.use_modulate:
            # :252-255: cond' = Wc (s_c . cond) + bc ; hid' = Wh (s_h . (hid + cond')) + bh with s = Linear(pooled) per expert —
            # the row scale rides in the gather, the (C, D, D) modulated weights of `modulated_flatten` never exist
            ops.gemv(cpooled, self.exp_mod_w[0], self.exp_mod_b[0], out=buf.MODC.view(B, E * D))
            ops.gemv(pooled, self.exp_mod_w[1], self.exp_mod_b[1], out=buf.MODH.view(B, E * D))
            ops.moe_gather_modulate(buf.COND.view(B * N, D), route["slot_token"], buf.MODC, E, C, N, out=buf.SNX)
            ops.gemm(buf.SNX.view(E, C, D), self.exp_w[0], out=buf.SL[1].view(E, C, D), bias=self.exp_b[0], variant=gv)
            ops.moe_gather_modulate(buf.EH, route["slot_token"], buf.MODH, E, C, N, addend=buf.SL[1], out=buf.SNX)
            ops.gemm(buf.SNX.view(E, C, D), self.exp_w[1], out=buf.SL[0].view(E, C, D), bias=self.exp_b[1], variant=gv)
        else:
            ops.moe_gather_modulate(buf.EH, route["slot_token"], None, E, C, N, out=buf.SL[0])
            ops.moe_gather_modulate(buf.COND.view(B * N, D), route["slot_token"], None, E, C, N, out=buf.SL[1])
            self._expert_branch(buf, 0, route, B, N)  # expert[0](hidden_chunk, temb_chunk)            temb = control_temb
            self._expert_branch(buf, 1, route, B, N)  # expert[1](condition_chunk, condition_temb_chunk)
        hc_h, hc_c = buf.HC[:, :N], buf.HC[:, N:]
        if self.use_shared_expert:
            # shared experts (:281-294): [0] sample = hidden, context = condition, temb = condition_temb
            self._joint_block(buf, self.shared[0], mods_s0[0], mods_s0[1], x_img, buf.COND, hc_h, hc_c)
            #                   [1] sample = [hidden | condition], context = control text, temb = control_temb, context_pre_only
            self._joint_block(buf, self.shared[1], mods_s1[0], mods_s1[1], buf.HC, buf.CENC, buf.HC, None)
        ops.moe_combine(buf.SL[0], route, C, buf.EH)
        ops.moe_combine(buf.SL[1], route, C, buf.EC)
        self._rec("moe.expert_hidden", buf.EH.view(B, N, D)); self._rec("moe.expert_cond", buf.EC.view(B, N, D))
        if not self.use_shared_expert:  # :279 skipped: control stream := expert_hidden + expert_cond (:561)
            ops.add(buf.EH.view(B, N, D), buf.EC.view(B, N, D), buf.CIN)
            self._rec("moe.ctrl_in", buf.CIN)
            return route
        self._rec("moe.shared_hidden", hc_h); self._rec("moe.shared_cond", hc_c)
        # control stream := (shared_hidden + expert_hidden) + (shared_cond + expert_cond)   (:294, :561)
        ops.add(hc_h, buf.EH.view(B, N, D), buf.CIN)
        ops.add(buf.CIN, hc_c, buf.CIN)
        ops.add(buf.CIN, buf.EC.view(B, N, D), buf.CIN)
        self._rec("moe.ctrl_in", buf.CIN)
        return route

    # ---------------------------------------------------------------------------------------------------------
    # forward (reference :625-710 + base_forward :583-623 + control_forward :542-581)
    # ---------------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, hidden_states, condition_hidden_states=None, conditioning_scale: float = 1.0, encoder_hidden_states=None,
                pooled_projections=None, condition_pooled_projections=None, timestep=None, joint_attention_kwargs=None,
                skip_layers=None, rts_uniform=None, **kwargs):
        """Reference signature (src/UniGenTransformer.py:625-637). hidden_states / condition_hidden_states are LATENTS
        (B, C, H, W); `timestep` is the raw scheduler timestep (0-1000, src/UniGenPipeline.py:382,396).
        `joint_attention_kwargs['scale']` (PEFT LoRA scale) is accepted and ignored (no adapter on the S-variant path)."""
        if not self._control_ready:
            raise ops.UgError("call init_condition_block(condition_nums=..., control_params=...) before forward")
        if encoder_hidden_states is None or condition_hidden_states is None or timestep is None or pooled_projections is None:
            raise ops.UgError("forward needs hidden_states, condition_hidden_states, encoder_hidden_states, pooled_projections and timestep")
        if joint_attention_kwargs and "ip_adapter_image_embeds" in joint_attention_kwargs:
            raise ops.UgError("ip_adapter_image_embeds is not covered by the B200-native path")
        a = self.arch
        B, Cc, Hh, Ww = hidden_states.shape
        if tuple(condition_hidden_states.shape) != (B, Cc, Hh, Ww):
            raise ops.UgError("condition latents must have the image latents' shape (Nc == N for the CoMoE pre-stage)")
        N, T = (Hh // a.patch_size) * (Ww // a.patch_size), encoder_hidden_states.shape[1]
        if T == N:
            raise ops.UgError("T == N: the reference MOELayer would also dispatch the text tensor (SURVEY.md §8 A9); unsupported")
        dev = self.device_
        f32 = lambda t: t.to(device=dev, dtype=torch.float32).contiguous()  # noqa: E731
        if rts_uniform is None:
            rts_uniform = torch.rand(B * N, self.expert_nums, device=dev, dtype=torch.float32)
        staged = dict(hs=hidden_states.to(dev), cs=condition_hidden_states.to(dev), es=encoder_hidden_states.to(dev),
                      pooled=f32(pooled_projections), cpooled=f32(condition_pooled_projections),
                      timestep=f32(timestep).reshape(-1).expand(B).contiguous(), u=f32(rts_uniform))
        key = (B, Hh, Ww, T, float(conditioning_scale), tuple((k, v.dtype) for k, v in staged.items()))
        out, add_losses, add_outputs = self._run_staged(key, staged, float(conditioning_scale))
        if self.clone_outputs:  # under graph replay `out` is the graph's static output: hand out a copy (see UniGenFlux.forward)
            cp = torch.empty(out.shape, device=out.device, dtype=out.dtype)
            ops.copy(out.view(B, 1, -1), cp.view(B, 1, -1))
            out = cp
            add_losses = {k: v.clone() for k, v in add_losses.items()}
            add_outputs = {k: v.clone() for k, v in add_outputs.items()}
        return out, add_losses, add_outputs

    def _forward_impl(self, conditioning_scale, hs, cs, es, pooled, cpooled, timestep, u):
        a, D = self.arch, self.inner_dim
        B, Cc, Hh, Ww = hs.shape
        hp, wp = Hh // a.patch_size, Ww // a.patch_size
        N, T = hp * wp, es.shape[1]
        buf = self._workspace(B, N, T)
        n0 = ops.launch_count()
        hs, cs, es = ops.to_bf16(hs.contiguous()), ops.to_bf16(cs.contiguous()), ops.to_bf16(es.contiguous())
        gv = self.gemm_variant
        x_img, x_txt = buf.X[:, :N], buf.X[:, N:]

        # ---- embeddings (:663-666) ----
        self._patch_embed(buf, self.pos_embed_w, hs, x_img)
        ops.gemm(es, self.context_embedder_w[0], out=x_txt, bias=self.context_embedder_w[1], variant=gv)
        t_emb = ops.timestep_embedding(timestep, batch=B)  # raw timestep: the SD3 forward does not rescale it (1-element view: broadcast)
        self._time_text(self.time_text, t_emb, pooled, buf.temb, buf.tmp)
        ctrl_pooled = pooled if self.use_pooled_prompt_embeds else torch.zeros_like(pooled)
        control_temb, condition_temb = buf.TE[0][:B], buf.TE[1][:B]  # row B of TE stays 0: the temb of an empty slot
        self._time_text(self.control_time_text, t_emb, ctrl_pooled, control_temb, buf.tmp)
        self._time_text(self.control_condition, t_emb, cpooled, condition_temb, buf.tmp)
        self._rec("temb", buf.temb); self._rec("x_embed", x_img); self._rec("context_embed", x_txt)

        # ---- AdaLN vectors of every block, once per step: two grouped-GEMV launches (device-resident job tables) — the first
        # block pair + pre-stage on the main stream, everything else on a side stream under the tensor-core-bound blocks ----
        mp = self._sd3_mod_plans(buf, B)
        m_base, m_ctrl, mods_s0, mods_s1, m_out = mp.m_base, mp.m_ctrl, mp.mods_s0, mp.mods_s1, mp.m_out
        ops.gemv_grouped(mp.early)
        main_stream = torch.cuda.current_stream()
        side = self._side_stream if self.overlap_mod_gemv else None
        if side is not None:
            side.wait_stream(main_stream)
        with torch.cuda.stream(side if side is not None else main_stream):
            ops.gemv_grouped(mp.late)
        joined = side is None

        # ---- 24 x [base MMDiT block -> control block -> zero-linear add] (:583-623) ----
        route = None
        n_base, n_ctrl = len(self.blocks), len(self.ctrl_blocks)
        for i, w in enumerate(self.blocks):
            if i == 1 and not joined:
                main_stream.wait_stream(side)
                joined = True
            self._joint_block(buf, w, m_base[i][0], m_base[i][1], x_img, x_txt, x_img, None if w.context_pre_only else x_txt)
            self._rec(f"block.{i}.base_hidden", x_img)
            j = int(i / (n_base / n_ctrl))
            if i == 0:   # first control call: CoMoE pre-stage on (hidden after block 0, base text after block 0) (:558-562)
                route = self._prestage(buf, B, N, T, x_img, x_txt, cs, mods_s0, mods_s1, u, pooled, cpooled)
                ctrl_in = buf.CIN
            else:
                ctrl_in = x_img
            wc = self.ctrl_blocks[j]
            self._joint_block(buf, wc, m_ctrl[j][0], m_ctrl[j][1], ctrl_in, buf.CENC, buf.CH, None)
            wa = self.add_blocks[j]
            ops.gemm(buf.CH, wa[0], out=x_img, bias=wa[1], alpha=float(conditioning_scale), residual=x_img, variant=gv)
            self._rec(f"block.{i}.ctrl_hidden", buf.CH); self._rec(f"block.{i}.hidden", x_img)
        if not joined:
            main_stream.wait_stream(side)

        # ---- norm_out + proj_out + un-patchify (:682-704) ----
        ops.ln_modulate(x_img, buf.NO, m_out[1], m_out[0])
        ops.gemm(buf.NO, self.proj_out_w[0], out=buf.OUT, bias=self.proj_out_w[1], variant=gv)
        self._rec("proj_out", buf.OUT)
        out = ops.unpatchify(buf.OUT, hp, wp, a.patch_size, a.out_channels)
        self._rec("velocity", out)
        self._last_route = route
        ops.note_capture_launches(ops.launch_count() - n0)
        return out, dict(moe_loss=route["l_aux"][0] * 0.1), dict(expert_counts=route["exp_counts"])


def shipped_control_params() -> Dict[str, Any]:
    """config/unigen.yaml:3-11 as shipped (the SD3 path runs with it unchanged)."""
    return dict(use_transformer_params=True, use_pooled_prompt_embeds=True, use_encoder_hidden_states=True,
                extra_conditioning_channels=0, expert_num_each_condition=3, use_shared_expert=True, use_consis_module=False,
                use_modulate=False)
