"""Host-side mirror of the reference's denoiser interface for the B200-native path.

`UniGenFlux` here keeps the reference's public surface — `init_condition_block(...)`, `forward(hidden_states,
condition_hidden_states, conditioning_scale, encoder_hidden_states, pooled_projections, condition_pooled_projections,
timestep, img_ids, txt_ids, guidance, condition_ids, joint_attention_kwargs, ...) -> (velocity, add_losses,
add_outputs)` (reference src/UniGenTransformer.py:712-716,1182-1271), `state_dict()/load_state_dict()` under the
reference's key names, `.config`, `.dtype`, `.trainable_control_modules` — while every arithmetic op of the step
runs in libunigen_b200.so (unigen_b200.ops).  torch supplies device memory, the stream and (optionally) CUDA-graph
capture; there is no eager/CPU fallback.

Data layout in HBM (bf16 unless noted)
  X    [B, T+N, D]   joint residual stream, TEXT ROWS FIRST — the `cat([text, image])` of base_forward (:1146) is free
  NX   [B, Smax, D]  LN+modulated operand, QKV [B, Smax, 3D] fused q|k|v, AO attention out, FF [B, Smax, 4D]
  CAT  [B, S, 5D]    single blocks: attention writes cols [0,D), GELU(proj_mlp) writes [D,5D) — `cat([attn, mlp])` is free
  MOD  fp32          AdaLN shift/scale/gate vectors of ALL blocks, computed once per step (temb is step-constant)
  weights            fused per block (to_q|to_k|to_v -> one [3D, D] matrix, experts stacked [E, D, D]); the reference's
                     parameter names are VIEWS into the fused storage, so state dicts load in place without copies.
"""
from __future__ import annotations

import collections
import math
import types
from typing import Any, Dict, List, Optional, Sequence, Tuple

import torch

from . import ops
from .ops import UG_ACT_GELU_TANH

BF16 = torch.bfloat16
FP8 = torch.float8_e4m3fn


class FluxArch:
    """diffusers FluxTransformer2DModel config fields read on the path + UniGen control_params (SURVEY.md §A.1)."""

    def __init__(self, num_layers=19, num_single_layers=38, attention_head_dim=128, num_attention_heads=24, in_channels=64,
                 joint_attention_dim=4096, pooled_projection_dim=768, guidance_embeds=False, axes_dims_rope=(16, 56, 56),
                 theta=10000.0):
        self.num_layers, self.num_single_layers = num_layers, num_single_layers
        self.attention_head_dim, self.num_attention_heads = attention_head_dim, num_attention_heads
        self.in_channels, self.joint_attention_dim = in_channels, joint_attention_dim
        self.pooled_projection_dim, self.guidance_embeds = pooled_projection_dim, guidance_embeds
        self.axes_dims_rope, self.theta = tuple(axes_dims_rope), theta
        self.hidden_size = num_layers and num_attention_heads * attention_head_dim

    @staticmethod
    def tiny():
        return FluxArch(num_layers=2, num_single_layers=4, attention_head_dim=64, num_attention_heads=6, axes_dims_rope=(8, 28, 28))


class _Weights:
    """Fused device storage + reference-name views."""

    def __init__(self, device):
        self.device = device
        self.views: Dict[str, torch.Tensor] = {}

    def alloc(self, *shape, dtype=BF16) -> torch.Tensor:
        return torch.zeros(*shape, device=self.device, dtype=dtype)

    def linear(self, name: str, out_f: int, in_f: int, w: Optional[torch.Tensor] = None, b: Optional[torch.Tensor] = None):
        w = self.alloc(out_f, in_f) if w is None else w
        b = self.alloc(out_f) if b is None else b
        self.views[name + ".weight"], self.views[name + ".bias"] = w, b
        return w, b

    def fused(self, names: Sequence[str], out_each: int, in_f: int):
        """One [len(names)*out_each, in_f] matrix (+ bias); names[i] is a row-slice view."""
        W, Bv = self.alloc(len(names) * out_each, in_f), self.alloc(len(names) * out_each)
        for i, n in enumerate(names):
            self.views[n + ".weight"] = W[i * out_each:(i + 1) * out_each]
            self.views[n + ".bias"] = Bv[i * out_each:(i + 1) * out_each]
        return W, Bv


class _DoubleBlockW:
    # linears `UniGenFlux.quantize_fp8()` / `UniCombineFlux.quantize_fp8()` convert; once they have, `fp8` is True and each of them is (W e4m3 [N, K], bias bf16 [N],
    # w_scale fp32 [N]) instead of (W bf16, bias)
    FP8_LINEARS = ("qkv", "add_qkv", "to_out", "to_add_out", "ff1", "ff2", "ffc1", "ffc2")
    fp8 = False

    def __init__(self, ws: _Weights, p: str, D: int, dh: int):
        self.norm1 = ws.linear(p + ".norm1.linear", 6 * D, D)
        self.norm1_ctx = ws.linear(p + ".norm1_context.linear", 6 * D, D)
        self.qkv = ws.fused([f"{p}.attn.to_q", f"{p}.attn.to_k", f"{p}.attn.to_v"], D, D)
        self.add_qkv = ws.fused([f"{p}.attn.add_q_proj", f"{p}.attn.add_k_proj", f"{p}.attn.add_v_proj"], D, D)
        self.to_out = ws.linear(p + ".attn.to_out.0", D, D)
        self.to_add_out = ws.linear(p + ".attn.to_add_out", D, D)
        self.rms = ws.alloc(2, dh)       # [norm_q; norm_k]
        self.rms_ctx = ws.alloc(2, dh)   # [norm_added_q; norm_added_k]
        ws.views[p + ".attn.norm_q.weight"], ws.views[p + ".attn.norm_k.weight"] = self.rms[0], self.rms[1]
        ws.views[p + ".attn.norm_added_q.weight"], ws.views[p + ".attn.norm_added_k.weight"] = self.rms_ctx[0], self.rms_ctx[1]
        self.ff1 = ws.linear(p + ".ff.net.0.proj", 4 * D, D)
        self.ff2 = ws.linear(p + ".ff.net.2", D, 4 * D)
        self.ffc1 = ws.linear(p + ".ff_context.net.0.proj", 4 * D, D)
        self.ffc2 = ws.linear(p + ".ff_context.net.2", D, 4 * D)


class _SingleBlockW:
    FP8_LINEARS = ("qkv", "mlp", "out")
    fp8 = False

    def __init__(self, ws: _Weights, p: str, D: int, dh: int):
        self.norm = ws.linear(p + ".norm.linear", 3 * D, D)
        self.qkv = ws.fused([f"{p}.attn.to_q", f"{p}.attn.to_k", f"{p}.attn.to_v"], D, D)
        self.mlp = ws.linear(p + ".proj_mlp", 4 * D, D)
        self.out = ws.linear(p + ".proj_out", D, 5 * D)
        self.rms = ws.alloc(2, dh)
        ws.views[p + ".attn.norm_q.weight"], ws.views[p + ".attn.norm_k.weight"] = self.rms[0], self.rms[1]


def quantize_block_linears(ws: _Weights, blocks) -> None:
    """Every linear named in a block's FP8_LINEARS becomes (W e4m3 [N, K], bias bf16 [N], w_scale fp32 [N]), one scale per output
    channel; the bf16 weight is released and its state-dict views are dropped (the bias stays). Marks the blocks `fp8`.
    A dotted name reaches a linear of a sub-object (`attn.qkv`); a linear or sub-object that is None (absent in this block
    layout, e.g. `to_add_out` of a context_pre_only block) is skipped."""
    views = ws.views
    for w in blocks:
        for name in w.FP8_LINEARS:
            *path, attr = name.split(".")
            owner = w
            for p in path:
                owner = getattr(owner, p) if owner is not None else None
            lin = getattr(owner, attr) if owner is not None else None
            if lin is None:
                continue
            W, bias = lin
            q, w_scale = ops.quant_rows_fp8(W)  # a row of W is an output channel
            ptr = W.untyped_storage().data_ptr()
            for k in [k for k, v in views.items() if k.endswith(".weight") and v.untyped_storage().data_ptr() == ptr]:
                del views[k]
            setattr(owner, attr, (q, bias, w_scale))
        w.fp8 = True


class _TimeTextW:
    def __init__(self, ws: _Weights, p: str, D: int, pooled: int, guidance: bool):
        self.t1 = ws.linear(p + ".timestep_embedder.linear_1", D, 256)
        self.t2 = ws.linear(p + ".timestep_embedder.linear_2", D, D)
        self.g1 = ws.linear(p + ".guidance_embedder.linear_1", D, 256) if guidance else None
        self.g2 = ws.linear(p + ".guidance_embedder.linear_2", D, D) if guidance else None
        self.p1 = ws.linear(p + ".text_embedder.linear_1", D, pooled)
        self.p2 = ws.linear(p + ".text_embedder.linear_2", D, D)


class _DenoiserBase(torch.nn.Module):
    """What the Flux (`UniGenFlux`) and SD3.5 (`UniGenSD3`, sd3.py) mirrors share: fused weight storage under the
    reference's state-dict names, the per-step AdaLN / time-text GEMV helpers, tracing and CUDA-graph replay."""

    def _init_base(self, device):
        self.device_ = torch.device(device)
        if self.device_.type != "cuda":
            raise ops.UgError(f"{type(self).__name__} (B200-native) needs a CUDA device: the hot path has no CPU fallback")
        self._ws = _Weights(self.device_)
        self._control_ready = False
        # one workspace per input shape, kept alive as long as a CUDA graph captured over it may be replayed (a graph holds
        # raw pointers into X / QKV / AO / ...): least-recently-used shapes are evicted TOGETHER with their graphs
        self._workspaces: "collections.OrderedDict[Any, Any]" = collections.OrderedDict()
        self.max_workspaces = 4
        self._buf = None
        self._graphs: Dict[Any, Any] = {}
        self.use_cuda_graph = False
        self.gemm_variant = 0
        self.attn_variant = 0
        self.overlap_mod_gemv = True  # AdaLN GEMVs (HBM-bound) on a side stream under the tensor-core-bound blocks
        self._side_stream = torch.cuda.Stream(device=self.device_)
        self.overlap_text_stream = True  # text-stream GEMMs of the double blocks on a second stream beside the image stream's
        self._text_stream = torch.cuda.Stream(device=self.device_)
        # QK-RMSNorm + RoPE inside the q|k|v projection GEMM's (staged) epilogue — north_star "fused into the Q/K load" — instead
        # of a separate in-place pass over the QKV buffer (-1.1 % per cfg3 step, same-box A/B in profiles/r02_ab_fuse_qk_norm.txt)
        self.fuse_qk_norm = True
        self.trace: Optional[Dict[str, torch.Tensor]] = None  # set to {} to record per-block intermediates
        self.clone_outputs = True  # forward returns copies, not views of the workspace / graph-static buffers
        self.linear_dtype = BF16  # float8_e4m3fn after quantize_fp8()

    @property
    def dtype(self):
        return BF16

    @property
    def device(self):
        return self.device_

    def state_dict(self, *args, **kwargs):  # reference key names, views into the fused storage
        return dict(self._ws.views)

    def parameters(self, recurse: bool = True):
        return iter(self._ws.views.values())

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        if self.linear_dtype != BF16:
            raise ops.UgError("load_state_dict on an fp8-quantised model: its block linears no longer hold bf16 weights — load the "
                              "checkpoint into a fresh model, then call quantize_fp8()")
        missing = [k for k in self._ws.views if k not in state_dict]
        unexpected = [k for k in state_dict if k not in self._ws.views]
        if strict and (missing or unexpected):
            raise RuntimeError(f"load_state_dict: missing {missing[:5]}... unexpected {unexpected[:5]}...")
        with torch.no_grad():
            for k, v in state_dict.items():
                if k in self._ws.views:
                    dst = self._ws.views[k]
                    if tuple(dst.shape) != tuple(v.shape):
                        raise RuntimeError(f"size mismatch for {k}: {tuple(v.shape)} vs {tuple(dst.shape)}")
                    dst.copy_(v.to(device=dst.device, dtype=dst.dtype))
        self._weights_loaded()
        return types.SimpleNamespace(missing_keys=missing, unexpected_keys=unexpected)

    def _weights_loaded(self):
        """Hook: derived (non-state-dict) device tensors are rebuilt after a load / random init."""

    @torch.no_grad()
    def init_random_(self, seed: int = 0, zero_linear_std: Optional[float] = 0.02):
        """nn.Linear / nn.Conv2d default init directly on the device (bench: the 18.7 B Flux parameters never exist on
        the host). Zero-linears (`controlnet_add_*`) get N(0, zero_linear_std), or true zeros for None."""
        if self.linear_dtype != BF16:
            raise ops.UgError("init_random_ on an fp8-quantised model: its quantised block weights are not in state_dict() any more "
                              "and would keep their values — initialise a fresh model, then call quantize_fp8()")
        gen = torch.Generator(device=self.device_).manual_seed(seed)
        for k, v in self._ws.views.items():
            if k.endswith(".pos_embed"):
                continue  # PatchEmbed's sincos buffer: a constant of the architecture, filled at construction
            if k.startswith("controlnet_add_"):
                if zero_linear_std is None:
                    v.zero_()
                else:
                    v.copy_(torch.randn(v.shape, device=v.device, generator=gen) * zero_linear_std)
            elif ".norm_q." in k or ".norm_k." in k or ".norm_added_" in k:
                v.fill_(1.0)
            else:
                w = self._ws.views[k[:-4] + "weight"] if k.endswith(".bias") else v
                bound = 1.0 / math.sqrt(w[0].numel())  # fan_in (Linear: in_features; Conv2d: C * kh * kw)
                v.copy_((torch.rand(v.shape, device=v.device, generator=gen) * 2 - 1) * bound)
        self._weights_loaded()
        return self

    def _time_text(self, w: "_TimeTextW", t_emb: torch.Tensor, pooled: torch.Tensor, out: torch.Tensor, tmp: torch.Tensor,
                   g_emb: Optional[torch.Tensor] = None, accumulate: bool = False):
        """CombinedTimestep(Guidance)TextProjEmbeddings (SURVEY.md §A.4); accumulate=True adds into `out`
        (merged_condition_temb = sum over conditions, reference :1314,1319)."""
        ops.gemv(t_emb, w.t1[0], w.t1[1], out=tmp, silu_out=True)
        ops.gemv(tmp, w.t2[0], w.t2[1], out=out, accumulate=accumulate)
        if g_emb is not None and w.g1 is not None:
            ops.gemv(g_emb, w.g1[0], w.g1[1], out=tmp, silu_out=True)
            ops.gemv(tmp, w.g2[0], w.g2[1], out=out, accumulate=True)
        ops.gemv(pooled, w.p1[0], w.p1[1], out=tmp, silu_out=True)
        ops.gemv(tmp, w.p2[0], w.p2[1], out=out, accumulate=True)
        return out

    def _mods(self, buf, slot: int, n_chunks: int, w, temb: torch.Tensor) -> List[torch.Tensor]:
        """AdaLN parameter vectors `linear(silu(temb)).chunk(n)`: fp32 [B, D] views into MOD."""
        D = self.inner_dim
        region = buf.MOD[:, slot * D:(slot + n_chunks) * D]
        ops.gemv(temb, w[0], w[1], out=region, silu_in=True)
        return [region[:, i * D:(i + 1) * D] for i in range(n_chunks)]

    def _rec(self, name: str, t: torch.Tensor):
        if self.trace is not None:
            self.trace[name] = t.detach().float().clone()

    def _fp8_blocks(self) -> list:
        """The blocks whose FP8_LINEARS `quantize_fp8()` converts (the model's base and control transformer blocks)."""
        raise NotImplementedError

    @torch.no_grad()
    def _quantize_fp8(self):
        """What every model's `quantize_fp8()` does: quantise the linears of `_fp8_blocks()` in place (once), then drop the
        workspaces and every CUDA graph captured over them — the pipeline's whole-loop graphs included — since they hold bf16
        operands only and point at the released weights."""
        if not self._control_ready:
            raise ops.UgError("call init_condition_block(condition_nums=..., control_params=...) before quantize_fp8()")
        if self.linear_dtype == FP8:
            return self
        quantize_block_linears(self._ws, self._fp8_blocks())
        self.linear_dtype = FP8
        from .pipeline import _GRAPHS_ATTR
        self.__dict__.pop(_GRAPHS_ATTR, None)
        self._workspaces.clear()
        self._graphs.clear()
        self._buf = None
        return self

    def _ln(self, w, x, nx, q, shift, scale):
        """LN + modulate of a block input into the bf16 operand `nx`, or (fp8 weight set) straight into q = (e4m3, row scales)."""
        if w.fp8:
            ops.ln_modulate_fp8(x, q[0], q[1], shift, scale)
        else:
            ops.ln_modulate(x, nx, shift, scale)

    def _linear(self, wl, x, q, out, quantize: bool = False, **epi):
        """One block linear: the bf16 GEMM of x with (W, bias), or for an fp8 (W e4m3, bias, w_scale) the fp8 GEMM of
        q = (e4m3 rows, row scales) — quantised from x first when `quantize` (operands no LN kernel produced)."""
        if len(wl) == 3:
            if quantize:
                ops.quant_rows_fp8(x, q[0], q[1])
            return ops.gemm_fp8(q[0], q[1], wl[0], wl[2], out=out, bias=wl[1], variant=self.gemm_variant, **epi)
        return ops.gemm(x, wl[0], out=out, bias=wl[1], variant=self.gemm_variant, **epi)

    def _cached_workspace(self, key, make):
        """Workspace for input shape `key` (built by `make()` on first use). Buffers of a shape stay where they are for as
        long as the shape is cached, so a graph captured over them stays valid when other shapes run in between; when the
        least-recently-used shape is evicted, the graphs captured over its buffers are dropped with it."""
        ws = self._workspaces
        b = ws.get(key)
        if b is None:
            while len(ws) >= max(int(self.max_workspaces), 1):
                _, old = ws.popitem(last=False)
                self._drop_graphs(old)
            b = ws[key] = make()
        else:
            ws.move_to_end(key)
            self._trim_workspaces()
        self._buf = b
        return b

    def _trim_workspaces(self):
        """Enforce `max_workspaces` (it may have been lowered): least recently used shapes go first, with their graphs."""
        ws = self._workspaces
        while len(ws) > max(int(self.max_workspaces), 1):
            _, old = ws.popitem(last=False)
            self._drop_graphs(old)

    def _drop_graphs(self, buf=None):
        """Forget the CUDA graphs captured over workspace `buf` (all graphs for None)."""
        if buf is None:
            self._graphs.clear()
            return
        for k in [k for k, g in self._graphs.items() if g[4] is buf]:
            del self._graphs[k]

    def _run_staged(self, key, staged: Dict[str, Optional[torch.Tensor]], *args):
        """`self._forward_impl(*args, **staged)`, eagerly or as a replay of a CUDA graph captured over static copies of
        the staged inputs (one graph per `key`). The graph record keeps the workspace it was captured over."""
        if not self.use_cuda_graph or self.trace is not None:
            return self._forward_impl(*args, **staged)
        g = self._graphs.get(key)
        if g is not None and not any(g[4] is b for b in self._workspaces.values()):
            del self._graphs[key]  # its workspace was evicted
            g = None
        if g is None:
            static = {k: (v.clone() if v is not None else None) for k, v in staged.items()}
            self._forward_impl(*args, **static)  # warm-up: attribute setup, workspace allocation
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out = self._forward_impl(*args, **static)
            g = self._graphs[key] = (graph, static, out, ops.launch_count_in_last_capture(), self._buf)
        graph, static, out, n_launch, buf = g
        ws_key = next(k for k, b in self._workspaces.items() if b is buf)
        self._workspaces.move_to_end(ws_key)
        self._trim_workspaces()
        self._buf = buf
        for k, v in staged.items():
            if v is not None:
                static[k].copy_(v)
        graph.replay()
        ops.add_launches(n_launch)
        return out


class UniGenFlux(_DenoiserBase):
    """B200-native drop-in for the reference `UniGenFlux` (Flux-arch denoiser + WeaveNet control branch + CoMoE)."""

    def __init__(self, arch: Optional[FluxArch] = None, device: Any = "cuda", **config):
        super().__init__()
        self.arch = arch or FluxArch(**config)
        self._init_base(device)
        a = self.arch
        self.config = types.SimpleNamespace(in_channels=a.in_channels, guidance_embeds=a.guidance_embeds,
                                            num_attention_heads=a.num_attention_heads, attention_head_dim=a.attention_head_dim,
                                            pooled_projection_dim=a.pooled_projection_dim, joint_attention_dim=a.joint_attention_dim,
                                            axes_dims_rope=a.axes_dims_rope, num_layers=a.num_layers,
                                            num_single_layers=a.num_single_layers)
        self.inner_dim = a.num_attention_heads * a.attention_head_dim
        D, dh = self.inner_dim, a.attention_head_dim
        ws = self._ws
        self.x_embedder_w = ws.linear("x_embedder", D, a.in_channels)
        self.context_embedder_w = ws.linear("context_embedder", D, a.joint_attention_dim)
        self.time_text = _TimeTextW(ws, "time_text_embed", D, a.pooled_projection_dim, a.guidance_embeds)
        self.double = [_DoubleBlockW(ws, f"transformer_blocks.{i}", D, dh) for i in range(a.num_layers)]
        self.single = [_SingleBlockW(ws, f"single_transformer_blocks.{i}", D, dh) for i in range(a.num_single_layers)]
        self.norm_out_w = ws.linear("norm_out.linear", 2 * D, D)
        # proj_out has only in_channels (64) output features: keep it as is, the GEMM masks the partial N tile
        self.proj_out_w = ws.linear("proj_out", a.in_channels, D)

    # ---------------------------------------------------------------------------------------------------------
    # reference API: construction
    # ---------------------------------------------------------------------------------------------------------
    _CONFIG_FIELDS = ("num_layers", "num_single_layers", "attention_head_dim", "num_attention_heads", "in_channels",
                      "joint_attention_dim", "pooled_projection_dim", "guidance_embeds", "axes_dims_rope")

    @classmethod
    def from_pretrained(cls, pretrained_model_name_or_path: str, subfolder: Optional[str] = None, torch_dtype=None,
                        device: Any = "cuda", revision: Optional[str] = None, variant: Optional[str] = None,
                        trust_pickle: bool = False, **kwargs):
        """`getattr(UniGenTransformer, basemodel).from_pretrained(f"{path}/transformer", revision=, variant=)` (infer.py:115-119,
        diffusers ModelMixin.from_pretrained): reads `config.json` (FluxTransformer2DModel fields) and the base weights
        (`diffusion_pytorch_model*.safetensors`, sharded or not) of a LOCAL diffusers transformer folder and returns the model
        with the base weights resident on `device`. The control branch is added afterwards by `init_condition_block(...)` and
        loaded with `load_state_dict(..., strict=False)`, exactly like the reference (infer.py:121-141). No hub download:
        `pretrained_model_name_or_path` must be a directory (this process has no network by design)."""
        import json
        import os
        from . import checkpoint
        path = os.path.join(pretrained_model_name_or_path, subfolder) if subfolder else pretrained_model_name_or_path
        cfg_file = os.path.join(path, "config.json")
        if not os.path.isfile(cfg_file):
            raise OSError(f"{path} does not contain config.json: from_pretrained needs a local diffusers transformer folder")
        with open(cfg_file) as f:
            cfg = json.load(f)
        if torch_dtype not in (None, BF16):
            import warnings
            warnings.warn(f"torch_dtype={torch_dtype}: the B200-native path stores weights and activations in bf16 (fp32 accumulate)")
        fields = {k: cfg[k] for k in cls._CONFIG_FIELDS if k in cfg}
        fields.update({k: v for k, v in kwargs.items() if k in cls._CONFIG_FIELDS})
        model = cls(FluxArch(**fields), device=device)
        sd = checkpoint.read_state_dict(path, trust_pickle=trust_pickle, variant=variant)
        own = model._ws.views
        missing = [k for k in own if k not in sd]
        if missing:
            raise RuntimeError(f"{path} lacks {len(missing)} base-model keys, e.g. {missing[:4]}")
        model.load_state_dict({k: v for k, v in sd.items() if k in own}, strict=False)
        model.name_or_path = pretrained_model_name_or_path
        return model

    def to(self, *args, **kwargs):
        """`transformer.to(accelerator.device, dtype=weight_dtype)` (infer.py:119): the weights already live on the CUDA device
        the model was built on, in bf16. Another CUDA device / a CPU target is an error (no fallback), a dtype is a no-op."""
        for a in list(args) + [kwargs.get("device")]:
            if isinstance(a, (str, torch.device)) and a is not None:
                d = torch.device(a)
                if d.type != "cuda" or (d.index is not None and d.index != (self.device_.index or 0)):
                    raise ops.UgError(f"the B200-native model lives on {self.device_}; moving it to {d} is not supported")
        return self

    def requires_grad_(self, requires_grad: bool = True):  # infer.py:143 `transformer.requires_grad_(False)`: inference-only path
        if requires_grad:
            raise ops.UgError("the B200-native path is forward-only (SURVEY.md §3.2: training is out of scope)")
        return self

    def quantize_fp8(self):
        """Opt-in fp8 (e4m3) transformer-block linears, in place; returns self. Every linear of the base and control double
        blocks (q|k|v, add_q|k|v, to_out, to_add_out, ff, ff_context) and single blocks (q|k|v, proj_mlp, proj_out) gets one fp32
        scale per output channel and is stored as e4m3; its bf16 copy is released (and leaves `state_dict()`). In every forward
        their operands are quantised per token row on the device and the GEMMs run on the fp8 tensor cores. Embedders, the
        CoMoE pre-stage (its expert, shared-expert and consistency blocks: routing stays bit-exact), the AdaLN GEMVs, the control
        add-linears, proj_out and attention stay bf16. Call after `from_pretrained` / `init_condition_block` and any
        `load_state_dict`. Afterwards `state_dict()` / `parameters()` no longer list the quantised weights (their biases and every
        bf16 tensor stay), and `load_state_dict` / `init_random_` raise `UgError`."""
        return self._quantize_fp8()

    def _fp8_blocks(self):
        return self.double + self.ctrl_double + self.single + self.ctrl_single

    def init_condition_block(self, condition_nums: int = 1, **kwargs):
        """reference src/UniGenTransformer.py:713-715 -> init_control_block(kwargs['control_params'])."""
        self.condition_nums = condition_nums
        self.init_control_block(kwargs.get("control_params", None))

    def init_control_block(self, control_params=None):
        """reference :717-783 (+ init_moe_block :806-923) for the canonical configuration (SURVEY.md §A.1)."""
        assert control_params is not None, ValueError("Please provice control net model parameter")
        get = control_params.get
        a, ws, D, dh = self.arch, self._ws, self.inner_dim, self.arch.attention_head_dim
        self.use_pooled_prompt_embeds = get("use_pooled_prompt_embeds", True)
        self.use_rope = get("use_rope", False)
        self.use_modulate = get("use_modulate", False)
        if not (self.use_rope or self.use_modulate):
            # the predecessor forbids it outright (MoeCombineTransformer.pyc L557-570) and the shipped transformer-block
            # experts are shape-broken with a per-token temb (SURVEY.md F5)
            raise ValueError("Warning: please use rope or modulated")
        self.use_shared_expert = bool(get("use_shared_expert", False))  # :863 (False: the routed experts alone, :1024 skipped)
        # :893-923 (V2): two joint blocks; moe_forward calls consis_module[0] twice and consis_module[1] never (:994, :998). Its
        # result only reaches the output through the tuple the shared-expert branch builds (:1024), so with
        # use_shared_expert=False the blocks hold weights but contribute nothing (tests/golden: moe_wiring).
        self.use_consis_module = bool(get("use_consis_module", False))
        dev = get("single_control_dev", 2)
        self.cn_joint_layers, self.cn_single_joint_layers = a.num_layers // dev, a.num_single_layers // dev
        self.single_block_control_method = get("single_block_control_method", "overall_add")
        self.use_single_trans_blocks = get("use_single_trans_blocks", True)
        self.expert_nums = get("expert_num", None) or (self.condition_nums + 1) * get("expert_num_each_condition", 3)
        self.top_k = get("top_num", 1)
        assert self.top_k == 1, "only top-1 gating (the shipped configuration) is implemented"
        self.num_local_experts = self.expert_nums
        self.cn_method = get("cn2base_method", "add")

        self.control_time_text = _TimeTextW(ws, "control_time_text_embed", D, a.pooled_projection_dim, a.guidance_embeds)
        self.control_condition = _TimeTextW(ws, "control_condition_embed", D, a.pooled_projection_dim, a.guidance_embeds)
        self.control_context_embedder_w = ws.linear("control_context_embedder", D, D)
        self.control_x_embedder_w = ws.linear("control_x_embedder", D, a.in_channels)
        self.ctrl_double = [_DoubleBlockW(ws, f"control_joint_trans_blocks.{j}", D, dh) for j in range(self.cn_joint_layers)]
        self.add_double = [ws.linear(f"controlnet_add_joint_blocks.{j}", D, D) for j in range(self.cn_joint_layers)]
        self.ctrl_single, self.add_single = [], []
        if self.use_single_trans_blocks:
            self.ctrl_single = [_SingleBlockW(ws, f"control_single_trans_blocks.{j}", D, dh)
                                for j in range(self.cn_single_joint_layers)]
            self.add_single = [ws.linear(f"controlnet_add_single_blocks.{j}", D, D) for j in range(self.cn_single_joint_layers)]
        E, P = self.expert_nums, a.pooled_projection_dim
        self.gate_wg = ws.alloc(E, D, dtype=torch.float32)  # evaluated in fp32 (SURVEY.md §A.5)
        ws.views["moe.moe_layer.gate.wg.weight"] = self.gate_wg
        # experts stacked: branch 0 = condition modulate, branch 1 = hidden modulate; [.0] = Linear(D,D), [.1] = Linear(P,D)
        self.exp_w = [ws.alloc(E, D, D), ws.alloc(E, D, D)]
        self.exp_b = [ws.alloc(E, D), ws.alloc(E, D)]
        self.exp_mod_w = [ws.alloc(E * D, P), ws.alloc(E * D, P)]
        self.exp_mod_b = [ws.alloc(E * D), ws.alloc(E * D)]
        for e in range(E):
            for br in (0, 1):
                p = f"moe.moe_layer.experts.deepspeed_experts.{e}.{br}"
                ws.views[p + ".0.weight"], ws.views[p + ".0.bias"] = self.exp_w[br][e], self.exp_b[br][e]
                ws.views[p + ".1.weight"] = self.exp_mod_w[br][e * D:(e + 1) * D]
                ws.views[p + ".1.bias"] = self.exp_mod_b[br][e * D:(e + 1) * D]
        self.shared = [_DoubleBlockW(ws, f"shared_expert.{s}", D, dh) for s in (0, 1)] if self.use_shared_expert else []
        self.consis = [_DoubleBlockW(ws, f"consis_module.{s}", D, dh) for s in (0, 1)] if self.use_consis_module else []
        self.trainable_control_modules = {k: None for k in (
            "control_pos_embed_input", "control_time_text_embed", "control_condition_embed", "control_context_embedder",
            "control_x_embedder", "control_joint_trans_blocks", "controlnet_add_joint_blocks", "control_single_trans_blocks",
            "controlnet_add_single_blocks", "moe") + (("shared_expert",) if self.use_shared_expert else ())
            + (("consis_module",) if self.use_consis_module else ())}
        self._control_ready = True
        if get("use_transformer_params", False):
            self.init_control_param()

    @torch.no_grad()
    def init_control_param(self):
        """reference :790-803: the control branch starts from the base model's weights — both control time-text embedders copy
        `time_text_embed`, control block j copies base block j (`load_state_dict(..., strict=False)` over the ModuleLists: the
        first cn_*_layers blocks match by index). `control_x_embedder` loads its OWN state dict there (a no-op, kept)."""
        v = self._ws.views

        def copy_prefix(dst: str, src: str):
            for k in [k for k in v if k.startswith(src + ".")]:
                kd = dst + k[len(src):]
                if kd in v and v[kd].shape == v[k].shape:
                    v[kd].copy_(v[k])

        copy_prefix("control_time_text_embed", "time_text_embed")
        copy_prefix("control_condition_embed", "time_text_embed")
        for j in range(self.cn_joint_layers):
            copy_prefix(f"control_joint_trans_blocks.{j}", f"transformer_blocks.{j}")
        for j in range(len(self.ctrl_single)):
            copy_prefix(f"control_single_trans_blocks.{j}", f"single_transformer_blocks.{j}")
        self._weights_loaded()

    # ---------------------------------------------------------------------------------------------------------
    # workspaces
    # ---------------------------------------------------------------------------------------------------------
    def _workspace(self, B: int, N: int, T: int):
        return self._cached_workspace((B, N, T), lambda: self._make_workspace(B, N, T))

    def _make_workspace(self, B: int, N: int, T: int):
        D, dev = self.inner_dim, self.device_
        S = T + N
        Smax = T + 2 * N  # shared_expert[1] runs over [txt | img | cond]
        consis = self.use_consis_module and self.use_shared_expert
        if consis:
            Smax = max(Smax, 3 * N)  # consis_module[0], second call: [img | experts' img | consis cond]
        E = self.expert_nums
        C = ops.moe_capacity(B * N, E)
        z = lambda *s, dt=BF16: torch.empty(*s, device=dev, dtype=dt)  # noqa: E731
        n_mod = (6 * 2 * (self.arch.num_layers + self.cn_joint_layers + 1 + self.condition_nums) + 3 * (self.arch.num_single_layers + len(self.ctrl_single)) + 2)
        if consis:
            n_mod += 6 * 2 * (1 + self.condition_nums)
        b = types.SimpleNamespace(
            X=z(B, S, D), NX=z(B, Smax, D), QKV=z(B, Smax, 3 * D), AO=z(B, Smax, D), FF=z(B, Smax, 4 * D),
            CAT=z(B, S, 5 * D), CH=z(B, N, D), CS=z(B, S, D), CENC=z(B, T, D), COND=z(B, N, D), HC=z(B, 2 * N, D),
            G=z(B * N, D), A=z(E * C, D), YC=z(E * C, D), YH=z(E * C, D), EH=z(B * N, D), EC=z(B * N, D), CIN=z(B, N, D),
            MOD=z(B, n_mod * D, dt=torch.float32), n_mod=n_mod, tmp=z(B, D, dt=torch.float32),
            # step-constant conditioning vectors [temb | control_temb | sum_c condition_temb | condition_temb_c ...] and their SiLU
            TEMBS=z(3 + self.condition_nums, B, D, dt=torch.float32), STEMBS=z(3 + self.condition_nums, B, D, dt=torch.float32),
            MODC=z(B, E, D, dt=torch.float32), MODH=z(B, E, D, dt=torch.float32),
            rope=z(S, self.arch.attention_head_dim, dt=torch.float32),
            rope0=z(2 * N, self.arch.attention_head_dim, dt=torch.float32),
            rope1=z(Smax, self.arch.attention_head_dim, dt=torch.float32),
            NO=z(B, N, D), OUT=z(B, N, self.arch.in_channels), capacity=C)
        b.temb, b.ctemb, b.cdtemb = b.TEMBS[0], b.TEMBS[1], b.TEMBS[2]
        b.cdtemb_c = [b.TEMBS[3 + c] for c in range(self.condition_nums)]
        b.mod_plans = None
        if self.linear_dtype == FP8:  # e4m3 operands (+ one fp32 scale per row) of the quantised block linears
            f8 = lambda *sh: z(*sh, dt=FP8)  # noqa: E731
            b.NXQ, b.NXS = f8(B, Smax, D), z(B, Smax, dt=torch.float32)
            b.AOQ, b.AOS = f8(B, Smax, D), z(B, Smax, dt=torch.float32)
            b.FFQ, b.FFS = f8(B, Smax, 4 * D), z(B, Smax, dt=torch.float32)
            b.CATQ, b.CATS = f8(B, S, 5 * D), z(B, S, dt=torch.float32)
        if consis:  # [experts' image output | consis condition output] and the id tables of the two consis_module[0] calls
            b.CONS = z(B, 2 * N, D)
            b.ropek0 = z(2 * N, self.arch.attention_head_dim, dt=torch.float32)
            b.ropek1 = z(3 * N, self.arch.attention_head_dim, dt=torch.float32)
        return b

    # ---------------------------------------------------------------------------------------------------------
    # building blocks (each line = one kernel launch in libunigen_b200.so)
    # ---------------------------------------------------------------------------------------------------------
    def _conditioning_vectors(self, buf, B, timestep, guidance, pooled, cond_pooled):
        """temb / control_temb / condition_temb (per condition and summed, :1048-1049, :1314-1319) into buf.TEMBS, then ONE SiLU pass
        over all of them (every AdaLN linear consumes silu(temb))."""
        n_cond = self.condition_nums
        t_emb = ops.timestep_embedding(timestep, scale=1000.0, batch=B)  # `timestep * 1000` (:1220) folded into the kernel
        g_emb = ops.timestep_embedding(guidance, scale=1000.0, batch=B) if guidance is not None else None
        self._time_text(self.time_text, t_emb, pooled, buf.temb, buf.tmp, g_emb)
        ctrl_pooled = pooled if self.use_pooled_prompt_embeds else torch.zeros_like(pooled)
        self._time_text(self.control_time_text, t_emb, ctrl_pooled, buf.ctemb, buf.tmp, g_emb)      # control_temb
        for c in range(n_cond):  # condition_temb per condition and their sum (what the control blocks are modulated by)
            self._time_text(self.control_condition, t_emb, cond_pooled[c], buf.cdtemb_c[c], buf.tmp, g_emb)
            self._time_text(self.control_condition, t_emb, cond_pooled[c], buf.cdtemb, buf.tmp, g_emb, accumulate=c > 0)
        ops.silu(buf.TEMBS, buf.STEMBS)

    def _mod_plans(self, buf, pool=None):
        """AdaLN job tables of this workspace (ops.GemvPlan: device-resident, built once): `early` = the linears the first
        block pair and the CoMoE pre-stage need, `late` = all others, `all` = both (sequence parallelism: one sharded launch
        writing into every rank's peer-mapped MOD). Also the fp32 [B, D] chunk views of MOD every block reads."""
        key = (buf.MOD.data_ptr(), id(pool))
        mp = buf.mod_plans
        if mp is not None and mp.key == key:
            return mp
        D, n_cond = self.inner_dim, self.condition_nums
        s_temb, s_ctemb, s_cdtemb = buf.STEMBS[0], buf.STEMBS[1], buf.STEMBS[2]
        slot = [0]
        early, late = [], []

        def job(w, x, n_chunks, dst):
            s0 = slot[0]
            slot[0] += n_chunks
            region = buf.MOD[:, s0 * D:(s0 + n_chunks) * D]
            dst.append((w[0], w[1], x, region, False))
            return [region[:, i * D:(i + 1) * D] for i in range(n_chunks)]

        mp = types.SimpleNamespace(key=key)
        mp.m_double = [(job(w.norm1, s_temb, 6, early if i == 0 else late), job(w.norm1_ctx, s_temb, 6, early if i == 0 else late))
                       for i, w in enumerate(self.double)]
        mp.m_cdouble = [(job(w.norm1, s_cdtemb, 6, early if j == 0 else late), job(w.norm1_ctx, s_cdtemb, 6, early if j == 0 else late))
                        for j, w in enumerate(self.ctrl_double)]
        mp.m_single = [job(w.norm, s_temb, 3, late) for w in self.single]
        mp.m_csingle = [job(w.norm, s_cdtemb, 3, late) for w in self.ctrl_single]
        mp.mods_s0, mp.mods_s1 = [None] * n_cond, None
        if self.use_shared_expert:  # shared_expert[0] is modulated by THIS condition's temb, shared_expert[1] by control_temb
            mp.mods_s0 = [(job(self.shared[0].norm1, buf.STEMBS[3 + c], 6, early), job(self.shared[0].norm1_ctx, buf.STEMBS[3 + c], 6, early))
                          for c in range(n_cond)]
            mp.mods_s1 = (job(self.shared[1].norm1, s_ctemb, 6, early), job(self.shared[1].norm1_ctx, s_ctemb, 6, early))
        mp.mods_k0, mp.mods_k1 = [None] * n_cond, None
        if self.use_consis_module and self.use_shared_expert:
            # consis_module[0]: first call modulated by THIS condition's temb, second call by control_temb (:994, :998)
            k0 = self.consis[0]
            mp.mods_k0 = [(job(k0.norm1, buf.STEMBS[3 + c], 6, early), job(k0.norm1_ctx, buf.STEMBS[3 + c], 6, early))
                          for c in range(n_cond)]
            mp.mods_k1 = (job(k0.norm1, s_ctemb, 6, early), job(k0.norm1_ctx, s_ctemb, 6, early))
        mp.m_out = job(self.norm_out_w, s_temb, 2, late)  # AdaLayerNormContinuous: (scale, shift)
        assert slot[0] <= buf.n_mod, (slot[0], buf.n_mod)
        dev = self.device_
        if pool is None:
            mp.early, mp.late, mp.all = ops.GemvPlan(early, dev), ops.GemvPlan(late, dev), None
        else:
            mp.early = mp.late = None
            mp.all = ops.GemvPlan(early + late, dev, pool=pool)
        buf.mod_plans = mp
        return mp

    def _rope(self, out: torch.Tensor, *id_tables: torch.Tensor):
        """FluxPosEmbed over `cat(id_tables)` written table by table into consecutive rows of `out` (no concat copy)."""
        a, r0 = self.arch, 0
        for ids in id_tables:
            ops.rope_table(ids, a.axes_dims_rope, a.theta, out=out[r0:r0 + ids.shape[0]])
            r0 += ids.shape[0]
        return out

    def _attend(self, buf, S: int, out: torch.Tensor):
        """Joint attention over rows [0, S) of the fused QKV buffer (q/k already normalised + rotated) -> out [B, S, D].
        The sequence-parallel subclass replaces this with the Ulysses exchange (parallel.py)."""
        a, D = self.arch, self.inner_dim
        ops.attention(buf.QKV[:, :S, 0:D], buf.QKV[:, :S, D:2 * D], buf.QKV[:, :S, 2 * D:3 * D], out, a.num_attention_heads,
                      a.attention_head_dim, variant=self.attn_variant)
        return out

    def _qk_norm(self, rms_w: torch.Tensor, rope_rows: Optional[torch.Tensor]):
        """Arguments of the fused QK-RMSNorm + RoPE epilogue of a q|k|v projection GEMM (ops.gemm qk_norm=...)."""
        if not self.fuse_qk_norm:
            return None
        return dict(weight=rms_w, head_dim=self.arch.attention_head_dim, d=self.inner_dim, cos_sin=rope_rows, eps=1e-6)

    def _joint_attention(self, buf, B, n_ctx, n_smp, rms_ctx, rms_smp, rope):
        """(RMSNorm(q,k)+RoPE in place on QKV rows unless it was fused into the projection GEMMs) + joint attention -> AO."""
        a = self.arch
        H, dh, D = a.num_attention_heads, a.attention_head_dim, self.inner_dim
        S = n_ctx + n_smp
        if not self.fuse_qk_norm:
            qk = buf.QKV[:, :S, :2 * D]
            if n_ctx:
                ops.qk_rmsnorm_rope(qk[:, :n_ctx], 2 * H, dh, rms_ctx, rope[:n_ctx] if rope is not None else None, heads_per_weight=H)
            if n_smp:
                ops.qk_rmsnorm_rope(qk[:, n_ctx:], 2 * H, dh, rms_smp, rope[n_ctx:S] if rope is not None else None, heads_per_weight=H)
        return self._attend(buf, S, buf.AO[:, :S])

    def _double_block(self, buf, w: _DoubleBlockW, mod_smp, mod_ctx, smp_in, ctx_in, smp_out, ctx_out, rope):
        """diffusers FluxTransformerBlock (SURVEY.md §A.2). smp/ctx = image-role / text-role streams ([B, n, D] views);
        outputs may alias inputs (in-place residual). ctx_out=None skips the context stream's post-attention half —
        exact whenever the caller discards `encoder_hidden_states` (control blocks, shared_expert[1]). Either stream may
        be empty on a sequence-parallel rank."""
        D = self.inner_dim
        B, n_smp, n_ctx = smp_in.shape[0], smp_in.shape[1], ctx_in.shape[1]
        S = n_ctx + n_smp
        sh_a, sc_a, g_a, sh_m, sc_m, g_m = mod_smp
        csh_a, csc_a, cg_a, csh_m, csc_m, cg_m = mod_ctx
        nx_c, nx_s = buf.NX[:, :n_ctx], buf.NX[:, n_ctx:S]
        qn_c = qn_s = qa_c = qa_s = qf_c = qf_s = None
        if w.fp8:  # e4m3 operands (+ one fp32 scale per row) of the same rows; the pre-stage's bf16 blocks never use them
            qn_c, qn_s = (buf.NXQ[:, :n_ctx], buf.NXS[:, :n_ctx]), (buf.NXQ[:, n_ctx:S], buf.NXS[:, n_ctx:S])
            qa_c, qa_s = (buf.AOQ[:, :n_ctx], buf.AOS[:, :n_ctx]), (buf.AOQ[:, n_ctx:S], buf.AOS[:, n_ctx:S])
            qf_c, qf_s = (buf.FFQ[:, :n_ctx], buf.FFS[:, :n_ctx]), (buf.FFQ[:, n_ctx:S], buf.FFS[:, n_ctx:S])
        # The text stream's GEMMs are small (M = 512 at cfg3: 24-96 tiles for 148 SMs); issued on a second stream they run
        # beside the image stream's GEMMs (disjoint rows of NX / QKV / FF) and fill the SMs those leave idle in their last wave.
        main = torch.cuda.current_stream()
        side = self._text_stream if (self.overlap_text_stream and ctx_out is not None and n_ctx and n_smp
                                     and not getattr(self, "_sp_active", False)) else None
        if n_ctx:
            if side is not None:
                side.wait_stream(main)
            with torch.cuda.stream(side if side is not None else main):
                self._ln(w, ctx_in, nx_c, qn_c, csh_a, csc_a)
                self._linear(w.add_qkv, nx_c, qn_c, out=buf.QKV[:, :n_ctx],
                             qk_norm=self._qk_norm(w.rms_ctx, rope[:n_ctx] if rope is not None else None))
        if n_smp:
            self._ln(w, smp_in, nx_s, qn_s, sh_a, sc_a)
            self._linear(w.qkv, nx_s, qn_s, out=buf.QKV[:, n_ctx:S],
                         qk_norm=self._qk_norm(w.rms, rope[n_ctx:S] if rope is not None else None))
        if side is not None:
            main.wait_stream(side)
        ao = self._joint_attention(buf, B, n_ctx, n_smp, w.rms_ctx, w.rms, rope)
        if ctx_out is not None and n_ctx:
            if side is not None:
                side.wait_stream(main)
            with torch.cuda.stream(side if side is not None else main):
                self._linear(w.to_add_out, ao[:, :n_ctx], qa_c, out=ctx_out, quantize=True, gate=cg_a, residual=ctx_in)
                self._ln(w, ctx_out, nx_c, qn_c, csh_m, csc_m)
                self._linear(w.ffc1, nx_c, qn_c, out=buf.FF[:, :n_ctx], act=UG_ACT_GELU_TANH)
                self._linear(w.ffc2, buf.FF[:, :n_ctx], qf_c, out=ctx_out, quantize=True, gate=cg_m, residual=ctx_out)
        if n_smp:
            # h = h + gate_msa * to_out(attn)
            self._linear(w.to_out, ao[:, n_ctx:S], qa_s, out=smp_out, quantize=True, gate=g_a, residual=smp_in)
            # h = h + gate_mlp * ff(LN(h) * (1 + scale_mlp) + shift_mlp)
            self._ln(w, smp_out, nx_s, qn_s, sh_m, sc_m)
            self._linear(w.ff1, nx_s, qn_s, out=buf.FF[:, n_ctx:S], act=UG_ACT_GELU_TANH)
            self._linear(w.ff2, buf.FF[:, n_ctx:S], qf_s, out=smp_out, quantize=True, gate=g_m, residual=smp_out)
        if side is not None:
            main.wait_stream(side)

    def _single_attention(self, buf, S: int, rms: torch.Tensor, rope, out: torch.Tensor):
        """(RMSNorm(q,k)+RoPE in place on the QKV rows unless fused into the projection GEMM) + attention over rows [0, S) ->
        `out` (the first D columns of CAT). The sequence-parallel subclass fuses both with the Ulysses exchange."""
        a, D = self.arch, self.inner_dim
        H, dh = a.num_attention_heads, a.attention_head_dim
        if not self.fuse_qk_norm:
            ops.qk_rmsnorm_rope(buf.QKV[:, :S, :2 * D], 2 * H, dh, rms, rope[:S] if rope is not None else None, heads_per_weight=H)
        return self._attend(buf, S, out)

    def _single_block(self, buf, w: _SingleBlockW, mod, x_in, x_out, rope):
        """diffusers FluxSingleTransformerBlock (SURVEY.md §A.3): x_out = x_in + gate * proj_out([attn | gelu(mlp)])."""
        a = self.arch
        H, dh, D = a.num_attention_heads, a.attention_head_dim, self.inner_dim
        B, S = x_in.shape[0], x_in.shape[1]
        shift, scale, gate = mod
        nx, cat = buf.NX[:, :S], buf.CAT[:, :S]
        qn = (buf.NXQ[:, :S], buf.NXS[:, :S]) if w.fp8 else None  # one quantised operand for both GEMMs that read nx
        qc = (buf.CATQ[:, :S], buf.CATS[:, :S]) if w.fp8 else None
        self._ln(w, x_in, nx, qn, shift, scale)
        self._linear(w.qkv, nx, qn, out=buf.QKV[:, :S], qk_norm=self._qk_norm(w.rms, rope[:S] if rope is not None else None))
        self._linear(w.mlp, nx, qn, out=cat[:, :, D:], act=UG_ACT_GELU_TANH)
        self._single_attention(buf, S, w.rms, rope, cat[:, :, :D])
        self._linear(w.out, cat, qc, out=x_out, quantize=True, gate=gate, residual=x_in)

    # ---------------------------------------------------------------------------------------------------------
    # CoMoE pre-stage (reference preprocess_moe_forward :1028-1068, moe_forward :969-1026, MOELayer.forward,
    # expert_forward :925-967) — runs once per step at the first control call
    # ---------------------------------------------------------------------------------------------------------
    def _prestage(self, buf, B, N, T, h_img, cond_tokens, pooled, cond_pooled, rts_uniform, mods_s0, mods_s1, cond_index,
                  txt_ids, img_ids, cond_ids, mods_k0=None, mods_k1=None):
        """One CoMoE pass for one condition; the control stream `CIN` accumulates over conditions
        (MultiCondtionUniGenFlux: merged_hidden_states = sum_c (expert_hidden + expert_cond), :1313-1316)."""
        a = self.arch
        D, E, C = self.inner_dim, self.expert_nums, buf.capacity
        gv = self.gemm_variant
        ops.gemm(cond_tokens, self.control_x_embedder_w[0], out=buf.COND, bias=self.control_x_embedder_w[1], variant=gv)
        self._rope(buf.rope0, cond_ids, img_ids)
        self._rope(buf.rope1, txt_ids, img_ids, cond_ids)
        # --- gate + Random-Token-Selection routing (DeepSpeed top1gating, SURVEY.md §A.5) ---
        g = buf.G.view(B, N, D)
        ops.add(h_img, buf.COND, g)
        tag = "moe" if cond_index == 0 and self.condition_nums == 1 else f"moe.cond{cond_index}"
        # the gate sees the bf16 sum, exactly what `hidden_states + condition_hidden_states` is in the reference's bf16 run
        self._rec(tag + ".cond_embed", buf.COND); self._rec(tag + ".gate_input", g)
        route = ops.moe_route(buf.G, self.gate_wg, rts_uniform, C)
        if self.trace is not None:
            for k in ("expert_idx", "slot", "prob", "slot_token", "exp_counts"):
                self.trace[f"{tag}.route.{k}"] = route[k].detach().clone()
        # --- condition-modulated experts: cond' = Wc (s_c . cond) + bc ; hid' = Wh (s_h . (hid + cond')) + bh ---
        ops.gemv(cond_pooled, self.exp_mod_w[0], self.exp_mod_b[0], out=buf.MODC.view(B, E * D))
        ops.gemv(pooled, self.exp_mod_w[1], self.exp_mod_b[1], out=buf.MODH.view(B, E * D))
        ops.moe_gather_modulate(buf.COND.view(B * N, D), route["slot_token"], buf.MODC, E, C, N, out=buf.A)
        ops.gemm(buf.A.view(E, C, D), self.exp_w[0], out=buf.YC.view(E, C, D), bias=self.exp_b[0], variant=gv)
        hid_flat = buf.EH  # contiguous copy of the image rows of X (they are strided inside the joint buffer)
        ops.copy(h_img, hid_flat.view(B, N, D))
        ops.moe_gather_modulate(hid_flat, route["slot_token"], buf.MODH, E, C, N, addend=buf.YC, out=buf.A)
        ops.gemm(buf.A.view(E, C, D), self.exp_w[1], out=buf.YH.view(E, C, D), bias=self.exp_b[1], variant=gv)
        # --- shared experts (V2, :1013-1022) ---
        hc_h, hc_c = buf.HC[:, :N], buf.HC[:, N:]
        if self.use_shared_expert:
            self._double_block(buf, self.shared[0], mods_s0[0], mods_s0[1], h_img, buf.COND, hc_h, hc_c, buf.rope0)
            self._double_block(buf, self.shared[1], mods_s1[0], mods_s1[1], buf.HC, buf.CENC, buf.HC, None, buf.rope1)
        # --- combine (gate-probability weighted, dropped tokens -> 0) and sum: ctrl_in (+)= (hid + EH) + (cond + EC) ---
        ops.moe_combine(buf.YH, route, C, buf.EH)
        ops.moe_combine(buf.YC, route, C, buf.EC)
        self._rec(tag + ".expert_hidden", buf.EH.view(B, N, D)); self._rec(tag + ".expert_cond", buf.EC.view(B, N, D))
        if self.use_consis_module and self.use_shared_expert:
            # --- consis module (V2, :982-1003): consis_module[0] over (hidden = experts' cond output, encoder = cond tokens) with
            # the condition's temb and ids, then over (hidden = [experts' image output | that result], encoder = image tokens)
            # with control_temb; its two halves are ADDED to the experts' outputs. The encoder-side results are discarded
            # (`_, x = block(...)`), so the context streams' post-attention halves are never computed (ctx_out=None).
            eh, ec = buf.EH.view(B, N, D), buf.EC.view(B, N, D)
            self._rope(buf.ropek0, cond_ids, cond_ids)
            self._rope(buf.ropek1, img_ids, img_ids, cond_ids)
            ops.copy(eh, buf.CONS[:, :N])
            self._double_block(buf, self.consis[0], mods_k0[0], mods_k0[1], ec, buf.COND, buf.CONS[:, N:], None, buf.ropek0)
            self._double_block(buf, self.consis[0], mods_k1[0], mods_k1[1], buf.CONS, h_img, buf.CONS, None, buf.ropek1)
            self._rec(tag + ".consis_hidden", buf.CONS[:, :N]); self._rec(tag + ".consis_cond", buf.CONS[:, N:])
            ops.add(eh, buf.CONS[:, :N], eh)
            ops.add(ec, buf.CONS[:, N:], ec)
        if not self.use_shared_expert:  # use_shared_expert=False (:1005): the control stream is the routed experts' output alone
            if cond_index == 0:
                ops.add(buf.EH.view(B, N, D), buf.EC.view(B, N, D), buf.CIN)
            else:
                ops.add(buf.CIN, buf.EH.view(B, N, D), buf.CIN)
                ops.add(buf.CIN, buf.EC.view(B, N, D), buf.CIN)
            return route
        self._rec(tag + ".shared_hidden", hc_h); self._rec(tag + ".shared_cond", hc_c)
        if cond_index == 0:
            ops.add(hc_h, buf.EH.view(B, N, D), buf.CIN)
        else:
            ops.add(buf.CIN, hc_h, buf.CIN)
            ops.add(buf.CIN, buf.EH.view(B, N, D), buf.CIN)
        ops.add(buf.CIN, hc_c, buf.CIN)
        ops.add(buf.CIN, buf.EC.view(B, N, D), buf.CIN)
        return route

    # ---------------------------------------------------------------------------------------------------------
    # forward (reference :1182-1271 + base_forward :1106-1180 + control_forward :1070-1104)
    # ---------------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, hidden_states, condition_hidden_states=None, conditioning_scale: float = 1.0,
                encoder_hidden_states=None, pooled_projections=None, condition_pooled_projections=None, timestep=None,
                img_ids=None, txt_ids=None, guidance=None, condition_ids=None, joint_attention_kwargs=None,
                skip_layers=None, rts_uniform=None, **kwargs):
        """Reference signature (src/UniGenTransformer.py:1182-1198). `joint_attention_kwargs['scale']` (PEFT LoRA scale)
        is accepted and ignored: the S-variant forward never applies an adapter (SURVEY.md F6)."""
        if not self._control_ready:
            raise ops.UgError("call init_condition_block(condition_nums=..., control_params=...) before forward")
        if encoder_hidden_states is None or condition_hidden_states is None or timestep is None:
            raise ops.UgError("forward needs hidden_states, condition_hidden_states, encoder_hidden_states and timestep")
        B, N, _ = hidden_states.shape
        T = encoder_hidden_states.shape[1]
        # MultiCondtionUniGenFlux passes LISTS (condition tokens / pooled embeddings / ids), reference :1297
        multi = isinstance(condition_hidden_states, (list, tuple))
        cond_list = list(condition_hidden_states) if multi else [condition_hidden_states]
        cpool_list = list(condition_pooled_projections) if multi else [condition_pooled_projections]
        cid_list = list(condition_ids) if multi else [condition_ids]
        if len(cond_list) != self.condition_nums or len(cpool_list) != len(cond_list) or len(cid_list) != len(cond_list):
            raise ops.UgError(f"expected {self.condition_nums} condition(s) (init_condition_block), got {len(cond_list)}")
        if any(c.shape[-2] != N for c in cond_list):
            raise ops.UgError("condition tokens must match the image token count (Nc == N) for the CoMoE pre-stage")
        if T == N:
            raise ops.UgError("T == N: the reference MOELayer would also dispatch the text tensor (SURVEY.md §8 A9); unsupported")
        dev = self.device_
        f32 = lambda t: t.to(device=dev, dtype=torch.float32).contiguous()  # noqa: E731
        sq = lambda t: t[0] if t.dim() == 3 else t  # noqa: E731  (3-D ids are accepted and squeezed, reference :1225-1236)
        if rts_uniform is None:
            # DeepSpeed draws this uniform tensor in train AND eval (SURVEY.md F7); torch RNG is plumbing here
            u_list = [torch.rand(B * N, self.expert_nums, device=dev, dtype=torch.float32) for _ in cond_list]
        else:
            u_list = list(rts_uniform) if isinstance(rts_uniform, (list, tuple)) else [rts_uniform]
        staged = dict(
            hs=hidden_states.to(dev), es=encoder_hidden_states.to(dev), pooled=f32(pooled_projections),
            timestep=f32(timestep), guidance=f32(guidance) if guidance is not None else None,
            txt_ids=f32(sq(txt_ids)), img_ids=f32(sq(img_ids)))
        for c in range(len(cond_list)):
            x = cond_list[c].to(dev)
            staged[f"cs{c}"] = x if x.dim() == 3 else x.unsqueeze(0)
            cp = f32(cpool_list[c])
            staged[f"cp{c}"] = cp if cp.dim() == 2 else cp.unsqueeze(0)
            staged[f"cid{c}"] = f32(sq(cid_list[c]))
            staged[f"u{c}"] = f32(u_list[c])
        key = (B, N, T, float(conditioning_scale), guidance is not None,
               tuple((k, v.dtype) for k, v in staged.items() if v is not None))
        out, add_losses, add_outputs = self._run_staged(key, staged, float(conditioning_scale))
        if self.clone_outputs:
            # the velocity lives in the workspace (and, under graph replay, in the graph's static output): hand out a copy so
            # that a second forward (cond / uncond passes held together) does not overwrite the first result
            out = ops.copy(out, torch.empty(out.shape, device=out.device, dtype=out.dtype))
            add_losses = {k: v.clone() for k, v in add_losses.items()}
            add_outputs = {k: v.clone() for k, v in add_outputs.items()}
        return out, add_losses, add_outputs

    def _forward_impl(self, conditioning_scale, hs, es, pooled, timestep, guidance, txt_ids, img_ids, **cond):
        a = self.arch
        n_cond = self.condition_nums
        cs = [cond[f"cs{c}"] for c in range(n_cond)]
        cond_pooled = [cond[f"cp{c}"] for c in range(n_cond)]
        condition_ids = [cond[f"cid{c}"] for c in range(n_cond)]
        rts_uniform = [cond[f"u{c}"] for c in range(n_cond)]
        D, H, dh = self.inner_dim, a.num_attention_heads, a.attention_head_dim
        B, N, _ = hs.shape
        T = es.shape[1]
        S = T + N
        buf = self._workspace(B, N, T)
        n0 = ops.launch_count()
        hs, es = ops.to_bf16(hs.contiguous()), ops.to_bf16(es.contiguous())
        cs = [ops.to_bf16(c.contiguous()) for c in cs]
        gv = self.gemm_variant

        # ---- embeddings (:1215-1239) ----
        x_txt, x_img = buf.X[:, :T], buf.X[:, T:]
        ops.gemm(hs, self.x_embedder_w[0], out=x_img, bias=self.x_embedder_w[1], variant=gv)
        ops.gemm(es, self.context_embedder_w[0], out=x_txt, bias=self.context_embedder_w[1], variant=gv)
        self._conditioning_vectors(buf, B, timestep, guidance, pooled, cond_pooled)
        self._rope(buf.rope, txt_ids, img_ids)
        self._rec("temb", buf.temb); self._rec("x_embed", x_img); self._rec("context_embed", x_txt)
        self._rec("control_temb", buf.ctemb); self._rec("condition_temb", buf.cdtemb)
        for c in range(n_cond):
            self._rec(f"condition_temb.{c}", buf.cdtemb_c[c])

        # ---- every block's AdaLN vectors, once per step (temb / condition_temb are step constants): ~10 GB of bf16 weights
        # streamed by TWO grouped-GEMV launches — what the first block pair and the pre-stage need on the main stream, the rest
        # on a side stream UNDER the tensor-core-bound block kernels ----
        mp = self._mod_plans(buf)
        m_double, m_cdouble, m_single, m_csingle = mp.m_double, mp.m_cdouble, mp.m_single, mp.m_csingle
        mods_s0, mods_s1, m_out = mp.mods_s0, mp.mods_s1, mp.m_out
        ops.gemv_grouped(mp.early)
        main_stream = torch.cuda.current_stream()
        side = self._side_stream if self.overlap_mod_gemv else None
        if side is not None:
            side.wait_stream(main_stream)
        with torch.cuda.stream(side if side is not None else main_stream):
            ops.gemv_grouped(mp.late)
        mods_joined = side is None

        # ---- 19 x [base double -> control double -> add] (:1124-1141) ----
        route = None
        n_cd = len(self.ctrl_double)
        for i, w in enumerate(self.double):
            if i == 1 and not mods_joined:  # everything after the first block pair needs the side-stream vectors
                main_stream.wait_stream(side)
                mods_joined = True
            self._double_block(buf, w, m_double[i][0], m_double[i][1], x_img, x_txt, x_img, x_txt, buf.rope)
            self._rec(f"double.{i}.base_hidden", x_img); self._rec(f"double.{i}.base_context", x_txt)
            j = int(i / (len(self.double) / n_cd))
            if route is None:  # first control call: CoMoE pre-stage, control stream := sum_c (expert_hidden + expert_cond)
                ops.gemm(x_txt, self.control_context_embedder_w[0], out=buf.CENC, bias=self.control_context_embedder_w[1], variant=gv)
                self._rec("moe.control_context", buf.CENC)
                for c in range(n_cond):
                    route = self._prestage(buf, B, N, T, x_img, cs[c], pooled, cond_pooled[c], rts_uniform[c], mods_s0[c],
                                           mods_s1, c, txt_ids, img_ids, condition_ids[c], mp.mods_k0[c], mp.mods_k1)
                self._rec("moe.ctrl_in", buf.CIN)
                ctrl_in = buf.CIN
            else:               # later calls: the control block reads the base stream
                ctrl_in = x_img
            self._double_block(buf, self.ctrl_double[j], m_cdouble[j][0], m_cdouble[j][1], ctrl_in, buf.CENC, buf.CH, None, buf.rope)
            wa = self.add_double[j]
            ops.gemm(buf.CH, wa[0], out=x_img, bias=wa[1], alpha=float(conditioning_scale), residual=x_img, variant=gv)
            self._rec(f"double.{i}.ctrl_hidden", buf.CH); self._rec(f"double.{i}.hidden", x_img)

        if not mods_joined:
            main_stream.wait_stream(side)
        # ---- 38 x [base single -> control single -> add] over the joint [text | image] stream (:1146-1172) ----
        n_cs = len(self.ctrl_single)
        for i, w in enumerate(self.single):
            self._single_block(buf, w, m_single[i], buf.X, buf.X, buf.rope)
            self._rec(f"single.{i}.base_hidden", buf.X)
            if n_cs:
                j = int(i / (len(self.single) / n_cs))
                self._single_block(buf, self.ctrl_single[j], m_csingle[j], buf.X, buf.CS, buf.rope)
                wa = self.add_single[j]
                self._rec(f"single.{i}.ctrl_hidden", buf.CS)
                if self.single_block_control_method == "overall_add":
                    ops.gemm(buf.CS, wa[0], out=buf.X, bias=wa[1], alpha=float(conditioning_scale), residual=buf.X, variant=gv)
                else:  # single_add: only the image rows receive the control signal
                    ops.gemm(buf.CS[:, T:], wa[0], out=x_img, bias=wa[1], alpha=float(conditioning_scale), residual=x_img, variant=gv)
            self._rec(f"single.{i}.hidden", buf.X)

        # ---- norm_out (AdaLayerNormContinuous: scale first, then shift) + proj_out (:1264-1265) ----
        ops.ln_modulate(x_img, buf.NO, m_out[1], m_out[0])
        ops.gemm(buf.NO, self.proj_out_w[0], out=buf.OUT, bias=self.proj_out_w[1], variant=gv)
        self._rec("velocity", buf.OUT)
        self._last_route = route
        ops.note_capture_launches(ops.launch_count() - n0)
        add_losses = dict(moe_loss=route["l_aux"][0] * 0.1)
        add_outputs = dict(expert_counts=route["exp_counts"])
        return buf.OUT, add_losses, add_outputs


class MultiCondtionUniGenFlux(UniGenFlux):
    """Reference `MultiCondtionUniGenFlux` (src/UniGenTransformer.py:1274-1450, spelling kept): `condition_hidden_states`,
    `condition_pooled_projections`, `condition_ids` (and the optional `rts_uniform`) are LISTS with one entry per condition;
    the CoMoE pre-stage runs once per condition, the control stream and condition_temb are summed, and moe_loss /
    expert_counts are those of the last condition. The base class already implements the list form."""


def canonical_control_params() -> Dict[str, Any]:
    """config/unigen.yaml:3-11 + `use_rope: True` (SURVEY.md §A.1)."""
    return dict(use_transformer_params=False, use_pooled_prompt_embeds=True, use_encoder_hidden_states=True, use_rope=True,
                expert_num_each_condition=3, top_num=1, use_modulate=False, use_shared_expert=True, use_consis_module=False,
                use_single_trans_blocks=True, single_block_control_method="overall_add", single_control_dev=2,
                cn2base_method="add")
