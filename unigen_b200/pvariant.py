"""B200-native P-variant: the predecessor's LoRA-switched joint blocks (SURVEY.md §A.7, §8 A11-A14).

Only stale bytecode of this design survives in the reference (`src/__pycache__/UniCombineTransformerBlock.cpython-312.pyc`
attn_forward L9-136 / block_forward L140-236 / single_block_forward L239-295 and `UniCombineTransformer2DModel...pyc`
forward L53-211), but it is the one artefact that exercises `enable_lora` (src/lora_switching_module.py) and the
condition-visibility rule BASELINE.json's north star names.  Here:

  * the joint sequence is one buffer  [ txt | img | c_1 | ... | c_n ]  (text first);
  * `enable_lora(modules, adapters)` is DATA: per row segment an adapter-group id. Group 0 = the "denoising" adapters
    (active_adapters minus condition types) stacked into one low-rank pair, group 1+i = the adapter named after
    condition i. The low-rank update runs inside the main GEMM: `ug_lora_down` (x @ A_g^T, skinny) feeds the fused
    epilogue of `ug_gemm_bf16` (acc += t . B_g[c], switched per row) — to_q|to_k|to_v are ONE GEMM with three LoRA pairs;
  * the visibility rule (txt,img -> everything; c_i -> {txt,img,c_i}; or the stricter c_i -> {c_i}) is the segment mask
    of `ug_attention_bf16`, bit-exactly expandable by `ug_expand_segment_mask`.
"""
from __future__ import annotations

import math
import types
from typing import Any, Dict, List, Optional, Sequence

import torch

from . import ops
from .lora_switching_module import LoraLayer
from .model import BF16, FP8, FluxArch, _DoubleBlockW, _SingleBlockW, _TimeTextW, _Weights, quantize_block_linears
from .ops import UG_ACT_GELU_TANH

DOUBLE_LORA = ("norm1.linear", "attn.to_q", "attn.to_k", "attn.to_v", "attn.to_out.0", "ff.net.2")
SINGLE_LORA = ("norm.linear", "proj_mlp", "proj_out", "attn.to_q", "attn.to_k", "attn.to_v")
LORA_BLOCK = 64  # columns per adapter group in the K-extension operand (one 128-byte swizzle row of bf16)


class _LoraPair:
    """A [groups, n_sub * R, K] and pre-scaled B [groups, N, R] stacks for one (possibly fused) linear."""

    def __init__(self, device, groups: int, rank: int, k: int, n_each: int, n_sub: int = 1):
        self.rank, self.n_sub, self.n_each = rank, n_sub, n_each
        self.a = torch.zeros(groups, n_sub * rank, k, device=device, dtype=BF16)
        self.b = torch.zeros(groups, n_sub * n_each, rank, device=device, dtype=BF16)
        self.bw: Optional[torch.Tensor] = None
        self.aw: Optional[torch.Tensor] = None
        # fp8 operands (UniCombineFlux.quantize_fp8): aw quantised per row (aq, aws) and W2 = bw / w_scale[c] of the linear
        self.w_scale: Optional[torch.Tensor] = None
        self.aq = self.aws = self.w2 = None

    def build_wide(self):
        """W2 operand of the K-extension form: [n_sub * n_each, groups * 64], block g = B_g with sub-linear j's columns at
        [j * rank, (j + 1) * rank) of the block (matching the column order of the stacked down-projection A_g)."""
        G, n_tot, r = self.b.shape
        if self.n_sub * r > LORA_BLOCK:
            raise ops.UgError(f"stacked LoRA rank {self.n_sub * r} exceeds the {LORA_BLOCK}-column K-extension block")
        # (re)built IN PLACE after the first call so that captured CUDA graphs keep valid operand pointers
        bw = self.bw.zero_() if self.bw is not None else torch.zeros(n_tot, G * LORA_BLOCK, device=self.b.device, dtype=BF16)
        for g in range(G):
            for j in range(self.n_sub):
                rows = slice(j * self.n_each, (j + 1) * self.n_each)
                bw[rows, g * LORA_BLOCK + j * r:g * LORA_BLOCK + (j + 1) * r] = self.b[g, rows]
        self.bw = bw
        # stacked down-projection for the tensor-core form: [groups * 64, K], group g's lora_A rows at the top of block g
        aw = self.aw.zero_() if self.aw is not None else torch.zeros(G * LORA_BLOCK, self.a.shape[2], device=self.a.device, dtype=BF16)
        for g in range(G):
            aw[g * LORA_BLOCK:g * LORA_BLOCK + self.a.shape[1]] = self.a[g]
        self.aw = aw
        if self.w_scale is not None:
            self._quantize_operands()

    def quantize_fp8(self, w_scale: torch.Tensor):
        """Operands of the fp8 form for a linear quantised with per-output-channel scales `w_scale`: the linear's GEMM
        dequantises its whole accumulator by a_s[r] * w_scale[c], so the K extension carries the update pre-divided —
        A2 = (x / a_s) A^T (the fp8 masked down-projection of the quantised x with Aq, aws and unit row scales) and
        W2 = bw / w_scale[c]. Rebuilt in place by build_wide."""
        self.w_scale = w_scale
        self.aq = torch.empty(self.aw.shape, device=self.aw.device, dtype=FP8)
        self.aws = torch.empty(self.aw.shape[0], device=self.aw.device, dtype=torch.float32)
        self.w2 = torch.empty_like(self.bw)
        self._quantize_operands()

    def _quantize_operands(self):
        ops.quant_rows_fp8(self.aw, self.aq, self.aws)
        self.w2.copy_(self.bw.float() / self.w_scale[:, None])


class UniCombineFlux(torch.nn.Module):
    """P-variant denoiser. forward(hidden_states, condition_latents=[...], condition_ids=[...], condition_types=[...],
    encoder_hidden_states, pooled_projections, timestep, img_ids, txt_ids, c_t=0) -> velocity (B, N, in_channels)."""

    def __init__(self, arch: Optional[FluxArch] = None, device: Any = "cuda", lora_rank: int = 4, max_conditions: int = 3,
                 strict_mask: bool = False):
        super().__init__()
        self.arch = arch or FluxArch()
        self.device_ = torch.device(device)
        if self.device_.type != "cuda":
            raise ops.UgError("UniCombineFlux (B200-native) needs a CUDA device: the hot path has no CPU fallback")
        a = self.arch
        self.inner_dim = D = a.num_attention_heads * a.attention_head_dim
        dh = a.attention_head_dim
        ws = self._ws = _Weights(self.device_)
        self.x_embedder_w = ws.linear("x_embedder", D, a.in_channels)
        self.context_embedder_w = ws.linear("context_embedder", D, a.joint_attention_dim)
        self.time_text = _TimeTextW(ws, "time_text_embed", D, a.pooled_projection_dim, a.guidance_embeds)
        self.double = [_DoubleBlockW(ws, f"transformer_blocks.{i}", D, dh) for i in range(a.num_layers)]
        self.single = [_SingleBlockW(ws, f"single_transformer_blocks.{i}", D, dh) for i in range(a.num_single_layers)]
        self.norm_out_w = ws.linear("norm_out.linear", 2 * D, D)
        self.proj_out_w = ws.linear("proj_out", a.in_channels, D)
        self.rank = lora_rank
        self.groups = 1 + max_conditions
        self.strict_mask = strict_mask
        self.lora: Dict[str, _LoraPair] = {}
        self.lora_layers: Dict[str, LoraLayer] = {}
        self._dirty: set = set()
        self.condition_types: List[str] = []
        self.trace: Optional[Dict[str, torch.Tensor]] = None
        self._bufs: Dict[Any, Any] = {}
        self.gemm_variant = 0
        self.attn_variant = 0
        self.fuse_qk_norm = True  # QK-RMSNorm + RoPE in the projection GEMMs' epilogue (lora_mode "mma"), see _fused_qk
        # "mma": the switched low-rank update rides the main GEMM's tensor-core loop as a K extension (A2 / W2 operand pair);
        # "epilogue": it is applied per output element on the CUDA cores in the epilogue (kept for comparison)
        self.lora_mode = "mma"
        self.lora_down_mode = "mma"  # "mma": tensor-core down-projection (masked grouped GEMM); "simt": ug_lora_down_wide
        self.overlap_mod_gemv = True  # AdaLN GEMVs (HBM-bound) on a side stream under the tensor-core-bound blocks
        self._side_stream = torch.cuda.Stream(device=self.device_)
        self.add_cond_attn = False  # model_config['add_cond_attn'] (UniCombineTransformerBlock.pyc L201-202)
        self.linear_dtype = BF16  # float8_e4m3fn after quantize_fp8()

    @property
    def dtype(self):
        return BF16

    def state_dict(self, *a, **k):
        return dict(self._ws.views)

    # ---------------------------------------------------------------------------------------------------------
    def load_state_dict(self, state_dict, adapters: Sequence[str] = (), condition_types: Sequence[str] = (),
                        scaling: Optional[Dict[str, float]] = None, strict: bool = False,
                        lora_alpha: Optional[Dict[str, float]] = None):
        """Base weights under diffusers names + PEFT LoRA weights `<linear>.lora_A/B.<adapter>.weight`. `condition_types`
        fixes which adapter belongs to which condition slot (group 1+i); every other adapter is a denoising adapter and is
        stacked into group 0 — exactly the partition `enable_lora` makes at every call site of the predecessor.
        Every LoRA-wrapped linear gets a `LoraLayer` carrier (`self.lora_layers[name]`: `.active_adapters`, `.scaling`,
        `.set_scale`) for the reference's hooks (unigen_b200.lora_switching_module.enable_lora); `lora_alpha[a]` (default r,
        the UniCombine convention) gives the initial `scaling = lora_alpha / r`, `scaling=` overrides it directly."""
        if self.linear_dtype != BF16:
            raise ops.UgError("load_state_dict on an fp8-quantised model: its block linears no longer hold bf16 weights — load the "
                              "checkpoint into a fresh model, then call quantize_fp8()")
        a, D = self.arch, self.inner_dim
        dev = self.device_
        with torch.no_grad():
            for k, v in state_dict.items():
                if k in self._ws.views:
                    self._ws.views[k].copy_(v.to(dev, self._ws.views[k].dtype))
        self.condition_types = list(condition_types)
        adapters = list(adapters)
        den = [x for x in adapters if x not in condition_types]
        R = max(self.rank * max(len(den), 1), self.rank)
        if R not in (4, 8, 12, 16):
            raise ops.UgError(f"stacked LoRA rank {R} not supported by the fused epilogue (4, 8, 12, 16)")
        self._group_sets = [den] + [[t] for t in condition_types]
        if len(self._group_sets) > self.groups:
            raise ops.UgError("more conditions than max_conditions")
        # raw low-rank weights per linear and adapter stay on the device: the scale tables are rebuilt from them whenever a
        # hook (enable_lora / set_scale / set_adapter) changes a carrier
        self._lora_raw: Dict[str, Dict[str, tuple]] = {}
        self.lora_layers: Dict[str, LoraLayer] = {}
        self._pair_of: Dict[str, str] = {}     # linear name -> key of the (fused) operand pair it belongs to
        self._pair_names: Dict[str, List[str]] = {}
        self._dirty = set()

        def register(names: Sequence[str], key: str):
            self._pair_names[key] = list(names)
            for name in names:
                raw, ranks = {}, {}
                for ad in adapters:
                    ka, kb = f"{name}.lora_A.{ad}.weight", f"{name}.lora_B.{ad}.weight"
                    if ka in state_dict:
                        raw[ad] = (state_dict[ka].to(dev, BF16), state_dict[kb].to(dev, BF16))
                        ranks[ad] = raw[ad][0].shape[0]
                self._lora_raw[name] = raw
                alpha = {ad: float((lora_alpha or {}).get(ad, ranks[ad])) for ad in raw}
                layer = LoraLayer(name, list(raw), ranks, alpha, on_change=self._lora_changed)
                if scaling is not None:
                    for ad in raw:
                        layer.scaling[ad] = float(scaling.get(ad, layer.scaling[ad]))
                self.lora_layers[name] = layer
                self._pair_of[name] = key

        def mk(key, names, k, n_each):
            register(names, key)
            p = _LoraPair(dev, self.groups, R, k, n_each, len(names))
            self._fill(p, names)
            p.build_wide()
            return p

        def mk_vec(key, name, k, n):  # AdaLN linears run as GEMVs: rank padded to a multiple of 8 (GEMV inner-dim granularity)
            register([name], key)
            Rp = (R + 7) // 8 * 8
            p = _LoraPair(dev, self.groups, Rp, k, n, 1)
            self._fill(p, [name])
            return p

        L = self.lora = {}
        L["x_embedder"] = mk("x_embedder", ["x_embedder"], a.in_channels, D)
        for i in range(a.num_layers):
            p = f"transformer_blocks.{i}"
            L[p + ".norm1"] = mk_vec(p + ".norm1", p + ".norm1.linear", D, 6 * D)
            L[p + ".qkv"] = mk(p + ".qkv", [p + ".attn.to_q", p + ".attn.to_k", p + ".attn.to_v"], D, D)
            L[p + ".to_out"] = mk(p + ".to_out", [p + ".attn.to_out.0"], D, D)
            L[p + ".ff2"] = mk(p + ".ff2", [p + ".ff.net.2"], 4 * D, D)
        for i in range(a.num_single_layers):
            p = f"single_transformer_blocks.{i}"
            L[p + ".norm"] = mk_vec(p + ".norm", p + ".norm.linear", D, 3 * D)
            L[p + ".qkv"] = mk(p + ".qkv", [p + ".attn.to_q", p + ".attn.to_k", p + ".attn.to_v"], D, D)
            L[p + ".mlp"] = mk(p + ".mlp", [p + ".proj_mlp"], D, 4 * D)
            L[p + ".out"] = mk(p + ".out", [p + ".proj_out"], 5 * D, D)
        self.R = R
        self._dirty.clear()
        return types.SimpleNamespace(missing_keys=[], unexpected_keys=[])

    def _fill(self, pair: _LoraPair, names: Sequence[str]):
        """(Re)write a pair's stacked operands IN PLACE from the raw adapter weights and the carriers' current scales:
        group g's B block = B_a * effective_scale(a) for the adapters a of that group (0 for an inactive / disabled adapter)."""
        pair.a.zero_()
        pair.b.zero_()
        for s_i, name in enumerate(names):
            layer, raw = self.lora_layers[name], self._lora_raw[name]
            for g, aset in enumerate(self._group_sets):
                off = 0
                for ad in aset:
                    if ad not in raw:
                        continue
                    A, Bm = raw[ad]
                    r = A.shape[0]
                    pair.a[g, s_i * pair.rank + off:s_i * pair.rank + off + r] = A
                    pair.b[g, s_i * pair.n_each:(s_i + 1) * pair.n_each, off:off + r] = (Bm.float() * layer.effective_scale(ad)).to(BF16)
                    off += r

    def _lora_changed(self, name: str):
        self._dirty.add(self._pair_of[name])

    def _sync_lora(self):
        """Apply pending hook changes (enable_lora / set_scale / set_adapter on a carrier) to the operand stacks."""
        for key in sorted(self._dirty):
            pair = self.lora[key]
            self._fill(pair, self._pair_names[key])
            if pair.bw is not None:
                pair.build_wide()
        self._dirty.clear()

    @torch.no_grad()
    def quantize_fp8(self):
        """Opt-in fp8 (e4m3) transformer-block linears, in place; returns self (a second call does nothing). The linears of the
        double blocks (q|k|v, add_q|k|v, to_out, to_add_out, ff, ff_context) and single blocks (q|k|v, proj_mlp, proj_out) get
        one fp32 scale per output channel and are stored as e4m3; their bf16 copies are released and leave `state_dict()`. In
        every forward their operands are quantised per token row on the device (once per operand, shared by the text, image /
        condition and LoRA GEMMs that read it) and the GEMMs run on the fp8 tensor cores. The switched LoRA update of the
        quantised linears stays exact in form: its down-projection runs on the quantised operand, and its bf16 K extension is
        pre-divided by the scales the fp8 GEMM multiplies with (`_LoraPair.quantize_fp8`); the LoRA hooks (`enable_lora`,
        `set_scale`, `set_adapter`) keep working and rewrite those operands in place. x_embedder and its LoRA, the context /
        time / text embedders, the AdaLN GEMVs and their LoRA, norm_out / proj_out and attention stay bf16. Call after
        `load_state_dict`; afterwards `load_state_dict`, `lora_mode="epilogue"` and the sequence-parallel subclass with
        `sp_enabled=True` raise `UgError`. CUDA graphs captured over
        this model before the call point at released weights: capture them again."""
        if self.linear_dtype == FP8:
            return self
        if not self.lora:
            raise ops.UgError("call load_state_dict(..., adapters=..., condition_types=...) before quantize_fp8()")
        quantize_block_linears(self._ws, self.double + self.single)
        for i, w in enumerate(self.double):
            for key, lin in (("qkv", w.qkv), ("to_out", w.to_out), ("ff2", w.ff2)):
                self.lora[f"transformer_blocks.{i}.{key}"].quantize_fp8(lin[2])
        for i, w in enumerate(self.single):
            for key, lin in (("qkv", w.qkv), ("mlp", w.mlp), ("out", w.out)):
                self.lora[f"single_transformer_blocks.{i}.{key}"].quantize_fp8(lin[2])
        self.linear_dtype = FP8
        return self

    def lora_modules(self) -> List[LoraLayer]:
        """The LoRA carriers of every switched linear, in registration order — what the reference passes to `enable_lora`."""
        return list(self.lora_layers.values())

    # ---------------------------------------------------------------------------------------------------------
    def _workspace(self, B, S):
        key = (B, S)
        if key in self._bufs:  # one workspace per shape, never freed while the model lives (captured graphs point into them)
            self._buf = self._bufs[key]
            self._fp8_buffers(self._buf, B, S)
            return self._buf
        D, dev = self.inner_dim, self.device_
        z = lambda *s, dt=BF16: torch.empty(*s, device=dev, dtype=dt)  # noqa: E731
        self._buf = self._bufs[key] = types.SimpleNamespace(
            X=z(B, S, D), NX=z(B, S, D), QKV=z(B, S, 3 * D), AO=z(B, S, D), FF=z(B, S, 4 * D), CAT=z(B, S, 5 * D),
            LT=z(B, S, 3 * self.R, dt=torch.float32), LTW=z(B, S, self.groups * LORA_BLOCK), temb=z(B, D, dt=torch.float32), ctemb=z(B, D, dt=torch.float32),
            tmp=z(B, D, dt=torch.float32), NO=None, mod_plans={},
            rope=z(S, self.arch.attention_head_dim, dt=torch.float32))
        self._fp8_buffers(self._buf, B, S)
        return self._buf

    def _fp8_buffers(self, buf, B, S):
        """e4m3 operands (+ one fp32 scale per row) of the quantised block linears: LN output, attention output, FF and CAT.
        Added to the shape's workspace on its first fp8 forward; the bf16 buffers keep their addresses."""
        if self.linear_dtype != FP8 or hasattr(buf, "NXQ"):
            return
        D, dev = self.inner_dim, self.device_
        q = lambda w: (torch.empty(B, S, w, device=dev, dtype=FP8), torch.empty(B, S, device=dev, dtype=torch.float32))  # noqa: E731
        buf.NXQ, buf.AOQ, buf.FFQ, buf.CATQ = q(D), q(D), q(4 * D), q(5 * D)

    def _rec(self, name, t):
        if self.trace is not None:
            self.trace[name] = t.detach().float().clone()

    def _time_text(self, t_emb, pooled, out, tmp):
        w = self.time_text
        ops.gemv(t_emb, w.t1[0], w.t1[1], out=tmp, silu_out=True)
        ops.gemv(tmp, w.t2[0], w.t2[1], out=out)
        ops.gemv(pooled, w.p1[0], w.p1[1], out=tmp, silu_out=True)
        ops.gemv(tmp, w.p2[0], w.p2[1], out=out, accumulate=True)

    def _mod_layout(self, B: int, n: int):
        """fp32 element offsets of the per-block AdaLN tables inside one flat buffer: double block i -> [2 + n, B, 6D] (row 0 =
        text stream / norm1_context, row 1 = image, rows 2.. = conditions), single block i -> [1 + n, B, 3D]; then the LoRA
        down-projections t_g [jobs, B, Rp] and the [1 + n, B, D] conditioning vectors with their SiLU."""
        D, G = self.inner_dim, 1 + n
        off, dbl, sgl = 0, [], []
        for _ in self.double:
            dbl.append(off)
            off += (2 + n) * B * 6 * D
        for _ in self.single:
            sgl.append(off)
            off += G * B * 3 * D
        n_lt = (len(self.double) + len(self.single)) * G
        lt = off
        off += n_lt * B * 16
        tembs = off
        off += G * B * D
        stembs = off
        off += G * B * D
        return dbl, sgl, lt, tembs, stembs, off

    def _mod_plans(self, buf, B: int, n: int, flat: Optional[torch.Tensor] = None, pool=None):
        """Every AdaLN `linear(silu(temb))` of the step — all blocks, all streams, with the switched LoRA update of norm1.linear /
        norm.linear (enable_lora per stream, pyc L154-156, L168-170, L251-253) — as THREE grouped-GEMV launches over
        device-resident job tables instead of ~4 GEMVs per block and adapter group:
          main : W silu(tembs) + b for the image / condition rows of every block (batch (1 + n) B: one weight pass serves all streams)
          ctx  : norm1_context for the text rows (batch B) + the LoRA down-projections t_g = A_g silu(temb_g)
          lora : table[g] += B_g t_g  (accumulating jobs; runs after `ctx`)
        With `pool` (sequence parallelism) the flat buffer lives in the peer pool and every rank computes 1/P of each launch."""
        key = (B, n, id(pool), flat.data_ptr() if flat is not None else 0)
        mp = buf.mod_plans.get(key)
        if mp is not None:
            return mp
        D, G, dev, L = self.inner_dim, 1 + n, self.device_, self.lora
        dbl_off, sgl_off, lt_off, t_off, st_off, total = self._mod_layout(B, n)
        if flat is None:
            flat = torch.zeros(total, device=dev, dtype=torch.float32)
        mp = types.SimpleNamespace(flat=flat)
        mp.tembs = flat[t_off:t_off + G * B * D].view(G, B, D)
        mp.stembs = flat[st_off:st_off + G * B * D].view(G, B, D)
        main, ctx, lora = [], [], []
        lt_i = [0]

        def lora_jobs(pair: _LoraPair, rows_of_group):
            for g in range(G):
                t = flat[lt_off + lt_i[0] * B * 16:lt_off + (lt_i[0] + 1) * B * 16].view(B, 16)[:, :pair.rank]
                lt_i[0] += 1
                ctx.append((pair.a[g], None, mp.stembs[g], t, False))
                lora.append((pair.b[g], None, t, rows_of_group(g), False, True))

        mp.dbl, mp.sgl = [], []
        for i, w in enumerate(self.double):
            tab = flat[dbl_off[i]:dbl_off[i] + (2 + n) * B * 6 * D].view(2 + n, B, 6 * D)
            ctx.append((w.norm1_ctx[0], w.norm1_ctx[1], mp.stembs[0], tab[0], False))
            main.append((w.norm1[0], w.norm1[1], mp.stembs.view(G * B, D), tab[1:].view(G * B, 6 * D), False))
            lora_jobs(L[f"transformer_blocks.{i}.norm1"], lambda g, tab=tab: tab[1 + g])
            mp.dbl.append((tab[0], tab[1:]))
        for i, w in enumerate(self.single):
            tab = flat[sgl_off[i]:sgl_off[i] + G * B * 3 * D].view(G, B, 3 * D)
            main.append((w.norm[0], w.norm[1], mp.stembs.view(G * B, D), tab.view(G * B, 3 * D), False))
            lora_jobs(L[f"single_transformer_blocks.{i}.norm"], lambda g, tab=tab: tab[g])
            mp.sgl.append(tab)
        mp.main, mp.ctx, mp.lora = (ops.GemvPlan(j, dev, pool=pool) for j in (main, ctx, lora))
        buf.mod_plans[key] = mp
        return mp

    def _mods(self, buf, B: int, n: int):
        """Fill the conditioning vectors' SiLU and launch the AdaLN job tables (see _mod_plans); returns the plan record with the
        per-block tables. The sequence-parallel subclass shards the launches and all-gathers through the peer pool."""
        mp = self._mod_plans(buf, B, n)
        mp.tembs[0].copy_(buf.temb)
        for j in range(n):
            mp.tembs[1 + j].copy_(buf.ctemb)
        ops.silu(mp.tembs, mp.stembs)
        ops.gemv_grouped(mp.main)
        ops.gemv_grouped(mp.ctx)
        ops.gemv_grouped(mp.lora)
        return mp

    @staticmethod
    def _chunks(row: torch.Tensor, n_chunks: int) -> List[torch.Tensor]:
        D = row.shape[-1] // n_chunks
        return [row[:, i * D:(i + 1) * D] for i in range(n_chunks)]

    @staticmethod
    def _rows(q, lo: int, hi: Optional[int] = None):
        """Rows [lo, hi) of a quantised operand (e4m3 [B, S, K], scales [B, S]); None stays None (bf16 weight set)."""
        return None if q is None else (q[0][:, lo:hi], q[1][:, lo:hi])

    def _linear(self, w, x, q, out, **kw):
        """Plain block linear: the bf16 GEMM of x, or for a quantised (W e4m3, bias, w_scale) the fp8 GEMM of q = (e4m3, scales)."""
        if len(w) == 3:
            return ops.gemm_fp8(q[0], q[1], w[0], w[2], out=out, bias=w[1], variant=self.gemm_variant, **kw)
        return ops.gemm(x, w[0], out=out, bias=w[1], variant=self.gemm_variant, **kw)

    def _lora_gemm(self, buf, x, w, pair: _LoraPair, seg_bounds, seg_group, out, q=None, **kw):
        """Main GEMM with the switched low-rank update fused into it. A quantised linear (W e4m3, bias, w_scale) takes the
        quantised operand q = (e4m3 rows, row scales) of x: the masked fp8 down-projection writes (x / a_s) A^T into the K
        extension, whose W2 is pre-divided by w_scale (see _LoraPair.quantize_fp8)."""
        if len(w) == 3:
            tw = buf.LTW[:, :x.shape[1]]
            ops.gemm_fp8(q[0], None, pair.aq, pair.aws, out=tw, variant=self.gemm_variant,
                         colmask=dict(block=LORA_BLOCK, seg_bounds=seg_bounds, seg_group=seg_group))
            return ops.gemm_fp8(q[0], q[1], w[0], w[2], out=out, bias=w[1], variant=self.gemm_variant, a2=tw, w2=pair.w2,
                                seg_bounds=seg_bounds if kw.get("gate_seg_stride") else None, **kw)
        if self.lora_mode == "mma":
            tw = buf.LTW[:, :x.shape[1]]
            if self.lora_down_mode == "mma" and x.shape[-1] >= 256:
                # down-projection on the tensor cores too: x @ [A_0; A_1; ...]^T, each row masked to its own group's block
                ops.gemm(x, pair.aw, out=tw, variant=self.gemm_variant, colmask=dict(block=LORA_BLOCK, seg_bounds=seg_bounds, seg_group=seg_group))
            else:
                ops.lora_down_wide(x, pair.a, seg_bounds, seg_group, out=tw, block=LORA_BLOCK)
            return ops.gemm(x, w[0], out=out, bias=w[1], variant=self.gemm_variant, a2=tw, w2=pair.bw,
                            seg_bounds=seg_bounds if kw.get("gate_seg_stride") else None, **kw)
        rt = pair.n_sub * pair.rank
        t = buf.LT[:, :x.shape[1], :rt]
        ops.lora_down(x, pair.a, seg_bounds, seg_group, out=t)
        return ops.gemm(x, w[0], out=out, bias=w[1], variant=self.gemm_variant,
                        lora=dict(t=t, b=pair.b, rank=pair.rank, block_n=pair.n_each, seg_bounds=seg_bounds,
                                  seg_group=seg_group), **kw)

    def _fused_qk(self) -> bool:
        """QK-RMSNorm + RoPE inside the projection GEMMs' epilogue (as in the S-variant); the LoRA-in-epilogue mode keeps the
        separate pass (its epilogue carries per-row LoRA state instead)."""
        return self.fuse_qk_norm and self.lora_mode == "mma"

    def _qk_norm(self, buf, rms, lo: int, hi: int):
        if not self._fused_qk():
            return None
        return dict(weight=rms, head_dim=self.arch.attention_head_dim, d=self.inner_dim, cos_sin=buf.rope[lo:hi], eps=1e-6)

    def _attention(self, buf, parts, out_name: str, bounds, vis):
        """QK-RMSNorm + RoPE on the q|k columns of row ranges `parts` = [(lo, hi, rms_weight)] (in place here unless the
        projection GEMMs already did it in their epilogue), then the joint attention with the segment-visibility rule ->
        buf.AO, or the first D columns of buf.CAT (single blocks).
        The sequence-parallel subclass (parallel.py) fuses both steps with the Ulysses exchange over peer memory."""
        a, D = self.arch, self.inner_dim
        H, dh = a.num_attention_heads, a.attention_head_dim
        if not self._fused_qk():
            for lo, hi, rms in parts:
                ops.qk_rmsnorm_rope(buf.QKV[:, lo:hi, :2 * D], 2 * H, dh, rms, buf.rope[lo:hi], heads_per_weight=H)
        out = buf.AO if out_name == "AO" else buf.CAT[:, :, :D]
        ops.attention(buf.QKV[:, :, 0:D], buf.QKV[:, :, D:2 * D], buf.QKV[:, :, 2 * D:], out, H, dh,
                      seg_bounds=bounds, seg_visible=vis, variant=self.attn_variant)

    # ---------------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, hidden_states, condition_latents, condition_ids, condition_types, encoder_hidden_states,
                pooled_projections, timestep, img_ids, txt_ids, c_t: float = 0.0, return_condition_latents: bool = False,
                **kwargs):
        """`return_condition_latents` (2DModel L203-209): also return the condition streams after the last single block."""
        a, D = self.arch, self.inner_dim
        H, dh = a.num_attention_heads, a.attention_head_dim
        dev = self.device_
        if list(condition_types) != self.condition_types[:len(condition_types)]:
            raise ops.UgError(f"condition_types {list(condition_types)} do not match the loaded adapters {self.condition_types}")
        if self.linear_dtype == FP8 and self.lora_mode != "mma":
            raise ops.UgError(f'lora_mode="{self.lora_mode}" on an fp8-quantised model: its switched update runs as the fp8 GEMM\'s '
                              'K extension (lora_mode="mma")')
        self._sync_lora()  # scale tables follow the LoRA hooks (lora_switching_module.enable_lora / LoraLayer.set_scale)
        n = len(condition_latents)
        B, N, _ = hidden_states.shape
        T = encoder_hidden_states.shape[1]
        ncs = [c.shape[1] for c in condition_latents]
        bounds = [0, T, T + N]
        for m in ncs:
            bounds.append(bounds[-1] + m)
        S = bounds[-1]
        buf = self._workspace(B, S)
        f32 = lambda t: t.to(device=dev, dtype=torch.float32).contiguous()  # noqa: E731
        gv = self.gemm_variant
        seg = lambda i: buf.X[:, bounds[i]:bounds[i + 1]]  # noqa: E731  (0 = txt, 1 = img, 2+j = cond j)
        # visibility: txt,img -> all ; c_i -> {txt,img,c_i}  (strict: c_i -> {c_i})
        nseg = 2 + n
        vis = [(1 << nseg) - 1, (1 << nseg) - 1] + [(1 << (2 + j)) | (0 if self.strict_mask else 0b11) for j in range(n)]

        # ---- embeddings (2DModel L92-99, L112-121, L144-149) ----
        hs = ops.to_bf16(hidden_states.to(dev).contiguous())
        es = ops.to_bf16(encoder_hidden_states.to(dev).contiguous())
        self._lora_gemm(buf, hs, self.x_embedder_w, self.lora["x_embedder"], [0, N], [0], seg(1))
        for j, c in enumerate(condition_latents):
            cj = ops.to_bf16(c.to(dev).contiguous())
            self._lora_gemm(buf, cj, self.x_embedder_w, self.lora["x_embedder"], [0, ncs[j]], [1 + j], seg(2 + j))
        ops.gemm(es, self.context_embedder_w[0], out=seg(0), bias=self.context_embedder_w[1], variant=gv)
        pooled = f32(pooled_projections)
        t1000 = f32(timestep) * 1000.0
        self._time_text(ops.timestep_embedding(t1000), pooled, buf.temb, buf.tmp)
        self._time_text(ops.timestep_embedding(torch.ones_like(t1000) * (c_t * 1000.0)), pooled, buf.ctemb, buf.tmp)
        ids = torch.cat([f32(txt_ids), f32(img_ids)] + [f32(ci) for ci in condition_ids], 0)
        ops.rope_table(ids, a.axes_dims_rope, a.theta, out=buf.rope)

        img_cond_bounds = [b - T for b in bounds[1:]]          # segments of rows [T, S): img, c_1..c_n
        img_cond_groups = list(range(0, 1 + n))               # den, c_1..c_n
        all_bounds = [0, T + N] + bounds[3:]                   # single blocks: [txt|img] share the denoising adapters
        all_groups = list(range(0, 1 + n))

        # ---- AdaLN vectors of every block and stream (temb / cond_temb are step constants): three grouped-GEMV launches ----
        L = self.lora
        mp = self._mods(buf, B, n)
        dbl_mods, sgl_mods = mp.dbl, mp.sgl
        # quantised block linears: one e4m3 operand (+ row scales) per LN output / attention output / FF / CAT, shared by every
        # GEMM that reads those rows (text, image / condition and LoRA down-projection)
        fp8 = self.linear_dtype == FP8
        qn, qa, qf, qc = ((buf.NXQ, buf.AOQ, buf.FFQ, buf.CATQ) if fp8 else (None,) * 4)
        rows = self._rows

        def ln(shift, scale, seg_bounds, seg_stride):
            if fp8:
                ops.ln_modulate_segs_fp8(buf.X, qn[0], qn[1], shift, scale, seg_bounds, seg_stride)
            else:
                ops.ln_modulate_segs(buf.X, buf.NX, shift, scale, seg_bounds, seg_stride)

        def quant(x, q):
            if fp8:
                ops.quant_rows_fp8(x, q[0], q[1])

        for i, w in enumerate(self.double):  # ---- block_forward ----
            p = f"transformer_blocks.{i}"
            # the image / condition streams' AdaLN vectors live in ONE [1+n, B, 6D] table so that the gated GEMMs below can
            # cover all of them in a single launch (ug_gemm_args.gate_seg_stride)
            m_txt = self._chunks(dbl_mods[i][0], 6)
            m_img = self._chunks(dbl_mods[i][1][0], 6)
            m_c = [self._chunks(dbl_mods[i][1][1 + j], 6) for j in range(n)]
            mods = [m_txt, m_img] + m_c
            ln(m_txt[0], m_txt[1], bounds, B * 6 * D)
            self._linear(w.add_qkv, buf.NX[:, :T], rows(qn, 0, T), buf.QKV[:, :T], qk_norm=self._qk_norm(buf, w.rms_ctx, 0, T))
            self._lora_gemm(buf, buf.NX[:, T:], w.qkv, L[p + ".qkv"], img_cond_bounds, img_cond_groups, buf.QKV[:, T:],
                            q=rows(qn, T, S), qk_norm=self._qk_norm(buf, w.rms, T, S))
            self._attention(buf, [(0, T, w.rms_ctx), (T, S, w.rms)], "AO", bounds, vis)
            quant(buf.AO, qa)
            self._linear(w.to_add_out, buf.AO[:, :T], rows(qa, 0, T), seg(0), gate=m_txt[2], residual=seg(0))
            # to_out[0]: LoRA group AND gate switched per stream inside one launch over [img | c_1 .. c_n]
            if not self.add_cond_attn:
                self._lora_gemm(buf, buf.AO[:, T:], w.to_out, L[p + ".to_out"], img_cond_bounds, img_cond_groups, buf.X[:, T:],
                                q=rows(qa, T, S), gate=m_img[2], gate_seg_stride=B * 6 * D, residual=buf.X[:, T:])
            else:
                # add_cond_attn (pyc L201-202): the GATED condition attention outputs are also added into the image stream, so
                # they are materialised once (gated, no residual) and added to both streams
                if any(m != N for m in ncs):
                    raise ops.UgError("add_cond_attn adds condition attention outputs to the image stream: needs Nc == N")
                g_out = buf.NX[:, T:]  # free until the MLP's LayerNorm pass
                self._lora_gemm(buf, buf.AO[:, T:], w.to_out, L[p + ".to_out"], img_cond_bounds, img_cond_groups, g_out,
                                q=rows(qa, T, S), gate=m_img[2], gate_seg_stride=B * 6 * D)
                ops.add(seg(1), g_out[:, :N], seg(1))
                for j in range(n):
                    gj = g_out[:, img_cond_bounds[1 + j]:img_cond_bounds[2 + j]]
                    ops.add(seg(2 + j), gj, seg(2 + j))
                    ops.add(seg(1), gj, seg(1))
            ln(m_txt[3], m_txt[4], bounds, B * 6 * D)
            # both up-projections first (disjoint rows of FF), so that one quantisation pass covers FF
            self._linear(w.ffc1, buf.NX[:, :T], rows(qn, 0, T), buf.FF[:, :T], act=UG_ACT_GELU_TANH)
            self._linear(w.ff1, buf.NX[:, T:], rows(qn, T, S), buf.FF[:, T:], act=UG_ACT_GELU_TANH)
            quant(buf.FF, qf)
            self._linear(w.ffc2, buf.FF[:, :T], rows(qf, 0, T), seg(0), gate=m_txt[5], residual=seg(0))
            self._lora_gemm(buf, buf.FF[:, T:], w.ff2, L[p + ".ff2"], img_cond_bounds, img_cond_groups, buf.X[:, T:],
                            q=rows(qf, T, S), gate=m_img[5], gate_seg_stride=B * 6 * D, residual=buf.X[:, T:])
            self._rec(f"double.{i}.hidden", seg(1)); self._rec(f"double.{i}.context", seg(0))
            for j in range(n):
                self._rec(f"double.{i}.cond{j}", seg(2 + j))

        for i, w in enumerate(self.single):  # ---- single_block_forward ----
            p = f"single_transformer_blocks.{i}"
            m_x = self._chunks(sgl_mods[i][0], 3)
            m_c = [self._chunks(sgl_mods[i][1 + j], 3) for j in range(n)]
            mods = [m_x] + m_c
            ln(m_x[0], m_x[1], all_bounds, B * 3 * D)
            self._lora_gemm(buf, buf.NX, w.qkv, L[p + ".qkv"], all_bounds, all_groups, buf.QKV, q=qn,
                            qk_norm=self._qk_norm(buf, w.rms, 0, S))
            self._lora_gemm(buf, buf.NX, w.mlp, L[p + ".mlp"], all_bounds, all_groups, buf.CAT[:, :, D:], q=qn, act=UG_ACT_GELU_TANH)
            self._attention(buf, [(0, S, w.rms)], "CAT", bounds, vis)
            quant(buf.CAT, qc)
            self._lora_gemm(buf, buf.CAT, w.out, L[p + ".out"], all_bounds, all_groups, buf.X, q=qc, gate=m_x[2],
                            gate_seg_stride=B * 3 * D, residual=buf.X)
            self._rec(f"single.{i}.hidden", buf.X[:, :T + N])
            for j in range(n):
                self._rec(f"single.{i}.cond{j}", seg(2 + j))

        e = torch.empty(B, 2 * D, device=dev, dtype=torch.float32)
        ops.gemv(buf.temb, self.norm_out_w[0], self.norm_out_w[1], out=e, silu_in=True)
        no = torch.empty(B, N, D, device=dev, dtype=BF16)
        ops.ln_modulate(seg(1), no, e[:, D:], e[:, :D])  # AdaLayerNormContinuous: scale first, then shift
        out = ops.gemm(no, self.proj_out_w[0], bias=self.proj_out_w[1], variant=gv)
        self._rec("velocity", out)
        if return_condition_latents:
            return out, [seg(2 + j).clone() for j in range(n)]
        return out
