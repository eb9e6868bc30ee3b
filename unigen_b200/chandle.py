"""ctypes view of the whole-step C handle (include/unigen_b200.h `ug_flux_*`, csrc/ug_flux.cu): what a non-Python host does —
create a handle from the architecture, bind every weight pointer under its reference state-dict name, size and supply one
workspace, call `ug_flux_forward` — driven from Python so that tests can compare it with `UniGenFlux.forward` (bit-identical:
same kernels, same order) and INTEGRATION.md can show a runnable binding. torch only supplies the device buffers."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence

import torch

from . import _lib, ops
from ._lib import FluxDesc, FluxInputs, FluxOutputs, check


class FluxStepHandle:
    """`ug_flux` handle over the weights of a native `UniGenFlux` (or any state dict laid out the way the header requires)."""

    def __init__(self, model):
        a = model.arch
        if getattr(model, "use_consis_module", False) and model.use_shared_expert:
            raise ops.UgError("ug_flux handle: use_consis_module is sequenced by the Python host only (unigen_b200.model)")
        if getattr(model, "linear_dtype", torch.bfloat16) != torch.bfloat16:
            raise ops.UgError("ug_flux handle: fp8-quantised block linears (quantize_fp8) run on the Python host only (unigen_b200.model)")
        d = FluxDesc()
        d.num_layers, d.num_single_layers, d.heads, d.head_dim = a.num_layers, a.num_single_layers, a.num_attention_heads, a.attention_head_dim
        d.in_channels, d.joint_dim, d.pooled_dim, d.guidance_embeds = a.in_channels, a.joint_attention_dim, a.pooled_projection_dim, int(a.guidance_embeds)
        for i, v in enumerate(a.axes_dims_rope):
            d.axes_dims_rope[i] = v
        d.theta = a.theta
        d.n_ctrl_double, d.n_ctrl_single = len(model.ctrl_double), len(model.ctrl_single)
        d.experts, d.condition_nums = model.expert_nums, model.condition_nums
        d.use_shared_expert = int(model.use_shared_expert)
        d.single_add = int(model.single_block_control_method != "overall_add")
        d.use_pooled_prompt_embeds = int(model.use_pooled_prompt_embeds)
        self.lib = _lib.load()
        self.h = C.c_void_p()
        check(self.lib.ug_flux_create(C.byref(d), C.byref(self.h)), "ug_flux_create")
        self.model, self.desc = model, d
        self._keep = []
        self.bind_state_dict(model.state_dict())
        self._ws: Dict[tuple, torch.Tensor] = {}

    def bind_state_dict(self, sd: Dict[str, torch.Tensor]) -> None:
        for name, t in sd.items():
            if not t.is_cuda or not t.is_contiguous():
                raise ops.UgError(f"{name}: weights must be contiguous CUDA tensors")
            dtype = {torch.bfloat16: 0, torch.float32: 1}[t.dtype]
            shape = (C.c_int64 * 4)(*list(t.shape) + [0] * (4 - t.dim()))
            check(self.lib.ug_flux_bind_weight(self.h, name.encode(), t.data_ptr(), dtype, shape, t.dim()), f"ug_flux_bind_weight({name})")
            self._keep.append(t)

    def workspace(self, B: int, N: int, T: int) -> torch.Tensor:
        key = (B, N, T)
        if key not in self._ws:
            n = int(self.lib.ug_flux_workspace_bytes(self.h, B, N, T))
            self._ws[key] = torch.empty(n, dtype=torch.uint8, device=self.model.device)
        return self._ws[key]

    @torch.no_grad()
    def forward(self, hidden_states, condition_hidden_states, encoder_hidden_states, pooled_projections, condition_pooled_projections,
                timestep, img_ids, txt_ids, condition_ids, rts_uniform, guidance=None, conditioning_scale: float = 1.0):
        """Same tensors as `UniGenFlux.forward` (lists for several conditions); returns (velocity, moe_loss, expert_counts)."""
        dev = self.model.device
        bf = lambda t: ops.to_bf16(t.to(dev).contiguous())  # noqa: E731
        f32 = lambda t: t.to(device=dev, dtype=torch.float32).contiguous()  # noqa: E731
        sq = lambda t: t[0] if t.dim() == 3 else t  # noqa: E731
        as_list = lambda v: list(v) if isinstance(v, (list, tuple)) else [v]  # noqa: E731
        hs, es = bf(hidden_states), bf(encoder_hidden_states)
        B, N, _ = hs.shape
        T = es.shape[1]
        inp = FluxInputs()
        inp.batch, inp.n_img, inp.n_txt, inp.conditioning_scale = B, N, T, float(conditioning_scale)
        keep = [hs, es, f32(pooled_projections), f32(timestep).reshape(-1), f32(sq(img_ids)), f32(sq(txt_ids))]
        inp.hidden_states, inp.encoder_hidden_states, inp.pooled_projections = hs.data_ptr(), es.data_ptr(), keep[2].data_ptr()
        inp.timestep, inp.timestep_stride = keep[3].data_ptr(), (1 if keep[3].numel() > 1 else 0)
        inp.img_ids, inp.txt_ids = keep[4].data_ptr(), keep[5].data_ptr()
        if guidance is not None:
            keep.append(f32(guidance))
            inp.guidance = keep[-1].data_ptr()
        for c, (cs, cp, ci, u) in enumerate(zip(as_list(condition_hidden_states), as_list(condition_pooled_projections),
                                                as_list(condition_ids), as_list(rts_uniform))):
            t = [bf(cs if cs.dim() == 3 else cs.unsqueeze(0)), f32(cp if cp.dim() == 2 else cp.unsqueeze(0)), f32(sq(ci)), f32(u)]
            keep += t
            inp.condition_hidden_states[c], inp.condition_pooled_projections[c] = t[0].data_ptr(), t[1].data_ptr()
            inp.condition_ids[c], inp.rts_uniform[c] = t[2].data_ptr(), t[3].data_ptr()
        out = FluxOutputs()
        vel = torch.empty(B, N, self.model.arch.in_channels, device=dev, dtype=torch.bfloat16)
        counts = torch.empty(self.model.expert_nums, device=dev, dtype=torch.int64)
        l_aux = torch.empty(1, device=dev, dtype=torch.float32)
        out.velocity, out.expert_counts, out.l_aux = vel.data_ptr(), counts.data_ptr(), l_aux.data_ptr()
        ws = self.workspace(B, N, T)
        check(self.lib.ug_flux_forward(self.h, C.byref(inp), C.byref(out), ws.data_ptr(), ws.numel(), ops._stream()), "ug_flux_forward")
        del keep
        return vel, l_aux[0] * 0.1, counts

    def close(self):
        if self.h:
            torch.cuda.synchronize()
            self.lib.ug_flux_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass
