"""GPU checks of the opt-in fp8 (e4m3, row-wise scaled) joint-block linears of the SD3.5 denoiser (`UniGenSD3.quantize_fp8()`):
the fp8 kernel paths SD3.5 reaches and nothing else does (the fused QK-RMSNorm epilogue without RoPE, K = 1536 / 6144 with
batched row scales, the fp8 LayerNorm at d = 1536), the interface, a quantised tiny model free-running against the fp32 oracle
whose block linears are fake-quantised the same way, every quantised block kind at SD3.5-medium width teacher-forced, and
graph replay / the whole-loop CFG graph / the pipeline entry on a quantised model."""
import dataclasses
import sys
from pathlib import Path

import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, str(Path(__file__).resolve().parent))
from test_fp8_cpu import dequant_ref, quant_rows_ref  # noqa: E402
from test_sd3_gpu import _dev, _setup, rel_l2  # noqa: E402

pytestmark = pytest.mark.gpu
FP8 = torch.float8_e4m3fn
BATCH, N_IMG, N_TXT, D = 4, 4096, 333, 1536  # cfg5: CFG-doubled batch 4, 1024^2 latents, 333 text tokens, SD3.5-medium width


def rnd(*shape, scale=1.0):
    return (torch.randn(*shape, device="cuda") * scale).to(torch.bfloat16)


def same_bytes(a, b):
    return torch.equal(a.view(torch.uint8).cpu(), b.view(torch.uint8).cpu())


@pytest.fixture(autouse=True)
def _seed():
    torch.manual_seed(0)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False


# ---------------------------------------------------------------------------------------------------------------------------
# kernel paths at the SD3.5 shapes
# ---------------------------------------------------------------------------------------------------------------------------
def _operands(ug, B, M, K, N):
    a, w = rnd(B, M, K), rnd(N, K, scale=K ** -0.5)
    qa, sa = ug.quant_rows_fp8(a)
    qw, sw = ug.quant_rows_fp8(w)
    assert sa.shape == (B, M)  # batched [B, rows] activation scales
    return qa, sa, qw, sw, dequant_ref(qa.float(), sa), dequant_ref(qw.float(), sw)


@pytest.mark.parametrize("variant", [0, 1, 2, 4, 5])
def test_gemm_fp8_fused_qk_rmsnorm_without_rope(ug, variant):
    """q|k|v projection of the joint rows (4 x (4096 + 333)) with the per-head RMSNorm (head_dim 64) in the epilogue and no RoPE
    table (SD3.5 has none): fp32 RMSNorm of the dequantised product on q / k, the plain product on v."""
    rows, H, dh = N_IMG + N_TXT, D // 64, 64
    qa, sa, qw, sw, ad, wd = _operands(ug, BATCH, rows, D, 3 * D)
    bias = rnd(3 * D)
    nw = (1 + 0.1 * torch.randn(2, dh)).to(torch.bfloat16).cuda()
    out = ug.gemm_fp8(qa, sa, qw, sw, bias=bias, variant=variant, qk_norm=dict(weight=nw, head_dim=dh, d=D, cos_sin=None, eps=1e-6))
    full = ad @ wd.t() + bias.float()
    y = full[:, :, :2 * D].reshape(BATCH, rows, 2, H, dh)
    want = (y * torch.rsqrt(y.pow(2).mean(-1, keepdim=True) + 1e-6) * nw.float()[None, None, :, None, :]).reshape(BATCH, rows, 2 * D)
    assert rel_l2(out[:, :, :2 * D], want) < 4e-3
    assert rel_l2(out[:, :, 2 * D:], full[:, :, 2 * D:]) < 6e-3


def test_gemm_fp8_fused_qk_rmsnorm_refuses_the_128_column_staged_tile(ug):
    qa, sa, qw, sw, _, _ = _operands(ug, 1, 256, D, 3 * D)
    nw = torch.ones(2, 64, device="cuda", dtype=torch.bfloat16)
    with pytest.raises(ug.UgError):
        ug.gemm_fp8(qa, sa, qw, sw, variant=6, qk_norm=dict(weight=nw, head_dim=64, d=D, cos_sin=None, eps=1e-6))


# (K, N, epilogue) of the image-stream block linears: to_out (and attn2.to_out), ff.net.0 (GELU), ff.net.2 (K = 4D)
EPILOGUE_SHAPES = [(D, D, "gate_residual"), (D, 4 * D, "gelu"), (4 * D, D, "gate_residual"), (D, D, "bias")]


@pytest.mark.parametrize("variant", [0, 1, 2, 3, 4, 5, 6])
@pytest.mark.parametrize("k,n,epi", EPILOGUE_SHAPES)
def test_gemm_fp8_sd3_shapes_epilogues(ug, variant, k, n, epi):
    """4 x 4096 image rows with batched [4, 4096] row scales at K = 1536 and K = 6144, in the epilogue each linear uses."""
    qa, sa, qw, sw, ad, wd = _operands(ug, BATCH, N_IMG, k, n)
    bias = rnd(n)
    acc = ad @ wd.t() + bias.float()
    if epi == "bias":
        out, want = ug.gemm_fp8(qa, sa, qw, sw, bias=bias, variant=variant), acc
    elif epi == "gelu":
        out = ug.gemm_fp8(qa, sa, qw, sw, bias=bias, act=ug.UG_ACT_GELU_TANH, variant=variant)
        want = F.gelu(acc, approximate="tanh")
    else:
        gate = torch.randn(BATCH, n, device="cuda")
        out = rnd(BATCH, N_IMG, n)
        want = out.float() + gate[:, None] * acc
        ug.gemm_fp8(qa, sa, qw, sw, out=out, bias=bias, gate=gate, residual=out, variant=variant)  # in place, as the blocks run it
    assert rel_l2(out, want) < 6e-3
    assert (out.float() - want).abs().max().item() < 0.25  # every tile written once


@pytest.mark.parametrize("B,rows", [(BATCH, N_IMG + N_TXT), (2, 333), (1, 1000)])
def test_ln_modulate_fp8_d1536_equals_quantised_ln_modulate(ug, B, rows):
    x = rnd(B, rows, D, scale=3.0)
    shift, scale = torch.randn(B, D, device="cuda") * 0.5, torch.randn(B, D, device="cuda") * 0.5
    nx = torch.empty_like(x)
    ug.ln_modulate(x, nx, shift, scale)
    qw, sw = ug.quant_rows_fp8(nx)
    q = torch.empty(B, rows, D, device="cuda", dtype=FP8)
    s = torch.empty(B, rows, device="cuda")
    ug.ln_modulate_fp8(x, q, s, shift, scale)
    assert same_bytes(q, qw) and torch.equal(s, sw)


def test_fp8_operands_of_the_context_rows_as_the_block_passes_them(ug):
    """Context rows [N, N + T) of the joint workspace buffers: LN of X[:, N:] into NXQ[:, N:] / NXS[:, N:] (modulation chunks are
    views into the wide MOD table), and FF[:, N:] (K = 4D) into FFQ[:, N:]; nothing outside the views is written."""
    S, mod = N_IMG + N_TXT, torch.randn(BATCH, 6 * D, device="cuda")
    x = rnd(BATCH, S, D, scale=2.0)
    shift, scale = mod[:, :D], mod[:, D:2 * D]
    nx = torch.empty(BATCH, N_TXT, D, device="cuda", dtype=torch.bfloat16)
    ug.ln_modulate(x[:, N_IMG:], nx, shift, scale)
    qw, sw = ug.quant_rows_fp8(nx)
    nxq, nxs = torch.zeros(BATCH, S, D, device="cuda", dtype=FP8), torch.zeros(BATCH, S, device="cuda")
    ug.ln_modulate_fp8(x[:, N_IMG:], nxq[:, N_IMG:], nxs[:, N_IMG:], shift, scale)
    assert same_bytes(nxq[:, N_IMG:], qw) and torch.equal(nxs[:, N_IMG:], sw)
    assert (nxq[:, :N_IMG].view(torch.uint8) == 0).all() and (nxs[:, :N_IMG] == 0).all()
    ff = rnd(BATCH, S, 4 * D)
    ffq, ffs = torch.zeros(BATCH, S, 4 * D, device="cuda", dtype=FP8), torch.zeros(BATCH, S, device="cuda")
    ug.quant_rows_fp8(ff[:, N_IMG:], ffq[:, N_IMG:], ffs[:, N_IMG:])
    qr, sr = quant_rows_ref(ff[:, N_IMG:].cpu())
    assert same_bytes(ffq[:, N_IMG:], qr) and torch.equal(ffs[:, N_IMG:].cpu(), sr)
    assert (ffq[:, :N_IMG].view(torch.uint8) == 0).all()


# ---------------------------------------------------------------------------------------------------------------------------
# model
# ---------------------------------------------------------------------------------------------------------------------------
QUANT_JOINT = (".attn.to_q", ".attn.to_k", ".attn.to_v", ".attn.add_q_proj", ".attn.add_k_proj", ".attn.add_v_proj",
               ".attn.to_out.0", ".attn.to_add_out", ".attn2.to_q", ".attn2.to_k", ".attn2.to_v", ".attn2.to_out.0",
               ".ff.net.0.proj", ".ff.net.2", ".ff_context.net.0.proj", ".ff_context.net.2")


def _quantised_prefix(prefix):
    head, _, rest = prefix.partition(".")
    idx, _, name = rest.partition(".")
    return head in ("transformer_blocks", "control_transformer_blocks") and idx.isdigit() and "." + name in QUANT_JOINT


def _covered_weights(dual, context_pre_only):
    """Weight views quantize_fp8() takes out of one joint block: q, k, v, add_q, add_k, add_v, to_out, ff.net.0, ff.net.2;
    + to_add_out, ff_context.net.0, ff_context.net.2 unless context_pre_only; + attn2 q, k, v, to_out with dual attention."""
    return 9 + (0 if context_pre_only else 3) + (4 if dual else 0)


@pytest.fixture
def fake_quant_sd3_oracle(monkeypatch):
    """`linear` of both oracle modules (the SD3 oracle imports it by name, feed_forward calls oracle.unigen_oracle.linear) with x
    quantised per token row (of its bf16 value, as the native operands are bf16) and W per output channel by the reference
    quantiser, for the quantised joint-block linears only."""
    from oracle import unigen_oracle as O
    from oracle import unigen_sd3_oracle as O3
    plain = O.linear

    def linear(sd, prefix, x):
        if not _quantised_prefix(prefix):
            return plain(sd, prefix, x)
        linear.quantised_calls += 1
        xd = dequant_ref(*quant_rows_ref(x.to(torch.bfloat16)))
        return F.linear(xd, dequant_ref(*quant_rows_ref(sd[prefix + ".weight"].to(torch.bfloat16))), sd.get(prefix + ".bias"))

    linear.quantised_calls = 0
    monkeypatch.setattr(O, "linear", linear)
    monkeypatch.setattr(O3, "linear", linear)
    return linear


def test_quantize_fp8_interface():
    from unigen_b200.model import FP8 as MFP8
    cfg, sd, inp, oracle, model = _setup()
    assert model.linear_dtype == torch.bfloat16
    n_before = len(model.state_dict())
    assert model.quantize_fp8() is model and model.linear_dtype == MFP8
    after = model.state_dict()
    assert model.quantize_fp8() is model and model.state_dict().keys() == after.keys()  # a second call changes nothing
    L = cfg.num_layers
    want = sum(_covered_weights(i in cfg.dual_attention_layers, i == L - 1) for i in range(L))           # base blocks
    want += sum(_covered_weights(j in cfg.dual_attention_layers, False) for j in range(L))              # control blocks
    assert n_before - len(after) == want
    assert not any(k.endswith(".weight") and _quantised_prefix(k[:-len(".weight")]) for k in after)
    assert all(k[:-len(".weight")] + ".bias" in after for k in sd if k.endswith(".weight") and _quantised_prefix(k[:-len(".weight")]))
    assert all(w.fp8 for w in model.blocks + model.ctrl_blocks) and not any(w.fp8 for w in model.shared)
    assert model.blocks[0].attn2.qkv[0].dtype == FP8 and model.blocks[-1].attn.to_add_out is None
    assert model.shared[1].attn2.qkv[0].dtype == torch.bfloat16 and model.experts[0].qkv_w.dtype == torch.bfloat16
    assert "shared_expert.0.attn.to_q.weight" in after and "controlnet_add_blocks.0.weight" in after
    assert len(list(model.parameters())) == len(after)


def test_refusals():
    from unigen_b200.ops import UgError
    from unigen_b200.sd3 import SD3Arch, UniGenSD3
    cfg, sd, inp, oracle, model = _setup()
    with pytest.raises(UgError):
        UniGenSD3(SD3Arch.tiny(), device="cuda").quantize_fp8()  # before init_condition_block
    model.quantize_fp8()
    with pytest.raises(UgError):
        model.load_state_dict(sd)
    with pytest.raises(UgError):
        model.init_random_(seed=1)
    with pytest.raises(UgError):
        model.init_control_param()


@pytest.mark.parametrize("use_modulate,use_shared", [(False, True), (True, True), (False, False)])
def test_tiny_quantised_model_matches_fake_quant_oracle(fake_quant_sd3_oracle, use_modulate, use_shared):
    """SD3Config.tiny() (4 layers, 2 dual, last context_pre_only) free-running against the fp32 oracle with fake-quantised block
    linears, with the bars of the bf16 model: every trace point rel-L2 <= 1e-2, velocity cosine >= 0.999, routing >= 99 %."""
    from oracle import unigen_sd3_oracle as O
    from unigen_b200.sd3 import shipped_control_params
    cfg = dataclasses.replace(O.SD3Config.tiny(), use_modulate=use_modulate, use_shared_expert=use_shared)
    params = dict(shipped_control_params(), use_modulate=use_modulate, use_shared_expert=use_shared)
    cfg, sd, inp, oracle, model = _setup(batch=2, seed=7, cfg=cfg, control_params=params)
    model.quantize_fp8()
    want, want_losses, _ = oracle.forward(**inp)
    assert fake_quant_sd3_oracle.quantised_calls >= 2 * cfg.num_layers * 9
    model.trace = {}
    got, losses, _ = model(**_dev(inp))
    torch.cuda.synchronize()
    worst = {name: rel_l2(model.trace[name], ref) for name, ref in oracle.trace.items()
             if name in model.trace and name.split(".")[-1] not in ("expert_idx", "slot", "prob")}
    assert len(worst) >= 3 * cfg.num_layers + 4
    bad = {k: v for k, v in worst.items() if v > 1e-2}
    assert not bad, f"per-block rel-L2 above 1e-2: {bad}"
    cos = F.cosine_similarity(got.float().cpu().flatten(), want.flatten(), dim=0).item()
    assert cos >= 0.999, cos
    idx = model._last_route["expert_idx"].cpu().long()
    assert (idx == oracle.trace["moe.expert_idx"]).float().mean().item() >= 0.99
    assert abs(losses["moe_loss"].item() - want_losses["moe_loss"].item()) < 2e-3


def test_full_width_blocks_match_fake_quant_oracle_teacher_forced(fake_quant_sd3_oracle, monkeypatch):
    """SD3.5-medium width (D = 1536, 24 heads of 64) at the real token counts (4096 image, 333 text), batch 2, reduced depth:
    4 base blocks (0, 1 dual, 3 context_pre_only) and 4 control blocks (0, 1 dual). Every quantised joint-block call of one
    forward is captured (inputs, temb, outputs) and the oracle's joint_block with fake-quantised linears is evaluated on exactly
    those inputs, in fp32 on the GPU with TF32 off: rel-L2 <= 1e-2 for every block kind."""
    from oracle import unigen_sd3_oracle as O3
    from unigen_b200.sd3 import SD3Arch, UniGenSD3, shipped_control_params
    B = 2
    model = UniGenSD3(SD3Arch(num_layers=4, dual_attention_layers=(0, 1)), device="cuda")
    model.init_condition_block(condition_nums=1, control_params=dict(shipped_control_params(), use_transformer_params=False))
    model.init_random_(seed=0)
    sd = {k: v.float().clone() for k, v in model.state_dict().items()
          if k.startswith(("transformer_blocks.", "control_transformer_blocks."))}
    model.quantize_fp8()
    calls = []
    joint_block = UniGenSD3._joint_block

    def spy(self, buf, w, mod_smp, mod_ctx, smp_in, ctx_in, smp_out, ctx_out):
        if not w.fp8:  # the bf16 shared experts of the pre-stage
            return joint_block(self, buf, w, mod_smp, mod_ctx, smp_in, ctx_in, smp_out, ctx_out)
        base = any(w is b for b in self.blocks)
        rec = dict(w=w, base=base, h=smp_in.float(), c=ctx_in.float(), temb=(buf.temb if base else buf.TE[1][:B]).clone())
        joint_block(self, buf, w, mod_smp, mod_ctx, smp_in, ctx_in, smp_out, ctx_out)
        rec["h_out"] = smp_out.float()
        rec["c_out"] = ctx_out.float() if ctx_out is not None else None
        calls.append(rec)

    monkeypatch.setattr(UniGenSD3, "_joint_block", spy)
    g = torch.Generator().manual_seed(1234)
    inp = dict(hidden_states=torch.randn(B, 16, 128, 128, generator=g), condition_hidden_states=torch.randn(B, 16, 128, 128, generator=g),
               encoder_hidden_states=torch.randn(B, N_TXT, 4096, generator=g), pooled_projections=torch.randn(B, 2048, generator=g),
               condition_pooled_projections=torch.randn(B, 2048, generator=g), timestep=torch.full((B,), 500.0),
               rts_uniform=torch.rand(B * N_IMG, model.expert_nums, generator=g))
    model(**_dev(inp))
    torch.cuda.synchronize()
    assert len(calls) == 8
    H, errs = model.arch.num_attention_heads, {}
    for rec in calls:
        w = rec["w"]
        blocks = model.blocks if rec["base"] else model.ctrl_blocks
        i = next(n for n, b in enumerate(blocks) if b is w)
        prefix = f"{'transformer_blocks' if rec['base'] else 'control_transformer_blocks'}.{i}"
        c_ref, h_ref = O3.joint_block(sd, prefix, H, rec["h"], rec["c"], rec["temb"], w.dual, w.context_pre_only)
        kind = ("control" if not rec["base"] else "context_pre_only base" if w.context_pre_only
                else "dual base" if w.dual else "plain base")
        errs[f"{prefix} ({kind}) sample"] = rel_l2(rec["h_out"], h_ref)
        if rec["c_out"] is not None:
            errs[f"{prefix} ({kind}) context"] = rel_l2(rec["c_out"], c_ref)
    kinds = {k.split("(")[1].split(")")[0] for k in errs}
    assert kinds == {"dual base", "plain base", "context_pre_only base", "control"}, kinds
    assert fake_quant_sd3_oracle.quantised_calls >= 8 * 9
    bad = {k: v for k, v in errs.items() if v > 1e-2}
    assert not bad, (bad, errs)


def test_quantised_graph_replay_equals_eager():
    cfg, sd, inp, oracle, model = _setup(height=320, width=192, text_len=333, batch=2, seed=5)
    model.quantize_fp8()
    d = _dev(inp)
    eager = model(**d)[0].clone()
    model.use_cuda_graph = True
    for _ in range(2):
        assert torch.equal(model(**d)[0], eager)


def test_quantised_whole_loop_cfg_graph_equals_stepwise_loop_and_pipeline_runs():
    from unigen_b200 import pipeline as PL
    cfg, sd, inp, oracle, model = _setup()
    d = _dev(inp)
    steps, g_scale = 3, 5.0
    gen = torch.Generator().manual_seed(3)
    B, Cc, Hh, Ww = d["hidden_states"].shape
    N = (Hh // 2) * (Ww // 2)
    rts = [torch.rand(2 * B * N, cfg.expert_nums, generator=gen).cuda() for _ in range(steps)]
    neg_es = torch.randn(d["encoder_hidden_states"].shape, generator=gen).to(torch.bfloat16).cuda()
    neg_pool = torch.randn(d["pooled_projections"].shape, generator=gen).cuda()
    lat = d["hidden_states"].to(torch.bfloat16)
    kw = dict(num_inference_steps=steps, guidance_scale=g_scale, negative_encoder_hidden_states=neg_es,
              negative_pooled_projections=neg_pool, rts_uniform=rts)
    args = (lat, d["condition_hidden_states"], d["encoder_hidden_states"], d["pooled_projections"], d["condition_pooled_projections"])
    bf16 = PL.denoise_sd3(model, *args, graph_loop=True, **kw)
    model.quantize_fp8()  # drops the bf16 loop graph with the workspaces it was captured over
    assert PL._GRAPHS_ATTR not in model.__dict__
    eager = PL.denoise_sd3(model, *args, graph_loop=False, **kw)
    graphed = [PL.denoise_sd3(model, *args, graph_loop=True, **kw) for _ in range(2)]
    assert torch.equal(graphed[0], eager) and torch.equal(graphed[1], eager)
    assert not torch.equal(eager, bf16)
    assert F.cosine_similarity(eager.float().flatten(), bf16.float().flatten(), dim=0).item() > 0.95
    pipe = PL.UniGenSD3Pipeline(model)
    out = pipe(control_image=d["condition_hidden_states"], num_inference_steps=steps, guidance_scale=g_scale, latents=lat,
               prompt_embeds=d["encoder_hidden_states"], negative_prompt_embeds=neg_es, pooled_prompt_embeds=d["pooled_projections"],
               negative_pooled_prompt_embeds=neg_pool, condition_pooled_prompt_embeds=d["condition_pooled_projections"],
               rts_uniform=rts).images
    assert torch.equal(out, eager)


def test_bf16_model_unchanged_when_another_model_is_quantised():
    cfg, sd, inp, oracle, model = _setup()
    d = _dev(inp)
    before = model(**d)[0].clone()
    _, _, _, _, other = _setup()
    other.quantize_fp8()
    other(**d)
    assert torch.equal(model(**d)[0], before)
