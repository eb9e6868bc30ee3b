"""GPU checks of the opt-in fp8 (e4m3, row-wise scaled) block linears: the quantisation kernels are bit-exact against the torch
reference quantiser, the fp8 GEMM matches an fp32 matmul of the dequantised operands in every epilogue and tile variant at the
cfg3 shapes, a quantised tiny model matches the fp32 oracle whose block linears are fake-quantised the same way (teacher-forced
per block), graph replay and the pipeline entry work on it, and every refusal raises."""
import sys
from pathlib import Path

import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, str(Path(__file__).resolve().parent))
from test_fp8_cpu import dequant_ref, quant_rows_ref  # noqa: E402

pytestmark = pytest.mark.gpu
FP8 = torch.float8_e4m3fn


def rel_l2(got, want):
    got, want = got.float().cpu(), want.float().cpu()
    return ((got - want).norm() / want.norm().clamp_min(1e-12)).item()


def rnd(*shape, scale=1.0):
    return (torch.randn(*shape, device="cuda") * scale).to(torch.bfloat16)


def same_bytes(a, b):
    return torch.equal(a.view(torch.uint8).cpu(), b.view(torch.uint8).cpu())


@pytest.fixture(autouse=True)
def _seed():
    torch.manual_seed(0)
    torch.backends.cuda.matmul.allow_tf32 = False


# ---------------------------------------------------------------------------------------------------------------------------
# quantisation kernels
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rows,k", [(4608, 3072), (4096, 12288), (4608, 15360)])
def test_quant_rows_fp8_is_bit_exact(ug, rows, k):
    x = rnd(rows, k)
    x[3] = 0                      # zero row: scale 1, q = 0
    x[9] *= 1e-3
    x[9, 123] = 3e4               # single-outlier row
    q, s = ug.quant_rows_fp8(x)
    qr, sr = quant_rows_ref(x.cpu())
    assert same_bytes(q, qr) and torch.equal(s.cpu(), sr)
    assert s[3].item() == 1.0 and (q[3].view(torch.uint8) == 0).all()


def test_quant_rows_fp8_strided_views(ug):
    """The single block's `cat` is a strided view ([attn | gelu(mlp)] rows inside a wider buffer); outputs may be views too."""
    big = rnd(2, 700, 5 * 384 + 64)
    x = big[:, 50:650, :5 * 384]
    qbuf = torch.zeros(2, 800, 5 * 384 + 128, device="cuda", dtype=FP8)
    sbuf = torch.zeros(2, 900, device="cuda")
    q, s = ug.quant_rows_fp8(x, qbuf[:, 100:700, :5 * 384], sbuf[:, 200:800])
    qr, sr = quant_rows_ref(x.cpu())
    assert same_bytes(q, qr) and torch.equal(s.cpu(), sr)
    assert (qbuf[:, :100].view(torch.uint8) == 0).all() and (sbuf[:, :200] == 0).all()  # nothing outside the views


def test_quant_rows_fp8_cfg3_cat_operand(ug):
    """The single block's proj_out operand at cfg3 exactly as the model passes it: CAT[:, :S] ([attn | gelu(mlp)], K = 5D = 15360)
    inside the workspace buffer, into CATQ[:, :S] / CATS[:, :S]; batch 2, so the batch stride is not rows * K. Also the gelu half
    alone (K = 12288 at row stride 5D)."""
    S, D, spare = 4608, 3072, 64
    cat = rnd(2, S + spare, 5 * D)
    catq = torch.zeros(2, S + spare, 5 * D, device="cuda", dtype=FP8)
    cats = torch.zeros(2, S + spare, device="cuda")
    for x, q_view, s_view in ((cat[:, :S], catq[:, :S], cats[:, :S]), (cat[:, :S, D:], catq[:, :S, D:], cats[:, :S])):
        q, s = ug.quant_rows_fp8(x, q_view, s_view)
        qr, sr = quant_rows_ref(x.cpu())
        assert same_bytes(q, qr) and torch.equal(s.cpu(), sr)
    assert (catq[:, S:].view(torch.uint8) == 0).all() and (cats[:, S:] == 0).all()


@pytest.mark.parametrize("B,rows,d", [(1, 4608, 3072), (2, 300, 384), (1, 700, 1024), (1, 513, 2560), (2, 130, 4096)])
def test_ln_modulate_fp8_equals_quantised_ln_modulate(ug, B, rows, d):
    """One kernel per row layout (rows / two-warp / one-warp kernels): quant_rows_fp8(ln_modulate(x)) bit for bit."""
    x = rnd(B, rows, d, scale=3.0)
    shift, scale = torch.randn(B, d, device="cuda") * 0.5, torch.randn(B, d, device="cuda") * 0.5
    nx = torch.empty_like(x)
    ug.ln_modulate(x, nx, shift, scale)
    qw, sw = ug.quant_rows_fp8(nx)
    q = torch.empty(B, rows, d, device="cuda", dtype=FP8)
    s = torch.empty(B, rows, device="cuda")
    ug.ln_modulate_fp8(x, q, s, shift, scale)
    assert same_bytes(q, qw) and torch.equal(s, sw)


# ---------------------------------------------------------------------------------------------------------------------------
# fp8 GEMM
# ---------------------------------------------------------------------------------------------------------------------------
def _operands(ug, B, M, K, N):
    a, w = rnd(B, M, K), rnd(N, K, scale=K ** -0.5)
    qa, sa = ug.quant_rows_fp8(a)
    qw, sw = ug.quant_rows_fp8(w)
    ad, wd = dequant_ref(qa.float(), sa), dequant_ref(qw.float(), sw)
    return qa, sa, qw, sw, ad, wd


# (M, K, N) of the cfg3 block linears: image / text rows of the double blocks (q|k|v, to_out, ff1, ff2) and the joint rows of
# the single blocks (q|k|v, proj_mlp, proj_out with K = 5D)
CFG3_SHAPES = [(4096, 3072, 9216), (4096, 12288, 3072), (512, 3072, 3072), (512, 3072, 12288), (4608, 3072, 12288), (4608, 15360, 3072)]


@pytest.mark.parametrize("variant", [0, 1, 2, 3, 4, 5, 6])
@pytest.mark.parametrize("mkn", CFG3_SHAPES)
def test_gemm_fp8_cfg3_shapes_bias(ug, variant, mkn):
    M, K, N = mkn
    qa, sa, qw, sw, ad, wd = _operands(ug, 1, M, K, N)
    bias = rnd(N)
    out = ug.gemm_fp8(qa, sa, qw, sw, bias=bias, variant=variant)
    want = ad[0] @ wd.t() + bias.float()
    assert rel_l2(out[0], want) < 6e-3
    assert (out[0].float() - want).abs().max().item() < 0.15  # every tile written once


@pytest.mark.parametrize("variant", [0, 1, 2, 3, 4, 5, 6])
def test_gemm_fp8_gelu_and_gated_residual_epilogues(ug, variant):
    """ff1 (bias + GELU-tanh) and ff2 (gate * alpha + in-place residual) at cfg3 image-stream shapes, batch 2."""
    qa, sa, qw, sw, ad, wd = _operands(ug, 2, 1000, 3072, 1536)
    bias = rnd(1536)
    out = ug.gemm_fp8(qa, sa, qw, sw, bias=bias, act=ug.UG_ACT_GELU_TANH, variant=variant)
    assert rel_l2(out, F.gelu(ad @ wd.t() + bias.float(), approximate="tanh")) < 6e-3
    gate = torch.randn(2, 1536, device="cuda")
    h = rnd(2, 1000, 1536)
    h0 = h.float().clone()
    ug.gemm_fp8(qa, sa, qw, sw, out=h, bias=bias, gate=gate, alpha=0.7, residual=h, variant=variant)
    assert rel_l2(h, h0 + 0.7 * gate[:, None] * (ad @ wd.t() + bias.float())) < 6e-3


@pytest.mark.parametrize("variant", [0, 1, 2, 4, 5])
@pytest.mark.parametrize("H,dh,rows", [(24, 128, 512), (6, 64, 333)])
def test_gemm_fp8_fused_qk_norm_rope(ug, variant, H, dh, rows):
    D, K = H * dh, 256
    axes = (16, 56, 56) if dh == 128 else (8, 28, 28)
    qa, sa, qw, sw, ad, wd = _operands(ug, 1, rows, K, 3 * D)
    bias = rnd(3 * D)
    nw = (1 + 0.1 * torch.randn(2, dh)).to(torch.bfloat16).cuda()
    ids = torch.stack([torch.zeros(rows), torch.arange(rows) // 20, torch.arange(rows) % 20], 1).float().cuda()
    table = ug.rope_table(ids, axes)
    out = ug.gemm_fp8(qa, sa, qw, sw, bias=bias, variant=variant, qk_norm=dict(weight=nw, head_dim=dh, d=D, cos_sin=table, eps=1e-6))
    full = ad @ wd.t() + bias.float()
    y = full[:, :, :2 * D].reshape(1, rows, 2, H, dh)
    y = y * torch.rsqrt(y.pow(2).mean(-1, keepdim=True) + 1e-6) * nw.float()[None, None, :, None, :]
    cs = table.view(rows, dh // 2, 2)
    c, s_ = cs[None, :, None, None, :, 0], cs[None, :, None, None, :, 1]
    y0, y1 = y[..., 0::2], y[..., 1::2]
    want = torch.stack([y0 * c - y1 * s_, y1 * c + y0 * s_], -1).reshape(1, rows, 2 * D)
    assert rel_l2(out[:, :, :2 * D], want) < 4e-3
    assert rel_l2(out[:, :, 2 * D:], full[:, :, 2 * D:]) < 6e-3


def test_gemm_fp8_agrees_with_torch_scaled_mm_rowwise(ug):
    M, K, N = 4096, 3072, 3072
    qa, sa, qw, sw, ad, wd = _operands(ug, 1, M, K, N)
    try:
        ref = torch._scaled_mm(qa[0], qw.t(), scale_a=sa[0].view(M, 1), scale_b=sw.view(1, N), out_dtype=torch.bfloat16)
    except (RuntimeError, NotImplementedError) as e:  # row-wise scaling is not offered by every torch build on sm_100
        pytest.skip(f"torch._scaled_mm row-wise unavailable here: {e}")
    out = ug.gemm_fp8(qa, sa, qw, sw)
    assert rel_l2(out[0], ref) < 6e-3


def test_gemm_fp8_rejects_what_it_does_not_cover(ug):
    import ctypes as C
    from unigen_b200 import _lib
    qa, sa, qw, sw, _, _ = _operands(ug, 1, 256, 256, 256)
    out = torch.empty(1, 256, 256, device="cuda", dtype=torch.bfloat16)
    with pytest.raises(ug.UgError):
        ug.gemm_fp8(qa.view(torch.uint8), sa, qw, sw)                      # not e4m3
    with pytest.raises(ug.UgError):
        ug.gemm_fp8(qa, sa[:, :100], qw, sw)                                # scale shape
    lib = _lib.load()

    def call(**kw):
        g = _lib.GemmArgs()
        g.a, g.a_row_stride, g.a_batch_stride, g.w, g.w_row_stride = qa.data_ptr(), 256, 256 * 256, qw.data_ptr(), 256
        g.c, g.c_row_stride, g.c_batch_stride = out.data_ptr(), 256, 256 * 256
        g.batch, g.rows, g.n, g.k, g.alpha = 1, 256, 256, 256, 1.0
        for k, v in kw.items():
            setattr(g, k, v)
        sc = _lib.GemmFp8Scales(sa.data_ptr(), 256, sw.data_ptr(), 0)
        return lib.ug_gemm_fp8(C.byref(g), C.byref(sc), None)

    assert call() == 0
    torch.cuda.synchronize()
    for bad in (dict(k=248), dict(colmask_block=32, lora_nseg=1), dict(lora_t=sa.data_ptr(), lora_b=qw.data_ptr(), lora_rank=4, lora_nseg=1),
                dict(a2=qa.data_ptr(), w2=qw.data_ptr(), k2=64, a2_row_stride=256, w2_row_stride=256)):
        assert call(**bad) == -1, bad
    assert lib.ug_gemm_fp8(C.byref(_lib.GemmArgs()), None, None) == -1


# ---------------------------------------------------------------------------------------------------------------------------
# model
# ---------------------------------------------------------------------------------------------------------------------------
QUANT_DOUBLE = (".attn.to_q", ".attn.to_k", ".attn.to_v", ".attn.add_q_proj", ".attn.add_k_proj", ".attn.add_v_proj",
                ".attn.to_out.0", ".attn.to_add_out", ".ff.net.0.proj", ".ff.net.2", ".ff_context.net.0.proj", ".ff_context.net.2")
QUANT_SINGLE = (".attn.to_q", ".attn.to_k", ".attn.to_v", ".proj_mlp", ".proj_out")


def _quantised_prefix(prefix):
    head, _, rest = prefix.partition(".")
    idx, _, name = rest.partition(".")
    if not idx.isdigit():
        return False
    if head in ("transformer_blocks", "control_joint_trans_blocks"):
        return "." + name in QUANT_DOUBLE
    if head in ("single_transformer_blocks", "control_single_trans_blocks"):
        return "." + name in QUANT_SINGLE
    return False


@pytest.fixture
def fake_quant_oracle(monkeypatch):
    """oracle.unigen_oracle.linear with x quantised per token row (of its bf16 value, as the native operands are bf16) and W per
    output channel by the reference quantiser, for the quantised block linears only."""
    from oracle import unigen_oracle as O
    plain = O.linear

    def linear(sd, prefix, x):
        if not _quantised_prefix(prefix):
            return plain(sd, prefix, x)
        linear.quantised_calls += 1
        W = sd[prefix + ".weight"]
        xd = dequant_ref(*quant_rows_ref(x.to(torch.bfloat16)))
        return F.linear(xd, dequant_ref(*quant_rows_ref(W.to(torch.bfloat16))), sd.get(prefix + ".bias"))

    linear.quantised_calls = 0
    monkeypatch.setattr(O, "linear", linear)
    return O


def _tiny(seed=0):
    from oracle import unigen_oracle as O
    from unigen_b200.model import FluxArch, UniGenFlux, canonical_control_params
    cfg = O.FluxConfig.tiny()
    sd = O.init_state_dict(cfg, seed=seed)
    sd = {k: (v if k.endswith("gate.wg.weight") else v.to(torch.bfloat16).float()) for k, v in sd.items()}
    inp = O.make_inputs(cfg, 256, 256, text_len=512)
    for k in ("hidden_states", "condition_hidden_states", "encoder_hidden_states"):
        inp[k] = inp[k].to(torch.bfloat16).float()
    model = UniGenFlux(FluxArch.tiny(), device="cuda")
    model.init_condition_block(condition_nums=1, control_params=canonical_control_params())
    model.load_state_dict(sd)
    return cfg, sd, inp, model


def _dev(inp):
    return {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in inp.items()}


def test_quantize_fp8_interface():
    from unigen_b200.model import FP8, MultiCondtionUniGenFlux
    cfg, sd, inp, model = _tiny()
    assert model.linear_dtype == torch.bfloat16
    n_before = len(model.state_dict())
    assert model.quantize_fp8() is model and model.linear_dtype == FP8
    assert model.quantize_fp8() is model
    gone = n_before - len(model.state_dict())
    assert gone == (2 + 1) * 12 + (4 + 2) * 5  # 12 weight views per double block, 5 per single block (base + control)
    assert all(w.fp8 for w in model.double + model.ctrl_double + model.single + model.ctrl_single)
    assert not any(w.fp8 for w in model.shared) and model.double[0].qkv[0].dtype == FP8
    assert issubclass(MultiCondtionUniGenFlux, type(model)) and hasattr(MultiCondtionUniGenFlux, "quantize_fp8")


def _fp8_parity(workload, monkeypatch):
    """tests/parity_fullsize.py's weave check (every block teacher-forced on the native block input: base / control double, the
    zero-linear adds, base / control single, the CoMoE pre-stage, norm_out + proj_out; routing given the native gate input; the
    free-running oracle forward) run over a QUANTISED native model against the fp32 oracle with fake-quantised block linears
    (fixture fake_quant_oracle). parity_fullsize builds, random-initialises and runs the model itself; the subclass below makes
    its first forward run once in bf16 on the same inputs (the velocity the fp8 one is compared with), then quantize_fp8() and
    the traced fp8 forward. Its state_dict() keeps returning the bf16 weights: the oracle quantises them itself."""
    import parity_fullsize as P
    from unigen_b200 import model as M
    box = {}

    class QuantisedOnFirstForward(M.UniGenFlux):
        def forward(self, **kw):
            if self.linear_dtype == torch.bfloat16:
                trace, self.trace = self.trace, None
                box["bf16_velocity"] = super().forward(**kw)[0].float().clone()
                box["bf16_state_dict"] = dict(super().state_dict())
                self.quantize_fp8()
                self.trace = trace
            out = super().forward(**kw)
            box["fp8_velocity"] = out[0].float().clone()
            return out

        def state_dict(self, *args, **kwargs):
            return box["bf16_state_dict"] if "bf16_state_dict" in box else super().state_dict()

    monkeypatch.setattr(M, "UniGenFlux", QuantisedOnFirstForward)
    from oracle import unigen_oracle as O
    rec = P.main(["--workload", workload])
    # the oracle side really was fake-quantised: base + control double blocks (12 quantised linears each) and base + control
    # single blocks (5 each) of the teacher-forced pass alone
    blocks = rec["per_block_rel_l2"]
    n_double = sum(k.startswith("double.") and k.endswith(".base_hidden") for k in blocks)
    n_single = sum(k.startswith("single.") and k.endswith(".base_hidden") for k in blocks)
    assert n_double and n_single and O.linear.quantised_calls >= 2 * 12 * n_double + 2 * 5 * n_single, O.linear.quantised_calls
    rec["free_running"]["note"] = ("native fp8 end to end vs the fp32 oracle with fake-quantised block linears end to end; the "
                                   "oracle routes on the unrounded fp32 sum, the native path on the bf16 sum")
    v8, v16 = box["fp8_velocity"], box["bf16_velocity"]
    rec["fp8_vs_bf16_native_velocity"] = {"cosine": F.cosine_similarity(v8.flatten(), v16.flatten(), dim=0).item(),
                                          "rel_l2": rel_l2(v8, v16), "note": "free-running, no bar"}
    rec["oracle"] = "fp32 oracle on the B200 (TF32 off), block linears fake-quantised (x per token row, W per output channel)"
    import json
    import os
    print(json.dumps({k: rec[k] for k in ("teacher_forced", "routing_given_native_gate_input", "free_running",
                                          "fp8_vs_bf16_native_velocity")}))
    if os.environ.get("UG_PARITY_OUT"):
        Path(os.environ["UG_PARITY_OUT"], f"r03_parity_fp8_{workload}.json").write_text(json.dumps(rec) + "\n")
    tf = rec["teacher_forced"]
    assert tf["max_rel_l2"] <= 1e-2, tf["worst"]
    assert rec["routing_given_native_gate_input"]["bit_exact"], rec["routing_given_native_gate_input"]
    assert torch.isfinite(v8).all()
    return rec


def test_tiny_quantised_model_matches_fake_quant_oracle_teacher_forced(fake_quant_oracle, monkeypatch):
    """Every block of the tiny weave (base and control double / single blocks included), teacher-forced: rel-L2 <= 1e-2;
    routing bit-exact given the native gate input."""
    rec = _fp8_parity("tiny", monkeypatch)
    assert any(".ctrl_hidden" in k for k in rec["per_block_rel_l2"])


def test_cfg3_quantised_model_matches_fake_quant_oracle_teacher_forced(fake_quant_oracle, monkeypatch):
    """The same at full size (1024^2 + 1 condition: 4096 + 4096 + 512 tokens, D = 3072, proj_out K = 15360, 19 + 38 base and
    9 + 19 control blocks): max rel-L2 <= 1e-2 over the whole weave, routing bit-exact; the free-running cosines against the
    fake-quant oracle and against the bf16 native model are reported."""
    rec = _fp8_parity("cfg3", monkeypatch)
    assert rec["teacher_forced"]["blocks_checked"] > 200


def test_bf16_model_unchanged_when_another_model_is_quantised():
    cfg, sd, inp, model = _tiny()
    dev = _dev(inp)
    before = model(**dev)[0].clone()
    _, _, _, other = _tiny()
    other.quantize_fp8()
    other(**dev)
    assert torch.equal(model(**dev)[0], before)


def test_quantised_whole_loop_graph_equals_stepwise_loop_and_pipeline_runs():
    from unigen_b200 import pipeline as PL
    cfg, sd, inp, model = _tiny()
    inp = _dev(inp)
    args = (inp["hidden_states"], inp["condition_hidden_states"], inp["encoder_hidden_states"], inp["pooled_projections"],
            inp["condition_pooled_projections"], inp["img_ids"], inp["txt_ids"], inp["condition_ids"])
    g = torch.Generator().manual_seed(5)
    rts = [torch.rand(256, cfg.expert_nums, generator=g).cuda() for _ in range(3)]
    bf16 = PL.denoise(model, *args, num_inference_steps=3, rts_uniform=rts, graph_loop=True)
    model.quantize_fp8()  # drops the bf16 loop graph with the workspaces it was captured over
    eager = PL.denoise(model, *args, num_inference_steps=3, rts_uniform=rts, graph_loop=False)
    graphed = [PL.denoise(model, *args, num_inference_steps=3, rts_uniform=rts, graph_loop=True) for _ in range(2)]
    assert torch.equal(graphed[0], eager) and torch.equal(graphed[1], eager)
    assert not torch.equal(eager, bf16)
    assert F.cosine_similarity(eager.float().flatten(), bf16.float().flatten(), dim=0).item() > 0.95
    from unigen_b200.condition import Condition
    pipe = PL.UniGenFLUXPipeline(model)
    cond = Condition("canny", inp["condition_hidden_states"].to(torch.bfloat16), height=256, width=256)
    out = pipe(prompt_embeds=inp["encoder_hidden_states"], pooled_prompt_embeds=inp["pooled_projections"], control_image=cond,
               condition_pooled_prompt_embeds=inp["condition_pooled_projections"], height=256, width=256, num_inference_steps=3,
               latents=inp["hidden_states"].to(torch.bfloat16), rts_uniform=rts, output_type="latent")
    assert out.images.shape == eager.shape and torch.isfinite(out.images.float()).all()


def test_refusals(tmp_path):
    from unigen_b200.chandle import FluxStepHandle
    from unigen_b200.model import FluxArch, UniGenFlux, canonical_control_params
    from unigen_b200.ops import UgError
    cfg, sd, inp, model = _tiny()
    with pytest.raises(UgError):
        UniGenFlux(FluxArch.tiny(), device="cuda").quantize_fp8()  # before init_condition_block
    model.quantize_fp8()
    with pytest.raises(UgError):
        model.load_state_dict(sd)
    with pytest.raises(UgError):
        model.init_random_(seed=1)
    with pytest.raises(UgError):
        FluxStepHandle(model)
    import torch.distributed as dist
    from unigen_b200.parallel import SequenceParallelUniGenFlux
    own = not dist.is_initialized()
    if own:
        dist.init_process_group("gloo", init_method=f"file://{tmp_path / 'pg'}", rank=0, world_size=1)
    try:
        sp = SequenceParallelUniGenFlux(FluxArch.tiny(), device="cuda")
        sp.init_condition_block(condition_nums=1, control_params=canonical_control_params())
        sp.load_state_dict(sd)
        sp.quantize_fp8()
        with pytest.raises(UgError):
            sp(**_dev(inp))
        sp.sp_enabled = False  # the same object as a single-GPU model (batch data parallelism) runs
        assert torch.isfinite(sp(**_dev(inp))[0].float()).all()
    finally:
        if own:
            dist.destroy_process_group()
