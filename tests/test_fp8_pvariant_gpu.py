"""GPU checks of the fp8 (e4m3, row-wise scaled) block linears of the LoRA-switched P-variant (`UniCombineFlux.quantize_fp8()`):
the mixed-kind GEMM (e4m3 main pair + bf16 K extension in one accumulator) against fp32 on the dequantised operands in every tile
variant and epilogue, the masked fp8 down-projection, the segmented fused LayerNorm bit for bit, the new entry point's refusals,
and the quantised model against the fp32 P-variant oracle whose switched linears are fake-quantised the same way."""
import math
import sys
from pathlib import Path

import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, str(Path(__file__).resolve().parent))
from test_fp8_cpu import dequant_ref, quant_rows_ref  # noqa: E402

pytestmark = pytest.mark.gpu
FP8 = torch.float8_e4m3fn
BLK = 64  # columns per adapter group in the K-extension operand


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


def _quant(ug, t):
    q, s = ug.quant_rows_fp8(t)
    return q, s, dequant_ref(q.float(), s)


# ---------------------------------------------------------------------------------------------------------------------------
# mixed-kind GEMM: e4m3 main pair + bf16 K extension
# ---------------------------------------------------------------------------------------------------------------------------
# (M, K, N) of the cfg4 P-variant block linears (1024^2 image + 3 conditions: 4096 + 3 x 4096 image / condition rows, 512 text
# rows, 16 896 joint rows of the single blocks; D = 3072)
CFG4_SHAPES = [(16384, 3072, 9216), (16384, 3072, 3072), (16384, 3072, 12288), (16384, 12288, 3072), (512, 3072, 9216),
               (16896, 3072, 9216), (16896, 3072, 12288), (16896, 15360, 3072)]
K2 = 4 * BLK  # 1 + 3 adapter groups


def _mixed_operands(ug, M, K, N, k2=K2, batch=1):
    """Random e4m3 main pair and a bf16 extension sized so that its share of the accumulator is comparable to the main one."""
    qa, sa, ad = _quant(ug, rnd(batch, M, K))
    qw, sw, wd = _quant(ug, rnd(N, K, scale=K ** -0.5))
    # pre-divided operands are large like the e4m3 values (x / a_s and B / w_s reach hundreds): sized so that the extension's
    # sum over k2 is about half the main pair's sum over K
    a2 = rnd(batch, M, k2, scale=100.0)
    w2 = rnd(N, k2, scale=50.0 * math.sqrt(K / k2))
    acc = (qa.float() @ qw.float().t() + a2.float() @ w2.float().t()) * sa[..., None] * sw
    main_only = ad @ wd.t()
    return qa, sa, qw, sw, a2, w2, acc, main_only


@pytest.mark.parametrize("variant,mkn", [(0, s) for s in CFG4_SHAPES] + [(v, (16384, 3072, 3072)) for v in range(1, 7)])
def test_gemm_fp8_lora_mixed_kind_accumulation(ug, variant, mkn):
    M, K, N = mkn
    qa, sa, qw, sw, a2, w2, acc, main_only = _mixed_operands(ug, M, K, N)
    bias = rnd(N)
    out = ug.gemm_fp8(qa, sa, qw, sw, bias=bias, variant=variant, a2=a2, w2=w2)
    want = acc + bias.float()
    assert rel_l2(out, want) < 6e-3
    assert rel_l2(main_only + bias.float(), want) > 0.1  # the extension is a visible part of the result


def _switched(ug, B=2, D=384, rank=4, seed=1):
    """The switched q|k|v update of a quantised linear over non-tile-aligned segments [txt: none | img: den | c1 | c2], built
    exactly as the model builds it: A2 = fp8 masked down-projection with unit activation scales, W2 = B / w_s."""
    g = torch.Generator().manual_seed(seed)
    bounds, groups = [0, 40, 300, 420, 555], [-1, 0, 1, 2]
    S, G = bounds[-1], 3
    x = rnd(B, S, D, scale=2.0)
    x[:, 77] = 0  # a zero row: scale 1, q = 0
    W = rnd(3 * D, D, scale=D ** -0.5)
    A = (torch.randn(G, 3, rank, D, generator=g) / math.sqrt(D)).to(torch.bfloat16)
    Bm = (torch.randn(G, 3, D, rank, generator=g) * 0.5 / math.sqrt(rank)).to(torch.bfloat16)
    aw = torch.zeros(G * BLK, D, dtype=torch.bfloat16)
    bw = torch.zeros(3 * D, G * BLK, dtype=torch.bfloat16)
    for gi in range(G):
        aw[gi * BLK:gi * BLK + 3 * rank] = A[gi].reshape(3 * rank, D)
        for sub in range(3):
            bw[sub * D:(sub + 1) * D, gi * BLK + sub * rank:gi * BLK + (sub + 1) * rank] = Bm[gi, sub]
    aw, bw = aw.cuda(), bw.cuda()
    q, s, xd = _quant(ug, x)
    qw, sw, wd = _quant(ug, W)
    aq, aws, awd = _quant(ug, aw)
    lin = xd @ wd.t()
    for si in range(4):
        gi = groups[si]
        if gi >= 0:
            rows = slice(bounds[si], bounds[si + 1])
            lin[:, rows] += (xd[:, rows] @ awd[gi * BLK:(gi + 1) * BLK].t()) @ bw[:, gi * BLK:(gi + 1) * BLK].float().t()
    w2 = (bw.float() / sw[:, None]).to(torch.bfloat16)
    return dict(x=x, q=q, s=s, xd=xd, qw=qw, sw=sw, aw=aw, aq=aq, aws=aws, awd=awd, bw=bw, w2=w2, lin=lin, bounds=bounds,
                groups=groups, S=S, D=D)


@pytest.mark.parametrize("variant", [0, 1, 2, 3, 4, 5, 6])
def test_gemm_fp8_lora_switched_update_gate_seg_residual(ug, variant):
    """The whole switched form over segments that are not tile-aligned: masked fp8 down-projection (variants 1-3: the column
    mask keeps the direct epilogue) feeding the K extension, with per-segment gates and the residual in the same launch."""
    t = _switched(ug)
    B, S, D = 2, t["S"], t["D"]
    cm = dict(block=BLK, seg_bounds=t["bounds"], seg_group=t["groups"])
    tw = torch.full((B, S, 3 * BLK), 7.0, device="cuda", dtype=torch.bfloat16)
    ug.gemm_fp8(t["q"], None, t["aq"], t["aws"], out=tw, variant=min(variant, 3), colmask=cm)
    gates = torch.randn(4, B, 3 * D, device="cuda")
    res = rnd(B, S, 3 * D)
    out = ug.gemm_fp8(t["q"], t["s"], t["qw"], t["sw"], variant=variant, a2=tw, w2=t["w2"], gate=gates[0],
                      gate_seg_stride=gates.stride(0), seg_bounds=t["bounds"], residual=res)
    want = res.float().clone()
    for si in range(4):
        rows = slice(t["bounds"][si], t["bounds"][si + 1])
        want[:, rows] += gates[si][:, None, :] * t["lin"][:, rows]
    assert rel_l2(out, want) < 6e-3
    # the un-adapted text rows equal the plain fp8 GEMM (the extension adds exact zeros there)
    plain = ug.gemm_fp8(t["q"], t["s"], t["qw"], t["sw"], variant=variant, gate=gates[0], residual=res)
    assert torch.equal(out[:, :40], plain[:, :40]) and not torch.equal(out[:, 40:], plain[:, 40:])


@pytest.mark.parametrize("variant", [1, 2, 3])
def test_masked_fp8_down_projection(ug, variant):
    """Zeros exactly where the bf16 column-mask GEMM puts them; values = (x / a_s) @ A^T with the quantised A."""
    t = _switched(ug)
    cm = dict(block=BLK, seg_bounds=t["bounds"], seg_group=t["groups"])
    ref16 = ug.gemm(t["x"], t["aw"], variant=variant, colmask=cm)
    tw = torch.full_like(ref16, 5.0)
    ug.gemm_fp8(t["q"], None, t["aq"], t["aws"], out=tw, variant=variant, colmask=cm)
    assert torch.equal(tw == 0, ref16 == 0)
    want = torch.zeros_like(tw, dtype=torch.float32)
    for si in range(4):
        gi = t["groups"][si]
        if gi >= 0:
            rows = slice(t["bounds"][si], t["bounds"][si + 1])
            want[:, rows, gi * BLK:(gi + 1) * BLK] = (t["xd"][:, rows] / t["s"][:, rows, None]) @ t["awd"][gi * BLK:(gi + 1) * BLK].t()
    assert rel_l2(tw, want) < 6e-3


@pytest.mark.parametrize("variant", [0, 1, 2, 3, 4, 5, 6])
def test_gemm_fp8_lora_gelu(ug, variant):
    qa, sa, qw, sw, a2, w2, acc, _ = _mixed_operands(ug, 1000, 3072, 1536, batch=2)
    bias = rnd(1536)
    out = ug.gemm_fp8(qa, sa, qw, sw, bias=bias, act=ug.UG_ACT_GELU_TANH, variant=variant, a2=a2, w2=w2)
    assert rel_l2(out, F.gelu(acc + bias.float(), approximate="tanh")) < 6e-3


@pytest.mark.parametrize("variant", [0, 1, 2, 4, 5])
@pytest.mark.parametrize("H,dh,rows", [(24, 128, 512), (6, 64, 333)])
def test_gemm_fp8_lora_fused_qk_norm_rope(ug, variant, H, dh, rows):
    D, K = H * dh, 256
    axes = (16, 56, 56) if dh == 128 else (8, 28, 28)
    qa, sa, qw, sw, a2, w2, acc, _ = _mixed_operands(ug, rows, K, 3 * D)
    bias = rnd(3 * D)
    nw = (1 + 0.1 * torch.randn(2, dh)).to(torch.bfloat16).cuda()
    ids = torch.stack([torch.zeros(rows), torch.arange(rows) // 20, torch.arange(rows) % 20], 1).float().cuda()
    table = ug.rope_table(ids, axes)
    out = ug.gemm_fp8(qa, sa, qw, sw, bias=bias, variant=variant, a2=a2, w2=w2,
                      qk_norm=dict(weight=nw, head_dim=dh, d=D, cos_sin=table, eps=1e-6))
    full = acc + bias.float()
    y = full[:, :, :2 * D].reshape(1, rows, 2, H, dh)
    y = y * torch.rsqrt(y.pow(2).mean(-1, keepdim=True) + 1e-6) * nw.float()[None, None, :, None, :]
    cs = table.view(rows, dh // 2, 2)
    c, s_ = cs[None, :, None, None, :, 0], cs[None, :, None, None, :, 1]
    y0, y1 = y[..., 0::2], y[..., 1::2]
    want = torch.stack([y0 * c - y1 * s_, y1 * c + y0 * s_], -1).reshape(1, rows, 2 * D)
    assert rel_l2(out[:, :, :2 * D], want) < 4e-3
    assert rel_l2(out[:, :, 2 * D:], full[:, :, 2 * D:]) < 6e-3


def test_gemm_fp8_lora_refusals(ug):
    import ctypes as C
    from unigen_b200 import _lib
    qa, sa, _ = _quant(ug, rnd(1, 256, 256))
    qw, sw, _ = _quant(ug, rnd(256, 256))
    a2, w2 = rnd(1, 256, 64), rnd(256, 64)
    out = torch.empty(1, 256, 256, device="cuda", dtype=torch.bfloat16)
    lib = _lib.load()

    def call(a_scale=sa.data_ptr(), w_scale=sw.data_ptr(), **kw):
        g = _lib.GemmArgs()
        g.a, g.a_row_stride, g.a_batch_stride, g.w, g.w_row_stride = qa.data_ptr(), 256, 256 * 256, qw.data_ptr(), 256
        g.c, g.c_row_stride, g.c_batch_stride = out.data_ptr(), 256, 256 * 256
        g.batch, g.rows, g.n, g.k, g.alpha = 1, 256, 256, 256, 1.0
        g.a2, g.a2_row_stride, g.a2_batch_stride, g.w2, g.w2_row_stride, g.k2 = a2.data_ptr(), 64, 256 * 64, w2.data_ptr(), 64, 64
        for k, v in kw.items():
            setattr(g, k, v)
        sc = _lib.GemmFp8Scales(a_scale, 256, w_scale, 0)
        return lib.ug_gemm_fp8_lora(C.byref(g), C.byref(sc), None)

    assert call() == 0
    assert call(a_scale=None) == 0  # NULL a_scale: unit row scales (the convention of the masked down-projection)
    torch.cuda.synchronize()
    for bad in (dict(k=248), dict(lora_t=sa.data_ptr(), lora_b=qw.data_ptr(), lora_rank=4, lora_nseg=1), dict(w_scale=None),
                dict(w2=None)):
        assert call(**bad) == -1, bad
    assert lib.ug_gemm_fp8_lora(C.byref(_lib.GemmArgs()), None, None) == -1
    # the plain entry point still refuses the K extension and the column mask
    with pytest.raises(ug.UgError):
        ug.gemm_fp8(qa, None, qw, sw)


# ---------------------------------------------------------------------------------------------------------------------------
# segmented LayerNorm-modulate with e4m3 output
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,d,bounds", [
    (2, 3072, [0, 512, 4608, 8704, 12800, 16896]),         # cfg4 double block: txt | img | c1 | c2 | c3
    (2, 3072, [0, 4608, 8704, 12800, 16896]),              # cfg4 single block: [txt|img] | c1 | c2 | c3
    (2, 384, [0, 40, 300, 420, 555]),                      # not aligned to anything
    (2, 384, [0, 77]),                                     # one segment
])
def test_ln_modulate_segs_fp8_equals_quantised_ln_modulate_segs(ug, B, d, bounds):
    rows, nseg = bounds[-1], len(bounds) - 1
    x = rnd(B, rows, d, scale=3.0)
    x[:, 5] = 0
    mods = torch.randn(nseg, B, 2 * d, device="cuda") * 0.5
    shift, scale = mods[0, :, :d], mods[0, :, d:]
    nx = torch.empty_like(x)
    ug.ln_modulate_segs(x, nx, shift, scale, bounds, mods.stride(0))
    qw, sw = ug.quant_rows_fp8(nx)
    q = torch.empty(B, rows, d, device="cuda", dtype=FP8)
    s = torch.empty(B, rows, device="cuda")
    ug.ln_modulate_segs_fp8(x, q, s, shift, scale, bounds, mods.stride(0))
    assert same_bytes(q, qw) and torch.equal(s, sw)


# ---------------------------------------------------------------------------------------------------------------------------
# model
# ---------------------------------------------------------------------------------------------------------------------------
QUANT_DOUBLE = (".attn.to_q", ".attn.to_k", ".attn.to_v", ".attn.add_q_proj", ".attn.add_k_proj", ".attn.add_v_proj",
                ".attn.to_out.0", ".attn.to_add_out", ".ff.net.0.proj", ".ff.net.2", ".ff_context.net.0.proj", ".ff_context.net.2")
QUANT_SINGLE = (".attn.to_q", ".attn.to_k", ".attn.to_v", ".proj_mlp", ".proj_out")


def _quantised_name(name):
    head, _, rest = name.partition(".")
    idx, _, sub = rest.partition(".")
    if not idx.isdigit():
        return False
    return "." + sub in {"transformer_blocks": QUANT_DOUBLE, "single_transformer_blocks": QUANT_SINGLE}.get(head, ())


def _fq(t):
    """Fake quantisation of the native operands: per row of the bf16 value (x per token, W per output channel, lora_A per row)."""
    return dequant_ref(*quant_rows_ref(t.to(torch.bfloat16)))


@pytest.fixture
def fake_quant_pvariant_oracle(monkeypatch):
    """oracle.unigen_oracle with the quantised linears of the P-variant fake-quantised: the switched ones (PVariantOracle.lin:
    x, W and every lora_A quantised, lora_B as is) and the plain ones the forward calls through `linear` (add_q|k|v_proj,
    to_add_out, ff.net.0.proj, ff_context)."""
    from oracle import unigen_oracle as O
    plain_linear, plain_lin = O.linear, O.PVariantOracle.lin
    calls = {"n": 0}

    def linear(sd, prefix, x):
        if not _quantised_name(prefix):
            return plain_linear(sd, prefix, x)
        calls["n"] += 1
        return F.linear(_fq(x), _fq(sd[prefix + ".weight"]), sd.get(prefix + ".bias"))

    def lin(self, name, x, active):
        if not _quantised_name(name):
            return plain_lin(self, name, x, active)
        calls["n"] += 1
        xd = _fq(x)
        y = F.linear(xd, _fq(self.sd[name + ".weight"]), self.sd.get(name + ".bias"))
        for a in active:
            ka = f"{name}.lora_A.{a}.weight"
            if ka in self.sd:
                y = y + F.linear(F.linear(xd, _fq(self.sd[ka])), self.sd[f"{name}.lora_B.{a}.weight"]) * self.scaling[a]
        return y

    monkeypatch.setattr(O, "linear", linear)
    monkeypatch.setattr(O.PVariantOracle, "lin", lin)
    O.fake_quant_calls = calls
    return O


def bf(x):
    return x.to(torch.bfloat16).float()


def _setup(n_cond=2, strict=False, seed=1, alpha=None):
    from oracle import unigen_oracle as O
    from unigen_b200.model import FluxArch
    from unigen_b200.pvariant import UniCombineFlux
    cfg = O.FluxConfig.tiny()
    types_ = ["depth", "canny", "subject"][:n_cond]
    adapters = ["denoise"] + types_
    sd = {k: bf(v) for k, v in O.init_pvariant_state_dict(cfg, adapters, rank=4, seed=seed).items()}
    inp = O.make_multi_inputs(cfg, 256, 256, condition_types=tuple(types_))
    for k in ("hidden_states", "encoder_hidden_states"):
        inp[k] = bf(inp[k])
    inp["condition_hidden_states"] = [bf(c) for c in inp["condition_hidden_states"]]
    model = UniCombineFlux(FluxArch.tiny(), device="cuda", lora_rank=4, strict_mask=strict)
    if alpha is None:
        model.load_state_dict(sd, adapters=adapters, condition_types=types_, scaling={a: 1.0 for a in adapters})
    else:
        model.load_state_dict(sd, adapters=adapters, condition_types=types_, lora_alpha=alpha)
    args = (inp["hidden_states"], inp["condition_hidden_states"], inp["condition_ids"], types_, inp["encoder_hidden_states"],
            inp["pooled_projections"], inp["timestep"], inp["img_ids"], inp["txt_ids"])
    return cfg, sd, adapters, args, model


def _cu(args):
    return [[t.cuda() for t in a] if isinstance(a, list) and a and torch.is_tensor(a[0]) else (a.cuda() if torch.is_tensor(a) else a)
            for a in args]


@pytest.mark.parametrize("case", ["n_cond1", "n_cond2", "strict_mask", "add_cond_attn"])
def test_tiny_quantised_pvariant_matches_fake_quant_oracle(fake_quant_pvariant_oracle, case):
    O = fake_quant_pvariant_oracle
    n_cond = 1 if case == "n_cond1" else 2
    cfg, sd, adapters, args, model = _setup(n_cond, strict=case == "strict_mask")
    oracle = O.PVariantOracle(cfg, sd, adapters, {a: 1.0 for a in adapters}, strict_mask=case == "strict_mask")
    oracle.record = True
    cond = case == "add_cond_attn"
    oracle.add_cond_attn = model.add_cond_attn = cond
    want = oracle.forward(*args, return_condition_latents=cond)
    # every quantised linear of the tiny weave went through the fake quantiser (12 per double block and stream call, 5 per single)
    assert O.fake_quant_calls["n"] >= 12 * cfg.num_layers + 5 * cfg.num_single_layers
    model.quantize_fp8()
    model.trace = {}
    got = model(*_cu(args), return_condition_latents=cond)
    if cond:
        (got, got_c), (want, want_c) = got, want
        assert len(got_c) == n_cond and all(rel_l2(g, w) < 1e-2 for g, w in zip(got_c, want_c))
    checked = {k: rel_l2(model.trace[k], v) for k, v in oracle.trace.items() if k in model.trace}
    # per double block: text, image and each condition stream; per single block: [text | image] and each condition stream
    assert len(checked) >= (2 + n_cond) * cfg.num_layers + (1 + n_cond) * cfg.num_single_layers
    bad = {k: v for k, v in checked.items() if v > 1e-2}
    assert not bad, bad
    cos = F.cosine_similarity(got.float().cpu().flatten(), want.flatten(), dim=0).item()
    assert cos >= 0.999 and rel_l2(got, want) < 1e-2, (cos, rel_l2(got, want))
    assert torch.isfinite(got.float()).all()


def _fp8_lora_operands(model):
    return [t for p in model.lora.values() if p.w_scale is not None for t in (p.aw, p.bw, p.aq, p.aws, p.w2)]


def test_lora_hooks_on_a_quantised_model_follow_the_fake_quant_oracle(fake_quant_pvariant_oracle):
    """enable_lora / set_adapter over the carriers of a quantised model change its output as the oracle's enable_lora changes
    the fake-quant oracle's, the alpha != r restore quirk included; the fp8-side LoRA operands are rewritten in place."""
    O = fake_quant_pvariant_oracle
    from unigen_b200.lora_switching_module import enable_lora
    alpha = {"denoise": 4.0, "depth": 4.0, "canny": 8.0}  # rank 4: canny has lora_alpha = 2 r
    cfg, sd, adapters, args, model = _setup(2, seed=2, alpha=alpha)
    model.quantize_fp8()
    mods = model.lora_modules()
    ptrs = [t.data_ptr() for t in _fp8_lora_operands(model)]
    assert len(ptrs) == 5 * 3 * (cfg.num_layers + cfg.num_single_layers)

    class Stub:
        def __init__(self):
            self.active_adapters, self.r, self.lora_alpha = list(adapters), {a: 4 for a in adapters}, dict(alpha)
            self.scaling = {a: alpha[a] / 4 for a in adapters}

        def set_scale(self, a, s):
            self.scaling[a] = s * self.lora_alpha[a] / self.r[a]

    stub = Stub()

    def oracle_out():
        return O.PVariantOracle(cfg, sd, adapters, dict(stub.scaling)).forward(*args)

    def native_out():
        return model(*_cu(args)).float().cpu()

    want0, got0 = oracle_out(), native_out()
    assert rel_l2(got0, want0) < 1e-2
    with O.enable_lora([stub], ["denoise", "depth"]), enable_lora(mods, ["denoise", "depth"]):
        assert stub.scaling["canny"] == 0 and all(m.scaling == stub.scaling for m in mods)
        want1, got1 = oracle_out(), native_out()
    assert rel_l2(got1, want1) < 1e-2
    assert rel_l2(want1, want0) > 5e-3 and rel_l2(got1, got0) > 5e-3
    assert stub.scaling == {"denoise": 1.0, "depth": 1.0, "canny": 4.0} and all(m.scaling == stub.scaling for m in mods)
    want2, got2 = oracle_out(), native_out()
    assert rel_l2(got2, want2) < 1e-2 and rel_l2(got2, got0) > 5e-3
    for m in mods:
        m.set_adapter(["denoise", "depth"])
    stub.scaling["canny"] = 0.0
    assert rel_l2(native_out(), oracle_out()) < 1e-2
    assert [t.data_ptr() for t in _fp8_lora_operands(model)] == ptrs


def test_quantised_pvariant_graph_replay_equals_eager():
    cfg, sd, adapters, args, model = _setup(2)
    model.quantize_fp8()
    args = _cu(args)
    eager = model(*args).clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        model(*args)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = model(*args)
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, eager)


def test_bf16_pvariant_unchanged_when_another_is_quantised():
    cfg, sd, adapters, args, model = _setup(2)
    args = _cu(args)
    before = model(*args).clone()
    _, _, _, _, other = _setup(2)
    other.quantize_fp8()
    other(*args)
    assert torch.equal(model(*args), before)


def test_quantize_fp8_interface_and_refusals(tmp_path):
    from unigen_b200.model import FP8, FluxArch
    from unigen_b200.ops import UgError
    from unigen_b200.pvariant import UniCombineFlux
    cfg, sd, adapters, args, model = _setup(2)
    with pytest.raises(UgError):
        UniCombineFlux(FluxArch.tiny(), device="cuda").quantize_fp8()  # before load_state_dict
    n_before, mods = len(model.state_dict()), model.lora_modules()
    assert model.quantize_fp8() is model and model.linear_dtype == FP8
    assert model.quantize_fp8() is model
    assert n_before - len(model.state_dict()) == 12 * cfg.num_layers + 5 * cfg.num_single_layers
    assert model.lora_modules() == mods
    assert all(w.fp8 for w in model.double + model.single) and model.double[0].qkv[0].dtype == FP8
    assert model.x_embedder_w[0].dtype == torch.bfloat16 and model.lora["x_embedder"].w_scale is None
    with pytest.raises(UgError):
        model.load_state_dict(sd, adapters=adapters, condition_types=args[3])
    model.lora_mode = "epilogue"
    with pytest.raises(UgError):
        model(*_cu(args))
    model.lora_mode = "mma"
    assert torch.isfinite(model(*_cu(args)).float()).all()
    import torch.distributed as dist
    from unigen_b200.parallel import SequenceParallelUniCombineFlux
    own = not dist.is_initialized()
    if own:
        dist.init_process_group("gloo", init_method=f"file://{tmp_path / 'pg'}", rank=0, world_size=1)
    try:
        sp = SequenceParallelUniCombineFlux(FluxArch.tiny(), device="cuda", lora_rank=4)
        sp.load_state_dict(sd, adapters=adapters, condition_types=args[3], scaling={a: 1.0 for a in adapters})
        sp.quantize_fp8()
        with pytest.raises(UgError):
            sp(*_cu(args))
        sp.sp_enabled = False  # the same object as a single-GPU model runs
        assert torch.equal(sp(*_cu(args)), model(*_cu(args)))
    finally:
        if own:
            dist.destroy_process_group()


def test_cfg4_quantised_pvariant_against_bf16():
    """Full size (1024^2 + 3 conditions, 16 896 tokens): the fp8 velocity against the bf16 one on the same weights and inputs,
    and the step time of both legs (eager launches, CUDA events)."""
    import bench
    from unigen_b200.pvariant import UniCombineFlux
    m16, inp, S = bench.build_pvariant(UniCombineFlux, "cuda", 3)
    m8, inp8, _ = bench.build_pvariant(UniCombineFlux, "cuda", 3)
    m8.quantize_fp8()
    ms = {}
    outs = {}
    for name, m in (("bf16", m16), ("fp8", m8)):
        outs[name] = m(*inp).float()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(2):
            m(*inp)
        b.record()
        b.synchronize()
        ms[name] = a.elapsed_time(b) / 2
    cos = F.cosine_similarity(outs["fp8"].flatten(), outs["bf16"].flatten(), dim=0).item()
    print(f"cfg4 P-variant ({S} tokens): velocity fp8 vs bf16 cosine {cos:.6f} rel-L2 {rel_l2(outs['fp8'], outs['bf16']):.4e}; "
          f"eager step bf16 {ms['bf16']:.1f} ms, fp8 {ms['fp8']:.1f} ms ({ms['bf16'] / ms['fp8']:.3f}x)")
    assert torch.isfinite(outs["fp8"]).all() and torch.isfinite(outs["bf16"]).all()
    assert cos >= 0.999
