"""Row reductions (LayerNorm-modulate, GroupNorm, per-head RMSNorm, row softmax) on the data where fp32 reductions go wrong:
rows with a large mean against their spread, a few huge channels, constant rows, values near 1e-20 and zeros.

Every reference is float64 on the CPU, computed from the same bf16 inputs the kernel reads. A bf16 output is compared with the
fp64 result rounded to bf16 (`want`):
  * every element is within one bf16 ulp of `want` (plus the element's fp32 error bound `err`, which only matters where the
    output cancels to near zero);
  * the count of elements that differ from `want` at all stays under 2 * sum_i min(1, err_i / ulp_i) + 4. An fp32 result off by
    at most err_i from the exact value rounds to a different bf16 neighbour only if a rounding boundary lies within err_i of the
    exact value, which for values spread over the bf16 grid happens with probability <= err_i / ulp_i. The factor 2 and the 4
    cover the spread of that count.
`err` restates the fp32 arithmetic each kernel is specified to do (U = 2^-24, the fp32 unit roundoff):
  * a mean of bf16 values: U * (2 |mean| + 4 mean|x|) (the fp32 sum, the division and the rounding of a mean stored as fp32);
  * an rstd: relative U * (8 + sqrt(n)) (a sum of n squares in blocked fp32 order, rsqrtf's 2 ulp, the products that follow);
  * each product / sum of the epilogue: 2 U of its magnitude.
A GroupNorm with a one-pass E[x^2] - mean^2 variance (rstd ~1e-3 off at mean / std = 100) fails both bars at mean / std >= 100."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

BF16, F64 = torch.bfloat16, torch.float64
U = 2.0 ** -24
KINDS = ("offset1", "offset1e2", "offset1e3", "outlier", "constant", "tiny", "zero")


def bf16_ulp(v):
    """Spacing of the bf16 grid at |v| (fp64 tensor); the smallest bf16 subnormal at 0."""
    _, e = torch.frexp(v.abs())
    ulp = torch.ldexp(torch.ones_like(v), (e - 8).clamp_min(-133))
    return torch.where(v == 0, torch.full_like(v, 2.0 ** -133), ulp)


def assert_bf16_matches(got, ref, err, what):
    """got: kernel output (bf16, any device); ref: fp64 reference; err: fp64 bound of the kernel's fp32 error (broadcastable)."""
    got = got.detach().cpu().to(F64)
    ref = ref.to(F64)
    err = torch.broadcast_to(err.to(F64), ref.shape)
    want = ref.to(BF16).to(F64)
    assert not torch.isnan(got).any(), f"{what}: NaN in the output"
    ulp = bf16_ulp(want)
    off = (got - want).abs() > ulp + err
    if off.any():
        i = off.nonzero()[0].tolist()
        raise AssertionError(f"{what}: {int(off.sum())} of {off.numel()} elements are more than one bf16 ulp from the fp64 reference; "
                             f"first at {i}: got {got[tuple(i)].item():.9g}, want {want[tuple(i)].item():.9g}, "
                             f"ref {ref[tuple(i)].item():.12g}, err bound {err[tuple(i)].item():.3g}")
    flips = int((got != want).sum())
    allowed = 2.0 * float((err / bf16_ulp(ref)).clamp(max=1.0).sum()) + 4
    assert flips <= allowed, (f"{what}: {flips} of {got.numel()} elements differ from bf16(fp64 reference), the fp32 arithmetic "
                              f"allows {allowed:.1f}")


def make_rows(kind, n, d, g):
    """n rows of d values of one kind (fp64 before the bf16 rounding)."""
    z = torch.randn(n, d, generator=g, dtype=F64)
    if kind.startswith("offset"):
        return float(kind[6:]) + z  # mean / std = 1, 1e2, 1e3 (bf16 spacing quantises the noise at 1e3; the reference sees it too)
    if kind == "outlier":
        for r in range(n):
            idx = torch.randperm(d, generator=g)[:2 + r % 3]
            mag = 1e3 * 30.0 ** torch.rand(len(idx), generator=g, dtype=F64)
            sign = torch.where(torch.rand(len(idx), generator=g) < 0.5, -1.0, 1.0).to(F64)
            z[r, idx] = sign * mag
        return z
    if kind == "constant":
        return torch.randn(n, 1, generator=g, dtype=F64).expand(n, d) * 5
    if kind == "tiny":
        return 1e-20 * z
    assert kind == "zero"
    return torch.zeros(n, d, dtype=F64)


def mean_err(x, dim):
    """Bound of the fp32 mean of bf16 values x (fp64) along dim (keepdim)."""
    return U * (2 * x.mean(dim, keepdim=True).abs() + 4 * x.abs().mean(dim, keepdim=True))


# ---------------------------------------------------------------------------------------------------------------------------
# a. LayerNorm (no affine) + (1 + scale) * x + shift
# ---------------------------------------------------------------------------------------------------------------------------
def ln_ref(x, shift, scale, eps=1e-6):
    """x: fp64 [..., d]; shift / scale: fp64 broadcastable. Returns (y, err)."""
    d = x.shape[-1]
    mu = x.mean(-1, keepdim=True)
    xc = x - mu
    r = 1.0 / torch.sqrt((xc * xc).mean(-1, keepdim=True) + eps)
    t = xc * r * (1 + scale)
    y = t + shift
    err = (mean_err(x, -1) * r * (1 + scale).abs() + U * (8 + math.sqrt(d)) * t.abs() + 2 * U * (shift.abs() + y.abs()))
    return y, err


def ln_inputs(B, R, d, seed):
    """bf16 [B, R, d] rows cycling through KINDS (row r of every sample has kind r % 7), shift / scale fp32 [B, d]."""
    g = torch.Generator().manual_seed(seed)
    x = torch.empty(B, R, d, dtype=F64)
    for i, kind in enumerate(KINDS):
        rows = list(range(i, R, len(KINDS)))
        if rows:
            x[:, rows] = make_rows(kind, B * len(rows), d, g).view(B, len(rows), d)
    shift = torch.randn(B, d, generator=g)
    scale = 0.5 * torch.randn(B, d, generator=g)
    return x.to(BF16), shift, scale


def strided(x, pad=8):
    """The same values as a view with a row stride of d + 2 * pad (16-byte aligned start)."""
    B, R, d = x.shape
    big = torch.full((B, R, d + 2 * pad), 3.0, dtype=x.dtype, device="cuda")
    v = big[:, :, pad:pad + d]
    v.copy_(x.cuda())
    return v


def out_buffer(B, R, d, pad=8):
    """Output view [B, R, d] with a row stride of d + 2 * pad, inside a buffer with one guard row; fill 7.0."""
    big = torch.full((B, R + 1, d + 2 * pad), 7.0, dtype=BF16, device="cuda")
    return big, big[:, :R, pad:pad + d]


def assert_guards(big, R, d, pad=8):
    assert (big[:, R] == 7.0).all(), "written past the last row"
    assert (big[:, :, :pad] == 7.0).all() and (big[:, :, pad + d:] == 7.0).all(), "written outside the row's columns"


def check_ln_rows(got, x, shift, scale, what):
    """got / x: [B, R, d]; shift / scale: per-row fp64 [B, R, d] (or broadcastable)."""
    xf = x.cpu().to(F64)
    want, err = ln_ref(xf, shift, scale)
    got = got.cpu()
    for i, kind in enumerate(KINDS):
        sl = (slice(None), slice(i, None, len(KINDS)))
        if got[sl].numel() == 0:
            continue
        assert_bf16_matches(got[sl], want[sl], err[sl], f"{what} [{kind} rows]")
        if kind in ("constant", "zero"):  # var = 0: (x - mean) is exactly 0, the output is exactly bf16(shift)
            assert torch.equal(got[sl], torch.broadcast_to(shift, want.shape)[sl].to(torch.float32).to(BF16)), f"{what} [{kind}]"


# (B, R, d): one-warp V=2 (d = 8, 40, 512), two-warp V=3 (d = 520), two-warp V=6 (2560), one-warp V=16 (3080, 4096),
# rows kernel (1536, 2048, 3072 with few rows; ragged last block), persistent stream kernel (3072, batch 1, 4608 rows)
LN_PLAIN = [(2, 21, 8), (1, 35, 40), (2, 30, 512), (2, 23, 520), (1, 29, 2560), (1, 22, 3080), (2, 21, 4096), (2, 23, 1536),
            (1, 29, 2048), (2, 25, 3072), (1, 4608, 3072)]


@pytest.mark.parametrize("B,R,d", LN_PLAIN)
def test_ln_modulate_hard_rows(ug, B, R, d):
    x, shift, scale = ln_inputs(B, R, d, seed=d + R)
    big, out = out_buffer(B, R, d)
    ug.ln_modulate(strided(x), out, shift.cuda(), scale.cuda())
    torch.cuda.synchronize()
    assert_guards(big, R, d)
    check_ln_rows(out, x, shift.to(F64)[:, None], scale.to(F64)[:, None], f"ln_modulate d={d}")


@pytest.mark.parametrize("B,R,d", LN_PLAIN)
def test_ln_modulate_fp8_hard_rows(ug, B, R, d):
    """The fp8 form: e4m3 rows + scales bit for bit equal to quant_rows_fp8(ln_modulate(x)), whose bf16 stage meets the bar."""
    x, shift, scale = ln_inputs(B, R, d, seed=d + R + 1)
    xs, sh, sc = strided(x), shift.cuda(), scale.cuda()
    nx = torch.empty(B, R, d, dtype=BF16, device="cuda")
    ug.ln_modulate(xs, nx, sh, sc)
    check_ln_rows(nx, x, shift.to(F64)[:, None], scale.to(F64)[:, None], f"ln_modulate d={d}")
    qw, sw = ug.quant_rows_fp8(nx)
    qbig = torch.full((B, R + 1, d + 16), 0x55, dtype=torch.uint8, device="cuda")
    q = qbig[:, :R, 8:8 + d].view(torch.float8_e4m3fn)
    s = torch.full((B, R + 1), -1.0, device="cuda")
    ug.ln_modulate_fp8(xs, q, s[:, :R], sh, sc)
    torch.cuda.synchronize()
    assert torch.equal(q.view(torch.uint8), qw.view(torch.uint8)) and torch.equal(s[:, :R], sw)
    assert (qbig[:, R] == 0x55).all() and (qbig[:, :, :8] == 0x55).all() and (qbig[:, :, 8 + d:] == 0x55).all()
    assert (s[:, R] == -1.0).all()


def seg_inputs(B, R, d, seed):
    x, _, _ = ln_inputs(B, R, d, seed)
    g = torch.Generator().manual_seed(seed + 7)
    bounds = [0, R // 3, R // 3 + 1, R]
    table = torch.randn(len(bounds) - 1, B, 2, d, generator=g)  # [segment, sample, shift | scale, d]
    table[:, :, 1] *= 0.5
    seg = torch.zeros(R, dtype=torch.long)
    for s in range(len(bounds) - 1):
        seg[bounds[s]:bounds[s + 1]] = s
    per_row = table[seg].permute(1, 0, 2, 3).to(F64)  # [B, R, 2, d]
    return x, bounds, table, per_row[:, :, 0], per_row[:, :, 1]


# d = 1536 (two-warp V=3) and 2560 / 3072 (two-warp V=6) take the warp kernels through the segment / slot entry points, plus
# one shape of every other warp kernel
LN_SEGS = [(2, 23, 1536), (1, 22, 2560), (2, 21, 3072), (2, 21, 40), (1, 23, 520), (1, 22, 4096)]


@pytest.mark.parametrize("B,R,d", LN_SEGS)
def test_ln_modulate_segs_hard_rows(ug, B, R, d):
    x, bounds, table, shift, scale = seg_inputs(B, R, d, seed=d + 3)
    tc = table.cuda()
    big, out = out_buffer(B, R, d)
    ug.ln_modulate_segs(strided(x), out, tc[0, :, 0], tc[0, :, 1], bounds, tc.stride(0))
    torch.cuda.synchronize()
    assert_guards(big, R, d)
    check_ln_rows(out, x, shift, scale, f"ln_modulate_segs d={d}")


@pytest.mark.parametrize("B,R,d", LN_SEGS)
def test_ln_modulate_segs_fp8_hard_rows(ug, B, R, d):
    x, bounds, table, shift, scale = seg_inputs(B, R, d, seed=d + 4)
    tc, xs = table.cuda(), strided(x)
    nx = torch.empty(B, R, d, dtype=BF16, device="cuda")
    ug.ln_modulate_segs(xs, nx, tc[0, :, 0], tc[0, :, 1], bounds, tc.stride(0))
    check_ln_rows(nx, x, shift, scale, f"ln_modulate_segs d={d}")
    qw, sw = ug.quant_rows_fp8(nx)
    q = torch.empty(B, R, d, dtype=torch.float8_e4m3fn, device="cuda")
    s = torch.empty(B, R, device="cuda")
    ug.ln_modulate_segs_fp8(xs, q, s, tc[0, :, 0], tc[0, :, 1], bounds, tc.stride(0))
    assert torch.equal(q.view(torch.uint8), qw.view(torch.uint8)) and torch.equal(s, sw)


@pytest.mark.parametrize("d", [40, 520, 1536, 2560, 3072, 4096])
def test_ln_modulate_slots_hard_rows(ug, d):
    E, C, B, N = 3, 9, 2, 40
    x, _, _ = ln_inputs(1, E * C, d, seed=d + 5)
    g = torch.Generator().manual_seed(d)
    slot_token = torch.randint(-1, B * N, (E * C,), generator=g, dtype=torch.int32)
    table = torch.randn(E, B + 1, 2, d, generator=g)
    table[:, :, 1] *= 0.5
    idx = torch.where(slot_token < 0, torch.full_like(slot_token, B), slot_token // N).long()
    e = torch.arange(E * C) // C
    per_row = table[e, idx].to(F64)  # [E * C, 2, d]
    tc = table.cuda()
    xs = strided(x)[0]
    big = torch.full((E * C + 1, d + 16), 7.0, dtype=BF16, device="cuda")
    out = big[:E * C, 8:8 + d]
    ug.ln_modulate_slots(xs, out, tc[:, :, 0], tc[:, :, 1], slot_token.cuda(), E, C, N, B)
    torch.cuda.synchronize()
    assert_guards(big[None], E * C, d)
    check_ln_rows(out[None], x, per_row[None, :, 0], per_row[None, :, 1], f"ln_modulate_slots d={d}")


# ---------------------------------------------------------------------------------------------------------------------------
# b. GroupNorm over NHWC
# ---------------------------------------------------------------------------------------------------------------------------
def gn_inputs(B, P, C, G, kinds, seed):
    """bf16 NHWC-flat [B, P, C]: group k of every image holds data of kind kinds[k % len(kinds)]."""
    g = torch.Generator().manual_seed(seed)
    cpg = C // G
    x = torch.empty(B, P, C, dtype=F64)
    for k in range(G):
        kind = kinds[k % len(kinds)]
        x[:, :, k * cpg:(k + 1) * cpg] = make_rows(kind, B, P * cpg, g).view(B, P, cpg)
    gamma = (1 + 0.2 * torch.randn(C, generator=g)).to(BF16)
    beta = (0.3 * torch.randn(C, generator=g)).to(BF16)
    return x.to(BF16), gamma, beta


def gn_ref(x, gamma, beta, G, silu, eps=1e-6, pixels=None):
    """fp64 GroupNorm (+ SiLU) of x [B, P, C] and its fp32 error bound; `pixels` selects the output pixels returned."""
    B, P, C = x.shape
    cpg = C // G
    xg = x.view(B, P, G, cpg)
    n = P * cpg
    mu = xg.mean((1, 3), keepdim=True)
    var = ((xg - mu) ** 2).mean((1, 3), keepdim=True)
    merr = U * (2 * mu.abs() + 4 * xg.abs().mean((1, 3), keepdim=True))
    r = 1.0 / torch.sqrt(var + eps)
    if pixels is not None:
        xg = xg[:, pixels]
    a = r * gamma.to(F64).view(G, cpg)
    t = (xg - mu) * a
    z = t + beta.to(F64).view(G, cpg)
    err = merr * a.abs() + U * (16 + math.sqrt(n)) * t.abs() + 2 * U * (beta.to(F64).view(G, cpg).abs() + z.abs())
    if silu:
        sig = torch.sigmoid(z)
        y = z * sig
        # __expf / __fdividef (MUFU ex2 + rcp): a few ulp, plus |z| U from rounding z * log2(e)
        # __fdividef returns 0 for divisors beyond 2^126: outputs below |z| 2^-126 may flush to zero
        err = err * (sig * (1 + z * (1 - sig))).abs() + U * (8 + 2 * z.abs()) * y.abs() + 2.0 ** -126 * (1 + z.abs())
        z = y
    return z.reshape(B, -1, C), err.reshape(B, -1, C)


def check_gn(got, x, gamma, beta, G, silu, kinds, what, pixels=None):
    B, P, C = x.shape
    cpg = C // G
    want, err = gn_ref(x.to(F64), gamma, beta, G, silu, pixels=pixels)
    got = got.cpu().view(B, P, C)
    if pixels is not None:
        got = got[:, pixels]
    failures = []
    for i, kind in enumerate(kinds):
        cols = [k * cpg + j for k in range(i, G, len(kinds)) for j in range(cpg)]
        if not cols:
            continue
        try:
            assert_bf16_matches(got[..., cols], want[..., cols], err[..., cols], f"{what} [{kind} groups]")
            if kind in ("constant", "zero"):  # var = 0: x - mean is exactly 0, the output is exactly bf16(beta) (SiLU of it)
                b = beta.float()[cols]
                exact = (b * torch.sigmoid(b.double()).float()).to(BF16) if silu else b.to(BF16)
                # SiLU runs on MUFU approximations: within one ulp of SiLU(beta), exactly beta without it
                if not silu:
                    assert torch.equal(got[..., cols], torch.broadcast_to(exact, got[..., cols].shape)), f"{what} [{kind}]"
        except AssertionError as e:
            failures.append(str(e))
    assert not failures, "\n".join(failures)


GN_SHAPES = [  # (B, H, W, C, G): cpg 2 / 4 / 16, C 64 / 128 / 192 / 512, pixels 1 / 63 / 64 * 64
    (3, 7, 9, 64, 32), (1, 1, 1, 128, 32), (3, 1, 1, 192, 48), (3, 64, 64, 192, 12), (1, 64, 64, 512, 32), (3, 9, 7, 128, 8),
    (1, 64, 64, 128, 64)]


@pytest.mark.parametrize("silu", [False, True])
@pytest.mark.parametrize("B,H,W,C,G", GN_SHAPES)
def test_groupnorm_hard_groups(ug, B, H, W, C, G, silu):
    ops = ug
    kinds = KINDS  # every shape has >= 7 groups: each kind gets at least one group
    x, gamma, beta = gn_inputs(B, H * W, C, G, kinds, seed=B + H + C + G)
    xn = x.view(B, H, W, C).cuda()
    got = ops.groupnorm(xn, gamma.cuda(), beta.cuda(), G, silu_act=silu)
    again = ops.groupnorm(xn, gamma.cuda(), beta.cuda(), G, silu_act=silu)
    inplace = xn.clone()
    ops.groupnorm(inplace, gamma.cuda(), beta.cuda(), G, silu_act=silu, out=inplace)
    torch.cuda.synchronize()
    assert torch.equal(got, again), "two runs on the same input differ"
    assert torch.equal(inplace, got), "in place (out = x) differs from out of place"
    check_gn(got, x, gamma, beta, G, silu, kinds, f"groupnorm B={B} {H}x{W} C={C} G={G} silu={silu}")


@pytest.mark.parametrize("ratio", ["offset1", "offset1e2", "offset1e3"])
def test_groupnorm_offset_ratio_issue_shape(ug, ratio):
    """The VAE's widest GroupNorm (64 x 64 pixels, c = 512, 32 groups) with every group at one mean / std ratio."""
    ops = ug
    x, gamma, beta = gn_inputs(1, 64 * 64, 512, 32, (ratio,), seed=11)
    got = ops.groupnorm(x.view(1, 64, 64, 512).cuda(), gamma.cuda(), beta.cuda(), 32, silu_act=True)
    check_gn(got, x, gamma, beta, 32, True, (ratio,), f"groupnorm 64x64 c=512 {ratio}")


def test_groupnorm_megapixel_many_chunks(ug):
    """One 1024 x 1024 image at c = 128: the statistics pass takes its maximum number of chunks (UG_GROUPNORM_MAX_CHUNKS)."""
    from unigen_b200 import _lib
    ops = ug
    P, C, G = 1024 * 1024, 128, 32
    assert (P + 63) // 64 >= _lib.UG_GROUPNORM_MAX_CHUNKS
    x, gamma, beta = gn_inputs(1, P, C, G, KINDS, seed=5)
    xn = x.view(1, 1024, 1024, C).cuda()
    got = ops.groupnorm(xn, gamma.cuda(), beta.cuda(), G, silu_act=True)
    again = ops.groupnorm(xn, gamma.cuda(), beta.cuda(), G, silu_act=True)
    torch.cuda.synchronize()
    assert torch.equal(got, again)
    pixels = torch.cat([torch.arange(0, P, 97), torch.tensor([P - 1])])
    check_gn(got, x, gamma, beta, G, True, KINDS, "groupnorm 1024x1024 c=128", pixels=pixels)


# ---------------------------------------------------------------------------------------------------------------------------
# c. Per-head RMSNorm (+ RoPE): qk_rmsnorm_rope, the fused epilogue of gemm / gemm_fp8, qkv_scatter
# ---------------------------------------------------------------------------------------------------------------------------
def head_inputs(S, H, dh, seed):
    """[S, H * dh] fp64 rows: head 0 all zero, head 1 N(0,1) * 1e3, head 2 N(0,1) with outlier channels, the rest N(0,1)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(S, H, dh, generator=g, dtype=F64)
    x[:, 0] = 0
    x[:, 1] *= 1e3
    for s in range(S):
        idx = torch.randperm(dh, generator=g)[:2 + s % 3]
        x[s, 2, idx] = torch.where(torch.rand(len(idx), generator=g) < 0.5, -1.0, 1.0).to(F64) * 1e3 * 30.0 ** torch.rand(
            len(idx), generator=g, dtype=F64)
    return x.reshape(S, H * dh)


def rms_rope_ref(x, w, cs, dh, eps=1e-6, xerr=None):
    """x fp64 [S, H * dh] (one weight w [dh] for every head), cs: fp64 [S, dh // 2, 2] or None; xerr: error bound of the fp32
    values the kernel normalises (a GEMM accumulator + bias). Returns (y, err)."""
    S = x.shape[0]
    xh = x.view(S, -1, dh)
    r = 1.0 / torch.sqrt((xh * xh).mean(-1, keepdim=True) + eps)
    t = xh * r * w.to(F64)
    rel = U * (12 + math.sqrt(dh))
    et = rel * t.abs() + (0 if xerr is None else xerr.view(S, -1, dh) * r * w.to(F64).abs())
    if cs is None:
        return t.reshape(S, -1), et.reshape(S, -1)
    c, s = cs[:, None, :, 0], cs[:, None, :, 1]
    t0, t1 = t[..., 0::2], t[..., 1::2]
    e0, e1 = et[..., 0::2], et[..., 1::2]
    y = torch.stack([t0 * c - t1 * s, t1 * c + t0 * s], -1).reshape(S, -1, dh)
    m = torch.stack([(t0 * c).abs() + (t1 * s).abs(), (t1 * c).abs() + (t0 * s).abs()], -1).reshape(S, -1, dh)
    me = torch.stack([e0 * c.abs() + e1 * s.abs(), e1 * c.abs() + e0 * s.abs()], -1).reshape(S, -1, dh)
    # cancellation in x0 cos - x1 sin: the floor 2^-20 x the head's RMS
    floor = 2.0 ** -20 * y.pow(2).mean(-1, keepdim=True).sqrt()
    return y.reshape(S, -1), (rel * m + me + floor).reshape(S, -1)


def rope(ug, S, dh):
    axes = (16, 56, 56) if dh == 128 else (8, 28, 28)
    ids = torch.stack([torch.zeros(S), torch.arange(S) // 13, torch.arange(S) % 13], 1).float()
    table = ug.rope_table(ids.cuda(), axes)
    return table, table.cpu().to(F64).view(S, dh // 2, 2)


def check_heads(got, ref, err, dh, what):
    got = got.cpu()
    assert (got.view(got.shape[0], -1, dh)[:, 0] == 0).all(), f"{what}: the all-zero head is not exactly 0"
    assert_bf16_matches(got, ref, err, what)


@pytest.mark.parametrize("dh", [64, 128])
@pytest.mark.parametrize("use_rope", [False, True])
def test_qk_rmsnorm_rope_hard_heads(ug, dh, use_rope):
    S, H = 77, 5
    x = torch.cat([head_inputs(S, H, dh, seed=dh), head_inputs(S, H, dh, seed=dh + 1)], 1).to(BF16)  # q heads | k heads
    w = (1 + 0.1 * torch.randn(2, dh, generator=torch.Generator().manual_seed(dh))).to(BF16)
    table, cs = rope(ug, S, dh)
    buf = torch.full((1, S, 2 * H * dh + 16), 7.0, dtype=BF16, device="cuda")
    qk = buf[:, :, 8:8 + 2 * H * dh]
    qk.copy_(x[None].cuda())
    ug.qk_rmsnorm_rope(qk, 2 * H, dh, w.cuda(), table if use_rope else None, heads_per_weight=H)
    torch.cuda.synchronize()
    assert (buf[..., :8] == 7.0).all() and (buf[..., 8 + 2 * H * dh:] == 7.0).all()
    for part in range(2):
        sl = slice(part * H * dh, (part + 1) * H * dh)
        ref, err = rms_rope_ref(x[:, sl].to(F64), w[part], cs if use_rope else None, dh)
        check_heads(qk[0, :, sl], ref, err, dh, f"qk_rmsnorm_rope dh={dh} rope={use_rope} part={part}")


def qkv_projection_inputs(S, H, dh, seed):
    """A q|k|v projection whose fp32 accumulator is exact: w = identity, so acc = x (+ bias); head 0 of q and of k has zero
    weight rows and a zero bias (an all-zero head)."""
    D = H * dh
    x = torch.cat([head_inputs(S, H, dh, seed), head_inputs(S, H, dh, seed + 1), torch.randn(S, D, dtype=F64)], 1).to(BF16)
    w = torch.eye(3 * D, dtype=BF16)
    bias = (0.25 * torch.randn(3 * D, generator=torch.Generator().manual_seed(seed))).to(BF16)
    for part in range(2):
        w[part * D:part * D + dh] = 0
        bias[part * D:part * D + dh] = 0
    return x, w, bias


def check_qkv(out, acc, acc_err, nw, cs, H, dh, what):
    """out [S, 3D] bf16 from the fused epilogue; acc: the exact fp64 accumulator + bias, acc_err: the fp32 error bound of it."""
    D = H * dh
    for part in range(2):
        sl = slice(part * D, (part + 1) * D)
        ref, err = rms_rope_ref(acc[:, sl], nw[part], cs, dh, xerr=acc_err[:, sl])
        check_heads(out[:, sl], ref, err, dh, f"{what} part={part}")
    assert_bf16_matches(out[:, 2 * D:], acc[:, 2 * D:], acc_err[:, 2 * D:], f"{what} v columns")


@pytest.mark.parametrize("variant", [0, 1, 2, 4, 5])
@pytest.mark.parametrize("dh", [64, 128])
@pytest.mark.parametrize("use_rope", [False, True])
def test_gemm_fused_qk_norm_hard_heads(ug, variant, dh, use_rope):
    S, H = 200, 384 // dh
    x, w, bias = qkv_projection_inputs(S, H, dh, seed=dh + variant)
    prod = x.to(F64) @ w.to(F64).t()
    acc, acc_err = prod + bias.to(F64), 3 * U * (prod.abs() + bias.to(F64).abs())  # + bias: cancellation is bounded by the terms
    nw = (1 + 0.1 * torch.randn(2, dh, generator=torch.Generator().manual_seed(3))).to(BF16)
    table, cs = rope(ug, S, dh)
    qk = dict(weight=nw.cuda(), head_dim=dh, d=H * dh, cos_sin=table if use_rope else None, eps=1e-6)
    out = ug.gemm(x[None].cuda(), w.cuda(), bias=bias.cuda(), variant=variant, qk_norm=qk)
    check_qkv(out[0], acc, acc_err, nw, cs if use_rope else None, H, dh, f"gemm qk_norm variant={variant} dh={dh} rope={use_rope}")


@pytest.mark.parametrize("dh", [64, 128])
def test_gemm_fp8_fused_qk_norm_hard_heads(ug, dh):
    """e4m3 operands with an exact accumulator: a = e4m3(x / a_scale) per row, w = identity (1.0 is an e4m3 value) with per-column
    scales 2^k, so acc * a_scale * w_scale carries two fp32 roundings."""
    S, H = 200, 384 // dh
    D = 3 * H * dh
    x, _, bias = qkv_projection_inputs(S, H, dh, seed=dh + 9)
    xf = x.to(torch.float32)
    a_s = (xf.abs().amax(1) / 448).clamp_min(1e-30)
    a_q = (xf / a_s[:, None]).to(torch.float8_e4m3fn)
    wq = torch.eye(D).to(torch.float8_e4m3fn)
    w_s = 2.0 ** torch.randint(-3, 4, (D,), generator=torch.Generator().manual_seed(dh)).float()
    for part in range(2):
        wq[part * H * dh:part * H * dh + dh] = 0
    prod = a_q.to(F64) * a_s.to(F64)[:, None] * (wq.to(F64).diagonal() * w_s.to(F64))[None]
    # acc * a_scale * w_scale + bias: three fp32 roundings, bounded by the terms (the bias may cancel the product)
    acc, acc_err = prod + bias.to(F64), 3 * U * (prod.abs() + bias.to(F64).abs())
    nw = (1 + 0.1 * torch.randn(2, dh, generator=torch.Generator().manual_seed(4))).to(BF16)
    table, cs = rope(ug, S, dh)
    qk = dict(weight=nw.cuda(), head_dim=dh, d=H * dh, cos_sin=table, eps=1e-6)
    out = ug.gemm_fp8(a_q[None].cuda(), a_s[None].cuda(), wq.cuda(), w_s.cuda(), bias=bias.cuda(), qk_norm=qk)
    check_qkv(out[0], acc, acc_err, nw, cs, H, dh, f"gemm_fp8 qk_norm dh={dh}")


@pytest.mark.parametrize("dh", [64, 128])
def test_qkv_scatter_one_rank_hard_heads(ug, dh):
    """qkv_scatter with one emulated rank: RMSNorm + RoPE of q / k heads into the receive buffer, v passed through."""
    from unigen_b200 import _lib
    S, H = 96, 4
    D = H * dh
    x, _, _ = qkv_projection_inputs(S, H, dh, seed=dh + 21)
    nw = (1 + 0.1 * torch.randn(2, dh, generator=torch.Generator().manual_seed(5))).to(BF16)
    table, cs = rope(ug, S, dh)
    off = 4096
    pool = torch.zeros(off + 3 * S * D * 2 + 4096, dtype=torch.uint8, device="cuda")
    t = _lib.PeerTable()
    t.world, t.rank = 1, 0
    t.base[0] = pool.data_ptr()
    rows = torch.zeros(S, 3 * D + 16, dtype=BF16, device="cuda")[:, 8:8 + 3 * D]
    rows.copy_(x.cuda())
    ug.qkv_scatter(t, rows, H, dh, nw.cuda(), table, off, S, 0)
    torch.cuda.synchronize()
    recv = pool[off:off + 3 * S * D * 2].view(BF16).view(3, S, D)
    assert (pool[off + 3 * S * D * 2:] == 0).all() and (pool[:off] == 0).all()
    check_qkv(recv.permute(1, 0, 2).reshape(S, 3 * D), x.to(F64), torch.zeros(S, 3 * D, dtype=F64), nw, cs, H, dh, f"qkv_scatter dh={dh}")
    assert torch.equal(recv[2].cpu(), x[:, 2 * D:])


# ---------------------------------------------------------------------------------------------------------------------------
# d. Row softmax in place
# ---------------------------------------------------------------------------------------------------------------------------
SOFTMAX_KINDS = ("normal", "equal", "offset3e4", "peaked", "neginf")


def softmax_rows(kind, n, cols, g):
    z = torch.randn(n, cols, generator=g, dtype=F64)
    if kind == "normal":
        return 3 * z
    if kind == "equal":
        return torch.full((n, cols), 1.5, dtype=F64)
    if kind == "offset3e4":  # bf16 spacing at 3e4 is 128: the noise is still resolved
        return 3e4 + 300 * z
    if kind == "peaked":
        z[torch.arange(n), torch.randint(0, cols, (n,), generator=g)] = z.max() + 80
        return z
    assert kind == "neginf"
    z = 3 * z
    z[torch.rand(n, cols, generator=g) < 0.3] = -math.inf
    z[:, 0] = 1.0  # never the whole row
    return z


@pytest.mark.parametrize("cols", [8, 1024, 16384, 16392, 65536])
def test_softmax_rows_hard_rows(ug, cols):
    g = torch.Generator().manual_seed(cols)
    per = 2
    x = torch.cat([softmax_rows(k, per, cols, g) for k in SOFTMAX_KINDS]).to(BF16)
    n = x.shape[0]
    buf = torch.full((n, cols + 64), 7.0, dtype=BF16, device="cuda")
    s = buf[:, :cols]  # row stride > cols, as in the chunked score buffer
    s.copy_(x.cuda())
    ug.softmax_rows_(s)
    torch.cuda.synchronize()
    assert (buf[:, cols:] == 7.0).all()
    xf = x.to(F64)
    m = xf.amax(-1, keepdim=True)
    e = torch.exp(xf - m)
    ref = e / e.sum(-1, keepdim=True)
    # exp2f((x - m) * log2 e): |x - m| U from the product, 2 ulp of exp2f; the fp32 row sum; the reciprocal and the product;
    # 2^-126: results below the fp32 normal range
    dm = (xf - m).abs().nan_to_num(posinf=0.0)
    err = U * (2 * dm + 8 + math.sqrt(cols)) * ref + 2.0 ** -126
    got = s.cpu()
    for i, kind in enumerate(SOFTMAX_KINDS):
        sl = slice(i * per, (i + 1) * per)
        assert_bf16_matches(got[sl], ref[sl], err[sl], f"softmax_rows cols={cols} [{kind} rows]")
    eq = got[per:2 * per]
    assert (eq.to(F64) - torch.tensor(1.0 / cols, dtype=F64).to(BF16).to(F64)).abs().max() <= bf16_ulp(torch.tensor(1.0 / cols, dtype=F64))
    pk = got[3 * per:4 * per].to(F64)
    assert (pk.max(-1).values == 1.0).all() and (pk.sort(-1).values[:, -2] < 1e-30).all()  # one-hot
    assert (got[4 * per:5 * per][x[4 * per:5 * per] == -math.inf] == 0).all()
