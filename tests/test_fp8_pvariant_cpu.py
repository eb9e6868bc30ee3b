"""CPU checks of the pre-division identity behind the fp8 P-variant linears (`UniCombineFlux.quantize_fp8()`): the fp8 GEMM
dequantises its whole accumulator as acc[r, c] * a_s[r] * w_s[c], so the switched LoRA update rides in the same accumulator as
  A2 = q @ Aq^T * aw_s   (= (x / a_s) @ A^T, masked to the row's adapter group)      W2 = (B * scaling) / w_s[c]
and  a_s w_s (q Wq^T + A2 W2^T)  equals  dequant(x) dequant(W)^T + (dequant(x) dequant(A)^T) B^T  exactly in real arithmetic.
Checked in fp32 with the reference quantiser on the operands `_LoraPair` stacks, with zero rows and segments without adapter."""
import math
import sys
from pathlib import Path

import pytest
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent))
from test_fp8_cpu import dequant_ref, quant_rows_ref  # noqa: E402

BLK = 64


def _case(seed, n_sub=3, rank=4, D=256, groups=4, bounds=(0, 40, 300, 420, 555), seg_group=(-1, 0, 1, 3)):
    from unigen_b200.pvariant import LORA_BLOCK, _LoraPair
    assert LORA_BLOCK == BLK
    g = torch.Generator().manual_seed(seed)
    S = bounds[-1]
    x = (torch.randn(S, D, generator=g) * torch.logspace(-2, 1, S).unsqueeze(1)).to(torch.bfloat16)
    x[7] = 0
    x[301] = 0
    W = (torch.randn(n_sub * D, D, generator=g) / math.sqrt(D)).to(torch.bfloat16)
    pair = _LoraPair("cpu", groups, rank, D, D, n_sub)
    for gi in range(groups):
        if gi == 2:
            continue  # a group with no adapter loaded: its A and B blocks stay zero
        pair.a[gi] = (torch.randn(n_sub * rank, D, generator=g) / math.sqrt(D)).to(torch.bfloat16)
        pair.b[gi] = (torch.randn(n_sub * D, rank, generator=g) * 0.7).to(torch.bfloat16)  # pre-scaled B
    pair.build_wide()
    return x, W, pair, list(bounds), list(seg_group)


def _group_of_rows(bounds, seg_group):
    return torch.cat([torch.full((bounds[i + 1] - bounds[i],), seg_group[i]) for i in range(len(seg_group))])


def _direct(x, W, pair, bounds, seg_group):
    """The quantised linear with its LoRA update the way the fake-quant oracle computes it: dequant(x) dequant(W)^T plus, per row,
    (dequant(x) dequant(A_g)^T) B_g^T with A quantised per row."""
    xd, Wd = dequant_ref(*quant_rows_ref(x)), dequant_ref(*quant_rows_ref(W))
    out = xd @ Wd.t()
    awd = dequant_ref(*quant_rows_ref(pair.aw))
    grp = _group_of_rows(bounds, seg_group)
    for gi in range(pair.a.shape[0]):
        m = grp == gi
        if m.any():
            blk = slice(gi * BLK, (gi + 1) * BLK)
            out[m] += (xd[m] @ awd[blk].t()) @ pair.bw[:, blk].float().t()
    return out


def _predivided(x, W, pair, bounds, seg_group, round_bf16=False):
    """What the fp8 kernels compute: masked down-projection with unit row scales, K extension pre-divided by w_s."""
    q, a_s = quant_rows_ref(x)
    qw, w_s = quant_rows_ref(W)
    aq, aw_s = quant_rows_ref(pair.aw)
    a2 = (q.float() @ aq.float().t()) * aw_s  # [S, groups * 64]
    grp = _group_of_rows(bounds, seg_group)
    keep = torch.zeros_like(a2, dtype=torch.bool)
    for gi in range(pair.a.shape[0]):
        keep[grp == gi, gi * BLK:(gi + 1) * BLK] = True
    a2 = torch.where(keep, a2, torch.zeros_like(a2))
    w2 = pair.bw.float() / w_s[:, None]
    if round_bf16:  # the operands the kernel reads are bf16
        a2, w2 = a2.to(torch.bfloat16).float(), w2.to(torch.bfloat16).float()
    acc = q.float() @ qw.float().t() + a2 @ w2.t()
    return acc * a_s[:, None] * w_s[None, :]


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_predivided_k_extension_equals_the_direct_lora_update(seed):
    x, W, pair, bounds, seg_group = _case(seed)
    want = _direct(x, W, pair, bounds, seg_group)
    got = _predivided(x, W, pair, bounds, seg_group)
    scale = want.abs().amax(1, keepdim=True).clamp_min(1e-30)
    assert ((got - want).abs() / scale).max().item() < 1e-5  # fp32 reassociation only
    # zero rows stay exactly zero; rows without an adapter equal the plain quantised linear exactly
    assert (got[7] == 0).all() and (got[301] == 0).all()
    q, a_s = quant_rows_ref(x)
    qw, w_s = quant_rows_ref(W)
    plain = (q.float() @ qw.float().t()) * a_s[:, None] * w_s[None, :]
    assert torch.equal(got[:40], plain[:40])
    # the update is visible on the adapted rows, and absent on the segment whose group has no adapter loaded
    assert not torch.allclose(got[40:300], plain[40:300])
    assert not torch.equal(got[420:], plain[420:])  # group 3 has an adapter
    grp2 = [0, 40, 300, 420, 555], [-1, 0, 2, 2]
    got2 = _predivided(x, W, pair, *grp2)
    assert torch.equal(got2[300:], plain[300:])


def test_bf16_operands_of_the_k_extension_stay_within_bf16_rounding():
    """The kernel reads A2 and W2 as bf16: the rounding costs about 2^-9 of the update, far below the fp8 error."""
    x, W, pair, bounds, seg_group = _case(5)
    want = _direct(x, W, pair, bounds, seg_group)
    got = _predivided(x, W, pair, bounds, seg_group, round_bf16=True)
    upd = want - _predivided(x, W, pair, [0, 555], [-1])
    assert ((got - want).norm() / upd.norm()).item() < 8e-3
