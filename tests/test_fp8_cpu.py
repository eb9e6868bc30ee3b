"""CPU checks of the fp8 (e4m3, row-wise scaled) block-linear path: the ctypes mirror of `ug_gemm_fp8_scales` matches the
header as gcc lays it out, and the torch reference quantiser the GPU tests compare against round-trips within half an e4m3
step of its row scale."""
import ctypes as C
import shutil
import subprocess
from pathlib import Path

import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
HEADER = ROOT / "include" / "unigen_b200.h"
E4M3_MAX = 448.0


def quant_rows_ref(x: torch.Tensor):
    """Row-wise e4m3 quantisation as the kernels define it: amax = max|x| per row (last dim); amax == 0 -> scale 1, q = 0;
    else inv = 448 / amax, scale = amax / 448 (fp32 IEEE divisions), q = e4m3(clamp(x * inv, +-448)) round-to-nearest-even.
    Returns (q float8_e4m3fn, scale fp32 [...rows])."""
    xf = x.float()
    amax = xf.abs().amax(dim=-1)
    nz = amax != 0
    inv = torch.where(nz, torch.tensor(E4M3_MAX) / torch.where(nz, amax, torch.ones_like(amax)), torch.zeros_like(amax))
    scale = torch.where(nz, amax / torch.tensor(E4M3_MAX), torch.ones_like(amax))
    q = (xf * inv.unsqueeze(-1)).clamp(-E4M3_MAX, E4M3_MAX).to(torch.float8_e4m3fn)
    q = torch.where(nz.unsqueeze(-1), q.view(torch.uint8), torch.zeros_like(q.view(torch.uint8))).view(torch.float8_e4m3fn)
    return q, scale


def dequant_ref(q: torch.Tensor, scale: torch.Tensor) -> torch.Tensor:
    return q.float() * scale.unsqueeze(-1)


def test_gemm_fp8_scales_offsets_match_a_compiled_probe(tmp_path):
    from unigen_b200 import _lib
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    cls = _lib.GemmFp8Scales
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(ug_gemm_fp8_scales));']
    lines += [f'  printf("{f} %zu\\n", offsetof(ug_gemm_fp8_scales, {f}));' for f, _ in cls._fields_]
    lines += ["  return 0;", "}"]
    src = tmp_path / "probe.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-std=c11", "-o", str(exe), str(src)], check=True)
    out = dict(ln.split() for ln in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(out["size"]) == C.sizeof(cls)
    for f, _ in cls._fields_:
        assert int(out[f]) == getattr(cls, f).offset, f


def test_reference_quantiser_round_trips_within_half_a_step():
    g = torch.Generator().manual_seed(0)
    x = (torch.randn(64, 512, generator=g) * torch.logspace(-3, 3, 64).unsqueeze(1)).to(torch.bfloat16)
    x[5, 17] = 1e4                              # single outlier row
    q, s = quant_rows_ref(x)
    assert q.dtype == torch.float8_e4m3fn and s.shape == (64,)
    xf = x.float()
    amax = xf.abs().amax(-1)
    assert torch.equal(s, amax / E4M3_MAX)
    assert (q.float().abs().amax(-1) == E4M3_MAX).all()   # the row maximum maps onto the top of the e4m3 range
    # e4m3 has 3 mantissa bits: in units of the row scale, the spacing around |y| is 2^(floor(log2|y|) - 3) (2^-9 below 2^-6)
    y = xf / s.unsqueeze(1)
    step = torch.exp2(torch.floor(torch.log2(y.abs().clamp_min(2.0 ** -6))) - 3)
    err = (dequant_ref(q, s) - xf).abs() / s.unsqueeze(1)
    assert (err <= 0.5 * step * (1 + 1e-5)).all()  # (ties land exactly on half a step; fp32 dequantisation adds ~1e-6)


def test_reference_quantiser_zero_rows():
    x = torch.zeros(3, 64, dtype=torch.bfloat16)
    x[1, 3] = -2.0
    x[2] = -0.0
    q, s = quant_rows_ref(x)
    assert s[0].item() == 1.0 and s[2].item() == 1.0 and s[1] == torch.tensor(2.0) / E4M3_MAX
    assert (q[0].view(torch.uint8) == 0).all() and (q[2].view(torch.uint8) == 0).all()   # +0 bytes, also for a -0 row
    assert q[1, 3].float().item() == -E4M3_MAX
