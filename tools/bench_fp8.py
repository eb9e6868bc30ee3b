"""fp8 (e4m3, row-wise scaled) block linears on one B200 at the cfg3 shapes, everything measured in ONE process and alternated:
  - isolated GEMMs at the cfg3 block-linear shapes: bf16 native (ug_gemm_bf16), fp8 native (ug_gemm_fp8) and torch._scaled_mm
    row-wise, CUDA events over back-to-back launches, TFLOP/s against the data-sheet dense 2 250 (bf16) / 4 500 (fp8);
  - the quantisation kernels (quant_rows_fp8, ln_modulate_fp8, with ln_modulate for reference) in GB/s of algorithmic bytes;
  - the cfg3 step (CUDA-graph replay) of a bf16 model and of the same weights after quantize_fp8(), alternating, plus the cosine
    of the two final velocities on the same inputs.
The card name, power limit and max SM clock are read in the same call.
python tools/bench_fp8.py [--rounds 3] [--steps 5] [--out FILE]   -> one JSON document"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

# (name, M, K, N) of the cfg3 block linears (1024^2 image: N = 4096 image tokens, T = 512 text tokens, D = 3072)
GEMMS = [("double.img.qkv", 4096, 3072, 9216), ("double.img.to_out", 4096, 3072, 3072), ("double.img.ff1", 4096, 3072, 12288),
         ("double.img.ff2", 4096, 12288, 3072), ("double.txt.qkv", 512, 3072, 9216), ("double.txt.ff2", 512, 12288, 3072),
         ("single.qkv", 4608, 3072, 9216), ("single.mlp", 4608, 3072, 12288), ("single.out", 4608, 15360, 3072)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def timed(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def bench_gemms(ops, rounds, iters):
    res = []
    for name, M, K, N in GEMMS:
        a, w = torch.randn(1, M, K, device="cuda").to(torch.bfloat16), (torch.randn(N, K, device="cuda") * K ** -0.5).to(torch.bfloat16)
        bias = torch.randn(N, device="cuda").to(torch.bfloat16)
        qa, sa = ops.quant_rows_fp8(a)
        qw, sw = ops.quant_rows_fp8(w)
        out = torch.empty(1, M, N, device="cuda", dtype=torch.bfloat16)
        legs = {"bf16_native": lambda: ops.gemm(a, w, out=out, bias=bias),
                "fp8_native": lambda: ops.gemm_fp8(qa, sa, qw, sw, out=out, bias=bias)}
        try:
            torch._scaled_mm(qa[0], qw.t(), scale_a=sa[0].view(M, 1), scale_b=sw.view(1, N), bias=bias, out_dtype=torch.bfloat16)
            legs["torch_scaled_mm_rowwise"] = lambda: torch._scaled_mm(qa[0], qw.t(), scale_a=sa[0].view(M, 1), scale_b=sw.view(1, N),
                                                                       bias=bias, out_dtype=torch.bfloat16)
        except (RuntimeError, NotImplementedError) as e:
            scaled_mm_error = f"{type(e).__name__}: {e}"[:200]
        else:
            scaled_mm_error = None
        for fn in legs.values():
            timed(fn, 3)  # warm-up: module load, algorithm choice
        ms = {k: [] for k in legs}
        for _ in range(rounds):
            for k, fn in legs.items():
                ms[k].append(timed(fn, iters))
        flop = 2.0 * M * K * N
        rec = {"name": name, "M": M, "K": K, "N": N}
        for k, v in ms.items():
            best = min(v)
            peak = 2250.0 if k == "bf16_native" else 4500.0
            rec[k] = {"ms": round(best, 4), "ms_all": [round(x, 4) for x in v], "tflops": round(flop / best / 1e9, 1),
                      "share_of_datasheet_dense": round(flop / best / 1e9 / peak, 3)}
        if scaled_mm_error:
            rec["torch_scaled_mm_rowwise"] = {"error": scaled_mm_error}
        rec["fp8_speedup_vs_bf16"] = round(rec["bf16_native"]["ms"] / rec["fp8_native"]["ms"], 3)
        res.append(rec)
        del a, w, qa, qw, out
    return res


def bench_quant(ops, rounds, iters):
    res = []
    for rows, k in ((4096, 3072), (4096, 12288), (4608, 15360)):
        x = torch.randn(1, rows, k, device="cuda").to(torch.bfloat16)
        q = torch.empty(1, rows, k, device="cuda", dtype=torch.float8_e4m3fn)
        s = torch.empty(1, rows, device="cuda")
        fn = lambda: ops.quant_rows_fp8(x, q, s)  # noqa: E731
        timed(fn, 3)
        best = min(timed(fn, iters) for _ in range(rounds))
        nbytes = rows * k * 3 + rows * 4
        res.append({"kernel": "quant_rows_fp8", "rows": rows, "k": k, "ms": round(best, 4), "GBps": round(nbytes / best / 1e6, 1)})
    rows, d = 4608, 3072
    x = torch.randn(1, rows, d, device="cuda").to(torch.bfloat16)
    shift, scale = torch.randn(1, d, device="cuda"), torch.randn(1, d, device="cuda")
    nx = torch.empty_like(x)
    q = torch.empty(1, rows, d, device="cuda", dtype=torch.float8_e4m3fn)
    s = torch.empty(1, rows, device="cuda")
    for name, fn, nbytes in (("ln_modulate (bf16 out)", lambda: ops.ln_modulate(x, nx, shift, scale), rows * d * 4),
                             ("ln_modulate_fp8", lambda: ops.ln_modulate_fp8(x, q, s, shift, scale), rows * d * 3 + rows * 4)):
        timed(fn, 3)
        best = min(timed(fn, iters) for _ in range(rounds))
        res.append({"kernel": name, "rows": rows, "k": d, "ms": round(best, 4), "GBps": round(nbytes / best / 1e6, 1)})
    return res


def cfg3_models_and_inputs():
    from unigen_b200.model import FluxArch, UniGenFlux, canonical_control_params
    arch = FluxArch()
    models = []
    for _ in range(2):
        m = UniGenFlux(arch, device="cuda")
        m.init_condition_block(condition_nums=1, control_params=canonical_control_params())
        m.init_random_(seed=0)
        m.use_cuda_graph = True
        models.append(m)
    models[1].quantize_fp8()
    N, T, E = 4096, 512, models[0].expert_nums
    g = torch.Generator().manual_seed(1234)
    ids = torch.zeros(64, 64, 3)
    ids[..., 1] += torch.arange(64)[:, None]
    ids[..., 2] += torch.arange(64)[None, :]
    ids = ids.reshape(N, 3)
    inp = dict(hidden_states=torch.randn(1, N, 64, generator=g).to(torch.bfloat16),
               condition_hidden_states=torch.randn(1, N, 64, generator=g).to(torch.bfloat16),
               encoder_hidden_states=torch.randn(1, T, 4096, generator=g).to(torch.bfloat16),
               pooled_projections=torch.randn(1, 768, generator=g), condition_pooled_projections=torch.randn(1, 768, generator=g),
               timestep=torch.full((1,), 0.75), img_ids=ids.clone(), txt_ids=torch.zeros(T, 3), condition_ids=ids.clone(),
               rts_uniform=torch.rand(N, E, generator=g))
    return models, {k: v.cuda() for k, v in inp.items()}


def bench_step(rounds, steps):
    models, inp = cfg3_models_and_inputs()
    outs = [m(**inp)[0] for m in models]  # warm-up: workspaces + graph capture
    for m in models:
        m(**inp)
    ms = {"bf16": [], "fp8": []}
    for _ in range(rounds):
        for name, m in zip(ms, models):
            ms[name].append(timed(lambda: m(**inp), steps))
    cos = torch.nn.functional.cosine_similarity(outs[0].float().flatten(), outs[1].float().flatten(), dim=0).item()
    rel = ((outs[1].float() - outs[0].float()).norm() / outs[0].float().norm()).item()
    rec = {k: {"ms_per_step": round(min(v), 2), "ms_all": [round(x, 2) for x in v]} for k, v in ms.items()}
    rec["fp8_speedup_vs_bf16"] = round(rec["bf16"]["ms_per_step"] / rec["fp8"]["ms_per_step"], 3)
    rec["velocity_fp8_vs_bf16"] = {"cosine": round(cos, 6), "rel_l2": round(rel, 5)}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--no-step", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from unigen_b200 import ops
    torch.backends.cuda.matmul.allow_tf32 = False
    ops.device_check()
    rec = {"what": "fp8 (e4m3 row-wise) vs bf16 block linears, cfg3 shapes, one process, alternating legs; isolated GEMMs with "
                   "warm L2 (same operands every launch), best of rounds",
           "card": card(), "gemm": bench_gemms(ops, args.rounds, args.iters), "quant": bench_quant(ops, args.rounds, args.iters)}
    if not args.no_step:
        rec["cfg3_step"] = bench_step(args.rounds, args.steps)
    rec["card_after"] = card()
    text = json.dumps(rec, indent=1)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
