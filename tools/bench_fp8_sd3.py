"""fp8 (e4m3, row-wise scaled) joint-block linears of the SD3.5 denoiser on one B200 at the cfg5 shapes, everything measured in
ONE process and alternated:
  - isolated GEMMs at the cfg5 block-linear shapes (forward batch 4, [4, rows] activation scales): bf16 native (ug_gemm_bf16),
    fp8 native (ug_gemm_fp8) and torch._scaled_mm row-wise, CUDA events over back-to-back launches, TFLOP/s against the
    data-sheet dense 2 250 (bf16) / 4 500 (fp8); and the fp8 GEMM in every tile variant at the two K = 1536 image shapes;
  - the quantisation kernels at d = 1536 and 6144 (quant_rows_fp8, ln_modulate_fp8, with ln_modulate for reference) in GB/s of
    algorithmic bytes;
  - the cfg5 step (SD3.5-medium UniGenSD3, 1024^2 + 1 condition, 333 text tokens, forward batch 4, CUDA-graph replay) of a bf16
    model and of the same seeded weights after quantize_fp8(), alternating, plus the cosine / rel-L2 of the two final velocities
    on the same inputs, and a per-kernel breakdown of one eager step of each (torch.profiler, run after the timed legs).
The card name, power limit and max SM clock are read in the same call.
python tools/bench_fp8_sd3.py [--rounds 3] [--steps 5] [--no-step] [--no-profile] [--out FILE]   -> one JSON document"""
import argparse
import json
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))
from bench_fp8 import card, timed  # noqa: E402

B, N_IMG, N_TXT, D = 4, 4096, 333, 1536
# (name, batch, rows, K, N) of the cfg5 joint-block linears (D = 1536: K = D, or 4D for ff.net.2)
GEMMS = [("img.qkv", B, N_IMG, D, 3 * D), ("txt.qkv", B, N_TXT, D, 3 * D), ("img.to_out", B, N_IMG, D, D),
         ("img.ff1", B, N_IMG, D, 4 * D), ("img.ff2", B, N_IMG, 4 * D, D), ("img.attn2_qkv", B, N_IMG, D, 3 * D)]


def bench_gemms(ops, rounds, iters):
    res = []
    for name, b, m, K, N in GEMMS:
        a, w = torch.randn(b, m, K, device="cuda").to(torch.bfloat16), (torch.randn(N, K, device="cuda") * K ** -0.5).to(torch.bfloat16)
        bias = torch.randn(N, device="cuda").to(torch.bfloat16)
        qa, sa = ops.quant_rows_fp8(a)  # [b, m, K] e4m3 + [b, m] row scales, as the model hands them over
        qw, sw = ops.quant_rows_fp8(w)
        out = torch.empty(b, m, N, device="cuda", dtype=torch.bfloat16)
        M = b * m
        qa2, sa2 = qa.view(M, K), sa.view(M, 1)
        legs = {"bf16_native": lambda: ops.gemm(a, w, out=out, bias=bias),
                "fp8_native": lambda: ops.gemm_fp8(qa, sa, qw, sw, out=out, bias=bias)}
        try:
            torch._scaled_mm(qa2, qw.t(), scale_a=sa2, scale_b=sw.view(1, N), bias=bias, out_dtype=torch.bfloat16)
            legs["torch_scaled_mm_rowwise"] = lambda: torch._scaled_mm(qa2, qw.t(), scale_a=sa2, scale_b=sw.view(1, N), bias=bias,
                                                                       out_dtype=torch.bfloat16)
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
        rec = {"name": name, "M": f"{b}x{m}", "K": K, "N": N}
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


def bench_fp8_tiles(ops, rounds, iters):
    """The fp8 GEMM in every tile variant (1-3: direct epilogue, 4-6: staged TMA-store epilogue; 0 = the auto pick) at the two
    K = 1536 image-stream shapes, where the fp8 main loop is short next to the epilogue."""
    res = []
    for name, b, m, K, N in (GEMMS[0], GEMMS[2]):
        a, w = torch.randn(b, m, K, device="cuda").to(torch.bfloat16), (torch.randn(N, K, device="cuda") * K ** -0.5).to(torch.bfloat16)
        bias = torch.randn(N, device="cuda").to(torch.bfloat16)
        qa, sa = ops.quant_rows_fp8(a)
        qw, sw = ops.quant_rows_fp8(w)
        out = torch.empty(b, m, N, device="cuda", dtype=torch.bfloat16)
        legs = {f"fp8_variant_{v}": (lambda v=v: ops.gemm_fp8(qa, sa, qw, sw, out=out, bias=bias, variant=v)) for v in range(7)}
        legs["bf16_variant_0"] = lambda: ops.gemm(a, w, out=out, bias=bias)
        for fn in legs.values():
            timed(fn, 3)
        ms = {k: [] for k in legs}
        for _ in range(rounds):
            for k, fn in legs.items():
                ms[k].append(timed(fn, iters))
        flop = 2.0 * b * m * K * N
        res.append({"name": name, "M": f"{b}x{m}", "K": K, "N": N,
                    **{k: {"ms": round(min(v), 4), "tflops": round(flop / min(v) / 1e9, 1)} for k, v in ms.items()}})
        del a, w, qa, qw, out
    return res


def bench_quant(ops, rounds, iters):
    res = []
    for rows, k in ((N_IMG + N_TXT, D), (N_IMG, 4 * D)):
        x = torch.randn(B, rows, k, device="cuda").to(torch.bfloat16)
        q = torch.empty(B, rows, k, device="cuda", dtype=torch.float8_e4m3fn)
        s = torch.empty(B, rows, device="cuda")
        fn = lambda: ops.quant_rows_fp8(x, q, s)  # noqa: E731
        timed(fn, 3)
        best = min(timed(fn, iters) for _ in range(rounds))
        nbytes = B * rows * (k * 3 + 4)
        res.append({"kernel": "quant_rows_fp8", "rows": f"{B}x{rows}", "k": k, "ms": round(best, 4), "GBps": round(nbytes / best / 1e6, 1)})
    rows = N_IMG + N_TXT
    x = torch.randn(B, rows, D, device="cuda").to(torch.bfloat16)
    shift, scale = torch.randn(B, D, device="cuda"), torch.randn(B, D, device="cuda")
    nx = torch.empty_like(x)
    q = torch.empty(B, rows, D, device="cuda", dtype=torch.float8_e4m3fn)
    s = torch.empty(B, rows, device="cuda")
    for name, fn, nbytes in (("ln_modulate (bf16 out)", lambda: ops.ln_modulate(x, nx, shift, scale), B * rows * D * 4),
                             ("ln_modulate_fp8", lambda: ops.ln_modulate_fp8(x, q, s, shift, scale), B * rows * (D * 3 + 4))):
        timed(fn, 3)
        best = min(timed(fn, iters) for _ in range(rounds))
        res.append({"kernel": name, "rows": f"{B}x{rows}", "k": D, "ms": round(best, 4), "GBps": round(nbytes / best / 1e6, 1)})
    return res


def cfg5_models_and_inputs():
    from unigen_b200.sd3 import SD3Arch, UniGenSD3, shipped_control_params
    models = []
    for _ in range(2):
        m = UniGenSD3(SD3Arch(), device="cuda")
        m.init_condition_block(condition_nums=1, control_params=shipped_control_params())
        m.init_random_(seed=0)
        m.use_cuda_graph = True
        models.append(m)
    models[1].quantize_fp8()
    lat = 1024 // 8
    g = torch.Generator().manual_seed(1234)
    inp = dict(hidden_states=torch.randn(B, 16, lat, lat, generator=g).bfloat16(),
               condition_hidden_states=torch.randn(B, 16, lat, lat, generator=g).bfloat16(),
               encoder_hidden_states=torch.randn(B, N_TXT, 4096, generator=g).bfloat16(),
               pooled_projections=torch.randn(B, 2048, generator=g), condition_pooled_projections=torch.randn(B, 2048, generator=g),
               timestep=torch.full((B,), 500.0), rts_uniform=torch.rand(B * N_IMG, models[0].expert_nums, generator=g))
    return models, {k: v.cuda() for k, v in inp.items()}


def kernel_breakdown(model, inp):
    """Device time per kernel of one eager forward (torch.profiler, CUDA activities), grouped by kernel name."""
    from torch.profiler import ProfilerActivity, profile
    model.use_cuda_graph = False
    model(**inp)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        model(**inp)
        torch.cuda.synchronize()
    rows = []
    for e in prof.key_averages():
        t = getattr(e, "self_device_time_total", 0) or getattr(e, "self_cuda_time_total", 0)
        if t > 0:
            rows.append((e.key, e.count, t / 1e3))
    rows.sort(key=lambda r: -r[2])
    total = sum(r[2] for r in rows)

    def group(name):
        n = name.lower()
        for key in ("attention", "gemv", "ln_modulate", "quant_rows", "gemm", "qk_rmsnorm"):
            if key in n:
                return key
        return "other"

    groups = {}
    for name, n, ms in rows:
        g = groups.setdefault(group(name), {"ms": 0.0, "launches": 0})
        g["ms"] += ms
        g["launches"] += n
    model.use_cuda_graph = True
    return {"kernel_ms_total": round(total, 2),
            "groups": {k: {"ms": round(v["ms"], 2), "launches": v["launches"], "share": round(v["ms"] / total, 3)}
                       for k, v in sorted(groups.items(), key=lambda kv: -kv[1]["ms"])},
            "top_kernels": [{"kernel": name[:120], "launches": n, "ms": round(ms, 3)} for name, n, ms in rows[:14]],
            "note": "one eager forward, kernels serialised by the profiler; compare shares, not totals, with the graph-replay step"}


def bench_step(rounds, steps, profile_step):
    models, inp = cfg5_models_and_inputs()
    outs = [m(**inp)[0] for m in models]  # warm-up: workspaces + graph capture
    for m in models:
        m(**inp)
    ms = {"bf16": [], "fp8": []}
    for _ in range(rounds):
        for name, m in zip(ms, models):
            ms[name].append(timed(lambda: m(**inp), steps))
    v16, v8 = outs[0].float(), outs[1].float()
    cos = torch.nn.functional.cosine_similarity(v8.flatten(), v16.flatten(), dim=0).item()
    rel = ((v8 - v16).norm() / v16.norm()).item()
    rec = {k: {"ms_per_step": round(min(v), 2), "ms_all": [round(x, 2) for x in v]} for k, v in ms.items()}
    rec["fp8_speedup_vs_bf16"] = round(rec["bf16"]["ms_per_step"] / rec["fp8"]["ms_per_step"], 3)
    rec["velocity_fp8_vs_bf16"] = {"cosine": round(cos, 6), "rel_l2": round(rel, 5), "note": "same seeded weights and inputs, no bar"}
    rec["finite"] = bool(torch.isfinite(v8).all() and torch.isfinite(v16).all())
    if profile_step:
        rec["kernel_breakdown"] = {name: kernel_breakdown(m, inp) for name, m in zip(("bf16", "fp8"), models)}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--no-step", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from unigen_b200 import ops
    torch.backends.cuda.matmul.allow_tf32 = False
    ops.device_check()
    rec = {"what": "fp8 (e4m3 row-wise) vs bf16 joint-block linears of UniGenSD3, cfg5 shapes (SD3.5-medium, 1024^2 + 1 condition, "
                   "333 text tokens, forward batch 4), one process, alternating legs; isolated GEMMs with warm L2 (same operands "
                   "every launch), best of rounds",
           "card": card(), "gemm": bench_gemms(ops, args.rounds, args.iters), "fp8_tiles": bench_fp8_tiles(ops, args.rounds, args.iters),
           "quant": bench_quant(ops, args.rounds, args.iters)}
    if not args.no_step:
        rec["cfg5_step"] = bench_step(args.rounds, args.steps, not args.no_profile)
    rec["card_after"] = card()
    text = json.dumps(rec, indent=1)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
