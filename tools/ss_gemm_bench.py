#!/usr/bin/env python3
"""Isolated timer of the conversion-free persistent prologue GEMM (gvd_gemm_f16ss) at the prologue's plain-mode shapes.

Every product runs through capi.op_linear_f16ss (operands packed to fp16x3 images, then the persistent GEMM); only the GEMM kernel's device
time is counted: torch.profiler with CUDA activities over --iters launches per shape after warm-up, kernels f16ss_persistent_kernel /
f16ss_pair_kernel.  Backend variants are selected with capi.set_backend and alternated inside one process (--rounds passes over all of them).
Q|K|V mode has no C-ABI op: bench.py's stages_ms_per_step["interact.qkv_proj"] times it inside the step.

Reported per shape and variant: ms per launch, algorithmic TFLOP/s (2 M N K), and the fraction of the 3-pass ceiling (every fp16x3 product
is 3 fp16 MMAs: the ceiling is 1/3 of the dense fp16 rate, 2250 TFLOP/s on NVIDIA's B200 data sheet for a 1000 W card).  The card name,
power limit and max SM clock are printed with the numbers.

    python tools/ss_gemm_bench.py [--variants 923,1947] [--iters 20] [--rounds 3] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

DENSE_FP16_TFLOPS = 2250.0            # NVIDIA B200 data sheet, dense, per GPU (1000 W)
KERNELS = ("f16ss_persistent_kernel", "f16ss_pair_kernel")


def shapes(opt, M):
    """(name, N, K, bias, act, want_c, want_img) of the prologue's plain-mode products, derived as gvd_model_create (gvd_api.cu) does."""
    rup4 = lambda x: (x + 3) // 4 * 4
    H, A, D, F = opt.rnn_size, opt.att_hid_size, opt.detect_size, opt.att_feat_size
    NC = D + 1
    PINp = rup4(F + 300 + D + 1)
    HP = rup4((H + 5) // 6) * len(range(0, H, (H + 5) // 6))
    return [("fc7", 2048, F, True, 1, True, True),               # region.fc7: C + image (the similarity GEMM streams it), bias + ReLU
            ("similarity", NC, 2048, True, 0, True, False),        # region.sim_gemm: 128-column tiles
            ("region_embedding", H, PINp, True, 1, True, True),   # region.pool_embed: C + image
            ("ffn1", H // 2, H, True, 1, False, True),            # interact.ffn1: image only
            ("ffn2", H, H // 2, True, 0, True, False),            # interact.ffn2: C
            ("wo", H, HP, False, 0, True, False),                 # interact.wo: C
            ("ctx2pool", A, H, True, 0, True, False)]             # region.ctx2pool: C


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        q = ""
    return q or "nvidia-smi unavailable"


def gemm_ms(fn, iters):
    """Mean device time per launch of the persistent GEMM kernel over `iters` calls of fn (torch.profiler, CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    tot, n = 0.0, 0
    for e in prof.events():
        if e.device_type.name == "CUDA" and any(k in e.name for k in KERNELS):
            tot += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
            n += 1
    assert n == iters, "expected %d GEMM launches, profiled %d" % (iters, n)
    return tot / n / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--M", type=int, default=100_000, help="rows (B=100 clips x R=1000 RoIs)")
    ap.add_argument("--variants", default="923,1947", help="comma list of backend flags, alternated")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--only", default="", help="comma list of shape names")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    from gvd_b200 import capi, synth
    assert torch.cuda.is_available(), "ss_gemm_bench needs a CUDA device"
    opt = synth.make_opt(t_attn_size=10)
    M = args.M
    variants = [int(v) for v in args.variants.split(",")]
    info = {"card": card(), "M": M, "iters": args.iters, "rounds": args.rounds,
            "ceiling_3pass_tflops": DENSE_FP16_TFLOPS / 3, "timing": "torch.profiler device time of the GEMM kernel, mean per launch"}
    print(json.dumps(info), flush=True)
    g = torch.Generator(device="cuda").manual_seed(7)
    rows = []
    old = capi.get_backend()
    for name, N, K, has_bias, act, want_c, want_img in shapes(opt, M):
        if args.only and name not in args.only.split(","):
            continue
        A = torch.randn(M, K, device="cuda", generator=g)
        W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
        b = torch.randn(N, device="cuda", generator=g) if has_bias else None
        fn = lambda: capi.op_linear_f16ss(A, W, b, act, want_img=want_img, want_c=want_c)
        ms = {v: [] for v in variants}
        for v in variants:
            capi.set_backend(v)
            for _ in range(args.warmup):
                fn()
        for _ in range(args.rounds):
            for v in variants:
                capi.set_backend(v)
                ms[v].append(gemm_ms(fn, args.iters))
        flop = 2.0 * M * N * K
        for v in variants:
            best, med = min(ms[v]), sorted(ms[v])[len(ms[v]) // 2]
            tf = flop / (med * 1e-3) / 1e12
            r = {"shape": name, "M": M, "N": N, "K": K, "out": "+".join(x for x, w in (("C", want_c), ("img", want_img)) if w),
                 "backend": v, "ms_median": round(med, 4), "ms_min": round(best, 4), "ms_all": [round(x, 4) for x in ms[v]],
                 "tflops": round(tf, 1), "frac_3pass": round(tf / info["ceiling_3pass_tflops"], 3)}
            rows.append(r)
            print(json.dumps(r), flush=True)
        del A, W, b
        torch.cuda.empty_cache()
    capi.set_backend(old)
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"info": info, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
