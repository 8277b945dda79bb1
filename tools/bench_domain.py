"""Step time of the config-2 workload at 128 x 128 and at 256 x 256 in one run: the sda_unet.yml ScoreUNet (random
init), L = 168 frames of 4 variables, k = 6 (156 windows per launch), CoarseGrain(6, 16), closed-form guidance, the
step of bench.py (window score, guidance + predictor; no corrections).  Reports ms per step, frames/s and the conv
TFLOP/s counted from shapes (115.134 GFLOP per window at 128 x 128, x (H W / 128^2) elsewhere), then, at 256 x 256,
the attention kernels' share of the step's kernel time (torch.profiler, a separate pass), one exact-grad step time and
the attention kernels' (and their backward's) share of that step.  Prints the GPU's name and power limit and one
JSON line."""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import sys
import warnings
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

GFLOP_PER_WINDOW_128 = 115.134  # conv FLOPs of one window's UNet forward at 128 x 128, counted from the layer shapes


def attention_shares(st) -> dict:
    """Shares of the kernel time of two profiled steps (torch.profiler, CUDA activities): every attention kernel, and
    the backward ones (attention_flash_bwd_*, attention_bwd_*) alone."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            st.timed(2, 0, torch.cuda.synchronize)
        events = prof.key_averages()
    tot = att = bwd = 0.0
    for e in events:
        t = e.device_time_total
        tot += t
        if "attention" in e.key:
            att += t
            if "bwd" in e.key:
                bwd += t
    return {"attention": round(att / max(tot, 1e-9), 5), "attention backward": round(bwd / max(tot, 1e-9), 5)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--sizes", type=int, nargs="+", default=[128, 256])
    args = ap.parse_args()

    import torch

    import bench
    import climate2weather_b200 as c2w
    from bench_ensemble import gpu_info

    if not torch.cuda.is_available():
        raise SystemExit("bench_domain.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda:0")
    C, k, nw = bench.C, bench.K_ORDER, bench.WINDOWS_PER_GPU
    L = nw + 2 * k
    torch.manual_seed(0)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, **bench.ARCH).requires_grad_(False).to(dev)
    cg = c2w.CoarseGrain(6, 16)

    def stepper(S, exact):
        truth = torch.randn(L, C, S, S, generator=torch.Generator().manual_seed(1))
        noise = torch.randn(L, C, S, S, generator=torch.Generator().manual_seed(2)).to(dev)
        with contextlib.redirect_stdout(io.StringIO()):
            return bench.Stepper(net, noise, cg(truth), cg, dev, nw, exact, shard=False)

    gpu = gpu_info()
    print(f"{gpu['name']}, power limit {gpu['power_limit']}, SM clock max {gpu['sm_max_clock']}")
    res = {}
    for S in args.sizes:
        st = stepper(S, False)
        ms = min(st.timed(args.steps, args.warmup, torch.cuda.synchronize) / args.steps for _ in range(args.rounds))
        gflop = GFLOP_PER_WINDOW_128 * (S * S) / (128 * 128) * nw
        res[S] = {"ms_per_step": round(ms, 3), "frames_per_s": round(L / ms * 1e3, 1),
                  "conv_tflops": round(gflop / ms, 1)}
        if S == max(args.sizes):  # attention share of the step's kernel time, in a profiled pass of its own
            res[S]["attention_share_of_kernel_time"] = attention_shares(st)["attention"]
            del st
            torch.cuda.empty_cache()
            ex = stepper(S, True)
            res[S]["exact_ms_per_step"] = round(
                min(ex.timed(max(2, args.steps // 4), 1, torch.cuda.synchronize) / max(2, args.steps // 4)
                    for _ in range(args.rounds)), 3)
            sh = attention_shares(ex)
            res[S]["exact_attention_share_of_kernel_time"] = sh["attention"]
            res[S]["exact_attention_backward_share_of_kernel_time"] = sh["attention backward"]
            del ex
        else:
            del st
        torch.cuda.empty_cache()
        print(f"{S}x{S}: {res[S]}", flush=True)
    print(json.dumps({"gpu": gpu, "workload": f"L={L} x {C}xSxS, k={k}, sda_unet.yml ScoreUNet (random init), {nw} "
                      "windows per launch, CoarseGrain(6, 16), closed-form guidance + predictor, 0 corrections",
                      "steps": args.steps, "rounds": args.rounds, "results": res}))


if __name__ == "__main__":
    main()
