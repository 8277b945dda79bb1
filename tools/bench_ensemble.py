"""Ensemble sampling in one device-resident run (SDAPipeline.sample_ensemble) against the members run one after the
other (M sequential SDAPipeline.sample calls, what the reference driver does), at the production ensemble shapes: the
sda_unet.yml ScoreUNet (random init), frames of 4 x 128 x 128, k = 6, CoarseGrain(6, 16), closed-form guidance, no
corrections, L in {13, 49, 121} frames x M in {1, 2, 4, 8} members.

Both arms sample the same M members from the same noise on the GPU (no host copies) and alternate, --rounds times:
the time of a whole call, host clock around work that ends in a device synchronise, over --steps denoising steps.
Each arm has its own score function, so its runtime, engine and workspace are built in one warm-up call per shape and
reused by the timed calls (steady state); a timed call still includes its noise load and its output copy.  Reported
per shape and arm: ms per step (the whole ensemble's) and frames/s (M L steps / time), best and all rounds; and whether
every member of the ensemble equals its sequential run bit for bit.  Prints the GPU's name and power limit and one JSON line."""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


def gpu_info() -> dict:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = (v.strip() for v in r.stdout.splitlines()[0].split(","))
    return {"name": name, "power_limit": power, "sm_max_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--lengths", type=int, nargs="+", default=[13, 49, 121])
    ap.add_argument("--members", type=int, nargs="+", default=[1, 2, 4, 8])
    args = ap.parse_args()

    import torch

    import bench
    import climate2weather_b200 as c2w

    if not torch.cuda.is_available():
        raise SystemExit("bench_ensemble.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda:0")
    C, H, W = bench.C, bench.H, bench.W
    torch.manual_seed(0)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, **bench.ARCH).requires_grad_(False).to(dev)
    pipe = c2w.SDAPipeline()
    cg = c2w.CoarseGrain(6, 16)

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):  # sample() prints its total time
            out = fn()
        torch.cuda.synchronize()
        return out, time.perf_counter() - t0

    results = []
    for L in args.lengths:
        truth = torch.randn(L, C, H, W, generator=torch.Generator().manual_seed(L))
        sfs = {}
        for arm in ("ensemble", "sequential"):
            sfs[arm] = c2w.DefaultScoreFunction(net, markov_order=bench.K_ORDER, noise_process=pipe)
            sfs[arm].condition_on(A=cg, y=cg(truth), std=bench.STD, gamma=bench.GAMMA, exact_grad=False)
        for M in args.members:
            noise = torch.randn(M, L, C, H, W, generator=torch.Generator().manual_seed(100 * L + M)).to(dev)
            arms = {
                "ensemble": lambda: pipe.sample_ensemble(sfs["ensemble"], noise, steps=args.steps,
                                                         show_progressbar=False),
                "sequential": lambda: torch.stack([pipe.sample(sfs["sequential"], noise[m], steps=args.steps,
                                                               show_progressbar=False) for m in range(M)]),
            }
            outs = {k: timed(fn)[0] for k, fn in arms.items()}  # warm-up: each arm's runtime, engine and workspace
            identical = all(torch.equal(outs["ensemble"][m], outs["sequential"][m]) for m in range(M))
            secs = {k: [] for k in arms}
            for _ in range(args.rounds):
                for k, fn in arms.items():
                    out, s = timed(fn)
                    secs[k].append(s)
                    identical &= all(torch.equal(out[m], outs[k][m]) for m in range(M))
            row = {"L": L, "M": M, "windows_per_member": L - 2 * bench.K_ORDER, "bit_identical": bool(identical)}
            for k, v in secs.items():
                row[k] = {"ms_per_step": [round(s / args.steps * 1e3, 3) for s in v],
                          "ms_per_step_best": round(min(v) / args.steps * 1e3, 3),
                          "frames_per_s_best": round(M * L * args.steps / min(v), 2)}
            row["speedup_best"] = round(min(secs["sequential"]) / min(secs["ensemble"]), 3)
            print(f"L={L:4d} M={M}: ensemble {row['ensemble']['ms_per_step_best']:9.3f} ms/step "
                  f"{row['ensemble']['frames_per_s_best']:8.2f} frames/s | sequential "
                  f"{row['sequential']['ms_per_step_best']:9.3f} ms/step {row['sequential']['frames_per_s_best']:8.2f} "
                  f"frames/s | x{row['speedup_best']:.3f} | bit-identical {identical}", flush=True)
            results.append(row)
            del noise, outs
    out = {"gpu": gpu_info(), "workload": f"{C}x{H}x{W} frames, sda_unet.yml ScoreUNet (random init), k={bench.K_ORDER}, "
           f"CoarseGrain(6, 16), closed-form guidance, 0 corrections, default windows per launch "
           f"(min(M (L - 2k), {c2w.DefaultScoreFunction.DEFAULT_WINDOWS})), whole sample calls in steady state",
           "steps": args.steps, "rounds": args.rounds, "results": results}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
