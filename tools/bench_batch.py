"""Batched sampling of independent problems in one device-resident run (SDAPipeline.sample_batch) against the same
problems run one after the other (M sequential SDAPipeline.sample calls) and against sample_ensemble on one shared
observation, at the production shapes: the sda_unet.yml ScoreUNet (random init), frames of 4 x 128 x 128, k = 6,
CoarseGrain(6, 16), closed-form guidance, no corrections, L in {13, 49, 121} frames x M in {1, 2, 4, 8} members.
Member m of the batch and of the sequential arm has its own truth and y; the ensemble arm conditions every member on
member 0's y, so the difference between the batch and the ensemble is what per-member observations cost.

The three arms sample the same noise on the GPU (no host copies) and alternate, --rounds times: the time of a whole
call, host clock around work that ends in a device synchronise, over --steps denoising steps.  Every arm's runtimes,
engine and workspace are built in one warm-up call per shape and reused by the timed calls (steady state); a timed call
still includes its noise load and its output copy.  Reported per shape and arm: ms per step (all members') and
frames/s (M L steps / time), best and all rounds; and whether every member of the batch equals its sequential run bit
for bit (in every round).  Prints the GPU's name and power limit and one JSON line."""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))


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
    from bench_ensemble import gpu_info

    if not torch.cuda.is_available():
        raise SystemExit("bench_batch.py measures on the GPU; no CUDA device found")
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

    def score_fn(y):
        sf = c2w.DefaultScoreFunction(net, markov_order=bench.K_ORDER, noise_process=pipe)
        with contextlib.redirect_stdout(io.StringIO()):
            sf.condition_on(A=cg, y=y, std=bench.STD, gamma=bench.GAMMA, exact_grad=False)
        return sf

    results = []
    for L in args.lengths:
        ys = [cg(torch.randn(L, C, H, W, generator=torch.Generator().manual_seed(1000 * L + m)))
              for m in range(max(args.members))]
        for M in args.members:
            batch_sfs = [score_fn(ys[m]) for m in range(M)]   # one per member, its own y
            seq_sfs = [score_fn(ys[m]) for m in range(M)]     # the same problems, run one after the other
            ens_sf = score_fn(ys[0])                          # one y for every member
            noise = torch.randn(M, L, C, H, W, generator=torch.Generator().manual_seed(100 * L + M)).to(dev)
            arms = {
                "batch": lambda: pipe.sample_batch(batch_sfs, noise, steps=args.steps, show_progressbar=False),
                "sequential": lambda: torch.stack([pipe.sample(seq_sfs[m], noise[m], steps=args.steps,
                                                               show_progressbar=False) for m in range(M)]),
                "ensemble": lambda: pipe.sample_ensemble(ens_sf, noise, steps=args.steps, show_progressbar=False),
            }
            outs = {k: timed(fn)[0] for k, fn in arms.items()}  # warm-up: each arm's runtimes, engine and workspace
            identical = all(torch.equal(outs["batch"][m], outs["sequential"][m]) for m in range(M))
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
            row["speedup_over_sequential_best"] = round(min(secs["sequential"]) / min(secs["batch"]), 3)
            row["batch_over_ensemble_best"] = round(min(secs["batch"]) / min(secs["ensemble"]), 3)
            print(f"L={L:4d} M={M}: batch {row['batch']['ms_per_step_best']:9.3f} ms/step "
                  f"{row['batch']['frames_per_s_best']:8.2f} frames/s | sequential "
                  f"{row['sequential']['ms_per_step_best']:9.3f} ms/step | ensemble (one y) "
                  f"{row['ensemble']['ms_per_step_best']:9.3f} ms/step | x{row['speedup_over_sequential_best']:.3f} "
                  f"over sequential, {row['batch_over_ensemble_best']:.3f} of the ensemble's time | "
                  f"bit-identical {identical}", flush=True)
            results.append(row)
            del noise, outs
    out = {"gpu": gpu_info(), "workload": f"{C}x{H}x{W} frames, sda_unet.yml ScoreUNet (random init), k={bench.K_ORDER}, "
           f"CoarseGrain(6, 16), a y per member, closed-form guidance, 0 corrections, default windows per launch "
           f"(min(M (L - 2k), {c2w.DefaultScoreFunction.DEFAULT_WINDOWS})), whole sample calls in steady state",
           "steps": args.steps, "rounds": args.rounds, "results": results}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
