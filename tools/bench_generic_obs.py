"""What the generic observation path costs (an observation operator A the fused guidance kernels do not implement, run
by torch with its VJP between c2w_x0_nchw and c2w_guided_step_dense), at bench.py's config-2 geometry: the
sda_unet.yml ScoreUNet (random init), L = 168 frames of 4 x 128 x 128, k = 6 (156 windows in one launch), bench.py's
std and gamma, the step of bench.py (window score, guidance + predictor; no corrections) on bench.py's 256-step
schedule.  Arms:

- fused:      CoarseGrain(6, 16) on the fused path (K6);
- generic:    the same operator forced through the generic path (the recogniser bypassed; there is no user switch);
- time_mean:  6-frame means of 16 x 16 tile means, an operator only the generic path runs;

closed-form guidance for all three, exact_grad for the first two (the generic path then runs the backward of every
window: it cannot know which frames an arbitrary A reads).  Each arm times --steps steps with CUDA events after
--warmup untimed ones; the arms alternate, --rounds times, best reported.  Prints the GPU's name and power limit and
one JSON line."""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()

    import torch
    import torch.nn.functional as F

    import bench
    import climate2weather_b200 as c2w
    from bench_ensemble import gpu_info
    from climate2weather_b200 import score

    if not torch.cuda.is_available():
        raise SystemExit("bench_generic_obs.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda:0")
    C, H, W, k = bench.C, bench.H, bench.W, bench.K_ORDER
    L = bench.WINDOWS_PER_GPU + 2 * k
    torch.manual_seed(0)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, **bench.ARCH).requires_grad_(False).to(dev)
    truth = torch.randn(L, C, H, W, generator=torch.Generator().manual_seed(1))
    noise = torch.randn(L, C, H, W, generator=torch.Generator().manual_seed(2)).to(dev)
    cg = c2w.CoarseGrain(6, 16)

    def time_mean(x):  # 6-frame means of 16 x 16 tile means: [L / 6, C, H / 16, W / 16]
        p = F.avg_pool2d(x, 16)
        return p.reshape(-1, 6, *p.shape[1:]).mean(1)

    def stepper(op, exact, generic):
        with contextlib.ExitStack() as stack:
            stack.enter_context(contextlib.redirect_stdout(io.StringIO()))
            if generic:  # the runtime (built in Stepper) routes the operator
                route = score._route_operator
                score._route_operator = lambda A, *a: score.GenericObservation(A)
                stack.callback(setattr, score, "_route_operator", route)
            st = bench.Stepper(net, noise, op(truth), op, dev, bench.WINDOWS_PER_GPU, exact, shard=False)
        kind = type(st.rt.cond["op"]).__name__
        assert (kind == "GenericObservation") == (generic or op is time_mean), kind
        return st

    arms = {
        "fused closed-form": stepper(cg, False, False),
        "generic closed-form": stepper(cg, False, True),
        "time_mean closed-form": stepper(time_mean, False, False),
        "fused exact": stepper(cg, True, False),
        "generic exact": stepper(cg, True, True),
    }
    ms = {a: [] for a in arms}
    for _ in range(args.rounds):
        for a, st in arms.items():
            ms[a].append(st.timed(args.steps, args.warmup, torch.cuda.synchronize) / args.steps)
    best = {a: min(v) for a, v in ms.items()}
    gpu = gpu_info()
    print(f"{gpu['name']}, power limit {gpu['power_limit']}, SM clock max {gpu['sm_max_clock']}")
    for a in arms:
        base = best["fused exact" if "exact" in a else "fused closed-form"]
        print(f"{a:24s} {best[a]:8.3f} ms/step (best of {args.rounds}; all {[round(v, 3) for v in ms[a]]}) "
              f"{100 * (best[a] / base - 1):+7.2f} % vs the fused path")
    print(json.dumps({"gpu": gpu, "workload": f"L={L} x {C}x{H}x{W}, k={k}, sda_unet.yml ScoreUNet (random init), "
                      f"{bench.WINDOWS_PER_GPU} windows per launch, guidance + predictor step, 0 corrections",
                      "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds,
                      "ms_per_step": {a: [round(v, 4) for v in ms[a]] for a in arms},
                      "ms_per_step_best": {a: round(v, 4) for a, v in best.items()}}))


if __name__ == "__main__":
    main()
