"""Cost of point observations (PointObservation) against the coarse-graining operator at config-2 shapes: the
sda_unet.yml ScoreUNet (random init), L = 168 frames of 4 x 128 x 128, k = 6, closed-form guidance.

* step time: ms per denoising step (window score + guidance/predictor), CUDA events over --steps steps after --warmup,
  for CoarseGrain(6, 16) and three point operators: (a) 1000 stations on every 6th frame, (b) 1000 stations on every
  frame, (c) every pixel of every 6th frame.  The variants run in turn, --rounds times, so the spread is visible.
* kernel time: c2w_guided_step against c2w_guided_step_points alone (mode 0 with t = t_next, which leaves x
  unchanged), CUDA events over --launches launches.  Bytes are algorithmic: read x and eps, write x (48 B per pixel of
  an owned frame) plus the point entries (4 B pixel + 32 B ysum/wsum each) and the CSR.  x and eps (44 MB each) fit
  the 126 MB L2, so the rate is an L2-assisted upper bound on the HBM rate.
Prints the GPU's name and power limit and one JSON line."""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
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
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--launches", type=int, default=200)
    args = ap.parse_args()

    import torch

    import bench
    import climate2weather_b200 as c2w

    if not torch.cuda.is_available():
        raise SystemExit("bench_point_obs.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda:0")
    L, C, H, W = bench.L_WEEK, bench.C, bench.H, bench.W
    net, noise, y_cg, cg = bench.make_problem(L)
    net = net.to(dev)
    truth = torch.randn(L, C, H, W, generator=torch.Generator().manual_seed(5))
    g = torch.Generator().manual_seed(7)
    st_rows = torch.randint(0, H, (1000,), generator=g)
    st_cols = torch.randint(0, W, (1000,), generator=g)
    rr, cc = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    ops = {
        "coarse_grain_t6_s16": (cg, y_cg),
        "points_1000_every6": c2w.PointObservation(list(range(0, L, 6)), st_rows, st_cols),
        "points_1000_every_frame": c2w.PointObservation(list(range(L)), st_rows, st_cols),
        "points_all_pixels_every6": c2w.PointObservation(list(range(0, L, 6)), rr.reshape(-1), cc.reshape(-1)),
    }
    for k, v in ops.items():
        if not isinstance(v, tuple):
            ops[k] = (v, v(truth))
    steppers = {k: bench.Stepper(net, noise, y, op, dev, bench.WINDOWS_PER_GPU, False, False) for k, (op, y) in ops.items()}
    for k, (op, y) in ops.items():
        if isinstance(op, c2w.PointObservation):
            # a pixel observed directly takes weight r^2 / (std^2 + gamma r^2), r = sigma/mu ~ 1e3 at t = 1: the
            # coarse-graining gamma (7e-4) would overshoot by ~1/gamma and the trajectory would leave the finite range;
            # gamma = 1 bounds the weight by 1 (the same number of bytes and launches either way)
            st = steppers[k]
            st.sf.condition_on(A=op, y=y, std=torch.tensor(bench.STD).reshape(1, C, 1), gamma=1.0, exact_grad=False)
            st.rt = st.sf.runtime(noise)
    step_ms = {k: [] for k in ops}
    for _ in range(args.rounds):
        for k, st in steppers.items():
            step_ms[k].append(st.timed(args.steps, args.warmup, torch.cuda.synchronize) / args.steps)

    finite = {k: int(st.rt.nan_flag.item()) == 0 for k, st in steppers.items()}
    kern = {}
    for k, st in steppers.items():
        rt = st.rt
        rt.reset_finite_check()
        rt.load(noise)
        for _ in range(10):
            rt.predictor(0.5, 0.5, 0.5, 0.5)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.launches):
            rt.predictor(0.5, 0.5, 0.5, 0.5)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.launches
        nbytes = rt.plan.own_n * H * W * C * 4 * 3
        if rt.points is not None:
            t = rt.points["tensors"]
            nbytes += sum(t[n].numel() * 4 for n in ("frame_slot", "strip_off", "pix", "ysum", "wsum"))
        kern[k] = {"kernel": "c2w_guided_step_points" if rt.points is not None else "c2w_guided_step",
                   "us": round(ms * 1e3, 2), "bytes": nbytes, "TBps": round(nbytes / (ms * 1e-3) / 1e12, 3),
                   "entries": int(rt.points["tensors"]["pix"].numel()) if rt.points is not None else None}
        assert int(rt.nan_flag.item()) == 0
    out = {"gpu": gpu_info(), "workload": f"L={L} frames of {C}x{H}x{W}, sda_unet.yml ScoreUNet (random init), "
           f"k={bench.K_ORDER}, {bench.WINDOWS_PER_GPU} windows per launch, closed-form guidance, predictor only",
           "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds,
           "step_ms": {k: [round(v, 4) for v in vs] for k, vs in step_ms.items()},
           "step_ms_min": {k: round(min(vs), 4) for k, vs in step_ms.items()},
           "trajectory_finite": finite, "kernel": kern, "kernel_note": "L2-assisted: x and eps (44 MB each) fit the 126 MB L2"}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
