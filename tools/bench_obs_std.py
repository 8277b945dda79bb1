"""Cost of a noise std per observation (c2w_guided_step_obs_std) against one std per variable, for a coarse field
(CoarseGrain, K6), stations (PointObservation, K6p) and both together (CombinedObservation, K6c), at config-2 shapes:
the sda_unet.yml ScoreUNet (random init), L = 168 frames of 4 x 128 x 128, k = 6, closed-form guidance.

* step time: ms per denoising step (window score + guidance/predictor), CUDA events over --steps steps after --warmup,
  for CoarseGrain(6, 16), 1000 stations on every 6th frame (100 of them on the pixel of another, so that stations with
  different std form runs of entries), and both, each with a per-variable std and with a std per observation (per tile
  and frame; per station and variable from three classes).  The six variants run in turn, --rounds times, so the
  run-to-run spread is visible next to any difference.
* kernel time: the guidance kernel of each variant alone (mode 0 with t = t_next, which leaves x unchanged), CUDA
  events over --launches launches.  Bytes are algorithmic: read x and eps, write x (48 B per pixel of an owned frame),
  plus the coarse y and std^2 block and the point entries, their std^2 and the CSR.  x and eps (44 MB each) fit the
  126 MB L2, so the rate is an L2-assisted upper bound on the HBM rate.
Prints the GPU's name and power limit, read in the same call, and one JSON line."""
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
        raise SystemExit("bench_obs_std.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda:0")
    L, C, H, W = bench.L_WEEK, bench.C, bench.H, bench.W
    net, noise, y_cg, cg = bench.make_problem(L)
    net = net.to(dev)
    truth = torch.randn(L, C, H, W, generator=torch.Generator().manual_seed(5))
    g = torch.Generator().manual_seed(7)
    st_rows = torch.randint(0, H, (1000,), generator=g)
    st_cols = torch.randint(0, W, (1000,), generator=g)
    st_rows[900:], st_cols[900:] = st_rows[:100], st_cols[:100]  # duplicated sites
    stations = c2w.PointObservation(list(range(0, L, 6)), st_rows, st_cols)
    both = c2w.CombinedObservation(cg, stations)
    std_c = torch.tensor(bench.STD)
    cs, ps = both.term_shapes((L, C, H, W))
    std_tile = std_c.reshape(1, C, 1, 1) * (1 + torch.rand(cs, generator=g))
    std_station = std_c.reshape(1, C, 1) * torch.tensor([1.0, 1.5, 2.0])[torch.randint(0, 3, (1, C, 1000), generator=g)]
    y_st = stations(truth)
    ops = {  # name -> (operator, y, std)
        "coarse_per_var": (cg, y_cg, std_c.reshape(1, C, 1, 1)),
        "coarse_per_obs": (cg, y_cg, std_tile),
        "points_per_var": (stations, y_st, std_c.reshape(1, C, 1)),
        "points_per_obs": (stations, y_st, std_station),
        "combined_per_var": (both, both.pack(y_cg, y_st, (L, C, H, W)), std_c),
        "combined_per_obs": (both, both.pack(y_cg, y_st, (L, C, H, W)), both.pack(std_tile, std_station.expand(ps),
                                                                                 (L, C, H, W))),
    }
    steppers = {k: bench.Stepper(net, noise, y_cg, cg, dev, bench.WINDOWS_PER_GPU, False, False) for k in ops}
    for k, (op, y, std) in ops.items():
        # a pixel observed directly takes weight r^2 / (std^2 + gamma r^2), r = sigma/mu ~ 1e3 at t = 1: gamma = 1
        # bounds it by 1 (bench_point_obs.py); the coarse variants keep the coarse gamma
        st = steppers[k]
        st.sf.condition_on(A=op, y=y, std=std, gamma=bench.GAMMA if op is cg else 1.0, exact_grad=False)
        st.rt = st.sf.runtime(noise)
        assert (st.rt.cond.get("obs_std") is not None) == k.endswith("per_obs"), k
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
        if not isinstance(rt.cond["op"], c2w.PointObservation):
            nbytes += rt.y_dev.numel() * 4
        if rt.coarse_std2_dev is not None:
            nbytes += rt.coarse_std2_dev.numel() * 4
        if rt.points is not None:
            t = rt.points["tensors"]
            nbytes += sum(v.numel() * 4 for v in t.values())
        name = {"coarse": "K6", "points": "K6p", "combined": "K6c"}[k.split("_")[0]]
        entry = "c2w_guided_step_obs_std" if k.endswith("per_obs") else \
            {"K6": "c2w_guided_step", "K6p": "c2w_guided_step_points", "K6c": "c2w_guided_step_combined"}[name]
        kern[k] = {"kernel": f"{entry} ({name})", "us": round(ms * 1e3, 2), "bytes": nbytes,
                   "TBps": round(nbytes / (ms * 1e-3) / 1e12, 3)}
        if rt.points is not None:
            kern[k]["entries"] = int(rt.points["tensors"]["pix"].numel())
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
