#!/usr/bin/env python
"""bench.py — guided-sampling frames/sec of the Climate2Weather hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Workloads (config.workload), all on the ScoreUNet of configs/sda_unet.yml (random init), 4 x 128 x 128 frames, Markov
order k = 6, 256 denoising steps, 0 corrections, tau 0.5, closed-form guidance (exact_grad False), observation = every
6th frame's 16x16 tile means (exp/configs/000_on-model-eval/s16_t6.yml):

  N = 1 (default)  BASELINE.json configs[1]: a 1-week hourly trajectory, L = 168 frames (156 windows), one GPU.
  N > 1 (default)  BASELINE.json configs[2]: a 1-month trajectory, L = 720 frames (708 windows) TIME-SHARDED over the
                   N GPUs with the k boundary frames exchanged after every update — strong scaling.  Rank 0 also times
                   the same 720-frame trajectory on ONE GPU in the same run (`strong_scaling` in the line).
  --config 4       BASELINE.json configs[3]: a 16-member ensemble of a synthetic year (L = 8760) over the N GPUs,
                   members as independent replicas (16 / N per GPU, exp/downscaling.py:96-99,248-261), windows chunked.
  --weak           the round-1 weak-scaling workload (L = 12 + 156 N).

A "step" is one denoising step over the whole trajectory: window score (UNet on every window of this rank) + fused
guidance and predictor update (+ halo exchange).  `value` = frames / (256 * mean step time): frames per second of a
full 256-step sampling run, state resident in HBM, timed with CUDA events over exactly K steps, max over ranks.
`e2e` = the same metric through the public API (SDAPipeline.sample) with pinned HOST noise in, HOST result out and
the per-step NaN-flag read the reference does (src/thor/pipelines.py:90), all inside the timed region.
`--impl reference` times the reference's CPU path (the oracle port, all host threads) on the same config.
`--dump-outputs DIR` saves what the last timed step computed (see `dump_outputs`): the inputs are seeded, so two builds
run with the same arguments can be compared array for array.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

SAMPLER_STEPS = 256
K_ORDER = 6
C, H, W = 4, 128, 128
WINDOWS_PER_GPU = 156
L_WEEK, L_MONTH, L_YEAR, MEMBERS = 168, 720, 8760, 16
T_STEP, S_STEP = 6, 16
STD = [0.1692666615037876, 0.0425178630338289, 0.3268027589410125, 0.3268027589410125]
GAMMA = 0.0007196856730011522
F_WIN_CONV = 115.134e9  # Conv2d FLOPs per window forward (SURVEY.md §8(d), BASELINE.md §2)
F_WIN = 116.0e9
FRAME_BYTES = C * H * W * 4
DUMP_BYTES = 64_000_000  # --dump-outputs: all .npy files together, headers included
ARCH = dict(channels=52, embedding_dim=512, hidden_channels=[128, 128, 256, 384, 512], hidden_blocks=[3, 3, 3, 3, 3],
            attention_levels=[4])


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured"
    return 1400.0, 6650.0, "fallback"


def k1_traffic():
    """DRAM bytes per K1 launch from the committed ncu capture of one step (profiles/k1_traffic.json, written by
    tools/ncu_traffic.py from `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum` over bench.py --profile)."""
    p = ROOT / "profiles" / "k1_traffic.json"
    if not p.exists():
        return None, None
    d = json.loads(p.read_text())
    return d.get("dram_bytes_per_launch"), d


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line).  The sampler is
    started BEFORE the warm-up (nvidia-smi needs a few hundred ms to come up) and every row is stamped on arrival;
    the summary uses the rows between mark_start() and mark_end()."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def mark_start(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        t0, t1 = self.t0 or 0.0, self.t1 or float("inf")
        inside = [r for ts, r in self.rows if t0 <= ts <= t1 + 0.05]
        rows = inside or [r for _, r in self.rows]
        sm, mx, reasons = [], 0, set()
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm),
                "window": "timed region" if inside else "whole run"}


def member_seed(seed: int, rank: int) -> int:
    """util.set_random_seed (util.py:27-29): hash((seed, rank)) % 2**31 — Python's tuple-of-ints hash is deterministic."""
    return hash((seed, rank)) % (1 << 31)


def make_problem(L: int, seed: int = 0, with_net: bool = True):
    import torch

    import climate2weather_b200 as c2w

    net = None
    if with_net:
        torch.manual_seed(0)
        net = c2w.ScoreUNet(activation=torch.nn.SiLU, **ARCH).requires_grad_(False)
    g = torch.Generator().manual_seed(seed + 1)
    noise = torch.randn(L, C, H, W, generator=g)
    truth = torch.randn(L, C, H, W, generator=g)
    cg = c2w.CoarseGrain(T_STEP, S_STEP)
    y = cg(truth)
    return net, noise, y, cg


def pick_workload(args, world: int):
    """(name, L, scaling, members_per_gpu)."""
    if args.config == 4:
        if MEMBERS % world:
            raise SystemExit(f"config 4: {MEMBERS} members do not divide over {world} GPUs")
        return "config4", args.frames or L_YEAR, "weak", MEMBERS // world
    if args.weak:
        return "config2-weak", args.frames or (2 * K_ORDER + WINDOWS_PER_GPU * world), "weak", 0
    if world == 1 and args.config in (None, 2):
        return "config2", args.frames or L_WEEK, "weak", 0
    return "config3", args.frames or L_MONTH, "strong", 0


def workload_config(name: str, L: int, world: int, members_per_gpu: int, exact: bool) -> dict:
    """The part of `config` both arms (ours and --impl reference) print identically: which BASELINE.json workload it is."""
    desc = {"config2": f"config2: guided PC sampling of a 1-week trajectory, L={L} frames",
            "config2-weak": f"config2 weak scaling: L={L} frames ({WINDOWS_PER_GPU} windows per GPU)",
            "config3": f"config3: time-sharded guided PC sampling of a 1-month trajectory, L={L} frames over {world} GPU(s)",
            "config4": f"config4: {MEMBERS}-member ensemble of a synthetic year, L={L} frames per member, "
                       f"{members_per_gpu} member(s) per GPU as independent replicas"}[name]
    return {"workload": f"{desc} of {C}x{H}x{W}, sda_unet.yml ScoreUNet k={K_ORDER}, {SAMPLER_STEPS} steps, 0 corrections, "
                        f"{'exact-grad (UNet VJP)' if exact else 'approx-grad'} guidance t_step={T_STEP} s_step={S_STEP}",
            "name": name, "frames": L, "members": MEMBERS if name == "config4" else 1, "sampler_steps": SAMPLER_STEPS,
            "windows": L - 2 * K_ORDER}


# ====================================================================================================== ours
class Stepper:
    """One resident trajectory (or this rank's shard of it) and its denoising step."""

    def __init__(self, net, noise, y, cg, dev, chunk, exact, shard):
        import torch

        import climate2weather_b200 as c2w
        from climate2weather_b200.score import _mu_sigma

        self.torch, self._mu_sigma = torch, _mu_sigma
        self.pipe = c2w.SDAPipeline()
        self.sf = c2w.BatchedScoreFunction(net, markov_order=K_ORDER, noise_process=self.pipe, batch_size=chunk, device=dev)
        self.sf.max_windows = chunk
        self.sf.condition_on(A=cg, y=y, std=torch.tensor(STD).reshape(1, C, 1, 1), gamma=GAMMA, exact_grad=exact)
        if shard:
            self.sf.enable_time_sharding()
        self.rt = self.sf.runtime(noise)
        self.group = None
        self.times = torch.linspace(1, 0, SAMPLER_STEPS + 1)
        self.noise = noise

    def load(self):
        self.rt.load(self.noise)

    def step(self, i: int):
        t = self.times[i % SAMPLER_STEPS]
        dt = 1 / SAMPLER_STEPS
        mu, sigma = self._mu_sigma(self.pipe, t)
        mu_n, sigma_n = self._mu_sigma(self.pipe, t - dt)
        self.rt.score(float(t), self.group)
        self.rt.predictor(mu, sigma, mu_n, sigma_n)
        self.rt.halo(self.group)

    def timed(self, steps: int, warmup: int, barrier, clocks=None):
        """ms for exactly `steps` steps (CUDA events on the launch stream), after `warmup` untimed steps."""
        torch = self.torch
        self.load()
        for i in range(warmup):
            self.step(i)
        self.load()  # restart the trajectory so the timed steps see the schedule from t = 1
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if clocks:
            clocks.mark_start()
        e0.record()
        for i in range(steps):
            self.step(i)
        e1.record()
        barrier()
        if clocks:
            clocks.mark_end()
        return e0.elapsed_time(e1)


def hbm_kernel_rates(lib, rt, dev, peak_gbs):
    """Achieved GB/s of the two HBM-bound kernels of a step, each timed alone with CUDA events over 20 launches.
    K6 guided predictor: algorithmic 3 x 4 x H x W x 4 B per owned frame (read x, read eps, write x).
    K0 window gather: algorithmic DRAM bytes = the local trajectory read once + the bf16 window batch written once
    (the 13x re-reads of a frame by neighbouring windows are L2 hits).
    Working sets (x, eps, the window batch) are re-touched every launch; at L = 168 x and eps (44 MB each) fit the
    126 MB L2, so K6's figure there is an L2-assisted upper bound — stated with the number (`l2_resident`)."""
    import torch

    from climate2weather_b200 import _lib as L_

    out = {}
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    n = 20
    rt.score(0.5)  # eps valid
    e0, e1 = ev(), ev()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        rt.predictor(0.9, 0.4, 0.9, 0.4)  # mu == mu_next, sigma == sigma_next: x is a fixed point, values stay finite
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    by = 3 * FRAME_BYTES * rt.plan.own_n
    out["K6_guided_predictor"] = {"GBps": round(by / ms / 1e6, 1), "frac": round(by / ms / 1e6 / peak_gbs, 4),
                                  "bytes_per_launch": by, "ms": round(ms, 5), "l2_resident": bool(by < 126e6)}
    nw = min(rt.engine.max_windows, rt.plan.win_hi - rt.plan.win_lo)
    xin = torch.empty(nw, H * W, 64, dtype=torch.bfloat16, device=dev)
    e0, e1 = ev(), ev()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        L_.check(lib.c2w_op_gather_windows(rt.x.data_ptr(), xin.data_ptr(), nw, H * W, C, 2 * K_ORDER + 1, 64, 0,
                                           torch.cuda.current_stream().cuda_stream), "gather")
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    by = (nw + 2 * K_ORDER) * FRAME_BYTES + nw * H * W * 64 * 2
    out["K0_gather_windows"] = {"GBps": round(by / ms / 1e6, 1), "frac": round(by / ms / 1e6 / peak_gbs, 4),
                                "bytes_per_launch": by, "ms": round(ms, 5), "l2_resident": bool(by < 126e6)}
    return out


def dump_outputs(out_dir: str, st: Stepper, rank: int) -> None:
    """Writes the state the last step left as float32 [frames, C, H, W] arrays: `x.npy`, the trajectory a caller of
    SDAPipeline.sample receives, and `eps.npy`, the window score that step computed.  A time-sharded run gathers the
    frames on rank 0, which writes them; in the ensemble, rank 0 writes its own member.  When the whole trajectory
    would exceed DUMP_BYTES, both arrays hold every s-th frame (0, s, 2s, ...) for the smallest s that fits."""
    import numpy as np

    from climate2weather_b200.sharding import gather_frames

    rt = st.rt
    group = st.sf.shard[2] if st.sf.shard else None
    arrays = {name: gather_frames(rt.owned(buf), rt.plan, group) for name, buf in (("x", rt.x), ("eps", rt.eps))}
    if rank != 0:
        return
    n = arrays["x"].shape[0]
    # 4 KB per file for the .npy header (128 B for these arrays)
    fit = max(1, (DUMP_BYTES - 4096 * len(arrays)) // (len(arrays) * FRAME_BYTES))
    stride = -(-n // min(n, fit))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a[::stride].cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist

    import climate2weather_b200 as c2w
    from climate2weather_b200 import _lib

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    name, L, scaling, members_per_gpu = pick_workload(args, world)
    lib = _lib.load()
    peak_tf, peak_gbs, peak_src = measured_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(v: float) -> float:
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    ensemble = name == "config4"
    seed = member_seed(0, rank) if ensemble else 0  # exp/downscaling.py:103: every rank seeds its own members
    net, noise, y, cg = make_problem(L, seed=seed)
    net = net.to(dev)

    # ---- strong scaling: the same trajectory on ONE GPU (rank 0), before the sharded run
    single = None
    if name == "config3" and world > 1 and not args.no_single:
        if rank == 0:
            s1 = Stepper(net, noise, y, cg, dev, args.chunk, args.exact_grad, shard=False)
            ks = max(2, min(args.steps, 6))
            ms1 = s1.timed(ks, 3, lambda: torch.cuda.synchronize()) / ks
            single = {"ms_per_step": round(ms1, 4), "value": round(L / (SAMPLER_STEPS * ms1 / 1e3), 3),
                      "windows": L - 2 * K_ORDER, "steps": ks}
            del s1
            torch.cuda.empty_cache()
        barrier()

    st = Stepper(net, noise, y, cg, dev, args.chunk, args.exact_grad, shard=(world > 1 and not ensemble))
    rt = st.rt
    n_win_local = rt.plan.win_hi - rt.plan.win_lo

    # ---- device-resident timed region: exactly K steps, CUDA events on the launch stream
    with ClockSampler(local_rank) as clocks:
        launches0 = lib.c2w_launch_count()
        ms_total = st.timed(args.steps, args.warmup, barrier, clocks)
        launches = lib.c2w_launch_count() - launches0
    launches = launches * args.steps // (args.steps + args.warmup)  # the counter also saw the warm-up steps
    if args.dump_outputs:  # before the roofline and e2e legs below step the same state further
        dump_outputs(args.dump_outputs, st, rank)
    ms_step = allmax(ms_total) / args.steps
    frames_total = L * (MEMBERS if ensemble else 1)
    # ensemble: each GPU runs its members one after the other -> a GPU-step of the job costs members_per_gpu steps
    value = frames_total / (SAMPLER_STEPS * ms_step * (members_per_gpu if ensemble else 1) / 1e3)
    rt.check_finite()

    # ---- roofline pass: event-time every forward-pass launch of a few steps (same process, right after)
    engs = rt.engines()
    for eng in engs:
        _lib.check(lib.c2w_set_timing(eng.handle, 1), "c2w_set_timing")
    # one untimed transition step (the GPU leaves the back-to-back regime: with an event pair around every launch it
    # idles between kernels), then per-step sums of up to 6 steps; the MEDIAN step is reported, min / max alongside
    nprof = 0 if args.profile else min(args.steps, 6 if not ensemble else 1)
    per_step = []  # (K1 ms, other ms, K1 launches)
    for i in range(nprof + (1 if nprof else 0)):
        st.step(i)
        acc = [0.0, 0.0, 0]
        for eng in engs:
            m_, c_ = (ctypes.c_double * 2)(), (ctypes.c_int64 * 2)()
            _lib.check(lib.c2w_timing_read(eng.handle, m_, c_), "c2w_timing_read")
            acc[0] += m_[0]
            acc[1] += m_[1]
            acc[2] += c_[0]
        if i > 0 or nprof == 0:
            per_step.append(acc)
    for eng in engs:
        _lib.check(lib.c2w_set_timing(eng.handle, 0), "c2w_set_timing")
    per_step.sort(key=lambda a: a[0])
    med = per_step[len(per_step) // 2] if per_step else [0.0, 0.0, 0]
    conv_ms_step, other_ms_step = med[0], med[1]
    n2 = [med[2], 0]
    k1_range = [round(per_step[0][0], 3), round(per_step[-1][0], 3)] if per_step else None
    # K1 work per step: every conv / 1x1 GEMM of the forward pass.  exact-grad (src/thor/score.py:28-33,51-52) adds, for
    # the windows whose output meets an observed frame (the others have a zero cotangent), a stashing forward and the
    # input-gradient conv of each layer (same FLOPs with Cin and Cout swapped)
    n_sel = rt.n_selected if args.exact_grad else 0
    n_rep = rt.n_repeated if args.exact_grad else 0  # windows whose forward runs twice (several stashing chunks)
    k1_flops_step = F_WIN_CONV * (n_win_local + n_sel + n_rep)
    conv_tf = k1_flops_step / (conv_ms_step * 1e-3) / 1e12 if conv_ms_step > 0 else 0.0
    traffic, traffic_src = k1_traffic()
    k1_per_step = n2[0]
    roofline = {
        "kernel": "conv_gemm_tcgen05_kernel (K1, all %d conv/GEMM launches of a step)" % k1_per_step,
        "bound": "tensor", "achieved": round(conv_tf, 1), "peak": peak_tf, "unit": "TFLOP/s",
        "frac": round(conv_tf / peak_tf, 4), "peak_source": f"{peak_src} bf16_tflops_sustained",
        "traffic": traffic, "traffic_source": (traffic_src or {}).get("source"),
        "algorithmic_flops_per_launch": k1_flops_step / max(k1_per_step, 1),
        "algorithmic_flops_per_step": k1_flops_step,
        "avg_launch_ms": round(conv_ms_step / max(1, n2[0]), 5), "k1_ms_per_step": round(conv_ms_step, 3),
        "k1_ms_per_step_min_max": k1_range, "timed_steps": len(per_step),
        "timing": "CUDA events around every launch, median of the event-timed steps (one transition step discarded)",
        "other_fwd_kernels_ms_per_step": round(other_ms_step, 3),
        "k1_share_of_step": round(conv_ms_step / ms_step, 4),
        "whole_step_frac": round(k1_flops_step / (ms_step * 1e-3) / 1e12 / peak_tf, 4),
    }
    hbm = None
    if not args.profile and not ensemble and not args.exact_grad:
        hbm = hbm_kernel_rates(lib, rt, dev, peak_gbs)

    # ---- end to end through the public API: pinned host noise in, host result out, per-step NaN-flag read
    e2e = None
    if not args.no_e2e:
        pipe2 = c2w.SDAPipeline()
        pipe2.nan_check_every = 1
        noise_pinned = noise.pin_memory()
        ke = max(1, args.e2e_steps)  # one full sample() call of this many denoising steps (independent of --steps)
        # untimed warm-up of the API path itself (3 steps): pinned-buffer allocation and, time-sharded, the first-use
        # NCCL connections of the final gather to rank 0
        pipe2.sample(st.sf, noise_pinned, steps=3, corrections=0, tau=0.5, show_progressbar=False)
        barrier()
        t0 = time.perf_counter()
        out = pipe2.sample(st.sf, noise_pinned, steps=ke, corrections=0, tau=0.5, show_progressbar=False)
        barrier()
        dt_e2e = allmax(time.perf_counter() - t0)
        if out is not None:  # time-sharded: the trajectory is assembled on rank 0 only
            assert out.device.type == "cpu" and tuple(out.shape) == (L, C, H, W) and bool(torch.isfinite(out).all())
        sharded = world > 1 and not ensemble
        e2e = {"value": round(frames_total / (SAMPLER_STEPS * dt_e2e * (members_per_gpu if ensemble else 1) / ke), 3),
               "unit": "frames/s",
               "h2d_bytes_per_step": int(rt.plan.n_local * FRAME_BYTES / ke),
               "d2h_bytes_per_step": int((L if (sharded and rank == 0) else rt.plan.own_n) * FRAME_BYTES / ke) + 4,
               "api": f"SDAPipeline.sample(BatchedScoreFunction, pinned host noise, steps={ke}) -> host tensor"
                      + (" on rank 0 (gather over NVLink)" if sharded else ""),
               "steps": ke}

    # ---- CPU baseline (rank 0, N = 1 only): the oracle port on the host cores, bounded sample
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu and not ensemble:
        cpu = cpu_reference(L, sample_windows=args.cpu_windows, steps=1)

    if rank == 0:
        x2 = (n_win_local + n_sel + n_rep) / n_win_local
        line = {
            "metric": "guided-sampling frames/sec", "value": round(value, 3), "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_step, 4), "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {**workload_config(name, L, world, members_per_gpu, args.exact_grad),
                       "windows_per_gpu": n_win_local, "vjp_windows_per_gpu": n_sel, "chunk_windows": rt.engine.max_windows,
                       "workspace_bytes": int(rt.engine.workspace.numel()),
                       "parallelism": (f"{members_per_gpu} replica member(s) per GPU x{world}" if ensemble
                                       else f"time-shard x{world}"),
                       "l2": "per-step working set (activations of a chunk + 144 MB packed weights) exceeds the 126 MB "
                             "L2; no explicit flush"},
            "clocks": clocks.summary(), "gpu_launches": int(launches),
            "roofline": roofline, "flops_per_step": F_WIN * n_win_local * world * x2,
            "achieved_tflops_whole_step": round(F_WIN * n_win_local * x2 / (ms_step * 1e-3) / 1e12, 1),
        }
        if hbm:
            line["hbm_kernels"] = dict(hbm, peak=peak_gbs, unit="GB/s", peak_source=f"{peak_src} hbm_gbs")
        if single:
            speedup = single["ms_per_step"] / ms_step
            line["strong_scaling"] = {"single_gpu": single, "speedup": round(speedup, 3),
                                      "efficiency": round(speedup / world, 4),
                                      "step_efficiency_window_normalised": round(
                                          single["ms_per_step"] / single["windows"] * n_win_local / ms_step, 4)}
        if e2e:
            line["e2e"] = e2e
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ====================================================================================================== training step
def run_train(args):
    """BASELINE.json configs[4]: the denoising-score-matching training step at the configured batch (run_training.sh:
    batch-gpu 128, 52 x 128 x 128 windows), the reference's own step body (training_loop.py:372-390)

        loss = pipeline.loss(net, x).mean(); loss.backward(); optimizer.step(); ema.update()

    on this package's ScoreUNet / AdamW / StandardEMA; DDP gradient all-reduce over NCCL for N > 1.  Metric: training
    samples/s (whole job); roofline: algorithmic 3 x 116 GFLOP per sample (forward + input-gradient + weight-gradient
    GEMMs) against the measured bf16 peak."""
    import torch
    import torch.distributed as dist

    import climate2weather_b200 as c2w
    from climate2weather_b200 import _lib, optim

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    peak_tf, _, peak_src = measured_peaks()
    B = args.batch
    torch.manual_seed(0)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, **ARCH).to(dev).train()
    model = net
    use_ddp = world > 1 and args.ddp == "torch"
    if use_ddp:  # the reference's own route: Fabric strategy="ddp" (train.py:93-100) = torch DDP hooks on our gradients
        model = torch.nn.parallel.DistributedDataParallel(net, device_ids=[local_rank])
    pipe = c2w.SDAPipeline()
    # default for N > 1: one in-place NCCL all-reduce of the flat gradient buffer inside optimizer.step()
    opt = optim.AdamW(net.parameters(), lr=1e-4, weight_decay=1e-3, betas=(0.9, 0.999),  # train.py:176-181
                      data_parallel_group=(None if (world > 1 and not use_ddp) else "none"), direct_grads=not use_ddp)
    if world > 1 and not use_ddp:
        opt.broadcast_parameters(0)
    ema = optim.StandardEMA(net, rates=[0.9999])
    opt.fuse_ema(ema)
    g = torch.Generator(device=dev).manual_seed(1 + rank)
    x = torch.rand(B, ARCH["channels"], H, W, generator=g, device=dev)  # quantile-normalised data lies in ~[0, 1]

    def step():
        opt.zero_grad()
        loss = pipe.loss(net=model, x=x).mean()
        loss.backward()
        opt.step()
        ema.update()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with ClockSampler(local_rank) as clocks:
        for _ in range(args.warmup):
            loss = step()
        barrier()
        launches0 = lib.c2w_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        clocks.mark_start()
        e0.record()
        for _ in range(args.steps):
            loss = step()
        e1.record()
        barrier()
        clocks.mark_end()
    launches = lib.c2w_launch_count() - launches0
    ms = torch.tensor([e0.elapsed_time(e1) / args.steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step = ms.item()
    assert bool(torch.isfinite(loss))
    flops = 3 * F_WIN * B
    # end to end: a fresh host batch every step (pinned), loss value read back
    xh = x.cpu().pin_memory()
    ke = max(2, min(args.steps, 8))
    barrier()
    t0 = time.perf_counter()
    for _ in range(ke):
        x.copy_(xh, non_blocking=True)
        lv = float(step().item())
    barrier()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    if rank == 0:
        line = {"metric": "DSM training samples/sec", "value": round(B * world / (ms_step / 1e3), 2), "unit": "samples/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_step, 3),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": f"config5: DSM training step, batch {B}/GPU x{world} of 52x128x128 windows, "
                                       "sda_unet.yml ScoreUNet (72.1 M parameters), AdamW lr 1e-4 wd 1e-3 + EMA 0.9999 "
                                       "(fused), per-sample diffusion times" + (("" if world == 1 else ", torch DDP all-reduce over NCCL" if use_ddp
                                                                  else ", flat-buffer gradient all-reduce over NCCL")),
                           "name": "config5", "batch_per_gpu": B, "global_batch": B * world,
                           "l2": "activations of a 128-sample batch (~14 GB) exceed the 126 MB L2; no explicit flush"},
                "clocks": clocks.summary(), "gpu_launches": int(launches),
                "roofline": {"kernel": "K1 forward / input-gradient convs + K10 weight-gradient GEMMs (whole step)",
                             "bound": "tensor", "achieved": round(flops / (ms_step * 1e-3) / 1e12, 1), "peak": peak_tf,
                             "unit": "TFLOP/s", "frac": round(flops / (ms_step * 1e-3) / 1e12 / peak_tf, 4),
                             "peak_source": f"{peak_src} bf16_tflops_sustained", "traffic": None,
                             "algorithmic_flops_per_step": flops},
                "loss": round(float(loss.item()), 5),
                "e2e": {"value": round(B * world * ke / dt.item(), 2), "unit": "samples/s",
                        "h2d_bytes_per_step": int(xh.numel() * 4), "d2h_bytes_per_step": 4, "steps": ke,
                        "api": "pipeline.loss(net, x).mean().backward(); optimizer.step(); ema.update() with a pinned host "
                               "batch copied in and the loss value read back every step"}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ====================================================================================================== reference arm
class CpuReference:
    """The oracle port of the reference path (fp32 torch on the host cores, all threads): guided predictor steps
    (BatchedScoreFunction.score_fn, src/thor/score.py:156-185, + closed-form guidance + SDAPipeline._sample_step) on a
    trajectory of `sample_windows` windows."""

    def __init__(self, sample_windows: int):
        import torch

        from oracle import pipeline_ref, score_ref, unet_ref

        self.torch, self.score_ref = torch, score_ref
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        self.sample_windows = sample_windows
        Ls = sample_windows + 2 * K_ORDER
        sd = unet_ref.init_state_dict(unet_ref.SDA_UNET, seed=0)
        self.net = unet_ref.RefNet(sd, unet_ref.SDA_UNET)
        g = torch.Generator().manual_seed(1)
        self.x = torch.randn(Ls, C, H, W, generator=g)
        self.y = score_ref.coarse_grain(torch.randn(Ls, C, H, W, generator=g), T_STEP, S_STEP)
        self.std = torch.tensor(STD).reshape(1, C, 1, 1)
        self.p = pipeline_ref.RefPipeline()
        self.ts = torch.linspace(1, 0, SAMPLER_STEPS + 1)
        self.i = 0

    def _guided(self, xx, tt):
        with self.torch.no_grad():
            eps = self.score_ref.window_score(self.net, xx, tt, K_ORDER, batch_size=32)
        return self.score_ref.guided_score_closed_form(eps, xx, tt, self.y, self.std, GAMMA, T_STEP, S_STEP)

    def step(self) -> float:
        """One guided predictor step; returns its wall time in seconds."""
        t0 = time.perf_counter()
        self.x = self.p.predictor(self._guided, self.x, self.ts[self.i % SAMPLER_STEPS], 1 / SAMPLER_STEPS)
        self.i += 1
        return time.perf_counter() - t0


def cpu_reference(L: int, sample_windows: int = 13, steps: int = 1):
    """cpu_baseline of the GPU line: `steps` guided predictor steps on a bounded sample of the workload, scaled to the
    full trajectory by the exact work ratio (cost is linear in windows, src/thor/score.py:143-185)."""
    n_win = L - 2 * K_ORDER
    sample_windows = min(sample_windows, n_win)
    ref = CpuReference(sample_windows)
    ref.step()  # untimed: thread pool, allocator and oneDNN primitive caches
    dt = sum(ref.step() for _ in range(steps)) / steps
    sec_per_window = dt / sample_windows
    value = L / (SAMPLER_STEPS * sec_per_window * n_win)
    return {"value": round(value, 6), "unit": "frames/s", "cores": ref.cores, "kind": "port",
            "sample": f"{steps} guided predictor step(s) on {sample_windows} of the {n_win} windows (L={sample_windows + 12} "
                      f"frames) after one untimed step, scaled x{n_win}/{sample_windows} (cost linear in windows)",
            "sec_per_window_eval": round(sec_per_window, 4), "threads": ref.cores}


def run_reference(args):
    """The reference arm: exactly --warmup untimed and --steps timed guided predictor steps of the oracle port on the
    host cores.  A step processes ALL windows of the config when that fits the time budget (--ref-budget-s for the whole
    run), otherwise a bounded sample of them — the same windows-per-step for every step, stated in `config`;
    `ms_per_step` is the MEASURED time of such a step and `value` scales it to the full trajectory by the window ratio."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    world = args.gpus
    name, L, scaling, members_per_gpu = pick_workload(args, world)
    n_win = L - 2 * K_ORDER
    t_start = time.perf_counter()
    probe = CpuReference(13)
    probe.step()                        # first-touch / thread-pool warm-up of the probe itself
    sec_per_window = probe.step() / 13  # one probe step prices a window
    del probe
    total_steps = args.steps + args.warmup
    budget = max(30.0, args.ref_budget_s - (time.perf_counter() - t_start))
    fit = int(budget / (total_steps * sec_per_window))
    ws = max(13, min(n_win, fit))
    if args.cpu_windows_ref:
        ws = min(n_win, args.cpu_windows_ref)
    ref = CpuReference(ws)
    for _ in range(args.warmup):
        ref.step()
    t0 = time.perf_counter()
    per = [ref.step() for _ in range(args.steps)]
    wall_timed = time.perf_counter() - t0
    ms_step_sample = 1e3 * wall_timed / args.steps
    sec_full_step = (wall_timed / args.steps) * n_win / ws
    value = L / (SAMPLER_STEPS * sec_full_step)  # one host runs one trajectory at a time: ensemble members are sequential
    cpu = {"value": round(value, 6), "unit": "frames/s", "cores": ref.cores, "kind": "port",
           "sample": f"{args.steps} timed guided predictor steps, each over {ws} of the {n_win} windows of the config"
                     + ("" if ws == n_win else f" (scaled x{n_win}/{ws}: cost is linear in windows)"),
           "sec_per_window_eval": round(wall_timed / args.steps / ws, 4), "threads": ref.cores,
           "step_s_min_max": [round(min(per), 3), round(max(per), 3)]}
    line = {"impl": "reference", "metric": "guided-sampling frames/sec", "value": round(value, 6), "unit": "frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_step_sample, 3),
            "ms_per_full_step_scaled": round(1e3 * sec_full_step, 3),
            "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {**workload_config(name, L, world, members_per_gpu, False),
                       "arm": "CPU oracle port of the reference path on the host cores", "windows_per_step": ws},
            "cpu_baseline": cpu,
            "e2e": {"value": round(value, 6), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "wall_s": round(time.perf_counter() - t_start, 1)}
    print(json.dumps(line), flush=True)


def run_reference_train(args):
    """Reference arm of config 5: the oracle port of the training step body (pipeline.loss(net, x).mean() -> backward
    through the fp32 UNet with torch autograd -> AdamW update, training_loop.py:372-390) on the host cores, on a bounded
    batch (--cpu-train-samples per step; cost is linear in the batch)."""
    import torch

    from oracle import pipeline_ref, unet_ref

    if int(os.environ.get("RANK", 0)) != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    t_start = time.perf_counter()
    sd = unet_ref.init_state_dict(unet_ref.SDA_UNET, seed=0)
    for v in sd.values():
        v.requires_grad_(True)
    net = unet_ref.RefNet(sd, unet_ref.SDA_UNET)
    opt = torch.optim.AdamW(list(sd.values()), lr=1e-4, weight_decay=1e-3)
    pipe = pipeline_ref.RefPipeline()
    b = max(1, args.cpu_train_samples)
    x = torch.rand(b, ARCH["channels"], H, W, generator=torch.Generator().manual_seed(1))

    def step():
        t0 = time.perf_counter()
        opt.zero_grad()
        pipe.loss(net, x).mean().backward()
        opt.step()
        return time.perf_counter() - t0

    for _ in range(args.warmup_train_ref):
        step()
    per = [step() for _ in range(args.steps)]
    sec = sum(per) / args.steps
    value = b / sec
    line = {"impl": "reference", "metric": "DSM training samples/sec", "value": round(value, 4), "unit": "samples/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup_train_ref,
            "ms_per_step": round(1e3 * sec, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"config5: DSM training step of the sda_unet.yml ScoreUNet on the host cores (oracle port, "
                                   f"torch autograd + torch.optim.AdamW), {b} samples of 52x128x128 per step",
                       "name": "config5", "batch_per_step": b},
            "cpu_baseline": {"value": round(value, 4), "unit": "samples/s", "cores": cores, "kind": "port",
                             "sample": f"{args.steps} timed steps of {b} samples each (the configured batch is 128 "
                                       "per GPU; cost is linear in the batch)"},
            "e2e": {"value": round(value, 4), "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "wall_s": round(time.perf_counter() - t_start, 1)}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=None, choices=[2, 3, 4],
                    help="BASELINE.json workload: 2 = 1 week on one GPU (default at N=1), 3 = 1 month time-sharded "
                         "(default at N>1), 4 = 16-member ensemble of a year as replicas")
    ap.add_argument("--weak", action="store_true", help="weak-scaling workload: L = 12 + 156 N frames")
    ap.add_argument("--frames", type=int, default=None, help="override the trajectory length L")
    ap.add_argument("--chunk", type=int, default=int(os.environ.get("C2W_CHUNK", 192)), help="windows per UNet launch")
    ap.add_argument("--e2e-steps", type=int, default=None,
                    help="denoising steps of the end-to-end sample() call (default: the real run's 256; 8 for config 4)")
    ap.add_argument("--cpu-windows", type=int, default=52, help="cpu_baseline sample of the GPU line")
    ap.add_argument("--cpu-windows-ref", type=int, default=0, help="reference arm: force this many windows per step")
    ap.add_argument("--ref-budget-s", type=float, default=420.0, help="reference arm: wall-time budget of the whole run")
    ap.add_argument("--exact-grad", action="store_true",
                    help="guidance through the UNet vector-Jacobian product (condition_on(exact_grad=True)); the shipped "
                         "experiment configs and the default bench line use the closed-form guidance")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-single", action="store_true", help="config 3: skip the one-GPU run of the same trajectory")
    ap.add_argument("--profile", action="store_true", help="short run for ncu: no warm-up floor, no roofline/e2e/cpu legs")
    ap.add_argument("--mode", default="sample", choices=["sample", "train"],
                    help="train: BASELINE config 5, the DSM training step (forward + backward + AdamW + EMA)")
    ap.add_argument("--batch", type=int, default=128, help="--mode train: samples per GPU (run_training.sh: 128)")
    ap.add_argument("--cpu-train-samples", type=int, default=2, help="--impl reference --mode train: samples per CPU step")
    ap.add_argument("--warmup-train-ref", type=int, default=1)
    ap.add_argument("--ddp", default="flat", choices=["flat", "torch"],
                    help="--mode train, N > 1: gradient averaging by one all-reduce of the flat buffer (default) or torch DDP")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, save the trajectory x and the score eps of the last step as "
                         "DIR/x.npy, DIR/eps.npy (float32, at most 64 MB together: every s-th frame of a longer "
                         "trajectory)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl, args.mode) != ("ours", "sample"):
        ap.error("--dump-outputs saves the sampling state of --impl ours --mode sample")
    if args.e2e_steps is None:
        args.e2e_steps = 8 if args.config == 4 else SAMPLER_STEPS
    if args.impl == "reference" and args.mode == "train":
        run_reference_train(args)
    elif args.impl == "reference":
        run_reference(args)
    elif args.mode == "train":
        if not args.profile:
            args.warmup = max(args.warmup, 3)
        run_train(args)
    else:
        if args.profile:
            args.no_e2e = args.no_cpu = args.no_single = True
        else:
            args.warmup = max(args.warmup, 3)
        run_ours(args)


if __name__ == "__main__":
    main()
