"""CPU tests (pytest -m "not gpu") of the host side: the C-ABI library loads and exports every symbol the header
declares (no compute calls), the time-shard plan partitions trajectories correctly, and the halo exchange /
frame gather work with world_size 2 over gloo.  The sharded-score equivalence is checked with the oracle's window
composition standing in for the UNet (src/thor/score.py:68-93 makes frame i depend on frames i-k..i+k only).
"""
import ctypes
import os
import re
import socket
import sys
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from climate2weather_b200 import _lib, sharding
from oracle import score_ref

ROOT = Path(__file__).resolve().parents[1]


# ------------------------------------------------------------------------------------------------ C ABI
def test_library_exports_every_header_symbol():
    """include/c2w_b200.h is the boundary: every function it declares must resolve in libc2w_b200.so, and the ctypes
    table must cover exactly that set."""
    text = (ROOT / "include" / "c2w_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    declared = set(re.findall(r"\b(c2w_[a-z0-9_]+)\s*\(", text))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.SIGNATURES), (declared ^ set(_lib.SIGNATURES))
    lib = _lib.load()  # raises C2WError if the library is missing, AttributeError if a symbol is
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.c2w_abi_version() >= 2
    # the ctypes mirrors of the header's structs have the layout the library was compiled with
    for which, mirror in enumerate((_lib.Config, _lib.Guide, _lib.AdamW, _lib.ConvDesc)):
        assert lib.c2w_struct_size(which) == ctypes.sizeof(mirror), mirror.__name__
    assert lib.c2w_struct_size(99) == -1


def test_no_cpu_path():
    """The product must fail loudly without a CUDA device (no CPU fallback)."""
    import climate2weather_b200 as c2w

    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    net = c2w.ScoreUNet(channels=20, embedding_dim=64, hidden_channels=(64,), hidden_blocks=(1,), attention_levels=(), activation=torch.nn.SiLU)
    with pytest.raises(_lib.C2WError):
        net(torch.zeros(1, 20, 16, 16), torch.tensor(0.5))
    sf = c2w.DefaultScoreFunction(net, markov_order=2, noise_process=c2w.SDAPipeline())
    with pytest.raises(_lib.C2WError):
        sf(torch.zeros(8, 4, 16, 16), torch.tensor(0.5))


def test_sampler_has_no_generic_torch_loop():
    """SDAPipeline.sample must not quietly run a torch-op loop for foreign score functions; with one of this package's
    score functions (proc_x0 hook or not) it needs the CUDA path and says so on a CPU box."""
    import climate2weather_b200 as c2w

    pipe = c2w.SDAPipeline()
    with pytest.raises(TypeError):
        pipe.sample(lambda x, t: x, torch.zeros(3, 4, 8, 8), steps=1)
    net = c2w.ScoreUNet(channels=20, embedding_dim=64, hidden_channels=(64,), hidden_blocks=(1,), attention_levels=(), activation=torch.nn.SiLU)
    sf = c2w.DefaultScoreFunction(net, markov_order=2, noise_process=pipe)
    if not torch.cuda.is_available():
        with pytest.raises(_lib.C2WError):
            pipe.sample(sf, torch.zeros(8, 4, 16, 16), steps=1, proc_x0=lambda v: v)
    # the schedule is the reference's (src/thor/pipelines.py:13-20): mu(0) = 1, sigma(0) = eta, mu(1) = eta
    t0, t1 = torch.tensor(0.0), torch.tensor(1.0)
    assert abs(float(pipe.mu(t0)) - 1.0) < 1e-6 and abs(float(pipe.sigma(t0)) - 1e-3) < 1e-6
    assert abs(float(pipe.mu(t1)) - 1e-3) < 1e-6 and abs(float(pipe.sigma(t1)) - 1.0) < 1e-5


def test_package_never_imports_oracle():
    """oracle/ is test infrastructure: nothing under climate2weather_b200/ may import it."""
    for f in (ROOT / "climate2weather_b200").rglob("*.py"):
        src = f.read_text()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f


# ------------------------------------------------------------------------------------------------ snapshots
def test_reference_snapshot_unpickles_through_compat():
    """A network snapshot pickled by the REFERENCE's own classes (tests/golden/make_golden.py: util.EasyDict with the
    fp16 model.score.ScoreUNet, thor.pipelines.SDAPipeline, dataset_kwargs — training_loop.py:250-266) loads through
    compat.install() into this package's classes with every parameter intact (exp/downscaling.py:110-126)."""
    import pickle

    import climate2weather_b200 as c2w
    import climate2weather_b200.compat as compat

    compat.install()
    with open(ROOT / "tests" / "golden" / "snapshot_tiny.pkl", "rb") as f:
        snap = pickle.load(f)
    exp = np.load(ROOT / "tests" / "golden" / "snapshot_tiny_expect.npz")
    assert snap["dataset_kwargs"]["train"]["window"] == 3 and snap.dataset_kwargs.train.window == 3
    assert isinstance(snap["pipeline"], c2w.SDAPipeline) and snap["pipeline"].eta == 1e-3
    net = snap["ema"]
    assert isinstance(net, c2w.ScoreUNet)
    assert (net.channels, net.embedding_dim) == (12, 64)
    assert net.hidden_channels == [64, 64] and net.hidden_blocks == [1, 1] and net.attention_levels == [1]
    sd = net.state_dict()
    assert list(sd.keys()) == [str(k) for k in exp["names"]]
    for k, want in zip(exp["names"], exp["sums"]):
        assert sd[str(k)].dtype == torch.float16
        assert abs(sd[str(k)].double().sum().item() - want) <= 1e-9 + 1e-12 * abs(want)
    net.eval()  # the calls exp/downscaling.py makes on it before sampling
    # a natively constructed net with the same architecture has the same parameter names
    native = c2w.ScoreUNet(12, 64, hidden_channels=[64, 64], hidden_blocks=[1, 1], attention_levels=[1], activation=torch.nn.SiLU)
    assert sorted(native.state_dict().keys()) == sorted(sd.keys())


# ------------------------------------------------------------------------------------------------ shard plan
@pytest.mark.parametrize("L,k,world", [(168, 6, 1), (168, 6, 2), (720, 6, 8), (25, 6, 2), (30, 2, 4), (8760, 6, 8),
                                       (13, 6, 1), (181, 6, 7)])
def test_plan_partitions_windows_and_frames(L, k, world):
    plans = [sharding.make_plan(L, k, r, world) for r in range(world)]
    nw = L - 2 * k
    # windows: contiguous, disjoint, cover [0, nw), balanced to within one
    assert plans[0].win_lo == 0 and plans[-1].win_hi == nw
    for a, b in zip(plans, plans[1:]):
        assert a.win_hi == b.win_lo
    sizes = [p.win_hi - p.win_lo for p in plans]
    assert max(sizes) - min(sizes) <= 1
    # owned frames: contiguous, disjoint, cover [0, L)
    assert plans[0].own_lo == 0 and plans[-1].own_hi == L
    for a, b in zip(plans, plans[1:]):
        assert a.own_hi == b.own_lo
    for p in plans:
        # local frames = every frame any local window touches; owned frames lie inside with k halo frames
        assert p.frame_lo == p.win_lo and p.frame_hi == p.win_hi + 2 * k
        assert p.frame_lo <= p.own_lo and p.own_hi <= p.frame_hi
        if p.rank > 0:
            assert p.own_lo - p.frame_lo == k
        if p.rank < world - 1:
            assert p.frame_hi - p.own_hi == k
        # every owned frame's score source (fold index map) is a window of this rank
        fi = score_ref.fold_index(L, k, 1)[:, 0, 0]
        src = fi[p.own_lo:p.own_hi]
        assert src.min() >= p.win_lo and src.max() < p.win_hi


def test_plan_rejects_too_many_ranks():
    with pytest.raises(ValueError):
        sharding.make_plan(12, 6, 0, 1)
    with pytest.raises(ValueError):
        sharding.make_plan(30, 6, 0, 8)


def _fake_net(u, t):
    """A window-local map with the UNet's signature: mixes every slot of a window into every output slot."""
    n, wc, H, W = u.shape
    return torch.tanh(u.flip(1) * 0.7 + u.mean(dim=1, keepdim=True) * (1.0 + t))


@pytest.mark.parametrize("L,k,world", [(40, 3, 2), (61, 6, 4), (25, 2, 3)])
def test_simulated_shards_reproduce_unsharded_score_bit_exact(L, k, world):
    """Each simulated rank evaluates only its windows on its local frames (with halos) and keeps its owned
    frames; the concatenation must equal the unsharded composition exactly (index work: bit-exact)."""
    C, H, W = 4, 4, 4
    x = torch.randn(L, C, H, W, generator=torch.Generator().manual_seed(L))
    t = torch.tensor(0.3)
    full = score_ref.window_score(_fake_net, x, t, k)
    nw = L - 2 * k
    parts = []
    for r in range(world):
        p = sharding.make_plan(L, k, r, world)
        u = score_ref.unfold(x[p.frame_lo:p.frame_hi], k)  # local windows == global windows [win_lo, win_hi)
        out = _fake_net(u, t)
        loc = torch.empty(p.own_n, C, H, W)
        for i in range(p.own_lo, p.own_hi):  # src/thor/score.py:76-88 on global indices
            if i < k:
                win, slot = 0, i
            elif i < L - k:
                win, slot = i - k, k
            else:
                win, slot = nw - 1, i - (L - 2 * k - 1)
            loc[i - p.own_lo] = out[win - p.win_lo, slot * C:(slot + 1) * C]
        parts.append(loc)
    assert torch.equal(torch.cat(parts), full)


# ------------------------------------------------------------------------------------------------ gloo, world 2
def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank: int, world: int, port: int, L: int, k: int, out_dir: str):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.manual_seed(0)
        shape = (4, 3, 2)
        x = torch.randn(L, *shape)
        p = sharding.make_plan(L, k, rank, world)
        # local copy with POISONED halos: only owned frames are valid before the exchange
        loc = x[p.frame_lo:p.frame_hi].clone()
        lo, hi = p.own_lo - p.frame_lo, p.own_hi - p.frame_lo
        loc[:lo] = float("nan")
        loc[hi:] = float("nan")
        sharding.exchange_halos(loc, p)
        ok_halo = torch.equal(loc, x[p.frame_lo:p.frame_hi])
        # "update" the owned frames rank-locally, exchange again, gather
        loc[lo:hi] = loc[lo:hi] * 2 + 1
        sharding.exchange_halos(loc, p)
        ok_halo2 = torch.equal(loc, x[p.frame_lo:p.frame_hi] * 2 + 1)
        full = sharding.all_gather_frames(loc[lo:hi].contiguous(), p)
        ok_gather = torch.equal(full, x * 2 + 1)
        # gather on one rank only (the sampler's default): dst gets the trajectory, the others nothing
        for dst in (0, world - 1):
            one = sharding.gather_frames(loc[lo:hi].contiguous(), p, dst=dst)
            ok_gather = ok_gather and ((one is None) if rank != dst else torch.equal(one, x * 2 + 1))
        # the corrector's scalar: sum over ranks of owned-frame sums == global sum
        s = (loc[lo:hi].double() ** 2).sum().reshape(1)
        dist.all_reduce(s)
        ok_sum = abs(s.item() - ((x * 2 + 1).double() ** 2).sum().item()) < 1e-6 * s.item()
        # adjoint exchange: every rank accumulated a contribution on ALL its local frames (halos included); after the
        # exchange each owned frame holds the sum over the ranks whose local range covers it
        def contrib(r):
            q = sharding.make_plan(L, k, r, world)
            return q, torch.randn(q.n_local, *shape, generator=torch.Generator().manual_seed(100 + r))
        total = torch.zeros(L, *shape)
        for r in range(world):
            q, c = contrib(r)
            total[q.frame_lo:q.frame_hi] += c
        _, mine = contrib(rank)
        sharding.exchange_halos_adjoint(mine, p)
        ok_adj = torch.allclose(mine[lo:hi], total[p.own_lo:p.own_hi], rtol=0, atol=1e-6)
        Path(out_dir, f"ok{rank}").write_text(f"{int(ok_halo)}{int(ok_halo2)}{int(ok_gather)}{int(ok_sum)}{int(ok_adj)}")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("L,k", [(40, 6), (31, 3)])
def test_halo_exchange_and_gather_gloo_world2(tmp_path, L, k):
    world = 2
    port = _free_port()
    mp.spawn(_worker, args=(world, port, L, k, str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        assert (tmp_path / f"ok{r}").read_text() == "11111"


# ------------------------------------------------------------------------------------------------ tile planning
def test_conv_tile_width_is_wave_aware():
    """Host-only planning query of the C ABI (no device call): the N-tile width per UNet level for the 156 windows of
    a one-week trajectory on 148 SMs — 128-wide activation-reuse tiles wherever a wider tile would leave the last wave
    of the persistent grid mostly empty (DESIGN.md, K1)."""
    from climate2weather_b200 import _lib

    lib = _lib.load()
    pick = lambda cout, H, W, n=156, c3=1, stride=1, sms=148: lib.c2w_conv_tile_width(cout, c3, n, H, W, stride, sms)
    assert pick(128, 128, 128) == 128 and pick(128, 64, 64) == 128 and pick(64, 128, 128) == 64
    assert pick(256, 32, 32) == 128   # 9 waves of 256 -> 17 waves of 128 with activation reuse
    assert pick(384, 16, 16) == 128   # 5 waves of 192 -> 7 waves of 128
    assert pick(512, 8, 8) == 128     # 2 waves of 256 -> 3 waves of 128 (two-image tiles)
    assert pick(384, 32, 32, stride=2) == 192 and pick(256, 64, 64, stride=2) == 256   # strided heads: streamed loop
    # attention GEMMs (78 M tiles): qkv 4 waves of 256; proj 3 waves of 128 beat 2 of 256 (16.5 vs 19.6 us measured)
    assert pick(1536, 8, 8, c3=0) == 256 and pick(512, 8, 8, c3=0) == 128
    assert pick(384, 12, 12) == 192   # images the 16 x 8 blocks do not tile
    assert pick(512, 8, 8, n=1) == 256  # a single M tile: nothing to balance
    assert lib.c2w_conv_tile_width(100, 1, 4, 8, 8, 1, 148) < 0


# ------------------------------------------------------------------------------------------------ reference-class surface
@pytest.mark.parametrize("L,k,C", [(13, 6, 4), (14, 6, 4), (26, 6, 4), (40, 6, 4), (5, 2, 4), (9, 2, 3), (7, 1, 1)])
def test_unfold_fold_batch_noise_mirrors_are_the_reference_index_maps(L, k, C):
    """DefaultScoreFunction.unfold / fold and BatchedScoreFunction._batch_noise / _window_score's slot selection
    (src/thor/score.py:68-88, :111-154) against the REFERENCE's own outputs on index-coded tensors (index_maps.npz)."""
    import climate2weather_b200 as c2w
    from climate2weather_b200.score import _pick_slots

    g = np.load(ROOT / "tests" / "golden" / "index_maps.npz")
    net = c2w.ScoreUNet(channels=C * (2 * k + 1), embedding_dim=64, hidden_channels=(64,), hidden_blocks=(1,),
                        attention_levels=(), activation=torch.nn.SiLU)
    pipe = c2w.SDAPipeline()
    sf = c2w.DefaultScoreFunction(net, markov_order=k, noise_process=pipe)
    code = (torch.arange(L)[:, None, None, None] * 1000 + torch.arange(C)[None, :, None, None] * 10
            + torch.arange(2)[None, None, :, None] * 2 + torch.arange(2)[None, None, None, :]).float()
    u = sf.unfold(code)
    assert np.array_equal(u.numpy().astype(np.int64), g[f"unfold_{L}_{k}_{C}"])
    nw = L - 2 * k
    wcode = (torch.arange(nw)[:, None, None, None] * 1000 + torch.arange((2 * k + 1) * C)[None, :, None, None]
             ).float().expand(nw, (2 * k + 1) * C, 1, 1)
    assert np.array_equal(sf.fold(wcode).numpy().astype(np.int64), g[f"fold_{L}_{k}_{C}"])
    for bs in (1, 2, 3, 16):
        bf = c2w.BatchedScoreFunction(net, markov_order=k, noise_process=pipe, batch_size=bs, device=torch.device("cpu"))
        batches = bf._batch_noise(code)
        assert len(batches) == -(-nw // bs) and sum(b.shape[0] for b in batches) == nw
        # the batched compose with an identity network (slot selection only), as the reference's score_fn loops it
        rows = [_pick_slots(b, k, i == 0, i == len(batches) - 1) for i, b in enumerate(batches)]
        assert np.array_equal(torch.cat(rows).numpy().astype(np.int64), g[f"batched_{L}_{k}_{C}_{bs}"])


def test_member_seeds_follow_the_reference_rule():
    """util.set_random_seed (util.py:27-29): hash((seed, rank)) % 2**31; SURVEY.md §8(d) probes (0,0) and (0,1)."""
    sys.path.insert(0, str(ROOT))
    import bench

    assert bench.member_seed(0, 0) == 397586535 and bench.member_seed(0, 1) == 16979904


def test_bench_workload_selection():
    """bench.py: N = 1 -> BASELINE config 2 (L = 168); N > 1 -> config 3 (L = 720, strong scaling); --config 4 -> the
    16-member ensemble of a year as replicas."""
    sys.path.insert(0, str(ROOT))
    import bench

    class A:
        config, weak, frames = None, False, None
    assert bench.pick_workload(A, 1) == ("config2", 168, "weak", 0)
    for n in (2, 4, 8):
        assert bench.pick_workload(A, n) == ("config3", 720, "strong", 0)
    A.config = 4
    assert bench.pick_workload(A, 8) == ("config4", 8760, "weak", 2)
    A.config, A.weak = None, True
    assert bench.pick_workload(A, 4) == ("config2-weak", 12 + 4 * 156, "weak", 0)


def test_bench_dump_outputs_keep_every_frame_or_a_fixed_stride_within_64_mb(tmp_path):
    """bench.py --dump-outputs: x and eps of every frame when both files fit 64 MB together, headers included (122
    frames do, 123 do not), otherwise the same every-s-th frames of both for the smallest s that fits; only rank 0
    writes."""
    import types

    sys.path.insert(0, str(ROOT))
    import bench

    for L, stride in ((20, 1), (122, 1), (123, 2), (200, 2)):
        x = torch.arange(L * bench.FRAME_BYTES // 4, dtype=torch.float32).reshape(L, bench.C, bench.H, bench.W)
        rt = types.SimpleNamespace(x=x, eps=-x, plan=sharding.make_plan(L, bench.K_ORDER, 0, 1), owned=lambda buf: buf)
        st = types.SimpleNamespace(rt=rt, sf=types.SimpleNamespace(shard=None))
        bench.dump_outputs(str(tmp_path / "rank1"), st, rank=1)
        assert not (tmp_path / "rank1").exists()
        out = tmp_path / str(L)
        bench.dump_outputs(str(out), st, rank=0)
        got = {n: np.load(out / f"{n}.npy") for n in ("x", "eps")}
        assert sum((out / f"{n}.npy").stat().st_size for n in got) <= bench.DUMP_BYTES
        assert got["x"].dtype == np.float32 and np.array_equal(got["x"], x[::stride].numpy()), L
        assert np.array_equal(got["eps"], -got["x"])


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours): one JSON line with the same metric, unit,
    direction and workload part of `config` as our arm, `impl: reference`, a `cpu_baseline` describing the run, an `e2e`
    equal to the line's value with zero copies — and exactly the steps / warm-up it was asked for (a bounded 13-window
    step here so the test stays short)."""
    import json
    import subprocess

    sys.path.insert(0, str(ROOT))
    import bench
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-windows-ref", "13"], capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "guided-sampling frames/sec" and line["unit"] == "frames/s"
    assert line["higher_is_better"] is True and line["steps"] == 1 and line["warmup"] == 0 and line["n_gpus"] == 1
    ours = bench.workload_config("config2", 168, 1, 0, False)
    assert {k: line["config"][k] for k in ours} == ours
    assert line["config"]["windows_per_step"] == 13
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "13 of the 156 windows" in cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["value"] > 0 and line["ms_per_step"] > 0


def test_bench_reference_training_arm_times_exactly_the_steps_asked_for():
    """`bench.py --impl reference --mode train --steps K` times K steps, not fewer (one sample per step here)."""
    import json
    import subprocess

    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--mode", "train",
                        "--steps", "4", "--cpu-train-samples", "1", "--warmup-train-ref", "0"],
                       capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 4 and line["cpu_baseline"]["sample"].startswith("4 timed steps of 1 samples")


@pytest.mark.parametrize("L,k,t_step", [(13, 6, 6), (14, 6, 6), (25, 6, 6), (168, 6, 6), (40, 2, 3), (31, 3, 4), (720, 6, 6),
                                        (50, 6, 1), (50, 6, 7)])
def test_observed_window_selection_is_exactly_the_fold_preimage_of_the_observed_frames(L, k, t_step):
    """exact_grad runs the UNet backward only for `observed_windows`: that must be EXACTLY the set of windows the
    reference's fold (src/thor/score.py:76-88, oracle fold_index pinned against it) takes an observed frame
    (f % t_step == 0, exp/downscaling.py:131) from — a missing window would drop a non-zero cotangent — and the shards
    of a time-sharded run must partition it."""
    from climate2weather_b200.score import observed_windows
    from climate2weather_b200.sharding import make_plan
    from oracle import score_ref
    nw = L - 2 * k
    f = score_ref.fold_index(L, k, 4)  # [L, C, (window, window-channel)]
    want = sorted({int(f[fr, 0, 0]) for fr in range(L) if fr % t_step == 0})
    assert observed_windows(0, nw, nw, L, k, t_step) == want
    for world in (2, 3, 8):
        if nw // world < max(k, 1):  # make_plan refuses shards narrower than the halo
            continue
        got = []
        for r in range(world):
            p = make_plan(L, k, r, world)
            got += observed_windows(p.win_lo, p.win_hi, p.n_win_global, L, k, t_step)
        assert got == want, world


# ------------------------------------------------------------------------------------------------ CoarseGrain conditioning
def test_coarse_grain_observation_shape_is_checked():
    """A CoarseGrain passed as `A` is checked against y like a recognised operator: y must broadcast to A(x), which is
    [ceil(L / t), C, H / s, W / s].  Too few observed frames would make the guidance kernel read past y, too large
    tiles would make it read y at the wrong offsets; both raise ValueError naming the two shapes."""
    import re

    from climate2weather_b200 import score as sc
    L, C, H, W = 11, 4, 32, 32
    op = sc.CoarseGrain(3, 8)
    assert sc._recognise_operator(op, L, C, H, W, (4, 4, 4, 4)) is op
    for bad in ((2, 4, 4, 4), (4, 4, 8, 8), (4, 3, 4, 4)):
        with pytest.raises(ValueError, match=re.escape(f"{bad}") + ".*" + re.escape("(4, 4, 4, 4)")):
            sc._recognise_operator(op, L, C, H, W, bad)
        with pytest.raises(ValueError, match=re.escape(f"{bad}")):
            sc.coarse_grain_observation(op, torch.zeros(bad), L, C, H, W)
    # a y that broadcasts (one observation for every observed frame) is uploaded as the full, contiguous A(x) shape
    y1 = torch.randn(1, C, 4, 4)
    assert sc._recognise_operator(op, L, C, H, W, tuple(y1.shape)) is op
    y = sc.coarse_grain_observation(op, y1, L, C, H, W)
    assert y.shape == (4, C, 4, 4) and y.is_contiguous() and all(torch.equal(y[m], y1[0]) for m in range(4))
    y4 = torch.randn(4, C, 4, 4)
    assert torch.equal(sc.coarse_grain_observation(op, y4, L, C, H, W), y4)
    # an opaque operator of the same family, recognised from the shapes, gets the same checks
    A = lambda x: torch.nn.functional.avg_pool2d(x[..., ::3, :, :, :], 8, stride=8)
    got = sc._recognise_operator(A, L, C, H, W, (4, 4, 4, 4))
    assert (got.t_step, got.s_step) == (3, 8)


@pytest.mark.parametrize("t,s,what", [(6, 1, "at most 32"), (6, 2, "at most 32"), (6, 5, "must divide"),
                                      (0, 16, "at least 1"), (6, 0, "at least 1"), (-1, 16, "at least 1")])
def test_coarse_grain_limits_raise_at_set_up(t, s, what):
    """(t, s) the guidance kernel cannot run are refused when the operator is recognised, not at the first guided step:
    s must divide H and W, leave at most 32 tiles per row (s >= 4 at 128 x 128), and t, s must be at least 1.  The same
    holds for an opaque operator recognised as that family."""
    from climate2weather_b200 import score as sc
    L, C, H, W = 13, 4, 128, 128
    op = sc.CoarseGrain(t, s)
    shape = (-(-L // t) if t >= 1 else 1, C, H // s if s >= 1 else 1, W // s if s >= 1 else 1)
    with pytest.raises(NotImplementedError, match=what):
        sc._recognise_operator(op, L, C, H, W, shape)
    with pytest.raises(NotImplementedError, match=what):
        sc.coarse_grain_observation(op, torch.zeros(shape), L, C, H, W)
    if t >= 1 and s in (1, 2):
        A = lambda x: torch.nn.functional.avg_pool2d(x[..., ::t, :, :, :], s, stride=s)
        with pytest.raises(NotImplementedError, match=what):
            sc._recognise_operator(A, L, C, H, W, shape)
    for ok in (4, 8, 16, 32, 64, 128):
        assert sc._recognise_operator(sc.CoarseGrain(6, ok), L, C, H, W, (3, C, H // ok, W // ok)).s_step == ok
