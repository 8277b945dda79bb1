"""GPU tests (pytest -m gpu) of guided sampling on a coarse field and point observations together (CombinedObservation,
c2w_guided_step_combined, K6c): the kernel through the C ABI at C = 1..8 against a float64 reference in this file,
bit-exact additivity against the coarse-only (K6) and point-only (K6p) kernels, the whole path against the oracle
(reference log_p + autograd through the same operator, flat y and flat std), bitwise invariance, and time sharding
against the single-GPU run (2 / 4 devices)."""
import ctypes
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle_op
from oracle import pipeline_ref
from test_gpu_frame_kernels import MU, SENTINEL, SIGMA, MU_N, SIGMA_N, f32, guide_ref, likelihood_params, randn, relerr
from test_gpu_point_obs import GAMMA, K, L, H, W, _net, rel_l2

pytestmark = pytest.mark.gpu

# (H, W, s): several tile rows per strip and up to 64 tiles per CTA; one 32 x 32 tile per strip; a ragged last strip
# (R = 21 of 48 rows); the shipped strip (R = 16); a map beyond 2048 pixels (R = 64); two that need more than 48 KB of
# dynamic shared memory: a 64 KB map (R = 128) and, at s = 1, 2048 one-pixel tiles (up to 64 KB of tile cotangents)
GRIDS = [(32, 32, 4), (32, 32, 8), (32, 32, 32), (48, 96, 3), (128, 128, 16), (128, 128, 64), (128, 128, 128),
         (64, 32, 1)]


@pytest.fixture(scope="module")
def lib():
    from climate2weather_b200 import _lib
    return _lib.load()


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def stream():
    return torch.cuda.current_stream().cuda_stream


def point_std2(C):
    return (np.array([0.03 + 0.011 * c for c in range(C)]) ** 2).astype(np.float32).astype(np.float64)


def point_operator(rng, frames, H, W, C, P=300, all_masked=False):
    """Stations at random pixels plus strip borders and a duplicated pixel; a random mask (or none set)."""
    import climate2weather_b200 as c2w
    rows, cols = rng.integers(0, H, P), rng.integers(0, W, P)
    rows[:4], cols[:4] = [0, H - 1, 5, 5], [0, W - 1, 7, 7]
    mask = np.zeros((len(frames), C, P), bool) if all_masked else rng.random((len(frames), C, P)) > 0.3
    op = c2w.PointObservation(list(frames), torch.from_numpy(rows), torch.from_numpy(cols), torch.from_numpy(mask))
    y = randn(rng, len(frames), C, P)
    return op, np.where(mask, y, np.nan).astype(np.float32)


def point_g_ref(op, y, x, eps, std2p, gamma, mu, sigma, frame0):
    """A_p^T((y - A_p x0)/var_p) in float64 on local frames of x [frames, H, W, C]."""
    x0 = (x.astype(np.float64) - sigma * eps.astype(np.float64)) / mu
    var = std2p + gamma * (sigma / mu) ** 2
    g = np.zeros_like(x0)
    mask = op.mask_for(x.shape[-1]).numpy()
    rows, cols = op.rows.numpy(), op.cols.numpy()
    for m, fgl in enumerate(op.frames.tolist()):
        f = fgl - frame0
        if not 0 <= f < x.shape[0]:
            continue
        for p in range(op.n_points):
            for c in range(x.shape[-1]):
                if mask[m, c, p]:
                    g[f, rows[p], cols[p], c] += (float(y[m, c, p]) - x0[f, rows[p], cols[p], c]) / var[c]
    return g


def plan_tensors(dev, op, y, Lg, C, H, W, lo, hi, strip, max_pix):
    from climate2weather_b200 import _lib, score as S
    pl = S.point_plan(op, torch.from_numpy(y), Lg, C, H, W, lo, hi, strip, max_pix)
    t = {n: torch.as_tensor(pl[n]).to(dev) for n in ("frame_slot", "strip_off", "pix", "ysum", "wsum")}
    for n in ("pix", "ysum", "wsum"):
        if t[n].numel() == 0:
            t[n] = torch.zeros(max(1, C), dtype=t[n].dtype, device=dev)
    ob = _lib.PointObs()
    ob.frame_slot, ob.strip_off, ob.pix = (t[n].data_ptr() for n in ("frame_slot", "strip_off", "pix"))
    ob.ysum, ob.wsum = t["ysum"].data_ptr(), t["wsum"].data_ptr()
    ob.n_slots, ob.strip_rows = pl["n_slots"], pl["strip_rows"]
    return ob, t, pl["n_strips"]


def launch(lib, dev, kind, x, eps, mode, t_step, s, yc, std2c, gamma, pts=None, std2p=None, frame0=0, own_lo=0,
           own_n=None, vjp=None):
    """One guidance launch: kind 'tile' (c2w_guided_step), 'points' (c2w_guided_step_points, std2 = std2p) or
    'combined'.  pts = (c2w_point_obs, tensors, n_strips).  Outputs start at SENTINEL; std2 / gamma past C are NaN."""
    from climate2weather_b200 import _lib
    F, H, W, C = x.shape
    own_n = F - own_lo if own_n is None else own_n
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
    xd, ed = up(x), up(eps)
    eo, co = torch.full_like(xd, SENTINEL), torch.full_like(xd, SENTINEL)
    n_part = own_n * (H // s if kind == "tile" else pts[2])
    parts = torch.full((n_part,), SENTINEL, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    yd = up(yc) if kind != "points" else None
    vd = up(vjp) if vjp is not None else None
    g = _lib.Guide()
    g.x, g.eps, g.eps_out = xd.data_ptr(), ed.data_ptr(), eo.data_ptr()
    g.y = yd.data_ptr() if yd is not None else None
    s2 = std2p if kind == "points" else std2c
    for c in range(8):
        g.std2[c] = float(s2[c]) if c < C else math.nan
        g.gamma[c] = float(gamma[c]) if c < C else math.nan
    g.mu, g.sigma, g.mu_next, g.sigma_next = MU, SIGMA, MU_N, SIGMA_N
    g.t_step, g.s_step, g.H, g.W = t_step, s, H, W
    g.frame_global0, g.own_lo, g.own_n, g.mode = frame0, own_lo, own_n, mode
    g.partials, g.nan_flag, g.cot_out = parts.data_ptr(), flag.data_ptr(), co.data_ptr()
    g.vjp = vd.data_ptr() if vd is not None else None
    g.halo, g.halo_k, g.channels = None, 0, C
    if kind == "tile":
        _lib.check(lib.c2w_guided_step(ctypes.byref(g), stream()), "c2w_guided_step")
    elif kind == "points":
        _lib.check(lib.c2w_guided_step_points(ctypes.byref(g), ctypes.byref(pts[0]), stream()), "points")
    else:
        ps = (ctypes.c_float * 8)(*[float(std2p[c]) if c < C else math.nan for c in range(8)])
        _lib.check(lib.c2w_guided_step_combined(ctypes.byref(g), ctypes.byref(pts[0]), ps, stream()), "combined")
    torch.cuda.synchronize()
    return dict(x=xd.cpu().numpy(), eps_out=eo.cpu().numpy(), cot=co.cpu().numpy(), partials=parts.cpu().numpy(),
                flag=int(flag.item()))


def check_combined(lib, dev, rng, C, H, W, s, Lg, t_step, frames, frame0=0, own_lo=0, own_n=None, nloc=None):
    """Modes 0 / 1 / 2, with and without vjp, against the float64 sum of the coarse and point references."""
    from climate2weather_b200 import score as S
    nloc = Lg if nloc is None else nloc
    own_n = nloc - own_lo if own_n is None else own_n
    x, eps, vjp = randn(rng, nloc, H, W, C), randn(rng, nloc, H, W, C), randn(rng, nloc, H, W, C)
    yc = randn(rng, -(-Lg // t_step), C, H // s, W // s)
    std2c, gamma = likelihood_params(C)
    std2p = point_std2(C)
    op, yp = point_operator(rng, frames, H, W, C)
    R = S.combined_strip_rows(H, W, s)
    g0 = frame0 + own_lo
    pts = plan_tensors(dev, op, yp, Lg, C, H, W, g0, g0 + own_n, R, S.COMBINED_STRIP_PIX)
    own = np.zeros(nloc, bool)
    own[own_lo:own_lo + own_n] = True
    mu, sigma, mu_n, sigma_n = f32(MU), f32(SIGMA), f32(MU_N), f32(SIGMA_N)
    base = guide_ref(x, eps, yc, std2c, gamma, mu, sigma, mu_n, sigma_n, t_step, s, frame0)
    gp = point_g_ref(op, yp, x, eps, std2p, gamma, mu, sigma, frame0)
    g = base["g"] + gp
    untouched = (g == 0)
    # each term on the frames only it observes, against its own scale: the point term (std ~ 0.03) dominates the
    # max-abs of the sum, so an error in the coarse term would hide behind it in the checks on the sum
    has_pts = np.array([bool(np.any(gp[f])) for f in range(nloc)])
    alone = [(own & base["observed"] & ~has_pts, base["g"]), (own & ~base["observed"] & has_pts, gp)]
    where = dict(C=C, H=H, W=W, s=s, t=t_step, frame0=frame0, own=(own_lo, own_n))
    for v in (None, vjp):
        corr = (sigma / mu) * (g if v is None else g - sigma * v.astype(np.float64))
        eps_g = eps - corr
        x_new = mu_n * (x - sigma * eps_g) / mu + sigma_n * eps_g
        kw = dict(pts=pts, std2p=std2p, frame0=frame0, own_lo=own_lo, own_n=own_n, vjp=v)
        out = launch(lib, dev, "combined", x, eps, 1, t_step, s, yc, std2c, gamma, **kw)
        assert relerr(out["eps_out"][own], eps_g[own]) < 1e-5, where
        assert relerr(out["eps_out"][own].astype(np.float64) - eps[own], -corr[own]) < 1e-5, where
        for sel, term in alone if v is None else ():  # with vjp, its term sets the scale instead
            if sel.any():
                # eps_g is stored in fp32: besides 1e-5 of the term's scale, allow the rounding of eps_g itself
                # (2^-23 |eps_g|), which at s = 128 (g ~ 1/s^2) is of the order of the correction
                got = out["eps_out"][sel].astype(np.float64)
                err = np.abs((got - eps[sel]) + (sigma / mu) * term[sel])
                assert np.all(err <= 1e-5 * np.abs((sigma / mu) * term[sel]).max() + 2.0 ** -23 * np.abs(got)), where
        if v is None:  # no observation of either term: eps_g == eps bit for bit
            sel = untouched & own[:, None, None, None]
            assert np.array_equal(out["eps_out"][sel], eps[sel]), where
        n_str = -(-H // R)
        sq = np.square(eps_g[own])
        want_p = np.stack([sq[:, i * R:(i + 1) * R].reshape(own_n, -1).sum(1) for i in range(n_str)], 1).reshape(-1)
        assert np.all(np.abs(out["partials"] - want_p) <= 1e-5 * want_p), where
        assert np.array_equal(out["x"], x) and np.all(out["eps_out"][~own] == SENTINEL) and out["flag"] == 0, where
        out = launch(lib, dev, "combined", x, eps, 0, t_step, s, yc, std2c, gamma, **kw)
        assert relerr(out["x"][own], x_new[own]) < 1e-5, where
        assert np.array_equal(out["x"][~own], x[~own]) and out["flag"] == 0, where
        out = launch(lib, dev, "combined", x, eps, 2, t_step, s, yc, std2c, gamma, **kw)
        assert relerr(out["cot"][own], g[own]) < 1e-5, where
        for sel, term in alone:
            if sel.any():
                assert relerr(out["cot"][sel], term[sel]) < 1e-5, where
        assert np.all(out["cot"][untouched & own[:, None, None, None]] == 0.0), where
        assert np.all(out["cot"][~own] == SENTINEL), where
    return base["observed"], gp


@pytest.mark.parametrize("H,W,s", GRIDS)
@pytest.mark.parametrize("C", range(1, 9))
def test_combined_kernel_vs_fp64(lib, dev, C, H, W, s):
    """L = 10, t_step = 3 (coarse frames 0, 3, 6, 9), stations on frames 3, 4, 9: frames observed by both terms (3, 9),
    by the coarse term only (0, 6), by the stations only (4) and by none."""
    rng = np.random.default_rng(1000 * C + s + H)
    observed, gp = check_combined(lib, dev, rng, C, H, W, s, 10, 3, (3, 4, 9))  # coarse alone: 0, 6; points alone: 4
    assert observed.tolist() == [f % 3 == 0 for f in range(10)]
    assert [bool(np.any(gp[f])) for f in range(10)] == [f in (3, 4, 9) for f in range(10)]


@pytest.mark.parametrize("H,W,s", [(48, 96, 3), (128, 128, 16), (128, 128, 64)])
@pytest.mark.parametrize("C", range(1, 9))
def test_combined_kernel_time_shard_slice_vs_fp64(lib, dev, C, H, W, s):
    """Local frames = global [4, 16) of 20, owned local [2, 10): coarse rows and station frames follow the global
    index; stations outside the owned frames are not in this rank's plan."""
    rng = np.random.default_rng(2000 + 10 * C + s)
    check_combined(lib, dev, rng, C, H, W, s, 20, 3, (1, 7, 9, 13, 15), frame0=4, own_lo=2, own_n=8, nloc=12)


@pytest.mark.parametrize("C", [1, 3, 4, 8])
def test_combined_is_the_sum_of_the_single_term_kernels(lib, dev, C):
    """Mode 2: the combined cotangent equals, bit for bit, the fp32 sum of the coarse-only (K6) and point-only (K6p)
    cotangents.  With the point mask all false, x after a predictor step and eps_g equal the coarse-only run bit for
    bit."""
    from climate2weather_b200 import score as S
    rng = np.random.default_rng(3000 + C)
    Lg, H, W, s, t = 10, 128, 128, 16, 3
    x, eps = randn(rng, Lg, H, W, C), randn(rng, Lg, H, W, C)
    yc = randn(rng, -(-Lg // t), C, H // s, W // s)
    std2c, gamma = likelihood_params(C)
    std2p = point_std2(C)
    op, yp = point_operator(rng, (0, 4, 9), H, W, C)
    R = S.combined_strip_rows(H, W, s)
    comb = plan_tensors(dev, op, yp, Lg, C, H, W, 0, Lg, R, S.COMBINED_STRIP_PIX)
    alone = plan_tensors(dev, op, yp, Lg, C, H, W, 0, Lg, S.point_strip_rows(H, W), S.POINT_STRIP_PIX)
    a = launch(lib, dev, "tile", x, eps, 2, t, s, yc, std2c, gamma)["cot"]
    b = launch(lib, dev, "points", x, eps, 2, t, s, None, std2c, gamma, pts=alone, std2p=std2p)["cot"]
    c = launch(lib, dev, "combined", x, eps, 2, t, s, yc, std2c, gamma, pts=comb, std2p=std2p)["cot"]
    assert np.array_equal(c, a + b)
    op0, yp0 = point_operator(rng, (0, 4, 9), H, W, C, all_masked=True)
    none = plan_tensors(dev, op0, yp0, Lg, C, H, W, 0, Lg, R, S.COMBINED_STRIP_PIX)
    for mode, key in ((0, "x"), (1, "eps_out")):
        want = launch(lib, dev, "tile", x, eps, mode, t, s, yc, std2c, gamma)[key]
        got = launch(lib, dev, "combined", x, eps, mode, t, s, yc, std2c, gamma, pts=none, std2p=std2p)[key]
        assert np.array_equal(got, want), mode


# ------------------------------------------------------------------------------------------------ whole path
def _combined(C, s=8, t=3, seed=7):
    """CoarseGrain(3, 8) with stations on irregular frames (masked, one fully masked point); the flat y (NaN under the
    mask), the same with zeros there (what the reference needs) and a flat std with a std per (term, variable)."""
    import climate2weather_b200 as c2w
    from test_gpu_point_obs import _points
    pts, yp, yp0 = _points(C, seed=seed)
    op = c2w.CombinedObservation(c2w.CoarseGrain(t, s), pts)
    g = torch.Generator().manual_seed(seed + 100)
    cs, _ = op.term_shapes((L, C, H, W))
    yc = torch.randn(cs, generator=g)
    std = op.pack([0.2 + 0.1 * c for c in range(C)], [0.05 + 0.03 * c for c in range(C)], (L, C, H, W))
    return op, op.pack(yc, yp, (L, C, H, W)), op.pack(yc, yp0, (L, C, H, W)), std


@pytest.mark.parametrize("C", [4, 3])
def test_combined_guided_path_vs_oracle(C):
    """The whole path against the fp32 oracle with the same operator object, flat y and flat std (reference log_p +
    autograd): closed-form guided score, a 3-step predictor-corrector run with the reference's noise draws, exact_grad
    with one stashing chunk and with several — the tolerances of test_point_guided_path_vs_oracle."""
    import climate2weather_b200 as c2w
    net, ref = _net(C, seed=31 + C)
    op, y, y0, std = _combined(C)
    g = torch.Generator().manual_seed(60 + C)
    x = torch.randn(L, C, H, W, generator=g)
    t = torch.tensor(0.45)
    pipe = c2w.SDAPipeline()
    sf = c2w.BatchedScoreFunction(net, markov_order=K, noise_process=pipe, batch_size=4, device="cuda:0")
    sf.condition_on(A=op, y=y, std=std, gamma=GAMMA, exact_grad=False)
    with torch.no_grad():
        want_g = oracle_op.guided_score_op(ref, x, t, K, y0, std, GAMMA, op, exact_grad=False)
    eg = relerr_t(sf(x, t), want_g)
    assert eg < 3e-2, eg
    ref_pipe = pipeline_ref.RefPipeline()
    score = lambda xx, tt: oracle_op.guided_score_op(ref, xx, tt, K, y0, std, GAMMA, op, exact_grad=False)
    torch.manual_seed(5)
    want_s = ref_pipe.sample(score, x, steps=3, corrections=1, tau=0.5)
    pipe.rng = "reference"
    torch.manual_seed(5)
    got_s = pipe.sample(sf, x, steps=3, corrections=1, tau=0.5, show_progressbar=False)
    es, ls = relerr_t(got_s, want_s), rel_l2(got_s, want_s)
    want_e = oracle_op.guided_score_op(ref, x, t, K, y0, std, GAMMA, op, exact_grad=True)
    d = relerr_t(want_g, want_e)
    ee = []
    for mw in (None, 2):
        sfe = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=c2w.SDAPipeline())
        sfe.max_windows = mw
        sfe.condition_on(A=op, y=y, std=std, gamma=GAMMA, exact_grad=True)
        ee.append(relerr_t(sfe(x.cuda(), t).cpu(), want_e))
    print(f"\nC={C}: guided {eg:.3e}, sampler max-abs ratio {es:.3e} rel-L2 {ls:.3e}, exact {ee} "
          f"(closed vs exact {d:.3e})")
    assert got_s.shape == x.shape and es < 5e-2 and ls < 3e-2
    for e in ee:
        assert e < 4e-2 and e < 0.5 * d, (ee, d)


def relerr_t(got, ref):
    got, ref = got.double().cpu(), ref.double().cpu()
    return ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


def test_combined_guidance_is_bitwise_invariant():
    """Bit-identical across windows per launch and across repeated runs (no atomics on data)."""
    import climate2weather_b200 as c2w
    net, _ = _net(4)
    op, y, _, std = _combined(4)
    x = torch.randn(L, 4, H, W, generator=torch.Generator().manual_seed(2))
    t = torch.tensor(0.3)
    outs, samples = [], []
    for mw in (None, 3, None):
        pipe = c2w.SDAPipeline()
        sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=pipe)
        sf.max_windows = mw
        sf.condition_on(A=op, y=y, std=std, gamma=GAMMA, exact_grad=False)
        outs.append(sf(x.cuda(), t).cpu())
        samples.append(pipe.sample(sf, x, steps=3, corrections=1, tau=0.5, show_progressbar=False, seed=9).cpu())
    for o in outs[1:]:
        assert torch.equal(o, outs[0])
    for s in samples[1:]:
        assert torch.equal(s, samples[0])
    assert torch.isfinite(samples[0]).all()


# ------------------------------------------------------------------------------------------------ time sharding
def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _problem(Ls):
    import climate2weather_b200 as c2w
    from test_gpu_point_obs import _problem as point_problem
    net, noise, pts, yp = point_problem(Ls)
    op = c2w.CombinedObservation(c2w.CoarseGrain(4, 8), pts)
    cs, _ = op.term_shapes(noise.shape)
    yc = torch.randn(cs, generator=torch.Generator().manual_seed(12))
    std = op.pack(0.2, 0.05, noise.shape)
    return net, noise, op, op.pack(yc, yp, noise.shape), std


def _sample(net, noise, op, y, std, dev, corrections, shard, exact=False):
    import climate2weather_b200 as c2w
    pipe = c2w.SDAPipeline()
    sf = c2w.BatchedScoreFunction(net.to(dev), markov_order=2, noise_process=pipe, batch_size=5, device=dev)
    sf.condition_on(A=op, y=y, std=std, gamma=1e-3, exact_grad=exact)
    if shard:
        sf.enable_time_sharding()
    return pipe.sample(sf, noise, steps=4, corrections=corrections, tau=0.5, show_progressbar=False, seed=77)


def _worker(rank, world, port, Ls, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        net, noise, op, y, std = _problem(Ls)
        for corr in (0, 1):
            out = _sample(net, noise, op, y, std, dev, corr, shard=True)
            if rank == 0:
                torch.save(out.cpu(), os.path.join(out_dir, f"sharded_c{corr}.pt"))
        out = _sample(net, noise, op, y, std, dev, 0, shard=True, exact=True)
        if rank == 0:
            torch.save(out.cpu(), os.path.join(out_dir, "sharded_exact.pt"))
        os.environ["C2W_HALO"] = "nccl"
        out = _sample(net, noise, op, y, std, dev, 0, shard=True)
        if rank == 0:
            torch.save(out.cpu(), os.path.join(out_dir, "sharded_c0_nccl.pt"))
        os.environ["C2W_HALO"] = "p2p"
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4])
def test_time_sharded_combined_sampling_matches_single_gpu(tmp_path, world):
    """Each rank splits y, uploads the coarse block and plans its own stations; bit-exact for predictor steps over both
    halo transports, 1e-5 with a correction, 1e-4 with exact_grad."""
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    Ls = 23
    net, noise, op, y, std = _problem(Ls)
    dev = torch.device("cuda:0")
    ref = {c: _sample(net, noise, op, y, std, dev, c, shard=False).cpu() for c in (0, 1)}
    mp.spawn(_worker, args=(world, _free_port(), Ls, str(tmp_path)), nprocs=world, join=True)
    got0 = torch.load(tmp_path / "sharded_c0.pt")
    got1 = torch.load(tmp_path / "sharded_c1.pt")
    assert torch.isfinite(got0).all() and torch.isfinite(got1).all()
    assert torch.equal(got0, ref[0]), float((got0 - ref[0]).abs().max())
    assert torch.equal(torch.load(tmp_path / "sharded_c0_nccl.pt"), ref[0])
    rel = ((got1 - ref[1]).abs().max() / ref[1].abs().max()).item()
    assert rel < 1e-5, rel
    want = _sample(net, noise, op, y, std, dev, 0, shard=False, exact=True).cpu()
    gote = torch.load(tmp_path / "sharded_exact.pt")
    rel = ((gote - want).abs().max() / want.abs().max()).item()
    assert rel < 1e-4, rel
    assert not torch.equal(want, ref[0])
