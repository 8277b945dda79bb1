"""GPU tests (pytest -m gpu) of guided sampling with a noise std per observation (c2w_guided_step_obs_std: the
per-observation instances of K6, K6p and K6c): each kernel through the C ABI at C = 1..8 against float64 references
that take a var per observation, bit-exact agreement with the per-variable kernels for a constant std, infinite std
as an unobserved tile or station, the whole path against the oracle with the same std tensor, bitwise invariance, and
time sharding against the single-GPU run (2 / 4 devices).

Tolerances: 1e-5 of the reference's max-abs (eps_g, the correction eps_g - eps on its own, x, the cotangent); each
mode-1 partial within 1e-5 relative; the whole path at the point tests' tolerances."""
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
from test_gpu_combined_obs import GRIDS, launch, plan_tensors, point_operator, relerr_t
from test_gpu_frame_kernels import MU, SENTINEL, SIGMA, MU_N, SIGMA_N, f32, likelihood_params, randn, relerr
from test_gpu_point_obs import GAMMA, K, L, H, W, _net, _points, rel_l2

pytestmark = pytest.mark.gpu

KINDS = ("coarse", "points", "combined")


@pytest.fixture(scope="module")
def lib():
    from climate2weather_b200 import _lib
    return _lib.load()


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def stream():
    return torch.cuda.current_stream().cuda_stream


def obs_plan(dev, op, y, std, Lg, C, H_, W_, lo, hi, strip, max_pix):
    """plan_tensors with a std per observation: (c2w_point_obs, tensors with "std2", n_strips)."""
    from climate2weather_b200 import _lib, score as S
    pl = S.point_plan(op, torch.from_numpy(y), Lg, C, H_, W_, lo, hi, strip, max_pix, std=torch.from_numpy(std))
    t = {n: torch.as_tensor(pl[n]).to(dev) for n in ("frame_slot", "strip_off", "pix", "ysum", "wsum", "std2")}
    for n in ("pix", "ysum", "wsum", "std2"):
        if t[n].numel() == 0:
            t[n] = torch.zeros(max(1, C), dtype=t[n].dtype, device=dev)
    ob = _lib.PointObs()
    ob.frame_slot, ob.strip_off, ob.pix = (t[n].data_ptr() for n in ("frame_slot", "strip_off", "pix"))
    ob.ysum, ob.wsum = t["ysum"].data_ptr(), t["wsum"].data_ptr()
    ob.n_slots, ob.strip_rows = pl["n_slots"], pl["strip_rows"]
    return ob, t, pl["n_strips"]


def launch_obs(lib, dev, x, eps, mode, t_step, s, yc, cstd2, gamma, pts=None, frame0=0, own_lo=0, own_n=None, vjp=None):
    """One c2w_guided_step_obs_std: the coarse term when yc is given (cstd2 in y's layout), the point term when pts is
    (its tensors hold "std2").  Outputs start at SENTINEL; g.std2 is NaN throughout and gamma past C is NaN."""
    from climate2weather_b200 import _lib
    F, H_, W_, C = x.shape
    own_n = F - own_lo if own_n is None else own_n
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
    xd, ed = up(x), up(eps)
    eo, co = torch.full_like(xd, SENTINEL), torch.full_like(xd, SENTINEL)
    n_part = own_n * (pts[2] if pts is not None else H_ // s)
    parts = torch.full((n_part,), SENTINEL, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    yd = up(yc) if yc is not None else None
    sd = up(cstd2) if yc is not None else None
    vd = up(vjp) if vjp is not None else None
    g = _lib.Guide()
    g.x, g.eps, g.eps_out = xd.data_ptr(), ed.data_ptr(), eo.data_ptr()
    g.y = yd.data_ptr() if yd is not None else None
    for c in range(8):
        g.std2[c] = math.nan
        g.gamma[c] = float(gamma[c]) if c < C else math.nan
    g.mu, g.sigma, g.mu_next, g.sigma_next = MU, SIGMA, MU_N, SIGMA_N
    g.t_step, g.s_step, g.H, g.W = (t_step, s, H_, W_) if yc is not None else (1, 1, H_, W_)
    g.frame_global0, g.own_lo, g.own_n, g.mode = frame0, own_lo, own_n, mode
    g.partials, g.nan_flag, g.cot_out = parts.data_ptr(), flag.data_ptr(), co.data_ptr()
    g.vjp = vd.data_ptr() if vd is not None else None
    g.halo, g.halo_k, g.channels = None, 0, C
    obs = ctypes.byref(pts[0]) if pts is not None else None
    entry = pts[1]["std2"].data_ptr() if pts is not None else None
    _lib.check(lib.c2w_guided_step_obs_std(ctypes.byref(g), obs, sd.data_ptr() if sd is not None else None, entry,
                                           stream()), "c2w_guided_step_obs_std")
    torch.cuda.synchronize()
    return dict(x=xd.cpu().numpy(), eps_out=eo.cpu().numpy(), cot=co.cpu().numpy(), partials=parts.cpu().numpy(),
                flag=int(flag.item()))


def tile_g_ref(x, eps, yc, cstd2, gamma, mu, sigma, t_step, s, frame0=0):
    """A_c^T((y - A_c x0)/var) in float64 with var = std2[m, c, ty, tx] + gamma_c (sigma/mu)^2 per tile."""
    x0 = (x.astype(np.float64) - sigma * eps.astype(np.float64)) / mu
    F, H_, W_, C = x.shape
    g = np.zeros_like(x0)
    observed = np.zeros(F, bool)
    for f in range(F):
        fg = frame0 + f
        if fg % t_step:
            continue
        mean = x0[f].reshape(H_ // s, s, W_ // s, s, C).mean(axis=(1, 3))
        r = yc[fg // t_step].astype(np.float64).transpose(1, 2, 0) - mean
        var = cstd2[fg // t_step].astype(np.float64).transpose(1, 2, 0) + gamma * (sigma / mu) ** 2
        g[f] = np.repeat(np.repeat(r / var / (s * s), s, axis=0), s, axis=1)
        observed[f] = True
    return g, observed


def point_g_ref(op, y, std, x, eps, gamma, mu, sigma, frame0):
    """A_p^T((y - A_p x0)/var) in float64 with var = std[m, c, p]^2 (fp32 square) + gamma_c (sigma/mu)^2."""
    x0 = (x.astype(np.float64) - sigma * eps.astype(np.float64)) / mu
    s2 = (std.astype(np.float32) * std.astype(np.float32)).astype(np.float64)
    g = np.zeros_like(x0)
    mask = op.mask_for(x.shape[-1]).numpy()
    rows, cols = op.rows.numpy(), op.cols.numpy()
    for m, fgl in enumerate(op.frames.tolist()):
        f = fgl - frame0
        if not 0 <= f < x.shape[0]:
            continue
        for c in range(x.shape[-1]):
            for p in np.nonzero(mask[m, c])[0]:
                g[f, rows[p], cols[p], c] += (float(y[m, c, p]) - x0[f, rows[p], cols[p], c]) / (
                    s2[m, c, p] + gamma[c] * (sigma / mu) ** 2)
    return g


def station_std(rng, op, C, classes=(0.03, 0.05, 0.08)):
    """A std per station and variable from a few classes (so duplicated pixels form runs), NaN under the mask."""
    std = np.asarray(classes, np.float32)[rng.integers(0, len(classes), (op.n_frames, C, op.n_points))]
    return np.where(op.mask_for(C).numpy(), std, np.nan).astype(np.float32)


def problem(dev, rng, kind, C, H_, W_, s, Lg, t_step, frames, frame0, own_lo, own_n, nloc):
    from climate2weather_b200 import score as S
    x, eps, vjp = randn(rng, nloc, H_, W_, C), randn(rng, nloc, H_, W_, C), randn(rng, nloc, H_, W_, C)
    gamma = likelihood_params(C)[1]
    yc = cstd2 = pts = None
    g = np.zeros((nloc, H_, W_, C))
    if kind != "points":
        yc = randn(rng, -(-Lg // t_step), C, H_ // s, W_ // s)
        cstd = (0.05 + 0.3 * rng.random(yc.shape)).astype(np.float32)
        cstd2 = cstd * cstd
        gc, _ = tile_g_ref(x, eps, yc, cstd2, gamma, f32(MU), f32(SIGMA), t_step, s, frame0)
        g += gc
    if kind != "coarse":
        op, yp = point_operator(rng, frames, H_, W_, C)
        pstd = station_std(rng, op, C)
        if kind == "combined":
            R, max_pix = S.combined_strip_rows(H_, W_, s), S.COMBINED_STRIP_PIX
        else:
            R, max_pix = S.point_strip_rows(H_, W_), S.POINT_STRIP_PIX
        g0 = frame0 + own_lo
        pts = obs_plan(dev, op, yp, pstd, Lg, C, H_, W_, g0, g0 + own_n, R, max_pix)
        g += point_g_ref(op, yp, pstd, x, eps, gamma, f32(MU), f32(SIGMA), frame0)
    return dict(x=x, eps=eps, vjp=vjp, gamma=gamma, yc=yc, cstd2=cstd2, pts=pts, g=g)


def check_obs(lib, dev, rng, kind, C, H_, W_, s, Lg, t_step, frames, frame0=0, own_lo=0, own_n=None, nloc=None):
    """Modes 0 / 1 / 2, with and without vjp, against the float64 reference with a var per observation."""
    nloc = Lg if nloc is None else nloc
    own_n = nloc - own_lo if own_n is None else own_n
    P = problem(dev, rng, kind, C, H_, W_, s, Lg, t_step, frames, frame0, own_lo, own_n, nloc)
    x, eps, g = P["x"], P["eps"], P["g"]
    mu, sigma, mu_n, sigma_n = f32(MU), f32(SIGMA), f32(MU_N), f32(SIGMA_N)
    own = np.zeros(nloc, bool)
    own[own_lo:own_lo + own_n] = True
    untouched = g == 0
    where = dict(kind=kind, C=C, H=H_, W=W_, s=s, frame0=frame0, own=(own_lo, own_n))
    n_str, R = (P["pts"][2], P["pts"][0].strip_rows) if P["pts"] is not None else (H_ // s, s)
    kw = dict(pts=P["pts"], frame0=frame0, own_lo=own_lo, own_n=own_n)
    for v in (None, P["vjp"]):
        corr = (sigma / mu) * (g if v is None else g - sigma * v.astype(np.float64))
        eps_g = eps - corr
        x_new = mu_n * (x - sigma * eps_g) / mu + sigma_n * eps_g
        out = launch_obs(lib, dev, x, eps, 1, t_step, s, P["yc"], P["cstd2"], P["gamma"], vjp=v, **kw)
        assert relerr(out["eps_out"][own], eps_g[own]) < 1e-5, where
        # the correction on its own: besides 1e-5 of its scale, allow the fp32 rounding of eps_g itself (2^-23 |eps_g|),
        # which at s = 128 (g ~ 1/s^2) is of the order of the correction (as test_gpu_combined_obs.check_combined)
        got = out["eps_out"][own].astype(np.float64)
        err = np.abs((got - eps[own]) + corr[own])
        assert np.all(err <= 1e-5 * np.abs(corr[own]).max() + 2.0 ** -23 * np.abs(got)), where
        if v is None:
            sel = untouched & own[:, None, None, None]
            assert np.array_equal(out["eps_out"][sel], eps[sel]), where
        sq = np.square(eps_g[own])
        want_p = np.stack([sq[:, i * R:(i + 1) * R].reshape(own_n, -1).sum(1) for i in range(n_str)], 1).reshape(-1)
        assert np.all(np.abs(out["partials"] - want_p) <= 1e-5 * want_p), where
        assert np.array_equal(out["x"], x) and np.all(out["eps_out"][~own] == SENTINEL) and out["flag"] == 0, where
        out = launch_obs(lib, dev, x, eps, 0, t_step, s, P["yc"], P["cstd2"], P["gamma"], vjp=v, **kw)
        assert relerr(out["x"][own], x_new[own]) < 1e-5, where
        assert np.array_equal(out["x"][~own], x[~own]) and out["flag"] == 0, where
        out = launch_obs(lib, dev, x, eps, 2, t_step, s, P["yc"], P["cstd2"], P["gamma"], vjp=v, **kw)
        assert relerr(out["cot"][own], g[own]) < 1e-5, where
        assert np.all(out["cot"][untouched & own[:, None, None, None]] == 0.0), where
        assert np.all(out["cot"][~own] == SENTINEL), where


@pytest.mark.parametrize("H_,W_,s", GRIDS)
@pytest.mark.parametrize("C", range(1, 9))
@pytest.mark.parametrize("kind", KINDS)
def test_obs_std_kernel_vs_fp64(lib, dev, kind, C, H_, W_, s):
    rng = np.random.default_rng(5000 + 1000 * KINDS.index(kind) + 10 * C + s + H_)
    check_obs(lib, dev, rng, kind, C, H_, W_, s, 10, 3, (3, 4, 9))


@pytest.mark.parametrize("C", range(1, 9))
@pytest.mark.parametrize("kind", KINDS)
def test_obs_std_kernel_time_shard_slice_vs_fp64(lib, dev, kind, C):
    """Local frames = global [4, 16) of 20, owned local [2, 10)."""
    rng = np.random.default_rng(7000 + 100 * KINDS.index(kind) + C)
    check_obs(lib, dev, rng, kind, C, 128, 128, 16, 20, 3, (1, 7, 9, 13, 15), frame0=4, own_lo=2, own_n=8, nloc=12)


@pytest.mark.parametrize("C", [1, 3, 4, 8])
@pytest.mark.parametrize("kind", KINDS)
def test_constant_std_is_bit_identical_to_the_per_variable_kernel(lib, dev, kind, C):
    """A std per observation equal to the per-variable one: x, eps_g, cotangent and partials bit for bit equal to
    K6, K6p or K6c, modes 0 / 1 / 2, with and without vjp."""
    from climate2weather_b200 import score as S
    rng = np.random.default_rng(8000 + C)
    Lg, H_, W_, s, t = 10, 128, 128, 16, 3
    x, eps, vjp = randn(rng, Lg, H_, W_, C), randn(rng, Lg, H_, W_, C), randn(rng, Lg, H_, W_, C)
    std2c, gamma = likelihood_params(C)
    pstd = np.array([0.03 + 0.011 * c for c in range(C)], np.float32)
    std2p = (pstd * pstd).astype(np.float64)
    yc = randn(rng, -(-Lg // t), C, H_ // s, W_ // s) if kind != "points" else None
    cstd2 = np.broadcast_to(std2c.astype(np.float32).reshape(1, C, 1, 1), yc.shape) if yc is not None else None
    pts = pts_obs = None
    if kind != "coarse":
        op, yp = point_operator(rng, (0, 4, 9), H_, W_, C)
        R, mp_ = ((S.combined_strip_rows(H_, W_, s), S.COMBINED_STRIP_PIX) if kind == "combined"
                  else (S.point_strip_rows(H_, W_), S.POINT_STRIP_PIX))
        pts = plan_tensors(dev, op, yp, Lg, C, H_, W_, 0, Lg, R, mp_)
        full = np.broadcast_to(pstd.reshape(1, C, 1), (op.n_frames, C, op.n_points))
        pts_obs = obs_plan(dev, op, yp, np.ascontiguousarray(full), Lg, C, H_, W_, 0, Lg, R, mp_)
    name = {"coarse": "tile", "points": "points", "combined": "combined"}[kind]
    for v in (None, vjp):
        for mode in (0, 1, 2):
            a = launch(lib, dev, name, x, eps, mode, t, s, yc, std2c, gamma, pts=pts, std2p=std2p, vjp=v)
            b = launch_obs(lib, dev, x, eps, mode, t, s, yc, cstd2, gamma, pts=pts_obs, vjp=v)
            for k in ("x", "eps_out", "cot", "partials"):
                assert a[k].tobytes() == b[k].tobytes(), (kind, C, mode, v is None, k)


@pytest.mark.parametrize("C", [1, 4, 5])
def test_infinite_std_leaves_eps_unguided(lib, dev, C):
    """An infinite-std tile (coarse) or station (point entries): eps_g == eps there bit for bit, without vjp; an
    infinite-std station through the plan equals that station masked out."""
    import climate2weather_b200 as c2w
    from climate2weather_b200 import score as S
    rng = np.random.default_rng(9000 + C)
    Lg, H_, W_, s, t = 10, 64, 64, 16, 3
    x, eps = randn(rng, Lg, H_, W_, C), randn(rng, Lg, H_, W_, C)
    gamma = likelihood_params(C)[1]
    yc = randn(rng, -(-Lg // t), C, H_ // s, W_ // s)
    cstd2 = np.full(yc.shape, 0.01, np.float32)
    cstd2[1, :, 2, 3] = np.inf  # frame 3, tile (2, 3)
    out = launch_obs(lib, dev, x, eps, 1, t, s, yc, cstd2, gamma)
    tile = (3, slice(2 * s, 3 * s), slice(3 * s, 4 * s))
    assert np.array_equal(out["eps_out"][tile], eps[tile])
    assert not np.array_equal(out["eps_out"][3], eps[3])
    # stations: a pixel whose whole run has infinite std, at the kernel
    op, yp = point_operator(rng, (4, 5), H_, W_, C, P=60)
    pstd = station_std(rng, op, C)
    R = S.point_strip_rows(H_, W_)
    pts = obs_plan(dev, op, yp, pstd, Lg, C, H_, W_, 0, Lg, R, S.POINT_STRIP_PIX)
    pix = pts[1]["pix"].cpu().numpy()
    s2 = pts[1]["std2"].cpu()
    s2[pix == pix[0]] = float("inf")
    pts[1]["std2"].copy_(s2.to(dev))
    out = launch_obs(lib, dev, x, eps, 1, t, s, None, None, gamma, pts=pts)
    f0 = pts[1]["frame_slot"].cpu().tolist().index(0)  # entry 0 lies on the frame of slot 0
    r, cc = divmod(int(pix[0]), W_)
    assert np.array_equal(out["eps_out"][f0, r, cc], eps[f0, r, cc])
    assert not np.array_equal(out["eps_out"][f0], eps[f0])
    # through the plan: a station with std = inf is the station masked out, for every output
    stdi = np.where(np.isnan(pstd), np.nan, 0.05).astype(np.float32)
    stdi[:, :, 1] = np.where(op.mask_for(C).numpy()[:, :, 1], np.inf, np.nan)
    mask = op.mask_for(C).clone()
    mask[:, :, 1] = False
    masked = c2w.PointObservation(op.frames, op.rows, op.cols, mask)
    a = obs_plan(dev, op, yp, stdi, Lg, C, H_, W_, 0, Lg, R, S.POINT_STRIP_PIX)
    b = obs_plan(dev, masked, yp, stdi, Lg, C, H_, W_, 0, Lg, R, S.POINT_STRIP_PIX)
    for mode in (0, 1, 2):
        oa = launch_obs(lib, dev, x, eps, mode, t, s, None, None, gamma, pts=a)
        ob = launch_obs(lib, dev, x, eps, mode, t, s, None, None, gamma, pts=b)
        for k in ("x", "eps_out", "cot", "partials"):
            assert oa[k].tobytes() == ob[k].tobytes(), (mode, k)


def test_obs_std_argument_checks(lib, dev):
    """A term given by half, or none, is refused with a message; the mirrored checks keep their messages."""
    from climate2weather_b200 import _lib
    g = _lib.Guide()
    y = torch.zeros(4, device=dev)
    g.y = y.data_ptr()
    g.channels, g.own_n, g.H, g.W, g.s_step, g.t_step, g.mu = 4, 1, 32, 32, 8, 1, 1.0
    rc = lib.c2w_guided_step_obs_std(ctypes.byref(g), None, None, None, stream())
    assert rc != 0 and b"coarse term needs both" in lib.c2w_last_error()
    g.y = None
    rc = lib.c2w_guided_step_obs_std(ctypes.byref(g), None, None, None, stream())
    assert rc != 0 and b"no observation term" in lib.c2w_last_error()
    ob = _lib.PointObs()
    rc = lib.c2w_guided_step_obs_std(ctypes.byref(g), ctypes.byref(ob), None, None, stream())
    assert rc != 0 and b"point term needs both" in lib.c2w_last_error()
    rc = lib.c2w_guided_step_obs_std(ctypes.byref(g), ctypes.byref(ob), None, y.data_ptr(), stream())
    assert rc != 0 and b"c2w_guided_step_points: bad argument" in lib.c2w_last_error()
    g.y, g.s_step = y.data_ptr(), 5
    rc = lib.c2w_guided_step_obs_std(ctypes.byref(g), None, y.data_ptr(), None, stream())
    assert rc != 0 and b"s_step=5 must divide" in lib.c2w_last_error()


# ------------------------------------------------------------------------------------------------ whole path
def _std_for(kind, op, C, seed):
    """A std per observation the package and the oracle both take: per frame and tile (coarse), per station and
    variable (points), a flat per-observation tensor (combined)."""
    g = torch.Generator().manual_seed(seed)
    if kind == "coarse":
        cs = (-(-L // op.t_step), C, H // op.s_step, W // op.s_step)
        return 0.1 + 0.3 * torch.rand(cs[0], 1, cs[2], cs[3], generator=g)
    if kind == "points":
        return 0.05 + 0.2 * torch.rand(1, C, op.n_points, generator=g)
    cs, ps = op.term_shapes((L, C, H, W))
    return op.pack(0.1 + 0.3 * torch.rand(cs, generator=g), 0.05 + 0.2 * torch.rand(ps, generator=g), (L, C, H, W))


def _operator(kind, C, seed=7):
    """(op, y for the package, y for the oracle)."""
    import climate2weather_b200 as c2w
    pts, yp, yp0 = _points(C, seed=seed)
    if kind == "points":
        return pts, yp, yp0
    cg = c2w.CoarseGrain(3, 8)
    yc = torch.randn(-(-L // 3), C, H // 8, W // 8, generator=torch.Generator().manual_seed(seed + 100))
    if kind == "coarse":
        return cg, yc, yc
    op = c2w.CombinedObservation(cg, pts)
    return op, op.pack(yc, yp, (L, C, H, W)), op.pack(yc, yp0, (L, C, H, W))


@pytest.mark.parametrize("C", [4, 3])
@pytest.mark.parametrize("kind", KINDS)
def test_obs_std_guided_path_vs_oracle(kind, C):
    """The whole path against the fp32 oracle with the same operator, y and std tensor: closed-form guided score, a
    3-step predictor-corrector run with the reference's noise draws, exact_grad with one stashing chunk and with
    several — the tolerances of test_point_guided_path_vs_oracle."""
    import climate2weather_b200 as c2w
    net, ref = _net(C, seed=41 + C)
    op, y, y0 = _operator(kind, C)
    std = _std_for(kind, op, C, 70 + C)
    g = torch.Generator().manual_seed(80 + C)
    x = torch.randn(L, C, H, W, generator=g)
    t = torch.tensor(0.45)
    pipe = c2w.SDAPipeline()
    sf = c2w.BatchedScoreFunction(net, markov_order=K, noise_process=pipe, batch_size=4, device="cuda:0")
    sf.condition_on(A=op, y=y, std=std, gamma=GAMMA, exact_grad=False)
    assert sf.runtime(x.cuda()).cond.get("obs_std") is not None  # the per-observation kernels run
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
    print(f"\n{kind} C={C}: guided {eg:.3e}, sampler max-abs ratio {es:.3e} rel-L2 {ls:.3e}, exact {ee} "
          f"(closed vs exact {d:.3e})")
    assert got_s.shape == x.shape and es < 5e-2 and ls < 3e-2
    for e in ee:
        assert e < 4e-2 and e < 0.5 * d, (ee, d)


@pytest.mark.parametrize("kind", KINDS)
def test_obs_std_guidance_is_bitwise_invariant(kind):
    """Bit-identical across windows per launch and across repeated runs (no atomics on data)."""
    import climate2weather_b200 as c2w
    net, _ = _net(4)
    op, y, _ = _operator(kind, 4)
    std = _std_for(kind, op, 4, 3)
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
    """test_gpu_combined_obs's sharding problem with a std per observation in both terms."""
    from test_gpu_combined_obs import _problem as combined_problem
    net, noise, op, y, _ = combined_problem(Ls)
    cs, ps = op.term_shapes(noise.shape)
    g = torch.Generator().manual_seed(13)
    std = op.pack(0.1 + 0.2 * torch.rand(cs, generator=g), 0.03 + 0.1 * torch.rand(ps, generator=g), noise.shape)
    return net, noise, op, y, std


def _sample(net, noise, op, y, std, dev, corrections, shard, exact=False):
    from test_gpu_combined_obs import _sample as combined_sample
    return combined_sample(net, noise, op, y, std, dev, corrections, shard, exact)


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
def test_time_sharded_obs_std_sampling_matches_single_gpu(tmp_path, world):
    """Each rank uploads the coarse std^2 block and plans its own stations with their std: bit-exact for predictor
    steps over both halo transports, 1e-5 with a correction, 1e-4 with exact_grad."""
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
