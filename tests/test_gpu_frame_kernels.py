"""The frame kernels that run after the UNet, at every variable count C = 1..8 they are instantiated for, against float64
references written in this file: K6 `c2w_guided_step` (modes 0, 1 and 2, closed-form and exact-gradient guidance), K7
`c2w_corrector_update_c` (with a given z and with its on-chip Philox4x32-10 noise) and `c2w_reduce_partials`.  Each
kernel is called through the C ABI on hand-built inputs.

Tolerances: fp32 elementwise arithmetic against fp64 -> 1e-5 of the reference's max-abs (the guidance correction
eps_g - eps on its own as well, so a wrong guidance term cannot hide behind eps); the corrector noise -> 1e-5 max(1, |z|);
the partial-sum reduction -> 1e-12 of sum |p| against math.fsum.  Ownership, unobserved frames and splits of a launch
are bit-exact.  The references are pinned on the CPU: K6's against torch.autograd of the log-likelihood, the Philox
one against the published Random123 known-answer vectors.
"""
import ctypes
import math

import numpy as np
import pytest
import torch

SENTINEL = 1234.5  # pre-fills every output buffer: a value no kernel computes here
MU, SIGMA, MU_N, SIGMA_N = 0.8, 0.6, 0.85, 0.52
# (H, W, s): the shipped case; 32 tiles per row (a 1024-thread CTA); one pixel per warp; H != W with s^2 < 32 and s not a
# power of two; one 32 x 32 tile per warp
GRIDS = [(128, 128, 16), (128, 128, 4), (32, 32, 1), (48, 96, 3), (128, 128, 32)]


@pytest.fixture(scope="module")
def lib():
    from climate2weather_b200 import _lib
    return _lib.load()


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def stream():
    return torch.cuda.current_stream().cuda_stream


def relerr(got, ref):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    return float(np.abs(got - ref).max() / max(np.abs(ref).max(), 1e-30))


def f32(v):
    return float(np.float32(v))


def likelihood_params(C):
    """std^2 and gamma per variable, all different from one another, as the fp32 values the kernel receives."""
    std = np.array([0.05 + 0.02 * c for c in range(C)])
    gamma = np.array([0.002 + 0.0013 * c for c in range(C)])
    return (std ** 2).astype(np.float32).astype(np.float64), gamma.astype(np.float32).astype(np.float64)


def randn(rng, *shape):
    return rng.standard_normal(shape).astype(np.float32)


# ------------------------------------------------------------------------------------------------ K6 reference
def guide_ref(x, eps, y, std2, gamma, mu, sigma, mu_n, sigma_n, t_step, s, frame0=0, vjp=None):
    """K6 in float64 for every local frame of x, eps, vjp ([frames, H, W, C]); local frame f is global frame0 + f, y is
    [ceil(L / t_step), C, H / s, W / s] or None.

      x0 = (x - sigma eps) / mu;  on observed frames r = y[m] - (s x s tile mean of x0),  var_c = std2_c + gamma_c (sigma/mu)^2
      g = r / var / s^2 on every pixel of the tile (zero on unobserved frames)
      eps_g = eps - (sigma/mu) (g - sigma vjp);  x' = mu' (x - sigma eps_g) / mu + sigma' eps_g"""
    x, eps = x.astype(np.float64), eps.astype(np.float64)
    F, H, W, C = x.shape
    x0 = (x - sigma * eps) / mu
    g = np.zeros_like(x)
    observed = np.zeros(F, dtype=bool)
    if y is not None:
        var = std2 + gamma * (sigma / mu) ** 2
        for f in range(F):
            fg = frame0 + f
            if fg % t_step:
                continue
            mean = x0[f].reshape(H // s, s, W // s, s, C).mean(axis=(1, 3))
            r = y[fg // t_step].astype(np.float64).transpose(1, 2, 0) - mean
            g[f] = np.repeat(np.repeat(r / var / (s * s), s, axis=0), s, axis=1)
            observed[f] = True
    corr = (sigma / mu) * (g if vjp is None else g - sigma * vjp.astype(np.float64))
    eps_g = eps - corr
    x_new = mu_n * (x - sigma * eps_g) / mu + sigma_n * eps_g
    return dict(g=g, corr=corr, eps_g=eps_g, x=x_new, observed=observed)


def c2w_guide(lib, dev, x, eps, y, mode, std2, gamma, t_step, s, frame0=0, own_lo=0, own_n=None, vjp=None,
              mu=MU, sigma=SIGMA, mu_n=MU_N, sigma_n=SIGMA_N):
    """One c2w_guided_step for any C on fp32 numpy inputs (x, eps, vjp: [frames, H, W, C]; y: [n_obs, C, Hs, Ws] or
    None).  eps_out, cot_out and the partials start as SENTINEL; std2 / gamma beyond C are NaN, so a kernel reading a
    variable that does not exist shows.  Returns the numpy outputs and the NaN flag."""
    from climate2weather_b200 import _lib
    F, H, W, C = x.shape
    own_n = F - own_lo if own_n is None else own_n
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
    xd, ed = up(x), up(eps)
    eo, co = torch.full_like(xd, SENTINEL), torch.full_like(xd, SENTINEL)
    parts = torch.full((own_n * (H // s),), SENTINEL, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    yd = up(y) if y is not None else None
    vd = up(vjp) if vjp is not None else None
    g = _lib.Guide()
    g.x, g.eps, g.eps_out = xd.data_ptr(), ed.data_ptr(), eo.data_ptr()
    g.y = yd.data_ptr() if yd is not None else None
    for c in range(8):
        g.std2[c] = float(std2[c]) if c < C else math.nan
        g.gamma[c] = float(gamma[c]) if c < C else math.nan
    g.mu, g.sigma, g.mu_next, g.sigma_next = mu, sigma, mu_n, sigma_n
    g.t_step, g.s_step, g.H, g.W = t_step, s, H, W
    g.frame_global0, g.own_lo, g.own_n, g.mode = frame0, own_lo, own_n, mode
    g.partials, g.nan_flag, g.cot_out = parts.data_ptr(), flag.data_ptr(), co.data_ptr()
    g.vjp = vd.data_ptr() if vd is not None else None
    g.halo, g.halo_k, g.channels = None, 0, C
    _lib.check(lib.c2w_guided_step(ctypes.byref(g), stream()), "c2w_guided_step")
    torch.cuda.synchronize()
    return dict(x=xd.cpu().numpy(), eps_out=eo.cpu().numpy(), cot=co.cpu().numpy(), partials=parts.cpu().numpy(),
                flag=int(flag.item()))


def check_guide(lib, dev, x, eps, y, std2, gamma, t_step, s, frame0=0, own_lo=0, own_n=None, vjp=None):
    """Modes 0, 1 and (with y) 2 of one input set against guide_ref: values on the owned frames, untouched buffers on the
    others, eps_g == eps on unobserved frames without vjp, every mode-1 partial, no NaN flag."""
    F, H, W, C = x.shape
    own_n = F - own_lo if own_n is None else own_n
    own = np.zeros(F, dtype=bool)
    own[own_lo:own_lo + own_n] = True
    p = (f32(MU), f32(SIGMA), f32(MU_N), f32(SIGMA_N))
    ref = guide_ref(x, eps, y, std2, gamma, *p, t_step, s, frame0, vjp)
    where = dict(C=C, H=H, W=W, s=s, t_step=t_step, vjp=vjp is not None, frame0=frame0, own=(own_lo, own_n))
    kw = dict(frame0=frame0, own_lo=own_lo, own_n=own_n, vjp=vjp)

    out = c2w_guide(lib, dev, x, eps, y, 1, std2, gamma, t_step, s, **kw)
    got = out["eps_out"][own]
    assert relerr(got, ref["eps_g"][own]) < 1e-5, where
    if np.abs(ref["corr"][own]).max() > 0:
        assert relerr(got.astype(np.float64) - eps[own], -ref["corr"][own]) < 1e-5, where
    unobs = own & ~ref["observed"]
    if vjp is None:
        assert np.array_equal(out["eps_out"][unobs], eps[unobs]), where
    # one partial per (owned frame, strip of s rows): the CTA's sum of eps_g^2, at partials[own_idx * (H / s) + strip]
    want_p = np.square(ref["eps_g"][own]).reshape(own_n, H // s, s * W * C).sum(axis=2).reshape(-1)
    assert np.all(np.abs(out["partials"] - want_p) <= 1e-5 * want_p), where
    assert np.array_equal(out["x"], x) and np.all(out["cot"] == SENTINEL), where
    assert np.all(out["eps_out"][~own] == SENTINEL) and out["flag"] == 0, where

    out = c2w_guide(lib, dev, x, eps, y, 0, std2, gamma, t_step, s, **kw)
    assert relerr(out["x"][own], ref["x"][own]) < 1e-5, where
    assert np.array_equal(out["x"][~own], x[~own]), where
    assert np.all(out["eps_out"] == SENTINEL) and np.all(out["cot"] == SENTINEL) and out["flag"] == 0, where

    if y is not None:  # the likelihood cotangent g alone: vjp, if passed, is not read
        out = c2w_guide(lib, dev, x, eps, y, 2, std2, gamma, t_step, s, **kw)
        assert relerr(out["cot"][own], ref["g"][own]) < 1e-5, where
        assert np.all(out["cot"][unobs] == 0.0), where
        assert np.all(out["cot"][~own] == SENTINEL), where
        assert np.array_equal(out["x"], x) and np.all(out["eps_out"] == SENTINEL) and out["flag"] == 0, where
    return ref


def test_guide_reference_matches_autograd():
    """guide_ref against the reference's own formulation (src/thor/score.py:44-60): eps - sigma * d/dx of
    -1/2 sum (y - A x0)^2 / var by torch.autograd in fp64, eps held constant, per-variable std and gamma, ragged
    observations (L = 10, t_step = 3)."""
    rng = np.random.default_rng(0)
    L, H, W, C, t, s = 10, 12, 18, 5, 3, 3
    x, eps = randn(rng, L, H, W, C), randn(rng, L, H, W, C)
    y = randn(rng, -(-L // t), C, H // s, W // s)
    std2, gamma = likelihood_params(C)
    ref = guide_ref(x, eps, y, std2, gamma, MU, SIGMA, MU_N, SIGMA_N, t, s)
    xt = torch.from_numpy(x).double().permute(0, 3, 1, 2).requires_grad_(True)
    et = torch.from_numpy(eps).double().permute(0, 3, 1, 2)
    x0 = (xt - SIGMA * et) / MU
    var = torch.from_numpy(std2 + gamma * (SIGMA / MU) ** 2).reshape(1, C, 1, 1)
    err = torch.from_numpy(y).double() - torch.nn.functional.avg_pool2d(x0[::t], s, stride=s)
    (J,) = torch.autograd.grad(-(err ** 2 / var).sum() / 2, xt)
    want = (et - SIGMA * J).permute(0, 2, 3, 1).numpy()
    assert relerr(ref["eps_g"], want) < 1e-12
    assert relerr(ref["g"], MU * J.permute(0, 2, 3, 1).numpy()) < 1e-12
    assert ref["observed"].tolist() == [f % t == 0 for f in range(L)]


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,s", GRIDS)
@pytest.mark.parametrize("C", range(1, 9))
def test_guided_step_vs_fp64(lib, dev, C, H, W, s):
    """K6, modes 0 / 1 / 2 with and without vjp, for t_step = 1 (every frame observed), 3 with L = 10 (the last
    observation is ragged) and t_step > L (frame 0 alone)."""
    rng = np.random.default_rng(100 * C + s)
    L = 10
    x, eps, vjp = randn(rng, L, H, W, C), randn(rng, L, H, W, C), randn(rng, L, H, W, C)
    std2, gamma = likelihood_params(C)
    for t_step in (1, 3, L + 2):
        y = randn(rng, -(-L // t_step), C, H // s, W // s)
        for v in (None, vjp):
            ref = check_guide(lib, dev, x, eps, y, std2, gamma, t_step, s, vjp=v)
            assert ref["observed"].sum() == -(-L // t_step)


@pytest.mark.gpu
@pytest.mark.parametrize("C", range(1, 9))
def test_guided_step_unconditioned_vs_fp64(lib, dev, C):
    """y = NULL: eps_g = eps without vjp (bit for bit), eps + sigma^2/mu vjp with it, and the plain predictor; mode 2
    is refused."""
    from climate2weather_b200 import _lib
    rng = np.random.default_rng(200 + C)
    L, H, W, s = 6, 48, 96, 3
    x, eps, vjp = randn(rng, L, H, W, C), randn(rng, L, H, W, C), randn(rng, L, H, W, C)
    std2, gamma = likelihood_params(C)
    for v in (None, vjp):
        check_guide(lib, dev, x, eps, None, std2, gamma, 1, s, vjp=v)
    with pytest.raises(_lib.C2WError, match="mode 2"):
        c2w_guide(lib, dev, x, eps, None, 2, std2, gamma, 1, s)


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,s", [(48, 96, 3), (128, 128, 16)])
@pytest.mark.parametrize("C", range(1, 9))
def test_guided_step_time_shard_slice_vs_fp64(lib, dev, C, H, W, s):
    """A time-sharded rank's slice: local frames = global [4, 16) of a 20-frame trajectory, owned local [2, 10), t_step
    3 -> observed global frames 6, 9, 12 (none at local 0).  Observation rows follow the global index; the halo frames
    stay untouched in x, eps_out and cot_out."""
    rng = np.random.default_rng(300 + C + s)
    Lg, f0, nloc, t = 20, 4, 12, 3
    x, eps, vjp = randn(rng, nloc, H, W, C), randn(rng, nloc, H, W, C), randn(rng, nloc, H, W, C)
    y = randn(rng, -(-Lg // t), C, H // s, W // s)
    std2, gamma = likelihood_params(C)
    for v in (None, vjp):
        ref = check_guide(lib, dev, x, eps, y, std2, gamma, t, s, frame0=f0, own_lo=2, own_n=8, vjp=v)
        assert np.nonzero(ref["observed"])[0].tolist() == [2, 5, 8, 11]


@pytest.mark.gpu
@pytest.mark.parametrize("C", range(1, 9))
def test_guided_step_nan_flag(lib, dev, C):
    """Mode 0 raises the NaN flag for a non-finite value of the last variable of an owned frame (observed or not), and
    not for one in a frame it does not own."""
    rng = np.random.default_rng(400 + C)
    L, H, W, s, t = 7, 32, 32, 8, 3
    x, eps = randn(rng, L, H, W, C), randn(rng, L, H, W, C)
    y = randn(rng, -(-L // t), C, H // s, W // s)
    std2, gamma = likelihood_params(C)
    for f, bad, want in ((3, math.inf, 1), (4, math.nan, 1), (0, math.nan, 0), (6, math.inf, 0)):
        xb = x.copy()
        xb[f, 5, 17, C - 1] = bad
        out = c2w_guide(lib, dev, xb, eps, y, 0, std2, gamma, t, s, own_lo=1, own_n=5)
        assert out["flag"] == want, (f, bad)


# ------------------------------------------------------------------------------------------------ K7 reference
_M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Random123 Philox4x32-10 on numpy arrays: ctr = 4 words, key = 2 words (uint32 values, broadcast)."""
    c0, c1, c2, c3 = (np.asarray(v, dtype=np.uint64) for v in ctr)
    k0, k1 = (np.asarray(v, dtype=np.uint64) for v in key)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _M32
        k0 = (k0 + np.uint64(0x9E3779B9)) & _M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & _M32
    return tuple(np.asarray(v).astype(np.uint32) for v in (c0, c1, c2, c3))


def box_muller(a, b):
    """The kernel's uniforms (float(a) + 0.5f) 2^-32 reproduced in float32, then log / sqrt / sincos in float64."""
    u1 = (a.astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -32)
    u2 = (b.astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -32)
    r = np.sqrt(-2.0 * np.log(u1.astype(np.float64)))
    th = np.pi * (np.float32(2.0) * u2).astype(np.float64)
    return r * np.cos(th), r * np.sin(th)


def philox_normals(pix, step_id, seed, C):
    """z [npix, C] of global pixels `pix`: for the group b of variables 4b..4b+3, counter = (pixel lo, pixel hi,
    step_id, b), key = (seed lo, seed hi); normals (r cos, r sin) of words (0, 1), then of words (2, 3)."""
    g = np.asarray(pix, dtype=np.uint64)
    seed = np.uint64(seed)
    out = np.empty((g.size, C))
    for b in range((C + 3) // 4):
        r = philox4x32_10((g & _M32, g >> np.uint64(32), step_id, b), (seed & _M32, seed >> np.uint64(32)))
        n = box_muller(r[0], r[1]) + box_muller(r[2], r[3])
        for e in range(min(4, C - 4 * b)):
            out[:, 4 * b + e] = n[e]
    return out


def test_philox_reference_known_answers():
    """The numpy Philox4x32-10 against Random123's published known-answer vectors (kat_vectors: philox4x32 10)."""
    kat = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
           ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
           ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
            (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for ctr, key, want in kat:
        assert tuple(int(v) for v in philox4x32_10(ctr, key)) == want
    # vectorised over counters: each lane is the scalar result
    ctr = (np.array([0, 0xFFFFFFFF, 0x243F6A88], dtype=np.uint32), np.array([0, 0xFFFFFFFF, 0x85A308D3], dtype=np.uint32),
           np.array([0, 0xFFFFFFFF, 0x13198A2E], dtype=np.uint32), np.array([0, 0xFFFFFFFF, 0x03707344], dtype=np.uint32))
    key = (np.array([0, 0xFFFFFFFF, 0xA4093822], dtype=np.uint32), np.array([0, 0xFFFFFFFF, 0x299F31D0], dtype=np.uint32))
    got = philox4x32_10(ctr, key)
    assert [tuple(int(w[i]) for w in got) for i in range(3)] == [w for _, _, w in kat]
    # the largest word gives u = 1 exactly (r = 0), the smallest u = 2^-33 (r = sqrt(66 ln 2))
    c, _ = box_muller(np.array([0xFFFFFFFF, 0], dtype=np.uint32), np.array([0, 0], dtype=np.uint32))
    assert c[0] == 0.0 and abs(c[1] - math.sqrt(66 * math.log(2))) < 1e-12


def corrector(lib, dev, x, eps, z, sumsq, count, tau, sigma_n, pix0, seed, step_id, npix=None, C=None):
    """One c2w_corrector_update_c over the first npix pixels of the device tensors x / eps / z ([pixels, C]);
    sumsq: python float (uploaded as the double the kernel reads).  Returns the NaN flag."""
    from climate2weather_b200 import _lib
    C = x.shape[-1] if C is None else C
    npix = x.numel() // C if npix is None else npix
    sq = torch.tensor([sumsq], dtype=torch.float64, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    _lib.check(lib.c2w_corrector_update_c(x.data_ptr(), eps.data_ptr(), z.data_ptr() if z is not None else None,
                                          sq.data_ptr(), float(count), tau, sigma_n, pix0, npix, C, seed, step_id,
                                          flag.data_ptr(), stream()), "c2w_corrector_update_c")
    torch.cuda.synchronize()
    return int(flag.item())


@pytest.mark.gpu
@pytest.mark.parametrize("C", range(1, 9))
def test_corrector_given_z_vs_fp64(lib, dev, C):
    """x <- x - (delta eps + sqrt(2 delta) z) sigma', delta = tau / float(sumsq / count) as the kernel rounds it, the
    rest in fp64; the NaN flag for a non-finite last variable inside the launch's pixels, not for one past them."""
    rng = np.random.default_rng(500 + C)
    npix = 3 * 17 * 19
    x, eps, z = randn(rng, npix + 1, C), randn(rng, npix + 1, C), randn(rng, npix + 1, C)
    tau, sgn = 0.37, 0.61
    sumsq = float(np.square(eps[:npix].astype(np.float64)).sum())
    count = npix * C
    delta = float(np.float32(tau) / np.float32(sumsq / count))
    e64, z64 = eps[:npix].astype(np.float64), z[:npix].astype(np.float64)
    want = x[:npix].astype(np.float64) - (delta * e64 + math.sqrt(2 * delta) * z64) * f32(sgn)
    xd, ed, zd = (torch.from_numpy(a).to(dev) for a in (x, eps, z))
    assert corrector(lib, dev, xd, ed, zd, sumsq, count, tau, sgn, 0, 0, 0, npix=npix) == 0
    got = xd.cpu().numpy()
    assert relerr(got[:npix], want) < 1e-5
    assert np.array_equal(got[npix], x[npix])  # past the launch: untouched
    for pixel, bad, want_flag in ((npix // 2, math.inf, 1), (npix - 1, math.nan, 1), (npix, math.nan, 0)):
        xb = x.copy()
        xb[pixel, C - 1] = bad
        assert corrector(lib, dev, torch.from_numpy(xb).to(dev), ed, zd, sumsq, count, tau, sgn, 0, 0, 0,
                         npix=npix) == want_flag, (pixel, bad)


@pytest.mark.gpu
@pytest.mark.parametrize("C", range(1, 9))
def test_corrector_philox_noise_vs_numpy(lib, dev, C):
    """On-chip noise against philox_normals.  x = eps = 0, delta = 0.5, sigma' = 1 make x = -z.  700,001 pixels: more
    than one grid-stride trip at 16 CTAs x 256 threads per SM on 148 SMs; the global pixel range crosses 2^32 (counter
    word 1) and the seed uses both key words.  Splitting the launch at an odd pixel gives the same bits; another seed
    or step gives other noise."""
    npix, pix0, seed, step = 700_001, 2 ** 32 - 350_000, 0x9E3779B97F4A7C15, 7
    x = torch.zeros(npix, C, device=dev)
    zero = torch.zeros_like(x)
    assert corrector(lib, dev, x, zero, None, 1.0, 1.0, 0.5, 1.0, pix0, seed, step) == 0
    got = -x.cpu().numpy().astype(np.float64)
    want = philox_normals(pix0 + np.arange(npix, dtype=np.uint64), step, seed, C)
    assert np.all(np.abs(got - want) <= 1e-5 * np.maximum(1.0, np.abs(want))), np.abs(got - want).max()
    assert abs(got.mean()) < 0.01 and abs(got.std() - 1) < 0.01
    # the same pixels in two launches split at an odd pixel (not a frame boundary): bit-identical
    cut = 333_333
    x2 = torch.zeros_like(x)
    corrector(lib, dev, x2, zero, None, 1.0, 1.0, 0.5, 1.0, pix0, seed, step, npix=cut)
    corrector(lib, dev, x2[cut:], zero[cut:], None, 1.0, 1.0, 0.5, 1.0, pix0 + cut, seed, step, npix=npix - cut)
    assert torch.equal(x2, x)
    # another seed (either key word) or step: other noise
    n = 4099
    base = -x[:n].cpu().numpy()
    for s2, t2 in ((seed + 1, step), (seed + (1 << 32), step), (seed, step + 1)):
        x3 = torch.zeros(n, C, device=dev)
        corrector(lib, dev, x3, zero[:n], None, 1.0, 1.0, 0.5, 1.0, pix0, s2, t2)
        other = -x3.cpu().numpy()
        assert np.mean(other == base) < 0.01, (s2, t2)
        want = philox_normals(pix0 + np.arange(n, dtype=np.uint64), t2, s2, C)
        assert np.all(np.abs(other - want) <= 1e-5 * np.maximum(1.0, np.abs(want))), (s2, t2)


# ------------------------------------------------------------------------------------------------ partial sums
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 7, 255, 256, 257, 1000, 65539])
def test_reduce_partials_vs_fsum(lib, dev, n):
    """c2w_reduce_partials: the double sum of n fp32 partials of mixed sign and magnitude (1e-3 .. 1e3) against
    math.fsum of the same values, within 1e-12 of sum |p|; two calls give the same bits."""
    from climate2weather_b200 import _lib
    rng = np.random.default_rng(n)
    p = (rng.choice([-1.0, 1.0], n) * 10.0 ** rng.uniform(-3, 3, n)).astype(np.float32)
    pd = torch.from_numpy(p).to(dev)
    outs = []
    for _ in range(2):
        out = torch.full((1,), math.nan, dtype=torch.float64, device=dev)
        _lib.check(lib.c2w_reduce_partials(pd.data_ptr(), n, out.data_ptr(), stream()), "c2w_reduce_partials")
        torch.cuda.synchronize()
        outs.append(out.item())
    want = math.fsum(float(v) for v in p)
    assert abs(outs[0] - want) <= 1e-12 * float(np.abs(p.astype(np.float64)).sum())
    assert np.float64(outs[0]).tobytes() == np.float64(outs[1]).tobytes()
