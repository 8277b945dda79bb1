"""GPU tests (pytest -m gpu) of guided sampling through any differentiable observation operator (the generic path:
c2w_x0_nchw -> A and its VJP in torch -> c2w_guided_step_dense).  The two kernels alone against float64 references,
the closed form against the oracle's torch.func.vjp through the same operator, the whole path against the reference's
log_p + autograd, the generic path against the fused one on the same operator, bitwise invariance (windows per launch,
repeats, autocast, inference mode), ensembles and batches against their members' own runs, and the NaN error.

The operators are the ones users bring: (a) a time mean of tile means, (b) bilinear interpolation at off-grid stations,
(c) a fixed dense regridding matrix, (d) wind speed sqrt(u^2 + v^2) at stations (nonlinear)."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from oracle import pipeline_ref, unet_ref

import oracle_op

pytestmark = pytest.mark.gpu

SMALL = dict(embedding_dim=64, hidden_channels=(64, 128), hidden_blocks=(1, 2), attention_levels=(1,), kernel_size=3)
GAMMA = 0.0007196856730011522
K, L, H, W = 2, 12, 32, 32


def relerr(got, ref):
    got, ref = got.double().cpu(), ref.double().cpu()
    return ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


def rel_l2(got, ref):
    got, ref = got.double().cpu(), ref.double().cpu()
    return ((got - ref).norm() / ref.norm().clamp_min(1e-30)).item()


# ------------------------------------------------------------------------------------------------ operators
class TimeMeanOfTileMeans:
    """(a) means over `tau` consecutive frames of s x s tile means: [L / tau, C, H / s, W / s]."""

    def __init__(self, tau=3, s=8):
        self.tau, self.s = tau, s

    def __call__(self, x):
        p = F.avg_pool2d(x, self.s)
        return p.reshape(-1, self.tau, *p.shape[1:]).mean(1)


class Bilinear:
    """(b) bilinear interpolation of every frame at P off-grid stations: [L, C, P]."""

    def __init__(self, P=40, seed=0):
        g = torch.Generator().manual_seed(seed)
        self.r = torch.rand(P, generator=g) * (H - 1.001)
        self.c = torch.rand(P, generator=g) * (W - 1.001)

    def __call__(self, x):
        r, c = self.r.to(x.device), self.c.to(x.device)
        r0, c0 = r.floor().long(), c.floor().long()
        fr, fc = (r - r0).to(x.dtype), (c - c0).to(x.dtype)
        v = lambda i, j: x[:, :, i, j]
        return ((1 - fr) * (1 - fc) * v(r0, c0) + (1 - fr) * fc * v(r0, c0 + 1) + fr * (1 - fc) * v(r0 + 1, c0)
                + fr * fc * v(r0 + 1, c0 + 1))


class Regrid:
    """(c) a fixed dense regridding matrix onto P cells: [L, C, P]."""

    def __init__(self, P=24, seed=1):
        m = torch.rand(P, H * W, generator=torch.Generator().manual_seed(seed))
        self.M = m / m.sum(1, keepdim=True)

    def __call__(self, x):
        return torch.einsum("pk,lck->lcp", self.M.to(x.device), x.reshape(*x.shape[:2], -1))


class WindSpeed:
    """(d) sqrt(u^2 + v^2) of variables 0 and 1 at P station pixels of every frame: [L, P]."""

    def __init__(self, P=30, seed=2):
        g = torch.Generator().manual_seed(seed)
        self.rows, self.cols = torch.randint(0, H, (P,), generator=g), torch.randint(0, W, (P,), generator=g)

    def __call__(self, x):
        u = x[:, 0, self.rows.to(x.device), self.cols.to(x.device)]
        v = x[:, 1, self.rows.to(x.device), self.cols.to(x.device)]
        return torch.sqrt(u * u + v * v)


class Subsample:
    """Every t-th frame at every s-th pixel (a strided slice: its VJP writes each pixel once)."""

    def __init__(self, t=2, s=4):
        self.t, self.s = t, s

    def __call__(self, x):
        return x[::self.t, :, ::self.s, ::self.s]


OPS = {"time_mean": TimeMeanOfTileMeans, "bilinear": Bilinear, "regrid": Regrid, "wind": WindSpeed}


def _problem(op, C, seed=0, Lp=L):
    """y = A(truth) + noise, a std that broadcasts against A(x) (per observation where it can) and gamma."""
    g = torch.Generator().manual_seed(seed + 10 * C)
    truth = torch.randn(Lp, C, H, W, generator=g)
    y = op(truth)
    y = y + 0.1 * torch.randn(y.shape, generator=g)
    std = 0.1 + 0.1 * torch.rand(y.shape[1:], generator=g)  # one std per (variable, site), shared by every frame
    return y, std


def _net(C, seed=3):
    import climate2weather_b200 as c2w
    cfg = dict(SMALL, channels=C * (2 * K + 1))
    torch.manual_seed(seed)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, **cfg)
    ref = unet_ref.RefNet({n: v.detach().clone() for n, v in net.state_dict().items()}, cfg)
    return net.to("cuda:0"), ref


# ------------------------------------------------------------------------------------------------ kernels alone
def _guide(lib, x, eps, mode, mu, sigma, mu_n, sigma_n, own_lo, own_n, C, Hh, Ww, vjp=None, eps_out=None, partials=None,
           nan_flag=None):
    from climate2weather_b200 import _lib
    g = _lib.Guide()
    g.x, g.eps, g.y = x.data_ptr(), eps.data_ptr(), None
    g.mu, g.sigma, g.mu_next, g.sigma_next = mu, sigma, mu_n, sigma_n
    g.t_step, g.s_step, g.H, g.W = 1, 1, Hh, Ww
    g.frame_global0, g.own_lo, g.own_n, g.mode, g.channels = 0, own_lo, own_n, mode, C
    g.nan_flag = nan_flag.data_ptr()
    g.vjp = vjp.data_ptr() if vjp is not None else None
    g.eps_out = eps_out.data_ptr() if eps_out is not None else None
    g.partials = partials.data_ptr() if partials is not None else None
    g.halo, g.halo_k = None, K
    return g


@pytest.mark.parametrize("Hh,Ww", [(32, 32), (48, 96), (128, 128)])
@pytest.mark.parametrize("C", range(1, 9))
def test_dense_kernels_vs_float64(C, Hh, Ww):
    """c2w_x0_nchw within 1e-6 of max-abs; c2w_guided_step_dense (modes 0 / 1, with and without a VJP term) within 1e-5
    of max-abs on x, eps_g and the correction, every partial within 1e-5 relative; eps_g == eps bit for bit where g is
    exactly 0 without a VJP term; mode 2 is refused."""
    from climate2weather_b200 import _lib
    from climate2weather_b200.score import point_strip_rows
    lib = _lib.load()
    dev = torch.device("cuda:0")
    st = torch.cuda.current_stream().cuda_stream
    Lf, own_lo, own_n = 6, 1, 4
    gen = torch.Generator().manual_seed(7 * C + Hh)
    x = torch.randn(Lf, Hh, Ww, C, generator=gen)
    eps = torch.randn(Lf, Hh, Ww, C, generator=gen)
    vjp = torch.randn(Lf, Hh, Ww, C, generator=gen)
    grad = torch.randn(own_n, C, Hh, Ww, generator=gen)
    grad[:, :, : Hh // 2] = 0.0  # g exactly 0 on the top half of every frame
    mu, sigma, mu_n, sigma_n = 0.8, 0.55, 0.9, 0.4
    xd, ed, vd, gd = (t.to(dev) for t in (x, eps, vjp, grad))
    flag = torch.zeros(1, dtype=torch.int32, device=dev)

    x0 = torch.empty(Lf, C, Hh, Ww, device=dev)
    _lib.check(lib.c2w_x0_nchw(xd.data_ptr(), ed.data_ptr(), mu, sigma, x0.data_ptr(), Lf, C, Hh * Ww, st), "x0")
    want_x0 = ((x.double() - sigma * eps.double()) / mu).permute(0, 3, 1, 2)
    assert relerr(x0, want_x0) < 1e-6

    R = point_strip_rows(Hh, Ww)
    n_strips = -(-Hh // R)
    g64 = grad.double().permute(0, 2, 3, 1)  # [own_n, H, W, C]
    sl = slice(own_lo, own_lo + own_n)
    for use_vjp in (False, True):
        gv = g64 - sigma * vjp.double()[sl] if use_vjp else g64
        want_e = eps.double()[sl] - (sigma / mu) * gv
        # mode 1: eps_g and the per-(frame, strip) partial sums of its squares
        eps_out = torch.full_like(ed, float("nan"))
        parts = torch.full((own_n * n_strips,), float("nan"), device=dev)
        gd_ = _guide(lib, xd, ed, 1, mu, sigma, 0.0, 0.0, own_lo, own_n, C, Hh, Ww, vd if use_vjp else None, eps_out,
                     parts, flag)
        _lib.check(lib.c2w_guided_step_dense(ctypes.byref(gd_), gd.data_ptr(), st), "dense mode 1")
        got_e = eps_out.cpu()[sl]
        assert relerr(got_e, want_e) < 1e-5
        assert relerr(eps[sl] - got_e, eps.double()[sl] - want_e) < 1e-5
        want_p = (want_e ** 2).reshape(own_n, Hh, Ww * C)
        want_p = torch.stack([want_p[:, i * R:(i + 1) * R].sum((1, 2)) for i in range(n_strips)], 1).reshape(-1)
        assert ((parts.cpu().double() - want_p).abs() / want_p).max().item() < 1e-5
        if not use_vjp:
            assert torch.equal(got_e[:, : Hh // 2], eps[sl][:, : Hh // 2])
        # mode 0: the predictor update of the owned frames in place, the others untouched
        xm = xd.clone()
        gd0 = _guide(lib, xm, ed, 0, mu, sigma, mu_n, sigma_n, own_lo, own_n, C, Hh, Ww, vd if use_vjp else None,
                     nan_flag=flag)
        _lib.check(lib.c2w_guided_step_dense(ctypes.byref(gd0), gd.data_ptr(), st), "dense mode 0")
        want_xm = mu_n * (x.double()[sl] - sigma * want_e) / mu + sigma_n * want_e
        got_xm = xm.cpu()
        assert relerr(got_xm[sl], want_xm) < 1e-5
        assert torch.equal(got_xm[:own_lo], x[:own_lo]) and torch.equal(got_xm[own_lo + own_n:], x[own_lo + own_n:])
    assert int(flag.item()) == 0
    bad = _guide(lib, xd, ed, 2, mu, sigma, 0.0, 0.0, own_lo, own_n, C, Hh, Ww, nan_flag=flag)
    assert lib.c2w_guided_step_dense(ctypes.byref(bad), gd.data_ptr(), st) != 0
    assert b"modes 0 and 1" in lib.c2w_last_error()


# ------------------------------------------------------------------------------------------------ vs the oracle
@pytest.mark.parametrize("name", list(OPS))
def test_generic_guidance_vs_closed_form(name):
    """sf(x, t) - eps against the oracle's A^T((y - A x0)/var)/mu through torch.func.vjp of the same operator, from the
    same GPU eps: 1e-5."""
    import climate2weather_b200 as c2w
    C = 4
    net, _ = _net(C)
    op = OPS[name]()
    y, std = _problem(op, C)
    x = torch.randn(L, C, H, W, generator=torch.Generator().manual_seed(21))
    sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=c2w.SDAPipeline())
    t = torch.tensor(0.45)
    eps = sf.score_fn(x.cuda(), t).cpu()
    sf.condition_on(A=op, y=y, std=std, gamma=GAMMA, exact_grad=False)
    got = sf(x.cuda(), t).cpu()
    assert type(sf.likelihood["op"]).__name__ == "GenericObservation"
    want = oracle_op.guided_score_closed_form_op(eps, x, t, y, std, GAMMA, op)
    e = relerr(got - eps, want - eps)
    print(f"\n{name}: correction rel-err {e:.3e}")
    assert e < 1e-5, e
    assert not torch.equal(got, eps)


@pytest.mark.parametrize("C,name", [(4, "time_mean"), (3, "wind")])
def test_generic_guided_path_vs_oracle(C, name):
    """The whole path against the fp32 oracle (the reference's log_p + autograd with the same A): closed-form guided
    score, a 3-step predictor-corrector run with the reference's noise draws, exact_grad with one stashing chunk and
    with several — the point-observation tests' tolerances."""
    import climate2weather_b200 as c2w
    net, ref = _net(C, seed=11 + C)
    op = OPS[name]()
    y, std = _problem(op, C, seed=1)
    x = torch.randn(L, C, H, W, generator=torch.Generator().manual_seed(50 + C))
    t = torch.tensor(0.45)
    pipe = c2w.SDAPipeline()
    sf = c2w.BatchedScoreFunction(net, markov_order=K, noise_process=pipe, batch_size=4, device="cuda:0")
    sf.condition_on(A=op, y=y, std=std, gamma=GAMMA, exact_grad=False)
    with torch.no_grad():
        want_g = oracle_op.guided_score_op(ref, x, t, K, y, std, GAMMA, op, exact_grad=False)
    eg = relerr(sf(x, t), want_g)
    assert eg < 3e-2, eg
    ref_pipe = pipeline_ref.RefPipeline()
    score = lambda xx, tt: oracle_op.guided_score_op(ref, xx, tt, K, y, std, GAMMA, op, exact_grad=False)
    torch.manual_seed(5)
    want_s = ref_pipe.sample(score, x, steps=3, corrections=1, tau=0.5)
    pipe.rng = "reference"
    torch.manual_seed(5)
    got_s = pipe.sample(sf, x, steps=3, corrections=1, tau=0.5, show_progressbar=False)
    es, ls = relerr(got_s, want_s), rel_l2(got_s, want_s)
    want_e = oracle_op.guided_score_op(ref, x, t, K, y, std, GAMMA, op, exact_grad=True)
    d = relerr(want_g, want_e)
    ee = []
    for mw in (None, 3):
        sfe = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=c2w.SDAPipeline())
        sfe.max_windows = mw
        sfe.condition_on(A=op, y=y, std=std, gamma=GAMMA, exact_grad=True)
        ee.append(relerr(sfe(x.cuda(), t).cpu(), want_e))
        rt = next(iter(sfe._runtimes.values()))
        assert rt.n_selected == L - 2 * K and (rt.n_repeated == 0) == (mw is None)
    print(f"\nC={C} {name}: guided {eg:.3e}, sampler max-abs ratio {es:.3e} rel-L2 {ls:.3e}, exact {ee} "
          f"(closed vs exact {d:.3e})")
    assert got_s.shape == x.shape and es < 5e-2 and ls < 3e-2
    for e in ee:
        assert e < 4e-2 and e < 0.5 * d, (ee, d)


def test_generic_path_matches_fused_on_the_same_operator(monkeypatch):
    """CoarseGrain(3, 8) through the generic path (the recogniser bypassed) against the fused K6 path: the closed-form
    guided score within 1e-5 relative (different summation orders, not bitwise)."""
    import climate2weather_b200 as c2w
    from climate2weather_b200 import score
    C = 4
    net, _ = _net(C)
    op = c2w.CoarseGrain(3, 8)
    y, _ = _problem(op, C, seed=4)
    x = torch.randn(L, C, H, W, generator=torch.Generator().manual_seed(8)).cuda()
    t = torch.tensor(0.35)
    out = {}
    for path in ("fused", "generic"):
        with monkeypatch.context() as mp:
            if path == "generic":
                mp.setattr(score, "_route_operator", lambda A, *a: score.GenericObservation(A))
            sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=c2w.SDAPipeline())
            sf.condition_on(A=op, y=y, std=0.15, gamma=GAMMA, exact_grad=False)
            out[path] = sf(x, t).cpu()
            assert (type(sf.likelihood["op"]).__name__ == "GenericObservation") == (path == "generic")
    e = relerr(out["generic"], out["fused"])
    print(f"\ngeneric vs fused rel-err {e:.3e}")
    assert e < 1e-5, e
    assert not torch.equal(out["generic"], sf.score_fn(x, t).cpu())


# ------------------------------------------------------------------------------------------------ bitwise
def _sample(sf, x, **kw):
    import climate2weather_b200 as c2w
    return c2w.SDAPipeline().sample(sf, x, steps=3, corrections=1, tau=0.5, show_progressbar=False, seed=9, **kw).cpu()


def test_generic_guidance_is_bitwise_invariant():
    """Bit-identical across windows per launch and repeats, and with sample() called inside
    torch.autocast("cuda", float16) and inside torch.inference_mode() (A runs in fp32 with autograd either way)."""
    import climate2weather_b200 as c2w
    net, _ = _net(4)
    op = TimeMeanOfTileMeans()
    y, std = _problem(op, 4)
    x = torch.randn(L, 4, H, W, generator=torch.Generator().manual_seed(2))
    t = torch.tensor(0.3)
    outs, samples = [], []
    for mw in (None, 3, None):
        sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=c2w.SDAPipeline())
        sf.max_windows = mw
        sf.condition_on(A=op, y=y, std=std, gamma=GAMMA, exact_grad=False)
        outs.append(sf(x.cuda(), t).cpu())
        samples.append(_sample(sf, x))
    for o in outs[1:]:
        assert torch.equal(o, outs[0])
    for s in samples[1:]:
        assert torch.equal(s, samples[0])
    assert torch.isfinite(samples[0]).all()
    sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=c2w.SDAPipeline())
    sf.condition_on(A=op, y=y, std=std, gamma=GAMMA, exact_grad=False)
    with torch.autocast("cuda", dtype=torch.float16):
        assert torch.equal(_sample(sf, x), samples[0])
        assert torch.equal(sf(x.cuda(), t).cpu(), outs[0])
    with torch.inference_mode():
        assert torch.equal(_sample(sf, x), samples[0])
        assert torch.equal(sf(x.cuda(), t).cpu(), outs[0])
    with torch.no_grad():
        assert torch.equal(_sample(sf, x), samples[0])


# ------------------------------------------------------------------------------------------------ ensembles, batches
@pytest.mark.parametrize("corrections", [0, 1])
def test_generic_ensemble_members_equal_their_own_runs(corrections):
    import climate2weather_b200 as c2w
    net, _ = _net(4)
    op = TimeMeanOfTileMeans()
    y, std = _problem(op, 4)
    M = 3
    noise = torch.randn(M, L, 4, H, W, generator=torch.Generator().manual_seed(12))
    seeds = [5, 123, 77]
    sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=c2w.SDAPipeline())
    sf.condition_on(A=op, y=y, std=std, gamma=GAMMA, exact_grad=False)
    pipe = c2w.SDAPipeline()
    ens = pipe.sample_ensemble(sf, noise, steps=3, corrections=corrections, tau=0.5, show_progressbar=False,
                               seeds=seeds).cpu()
    for m in range(M):
        own = pipe.sample(sf, noise[m], steps=3, corrections=corrections, tau=0.5, show_progressbar=False,
                          seed=seeds[m]).cpu()
        assert torch.equal(ens[m], own), m
    assert not torch.equal(ens[0], ens[1])


def test_generic_batch_members_equal_their_own_runs():
    """Members with different generic operators, y, std and gamma, each bit-identical to its own run; a batch of one
    score function M times equals the ensemble of it."""
    import climate2weather_b200 as c2w
    net, _ = _net(4)
    ops = [TimeMeanOfTileMeans(3, 8), Subsample(2, 4), TimeMeanOfTileMeans(2, 4)]
    sfs = []
    for m, op in enumerate(ops):
        y, std = _problem(op, 4, seed=30 + m)
        sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=c2w.SDAPipeline())
        sf.condition_on(A=op, y=y, std=std, gamma=GAMMA * (m + 1), exact_grad=False)
        sfs.append(sf)
    M = len(sfs)
    noise = torch.randn(M, L, 4, H, W, generator=torch.Generator().manual_seed(13))
    seeds = [4, 8, 15]
    pipe = c2w.SDAPipeline()
    for corrections in (0, 1):
        got = pipe.sample_batch(sfs, noise, steps=3, corrections=corrections, tau=0.5, show_progressbar=False,
                                seeds=seeds).cpu()
        for m in range(M):
            own = pipe.sample(sfs[m], noise[m], steps=3, corrections=corrections, tau=0.5, show_progressbar=False,
                              seed=seeds[m]).cpu()
            assert torch.equal(got[m], own), (corrections, m)
    same = pipe.sample_batch([sfs[0]] * M, noise, steps=3, corrections=1, tau=0.5, show_progressbar=False,
                             seeds=seeds).cpu()
    ens = pipe.sample_ensemble(sfs[0], noise, steps=3, corrections=1, tau=0.5, show_progressbar=False,
                               seeds=seeds).cpu()
    assert torch.equal(same, ens)


def test_nan_in_y_raises():
    import climate2weather_b200 as c2w
    net, _ = _net(4)
    op = TimeMeanOfTileMeans()
    y, std = _problem(op, 4)
    y[1, 2, 0, 1] = float("nan")
    sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=c2w.SDAPipeline())
    sf.condition_on(A=op, y=y, std=std, gamma=GAMMA, exact_grad=False)
    with pytest.raises(ValueError, match="NaN detected in sample"):
        c2w.SDAPipeline().sample(sf, torch.randn(L, 4, H, W), steps=2, show_progressbar=False)
