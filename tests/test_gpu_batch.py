"""GPU tests (pytest -m gpu) of batched sampling of independent problems (SDAPipeline.sample_batch): the batch guidance
step (c2w_guided_step_batch) against the single-trajectory entry points member by member, the contract
that member m equals sample(score_fns[m], noise[m], seed=seeds[m]) bit for bit for every operator with per-member
observations, std forms and gamma, the ensemble cross-check, hooks, traces, the NaN error and the runtime cache."""
import pytest
import torch

from test_gpu_ensemble import GAMMA, KINDS, SMALL

pytestmark = pytest.mark.gpu

K, L, H, W = 2, 11, 32, 32
M = 3


def _net(C, seed=3):
    import climate2weather_b200 as c2w
    torch.manual_seed(seed)
    return c2w.ScoreUNet(activation=torch.nn.SiLU, channels=C * (2 * K + 1), **SMALL).to("cuda:0")


def _condition(sf, kind, C, m, Lm=L, Hm=H, Wm=W, s=8, t=3, form=None):
    """Conditions member m on its own observation of the given kind: its own y, stations (count, frames, mask), gamma,
    and a std whose form depends on m (one value, per variable, per observation) unless the kind fixes it or `form`
    ("var" / "obs") overrides it."""
    import climate2weather_b200 as c2w
    g = torch.Generator().manual_seed(100 * m + 7 * C + Hm)
    P = 20 + 17 * m
    rows, cols = torch.randint(0, Hm, (P,), generator=g), torch.randint(0, Wm, (P,), generator=g)
    rows[1], cols[1] = rows[0], cols[0]
    F = 2 + m
    frames = torch.randperm(Lm, generator=g)[:F]
    mask = torch.rand(F, C, P, generator=g) > 0.2 + 0.1 * m
    pts = c2w.PointObservation(frames, rows, cols, mask)
    py = torch.randn(F, C, P, generator=g).masked_fill(~mask, float("nan"))
    cg = c2w.CoarseGrain(t, s)
    cshape = (-(-Lm // t), C, Hm // s, Wm // s)
    cy = torch.randn(cshape, generator=g)
    gamma = [GAMMA * (1 + m + 0.5 * c) for c in range(C)] if m % 2 else GAMMA * (1 + m)
    var = [0.1 + 0.05 * c + 0.02 * m for c in range(C)]
    one = 0.15 + 0.05 * m
    form = form or ("one", "var", "obs")[m % 3]
    shape = (Lm, C, Hm, Wm)
    if kind == "none":
        return
    if kind in ("coarse", "coarse_std_tile"):
        if kind == "coarse_std_tile" or form == "obs":
            std = 0.05 + torch.rand(1, 1, Hm // s, Wm // s, generator=g)
        else:
            std = one if form == "one" else var
        sf.condition_on(A=cg, y=cy, std=std, gamma=gamma, exact_grad=False)
    elif kind == "coarse_opaque":
        sf.condition_on(A=lambda x: torch.nn.functional.avg_pool2d(x[::t], s), y=cy, std=one if form != "var" else var,
                        gamma=gamma, exact_grad=False)
    elif kind in ("points", "points_std_station"):
        if kind == "points_std_station" or form == "obs":
            std = (0.05 + torch.rand(1, 1, P, generator=g)).expand(F, C, P)
        else:
            std = one if form == "one" else torch.tensor(var).reshape(1, C, 1)
        sf.condition_on(A=pts, y=py, std=std, gamma=gamma, exact_grad=False)
    elif kind in ("combined", "combined_std_obs"):
        op = c2w.CombinedObservation(cg, pts)
        if kind == "combined_std_obs" or form == "obs":
            std = op.pack(0.05 + torch.rand(cshape, generator=g), 0.05 + torch.rand(F, C, P, generator=g), shape)
        else:
            std = one if form == "one" else op.pack(0.3 + 0.1 * m, torch.tensor(var), shape)
        sf.condition_on(A=op, y=op.pack(cy, py, shape), std=std, gamma=gamma, exact_grad=False)
    else:
        raise ValueError(kind)


def _members(net, kind, C, mw=None, **kw):
    import climate2weather_b200 as c2w
    pipe = c2w.SDAPipeline()
    sfs = []
    for m in range(M):
        sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=pipe)
        sf.max_windows = mw
        _condition(sf, kind, C, m, **kw)
        sfs.append(sf)
    return pipe, sfs


# ------------------------------------------------------------------------------------------------ kernel level
GRIDS = [(32, 32, 8), (48, 96, 3), (128, 128, 16)]


@pytest.mark.parametrize("Hm,Wm,s", GRIDS)
@pytest.mark.parametrize("C", range(1, 9))
def test_batch_guidance_equals_single_guidance_per_member(C, Hm, Wm, s, monkeypatch):
    """c2w_guided_step_batch (through the runtime's _guide) at modes 0 / 1 / 2, with and without a VJP term, for the
    coarse, point and combined terms, per variable, per observation and mixed, against the single-trajectory entry
    points on each member's slice with its own y, std and gamma: x, eps_g, the cotangent and each member's partials,
    bit for bit.  The guidance step reads no network: the runtimes are built without an engine, so that grids the
    UNet does not take (48 x 96) are covered too."""
    import climate2weather_b200 as c2w
    monkeypatch.setattr(c2w.score._Runtime, "refresh_engine", lambda self: None)
    net = _net(C)
    Lm = 7
    gen = torch.Generator().manual_seed(C + Hm)
    x = torch.randn(M, Lm, C, Hm, Wm, generator=gen).cuda()
    eps = torch.randn(M, Lm, Hm, Wm, C, generator=gen).cuda()
    vjp = torch.randn(M, Lm, Hm, Wm, C, generator=gen).cuda()
    for kind in ("coarse", "points", "combined"):
        for form in ("var", "obs", None):  # None: the members' forms differ
            pipe, sfs = _members(net, kind, C, Lm=Lm, Hm=Hm, Wm=Wm, s=s, t=2, form=form)
            bat = pipe._batch_runtime(sfs, x)
            assert bat.batch is not None and bat.batch["per_obs"] == (form != "var")
            singles = [sf.runtime(x[m]) for m, sf in enumerate(sfs)]
            for mode in (0, 1, 2):
                for with_vjp in ((False, True) if mode != 2 else (False,)):
                    for rt, xs, es, vs in [(bat, x, eps.reshape(M * Lm, Hm, Wm, C), vjp.reshape(M * Lm, Hm, Wm, C))] + \
                            [(singles[m], x[m], eps[m], vjp[m]) for m in range(M)]:
                        rt.load(xs)
                        rt.eps.copy_(es)
                        rt.cot = torch.zeros_like(rt.x)
                        rt.exact, rt.vjp = with_vjp, vs.contiguous() if with_vjp else None  # the kernels' vjp term
                        rt._guide(mode, 0.8, 0.5, 0.9, 0.4)
                        rt.exact, rt.vjp = False, None
                    seg = bat._n_part // M if mode == 1 else 0
                    for m, one in enumerate(singles):
                        sl = slice(m * Lm, (m + 1) * Lm)
                        what = (kind, form, mode, with_vjp, m)
                        assert torch.equal(bat.x[sl], one.x), what
                        if mode == 1:
                            assert torch.equal(bat.eps_g[sl], one.eps_g), what
                            assert seg == one._n_part, what
                            assert torch.equal(bat.partials[m * seg:(m + 1) * seg], one.partials[:seg]), what
                        if mode == 2:
                            assert torch.equal(bat.cot[sl], one.cot), what


# ------------------------------------------------------------------------------------------------ the contract
@pytest.mark.parametrize("corrections", [0, 2])
@pytest.mark.parametrize("C", [4, 3])
@pytest.mark.parametrize("kind", KINDS)
def test_batch_equals_sequential_samples(kind, C, corrections):
    """Member m of sample_batch(score_fns, noise, seeds=s) is bit-identical to sample(score_fns[m], noise[m],
    seed=s[m]), with per-member observations, stations, std forms and gamma, at the default max_windows (one launch of
    21 windows) and at 4, which splits members across launches."""
    net = _net(C)
    noise = torch.randn(M, L, C, H, W, generator=torch.Generator().manual_seed(7))
    seeds = [11, 2 ** 40 + 3, 12345]
    for mw in (None, 4):
        pipe, sfs = _members(net, kind, C, mw)
        out = pipe.sample_batch(sfs, noise, steps=3, corrections=corrections, show_progressbar=False, seeds=seeds)
        assert out.shape == noise.shape and out.device == noise.device
        for m in range(M):
            one = pipe.sample(sfs[m], noise[m], steps=3, corrections=corrections, show_progressbar=False, seed=seeds[m])
            assert torch.equal(out[m], one), (kind, C, corrections, mw, m)


def _coarse_members(net, Lm, t, seed):
    import climate2weather_b200 as c2w
    pipe = c2w.SDAPipeline()
    sfs = []
    for m in range(M):
        truth = torch.randn(Lm, 4, H, W, generator=torch.Generator().manual_seed(seed + m))
        cg = c2w.CoarseGrain(t, 8)
        sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=pipe)
        sf.condition_on(A=cg, y=cg(truth), std=0.1 + 0.1 * m, gamma=GAMMA * (m + 1), exact_grad=False)
        sfs.append(sf)
    return pipe, sfs


def test_batch_keeps_a_members_conv_tile_widths():
    """The 384-channel level whose tile width flips between a member's 37 windows and the batch's 111."""
    import climate2weather_b200 as c2w
    torch.manual_seed(5)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, channels=4 * (2 * K + 1), embedding_dim=64, hidden_channels=(64, 384),
                        hidden_blocks=(1, 1), attention_levels=(), kernel_size=3).to("cuda:0")
    Lm = 41
    pipe, sfs = _coarse_members(net, Lm, 3, 1)
    noise = torch.randn(M, Lm, 4, H, W, generator=torch.Generator().manual_seed(2))
    out = pipe.sample_batch(sfs, noise, steps=2, corrections=1, show_progressbar=False, seeds=[0, 1, 2])
    for m in range(M):
        one = pipe.sample(sfs[m], noise[m], steps=2, corrections=1, show_progressbar=False, seed=m)
        assert torch.equal(out[m], one), m


def test_batch_keeps_a_members_conv_variant():
    """One window per member (L = 2k + 1): the 128-channel 8 x 8 level's main loop flips with the window count."""
    import climate2weather_b200 as c2w
    torch.manual_seed(6)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, channels=4 * (2 * K + 1), embedding_dim=64,
                        hidden_channels=(64, 128, 128), hidden_blocks=(1, 1, 1), attention_levels=(),
                        kernel_size=3).to("cuda:0")
    Lm = 2 * K + 1
    pipe, sfs = _coarse_members(net, Lm, 2, 3)
    noise = torch.randn(M, Lm, 4, H, W, generator=torch.Generator().manual_seed(4))
    out = pipe.sample_batch(sfs, noise, steps=3, corrections=1, show_progressbar=False, seeds=[7, 8, 9])
    for m in range(M):
        one = pipe.sample(sfs[m], noise[m], steps=3, corrections=1, show_progressbar=False, seed=7 + m)
        assert torch.equal(out[m], one), m


@pytest.mark.parametrize("kind", ["coarse", "points", "combined_std_obs"])
def test_batch_of_one_score_function_equals_the_ensemble(kind):
    import climate2weather_b200 as c2w
    net = _net(4)
    pipe = c2w.SDAPipeline()
    sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=pipe)
    _condition(sf, kind, 4, 1)
    noise = torch.randn(M, L, 4, H, W, generator=torch.Generator().manual_seed(9))
    seeds = [3, 4, 5]
    ens = pipe.sample_ensemble(sf, noise, steps=3, corrections=1, show_progressbar=False, seeds=seeds)
    bat = pipe.sample_batch([sf] * M, noise, steps=3, corrections=1, show_progressbar=False, seeds=seeds)
    assert torch.equal(bat, ens)


def test_default_seeds_hook_and_traces():
    """Default seeds drawn in member order, a proc_x0 hook called once per member on [L, C, H, W], and trace_at traces
    of shape [M, L, C, H, W]."""
    C = 4
    net = _net(C)
    pipe, sfs = _members(net, "points", C)
    pipe.trace_at = [2]
    shapes = []

    def hook(x0):
        shapes.append(tuple(x0.shape))
        return x0.clamp(-1.5, 1.5)

    noise = torch.randn(M, L, C, H, W, generator=torch.Generator().manual_seed(1))
    torch.manual_seed(123)
    singles, traces = [], []
    for m in range(M):
        singles.append(pipe.sample(sfs[m], noise[m], steps=3, corrections=1, proc_x0=hook, show_progressbar=False))
        traces.append(pipe.traces[2])
    shapes.clear()
    torch.manual_seed(123)
    out = pipe.sample_batch(sfs, noise, steps=3, corrections=1, proc_x0=hook, show_progressbar=False)
    assert shapes == [(L, C, H, W)] * (3 * M)
    assert pipe.traces[2].shape == (M, L, C, H, W)
    for m in range(M):
        assert torch.equal(out[m], singles[m]), m
        assert torch.equal(pipe.traces[2][m], traces[m]), m


def test_non_finite_member_raises_the_reference_error():
    net = _net(4)
    pipe, sfs = _members(net, "coarse", 4)
    noise = torch.randn(M, L, 4, H, W)
    noise[1, 5, 2, 7, 7] = float("inf")
    with pytest.raises(ValueError, match="NaN detected in sample"):
        pipe.sample_batch(sfs, noise, steps=2, show_progressbar=False)


def test_second_call_reuses_the_runtime_and_reconditioning_changes_one_member():
    C = 4
    net = _net(C)
    pipe, sfs = _members(net, "combined", C)
    noise = torch.randn(M, L, C, H, W, generator=torch.Generator().manual_seed(2))
    seeds = [1, 2, 3]
    first = pipe.sample_batch(sfs, noise, steps=2, corrections=1, show_progressbar=False, seeds=seeds)
    rt, eng, pts = pipe._batch_cache[2], pipe._batch_cache[2].engine, pipe._batch_cache[2].points
    again = pipe.sample_batch(sfs, noise, steps=2, corrections=1, show_progressbar=False, seeds=seeds)
    assert torch.equal(first, again)
    assert pipe._batch_cache[2] is rt and rt.engine is eng and rt.points is pts  # neither engine nor plans rebuilt
    _condition(sfs[1], "combined", C, 5)  # member 1 gets another observation
    third = pipe.sample_batch(sfs, noise, steps=2, corrections=1, show_progressbar=False, seeds=seeds)
    assert pipe._batch_cache[2] is rt and rt.engine is eng and rt.points is not pts
    assert torch.equal(third[0], first[0]) and torch.equal(third[2], first[2])
    assert not torch.equal(third[1], first[1])
    one = pipe.sample(sfs[1], noise[1], steps=2, corrections=1, show_progressbar=False, seed=seeds[1])
    assert torch.equal(third[1], one)
