"""GPU tests (pytest -m gpu) of ensemble sampling (SDAPipeline.sample_ensemble): the member-major gather and fold with
index-coded networks (integers out, any chunking of the windows over launches), the contract that member m equals
sample(noise[m], seed=seeds[m]) bit for bit for every operator, the member kernels (segmented reduction, member
corrector, member guidance step) against the single-trajectory entry points member by member, and the NaN error."""
import numpy as np
import pytest
import torch

from oracle import score_ref
from test_gpu_parity import _index_coded_net

pytestmark = pytest.mark.gpu

SMALL = dict(embedding_dim=64, hidden_channels=(64, 128), hidden_blocks=(1, 2), attention_levels=(1,), kernel_size=3)
K, L, H, W = 2, 11, 32, 32
GAMMA = 0.0007196856730011522


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


# ------------------------------------------------------------------------------------------------ gather + fold
@pytest.mark.parametrize("C", [4, 3])
@pytest.mark.parametrize("Lm,M", [(Lm, M) for Lm in (13, 14, 26) for M in (1, 2, 3)])
def test_member_gather_and_fold_index_bit_exact(dev, C, Lm, M):
    """c2w_window_score_members on index-coded networks at k = 6: every frame of every member must hold, as an integer,
    the (window, window-channel, pixel) the reference's fold of that member alone names — for chunkings where one launch
    holds windows of two or three members, with a ragged last chunk (K0 tiled per member for C = 4; K1's compose
    epilogue for C = 4, compose_generic_kernel for C = 3)."""
    k, Hh, Ww = 6, 64, 64
    nw = Lm - 2 * k
    n = M * nw
    f = score_ref.fold_index(Lm, k, C)
    frames = torch.arange(M * Lm, dtype=torch.float32).reshape(M * Lm, 1, 1, 1).expand(M * Lm, Hh, Ww, C).contiguous()
    hh, ww, cc = torch.meshgrid(torch.arange(Hh), torch.arange(Ww), torch.arange(C), indexing="ij")
    pix = ((hh * Ww + ww + 64 * cc + 17 * torch.arange(M * Lm).reshape(-1, 1, 1, 1)) % 251).float()  # [F, H, W, C]
    member_base = (torch.arange(M) * Lm).repeat_interleave(Lm).reshape(-1, 1, 1, 1).float()
    want = {
        "window": member_base + torch.from_numpy(f[..., 0]).float().repeat(M, 1).reshape(M * Lm, 1, 1, C),
        "slot": torch.from_numpy(f[..., 1]).float().repeat(M, 1).reshape(M * Lm, 1, 1, C).expand(M * Lm, Hh, Ww, C),
        "pixel": pix,
    }
    chunks = sorted({1, 5, nw + 1, 2 * nw - 1, n})  # n: one launch for the whole ensemble
    for mode in ("window", "slot", "pixel"):
        net = _index_coded_net(dev, k, C, mode)
        x = (pix if mode == "pixel" else frames).to(dev)
        for mw in chunks:
            eng = net.engine(C, 2 * k + 1, Hh, Ww, dev, max_windows=mw, vjp=False)
            eps = torch.full_like(x, float("nan"))
            eng.window_score_members(x, M, Lm, 0, n, 0.5, eps)
            torch.cuda.synchronize()
            got = eps.cpu()
            exp = want[mode].expand_as(got)
            assert torch.equal(got, exp), (mode, mw, (got != exp).nonzero()[:4].tolist())


# ------------------------------------------------------------------------------------------------ the contract
def _net(C, seed=3):
    import climate2weather_b200 as c2w
    torch.manual_seed(seed)
    return c2w.ScoreUNet(activation=torch.nn.SiLU, channels=C * (2 * K + 1), **SMALL).to("cuda:0")


def _condition(sf, kind, C):
    """Conditions sf on one operator of each kind the fused path runs (the same observation for every member)."""
    import climate2weather_b200 as c2w
    g = torch.Generator().manual_seed(40 + C)
    P = 60
    rows, cols = torch.randint(0, H, (P,), generator=g), torch.randint(0, W, (P,), generator=g)
    rows[1], cols[1] = rows[0], cols[0]
    mask = torch.rand(4, C, P, generator=g) > 0.25
    pts = c2w.PointObservation([9, 0, 3, 10], rows, cols, mask)
    py = torch.randn(4, C, P, generator=g).masked_fill(~mask, float("nan"))
    cg = c2w.CoarseGrain(3, 8)
    cy = torch.randn(-(-L // 3), C, H // 8, W // 8, generator=g)
    std = [0.1 + 0.05 * c for c in range(C)]
    if kind == "none":
        return
    if kind == "coarse":
        sf.condition_on(A=cg, y=cy, std=std, gamma=GAMMA, exact_grad=False)
    elif kind == "coarse_opaque":  # recognised as AvgPool2d(s)(x[::t])
        sf.condition_on(A=lambda x: torch.nn.functional.avg_pool2d(x[::3], 8), y=cy, std=0.2, gamma=GAMMA,
                        exact_grad=False)
    elif kind == "points":
        sf.condition_on(A=pts, y=py, std=torch.tensor(std).reshape(1, C, 1), gamma=GAMMA, exact_grad=False)
    elif kind == "combined":
        op = c2w.CombinedObservation(cg, pts)
        shape = (L, C, H, W)
        sf.condition_on(A=op, y=op.pack(cy, py, shape), std=op.pack(0.3, torch.tensor(std), shape), gamma=GAMMA,
                        exact_grad=False)
    elif kind == "coarse_std_tile":
        s = 0.05 + torch.rand(1, 1, H // 8, W // 8, generator=g)
        sf.condition_on(A=cg, y=cy, std=s, gamma=GAMMA, exact_grad=False)
    elif kind == "points_std_station":
        s = 0.05 + torch.rand(1, 1, P, generator=g)
        sf.condition_on(A=pts, y=py, std=s.expand(4, C, P), gamma=GAMMA, exact_grad=False)
    elif kind == "combined_std_obs":
        op = c2w.CombinedObservation(cg, pts)
        shape = (L, C, H, W)
        s = op.pack(0.05 + torch.rand(cy.shape, generator=g), 0.05 + torch.rand(4, C, P, generator=g), shape)
        sf.condition_on(A=op, y=op.pack(cy, py, shape), std=s, gamma=GAMMA, exact_grad=False)
    else:
        raise ValueError(kind)


KINDS = ["none", "coarse", "coarse_opaque", "points", "combined", "coarse_std_tile", "points_std_station",
         "combined_std_obs"]


@pytest.mark.parametrize("corrections", [0, 2])
@pytest.mark.parametrize("C", [4, 3])
@pytest.mark.parametrize("kind", KINDS)
def test_ensemble_equals_sequential_samples(kind, C, corrections):
    """Member m of sample_ensemble(noise, seeds=s) is bit-identical to sample(noise[m], seed=s[m]) with the same
    max_windows: the default (one launch of 21 windows for the ensemble, 7 per member) and 4, which splits members
    across launches.  max_windows is read when a score function builds its runtime: a fresh one per setting."""
    import climate2weather_b200 as c2w
    net = _net(C)
    pipe = c2w.SDAPipeline()
    M = 3
    noise = torch.randn(M, L, C, H, W, generator=torch.Generator().manual_seed(7))
    seeds = [11, 2 ** 40 + 3, 12345]
    for mw in (None, 4):
        sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=pipe)
        sf.max_windows = mw
        _condition(sf, kind, C)
        ens = pipe.sample_ensemble(sf, noise, steps=3, corrections=corrections, show_progressbar=False, seeds=seeds)
        assert ens.shape == noise.shape and ens.device == noise.device
        assert sf.runtime(noise, members=M).engine.max_windows == (mw or M * (L - 2 * K))
        for m in range(M):
            one = pipe.sample(sf, noise[m], steps=3, corrections=corrections, show_progressbar=False, seed=seeds[m])
            assert torch.equal(ens[m], one), (kind, C, corrections, mw, m)


@pytest.mark.parametrize("M,max_windows", [(2, None), (3, None), (3, 20)])
def test_ensemble_keeps_a_members_conv_tile_widths(M, max_windows):
    """K1's tile width is picked from the windows per launch, and it decides the main loop and the order of the fp32
    sums.  With 384 channels at 16 x 16 a member's 37 windows and an ensemble's 74 or 111 pick different widths; the
    ensemble workspace must still plan a member's, so the members stay bit-identical to their own runs."""
    import climate2weather_b200 as c2w
    from climate2weather_b200 import _lib
    lib = _lib.load()
    assert lib.c2w_conv_tile_width(384, 1, 37, 16, 16, 1, 148) != lib.c2w_conv_tile_width(384, 1, M * 37, 16, 16, 1, 148)
    C, Lm = 4, 41
    torch.manual_seed(5)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, channels=C * (2 * K + 1), embedding_dim=64, hidden_channels=(64, 384),
                        hidden_blocks=(1, 1), attention_levels=(), kernel_size=3).to("cuda:0")
    pipe = c2w.SDAPipeline()
    sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=pipe)
    sf.max_windows = max_windows
    truth = torch.randn(Lm, C, H, W, generator=torch.Generator().manual_seed(1))
    cg = c2w.CoarseGrain(3, 8)
    sf.condition_on(A=cg, y=cg(truth), std=0.2, gamma=GAMMA, exact_grad=False)
    noise = torch.randn(M, Lm, C, H, W, generator=torch.Generator().manual_seed(2))
    seeds = list(range(M))
    ens = pipe.sample_ensemble(sf, noise, steps=2, corrections=1, show_progressbar=False, seeds=seeds)
    for m in range(M):
        one = pipe.sample(sf, noise[m], steps=2, corrections=1, show_progressbar=False, seed=seeds[m])
        assert torch.equal(ens[m], one), (M, max_windows, m)


@pytest.mark.parametrize("M", [3, 4])
def test_ensemble_keeps_a_members_conv_variant(M):
    """The CTA pair and the main loop are picked from the windows per launch too.  With one window per member
    (L = 2k + 1, validation sampling) a 128-channel 8 x 8 level is one M tile: the member's run takes the streamed main
    loop with the fused LayerNorm, while three or more windows would take the two-image activation-reuse loop (another
    order of the fp32 sums) and a separate LayerNorm.  The ensemble must plan the member's variant."""
    import climate2weather_b200 as c2w
    C, Lm = 4, 2 * K + 1
    torch.manual_seed(6)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, channels=C * (2 * K + 1), embedding_dim=64,
                        hidden_channels=(64, 128, 128), hidden_blocks=(1, 1, 1), attention_levels=(),
                        kernel_size=3).to("cuda:0")
    pipe = c2w.SDAPipeline()
    sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=pipe)
    truth = torch.randn(Lm, C, H, W, generator=torch.Generator().manual_seed(3))
    cg = c2w.CoarseGrain(2, 8)
    sf.condition_on(A=cg, y=cg(truth), std=0.2, gamma=GAMMA, exact_grad=False)
    noise = torch.randn(M, Lm, C, H, W, generator=torch.Generator().manual_seed(4))
    seeds = [7 + m for m in range(M)]
    ens = pipe.sample_ensemble(sf, noise, steps=3, corrections=1, show_progressbar=False, seeds=seeds)
    for m in range(M):
        one = pipe.sample(sf, noise[m], steps=3, corrections=1, show_progressbar=False, seed=seeds[m])
        assert torch.equal(ens[m], one), (M, m)


def test_one_member_default_seeds_hook_and_traces():
    """M = 1 and M = 3 with default seeds (drawn in member order, as sequential calls draw them), a proc_x0 hook
    called once per member on [L, C, H, W], and trace_at traces of shape [M, L, C, H, W]."""
    import climate2weather_b200 as c2w
    C = 4
    net = _net(C)
    pipe = c2w.SDAPipeline()
    pipe.trace_at = [2]
    sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=pipe)
    _condition(sf, "points", C)
    shapes = []

    def hook(x0):
        shapes.append(tuple(x0.shape))
        return x0.clamp(-1.5, 1.5)

    for M in (1, 3):
        noise = torch.randn(M, L, C, H, W, generator=torch.Generator().manual_seed(M))
        torch.manual_seed(123)
        singles, traces = [], []
        for m in range(M):
            singles.append(pipe.sample(sf, noise[m], steps=3, corrections=1, proc_x0=hook, show_progressbar=False))
            traces.append(pipe.traces[2])
        shapes.clear()
        torch.manual_seed(123)
        ens = pipe.sample_ensemble(sf, noise, steps=3, corrections=1, proc_x0=hook, show_progressbar=False)
        assert shapes == [(L, C, H, W)] * (3 * M)
        assert pipe.traces[2].shape == (M, L, C, H, W)
        for m in range(M):
            assert torch.equal(ens[m], singles[m]), (M, m)
            assert torch.equal(pipe.traces[2][m], traces[m]), (M, m)


def test_non_finite_member_raises_the_reference_error():
    import climate2weather_b200 as c2w
    net = _net(4)
    pipe = c2w.SDAPipeline()
    sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=pipe)
    noise = torch.randn(3, L, 4, H, W)
    noise[1, 5, 2, 7, 7] = float("inf")
    with pytest.raises(ValueError, match="NaN detected in sample"):
        pipe.sample_ensemble(sf, noise, steps=2, show_progressbar=False)


# ------------------------------------------------------------------------------------------------ the member kernels
def test_segmented_reduction_equals_single_reductions(dev):
    from climate2weather_b200 import _lib
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    for M, seg in ((5, 1000), (3, 7), (4, 300), (1, 4096)):
        parts = (torch.randn(M * seg, generator=torch.Generator().manual_seed(seg)) ** 2 * 1e3).to(dev)
        got = torch.zeros(M, dtype=torch.float64, device=dev)
        _lib.check(lib.c2w_reduce_partials_members(parts.data_ptr(), M, seg, got.data_ptr(), st), "members")
        for m in range(M):
            one = torch.zeros(1, dtype=torch.float64, device=dev)
            _lib.check(lib.c2w_reduce_partials(parts[m * seg:].data_ptr(), seg, one.data_ptr(), st), "single")
            assert torch.equal(got[m:m + 1], one), (M, seg, m)


@pytest.mark.parametrize("C", range(1, 9))
def test_member_corrector_equals_single_corrector(dev, C):
    from climate2weather_b200 import _lib
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    M, npix = 3, 5 * 24 * 24
    g = torch.Generator().manual_seed(C)
    x = torch.randn(M * npix * C, generator=g).to(dev)
    eps = torch.randn(M * npix * C, generator=g).to(dev)
    sumsq = (torch.rand(M, generator=g, dtype=torch.float64) * 1e4 + 1.0).to(dev)
    seeds = [5, 2 ** 63 + 9, 77]
    seeds_dev = torch.from_numpy(np.array(seeds, dtype=np.uint64).view(np.int64)).to(dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    got = x.clone()
    _lib.check(lib.c2w_corrector_update_members(got.data_ptr(), eps.data_ptr(), sumsq.data_ptr(), float(npix * C), 0.7,
                                                0.3, M, npix, C, seeds_dev.data_ptr(), 9, flag.data_ptr(), st), "members")
    for m in range(M):
        want = x[m * npix * C:(m + 1) * npix * C].clone()
        _lib.check(lib.c2w_corrector_update_c(want.data_ptr(), eps[m * npix * C:].data_ptr(), None,
                                              sumsq[m:].data_ptr(), float(npix * C), 0.7, 0.3, 0, npix, C, seeds[m], 9,
                                              flag.data_ptr(), st), "single")
        assert torch.equal(got[m * npix * C:(m + 1) * npix * C], want), (C, m)


@pytest.mark.parametrize("C", range(1, 9))
def test_member_guidance_equals_single_guidance_per_member(C):
    """c2w_guided_step_members (through the runtime's _guide) at modes 0 / 1 / 2 for every operator against the
    single-trajectory entry points on each member's slice: x, eps_g, the partials (one segment per member), the
    cotangent, bit for bit."""
    import climate2weather_b200 as c2w
    net = _net(C)
    pipe = c2w.SDAPipeline()
    M = 3
    for kind in KINDS:
        sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=pipe)
        _condition(sf, kind, C)
        gen = torch.Generator().manual_seed(C)
        x = torch.randn(M, L, C, H, W, generator=gen).cuda()
        eps = torch.randn(M, L, H, W, C, generator=gen).cuda()
        for mode in (0, 1) if kind == "none" else (0, 1, 2):  # mode 2 needs an observation
            ens = sf.runtime(x, members=M)
            ens.load(x)
            ens.eps.copy_(eps.reshape(M * L, H, W, C))
            ens.cot = torch.zeros_like(ens.x)
            ens._guide(mode, 0.8, 0.5, 0.9, 0.4)
            e_x, e_eg, e_cot = ens.x.clone(), None if mode != 1 else ens.eps_g.clone(), ens.cot.clone()
            e_part = ens.partials[:ens._n_part].clone() if mode == 1 else None
            for m in range(M):
                one = sf.runtime(x[m])
                one.load(x[m])
                one.eps.copy_(eps[m])
                one.cot = torch.zeros_like(one.x)
                one._guide(mode, 0.8, 0.5, 0.9, 0.4)
                sl = slice(m * L, (m + 1) * L)
                assert torch.equal(e_x[sl], one.x), (kind, mode, m)
                if mode == 1:
                    assert torch.equal(e_eg[sl], one.eps_g), (kind, mode, m)
                    seg = ens._n_part // M
                    assert seg == one._n_part
                    assert torch.equal(e_part[m * seg:(m + 1) * seg], one.partials[:seg]), (kind, mode, m)
                if mode == 2:
                    assert torch.equal(e_cot[sl], one.cot), (kind, mode, m)
