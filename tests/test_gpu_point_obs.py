"""GPU tests (pytest -m gpu) of guided sampling with point observations (PointObservation, c2w_guided_step_points):
the guidance kernel alone against the oracle's closed form computed from the same GPU score, locality of the correction,
the whole path against the fp32 oracle (same metrics and tolerances as test_other_variable_counts_vs_oracle), bitwise
invariance, hard conditioning, and time sharding against the single-GPU run (2 / 4 devices)."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import pipeline_ref, score_ref, unet_ref

import oracle_op

pytestmark = pytest.mark.gpu

SMALL = dict(channels=20, embedding_dim=64, hidden_channels=(64, 128), hidden_blocks=(1, 2), attention_levels=(1,),
             kernel_size=3)
GAMMA = 0.0007196856730011522
K, L, H, W = 2, 11, 32, 32


def relerr(got, ref):
    got, ref = got.double().cpu(), ref.double().cpu()
    return ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


def rel_l2(got, ref):
    got, ref = got.double().cpu(), ref.double().cpu()
    return ((got - ref).norm() / ref.norm().clamp_min(1e-30)).item()


def _net(C, seed=3):
    import climate2weather_b200 as c2w
    cfg = dict(SMALL, channels=C * (2 * K + 1))
    torch.manual_seed(seed)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, **cfg)
    ref = unet_ref.RefNet({n: v.detach().clone() for n, v in net.state_dict().items()}, cfg)
    return net.to("cuda:0"), ref


def _points(C, n_frames=L, frames=(9, 0, 3, 4, 10), P=150, seed=7):
    """Irregular observed frames, duplicated pixels, corners, strip borders and a mask with a fully masked point.
    Returns the operator, y with NaN under the mask, and the same y with zeros there (what the reference needs)."""
    import climate2weather_b200 as c2w
    g = torch.Generator().manual_seed(seed + C)
    rows = torch.randint(0, H, (P,), generator=g)
    cols = torch.randint(0, W, (P,), generator=g)
    rows[:6] = torch.tensor([5, 5, 0, H - 1, 15, 16])
    cols[:6] = torch.tensor([7, 7, 0, W - 1, 3, 3])
    mask = torch.rand(len(frames), C, P, generator=g) > 0.25
    mask[:, :, 6] = False
    op = c2w.PointObservation(list(frames), rows, cols, mask)
    y = torch.randn(len(frames), C, P, generator=g)
    y_nan = y.masked_fill(~mask, float("nan"))
    return op, y_nan, y.masked_fill(~mask, 0.0)


def _std(C):
    """Per-variable std, shaped to broadcast against y [F, C, P] in the oracle (the package takes any shape)."""
    return torch.tensor([0.1 + 0.05 * c for c in range(C)]).reshape(1, C, 1)


@pytest.mark.parametrize("C", [4, 3, 1, 8])
def test_point_guidance_kernel_vs_closed_form(C):
    """sf(x, t) - eps (the kernel's correction) against the oracle's A^T((y - A x0)/var) through torch.func.vjp of the
    same operator, from the same GPU eps: fp32 elementwise -> 1e-5; one predictor step the same way; the correction is
    exactly zero (eps_g == eps bit for bit) on frames and at pixels without an observation."""
    import climate2weather_b200 as c2w
    net, _ = _net(C)
    op, y, y0 = _points(C)
    g = torch.Generator().manual_seed(21 + C)
    x = torch.randn(L, C, H, W, generator=g)
    std = _std(C)
    pipe = c2w.SDAPipeline()
    sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=pipe)
    t = torch.tensor(0.45)
    eps = sf.score_fn(x.cuda(), t).cpu()
    sf.condition_on(A=op, y=y, std=std, gamma=GAMMA, exact_grad=False)
    got = sf(x.cuda(), t).cpu()
    want = oracle_op.guided_score_closed_form_op(eps, x, t, y0, std, GAMMA, op)
    e = relerr(got - eps, want - eps)
    print(f"\nC={C}: kernel correction rel-err {e:.3e}")
    assert e < 1e-5, e
    touched = torch.zeros(L, 1, H, W, dtype=torch.bool)
    touched[op.frames[:, None], 0, op.rows[None, :], op.cols[None, :]] = True
    untouched = (~touched).expand(L, C, H, W)
    assert torch.equal(got[untouched], eps[untouched])
    assert not torch.equal(got, eps)
    # one fused guidance + predictor step from t to t - 0.1 on the resident state
    mu, sigma = pipe.mu(t), pipe.sigma(t)
    mu_n, sigma_n = pipe.mu(t - 0.1), pipe.sigma(t - 0.1)
    want_x = mu_n * (x - sigma * want) / mu + sigma_n * want
    rt = sf.runtime(x.cuda())
    rt.load(x.cuda())
    rt.score(float(t))
    rt.predictor(float(mu), float(sigma), float(mu_n), float(sigma_n))
    got_x = rt.owned(rt.x).cpu()
    ex = relerr(got_x, want_x)
    assert ex < 1e-5, ex


@pytest.mark.parametrize("C", [4, 3])
def test_point_guided_path_vs_oracle(C):
    """The whole path against the fp32 oracle with the same operator object (reference log_p + autograd): closed-form
    guided score, a 3-step predictor-corrector run with the reference's noise draws, exact_grad with one stashing chunk
    and with several — the tolerances of test_other_variable_counts_vs_oracle."""
    import climate2weather_b200 as c2w
    net, ref = _net(C, seed=11 + C)
    op, y, y0 = _points(C)
    g = torch.Generator().manual_seed(50 + C)
    x = torch.randn(L, C, H, W, generator=g)
    std = _std(C)
    t = torch.tensor(0.45)
    pipe = c2w.SDAPipeline()
    sf = c2w.BatchedScoreFunction(net, markov_order=K, noise_process=pipe, batch_size=4, device="cuda:0")
    sf.condition_on(A=op, y=y, std=std, gamma=GAMMA, exact_grad=False)
    with torch.no_grad():
        want_g = oracle_op.guided_score_op(ref, x, t, K, y0, std, GAMMA, op, exact_grad=False)
    eg = relerr(sf(x, t), want_g)
    assert eg < 3e-2, eg
    ref_pipe = pipeline_ref.RefPipeline()
    score = lambda xx, tt: oracle_op.guided_score_op(ref, xx, tt, K, y0, std, GAMMA, op, exact_grad=False)
    torch.manual_seed(5)
    want_s = ref_pipe.sample(score, x, steps=3, corrections=1, tau=0.5)
    pipe.rng = "reference"
    torch.manual_seed(5)
    got_s = pipe.sample(sf, x, steps=3, corrections=1, tau=0.5, show_progressbar=False)
    es, ls = relerr(got_s, want_s), rel_l2(got_s, want_s)
    want_e = oracle_op.guided_score_op(ref, x, t, K, y0, std, GAMMA, op, exact_grad=True)
    d = relerr(want_g, want_e)
    ee = []
    for mw in (None, 2):
        sfe = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=c2w.SDAPipeline())
        sfe.max_windows = mw
        sfe.condition_on(A=op, y=y, std=std, gamma=GAMMA, exact_grad=True)
        ee.append(relerr(sfe(x.cuda(), t).cpu(), want_e))
    print(f"\nC={C}: guided {eg:.3e}, sampler max-abs ratio {es:.3e} rel-L2 {ls:.3e}, exact {ee} "
          f"(closed vs exact {d:.3e})")
    assert got_s.shape == x.shape and es < 5e-2 and ls < 3e-2
    for e in ee:
        assert e < 4e-2 and e < 0.5 * d, (ee, d)


def test_point_guidance_is_bitwise_invariant():
    """Bit-identical across windows per launch and across repeated runs (no atomics on data)."""
    import climate2weather_b200 as c2w
    net, _ = _net(4)
    op, y, _ = _points(4)
    x = torch.randn(L, 4, H, W, generator=torch.Generator().manual_seed(2))
    t = torch.tensor(0.3)
    outs, samples = [], []
    for mw in (None, 3, None):
        pipe = c2w.SDAPipeline()
        sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=pipe)
        sf.max_windows = mw
        sf.condition_on(A=op, y=y, std=0.1, gamma=GAMMA, exact_grad=False)
        outs.append(sf(x.cuda(), t).cpu())
        samples.append(pipe.sample(sf, x, steps=3, corrections=1, tau=0.5, show_progressbar=False, seed=9).cpu())
    for o in outs[1:]:
        assert torch.equal(o, outs[0])
    for s in samples[1:]:
        assert torch.equal(s, samples[0])
    assert torch.isfinite(samples[0]).all()


def test_hard_conditioning_pins_the_observed_frames():
    """Every pixel of frames 0..k-1 observed with std 1e-3: the sampled frames end on y.  gamma = 1 keeps the
    Tweedie update from overshooting while sigma/mu is large (weight r^2 / (std^2 + gamma r^2) <= 1/gamma); at the
    last step r^2 >> std^2, so x0 is y to ~1e-4 and the final x is y + sigma(0) eps_g with sigma(0) = eta = 1e-3."""
    import climate2weather_b200 as c2w
    net, _ = _net(4)
    rr, cc = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    op = c2w.PointObservation(list(range(K)), rr.reshape(-1), cc.reshape(-1))
    g = torch.Generator().manual_seed(13)
    y = torch.randn(K, 4, H * W, generator=g)
    noise = torch.randn(L, 4, H, W, generator=g)
    pipe = c2w.SDAPipeline()
    sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=pipe)
    sf.condition_on(A=op, y=y, std=1e-3, gamma=1.0, exact_grad=False)
    out = pipe.sample(sf, noise, steps=16, show_progressbar=False, device="cuda:0").cpu()
    err = (op(out) - y).abs().max().item()
    free = (out[K:].std()).item()
    print(f"\nhard conditioning: max |A x - y| = {err:.3e} (unobserved frames std {free:.3f})")
    assert err < 5e-2, err


# ------------------------------------------------------------------------------------------------ time sharding
def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _problem(Ls):
    import climate2weather_b200 as c2w
    torch.manual_seed(3)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, **SMALL)
    g = torch.Generator().manual_seed(11)
    noise = torch.randn(Ls, 4, 32, 32, generator=g)
    frames = [0, 1, 5, 6, 11, 12, 16, Ls - 1]  # shard boundaries fall between and on observed frames
    rows = torch.randint(0, 32, (200,), generator=g)
    cols = torch.randint(0, 32, (200,), generator=g)
    mask = torch.rand(len(frames), 4, 200, generator=g) > 0.2
    op = c2w.PointObservation(frames, rows, cols, mask)
    y = torch.randn(len(frames), 4, 200, generator=g).masked_fill(~mask, float("nan"))
    return net, noise, op, y


def _sample(net, noise, op, y, dev, corrections, shard, exact=False):
    import climate2weather_b200 as c2w
    pipe = c2w.SDAPipeline()
    sf = c2w.BatchedScoreFunction(net.to(dev), markov_order=2, noise_process=pipe, batch_size=5, device=dev)
    sf.condition_on(A=op, y=y, std=0.1, gamma=1e-3, exact_grad=exact)
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
        net, noise, op, y = _problem(Ls)
        for corr in (0, 1):
            out = _sample(net, noise, op, y, dev, corr, shard=True)
            if rank == 0:
                torch.save(out.cpu(), os.path.join(out_dir, f"sharded_c{corr}.pt"))
        out = _sample(net, noise, op, y, dev, 0, shard=True, exact=True)
        if rank == 0:
            torch.save(out.cpu(), os.path.join(out_dir, "sharded_exact.pt"))
        os.environ["C2W_HALO"] = "nccl"
        out = _sample(net, noise, op, y, dev, 0, shard=True)
        if rank == 0:
            torch.save(out.cpu(), os.path.join(out_dir, "sharded_c0_nccl.pt"))
        os.environ["C2W_HALO"] = "p2p"
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4])
def test_time_sharded_point_sampling_matches_single_gpu(tmp_path, world):
    """Each rank plans its own frames; bit-exact for predictor steps over both halo transports, 1e-5 with a
    correction (the global mean(eps^2) sums in another order), 1e-4 with exact_grad (reverse halo accumulation)."""
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    Ls = 23
    net, noise, op, y = _problem(Ls)
    dev = torch.device("cuda:0")
    ref = {c: _sample(net, noise, op, y, dev, c, shard=False).cpu() for c in (0, 1)}
    mp.spawn(_worker, args=(world, _free_port(), Ls, str(tmp_path)), nprocs=world, join=True)
    got0 = torch.load(tmp_path / "sharded_c0.pt")
    got1 = torch.load(tmp_path / "sharded_c1.pt")
    assert torch.isfinite(got0).all() and torch.isfinite(got1).all()
    assert torch.equal(got0, ref[0]), float((got0 - ref[0]).abs().max())
    assert torch.equal(torch.load(tmp_path / "sharded_c0_nccl.pt"), ref[0])
    rel = ((got1 - ref[1]).abs().max() / ref[1].abs().max()).item()
    assert rel < 1e-5, rel
    want = _sample(net, noise, op, y, dev, 0, shard=False, exact=True).cpu()
    gote = torch.load(tmp_path / "sharded_exact.pt")
    rel = ((gote - want).abs().max() / want.abs().max()).item()
    assert rel < 1e-4, rel
    assert not torch.equal(want, ref[0])
