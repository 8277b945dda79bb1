"""The sampling and training paths at 256 x 256 (a net with 512-channel attention at its deepest level: 256 tokens, the
tiled attention kernels): composed window score, closed-form and exact guided score and a 3-step predictor-corrector
run against the fp32 oracle with CoarseGrain and PointObservation; a training step's parameter gradients against fp32
autograd; sample() bit-identical across max_windows; sample_ensemble members bit-identical to their own runs; a
time-sharded run bit-identical to one GPU (skipped below 2 GPUs)."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle_op
from oracle import pipeline_ref, score_ref, unet_ref

pytestmark = pytest.mark.gpu

C, K, L, H, W = 4, 1, 5, 256, 256
NET = dict(channels=C * (2 * K + 1), embedding_dim=64, hidden_channels=(64, 64, 64, 64, 512),
           hidden_blocks=(1, 1, 1, 1, 1), attention_levels=(4,), kernel_size=3)
GAMMA = 0.0007196856730011522


def relerr(got, ref):
    got, ref = got.double().cpu(), ref.double().cpu()
    return ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


def rel_l2(got, ref):
    got, ref = got.double().cpu(), ref.double().cpu()
    return ((got - ref).norm() / ref.norm().clamp_min(1e-30)).item()


def _net(seed=3, cfg=NET):
    import climate2weather_b200 as c2w
    torch.manual_seed(seed)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, **cfg)
    ref = unet_ref.RefNet({n: v.detach().clone() for n, v in net.state_dict().items()}, cfg)
    return net.to("cuda:0"), ref


def _operator(kind, seed=7):
    """(operator, y for the package, y for the oracle, std broadcasting against y in the oracle)."""
    import climate2weather_b200 as c2w
    g = torch.Generator().manual_seed(seed)
    if kind == "coarse":
        op = c2w.CoarseGrain(2, 16)
        y = torch.randn(-(-L // 2), C, H // 16, W // 16, generator=g)
        return op, y, y, torch.tensor([0.1 + 0.05 * c for c in range(C)]).reshape(1, C, 1, 1)
    P = 300
    rows, cols = torch.randint(0, H, (P,), generator=g), torch.randint(0, W, (P,), generator=g)
    rows[:4], cols[:4] = torch.tensor([0, H - 1, 128, 128]), torch.tensor([0, W - 1, 127, 128])
    mask = torch.rand(3, C, P, generator=g) > 0.25
    op = c2w.PointObservation([4, 0, 2], rows, cols, mask)
    y = torch.randn(3, C, P, generator=g)
    return op, y.masked_fill(~mask, float("nan")), y.masked_fill(~mask, 0.0), \
        torch.tensor([0.1 + 0.05 * c for c in range(C)]).reshape(1, C, 1)


@pytest.mark.parametrize("kind", ["coarse", "points"])
def test_guided_paths_vs_oracle(kind):
    """The tolerances of test_other_variable_counts_vs_oracle and test_point_guided_path_vs_oracle."""
    import climate2weather_b200 as c2w
    dev = torch.device("cuda:0")
    net, ref = _net(11)
    op, y, y0, std = _operator(kind)
    x = torch.randn(L, C, H, W, generator=torch.Generator().manual_seed(50))
    t = torch.tensor(0.45)
    pipe = c2w.SDAPipeline()
    with torch.no_grad():
        want = score_ref.window_score(ref, x, t, K)
    sf0 = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=pipe)
    e = relerr(sf0.score_fn(x.to(dev), t).cpu(), want)
    assert e < 3e-2, e
    sf = c2w.BatchedScoreFunction(net, markov_order=K, noise_process=pipe, batch_size=2, device=dev)
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
    assert got_s.shape == x.shape and es < 5e-2 and ls < 3e-2, (es, ls)
    want_e = oracle_op.guided_score_op(ref, x, t, K, y0, std, GAMMA, op, exact_grad=True)
    d = relerr(want_g, want_e)
    for mw in (None, 2):
        sfe = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=c2w.SDAPipeline())
        sfe.max_windows = mw
        sfe.condition_on(A=op, y=y, std=std, gamma=GAMMA, exact_grad=True)
        ee = relerr(sfe(x.to(dev), t).cpu(), want_e)
        assert ee < 4e-2 and ee < 0.5 * d, (mw, ee, d)


def test_sample_and_ensemble_bit_identical():
    """sample() is bit-identical across max_windows, and each sample_ensemble member to its own run."""
    import climate2weather_b200 as c2w
    net, _ = _net(3)
    op, y, _, std = _operator("coarse")
    pipe = c2w.SDAPipeline()
    noise = torch.randn(2, L, C, H, W, generator=torch.Generator().manual_seed(7))
    seeds = [11, 12345]
    runs = []
    for mw in (None, 1, 2):
        sf = c2w.DefaultScoreFunction(net, markov_order=K, noise_process=pipe)
        sf.max_windows = mw
        sf.condition_on(A=op, y=y, std=std, gamma=GAMMA, exact_grad=False)
        runs.append(pipe.sample(sf, noise[0], steps=3, corrections=1, tau=0.5, show_progressbar=False, seed=seeds[0]))
        if mw is None:
            ens = pipe.sample_ensemble(sf, noise, steps=3, corrections=1, tau=0.5, show_progressbar=False, seeds=seeds)
            for m in range(2):
                one = pipe.sample(sf, noise[m], steps=3, corrections=1, tau=0.5, show_progressbar=False, seed=seeds[m])
                assert torch.equal(ens[m], one), m
    assert torch.isfinite(runs[0]).all()
    assert torch.equal(runs[0], runs[1]) and torch.equal(runs[0], runs[2])


def test_training_step_gradients_vs_oracle():
    """Batch 2 at 256 x 256: loss and every parameter gradient against the fp32 oracle's autograd."""
    import climate2weather_b200 as c2w
    dev = torch.device("cuda:0")
    cfg = dict(NET, channels=20)
    torch.manual_seed(0)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, **cfg)
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in net.state_dict().items()}
    net = net.to(dev)
    g = torch.Generator().manual_seed(4)
    x = torch.randn(2, 20, H, W, generator=g)
    t = torch.tensor([0.15, 0.8]).reshape(2, 1, 1, 1)
    eps = torch.randn(2, 20, H, W, generator=g)
    pipe = c2w.SDAPipeline()
    xt = pipe.mu(t) * x + pipe.sigma(t) * eps
    out = net(xt.to(dev), t.to(dev))
    loss = ((out - eps.to(dev)) ** 2).mean()
    loss.backward()
    want_loss = pipeline_ref.RefPipeline().loss(unet_ref.RefNet(sd, cfg), x, t=t, eps=eps).mean()
    want = dict(zip(sd.keys(), torch.autograd.grad(want_loss, list(sd.values()))))
    assert abs(loss.item() - want_loss.item()) <= 2e-3 * want_loss.item()
    errs = {n: rel_l2(p.grad, want[n]) for n, p in net.named_parameters()}
    worst = max(errs, key=errs.get)
    assert errs[worst] <= 5e-2, (worst, errs[worst])


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _sample(net, noise, op, y, std, dev, shard):
    import climate2weather_b200 as c2w
    pipe = c2w.SDAPipeline()
    sf = c2w.BatchedScoreFunction(net.to(dev), markov_order=K, noise_process=pipe, batch_size=2, device=dev)
    sf.condition_on(A=op, y=y, std=std, gamma=GAMMA, exact_grad=False)
    if shard:
        sf.enable_time_sharding()
    return pipe.sample(sf, noise, steps=3, corrections=0, tau=0.5, show_progressbar=False, seed=77)


def _shard_problem():
    torch.manual_seed(3)
    import climate2weather_b200 as c2w
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, **NET)
    op, y, _, std = _operator("points")
    noise = torch.randn(L + 4, C, H, W, generator=torch.Generator().manual_seed(9))
    return net, noise, op, y, std


def _worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        net, noise, op, y, std = _shard_problem()
        out = _sample(net, noise, op, y, std, dev, shard=True)
        if rank == 0:
            torch.save(out.cpu(), os.path.join(out_dir, "sharded.pt"))
    finally:
        dist.destroy_process_group()


def test_time_sharded_matches_single_gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    net, noise, op, y, std = _shard_problem()
    want = _sample(net, noise, op, y, std, torch.device("cuda:0"), shard=False).cpu()
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    assert torch.equal(torch.load(tmp_path / "sharded.pt"), want)
