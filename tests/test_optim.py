"""N2, optimiser half (SURVEY.md §8(f)): `optimizer.step()` + `ema.update()` of training_loop.py:381-390 as one fused
pass (`c2w_adamw_ema_step`, climate2weather_b200/optim.py).

CPU: the oracle (oracle/optim_ref.py) is pinned against torch.optim.AdamW itself and, where C2W_REFERENCE names a
checkout of the reference, against the reference's own thor/ema.py.  GPU (`-m gpu`): the fused kernel against the
oracle over several steps with a changing learning rate, gradients set directly and through autograd, and its HBM rate
at the reference model's 72.1 M parameters.
"""
import importlib.util
import os
import pathlib

import pytest
import torch

from oracle import optim_ref

REF = os.environ.get("C2W_REFERENCE")  # a checkout of schmidtjonathan/Climate2Weather
REF_EMA = pathlib.Path(REF, "src/thor/ema.py") if REF else None
HP = dict(lr=3e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-3)  # train.py:176-181


def _tiny_net(seed=0):
    torch.manual_seed(seed)
    return torch.nn.Sequential(torch.nn.Conv2d(3, 5, 3, padding=1), torch.nn.SiLU(), torch.nn.Flatten(),
                               torch.nn.Linear(5 * 4 * 4, 7), torch.nn.Linear(7, 1, bias=False))


def _grads(params, step):
    g = torch.Generator().manual_seed(100 + step)
    return [torch.randn(p.shape, generator=g, dtype=torch.float64) * (0.1 + 0.05 * step) for p in params]


# ---------------------------------------------------------------------------------------------------- CPU
def test_oracle_matches_torch_adamw():
    net = _tiny_net().double()
    params = list(net.parameters())
    ref = optim_ref.AdamWEMARef(params, **HP)
    opt = torch.optim.AdamW(params, **HP)
    for step in range(6):
        lr = HP["lr"] * (1.0 - step / 10.0)  # linear schedule, re-set every step like training_loop.py:380-382
        for g in opt.param_groups:
            g["lr"] = lr
        ref.lr = lr
        grads = _grads(params, step)
        for p, g in zip(params, grads):
            p.grad = g.clone()
        opt.step()
        ref.step(grads)
        for p, q in zip(params, ref.p):
            assert torch.allclose(p.detach(), q, rtol=1e-12, atol=1e-14)


def test_oracle_ema_matches_torch_ema():
    """The oracle's EMA over 5 compounding AdamW steps, element for element, against torch's own EMA
    (torch.optim.swa_utils.get_ema_multi_avg_fn): W_0 = the initial weights, W_t+1 = rate W_t + (1 - rate) p_t+1, the
    rule the oracle restates from the reference's StandardEMA (ema.py:14,24-27)."""
    from torch.optim.swa_utils import get_ema_multi_avg_fn

    net = _tiny_net().double()
    params = list(net.parameters())
    ema = [p.detach().clone() for p in params]
    ema_update = get_ema_multi_avg_fn(0.99)
    ref = optim_ref.AdamWEMARef(params, ema_rate=0.99, **HP)
    opt = torch.optim.AdamW(params, **HP)
    for step in range(5):
        grads = _grads(params, step)
        for p, g in zip(params, grads):
            p.grad = g.clone()
        opt.step()
        ema_update(ema, [p.detach() for p in params], step)
        ref.step(grads)
    for p, q in zip(ema, ref.ema):
        assert torch.allclose(p, q, rtol=1e-12, atol=1e-14)


@pytest.mark.skipif(REF_EMA is None or not REF_EMA.exists(), reason="C2W_REFERENCE does not name a reference checkout")
def test_oracle_ema_matches_reference_ema():
    spec = importlib.util.spec_from_file_location("_ref_ema", REF_EMA)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)  # the reference's own StandardEMA
    net = _tiny_net().double()
    params = list(net.parameters())
    ema = mod.StandardEMA(net, rates=[0.99])
    ref = optim_ref.AdamWEMARef(params, ema_rate=0.99, **HP)
    opt = torch.optim.AdamW(params, **HP)
    for step in range(5):
        grads = _grads(params, step)
        for p, g in zip(params, grads):
            p.grad = g.clone()
        opt.step()
        ema.update(cur_ndata=0, batch_size=1)
        ref.step(grads)
    for p, q in zip(ema.emas[0].parameters(), ref.ema):
        assert torch.allclose(p.detach(), q, rtol=1e-12, atol=1e-14)


def test_optimizer_has_no_cpu_path():
    from climate2weather_b200 import _lib, optim

    with pytest.raises((_lib.C2WError, OSError)):
        optim.AdamW(_tiny_net().parameters(), **HP)


# ---------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("fused_ema", [True, False])
def test_fused_adamw_ema_vs_oracle(fused_ema):
    from climate2weather_b200 import optim

    dev = torch.device("cuda:0")
    net = _tiny_net(1).to(dev)
    cpu_params = [p.detach().cpu() for p in net.parameters()]
    ref = optim_ref.AdamWEMARef(cpu_params, ema_rate=0.99, **HP)
    opt = optim.AdamW(net.parameters(), loss_scaling=4.0, **HP)
    ema = optim.StandardEMA(net, rates=[0.99])
    if fused_ema:
        opt.fuse_ema(ema)
    x = torch.randn(2, 3, 4, 4, generator=torch.Generator().manual_seed(9)).to(dev)
    for step in range(6):
        lr = HP["lr"] * (1.0 - step / 10.0)
        for g in opt.param_groups:
            g["lr"] = lr
        ref.lr = lr
        opt.zero_grad()
        if step < 4:  # gradients written into the flat views directly
            grads = _grads(cpu_params, step)
            for p, g in zip(net.parameters(), grads):
                p.grad.copy_(g.to(dev).float())
        else:         # gradients accumulated by autograd (two backward passes, like gradient accumulation rounds)
            for _ in range(2):
                (net(x) ** 2).mean().mul(4.0).backward()
            grads = [p.grad.detach().cpu().double() for p in net.parameters()]
        opt.step()
        ema.update(cur_ndata=0, batch_size=1)
        ref.step(grads, grad_scale=0.25)
        for p, q in zip(net.parameters(), ref.p):
            assert torch.allclose(p.detach().cpu().double(), q, rtol=2e-5, atol=2e-7), step
    for p, q in zip(ema.emas[0].parameters(), ref.ema):
        assert torch.allclose(p.detach().cpu().double(), q, rtol=2e-5, atol=2e-7)
    out = net(x)  # the module still runs on its (flat-buffer) parameters
    assert torch.isfinite(out).all()


@pytest.mark.gpu
def test_fused_adamw_ema_rate():
    import ctypes

    from climate2weather_b200 import _lib

    lib = _lib.load()
    dev = torch.device("cuda:0")
    n = 72_100_000  # parameters of the reference ScoreUNet (sda_unet.yml)
    bufs = [torch.randn(n, device=dev) * 0.01 for _ in range(2)] + [torch.zeros(n, device=dev) for _ in range(2)]
    p, g, m, v = bufs
    ema = p.clone()
    hp = _lib.AdamW(3e-4, 0.9, 0.999, 1e-8, 1e-3, 0.9999, 1.0, 1)
    st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    call = lambda: lib.c2w_adamw_ema_step(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), ema.data_ptr(), n,
                                          ctypes.byref(hp), st)
    for _ in range(2):
        assert call() == 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        call()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    gbs = 36.0 * n / ms / 1e6
    print(f"\nc2w_adamw_ema_step: {n / 1e6:.1f} M parameters, {ms:.3f} ms, {gbs:.0f} GB/s (36 B per parameter)")
    assert torch.isfinite(p).all() and gbs > 2000


@pytest.mark.gpu
def test_engine_repacks_after_optimizer_and_ema_steps():
    """Advisor finding (round 1): the fused step updates the flat buffers through raw pointers, which does not bump
    Tensor._version — the packed-weight engine cache must be invalidated explicitly.  forward -> step -> forward has to
    change, and must equal a forward of a FRESH network holding the updated weights; same for the EMA copy."""
    import climate2weather_b200 as c2w
    from climate2weather_b200 import optim

    dev = torch.device("cuda:0")
    cfg = dict(channels=20, embedding_dim=64, hidden_channels=(64, 128), hidden_blocks=(1, 1), attention_levels=(1,))
    torch.manual_seed(0)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, **cfg).to(dev)
    x = torch.randn(2, 20, 32, 32, generator=torch.Generator().manual_seed(1)).to(dev)
    t = torch.tensor(0.4)
    opt = optim.AdamW(net.parameters(), lr=1e-2, weight_decay=0.0)
    ema = optim.StandardEMA(net, rates=[0.5])
    opt.fuse_ema(ema)
    gout = torch.randn(2, 20, 32, 32, generator=torch.Generator().manual_seed(3)).to(dev)
    with torch.no_grad():
        y0 = net(x, t)
        e0 = ema.emas[0](x, t)
        _, gin0 = net.engine(20, 1, 32, 32, dev, max_windows=2, vjp=True).unet_vjp(x, 0.4, gout)  # packed before the step
    assert torch.equal(y0, e0)
    opt.zero_grad()
    g = torch.Generator().manual_seed(2)
    for p in net.parameters():
        p.grad.copy_(torch.randn(p.shape, generator=g).to(dev))
    opt.step()
    ema.update()
    with torch.no_grad():
        y1 = net(x, t)
        e1 = ema.emas[0](x, t)
    assert not torch.equal(y1, y0) and not torch.equal(e1, e0) and not torch.equal(e1, y1)
    for trained, got in ((net, y1), (ema.emas[0], e1)):
        fresh = c2w.ScoreUNet(activation=torch.nn.SiLU, **cfg)
        fresh.load_state_dict({k: v.detach().cpu().clone() for k, v in trained.state_dict().items()})
        with torch.no_grad():
            want = fresh.to(dev)(x, t)
        assert torch.equal(got, want)
    # the flipped / transposed input-gradient operands are re-packed too
    fresh = c2w.ScoreUNet(activation=torch.nn.SiLU, **cfg)
    fresh.load_state_dict({k: v.detach().cpu().clone() for k, v in net.state_dict().items()})
    _, gin1 = net.engine(20, 1, 32, 32, dev, max_windows=2, vjp=True).unet_vjp(x, 0.4, gout)
    _, want = fresh.to(dev).engine(20, 1, 32, 32, dev, max_windows=2, vjp=True).unet_vjp(x, 0.4, gout)
    assert torch.equal(gin1, want) and not torch.equal(gin1, gin0)


@pytest.mark.gpu
def test_adamw_state_dict_roundtrip_and_pickle():
    """Checkpointing as training_loop.py:131-138 / src/thor/checkpoint.py:17-30 do it: state_dict() in torch.optim
    layout, load_state_dict() restores the moments and the step count (bias correction continues), and the object
    pickles (the ctypes handle is excluded)."""
    import pickle

    from climate2weather_b200 import optim

    dev = torch.device("cuda:0")
    net_a, net_b = _tiny_net(3).to(dev), _tiny_net(3).to(dev)
    a, b = optim.AdamW(net_a.parameters(), **HP), optim.AdamW(net_b.parameters(), **HP)

    def step(opt, net, s):
        opt.zero_grad()
        for p, g in zip(net.parameters(), _grads([q.detach().cpu() for q in net.parameters()], s)):
            p.grad.copy_(g.to(dev).float())
        opt.step()

    for s in range(3):
        step(a, net_a, s)
    sd = a.state_dict()
    assert set(sd) >= {"state", "param_groups"} and sd["param_groups"][0]["params"] == list(range(len(a.params)))
    assert float(sd["state"][0]["step"]) == 3.0
    # resume: fresh optimizer over a copy of the trained parameters
    net_b.load_state_dict(net_a.state_dict())
    b.load_state_dict(pickle.loads(pickle.dumps(sd)))
    assert b.step_count == 3
    step(a, net_a, 3)
    step(b, net_b, 3)
    for p, q in zip(net_a.parameters(), net_b.parameters()):
        assert torch.equal(p, q)
    # a parameter that left the flat buffer is re-adopted instead of silently ignored
    first = next(net_b.parameters())
    first.data = first.data.clone()
    step(a, net_a, 4)
    step(b, net_b, 4)
    for p, q in zip(net_a.parameters(), net_b.parameters()):
        assert torch.equal(p, q)
    c = pickle.loads(pickle.dumps(b))
    assert c.step_count == b.step_count and torch.equal(c.exp_avg, b.exp_avg)
