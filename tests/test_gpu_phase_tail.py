"""The phase form of the ascent tails: conv3x3(nearest x2 (z)) computed at the low resolution as four 2x2 convs, one
per output phase (a, b) of pixel (2i + a, 2j + b), with merged weights (c2w_pack_phase_weights, c2w_op_conv_phase).

- the weight merge against numpy (CPU);
- bit-exact against conv3x3 of the explicitly upsampled input with integer data, where every merged weight, product
  and sum is exact, with and without the residual, at image borders and odd batches, and the fused LayerNorm output
  against the upsampled-input kernel's;
- accuracy against fp64 conv2d(interpolate(z, nearest)) with real-valued data;
- after a parameter change, c2w_refresh_weights re-packs the phase weights as a freshly built engine packs them.
"""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from climate2weather_b200 import _lib


@pytest.fixture(scope="module")
def lib():
    return _lib.load()


def _numpy_phase_weights(w, cin_pad, cout_pad):
    """w: fp32 [cout, cin, 3, 3] -> fp32 [4, cout_pad, 4 * cin_pad] (phase 2a + b, tap 2 tr + ts), merged in fp64."""
    rows = {(0, 0): [0], (0, 1): [1, 2], (1, 0): [0, 1], (1, 1): [2]}  # (phase a, tap tr) -> filter rows
    cout, cin = w.shape[:2]
    out = np.zeros((4, cout_pad, 4, cin_pad))
    for a in range(2):
        for b in range(2):
            for tr in range(2):
                for ts in range(2):
                    m = w[:, :, rows[a, tr]][:, :, :, rows[b, ts]].astype(np.float64).sum(axis=(2, 3))
                    out[2 * a + b, :cout, 2 * tr + ts, :cin] = m
    return out.reshape(4, cout_pad, 4 * cin_pad)


def _pack(lib, w, cin_pad, cout_pad):
    cout, cin = w.shape[:2]
    wc = torch.as_tensor(w, dtype=torch.float32).contiguous()
    out = torch.empty(4, cout_pad, 4 * cin_pad, dtype=torch.bfloat16)
    _lib.check(lib.c2w_pack_phase_weights(wc.data_ptr(), cout, cin, cin_pad, cout_pad, out.data_ptr()),
               "c2w_pack_phase_weights")
    return out


@pytest.mark.parametrize("cout,cin,cin_pad,cout_pad", [(128, 128, 128, 128), (64, 128, 128, 64), (52, 70, 128, 64)])
def test_phase_weight_packing_matches_numpy_merge(lib, cout, cin, cin_pad, cout_pad):
    rng = np.random.default_rng(cout + cin)
    w = rng.standard_normal((cout, cin, 3, 3)).astype(np.float32)
    got = _pack(lib, w, cin_pad, cout_pad).float().numpy()
    want = torch.from_numpy(_numpy_phase_weights(w, cin_pad, cout_pad)).to(torch.bfloat16).float().numpy()
    # one bf16 rounding of the fp32 sum: the rounded fp64 sum, or one bf16 step from it where the two straddle a rounding
    # boundary
    diff = np.abs(got - want)
    assert (diff <= np.abs(want) * 2.0 ** -7 + 1e-30).all()
    assert (diff == 0).mean() > 0.99
    # integer weights: every merge is exact
    wi = rng.integers(-3, 4, (cout, cin, 3, 3)).astype(np.float32)
    assert np.array_equal(_pack(lib, wi, cin_pad, cout_pad).float().numpy(), _numpy_phase_weights(wi, cin_pad, cout_pad))


def _run_phase(lib, dev, z, wph, bias, mode, res=None, ln=False):
    n, H, W, cin = z.shape
    cout = bias.numel()
    out = (res.clone() if mode == 2 else torch.empty(n, 2 * H, 2 * W, cout, dtype=torch.bfloat16, device=dev))
    ln_out = torch.empty_like(out) if ln else None
    d = _lib.ConvDesc()
    d.x, d.n_img, d.H, d.W, d.cin, d.stride, d.conv3x3 = z.data_ptr(), n, H, W, cin, 1, 1
    d.w_packed, d.cout_pad, d.bias, d.mode = wph.data_ptr(), cout, bias.data_ptr(), mode
    d.res = out.data_ptr() if mode == 2 else None
    d.out = out.data_ptr()
    d.out_f32 = None
    d.bn, d.variant, d.max_ctas, d.skip_loads = 0, -1, 0, 0
    d.ln_out = ln_out.data_ptr() if ln else None
    d.ln_mod = None
    d.ln_upsample = 0
    _lib.check(lib.c2w_op_conv_phase(ctypes.byref(d), torch.cuda.current_stream().cuda_stream), "c2w_op_conv_phase")
    torch.cuda.synchronize()
    return out, ln_out


def _run_upsampled(lib, dev, up, w, bias, mode, res=None, ln=False):
    """The 3x3 conv of the upsampled input through c2w_op_conv_ex (the engine's path before the phase form)."""
    n, H, W, cin = up.shape
    cout = bias.numel()
    wp = torch.as_tensor(w).permute(0, 2, 3, 1).reshape(cout, 9 * cin).to(dev, torch.bfloat16).contiguous()
    out = (res.clone() if mode == 2 else torch.empty(n, H, W, cout, dtype=torch.bfloat16, device=dev))
    ln_out = torch.empty_like(out) if ln else None
    d = _lib.ConvDesc()
    d.x, d.n_img, d.H, d.W, d.cin, d.stride, d.conv3x3 = up.data_ptr(), n, H, W, cin, 1, 1
    d.w_packed, d.cout_pad, d.bias, d.mode = wp.data_ptr(), cout, bias.data_ptr(), mode
    d.res = out.data_ptr() if mode == 2 else None
    d.out = out.data_ptr()
    d.out_f32 = None
    d.bn, d.variant, d.max_ctas, d.skip_loads = cout, -1, 0, 0
    d.ln_out = ln_out.data_ptr() if ln else None
    d.ln_mod = None
    d.ln_upsample = 0
    _lib.check(lib.c2w_op_conv_ex(ctypes.byref(d), torch.cuda.current_stream().cuda_stream), "c2w_op_conv_ex")
    torch.cuda.synchronize()
    return out, ln_out


def _reference(z, w, bias, res=None):
    """fp64 conv2d(interpolate(z, nearest x2)) + bias [+ res], NHWC in and out."""
    x = z.double().permute(0, 3, 1, 2)
    up = F.interpolate(x, scale_factor=2, mode="nearest")
    y = F.conv2d(up, torch.as_tensor(w, dtype=torch.float64, device=z.device), torch.as_tensor(bias).double(),
                 padding=1)
    y = y.permute(0, 2, 3, 1)
    return y if res is None else y + res.double()


# (n, H, W, cin, cout) at the LOW resolution: the config-2 tails (level 1: 128 -> 128 at 64^2, level 2: 256 -> 128 at
# 32^2, level 3: 384 -> 256 at 16^2, two N tiles), a 64-channel tail, odd batches and non-square images
TAIL_SHAPES = [(1, 64, 64, 128, 128), (3, 32, 32, 256, 128), (3, 16, 16, 384, 256), (2, 16, 16, 128, 64),
               (3, 16, 32, 64, 64), (1, 16, 16, 256, 128)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,H,W,cin,cout", TAIL_SHAPES)
@pytest.mark.parametrize("mode", [0, 2])
def test_phase_tail_bit_exact_against_upsampled_conv(lib, n, H, W, cin, cout, mode):
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(n * 7 + H + cin + cout + mode)
    z = torch.randint(-4, 5, (n, H, W, cin), generator=g).float()
    w = torch.randint(-2, 3, (cout, cin, 3, 3), generator=g).float()
    bias = torch.randint(-3, 4, (cout,), generator=g).float().to(dev)
    wph = _pack(lib, w.numpy(), cin, cout).to(dev)
    zb = z.to(dev, torch.bfloat16).contiguous()
    res = torch.randint(-8, 9, (n, 2 * H, 2 * W, cout), generator=g).to(dev, torch.bfloat16) if mode == 2 else None
    ln = cout <= 128  # the fused LayerNorm needs one N tile per pixel
    got, ln_got = _run_phase(lib, dev, zb, wph, bias, mode, res, ln=ln)
    want = _reference(zb, w.to(dev), bias, res).to(torch.bfloat16)
    assert torch.equal(got, want), f"{(got != want).sum().item()} of {want.numel()} outputs differ"
    # the fused LayerNorm of the phase tiles, written to the output pixels, equals the upsampled-input kernel's
    up = zb.repeat_interleave(2, dim=1).repeat_interleave(2, dim=2).contiguous()
    old, ln_old = _run_upsampled(lib, dev, up, w.numpy(), bias, mode, res, ln=ln)
    assert torch.equal(old, want)
    if ln:
        assert torch.equal(ln_got, ln_old)


@pytest.mark.gpu
@pytest.mark.parametrize("n,H,W,cin,cout", TAIL_SHAPES)
def test_phase_tail_accuracy(lib, n, H, W, cin, cout):
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(H * W + cin + cout + n)
    z = torch.randn(n, H, W, cin, generator=g)
    w = torch.randn(cout, cin, 3, 3, generator=g) / (3.0 * cin ** 0.5)
    bias = (0.1 * torch.randn(cout, generator=g)).to(dev)
    res = torch.randn(n, 2 * H, 2 * W, cout, generator=g).to(dev, torch.bfloat16)
    zb = z.to(dev, torch.bfloat16).contiguous()
    got, _ = _run_phase(lib, dev, zb, _pack(lib, w.numpy(), cin, cout).to(dev), bias, 2, res)
    want = _reference(zb, w.to(dev), bias, res)
    err = (got.double() - want).abs().max().item() / want.abs().max().item()
    assert err < 2.0 ** -7, err


@pytest.mark.gpu
def test_refreshed_phase_weights_equal_a_fresh_engine():
    import climate2weather_b200 as c2w
    from climate2weather_b200.model import Engine

    dev = torch.device("cuda:0")
    torch.manual_seed(3)
    # both tails take the phase form: 128 -> 64 from 32^2 and 128 -> 128 from 16^2
    net = c2w.ScoreUNet(channels=12, embedding_dim=64, hidden_channels=(64, 128, 128), hidden_blocks=(1, 1, 1),
                        attention_levels=(), kernel_size=3, activation=torch.nn.SiLU).to(dev)
    x = torch.randn(5, 12, 64, 64, device=dev)
    eng = Engine(net, 4, 3, 64, 64, dev, 8)
    before = eng.unet_forward(x, 0.3)
    with torch.no_grad():
        for name, p in net.named_parameters():
            if "tails" in name:
                p.mul_(1.5).add_(0.01)
    eng.refresh_weights(net)
    torch.cuda.synchronize()
    after = eng.unet_forward(x, 0.3)
    fresh = Engine(net, 4, 3, 64, 64, dev, 8).unet_forward(x, 0.3)
    assert not torch.equal(after, before)
    assert torch.equal(after, fresh)
