"""Exact, index-coded tests of K1's activation-reuse main loop (variant 5: CTA pair, 16 x 8 spatial tiles, one halo'd
unit per channel block whose nine taps are sub-views of it).

Inputs are small integers and each output channel reads one or two (tap, input channel) pairs with weights +-1 / +-2,
so every sum is exact in bf16 and fp32: the expected output is plain integer indexing and must match bit for bit.
Across the output channels every (filter row, filter column, channel block) appears, so a tap read from the wrong row,
column or channel block of the unit shows up as a wrong value.
"""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def lib():
    from climate2weather_b200 import _lib
    return _lib.load()


def _problem(n, H, W, cin, cout, seed):
    """Integer input x [n, H, W, cin], per-output-channel (tap, ci, weight) picks, packed weights and integer bias."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randint(-4, 5, (n, H, W, cin), generator=g).float()
    cb_count = cin // 64
    picks = []
    for co in range(cout):
        tap, cb = co % 9, (co // 9) % cb_count
        terms = [(tap, cb * 64 + (7 * co + 3) % 64, (1.0, -1.0, 2.0, -2.0)[co % 4])]
        if co % 3 == 0:  # a second term from another tap and channel block
            terms.append(((tap + 4) % 9, ((cb + 1) % cb_count) * 64 + (5 * co + 1) % 64, (-2.0, 1.0)[co % 2]))
        picks.append(terms)
    wp = torch.zeros(cout, 9, cin)
    for co, terms in enumerate(picks):
        for tap, ci, wv in terms:
            wp[co, tap, ci] += wv
    bias = torch.tensor([float(co % 5 - 2) for co in range(cout)])
    return x, picks, wp.reshape(cout, 9 * cin), bias


def _reference(x, picks, bias, dr=0, ds=0):
    """out[n, h, w, co] = bias[co] + sum w * x[n, h + r - 1 + dr, w + s - 1 + ds, ci] (zero outside the image)."""
    n, H, W, _ = x.shape
    xp = torch.zeros(n, H + 4, W + 4, x.shape[3])
    xp[:, 2:H + 2, 2:W + 2] = x
    out = bias.repeat(n, H, W, 1)
    for co, terms in enumerate(picks):
        for tap, ci, wv in terms:
            r, s = divmod(tap, 3)
            h0, w0 = r + 1 + dr, s + 1 + ds
            out[..., co] += wv * xp[:, h0:h0 + H, w0:w0 + W, ci]
    return out.reshape(n * H * W, -1)


def _run(lib, dev, x, wp, bias, n, H, W, mode, bn, res=None, ln=False):
    from climate2weather_b200 import _lib
    cin, cout = x.shape[3], wp.shape[0]
    M = n * H * W
    xb = x.to(dev, torch.bfloat16).contiguous()
    wb = wp.to(dev, torch.bfloat16).contiguous()
    bd = bias.to(dev)
    out = res.to(dev, torch.bfloat16).clone() if mode == 2 else torch.empty(M, cout, device=dev, dtype=torch.bfloat16)
    out32 = torch.empty(M, cout, device=dev) if mode == 4 else None
    ln_out = torch.empty(M, cout, device=dev, dtype=torch.bfloat16) if ln else None
    d = _lib.ConvDesc()
    d.x, d.n_img, d.H, d.W, d.cin, d.stride, d.conv3x3 = xb.data_ptr(), n, H, W, cin, 1, 1
    d.w_packed, d.cout_pad, d.bias, d.mode = wb.data_ptr(), cout, bd.data_ptr(), mode
    d.res = out.data_ptr() if mode == 2 else None
    d.out = out.data_ptr()
    d.out_f32 = out32.data_ptr() if mode == 4 else None
    d.bn, d.variant, d.max_ctas, d.skip_loads = bn, 5, 0, 0
    d.ln_out = ln_out.data_ptr() if ln else None
    d.ln_mod = None
    d.ln_upsample = 0
    _lib.check(lib.c2w_op_conv_ex(ctypes.byref(d), torch.cuda.current_stream().cuda_stream), "c2w_op_conv_ex")
    torch.cuda.synchronize()
    return (out32 if mode == 4 else out.float()).cpu()


@pytest.mark.parametrize("n,H,W,cin,cout,bn,mode,ln", [
    (1, 128, 128, 128, 128, 128, 0, False),
    (1, 128, 128, 256, 128, 128, 2, False),
    (2, 64, 64, 128, 128, 128, 2, False),
    (2, 64, 64, 256, 256, 128, 0, False),   # two N tiles per M tile
    (3, 16, 8, 128, 128, 128, 0, False),    # one tile column: both halo columns outside the image
    (3, 8, 16, 128, 128, 128, 2, False),    # two-image form (8-row images), odd image count
    (5, 8, 8, 256, 128, 128, 0, False),     # two-image form, one tile column, odd image count
    (2, 32, 32, 64, 128, 128, 0, False),    # one channel block
    (2, 64, 64, 128, 64, 64, 0, False),
    (2, 64, 64, 256, 64, 64, 2, False),
    (3, 16, 8, 128, 64, 64, 4, False),      # fp32 output straight from the accumulator
    (2, 32, 32, 64, 64, 64, 4, False),
    (2, 64, 64, 128, 128, 128, 2, True),    # fused LayerNorm kernel: its conv output
    (2, 32, 32, 128, 64, 64, 0, True),
])
def test_activation_reuse_taps_bit_exact(lib, dev, n, H, W, cin, cout, bn, mode, ln):
    x, picks, wp, bias = _problem(n, H, W, cin, cout, seed=n * 1000 + H + W + cin + cout + mode)
    want = _reference(x, picks, bias)
    # the coding is sensitive to a tap read one row or one column off
    for dr, ds in ((0, 1), (0, -1), (1, 0), (-1, 0)):
        assert not torch.equal(_reference(x, picks, bias, dr, ds), want)
    res = None
    if mode == 2:
        res = torch.randint(-8, 9, (n * H * W, cout), generator=torch.Generator().manual_seed(cout + H)).float()
        want = want + res
    got = _run(lib, dev, x, wp, bias, n, H, W, mode, bn, res=res, ln=ln)
    assert torch.equal(got, want), f"{(got != want).sum().item()} of {want.numel()} outputs differ"
