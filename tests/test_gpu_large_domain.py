"""Domains wider than 128 pixels: K1's streamed main loop over 128-pixel row segments, the tiled attention kernels
beyond 64 tokens (forward and backward), and the whole network at 128 x 256 and 256 x 256 against the fp32 oracle."""
import ctypes
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import unet_ref

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def lib():
    from climate2weather_b200 import _lib
    return _lib.load()


def stream():
    return torch.cuda.current_stream().cuda_stream


def relerr(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def rel_l2(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def _conv(lib, dev, x, w, bias, stride, mode, bn, variant, res=None, ln=False):
    """c2w_op_conv_ex on NHWC x [n, H, W, cin] with OIHW fp32 w; returns (out [n, Ho, Wo, cout] fp32, ln_out)."""
    from climate2weather_b200 import _lib
    n, H, W, cin = x.shape
    cout = w.shape[0]
    Ho, Wo = H // stride, W // stride
    M = n * Ho * Wo
    xb = x.to(dev, torch.bfloat16).contiguous()
    wp = w.permute(0, 2, 3, 1).reshape(cout, 9 * cin).to(dev, torch.bfloat16).contiguous()
    bd = bias.to(dev)
    out = res.reshape(M, cout).to(dev, torch.bfloat16).clone() if mode == 2 else \
        torch.zeros(M, cout, device=dev, dtype=torch.bfloat16)
    out32 = torch.zeros(M, cout, device=dev) if mode == 4 else None
    ln_out = torch.zeros(M, cout, device=dev, dtype=torch.bfloat16) if ln else None
    d = _lib.ConvDesc()
    d.x, d.n_img, d.H, d.W, d.cin, d.stride, d.conv3x3 = xb.data_ptr(), n, H, W, cin, stride, 1
    d.w_packed, d.cout_pad, d.bias, d.mode = wp.data_ptr(), cout, bd.data_ptr(), mode
    d.res = out.data_ptr() if mode == 2 else None
    d.out = out.data_ptr()
    d.out_f32 = out32.data_ptr() if mode == 4 else None
    d.bn, d.variant, d.max_ctas, d.skip_loads = bn, variant, 0, 0
    d.ln_out = ln_out.data_ptr() if ln else None
    d.ln_mod = None
    d.ln_upsample = 0
    _lib.check(lib.c2w_op_conv_ex(ctypes.byref(d), stream()), "c2w_op_conv_ex")
    torch.cuda.synchronize()
    got = (out32 if mode == 4 else out.float()).cpu().reshape(n, Ho, Wo, cout)
    return got, (ln_out.float().cpu().reshape(n, Ho, Wo, cout) if ln else None)


def _torch_conv(x, w, bias, stride, dtype=torch.float32):
    y = F.conv2d(x.permute(0, 3, 1, 2).to(dtype), w.to(dtype), bias.to(dtype), stride=stride, padding=1)
    return y.permute(0, 2, 3, 1)


# (n, H, W, cin, cout, stride, mode, bn, variant): variant 1 = CTA pair on the streamed loop (no activation reuse),
# -1 = the library's pick (256-wide N tile, streamed)
K1_SHAPES = [
    (2, 8, 256, 128, 128, 1, 0, 128, 1),     # two row segments per row
    (1, 4, 512, 64, 64, 1, 2, 64, 1),        # four segments, residual epilogue
    (2, 16, 256, 128, 128, 2, 0, 128, 1),    # stride-2 head 256 -> 128 (one segment)
    (1, 8, 512, 64, 128, 2, 0, 128, 1),      # stride-2 head 512 -> 256 (two segments)
    (1, 8, 256, 256, 256, 1, 0, 256, -1),    # 256-wide N tile at a 256-wide level
    (2, 8, 256, 128, 64, 1, 4, 64, 1),       # fp32 epilogue
    (1, 6, 256, 64, 64, 1, 0, 64, 0),        # one CTA per MMA
]


@pytest.mark.parametrize("n,H,W,cin,cout,stride,mode,bn,variant", K1_SHAPES)
def test_k1_row_segments_bit_exact(lib, dev, n, H, W, cin, cout, stride, mode, bn, variant):
    """Small-integer data with sparse +-1 weights: every sum is exact in bf16, so the output must equal torch's."""
    g = torch.Generator().manual_seed(n * 7 + H + W + cin + cout + stride + mode)
    x = torch.randint(-2, 3, (n, H, W, cin), generator=g).float()
    w = torch.randint(-1, 2, (cout, cin, 3, 3), generator=g).float() * (torch.rand(cout, cin, 3, 3, generator=g) < 1 / 32)
    bias = torch.randint(-3, 4, (cout,), generator=g).float()
    want = _torch_conv(x, w, bias, stride)
    res = None
    if mode == 2:
        res = torch.randint(-8, 9, want.shape, generator=g).float()
        want = want + res
    got, _ = _conv(lib, dev, x, w, bias, stride, mode, bn, variant, res=res)
    assert torch.equal(got, want), f"{(got != want).sum().item()} of {want.numel()} outputs differ"


@pytest.mark.parametrize("n,H,W,cin,cout,stride,mode,bn,variant", K1_SHAPES)
def test_k1_row_segments_accuracy(lib, dev, n, H, W, cin, cout, stride, mode, bn, variant):
    g = torch.Generator().manual_seed(H * W + cout)
    x = torch.randn(n, H, W, cin, generator=g)
    w = torch.randn(cout, cin, 3, 3, generator=g) / (3 * cin ** 0.5)
    bias = torch.randn(cout, generator=g)
    xb = x.bfloat16().double()
    want = _torch_conv(xb, w.bfloat16().double(), bias.double(), stride, torch.float64)
    res = None
    if mode == 2:
        res = torch.randn(want.shape, generator=g)
        want = want + res.bfloat16().double()
    got, _ = _conv(lib, dev, x, w, bias, stride, mode, bn, variant, res=res)
    assert relerr(got, want) < 2 ** -7


@pytest.mark.parametrize("mode", [0, 2])
def test_k1_row_segments_fused_layernorm(lib, dev, mode):
    """Fused LayerNorm epilogue (one N tile = all channels) on the streamed loop at 256 wide."""
    n, H, W, C = 2, 4, 256, 128
    g = torch.Generator().manual_seed(5 + mode)
    x = torch.randn(n, H, W, C, generator=g)
    w = torch.randn(C, C, 3, 3, generator=g) / (3 * C ** 0.5)
    bias = torch.randn(C, generator=g)
    res = torch.randn(n, H, W, C, generator=g) if mode == 2 else None
    got, ln = _conv(lib, dev, x, w, bias, 1, mode, 128, 1, res=res, ln=True)
    ref = unet_ref.channel_layernorm(got.permute(0, 3, 1, 2)).permute(0, 2, 3, 1)
    assert relerr(ln, ref) < 2 ** -7


def _attn_ref(qkv, C):
    q, k, v = qkv.float().cpu().split(C, dim=2)
    s = 1 / math.sqrt(math.sqrt(C))
    return torch.einsum("bts,bsc->btc", torch.softmax(torch.einsum("btc,bsc->bts", q * s, k * s), dim=-1), v)


# T = 96, 136, 200: a partial last block of queries and keys (masked keys, rows past T never stored)
ATTN = [(128, 512), (256, 512), (256, 256), (1024, 128), (1024, 512), (192, 384), (320, 192), (128, 128), (256, 128),
        (96, 512), (136, 512), (200, 512)]


@pytest.mark.parametrize("T,C", ATTN)
def test_attention_tiled_forward(lib, dev, T, C):
    from climate2weather_b200 import _lib
    g = torch.Generator().manual_seed(T + C)
    n = 3
    qkv = torch.randn(n, T, 3 * C, generator=g).to(dev).to(torch.bfloat16)
    outs = []
    for _ in range(2):
        out = torch.empty(n, T, C, device=dev, dtype=torch.bfloat16)
        _lib.check(lib.c2w_op_attention(qkv.data_ptr(), out.data_ptr(), n, T, C, stream()), "c2w_op_attention")
        torch.cuda.synchronize()
        outs.append(out.cpu())
    assert torch.equal(outs[0], outs[1])
    assert relerr(outs[0], _attn_ref(qkv, C)) < 2 ** -7


@pytest.mark.parametrize("T,C", ATTN)
def test_attention_tiled_backward(lib, dev, T, C):
    from climate2weather_b200 import _lib
    g = torch.Generator().manual_seed(T * C)
    n = 2
    qkv = torch.randn(n, T, 3 * C, generator=g).to(torch.bfloat16)
    go = torch.randn(n, T, C, generator=g).to(torch.bfloat16)
    qkv_d, go_d = qkv.to(dev), go.to(dev)
    scratch = torch.empty(2 * n * T * T, device=dev)
    outs = []
    for _ in range(2):
        gq = torch.empty(n, T, 3 * C, device=dev, dtype=torch.bfloat16)
        _lib.check(lib.c2w_op_attention_bwd(qkv_d.data_ptr(), go_d.data_ptr(), gq.data_ptr(), scratch.data_ptr(), n, T,
                                            C, stream()), "attention_bwd")
        torch.cuda.synchronize()
        outs.append(gq.cpu())
    assert torch.equal(outs[0], outs[1])
    leaf = qkv.float().requires_grad_(True)
    (want,) = torch.autograd.grad(_attn_ref(leaf, C), leaf, go.float())
    assert relerr(outs[0], want) < 2 ** -6
    assert rel_l2(outs[0], want) < 2 ** -6


NET = dict(channels=20, embedding_dim=64, hidden_channels=(64, 64, 64, 64, 512), hidden_blocks=(1, 1, 1, 1, 1),
           attention_levels=(4,), kernel_size=3)


def _net(dev, seed):
    import climate2weather_b200 as c2w
    torch.manual_seed(seed)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, **NET)
    ref = unet_ref.RefNet({k: v.detach().clone() for k, v in net.state_dict().items()}, NET)
    return net.to(dev), ref


@pytest.mark.parametrize("H,W", [(128, 256), (256, 256)])
def test_unet_large_domain_vs_oracle(dev, H, W):
    """Attention at the deepest level with 512 channels (128 / 256 tokens: the tiled kernels): forward and input-VJP
    against fp32 autograd through the oracle, with the parity tests' tolerances."""
    net, ref = _net(dev, H + W)
    n = 2
    g = torch.Generator().manual_seed(n)
    x = torch.randn(n, NET["channels"], H, W, generator=g)
    gout = torch.randn(n, NET["channels"], H, W, generator=g)
    t = torch.tensor(0.45)
    xg = x.clone().requires_grad_(True)
    want_out = ref(xg, t)
    (want_gin,) = torch.autograd.grad(want_out, xg, gout)
    with torch.no_grad():
        got = net(x.to(dev), t)
    assert relerr(got, want_out.detach()) < 3e-2 and rel_l2(got, want_out.detach()) < 2e-2
    eng = net.engine(NET["channels"], 1, H, W, dev, max_windows=n, vjp=True)
    out, gin = eng.unet_vjp(x.to(dev), 0.45, gout.to(dev))
    assert relerr(out, want_out.detach()) < 3e-2
    assert relerr(gin, want_gin) < 3e-2 and rel_l2(gin, want_gin) < 2e-2


def test_unet_large_domain_chunking_bit_identical(dev):
    """The same windows through 1-, 2- and 3-window workspaces give the same bits at 256 x 256."""
    net, _ = _net(dev, 3)
    x = torch.randn(3, NET["channels"], 256, 256, generator=torch.Generator().manual_seed(4)).to(dev)
    outs = []
    for mw in (1, 2, 3):
        eng = net.engine(NET["channels"], 1, 256, 256, dev, max_windows=mw)
        outs.append(eng.unet_forward(x, 0.3).cpu())
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])
