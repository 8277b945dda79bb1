"""GPU parity tests (pytest -m gpu): the CUDA path, called through the C ABI (ctypes) and through the Python mirror
of the reference classes, against the CPU oracle (oracle/) and the committed golden fixtures.

Tolerances (stated per test): integer/index work is bit-exact; tensor-core layers use bf16 operands with fp32
accumulation against an fp32 oracle, so per-layer error is ~2^-8 relative to the tensor scale and the whole UNet
(70 convs, bf16 residual stream) is held to 3e-2 of the output's max-abs; the fp32 elementwise kernels (guidance,
predictor, corrector) are held to 1e-5.
"""
import ctypes
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import pipeline_ref, score_ref, unet_ref

pytestmark = pytest.mark.gpu

SMALL = dict(channels=20, embedding_dim=64, hidden_channels=(64, 128), hidden_blocks=(1, 2), attention_levels=(1,),
             kernel_size=3)
STD = [0.1692666615037876, 0.0425178630338289, 0.3268027589410125, 0.3268027589410125]
GAMMA = 0.0007196856730011522


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def lib():
    from climate2weather_b200 import _lib
    return _lib.load()


def stream():
    return torch.cuda.current_stream().cuda_stream


def relerr(got, ref):
    got, ref = got.double().cpu(), ref.double().cpu()
    return ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


def rel_l2(got, ref):
    """||got - ref||_2 / ||ref||_2 over the whole tensor: the average-case companion of `relerr` (a max-abs ratio can
    hide a uniformly wrong tensor behind one large reference value)."""
    got, ref = got.double().cpu(), ref.double().cpu()
    return ((got - ref).norm() / ref.norm().clamp_min(1e-30)).item()


def frame_rel_l2(got, ref):
    """Worst per-frame (leading axis) relative L2 error."""
    got, ref = got.double().cpu().flatten(1), ref.double().cpu().flatten(1)
    return ((got - ref).norm(dim=1) / ref.norm(dim=1).clamp_min(1e-30)).max().item()


def pack_w(w, cin_pad, cout_pad):
    cout, cin = w.shape[:2]
    taps = w[0, 0].numel()
    wp = torch.zeros(cout_pad, taps, cin_pad, device=w.device)
    wp[:cout, :, :cin] = w.reshape(cout, cin, taps).permute(0, 2, 1)
    return wp.reshape(cout_pad, taps * cin_pad).to(torch.bfloat16).contiguous()


# ------------------------------------------------------------------------------------------------ K1
@pytest.mark.parametrize("n,H,W,cin,cout,mode", [
    (2, 128, 128, 128, 128, 1), (2, 128, 128, 52, 128, 0), (1, 128, 128, 128, 52, 4), (3, 64, 64, 128, 128, 2),
    (3, 32, 32, 256, 256, 1), (3, 16, 16, 384, 384, 2), (3, 8, 8, 512, 512, 1), (2, 16, 16, 512, 384, 0),
    (1, 8, 8, 64, 64, 0), (5, 16, 16, 64, 192, 1)])
def test_conv3x3_vs_torch(lib, dev, n, H, W, cin, cout, mode):
    """K1 vs F.conv2d in fp32 on the same bf16-rounded operands: only accumulation order and the bf16 output
    rounding differ -> 2^-7 of the output scale (fp32 output mode: 1e-4)."""
    from climate2weather_b200 import _lib
    g = torch.Generator().manual_seed(n * 1000 + cin + cout)
    cin_pad, cout_pad = (cin + 63) // 64 * 64, (cout + 63) // 64 * 64
    x = torch.randn(n, cin, H, W, generator=g).to(dev)
    w = (torch.randn(cout, cin, 3, 3, generator=g) / (3 * math.sqrt(cin))).to(dev)
    b = torch.randn(cout, generator=g).to(dev)
    xb = torch.zeros(n, H, W, cin_pad, device=dev, dtype=torch.bfloat16)
    xb[..., :cin] = x.permute(0, 2, 3, 1).to(torch.bfloat16)
    wp = pack_w(w, cin_pad, cout_pad)
    bp = torch.zeros(cout_pad, device=dev)
    bp[:cout] = b
    M = n * H * W
    res = torch.randn(M, cout_pad, generator=g).to(dev).to(torch.bfloat16)
    out = res.clone() if mode in (2, 5) else torch.empty(M, cout_pad, device=dev, dtype=torch.bfloat16)
    out32 = torch.empty(M, cout_pad, device=dev) if mode == 4 else None
    _lib.check(lib.c2w_op_conv(xb.data_ptr(), n, H, W, cin_pad, wp.data_ptr(), cout_pad, bp.data_ptr(), mode,
                               out.data_ptr() if mode == 2 else None, out.data_ptr(),
                               out32.data_ptr() if mode == 4 else None, 1, 0, 0, stream()), "c2w_op_conv")
    torch.cuda.synchronize()
    ref = F.conv2d(xb[..., :cin].float().permute(0, 3, 1, 2), w.to(torch.bfloat16).float(), b, padding=1)
    if mode == 1:
        ref = F.silu(ref)
    ref = ref.permute(0, 2, 3, 1).reshape(M, cout)
    if mode == 2:
        ref = ref + res[:, :cout].float()
    got = (out32 if mode == 4 else out.float())[:, :cout]
    assert relerr(got, ref) < (1e-4 if mode == 4 else 2 ** -7)
    if cout_pad > cout and mode != 2:  # padded output channels carry exact zeros (zero weights, zero bias)
        pad = (out32 if mode == 4 else out.float())[:, cout:]
        assert float(pad.abs().max()) == 0.0


def test_gemm_mode_vs_torch(lib, dev):
    """Plain GEMM mode (1x1 Conv1d of the attention blocks): bf16 output 2^-7; fp32 output 1e-4, in 64-wide tiles, one or
    several per row (the picked tile for mode 4 with bn = 0)."""
    from climate2weather_b200 import _lib
    g = torch.Generator().manual_seed(7)
    for M, K, N, f32 in [(256, 128, 128, False), (64, 512, 1536, False), (200, 576, 64, True), (384, 512, 512, False),
                         (200, 128, 192, True)]:
        a = torch.randn(M, K, generator=g).to(dev).to(torch.bfloat16)
        w = (torch.randn(N, K, generator=g) / math.sqrt(K)).to(dev).to(torch.bfloat16)
        b = torch.randn(N, generator=g).to(dev)
        out32 = torch.empty(M, N, device=dev) if f32 else None
        out = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
        _lib.check(lib.c2w_op_conv(a.data_ptr(), 1, 1, M, K, w.data_ptr(), N, b.data_ptr(), 4 if f32 else 0, None,
                                   None if f32 else out.data_ptr(), out32.data_ptr() if f32 else None, 0, 0, 0, stream()),
                   "c2w_op_conv(gemm)")
        torch.cuda.synchronize()
        ref = a.float() @ w.float().t() + b
        assert relerr(out32 if f32 else out.float(), ref) < (1e-4 if f32 else 2 ** -7)


def _conv_ex(lib, xb, wp, bp, mode, n, H, W, stride=1, res=None, variant=-1, bn=0, ln_mod=None, ln=False, ln_up=0,
             f32=False, max_ctas=0):
    """One c2w_op_conv_ex launch on NHWC bf16 input xb [n, H, W, cin_pad]; returns (out, ln_out)."""
    from climate2weather_b200 import _lib
    dev = xb.device
    cout_pad = wp.shape[0]
    Ho, Wo = H // stride, W // stride
    M = n * Ho * Wo
    out = res.clone() if mode in (2, 5) else torch.empty(M, cout_pad, device=dev, dtype=torch.bfloat16)
    out32 = torch.empty(M, cout_pad, device=dev) if f32 else None
    up = 2 if ln_up else 1
    ln_out = torch.full((n, Ho * up, Wo * up, cout_pad), 7.0, device=dev, dtype=torch.bfloat16) if ln else None
    d = _lib.ConvDesc()
    d.x, d.n_img, d.H, d.W, d.cin, d.stride, d.conv3x3 = xb.data_ptr(), n, H, W, xb.shape[-1], stride, 1
    d.w_packed, d.cout_pad, d.bias, d.mode = wp.data_ptr(), cout_pad, bp.data_ptr(), mode
    d.res = out.data_ptr() if mode in (2, 5) else None
    d.out = out.data_ptr()
    d.out_f32 = out32.data_ptr() if f32 else None
    d.bn, d.variant, d.max_ctas, d.skip_loads = bn, variant, max_ctas, 0
    d.ln_out = ln_out.data_ptr() if ln else None
    d.ln_mod = ln_mod.data_ptr() if ln_mod is not None else None
    d.ln_upsample = ln_up
    _lib.check(lib.c2w_op_conv_ex(ctypes.byref(d), stream()), "c2w_op_conv_ex")
    torch.cuda.synchronize()
    return (out32 if f32 else out), ln_out


def _conv_problem(dev, n, H, W, cin, cout, seed):
    g = torch.Generator().manual_seed(seed)
    cin_pad, cout_pad = (cin + 63) // 64 * 64, (cout + 63) // 64 * 64
    x = torch.randn(n, cin, H, W, generator=g).to(dev)
    w = (torch.randn(cout, cin, 3, 3, generator=g) / (3 * math.sqrt(cin))).to(dev)
    b = torch.randn(cout, generator=g).to(dev)
    xb = torch.zeros(n, H, W, cin_pad, device=dev, dtype=torch.bfloat16)
    xb[..., :cin] = x.permute(0, 2, 3, 1).to(torch.bfloat16)
    wp = pack_w(w, cin_pad, cout_pad)
    bp = torch.zeros(cout_pad, device=dev)
    bp[:cout] = b
    return g, xb, w, b, wp, bp


@pytest.mark.parametrize("variant", [0, 1, 5])
@pytest.mark.parametrize("n,H,W,cin,cout,mode", [
    (2, 128, 128, 128, 128, 1), (3, 64, 64, 128, 128, 2), (5, 32, 32, 128, 128, 0), (1, 128, 128, 64, 128, 1),
    (3, 16, 16, 256, 128, 2), (1, 16, 8, 64, 128, 0), (2, 64, 64, 128, 52, 4), (2, 32, 32, 128, 64, 1)])
def test_conv3x3_kernel_variants(lib, dev, variant, n, H, W, cin, cout, mode):
    """Single CTA (0), CTA pair / cta_group::2 (1) and CTA pair with the activation-reuse main loop (5: 16 x 8 spatial
    tiles, one halo'd load per filter column reused by the three filter rows) compute the same conv; odd tile counts
    exercise the pair's out-of-range half."""
    g, xb, w, b, wp, bp = _conv_problem(dev, n, H, W, cin, cout, 11 * n + cin)
    M = n * H * W
    res = torch.randn(M, wp.shape[0], generator=g).to(dev).to(torch.bfloat16)
    got, _ = _conv_ex(lib, xb, wp, bp, mode, n, H, W, res=res, variant=variant, f32=(mode == 4))
    ref = F.conv2d(xb[..., :cin].float().permute(0, 3, 1, 2), w.to(torch.bfloat16).float(), b, padding=1)
    if mode == 1:
        ref = F.silu(ref)
    ref = ref.permute(0, 2, 3, 1).reshape(M, cout)
    if mode == 2:
        ref = ref + res[:, :cout].float()
    assert relerr(got.float()[:, :cout], ref) < (1e-4 if mode == 4 else 2 ** -7)


@pytest.mark.parametrize("n,H,W,cin,cout,mode", [
    (6, 8, 8, 512, 512, 1), (5, 8, 8, 128, 256, 2), (4, 8, 16, 64, 128, 0), (3, 8, 8, 192, 384, 2),
    (7, 16, 16, 384, 384, 1), (2, 16, 16, 512, 384, 2), (3, 32, 32, 256, 256, 1)])
def test_conv3x3_activation_reuse_wide_and_two_image_tiles(lib, dev, n, H, W, cin, cout, mode):
    """Activation reuse with 128-wide N tiles on layers wider than one tile (several N tiles per M tile), and its
    two-image form on 8-row images (tile row = (image row, image, pixel); odd image counts leave half a tile out of
    range) against the streamed single-CTA kernel's reference."""
    g, xb, w, b, wp, bp = _conv_problem(dev, n, H, W, cin, cout, 13 * n + cout)
    M = n * H * W
    res = torch.randn(M, wp.shape[0], generator=g).to(dev).to(torch.bfloat16)
    got, _ = _conv_ex(lib, xb, wp, bp, mode, n, H, W, res=res, variant=5, bn=128)
    ref = F.conv2d(xb[..., :cin].float().permute(0, 3, 1, 2), w.to(torch.bfloat16).float(), b, padding=1)
    if mode == 1:
        ref = F.silu(ref)
    ref = ref.permute(0, 2, 3, 1).reshape(M, cout)
    if mode == 2:
        ref = ref + res[:, :cout].float()
    assert relerr(got.float()[:, :cout], ref) < 2 ** -7


@pytest.mark.parametrize("n,H,W,cin,cout,variant,bn", [
    (2, 128, 128, 128, 128, 5, 0), (3, 32, 32, 256, 256, 1, 256), (3, 32, 32, 256, 256, 5, 128), (5, 8, 8, 512, 512, 5, 128),
    (2, 16, 16, 384, 384, 1, 192)])
def test_conv3x3_times_dsilu_in_place(lib, dev, n, H, W, cin, cout, variant, bn):
    """Epilogue mode 5 of the input-gradient pass: out <- conv(x) * silu'(out), the pre-activation prefetched into the
    staging tile like a residual and overwritten in place."""
    g, xb, w, b, wp, bp = _conv_problem(dev, n, H, W, cin, cout, 17 * n + cout)
    M = n * H * W
    pre = (2.0 * torch.randn(M, wp.shape[0], generator=g)).to(dev).to(torch.bfloat16)
    got, _ = _conv_ex(lib, xb, wp, bp, 5, n, H, W, res=pre, variant=variant, bn=bn)
    ref = F.conv2d(xb[..., :cin].float().permute(0, 3, 1, 2), w.to(torch.bfloat16).float(), b, padding=1)
    ref = ref.permute(0, 2, 3, 1).reshape(M, cout)
    x = pre[:, :cout].float()
    sg = torch.sigmoid(x)
    ref = ref * (sg * (1 + x * (1 - sg)))
    assert relerr(got.float()[:, :cout], ref) < 2 ** -7


@pytest.mark.parametrize("variant", [0, 1])
@pytest.mark.parametrize("n,H,W,cin,cout", [(2, 128, 128, 128, 128), (3, 64, 64, 128, 256), (3, 32, 32, 256, 384),
                                            (5, 16, 16, 384, 512), (1, 16, 32, 64, 64)])
def test_conv3x3_stride2_vs_torch(lib, dev, variant, n, H, W, cin, cout):
    """Head convs of levels > 0 (model/nn.py:169-176): stride 2, pad 1, read straight from the NHWC input through
    an element-strided tensor map."""
    g, xb, w, b, wp, bp = _conv_problem(dev, n, H, W, cin, cout, 5 * n + cout)
    got, _ = _conv_ex(lib, xb, wp, bp, 0, n, H, W, stride=2, variant=variant)
    ref = F.conv2d(xb[..., :cin].float().permute(0, 3, 1, 2), w.to(torch.bfloat16).float(), b, padding=1, stride=2)
    ref = ref.permute(0, 2, 3, 1).reshape(-1, cout)
    assert relerr(got.float()[:, :cout], ref) < 2 ** -7


@pytest.mark.parametrize("n,H,W,C,mode,up,use_mod,variant", [
    (2, 128, 128, 128, 2, 0, True, 1), (2, 64, 64, 128, 0, 0, True, 1), (3, 32, 32, 256, 2, 0, True, 1),
    (2, 128, 128, 128, 2, 0, True, 5), (3, 64, 64, 128, 2, 1, False, 5), (1, 32, 32, 128, 0, 0, True, 5),
    (3, 32, 32, 256, 2, 1, False, 1), (2, 64, 64, 128, 2, 1, False, 0), (1, 16, 16, 64, 0, 0, True, 0)])
def test_conv3x3_fused_layernorm(lib, dev, n, H, W, C, mode, up, use_mod, variant):
    """Conv epilogue that also emits LN(out + mod) (model/nn.py:154,183-184): must equal the standalone K2 semantics
    applied to the bf16 conv output -> 2^-7 of the normalised scale."""
    g, xb, w, b, wp, bp = _conv_problem(dev, n, H, W, C, C, 17 * n + C + up)
    M = n * H * W
    res = torch.randn(M, C, generator=g).to(dev).to(torch.bfloat16)
    mod = torch.randn(C, generator=g).to(dev) if use_mod else None
    out, ln_out = _conv_ex(lib, xb, wp, bp, mode, n, H, W, res=res, variant=variant, ln=True, ln_mod=mod, ln_up=up)
    ref = F.conv2d(xb.float().permute(0, 3, 1, 2), w.to(torch.bfloat16).float(), b, padding=1)
    ref = ref.permute(0, 2, 3, 1).reshape(M, C)
    if mode == 2:
        ref = ref + res.float()
    assert relerr(out.float(), ref) < 2 ** -7
    v = out.float().reshape(n, H, W, C).permute(0, 3, 1, 2).cpu()
    if use_mod:
        v = v + mod.cpu()[None, :, None, None]
    lref = unet_ref.channel_layernorm(v)
    if up:
        lref = F.interpolate(lref, scale_factor=2, mode="nearest")
    assert relerr(ln_out.float().cpu().permute(0, 3, 1, 2), lref) < 2 ** -7


# ------------------------------------------------------------------------------------------------ K2 / K4 / K0
@pytest.mark.parametrize("C", [64, 128, 256, 384, 512])
@pytest.mark.parametrize("up", [0, 1])
def test_channel_layernorm(lib, dev, C, up):
    """K2 vs the oracle's zuko-LayerNorm restatement (unbiased variance): fp32 math, bf16 output -> 2^-8."""
    from climate2weather_b200 import _lib
    g = torch.Generator().manual_seed(C + up)
    n, H, W = 3, 8, 16
    x = (torch.randn(n, H, W, C, generator=g) * 2 + 0.5).to(dev).to(torch.bfloat16)
    mod = torch.randn(C, generator=g).to(dev)
    out = torch.empty(n, H * (2 if up else 1), W * (2 if up else 1), C, device=dev, dtype=torch.bfloat16)
    _lib.check(lib.c2w_op_layernorm(x.data_ptr(), None if up else mod.data_ptr(), out.data_ptr(), n * H * W, C, H, W,
                                    up, stream()), "c2w_op_layernorm")
    torch.cuda.synchronize()
    v = x.float().cpu().permute(0, 3, 1, 2) + (0 if up else mod.cpu()[None, :, None, None])
    ref = unet_ref.channel_layernorm(v)
    if up:
        ref = F.interpolate(ref, scale_factor=2, mode="nearest")
    assert relerr(out.float().cpu().permute(0, 3, 1, 2), ref) < 2 ** -8


@pytest.mark.parametrize("T,C", [(64, 512), (256, 128), (16, 64), (64, 128), (64, 256)])
def test_attention_core(lib, dev, T, C):
    """K4 vs model/nn.py:74-85 semantics in fp32 on the same bf16 q, k, v: bf16 output rounding only."""
    from climate2weather_b200 import _lib
    g = torch.Generator().manual_seed(T + C)
    n = 3
    qkv = torch.randn(n, T, 3 * C, generator=g).to(dev).to(torch.bfloat16)
    out = torch.empty(n, T, C, device=dev, dtype=torch.bfloat16)
    _lib.check(lib.c2w_op_attention(qkv.data_ptr(), out.data_ptr(), n, T, C, stream()), "c2w_op_attention")
    torch.cuda.synchronize()
    q, k, v = qkv.float().cpu().split(C, dim=2)
    s = 1 / math.sqrt(math.sqrt(C))
    w = torch.softmax(torch.einsum("btc,bsc->bts", q * s, k * s), dim=-1)
    ref = torch.einsum("bts,bsc->btc", w, v)
    assert relerr(out.float().cpu(), ref) < 2 ** -7


@pytest.mark.parametrize("L,k,first,n", [(16, 6, 0, 4), (16, 6, 2, 2), (9, 2, 1, 4)])
@pytest.mark.parametrize("H,W", [(4, 8), (16, 16), (8, 24)])  # 256 pixels: the tiled kernel (64-pixel tiles); others: generic
@pytest.mark.parametrize("C", [1, 3, 4, 5, 8])  # C != 4: the scalar lanes; k = 6, C = 5 -> 65 channels straddle 64
def test_gather_windows_bit_exact(lib, dev, C, L, k, first, n, H, W):
    """K0 vs the oracle unfold index map (src/thor/score.py:68-74): pure indexing + one bf16 rounding; the channels
    past w*C up to cin_pad = 64 * ceil(w*C / 64) are zero."""
    from climate2weather_b200 import _lib
    w = 2 * k + 1
    cin_pad = 64 * -(-w * C // 64)
    x = torch.randn(L, C, H, W, generator=torch.Generator().manual_seed(L))
    traj = x.permute(0, 2, 3, 1).contiguous().to(dev)
    out = torch.full((n, H * W, cin_pad), 7.0, device=dev, dtype=torch.bfloat16)
    _lib.check(lib.c2w_op_gather_windows(traj.data_ptr(), out.data_ptr(), n, H * W, C, w, cin_pad, first, stream()),
               "gather")
    torch.cuda.synchronize()
    ref = score_ref.unfold(x, k)[first:first + n].reshape(n, w * C, H * W).permute(0, 2, 1).to(torch.bfloat16)
    assert torch.equal(out[..., :w * C].cpu(), ref)
    assert float(out[..., w * C:].abs().max()) == 0.0  # w * C is never a multiple of 64 here


# ------------------------------------------------------------------------------------------------ whole network
def make_small(dev, seed=3):
    import climate2weather_b200 as c2w
    torch.manual_seed(seed)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, **SMALL)
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    return net.to(dev), unet_ref.RefNet(sd, SMALL)


def test_modulation_vs_oracle(lib, dev):
    """K3: time embedding MLP and every block's modulation vector, fp32 -> 1e-5."""
    from climate2weather_b200 import _lib
    net, ref = make_small(dev)
    eng = net.engine(20, 1, 32, 32, dev)
    nmod = lib.c2w_total_mod_channels(eng.handle)
    emb = torch.empty(64, device=dev)
    mods = torch.empty(nmod, device=dev)
    _lib.check(lib.c2w_op_modulation(eng.handle, 0.37, emb.data_ptr(), mods.data_ptr(), stream()), "modulation")
    torch.cuda.synchronize()
    e_ref = unet_ref.time_modulation(ref.sd, torch.tensor(0.37))[0]
    assert relerr(emb, e_ref) < 1e-5
    p = "unet.descent.0.0.project.0"
    m_ref = F.linear(e_ref, ref.sd[p + ".weight"], ref.sd[p + ".bias"])
    assert relerr(mods[:64], m_ref) < 1e-5


def test_unet_forward_small_vs_oracle(dev):
    net, ref = make_small(dev)
    x = torch.randn(3, 20, 32, 32, generator=torch.Generator().manual_seed(11))
    t = torch.tensor(0.6)
    with torch.no_grad():
        want = ref(x, t)
        got = net(x.to(dev), t)
    e = relerr(got, want)
    print(f"\nsmall UNet forward rel-err (max-abs / max-abs): {e:.3e}")
    assert e < 3e-2


@pytest.mark.parametrize("cfg,H,W,n", [
    (dict(channels=12, embedding_dim=64, hidden_channels=(64, 192), hidden_blocks=(2, 1), attention_levels=()), 32, 64, 3),
    (dict(channels=36, embedding_dim=128, hidden_channels=(128, 256, 320), hidden_blocks=(1, 1, 2), attention_levels=(2,)),
     32, 32, 2),
    (dict(channels=52, embedding_dim=64, hidden_channels=(64, 64, 64, 128), hidden_blocks=(1, 1, 1, 1),
          attention_levels=(3,)), 64, 64, 5),
    (dict(channels=20, embedding_dim=64, hidden_channels=(128,), hidden_blocks=(3,), attention_levels=()), 16, 128, 7),
])
def test_unet_forward_other_architectures(dev, cfg, H, W, n):
    """Architectures and patch shapes other than the two fixtures (non-square patches, channel counts that map to
    the 64/128/192/256-wide tiles, attention at different depths, odd window counts): forward and input-VJP against
    the fp32 oracle."""
    import climate2weather_b200 as c2w
    cfg = dict(cfg, kernel_size=3)
    torch.manual_seed(H + W + n)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, **cfg)
    ref = unet_ref.RefNet({k: v.detach().clone() for k, v in net.state_dict().items()}, cfg)
    net = net.to(dev)
    g = torch.Generator().manual_seed(n)
    x = torch.randn(n, cfg["channels"], H, W, generator=g)
    gout = torch.randn(n, cfg["channels"], H, W, generator=g)
    t = torch.tensor(0.45)
    want_out, want_gin = _autograd_vjp(ref, x, t, gout)
    with torch.no_grad():
        got = net(x.to(dev), t)
    assert relerr(got, want_out) < 3e-2
    eng = net.engine(cfg["channels"], 1, H, W, dev, max_windows=n, vjp=True)
    out, gin = eng.unet_vjp(x.to(dev), 0.45, gout.to(dev))
    assert relerr(out, want_out) < 3e-2 and relerr(gin, want_gin) < 5e-2


def test_unet_forward_full_vs_golden(dev, golden_dir):
    """configs/sda_unet.yml architecture, seed-0 weights, one window: against the REFERENCE's own output slice."""
    import climate2weather_b200 as c2w
    g = np.load(golden_dir / "full_arch.npz")
    torch.manual_seed(0)
    net = c2w.ScoreUNet(52, 512, hidden_channels=[128, 128, 256, 384, 512], hidden_blocks=[3] * 5, attention_levels=[4], activation=torch.nn.SiLU)
    x = torch.randn(1, 52, 128, 128, generator=torch.Generator().manual_seed(int(g["x_seed"])))
    with torch.no_grad():
        y = net.to(dev)(x.to(dev), torch.tensor(float(g["t"])))
    e = relerr(y[0, :, ::8, ::8], torch.from_numpy(g["out_slice"]))
    e2 = rel_l2(y[0, :, ::8, ::8], torch.from_numpy(g["out_slice"]))
    print(f"\nfull UNet forward vs reference slice: max-abs ratio {e:.3e}, rel-L2 {e2:.3e}; "
          f"std {y.std().item():.4f} vs {float(g['out_std']):.4f}")
    assert e < 3e-2 and e2 < 2e-2
    assert abs(y.std().item() - float(g["out_std"])) < 1e-2 * float(g["out_std"])


def test_window_score_vs_oracle_and_chunk_invariance(dev, golden_dir):
    """Default / Batched composition (src/thor/score.py:76-88, :111-185): the values against the reference's golden
    output, and BIT-EXACT equality across chunk sizes (the index map must not depend on batching)."""
    import climate2weather_b200 as c2w
    g = np.load(golden_dir / "small_path.npz")
    net, _ = make_small(dev)
    pipe = c2w.SDAPipeline()
    x = torch.from_numpy(g["x"])
    t = torch.tensor(float(g["t"]))
    outs = []
    for mw in (None, 1, 2, 3, 5):
        sf = c2w.DefaultScoreFunction(net, markov_order=2, noise_process=pipe)
        sf.max_windows = mw
        outs.append(sf(x.to(dev), t).cpu())
    e = relerr(outs[0], torch.from_numpy(g["eps_default"]))
    e2, ef = rel_l2(outs[0], torch.from_numpy(g["eps_default"])), frame_rel_l2(outs[0], torch.from_numpy(g["eps_default"]))
    print(f"\nwindow score vs reference: max-abs ratio {e:.3e}, rel-L2 {e2:.3e}, worst frame rel-L2 {ef:.3e}")
    assert e < 3e-2 and e2 < 2e-2 and ef < 3e-2
    for o in outs[1:]:
        assert torch.equal(o, outs[0])
    bf = c2w.BatchedScoreFunction(net, markov_order=2, noise_process=pipe, batch_size=3, device=dev)
    assert torch.equal(bf(x, t), outs[0])  # CPU tensor in, CPU tensor out, like the reference


def _index_coded_net(dev, k, C, mode):
    """One-level ScoreUNet (head conv -> one residual block -> tail conv, the launch sequence of level 0 of the real
    net incl. the fused compose epilogue) whose weights make the output an INTEGER CODE of where it came from:

      the residual block is switched off (second conv zero) and the head conv copies window channel (tau, c) through
      (centre tap 1), so the 128-channel stream holds the gathered window in its first w*C channels; the tail is
        "window": out[(tau, c)] = in[(0, c)]        -> with x[f] = f the UNet output is the WINDOW index j
        "slot"  : weights 0, bias[(tau, c)] = tau*C + c   -> the output is the window-CHANNEL index
        "pixel" : out[(tau, c)] = in[(tau, c)]      -> the output is the input pixel (fold o unfold = id)
        "centre-sum": out[(k, c)] = sum_tau in[(tau, c)], every other output zero
    All values are small integers, exact in bf16 operands and fp32 accumulators.  The residual branch ends in a zero
    conv, so its input gradient is exactly 0 and the input-gradient pass is the transpose of the tail alone."""
    import climate2weather_b200 as c2w
    w = 2 * k + 1
    net = c2w.ScoreUNet(channels=C * w, embedding_dim=64, hidden_channels=[128], hidden_blocks=[1], attention_levels=[], activation=torch.nn.SiLU)
    sd = {name: torch.zeros_like(p) for name, p in net.state_dict().items()}
    for ch in range(C * w):
        sd["unet.heads.0.weight"][ch, ch, 1, 1] = 1.0
        if mode == "window":
            sd["unet.tails.0.weight"][ch, ch % C, 1, 1] = 1.0
        elif mode == "pixel":
            sd["unet.tails.0.weight"][ch, ch, 1, 1] = 1.0
        elif mode == "centre-sum":
            sd["unet.tails.0.weight"][k * C + ch % C, ch, 1, 1] = 1.0
        else:
            sd["unet.tails.0.bias"][ch] = float(ch)
    net.load_state_dict(sd)
    return net.to(dev)


_COMPOSE_CASES = [
    (13, 128, 128, (None, 1)),             # one window: head, centre and tail slots all come from window 0
    (14, 128, 128, (None, 1, 2)),          # two windows; chunk 1 -> first batch != last batch
    (26, 128, 128, (None, 1, 3, 5, 14)),   # ragged last batch (3, 5), first == last (14)
    (40, 16, 64, (None, 7)),
]
_COMPOSE_L168 = (168, 128, 128, (None, 32, 100))  # BASELINE config 2 geometry: 156 windows (C = 4 and one other count)


@pytest.mark.parametrize("C,L,H,W,chunks", [(C,) + case for C in range(1, 9) for case in _COMPOSE_CASES] +
                         [(C,) + _COMPOSE_L168 for C in (4, 3)])
def test_compose_index_bit_exact(dev, golden_dir, C, L, H, W, chunks):
    """K0 gather + the fold (K5 compose epilogue for C = 4, compose_generic_kernel for any other count;
    src/thor/score.py:68-88, :111-154) through c2w_window_score on index-coded networks at k = 6: the composed output
    must equal, as INTEGERS, the (window, window-channel, pixel) the oracle's fold map names — for every chunking of the
    window range (the batched variant emits the head slots with the first batch and the tail slots with the last,
    src/thor/score.py:124-141)."""
    import climate2weather_b200 as c2w
    k = 6
    f = score_ref.fold_index(L, k, C)  # [L, C, (window, window-channel)], pinned against the reference (index_maps.npz)
    key = f"fold_{L}_{k}_{C}"
    idx = np.load(golden_dir / "index_maps.npz")
    if key in idx.files:  # the reference's own fold on a (window*1000 + channel)-coded tensor
        assert np.array_equal(idx[key][:, :, 0, 0], f[..., 0] * 1000 + f[..., 1])
    pipe = c2w.SDAPipeline()
    t = torch.tensor(0.5)
    frame_code = torch.arange(L, dtype=torch.float32).reshape(L, 1, 1, 1).expand(L, C, H, W).contiguous()
    hh, ww, cc = torch.meshgrid(torch.arange(H), torch.arange(W), torch.arange(C), indexing="ij")
    pix_code = ((hh * W + ww + 64 * cc) % 251).permute(2, 0, 1).float()  # [C, H, W], < 256: exact in bf16
    pix_x = ((pix_code[None] + 17 * frame_code) % 251).contiguous()  # varies with frame, channel and pixel
    want = {
        "window": torch.from_numpy(f[..., 0]).float().reshape(L, C, 1, 1).expand(L, C, H, W),
        "slot": torch.from_numpy(f[..., 1]).float().reshape(L, C, 1, 1).expand(L, C, H, W),
        "pixel": pix_x,
    }
    for mode in ("window", "slot", "pixel"):
        net = _index_coded_net(dev, k, C, mode)
        x = pix_x if mode == "pixel" else frame_code
        for mw in chunks:
            sf = c2w.DefaultScoreFunction(net, markov_order=k, noise_process=pipe)
            sf.max_windows = mw
            got = sf.score_fn(x.to(dev), t).cpu()
            assert got.dtype == torch.float32
            assert torch.equal(got, want[mode]), (mode, mw, (got != want[mode]).nonzero()[:4].tolist())


@pytest.mark.parametrize("C,L,split", [(C, L, split) for C in range(1, 9) for L, split in
                                        ((13, "all"), (14, "halves"), (26, "every3"))] +
                         [(C, 168, "observed") for C in (4, 3)])
def test_compose_by_window_lists_bit_exact(dev, C, L, split):
    """c2w_window_score_sel with a score output (exact_grad: the observed selection on the stashing engine, the others on
    the plain one): two window LISTS fold into one eps exactly like the contiguous c2w_window_score — integers out of
    index-coded networks at k = 6, H = W = 128, C variables per frame; lists shorter and longer than a chunk, first /
    last window in either."""
    import climate2weather_b200 as c2w
    k, H, W = 6, 128, 128
    nw = L - 2 * k
    f = score_ref.fold_index(L, k, C)
    frame_code = torch.arange(L, dtype=torch.float32).reshape(L, 1, 1, 1).expand(L, C, H, W).contiguous()
    every = {"all": [list(range(nw)), []], "halves": [[1], [0]], "every3": [[j for j in range(nw) if j % 3 == 0],
             [j for j in range(nw) if j % 3]], "observed": [[j for j in range(nw) if (j + k) % 6 == 0 or j in (0, nw - 1)],
             [j for j in range(nw) if not ((j + k) % 6 == 0 or j in (0, nw - 1))]]}[split]
    for mode in ("window", "slot"):
        net = _index_coded_net(dev, k, C, mode)
        x = frame_code.permute(0, 2, 3, 1).contiguous().to(dev)
        eps = torch.full_like(x, float("nan"))
        plain = net.engine(C, 2 * k + 1, H, W, dev, max_windows=5, vjp=False)       # lists longer than a chunk
        stash = net.engine(C, 2 * k + 1, H, W, dev, max_windows=max(1, len(every[0])), vjp=True)
        if every[1]:
            plain.window_score_sel(x, 0, torch.tensor(every[1], dtype=torch.int32, device=dev), 0.5, nw, eps)
        stash.window_score_sel(x, 0, torch.tensor(every[0], dtype=torch.int32, device=dev), 0.5, nw, eps)
        torch.cuda.synchronize()
        got = eps.permute(0, 3, 1, 2).cpu()
        want = torch.from_numpy(f[..., 0 if mode == "window" else 1]).float().reshape(L, C, 1, 1).expand(L, C, H, W)
        assert torch.equal(got, want), (mode, split, (got != want).nonzero()[:4].tolist())


@pytest.mark.parametrize("C,k", [(C, 2) for C in range(1, 9)] + [(5, 6), (8, 6)])  # k = 6: C * w > 64 channels
def test_window_adjoint_index_bit_exact(dev, C, k):
    """The window adjoints (compose_adjoint_kernel -> input-gradient pass -> unfold_adjoint_kernel) as exact integers,
    through c2w_window_score_backward (range form) and c2w_window_score_backward_sel (list form), each right after its
    stashing forward; integer cot and base in [-8, 8] (vjp accumulates onto base):
      "pixel" (identity Jacobian): vjp[f] = base[f] + cot[f] if the source window of frame f (score_ref.fold_index:
          centre slot, or the head / tail slots of the first / last window) is in the set, else base[f] to the bit;
      "centre-sum": vjp[f] = base[f] + sum over windows j of the set with j <= f <= j + 2k of cot[j + k].
    On the whole trajectory (first / last window in and out of the set) and on time-sharded local slices
    (frame_global0 > 0)."""
    nw, H, W = 8, 32, 32
    w, L = 2 * k + 1, nw + 2 * k
    src = score_ref.fold_index(L, k, C)[:, 0, 0]  # source window of each global frame
    g = torch.Generator().manual_seed(90 + C)
    x, cot, base = (torch.randint(-8, 9, (L, H, W, C), generator=g).float() for _ in range(3))
    # (local slice [lo, hi), window sets: ranges (first, n) and lists); a set's windows lie inside the slice
    cases = [((0, L), [(0, nw), (0, 3), (5, 3), (2, 4)], [[0, 2, 5, 7], [1, 4, 6], [7], [0]]),
             ((3, L), [(3, 5), (4, 2)], [[3, 5, 7], [4, 6]]),   # the last rank's slice: holds the last window
             ((2, 6 + 2 * k), [(2, 4)], [[2, 5], [3, 4, 5]])]   # a middle rank's slice
    for mode in ("pixel", "centre-sum"):
        net = _index_coded_net(dev, k, C, mode)
        eng = net.engine(C, w, H, W, dev, max_windows=nw, vjp=True)
        for (lo, hi), ranges, lists in cases:
            xd, cd = (v[lo:hi].contiguous().to(dev) for v in (x, cot))
            for wins, contiguous in [(list(range(a, a + n)), True) for a, n in ranges] + [(li, False) for li in lists]:
                want = base.clone()
                for f in range(L):
                    if mode == "pixel":
                        want[f] += cot[f] if src[f] in wins else 0.0
                    else:
                        for j in wins:
                            if j <= f <= j + 2 * k:
                                want[f] += cot[j + k]
                want = want[lo:hi]
                got = []
                if contiguous:
                    v = base[lo:hi].contiguous().to(dev)
                    eng.window_score(xd, lo, wins[0], len(wins), nw, 0.5, torch.empty_like(xd))
                    eng.window_score_backward(cd, lo, wins[0], len(wins), nw, v)
                    got.append(("range", v))
                wl = torch.tensor(wins, dtype=torch.int32, device=dev)
                pos = torch.full((nw,), -1, dtype=torch.int32)
                pos[wins] = torch.arange(len(wins), dtype=torch.int32)
                v = base[lo:hi].contiguous().to(dev)
                eng.window_score_sel(xd, lo, wl, 0.5, nw)
                eng.window_score_backward_sel(cd, lo, wl, pos.to(dev), nw, v)
                got.append(("list", v))
                torch.cuda.synchronize()
                for form, v in got:
                    v = v.cpu()
                    assert torch.equal(v, want), (mode, form, (lo, hi), wins, (v != want).nonzero()[:4].tolist())


# ------------------------------------------------------------------------------------------------ K6 / K7
def _guide_call(lib, dev, x, eps, y, mode, mu, sigma, mu_n, sigma_n, t_step, s_step, own_lo=0, own_n=None, frame0=0):
    from climate2weather_b200 import _lib
    L, C, H, W = x.shape
    xd = x.permute(0, 2, 3, 1).contiguous().to(dev)
    ed = eps.permute(0, 2, 3, 1).contiguous().to(dev)
    own_n = L if own_n is None else own_n
    g = _lib.Guide()
    g.x, g.eps = xd.data_ptr(), ed.data_ptr()
    eo = torch.zeros_like(xd)
    parts = torch.zeros(own_n * (H // s_step), device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    yd = y.to(dev).contiguous() if y is not None else None
    g.eps_out, g.partials, g.nan_flag = eo.data_ptr(), parts.data_ptr(), flag.data_ptr()
    g.y = yd.data_ptr() if yd is not None else None
    for i in range(4):
        g.std2[i] = STD[i] ** 2
        g.gamma[i] = GAMMA
    g.mu, g.sigma, g.mu_next, g.sigma_next = mu, sigma, mu_n, sigma_n
    g.t_step, g.s_step, g.H, g.W = t_step, s_step, H, W
    g.frame_global0, g.own_lo, g.own_n, g.mode = frame0, own_lo, own_n, mode
    _lib.check(lib.c2w_guided_step(ctypes.byref(g), stream()), "c2w_guided_step")
    torch.cuda.synchronize()
    return xd.permute(0, 3, 1, 2).cpu(), eo.permute(0, 3, 1, 2).cpu(), parts.cpu(), int(flag.item())


def test_guided_eps_and_predictor_vs_oracle(lib, dev):
    """K6 against the oracle's autograd guidance (exact_grad=False, src/thor/score.py:44-60) and predictor
    (src/thor/pipelines.py:41-46) on the shipped operator (t_step 6, s_step 16, 128x128): fp32 -> 1e-5 relative."""
    g = torch.Generator().manual_seed(21)
    L, C, H, W = 14, 4, 128, 128
    x = torch.randn(L, C, H, W, generator=g)
    eps = torch.randn(L, C, H, W, generator=g)
    y = score_ref.coarse_grain(torch.randn(L, C, H, W, generator=g), 6, 16)
    std = torch.tensor(STD).reshape(1, 4, 1, 1)
    p = pipeline_ref.RefPipeline()
    for tval in (0.95, 0.5, 0.05):
        t = torch.tensor(tval)
        tn = t - 1 / 256
        mu, sg, mun, sgn = (float(v) for v in (p.mu(t), p.sigma(t), p.mu(tn), p.sigma(tn)))
        want_eps = score_ref.guided_score_closed_form(eps, x, t, y, std, GAMMA, 6, 16)
        _, got_eps, parts, flag = _guide_call(lib, dev, x, eps, y, 1, mu, sg, 0.0, 0.0, 6, 16)
        assert flag == 0
        assert relerr(got_eps, want_eps) < 1e-5
        assert abs(parts.double().sum().item() / want_eps.double().square().sum().item() - 1) < 1e-5
        want_x = p.mu(tn) * ((x - p.sigma(t) * want_eps) / p.mu(t)) + p.sigma(tn) * want_eps
        got_x, _, _, flag = _guide_call(lib, dev, x, eps, y, 0, mu, sg, mun, sgn, 6, 16)
        assert flag == 0
        assert relerr(got_x, want_x) < 1e-5


def test_guided_step_matches_reference_autograd(lib, dev):
    """Same kernel against the reference formulation itself (jacrev == autograd.grad of log p) on a small case."""
    g = torch.Generator().manual_seed(5)
    L, C, H, W = 7, 4, 16, 16
    x = torch.randn(L, C, H, W, generator=g)
    eps = torch.randn(L, C, H, W, generator=g)
    y = score_ref.coarse_grain(torch.randn(L, C, H, W, generator=g), 3, 8)
    std = torch.tensor(STD).reshape(1, 4, 1, 1)
    t = torch.tensor(0.4)
    mu, sg = (float(v) for v in score_ref.mu_sigma(t))
    # autograd with eps held constant (torch.set_grad_enabled(False) around the network, src/thor/score.py:51-52)
    xg = x.clone().requires_grad_(True)
    x0 = (xg - sg * eps) / mu
    err = y - score_ref.coarse_grain(x0, 3, 8)
    var = std ** 2 + GAMMA * (sg / mu) ** 2
    (J,) = torch.autograd.grad(-(err ** 2 / var).sum() / 2, xg)
    _, got, _, _ = _guide_call(lib, dev, x, eps, y, 1, mu, sg, 0.0, 0.0, 3, 8)
    assert relerr(got, eps - sg * J) < 1e-5


def test_guided_step_unconditioned_and_sharded_frames(lib, dev):
    """y = NULL is the plain predictor; with frame_global0 != 0 observed frames follow the GLOBAL index."""
    g = torch.Generator().manual_seed(6)
    L, C, H, W = 12, 4, 32, 32
    x = torch.randn(L, C, H, W, generator=g)
    eps = torch.randn(L, C, H, W, generator=g)
    got_x, _, _, _ = _guide_call(lib, dev, x, eps, None, 0, 0.8, 0.6, 0.85, 0.52, 1, 16)
    want = 0.85 * ((x - 0.6 * eps) / 0.8) + 0.52 * eps
    assert relerr(got_x, want) < 1e-6
    y = score_ref.coarse_grain(torch.randn(L, C, H, W, generator=g), 6, 16)
    std = torch.tensor(STD).reshape(1, 4, 1, 1)
    t = torch.tensor(0.5)
    mu, sg = (float(v) for v in score_ref.mu_sigma(t))
    want = score_ref.guided_score_closed_form(eps, x, t, y, std, GAMMA, 6, 16)
    # local shard = global frames [4, 12); only frames [5, 11) are owned
    _, got, _, _ = _guide_call(lib, dev, x[4:], eps[4:], y, 1, mu, sg, 0, 0, 6, 16, own_lo=1, own_n=6, frame0=4)
    assert relerr(got[1:7], want[5:11]) < 1e-5
    assert float(got[0].abs().max()) == 0.0 and float(got[7].abs().max()) == 0.0  # not owned -> untouched


def test_corrector_update_vs_oracle(lib, dev):
    from climate2weather_b200 import _lib
    g = torch.Generator().manual_seed(8)
    L, C, H, W = 6, 4, 16, 16
    x, eps, z = (torch.randn(L, C, H, W, generator=g) for _ in range(3))
    tau, sgn = 0.5, 0.7
    delta = tau / eps.square().mean()
    want = x - (delta * eps + torch.sqrt(2 * delta) * z) * sgn
    xd, ed, zd = (v.permute(0, 2, 3, 1).contiguous().to(dev) for v in (x, eps, z))
    sumsq = eps.double().square().sum().reshape(1).to(dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    _lib.check(lib.c2w_corrector_update(xd.data_ptr(), ed.data_ptr(), zd.data_ptr(), sumsq.data_ptr(),
                                        float(x.numel()), tau, sgn, 0, L * H * W, 0, 0, flag.data_ptr(), stream()), "corr")
    torch.cuda.synchronize()
    assert relerr(xd.permute(0, 3, 1, 2), want) < 1e-5 and int(flag.item()) == 0
    # on-chip Philox: unit-variance, zero-mean, and identical for any split of the pixel range (sharding-invariant)
    x0 = torch.zeros(L, H, W, C, device=dev)
    e0 = torch.zeros_like(x0)
    one = torch.ones(1, dtype=torch.float64, device=dev)  # delta = tau / (1/count) -> choose count so delta = 0.5
    _lib.check(lib.c2w_corrector_update(x0.data_ptr(), e0.data_ptr(), None, one.data_ptr(), 1.0, 0.5, 1.0, 0,
                                        L * H * W, 1234, 3, flag.data_ptr(), stream()), "corr")
    xa = x0.clone()
    x1 = torch.zeros_like(x0)
    half = (L // 2) * H * W
    _lib.check(lib.c2w_corrector_update(x1.data_ptr(), e0.data_ptr(), None, one.data_ptr(), 1.0, 0.5, 1.0, 0, half,
                                        1234, 3, flag.data_ptr(), stream()), "corr")
    _lib.check(lib.c2w_corrector_update(x1.reshape(-1)[half * 4:].data_ptr(), e0.data_ptr(), None, one.data_ptr(), 1.0,
                                        0.5, 1.0, half, L * H * W - half, 1234, 3, flag.data_ptr(), stream()), "corr")
    torch.cuda.synchronize()
    assert torch.equal(xa, x1)
    zgen = -xa  # x = 0 - (0 + sqrt(2*0.5) z) * 1
    assert abs(zgen.mean().item()) < 0.05 and abs(zgen.std().item() - 1) < 0.05


# ------------------------------------------------------------------------------------------------ sampler
def test_sampler_vs_reference_golden(dev, golden_dir):
    """Guided predictor-corrector (steps=3, corrections=1) and predictor-only (steps=4) runs with the reference's
    own noise stream, against the reference's outputs.  Tolerance 5e-2 of max-abs: the UNet's bf16 error is
    amplified by 1/mu(t) ~ 1e3 in the first steps (SURVEY.md §7 hard parts)."""
    import climate2weather_b200 as c2w
    g = np.load(golden_dir / "small_path.npz")
    net, _ = make_small(dev)
    pipe = c2w.SDAPipeline()
    pipe.rng = "reference"
    x = torch.from_numpy(g["x"])
    y = torch.from_numpy(g["yobs"])
    std = torch.tensor(STD).reshape(1, 4, 1, 1)
    pool = torch.nn.AvgPool2d(8, stride=8, padding=0)
    sf = c2w.BatchedScoreFunction(net, markov_order=2, noise_process=pipe, batch_size=4, device=dev)
    sf.condition_on(A=lambda v: pool(v[..., ::3, :, :, :]), y=y, std=std, gamma=GAMMA, exact_grad=False)
    ge = relerr(sf(x, torch.tensor(float(g["t"]))), torch.from_numpy(g["eps_guided_approx"]))
    print(f"\nguided eps rel-err vs reference: {ge:.3e}")
    assert ge < 3e-2
    torch.manual_seed(5)
    s1 = pipe.sample(sf, x, steps=3, corrections=1, tau=0.5, show_progressbar=False)
    e1 = relerr(s1, torch.from_numpy(g["sample_c1"]))
    s0 = pipe.sample(sf, x, steps=4, corrections=0, tau=0.5, show_progressbar=False)
    e0 = relerr(s0, torch.from_numpy(g["sample_c0"]))
    l1, l0 = rel_l2(s1, torch.from_numpy(g["sample_c1"])), rel_l2(s0, torch.from_numpy(g["sample_c0"]))
    f1, f0 = frame_rel_l2(s1, torch.from_numpy(g["sample_c1"])), frame_rel_l2(s0, torch.from_numpy(g["sample_c0"]))
    print(f"sampler vs reference: max-abs ratio c1 {e1:.3e} c0 {e0:.3e}; rel-L2 c1 {l1:.3e} c0 {l0:.3e}; "
          f"worst frame rel-L2 c1 {f1:.3e} c0 {f0:.3e}")
    assert s1.device.type == "cpu" and s1.shape == x.shape
    assert e1 < 5e-2 and e0 < 5e-2 and l1 < 3e-2 and l0 < 3e-2 and f1 < 5e-2 and f0 < 5e-2
    sf1 = c2w.DefaultScoreFunction(net, markov_order=2, noise_process=pipe)
    s2 = pipe.sample(sf1, x[:5], steps=3, show_progressbar=False, device=dev)
    assert s2.is_cuda
    assert relerr(s2, torch.from_numpy(g["sample_one_window"])) < 5e-2


@pytest.mark.parametrize("C", [1, 2, 3, 6, 8])
def test_other_variable_counts_vs_oracle(dev, C):
    """The reference's score functions and sampler are written for any number of variables per frame
    (src/thor/score.py:68-88, :111-154); the shipped configs have C = 4 (exp/downscaling.py:101), which is the fused
    float4 path.  C != 4 runs the separate fold kernel and the scalar-access instances of the guidance / corrector /
    adjoint kernels: composed score, closed-form and exact-gradient guided score and a short predictor-corrector run
    against the fp32 oracle, same tolerances as the 4-variable tests; the fold is index work -> chunk-invariant to the
    bit; the backward over a window range equals the backward over the same windows as a list."""
    import climate2weather_b200 as c2w
    k, L, H, W = 2, 11, 32, 32
    cfg = dict(SMALL, channels=C * (2 * k + 1))
    torch.manual_seed(11 + C)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, **cfg)
    ref = unet_ref.RefNet({n: v.detach().clone() for n, v in net.state_dict().items()}, cfg)
    net = net.to(dev)
    g = torch.Generator().manual_seed(50 + C)
    x = torch.randn(L, C, H, W, generator=g)
    y = score_ref.coarse_grain(torch.randn(L, C, H, W, generator=g), 3, 8)
    std = torch.tensor([0.1 + 0.05 * c for c in range(C)]).reshape(1, C, 1, 1)
    t = torch.tensor(0.45)
    pipe = c2w.SDAPipeline()
    with torch.no_grad():
        want = score_ref.window_score(ref, x, t, k)
    outs = []
    for mw in (None, 3):
        sf = c2w.DefaultScoreFunction(net, markov_order=k, noise_process=pipe)
        sf.max_windows = mw
        outs.append(sf.score_fn(x.to(dev), t).cpu())
    e = relerr(outs[0], want)
    assert outs[0].shape == x.shape and e < 3e-2, e
    assert torch.equal(outs[0], outs[1])
    # closed-form guidance (exact_grad=False, every shipped config)
    sf = c2w.BatchedScoreFunction(net, markov_order=k, noise_process=pipe, batch_size=4, device=dev)
    sf.condition_on(A=c2w.CoarseGrain(3, 8), y=y, std=std, gamma=GAMMA, exact_grad=False)
    with torch.no_grad():
        want_g = score_ref.guided_score(ref, x, t, k, y, std, GAMMA, 3, 8, exact_grad=False)
    eg = relerr(sf(x, t), want_g)
    assert eg < 3e-2, eg
    # predictor + one Langevin correction per step, the corrector noise drawn as the reference draws it
    ref_pipe = pipeline_ref.RefPipeline()
    score = lambda xx, tt: score_ref.guided_score(ref, xx, tt, k, y, std, GAMMA, 3, 8, exact_grad=False)
    torch.manual_seed(5)
    want_s = ref_pipe.sample(score, x, steps=3, corrections=1, tau=0.5)
    pipe.rng = "reference"
    torch.manual_seed(5)
    got_s = pipe.sample(sf, x, steps=3, corrections=1, tau=0.5, show_progressbar=False)
    es, ls = relerr(got_s, want_s), rel_l2(got_s, want_s)
    print(f"\nC={C}: score {e:.3e}, guided {eg:.3e}, sampler max-abs ratio {es:.3e} rel-L2 {ls:.3e}")
    assert got_s.shape == x.shape and es < 5e-2 and ls < 3e-2
    # on-chip Philox noise: finite
    pipe2 = c2w.SDAPipeline()
    assert torch.isfinite(pipe2.sample(sf, x, steps=2, corrections=1, tau=0.5, show_progressbar=False, seed=3)).all()
    # exact_grad=True (gradient through the UNet, src/thor/score.py:28-35): one stashing chunk and several
    want_e = score_ref.guided_score(ref, x, t, k, y, std, GAMMA, 3, 8, exact_grad=True)
    for mw in (None, 2):
        sfe = c2w.DefaultScoreFunction(net, markov_order=k, noise_process=pipe2)
        sfe.max_windows = mw
        sfe.condition_on(A=c2w.CoarseGrain(3, 8), y=y, std=std, gamma=GAMMA, exact_grad=True)
        ee = relerr(sfe(x.to(dev), t).cpu(), want_e)
        assert ee < 4e-2 and ee < 0.5 * relerr(want_g, want_e), (mw, ee)
    _assert_backward_range_equals_list(net, x, k, t, dev)


def test_per_sample_times_and_dsm_loss(dev, golden_dir):
    """ScoreUNet with one diffusion time per sample (model/score.py:61) and SDAPipeline.loss
    (src/thor/pipelines.py:27-35) against the oracle with the same t and eps; chunked through a 2-window workspace."""
    import climate2weather_b200 as c2w
    net, ref = make_small(dev)
    g = torch.Generator().manual_seed(41)
    x = torch.randn(5, 20, 32, 32, generator=g)
    t = torch.tensor([0.05, 0.9, 0.33, 0.33, 0.71])
    want = ref(x, t.reshape(-1, 1, 1, 1))
    net.DEFAULT_MAX_WINDOWS = 2
    with torch.no_grad():
        got = net(x.to(dev), t.reshape(-1, 1, 1, 1).to(dev))
    e = relerr(got, want)
    print(f"\nper-sample-t forward rel-err vs oracle: {e:.3e}")
    assert e < 3e-2
    # each sample must equal the single-t call at its own time (the modulation is per sample, nothing else is)
    with torch.no_grad():
        one = net(x[1:2].to(dev), torch.tensor(0.9))
    assert relerr(got[1:2], one) < 1e-2
    # DSM loss: same draws as the oracle (torch.rand for t, then randn_like for eps, on the CPU generator)
    pipe = c2w.SDAPipeline()
    torch.manual_seed(7)
    tt = torch.rand(5, 1, 1, 1)
    eps = torch.randn_like(x)
    want_loss = pipeline_ref.RefPipeline().loss(ref, x, t=tt, eps=eps)
    torch.manual_seed(7)
    xt = pipe.mu(tt) * x + pipe.sigma(tt) * eps
    with torch.no_grad():
        got_loss = (net(xt.to(dev), tt.to(dev)).cpu() - eps) ** 2
    assert relerr(got_loss, want_loss) < 6e-2  # squared error of a 3e-2 output


def test_reference_snapshot_forward(dev, golden_dir):
    """The unpickled reference snapshot (fp16 EMA module) runs through the CUDA path and reproduces the reference's
    own forward on the same weights (fixture from tests/golden/make_golden.py)."""
    import pickle

    import climate2weather_b200.compat as compat
    compat.install()
    with open(golden_dir / "snapshot_tiny.pkl", "rb") as f:
        snap = pickle.load(f)
    exp = np.load(golden_dir / "snapshot_tiny_expect.npz")
    net = snap["ema"].to(dev).eval()
    with torch.no_grad():
        y = net(torch.from_numpy(exp["x"]).to(dev), torch.tensor(float(exp["t"])))
    e = relerr(y, torch.from_numpy(exp["y"]))
    print(f"\nsnapshot forward rel-err vs reference: {e:.3e}")
    assert e < 3e-2


@pytest.mark.parametrize("every", [0, 1])
def test_sampler_raises_on_nan_like_the_reference(dev, every):
    """src/thor/pipelines.py:90-91: `raise ValueError("NaN detected in sample")`.  With a per-step check the flag is
    read asynchronously and inspected one step later; without it, at the end — both raise the reference's error, and a
    clean run with the per-step check returns the same trajectory as one without."""
    import climate2weather_b200 as c2w

    torch.manual_seed(5)
    net = c2w.ScoreUNet(activation=torch.nn.SiLU, **SMALL).to(dev)
    pipe = c2w.SDAPipeline()
    pipe.nan_check_every = every
    sf = c2w.BatchedScoreFunction(net, markov_order=2, noise_process=pipe, batch_size=4, device=dev)
    g = torch.Generator().manual_seed(6)
    noise = torch.randn(9, 4, 32, 32, generator=g)
    clean = pipe.sample(sf, noise, steps=4, show_progressbar=False)
    assert torch.isfinite(clean).all()
    pipe0 = c2w.SDAPipeline()
    assert torch.equal(clean, pipe0.sample(sf, noise, steps=4, show_progressbar=False))
    bad = noise.clone()
    bad[4, 1, 7, 9] = float("nan")
    with pytest.raises(ValueError, match="NaN detected in sample"):
        pipe.sample(sf, bad, steps=4, show_progressbar=False)
    # and the runtime recovers for the next trajectory
    assert torch.equal(clean, pipe.sample(sf, noise, steps=4, show_progressbar=False))


def test_driver_flow_from_snapshot(dev, golden_dir):
    """The hot-path lines of exp/downscaling.py:_run_impl, in order, on the reference-pickled snapshot fixture:
    pickle.load -> markov order from dataset_kwargs (:110-118) -> net.eval() (:125) -> A = AvgPool2d(s)(x[::t]) closure
    (:129-132) -> BatchedScoreFunction(...) (:208-214) -> condition_on(A=, y=, std=[1,C,1,1], gamma=, exact_grad=False)
    (:236-242) -> pipeline.sample(score_fn, noise (CPU), steps=, corrections=, tau=) (:254-261) -> .float().cpu().numpy().
    The same flow through the oracle on the snapshot's (fp16) weights is the ground truth."""
    import pickle

    import climate2weather_b200.compat as compat
    compat.install()
    from thor.score import BatchedScoreFunction  # resolves to this package, as in the driver

    with open(golden_dir / "snapshot_tiny.pkl", "rb") as f:
        snapshot_data = pickle.load(f)
    markov_window = snapshot_data["dataset_kwargs"]["train"]["window"]
    markov_order = markov_window // 2
    pipeline = snapshot_data["pipeline"]
    net = snapshot_data["ema"].to(dev)
    net.eval()
    t_step, s_step = 2, 4
    pool = torch.nn.AvgPool2d(s_step, stride=s_step, padding=0)

    def A(x):
        return pool(x[..., ::t_step, :, :, :])

    g = torch.Generator().manual_seed(17)
    L, C, H, W = 9, 4, 16, 16
    truth = torch.randn(L, C, H, W, generator=g)
    y = A(truth)
    std = torch.tensor(STD).reshape(1, C, 1, 1)
    score_function = BatchedScoreFunction(net, markov_order=markov_order, noise_process=pipeline, batch_size=4,
                                          device=dev)
    score_function.condition_on(A=A, y=y, std=std, gamma=GAMMA, exact_grad=False)
    noise = torch.randn(L, C, H, W, generator=g)
    out = pipeline.sample(score_function, noise, steps=5, corrections=0, tau=0.5, show_progressbar=False)
    out_np = out.to(torch.float32).cpu().numpy()
    assert out_np.shape == (L, C, H, W) and np.isfinite(out_np).all()
    # ground truth: oracle network on the snapshot's weights, oracle guidance and sampler
    cfg = dict(channels=12, embedding_dim=64, hidden_channels=(64, 64), hidden_blocks=(1, 1), attention_levels=(1,),
               kernel_size=3)
    ref = unet_ref.RefNet({k: v.float().cpu() for k, v in net.state_dict().items()}, cfg)

    def guided(xx, tt):
        with torch.no_grad():
            eps = score_ref.window_score(ref, xx, tt, markov_order, batch_size=4)
        return score_ref.guided_score_closed_form(eps, xx, tt, y, std, GAMMA, t_step, s_step)

    want = pipeline_ref.RefPipeline().sample(guided, noise, steps=5, corrections=0, tau=0.5)
    e = relerr(out, want)
    print(f"\ndriver flow (snapshot -> guided sampling) rel-err vs oracle: {e:.3e}")
    assert e < 5e-2


# ------------------------------------------------------------------------------------------------ VJP (exact_grad)
@pytest.mark.parametrize("C", [64, 128, 384, 512])
@pytest.mark.parametrize("down", [0, 1])
def test_layernorm_backward_vs_autograd(lib, dev, C, down):
    """LayerNorm forward (with its 1/std stash) + backward kernel vs torch autograd of the oracle LayerNorm:
    bf16 in/out, fp32 math -> 2^-6 of the gradient scale."""
    from climate2weather_b200 import _lib
    g = torch.Generator().manual_seed(C + down)
    n, H, W = 2, 4, 8
    x = (torch.randn(n, H, W, C, generator=g) * 1.5 + 0.3).to(torch.bfloat16)
    mod = torch.randn(C, generator=g)
    up = 2 if down else 1
    gy = torch.randn(n, H * up, W * up, C, generator=g).to(torch.bfloat16)
    gres = torch.randn(n, H, W, C, generator=g).to(torch.bfloat16)
    xd, gyd, gresd, modd = x.to(dev), gy.to(dev), gres.to(dev), mod.to(dev)
    y = torch.empty(n, H, W, C, device=dev, dtype=torch.bfloat16)
    inv = torch.empty(n * H * W, device=dev)
    _lib.check(lib.c2w_op_layernorm_inv(xd.data_ptr(), modd.data_ptr(), y.data_ptr(), inv.data_ptr(), n * H * W, C,
                                        stream()), "ln_inv")
    if down:  # the backward reads y from the first pixel of each 2x2 block of the upsampled tensor
        ysrc = y.repeat_interleave(2, dim=1).repeat_interleave(2, dim=2).contiguous()
    else:
        ysrc = y
    out = torch.empty(n, H, W, C, device=dev, dtype=torch.bfloat16)
    _lib.check(lib.c2w_op_layernorm_bwd(gyd.data_ptr(), ysrc.data_ptr(), inv.data_ptr(), gresd.data_ptr(), out.data_ptr(),
                                        n * H * W, C, H, W, down, stream()), "ln_bwd")
    torch.cuda.synchronize()
    v = (x.float() + mod).permute(0, 3, 1, 2).requires_grad_(True)
    yr = unet_ref.channel_layernorm(v)
    if down:
        yr = F.interpolate(yr, scale_factor=2, mode="nearest")
    (gv,) = torch.autograd.grad(yr, v, gy.float().permute(0, 3, 1, 2))
    want = gv.permute(0, 2, 3, 1) + gres.float()
    assert relerr(out.float().cpu(), want) < 2 ** -6


@pytest.mark.parametrize("T,C", [(64, 512), (64, 256), (64, 128), (16, 64), (256, 128)])  # T = 64: the tensor-core kernel
def test_attention_backward_vs_autograd(lib, dev, T, C):
    from climate2weather_b200 import _lib
    g = torch.Generator().manual_seed(T * C)
    n = 2
    qkv = torch.randn(n, T, 3 * C, generator=g).to(torch.bfloat16)
    go = torch.randn(n, T, C, generator=g).to(torch.bfloat16)
    gq = torch.empty(n, T, 3 * C, device=dev, dtype=torch.bfloat16)
    qkv_d, go_d = qkv.to(dev), go.to(dev)  # keep the device copies alive across the launch
    scratch = torch.empty(2 * n * T * T, device=dev)
    _lib.check(lib.c2w_op_attention_bwd(qkv_d.data_ptr(), go_d.data_ptr(), gq.data_ptr(), scratch.data_ptr(), n, T, C,
                                        stream()), "attention_bwd")
    torch.cuda.synchronize()
    leaf = qkv.float().requires_grad_(True)
    q, k, v = leaf.split(C, dim=2)
    sc = 1 / math.sqrt(math.sqrt(C))
    w = torch.softmax(torch.einsum("btc,bsc->bts", q * sc, k * sc), dim=-1)
    o = torch.einsum("bts,bsc->btc", w, v)
    (want,) = torch.autograd.grad(o, leaf, go.float())
    assert relerr(gq.float().cpu(), want) < 2 ** -6
    assert rel_l2(gq.float().cpu(), want) < 2 ** -6


def _autograd_vjp(ref, x, t, gout):
    xg = x.clone().requires_grad_(True)
    out = ref(xg, t)
    (gin,) = torch.autograd.grad(out, xg, gout)
    return out.detach(), gin


def test_unet_vjp_small_vs_oracle_autograd(dev):
    """c2w_unet_vjp (stashing forward + input-gradient pass on tensor cores) vs torch.autograd through the fp32 oracle
    network: bf16 activations and gradients through ~12 convs -> 4e-2 of the gradient's max-abs; also through
    torch.autograd on the ScoreUNet module itself (the route torch.func / jacrev-style callers take)."""
    net, ref = make_small(dev)
    g = torch.Generator().manual_seed(21)
    x = torch.randn(3, 20, 32, 32, generator=g)
    gout = torch.randn(3, 20, 32, 32, generator=g)
    t = torch.tensor(0.4)
    want_out, want = _autograd_vjp(ref, x, t, gout)
    eng = net.engine(20, 1, 32, 32, dev, max_windows=2, vjp=True)  # 3 windows through a 2-window workspace: chunked
    out, gin = eng.unet_vjp(x.to(dev), 0.4, gout.to(dev))
    e_out, e = relerr(out, want_out), relerr(gin, want)
    print(f"\nsmall UNet VJP rel-err vs autograd: {e:.3e} (forward {e_out:.3e})")
    assert e_out < 3e-2 and e < 4e-2
    xg = x.to(dev).requires_grad_(True)
    net.requires_grad_(False)  # frozen, like every sampling snapshot (training_loop.py:257)
    y = net(xg, t)
    (gin2,) = torch.autograd.grad(y, xg, gout.to(dev))
    assert torch.equal(gin2, gin)


def test_unet_vjp_full_arch_vs_oracle_autograd(dev):
    """configs/sda_unet.yml architecture (70 convs, attention at level 4, all fusion paths), one window."""
    import climate2weather_b200 as c2w
    cfg = unet_ref.SDA_UNET
    torch.manual_seed(0)
    net = c2w.ScoreUNet(52, 512, hidden_channels=[128, 128, 256, 384, 512], hidden_blocks=[3] * 5, attention_levels=[4], activation=torch.nn.SiLU)
    ref = unet_ref.RefNet({k: v.detach().clone() for k, v in net.state_dict().items()}, cfg)
    g = torch.Generator().manual_seed(5)
    x = torch.randn(1, 52, 128, 128, generator=g)
    gout = torch.randn(1, 52, 128, 128, generator=g)
    t = torch.tensor(0.6)
    want_out, want = _autograd_vjp(ref, x, t, gout)
    eng = net.to(dev).engine(52, 1, 128, 128, dev, max_windows=1, vjp=True)
    out, gin = eng.unet_vjp(x.to(dev), 0.6, gout.to(dev))
    e_out, e = relerr(out, want_out), relerr(gin, want)
    print(f"\nfull UNet VJP rel-err vs autograd: {e:.3e} (forward {e_out:.3e})")
    assert e_out < 3e-2 and e < 5e-2


def _assert_backward_range_equals_list(net, x, k, t, dev):
    """c2w_window_score_backward over the contiguous windows [1, nw - 1) and c2w_window_score_backward_sel over the same
    windows as a list accumulate the same vjp to the bit, and leave the frames no window touches (the first and the
    last) as they were."""
    L, C, H, W = x.shape
    nw = L - 2 * k
    wins = list(range(1, nw - 1))
    eng = net.engine(C, 2 * k + 1, H, W, dev, max_windows=len(wins), vjp=True)
    g = torch.Generator().manual_seed(77 + C)
    xd = x.permute(0, 2, 3, 1).contiguous().to(dev)
    cot = torch.randn(L, H, W, C, generator=g).to(dev)
    base = torch.randn(L, H, W, C, generator=g).to(dev)
    v_range, v_list = base.clone(), base.clone()
    eng.window_score(xd, 0, wins[0], len(wins), nw, float(t), torch.empty_like(xd))
    eng.window_score_backward(cot, 0, wins[0], len(wins), nw, v_range)
    win_list = torch.tensor(wins, dtype=torch.int32, device=dev)
    pos = torch.full((nw,), -1, dtype=torch.int32)
    pos[wins] = torch.arange(len(wins), dtype=torch.int32)
    pos = pos.to(dev)
    eng.window_score_sel(xd, 0, win_list, float(t), nw)
    eng.window_score_backward_sel(cot, 0, win_list, pos, nw, v_list)
    torch.cuda.synchronize()
    assert torch.equal(v_range, v_list)
    assert torch.equal(v_range[[0, L - 1]], base[[0, L - 1]])
    assert not torch.equal(v_range[1:L - 1], base[1:L - 1])


def test_exact_grad_guided_score_vs_oracle(dev):
    """condition_on(exact_grad=True): eps - sigma * d log p / dx with the gradient THROUGH the UNet
    (src/thor/score.py:28-35,48-60), against the oracle's autograd formulation; the chunked backward (2 or 3 windows
    per chunk) accumulates a frame's contributions in a different fp32 order -> 1e-5 between chunked runs;
    exact must differ from the closed-form approximation."""
    import climate2weather_b200 as c2w
    net, ref = make_small(dev)
    g = torch.Generator().manual_seed(31)
    L, k = 11, 2
    x = torch.randn(L, 4, 32, 32, generator=g)
    y = score_ref.coarse_grain(torch.randn(L, 4, 32, 32, generator=g), 3, 8)
    std = torch.tensor(STD).reshape(1, 4, 1, 1)
    t = torch.tensor(0.35)
    want = score_ref.guided_score(ref, x, t, k, y, std, GAMMA, 3, 8, exact_grad=True)
    approx = score_ref.guided_score(ref, x, t, k, y, std, GAMMA, 3, 8, exact_grad=False)
    outs = []
    for mw in (None, 2, 3):
        sf = c2w.DefaultScoreFunction(net, markov_order=k, noise_process=c2w.SDAPipeline())
        sf.max_windows = mw
        sf.condition_on(A=c2w.CoarseGrain(3, 8), y=y, std=std, gamma=GAMMA, exact_grad=True)
        outs.append(sf(x.to(dev), t).cpu())
    e = relerr(outs[0], want)
    d = relerr(approx, want)
    print(f"\nexact-grad guided score rel-err vs oracle: {e:.3e} (closed-form approximation differs by {d:.3e})")
    assert e < 4e-2 and e < 0.5 * d
    # several stashing chunks: every window's score comes from the plain engine and the chunks repeat the selection's
    # forward; one chunk: the selection's score is the stashing engine's own output (bf16 rounding at other points)
    assert relerr(outs[2], outs[1]) < 1e-5
    for o in outs[1:]:
        assert relerr(o, want) < 4e-2 and relerr(o, outs[0]) < 2e-2
    _assert_backward_range_equals_list(net, x, k, t, dev)
    # a short exact-grad sampling run stays finite and differs from the approximate one
    pipe = c2w.SDAPipeline()
    sf = c2w.DefaultScoreFunction(net, markov_order=k, noise_process=pipe)
    sf.condition_on(A=c2w.CoarseGrain(3, 8), y=y, std=std, gamma=GAMMA, exact_grad=True)
    out = pipe.sample(sf, x, steps=3, corrections=1, tau=0.5, show_progressbar=False, seed=5)
    assert torch.isfinite(out).all()


def test_sampler_proc_x0_hook(dev, golden_dir):
    """SDAPipeline.sample(proc_x0=...) (src/thor/pipelines.py:41-46): the hook sees x0 = (x - sigma eps)/mu as an NCHW
    tensor once per step; an identity hook reproduces the fused predictor (fp32 rounding of the split update only), a
    clamping hook changes the sample exactly as re-noising the clamped x0 does."""
    import climate2weather_b200 as c2w
    g = np.load(golden_dir / "small_path.npz")
    net, _ = make_small(dev)
    pipe = c2w.SDAPipeline()
    x = torch.from_numpy(g["x"])
    y = torch.from_numpy(g["yobs"])
    sf = c2w.BatchedScoreFunction(net, markov_order=2, noise_process=pipe, batch_size=4, device=dev)
    sf.condition_on(A=c2w.CoarseGrain(3, 8), y=y, std=torch.tensor(STD).reshape(1, 4, 1, 1), gamma=GAMMA, exact_grad=False)
    base = pipe.sample(sf, x, steps=4, corrections=0, tau=0.5, show_progressbar=False)
    seen = []

    def ident(x0):
        seen.append(x0.detach().clone())
        assert x0.is_cuda
        return x0

    same = pipe.sample(sf, x, steps=4, corrections=0, tau=0.5, show_progressbar=False, proc_x0=ident)
    assert [tuple(s.shape) for s in seen] == [tuple(x.shape)] * 4
    assert relerr(same, base) < 1e-5 and rel_l2(same, base) < 1e-5
    # clamp x0 in the LAST step only: the sample is mu(0) proc(x0) + sigma(0) eps, so it must move by exactly
    # mu(0) (clamp(x0) - x0) with mu(0) = 1 relative to the identity-hook run
    calls = {"n": 0}

    def clamp_last(x0):
        calls["n"] += 1
        return x0.clamp(-0.5, 0.5) if calls["n"] == 4 else x0

    clamped = pipe.sample(sf, x, steps=4, corrections=0, tau=0.5, show_progressbar=False, proc_x0=clamp_last)
    x0_last = seen[3].cpu()
    want = same + float(pipe.mu(torch.tensor(0.0))) * (x0_last.clamp(-0.5, 0.5) - x0_last)
    assert not torch.equal(clamped, same)
    assert rel_l2(clamped, want) < 1e-5


def test_bench_dump_outputs_hold_the_state_after_exactly_steps_steps(tmp_path):
    """bench.py --steps K --dump-outputs DIR on a short trajectory: x.npy and eps.npy are the state after exactly K
    timed steps and the window score of the K-th.  K = 1 is replayed from the seeded noise by the oracle predictor with
    closed-form guidance on the dumped eps (fp32 elementwise, 1e-5); K = 2 replays its second step from K = 1's x,
    whose window score came from another process (bf16 tolerance, 1e-3: a missing or extra step moves x by ~10 % of
    its scale)."""
    import json
    import subprocess
    import sys

    import bench

    L = 20
    _, noise, y, _ = bench.make_problem(L, with_net=False)
    std = torch.tensor(bench.STD).reshape(1, 4, 1, 1)
    times = torch.linspace(1, 0, bench.SAMPLER_STEPS + 1)
    pipe = pipeline_ref.RefPipeline()
    x = noise
    for k in (1, 2):
        out = tmp_path / f"steps{k}"
        r = subprocess.run([sys.executable, str(bench.ROOT / "bench.py"), "--frames", str(L), "--steps", str(k),
                            "--warmup", "0", "--no-cpu", "--no-e2e", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=900, cwd=str(bench.ROOT))
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == k
        got, eps = (torch.from_numpy(np.load(out / f"{n}.npy")) for n in ("x", "eps"))
        assert got.shape == eps.shape == (L, 4, 128, 128)

        def guided(xx, tt, eps=eps):
            return score_ref.guided_score_closed_form(eps, xx, tt, y, std, bench.GAMMA, bench.T_STEP, bench.S_STEP)

        want = pipe.predictor(guided, x, times[k - 1], 1 / bench.SAMPLER_STEPS)
        assert relerr(got, want) < (1e-5 if k == 1 else 1e-3), (k, relerr(got, want))
        x = got
