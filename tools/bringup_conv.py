"""GPU bring-up for K1 (tcgen05 implicit-GEMM conv): numerics vs torch fp32 conv on the same bf16-rounded
operands, then a timing sweep of the dominant shapes.  Run on a B200 via gpurun:
    python tools/bringup_conv.py [--time]
"""
import ctypes
import json
import os
import sys
import time
from pathlib import Path

import torch
import torch.nn.functional as F

ROOT = Path(__file__).resolve().parents[1]
lib = ctypes.CDLL(os.environ.get("C2W_LIB") or str(ROOT / "climate2weather_b200" / "libc2w_b200.so"))
lib.c2w_op_conv.restype = ctypes.c_int
lib.c2w_op_conv.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                            ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                            ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                            ctypes.c_void_p]
try:
    lib.c2w_last_error.restype = ctypes.c_char_p
except AttributeError:
    pass

dev = torch.device("cuda:0")


def pack_w(w, cin_pad, cout_pad):
    cout, cin, kh, kw = w.shape
    wp = torch.zeros(cout_pad, kh, kw, cin_pad, device=w.device, dtype=torch.float32)
    wp[:cout, :, :, :cin] = w.permute(0, 2, 3, 1)
    return wp.reshape(cout_pad, kh * kw * cin_pad).to(torch.bfloat16).contiguous()


def run_conv(x_nhwc, wp, bias, mode, res=None, conv3x3=True, f32=False, bn=0, max_ctas=0):
    n, H, W, cin = x_nhwc.shape
    cout_pad = wp.shape[0]
    M = n * H * W
    out = torch.empty(M, cout_pad, device=dev, dtype=torch.bfloat16) if not f32 else None
    out32 = torch.empty(M, cout_pad, device=dev, dtype=torch.float32) if f32 else None
    if mode == 2 and res is not None:
        out.copy_(res)  # in-place residual
    rc = lib.c2w_op_conv(x_nhwc.data_ptr(), n, H, W, cin, wp.data_ptr(), cout_pad, bias.data_ptr(), mode,
                         out.data_ptr() if (mode == 2) else None, out.data_ptr() if out is not None else None,
                         out32.data_ptr() if f32 else None, 1 if conv3x3 else 0, bn, max_ctas,
                         torch.cuda.current_stream().cuda_stream)
    if rc != 0:
        raise RuntimeError(f"c2w_op_conv rc={rc}")
    torch.cuda.synchronize()
    return out32 if f32 else out


def check(name, n, H, W, cin, cout, mode, seed=0, **kw):
    g = torch.Generator(device="cpu").manual_seed(seed)
    cin_pad = (cin + 63) // 64 * 64
    cout_pad = (cout + 63) // 64 * 64
    x = torch.randn(n, cin, H, W, generator=g).to(dev)
    w = (torch.randn(cout, cin, 3, 3, generator=g) / (3 * cin ** 0.5)).to(dev)
    b = torch.randn(cout, generator=g).to(dev)
    xb = torch.zeros(n, H, W, cin_pad, device=dev, dtype=torch.bfloat16)
    xb[..., :cin] = x.permute(0, 2, 3, 1).to(torch.bfloat16)
    wp = pack_w(w, cin_pad, cout_pad)
    bp = torch.zeros(cout_pad, device=dev)
    bp[:cout] = b
    res = None
    if mode == 2:
        res = torch.randn(n * H * W, cout_pad, generator=g).to(dev).to(torch.bfloat16)
    got = run_conv(xb, wp, bp, 4 if mode == 4 else mode, res=res, f32=(mode == 4), **kw).float()
    # reference on the same rounded operands, fp32 math
    xr = xb[..., :cin].float().permute(0, 3, 1, 2)
    wr = w.to(torch.bfloat16).float()
    ref = F.conv2d(xr, wr, b, padding=1)
    if mode == 1:
        ref = F.silu(ref)
    ref = ref.permute(0, 2, 3, 1).reshape(n * H * W, cout)
    if mode == 2:
        ref = ref + res[:, :cout].float()
    err = (got[:, :cout] - ref).abs().max().item()
    scale = ref.abs().max().item()
    tol = 2e-2 * scale if mode != 4 else 2e-3 * scale
    ok = err <= tol and torch.isfinite(got).all().item()
    print(f"{'PASS' if ok else 'FAIL'} {name}: n={n} {H}x{W} {cin}->{cout} mode={mode} max_err={err:.3e} "
          f"ref_max={scale:.3e}", flush=True)
    return ok


def check_gemm(name, M, K, N, seed=1):
    g = torch.Generator(device="cpu").manual_seed(seed)
    a = torch.randn(M, K, generator=g).to(dev).to(torch.bfloat16)
    w = (torch.randn(N, K, generator=g) / K ** 0.5).to(dev).to(torch.bfloat16)
    b = torch.randn(N, generator=g).to(dev)
    got = run_conv(a.reshape(1, 1, M, K), w, b, 0, conv3x3=False, f32=False).float()
    ref = a.float() @ w.float().t() + b
    err = (got - ref).abs().max().item()
    ok = err <= 2e-2 * ref.abs().max().item()
    print(f"{'PASS' if ok else 'FAIL'} {name}: gemm M={M} K={K} N={N} max_err={err:.3e}", flush=True)
    return ok


def timeit(name, n, H, W, cin, cout, iters=20, variant=-1, bn=0, skip_loads=0, ln=False, res=False, cudnn=True, warm=3,
           **kw):
    sys.path.insert(0, str(ROOT))
    from climate2weather_b200 import _lib
    cin_pad = (cin + 63) // 64 * 64
    cout_pad = (cout + 63) // 64 * 64
    xb = torch.randn(n, H, W, cin_pad, device=dev).to(torch.bfloat16)
    wp = (torch.randn(cout_pad, 9 * cin_pad, device=dev) / 30).to(torch.bfloat16)
    bp = torch.zeros(cout_pad, device=dev)
    out = torch.empty(n * H * W, cout_pad, device=dev, dtype=torch.bfloat16)
    ln_out = torch.empty(n * H * W, cout_pad, device=dev, dtype=torch.bfloat16) if ln else None
    mod = torch.randn(cout_pad, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    L = _lib.load()
    d = _lib.ConvDesc()
    d.x, d.n_img, d.H, d.W, d.cin, d.stride, d.conv3x3 = xb.data_ptr(), n, H, W, cin_pad, 1, 1
    d.w_packed, d.cout_pad, d.bias, d.mode = wp.data_ptr(), cout_pad, bp.data_ptr(), (2 if (ln or res) else 1)
    d.res = out.data_ptr() if (ln or res) else None
    d.out = out.data_ptr()
    d.bn, d.variant, d.max_ctas, d.skip_loads = bn, variant, 0, skip_loads
    d.ln_out = ln_out.data_ptr() if ln else None
    d.ln_mod = mod.data_ptr() if ln else None
    stats = torch.zeros(148 * 12, dtype=torch.int64, device=dev) if "--stats" in sys.argv else None
    d.stats = stats.data_ptr() if stats is not None else None

    def call():
        rc = L.c2w_op_conv_ex(ctypes.byref(d), st)
        assert rc == 0, L.c2w_last_error()

    for _ in range(warm):
        call()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        call()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    if stats is not None:
        st = stats.reshape(148, 12).double().cpu()
        lead = st[0::2]  # leader CTAs hold the MMA counters
        f = lambda v: f"{v.mean().item() / 1e3:.0f}k"
        print(f"  [{name}] cycles/launch: producer total {f(st[:, 0])} wait-empty {f(st[:, 1])} | mma total {f(lead[:, 2])} "
              f"wait-full {f(lead[:, 3])} wait-tmem {f(lead[:, 4])} | epilogue total {f(st[:, 5])} wait-acc {f(st[:, 6])} "
              f"wait-staging {f(st[:, 7])} pass1(incl) {f(st[:, 8])} wait-tile {f(st[:, 9])} LN(incl) {f(st[:, 10])}",
              flush=True)
    flops = 2.0 * n * H * W * cout_pad * 9 * cin_pad
    tf = flops / ms / 1e9
    if not cudnn:
        print(json.dumps({"shape": name, "n": n, "H": H, "W": W, "cin": cin, "cout": cout, "ms": round(ms, 4),
                          "tflops": round(tf, 1)}), flush=True)
        return
    # cuDNN bf16 channels_last for comparison (library bar)
    xc = xb.permute(0, 3, 1, 2)  # NCHW view of NHWC memory == channels_last
    wc = wp.reshape(cout_pad, 3, 3, cin_pad).permute(0, 3, 1, 2).contiguous(memory_format=torch.channels_last)
    for _ in range(3):
        F.conv2d(xc, wc, None, padding=1)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        F.conv2d(xc, wc, None, padding=1)
    e1.record()
    torch.cuda.synchronize()
    ms_dnn = e0.elapsed_time(e1) / iters
    print(json.dumps({"shape": name, "n": n, "H": H, "W": W, "cin": cin, "cout": cout, "ms": round(ms, 4),
                      "tflops": round(tf, 1), "cudnn_ms": round(ms_dnn, 4),
                      "cudnn_tflops": round(flops / ms_dnn / 1e9, 1)}), flush=True)


def main():
    print(torch.cuda.get_device_name(0), flush=True)
    if "--only-g2" in sys.argv:  # short run for `ncu --set full -k regex:conv_gemm`
        timeit("G2", 32, 128, 128, 128, 128, iters=5, cudnn=False)
        return 0
    if "--ncu-variants" in sys.argv:  # `ncu --set full -k regex:conv_gemm -c 8`: 2 launches each of the four main variants
        timeit("G2 plain AR <128,2,0,1>", 32, 128, 128, 128, 128, iters=1, warm=1, variant=5, cudnn=False)
        timeit("G2 residual AR <128,2,0,1>", 32, 128, 128, 128, 128, iters=1, warm=1, variant=5, res=True, cudnn=False)
        timeit("G2 residual+LN AR <128,2,1,1>", 32, 128, 128, 128, 128, iters=1, warm=1, variant=5, ln=True, cudnn=False)
        timeit("G8 residual+LN <256,2,1,0>", 64, 32, 32, 256, 256, iters=1, warm=1, variant=1, bn=256, ln=True, cudnn=False)
        return 0
    if "--res" in sys.argv:  # residual convs only 
        for _ in range(2):
            timeit("G2 cg2+AR res", 32, 128, 128, 128, 128, variant=5, res=True, cudnn=False)
            timeit("G2 cg2+AR res+LN", 32, 128, 128, 128, 128, variant=5, ln=True, cudnn=False)
            timeit("G5 cg2+AR res+LN", 64, 64, 64, 128, 128, variant=5, ln=True, cudnn=False)
        return 0
    if "--noaux" in sys.argv:  # residual convs with the residual prefetch disabled (does it delay the operand loads?)
        for sk in (0, 5, 0, 5):
            timeit(f"G2 cg2+AR res skip={sk}", 32, 128, 128, 128, 128, variant=5, skip_loads=sk, res=True, cudnn=False)
            timeit(f"G2 cg2+AR res+LN skip={sk}", 32, 128, 128, 128, 128, variant=5, skip_loads=sk, ln=True, cudnn=False)
        return 0
    if "--lnfloor" in sys.argv:  # role counters of the LayerNorm conv with and without operand loads (use --stats)
        for sk in (0, 1):
            timeit(f"G2 cg2+AR res skip={sk}", 32, 128, 128, 128, 128, variant=5, skip_loads=sk, res=True, cudnn=False)
            timeit(f"G2 cg2+AR res+LN skip={sk}", 32, 128, 128, 128, 128, variant=5, skip_loads=sk, ln=True, cudnn=False)
        return 0
    if "--which" in sys.argv:  # residual convs (3-deep ring): drop the weight loads (3) or the activation loads (4)
        for sk in (0, 3, 4, 1):
            timeit(f"G2 cg2+AR res skip={sk}", 32, 128, 128, 128, 128, variant=5, skip_loads=sk, res=True, cudnn=False)
            timeit(f"G2 cg2+AR res+LN skip={sk}", 32, 128, 128, 128, 128, variant=5, skip_loads=sk, ln=True, cudnn=False)
            timeit(f"G2 cg2+AR skip={sk}", 32, 128, 128, 128, 128, variant=5, skip_loads=sk, cudnn=False)
        return 0
    if "--halfb" in sys.argv:  # what would a 256-row M tile sharing one weight load buy?  (timing only)
        for sk in (0, 2, 0, 2):
            timeit(f"G2 cg2+AR skip={sk}", 32, 128, 128, 128, 128, variant=5, skip_loads=sk, cudnn=False)
            timeit(f"G2 cg2+AR res skip={sk}", 32, 128, 128, 128, 128, variant=5, skip_loads=sk, res=True, cudnn=False)
            timeit(f"G2 cg2+AR res+LN skip={sk}", 32, 128, 128, 128, 128, variant=5, skip_loads=sk, ln=True, cudnn=False)
        return 0
    if "--ar" in sys.argv:  # the activation-reuse instances at the step's layer shapes, timing only
        for _ in range(2):
            timeit("G2 128x128x128 AR", 32, 128, 128, 128, 128, variant=5, cudnn=False)
            timeit("G2 128x128x128 AR res", 32, 128, 128, 128, 128, variant=5, res=True, cudnn=False)
            timeit("G2 128x128x128 AR res+LN", 32, 128, 128, 128, 128, variant=5, ln=True, cudnn=False)
            timeit("G5 64x64x128 AR res+LN", 64, 64, 64, 128, 128, variant=5, ln=True, cudnn=False)
            timeit("G6 64x64 256->128 AR", 64, 64, 64, 256, 128, variant=5, cudnn=False)
            timeit("L2 32x32x256 bn128 AR", 156, 32, 32, 256, 256, variant=5, bn=128, cudnn=False)
            timeit("L3 16x16x384 bn128 AR", 156, 16, 16, 384, 384, variant=5, bn=128, cudnn=False)
            timeit("L4 8x8x512 bn128 AR (two-image)", 156, 8, 8, 512, 512, variant=5, bn=128, cudnn=False)
            timeit("G2 128x128x128 AR bn64", 32, 128, 128, 128, 64, variant=5, bn=64, cudnn=False)
        return 0
    if "--tiles" in sys.argv:  # N-tile choice per level at the real window count (conv_pick_bn_tiled's cost model)
        n = 156
        for res in (False, True):
            r = " res" if res else ""
            for name, H, C, cases in (("L2 32x32x256", 32, 256, ((256, 1), (128, 5), (128, 1))),
                                      ("L3 16x16x384", 16, 384, ((192, 1), (128, 5), (128, 1))),
                                      ("L4 8x8x512", 8, 512, ((256, 1), (128, 5), (128, 1), (256, 0)))):
                for bn, var in cases:
                    timeit(f"{name} bn{bn} v{var}{r}", n, H, H, C, C, variant=var, bn=bn, res=res, cudnn=False)
        timeit("L3 16x16 512->384 bn192 v1", n, 16, 16, 512, 384, variant=1, bn=192, cudnn=False)
        timeit("L3 16x16 512->384 bn128 v5", n, 16, 16, 512, 384, variant=5, bn=128, cudnn=False)
        timeit("L2 32x32 384->256 bn256 v1", n, 32, 32, 384, 256, variant=1, bn=256, cudnn=False)
        timeit("L2 32x32 384->256 bn128 v5", n, 32, 32, 384, 256, variant=5, bn=128, cudnn=False)
        return 0
    ok = True
    ok &= check_gemm("gemm-basic", 256, 128, 128)
    ok &= check_gemm("gemm-k512-n256", 384, 512, 256)
    ok &= check_gemm("gemm-m64", 64, 512, 1536)
    ok &= check("conv-w128-c64", 1, 128, 128, 64, 128, 0)
    ok &= check("conv-G2", 2, 128, 128, 128, 128, 1)
    ok &= check("conv-G2-res", 2, 128, 128, 128, 128, 2)
    ok &= check("conv-G1(52)", 2, 128, 128, 52, 128, 0)
    ok &= check("conv-G3(->52) f32", 2, 128, 128, 128, 52, 4)
    ok &= check("conv-w64", 3, 64, 64, 128, 128, 1)
    ok &= check("conv-w32-256", 3, 32, 32, 256, 256, 2)
    ok &= check("conv-w16-384", 3, 16, 16, 384, 384, 1)
    ok &= check("conv-w8-512", 3, 8, 8, 512, 512, 2)
    ok &= check("conv-w16-512->384", 2, 16, 16, 512, 384, 0)
    ok &= check("conv-G2-bn64", 2, 128, 128, 128, 128, 1, bn=64)
    ok &= check("conv-G2-few-ctas", 4, 128, 128, 128, 128, 1, max_ctas=7)
    print("ALL PASS" if ok else "SOME FAILED", flush=True)
    if "--time" in sys.argv:
        timeit("G2 cg1", 32, 128, 128, 128, 128, variant=0)
        timeit("G2 cg2", 32, 128, 128, 128, 128, variant=1, cudnn=False)
        timeit("G2 cg2+AR", 32, 128, 128, 128, 128, variant=5, cudnn=False)
        timeit("G2 cg2+AR res", 32, 128, 128, 128, 128, variant=5, res=True, cudnn=False)
        timeit("G2 cg2+AR res+LN", 32, 128, 128, 128, 128, variant=5, ln=True, cudnn=False)
        timeit("G5 cg2+AR", 64, 64, 64, 128, 128, variant=5, cudnn=False)
        timeit("G6 cg2+AR (256->128)", 64, 64, 64, 256, 128, variant=5, cudnn=False)
        timeit("G2 cg2 res", 32, 128, 128, 128, 128, variant=1, res=True, cudnn=False)
        timeit("G2 cg2+LN", 32, 128, 128, 128, 128, variant=1, ln=True, cudnn=False)
        timeit("G5 cg2", 64, 64, 64, 128, 128, variant=1, cudnn=False)
        if os.environ.get("C2W_LIB"):  # diagnostics build only (-DC2W_DIAG): no TMA traffic after priming
            timeit("G2 cg1 noloads", 32, 128, 128, 128, 128, variant=0, skip_loads=1, cudnn=False)
            timeit("G2 cg2 noloads", 32, 128, 128, 128, 128, variant=1, skip_loads=1, cudnn=False)
        timeit("G5 cg2 (cudnn)", 64, 64, 64, 128, 128, variant=1)
        timeit("G8 cg1", 64, 32, 32, 256, 256, variant=0)
        timeit("G8 cg2", 64, 32, 32, 256, 256, variant=1, cudnn=False)
        timeit("G11 cg1", 128, 16, 16, 384, 384, variant=0)
        timeit("G11 cg2", 128, 16, 16, 384, 384, variant=1, cudnn=False)
        timeit("G14 cg1", 156, 8, 8, 512, 512, variant=0)
        timeit("G14 cg2", 156, 8, 8, 512, 512, variant=1, cudnn=False)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
