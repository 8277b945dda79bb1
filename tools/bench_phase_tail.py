"""Times the ascent-tail conv of config 2 (156 windows) both ways, each launch in isolation with CUDA events:
the 3x3 conv of the nearest x2 upsampled LayerNorm output (c2w_op_conv_ex) and its phase form at the low resolution
(c2w_op_conv_phase), both with the residual epilogue and with and without the fused LayerNorm of the output.
Prints the time per launch and the achieved TFLOP/s counted with the 3x3 conv's FLOPs and with the phase form's.

    python tools/bench_phase_tail.py [--windows 156] [--iters 50]
"""
import argparse
import ctypes
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from climate2weather_b200 import _lib  # noqa: E402

# (name, low-res H = W, cin, cout): the config-2 tails that take the phase form (level 3: two 128-wide N tiles, so its
# LayerNorm is a launch of its own; the upsampled form fuses it into one 256-wide tile)
TAILS = [("level-1 tail 128->128 @128^2", 64, 128, 128), ("level-2 tail 256->128 @64^2", 32, 256, 128),
         ("level-3 tail 384->256 @32^2", 16, 384, 256)]


def _desc(x, n, H, cin, w, cout, bias, out, ln_out, bn=0):
    d = _lib.ConvDesc()
    d.x, d.n_img, d.H, d.W, d.cin, d.stride, d.conv3x3 = x.data_ptr(), n, H, H, cin, 1, 1
    d.w_packed, d.cout_pad, d.bias, d.mode = w.data_ptr(), cout, bias.data_ptr(), 2
    d.res, d.out, d.out_f32 = out.data_ptr(), out.data_ptr(), None
    d.bn, d.variant, d.max_ctas, d.skip_loads = bn or cout, -1, 0, 0
    d.ln_out = ln_out.data_ptr() if ln_out is not None else None
    d.ln_mod, d.ln_upsample = None, 0
    return d


def _time(fn, iters):
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3  # us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=156)
    ap.add_argument("--iters", type=int, default=50)
    a = ap.parse_args()
    lib = _lib.load()
    dev = torch.device("cuda:0")
    st = torch.cuda.current_stream().cuda_stream
    p = torch.cuda.get_device_properties(dev)
    print(f"# {p.name}, {a.windows} windows, mean of {a.iters} back-to-back launches after 3 warm-up launches")
    n = a.windows
    for name, H, cin, cout in TAILS:
        z = torch.randn(n, H, H, cin, device=dev).to(torch.bfloat16)
        up = z.repeat_interleave(2, dim=1).repeat_interleave(2, dim=2).contiguous()
        w = torch.randn(cout, cin, 3, 3) / (3 * cin ** 0.5)
        w9 = w.permute(0, 2, 3, 1).reshape(cout, 9 * cin).to(dev, torch.bfloat16).contiguous()
        wph = torch.empty(4, cout, 4 * cin, dtype=torch.bfloat16)
        _lib.check(lib.c2w_pack_phase_weights(w.contiguous().data_ptr(), cout, cin, cin, cout, wph.data_ptr()), "pack")
        wph = wph.to(dev)
        bias = torch.zeros(cout, device=dev)
        out = torch.zeros(n, 2 * H, 2 * H, cout, device=dev, dtype=torch.bfloat16)
        ln_out = torch.empty_like(out)
        flop9 = 2.0 * n * (2 * H) ** 2 * cout * 9 * cin
        flop4 = 2.0 * n * H * H * 4 * cout * 4 * cin
        for ln in (False, True):
            d_old = _desc(up, n, 2 * H, cin, w9, cout, bias, out, ln_out if ln else None)
            d_new = _desc(z, n, H, cin, wph, cout, bias, out, ln_out if ln else None, bn=min(cout, 128))
            t_old = _time(lambda: _lib.check(lib.c2w_op_conv_ex(ctypes.byref(d_old), st), "conv"), a.iters)
            tag = name + (" +res +LN" if ln else " +res")
            if ln and cout > 128:  # two N tiles: no fused LayerNorm in the phase form (see the separate launch below)
                print(f"{tag:40s} upsampled 3x3: {t_old:7.1f} us {flop9 / t_old / 1e6:6.0f} TFLOP/s")
                continue
            t_new = _time(lambda: _lib.check(lib.c2w_op_conv_phase(ctypes.byref(d_new), st), "phase"), a.iters)
            print(f"{tag:40s} upsampled 3x3: {t_old:7.1f} us {flop9 / t_old / 1e6:6.0f} TFLOP/s | "
                  f"phase: {t_new:7.1f} us {flop9 / t_new / 1e6:6.0f} TFLOP/s (3x3 FLOPs) "
                  f"{flop4 / t_new / 1e6:6.0f} TFLOP/s (2x2 FLOPs) | {t_new / t_old - 1:+.1%}")
        # the LayerNorm as a launch of its own after the phase conv without it
        d_new = _desc(z, n, H, cin, wph, cout, bias, out, None, bn=min(cout, 128))
        npix = n * 4 * H * H

        def phase_then_ln():
            _lib.check(lib.c2w_op_conv_phase(ctypes.byref(d_new), st), "phase")
            _lib.check(lib.c2w_op_layernorm(out.data_ptr(), None, ln_out.data_ptr(), npix, cout, 2 * H, 2 * H, 0, st),
                       "layernorm")
        t_sep = _time(phase_then_ln, a.iters)
        print(f"{name + ' +res, then LayerNorm launch':40s} phase + separate LayerNorm: {t_sep:7.1f} us")


if __name__ == "__main__":
    main()
