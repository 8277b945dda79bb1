"""sha256 of K1's outputs at the parity tests' conv shapes (tests/test_gpu_parity.py), seeded, one line per launch.
Run once per library build (C2W_LIB selects another build of the same ABI) and diff the outputs:
    python tools/k1_output_hashes.py > new.txt; C2W_LIB=... python tools/k1_output_hashes.py > parent.txt
"""
import ctypes
import hashlib
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from climate2weather_b200 import _lib  # noqa: E402

# (n, H, W, cin, cout, mode, variant, bn, ln): test_conv3x3_kernel_variants, ..._wide_and_two_image_tiles,
# ..._times_dsilu_in_place and ..._fused_layernorm
SHAPES = [(n, H, W, ci, co, m, v, 0, False) for v in (-1, 1, 5) for n, H, W, ci, co, m in [
    (2, 128, 128, 128, 128, 1), (3, 64, 64, 128, 128, 2), (5, 32, 32, 128, 128, 0), (1, 128, 128, 64, 128, 1),
    (3, 16, 16, 256, 128, 2), (1, 16, 8, 64, 128, 0), (2, 64, 64, 128, 64, 4), (2, 32, 32, 128, 64, 1)]]
SHAPES += [(n, H, W, ci, co, m, 5, 128, False) for n, H, W, ci, co, m in [
    (6, 8, 8, 512, 512, 1), (5, 8, 8, 128, 256, 2), (4, 8, 16, 64, 128, 0), (3, 8, 8, 192, 384, 2),
    (7, 16, 16, 384, 384, 1), (2, 16, 16, 512, 384, 2), (3, 32, 32, 256, 256, 1)]]
SHAPES += [(2, 128, 128, 128, 128, 5, 5, 0, False), (3, 32, 32, 256, 256, 5, 5, 128, False),
           (5, 8, 8, 512, 512, 5, 5, 128, False)]
SHAPES += [(n, H, W, C, C, m, v, 0, True) for n, H, W, C, m, v in [
    (2, 128, 128, 128, 2, 5), (1, 32, 32, 128, 0, 5), (2, 64, 64, 128, 2, 1), (2, 32, 32, 64, 0, 5)]]


def main():
    lib = _lib.load()
    dev = torch.device("cuda:0")
    for i, (n, H, W, cin, cout, mode, variant, bn, ln) in enumerate(SHAPES):
        g = torch.Generator().manual_seed(1000 + i)
        M = n * H * W
        xb = torch.randn(n, H, W, cin, generator=g).to(dev, torch.bfloat16)
        wp = (torch.randn(cout, 9 * cin, generator=g) / (3 * cin ** 0.5)).to(dev, torch.bfloat16)
        bp = torch.randn(cout, generator=g).to(dev)
        aux = (2.0 * torch.randn(M, cout, generator=g)).to(dev, torch.bfloat16)
        out = aux.clone() if mode in (2, 5) else torch.zeros(M, cout, device=dev, dtype=torch.bfloat16)
        out32 = torch.zeros(M, cout, device=dev) if mode == 4 else None
        ln_out = torch.zeros(M, cout, device=dev, dtype=torch.bfloat16) if ln else None
        d = _lib.ConvDesc()
        d.x, d.n_img, d.H, d.W, d.cin, d.stride, d.conv3x3 = xb.data_ptr(), n, H, W, cin, 1, 1
        d.w_packed, d.cout_pad, d.bias, d.mode = wp.data_ptr(), cout, bp.data_ptr(), mode
        d.res = out.data_ptr() if mode in (2, 5) else None
        d.out = out.data_ptr()
        d.out_f32 = out32.data_ptr() if out32 is not None else None
        d.bn, d.variant, d.max_ctas, d.skip_loads = bn, variant, 0, 0
        d.ln_out = ln_out.data_ptr() if ln else None
        _lib.check(lib.c2w_op_conv_ex(ctypes.byref(d), torch.cuda.current_stream().cuda_stream), "c2w_op_conv_ex")
        torch.cuda.synchronize()
        h = hashlib.sha256((out32 if out32 is not None else out).cpu().view(torch.uint8).numpy().tobytes())
        if ln:
            h.update(ln_out.cpu().view(torch.uint8).numpy().tobytes())
        print(f"n={n} H={H} W={W} cin={cin} cout={cout} mode={mode} variant={variant} bn={bn} ln={int(ln)} "
              f"{h.hexdigest()}", flush=True)


if __name__ == "__main__":
    main()
