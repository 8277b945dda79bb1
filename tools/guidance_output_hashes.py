"""sha256 of every output of the existing guidance entry points (c2w_guided_step, _points, _combined, _obs_std and
_members), seeded, one line per call: C = 1..8 on L = 11 frames of 32 x 32 (s = 8) and 128 x 128 (s = 16), t_step = 3,
modes 0 / 1 / 2, with and without a VJP term (x, eps_out, cot_out, partials, NaN flag).  Only entry points every
library of ABI 3 since the ensemble change exports are called, so one build's output can be diffed against another's:
    python tools/guidance_output_hashes.py > new.txt; python tools/guidance_output_hashes.py --lib OTHER.so > old.txt
"""
import argparse
import ctypes as C
import hashlib
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from climate2weather_b200 import _lib  # noqa: E402
from climate2weather_b200.score import PointObservation, combined_strip_rows, point_plan, point_strip_rows  # noqa: E402

_vp, _i = C.c_void_p, C.c_int
ENTRIES = {
    "c2w_guided_step": [C.POINTER(_lib.Guide), _vp],
    "c2w_guided_step_points": [C.POINTER(_lib.Guide), C.POINTER(_lib.PointObs), _vp],
    "c2w_guided_step_combined": [C.POINTER(_lib.Guide), C.POINTER(_lib.PointObs), C.POINTER(C.c_float), _vp],
    "c2w_guided_step_obs_std": [C.POINTER(_lib.Guide), C.POINTER(_lib.PointObs), _vp, _vp, _vp],
    "c2w_guided_step_members": [C.POINTER(_lib.Guide), C.c_int32, C.POINTER(_lib.PointObs), C.POINTER(C.c_float), _vp,
                                _vp, _vp],
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=str(_lib.LIB_PATH))
    args = ap.parse_args()
    lib = C.CDLL(args.lib)
    for name, argt in ENTRIES.items():
        getattr(lib, name).restype, getattr(lib, name).argtypes = _i, argt
    lib.c2w_last_error.restype = C.c_char_p
    dev = torch.device("cuda:0")
    st = torch.cuda.current_stream().cuda_stream
    L, t = 11, 3
    for Hh, s in ((32, 8), (128, 16)):
        Ww = Hh
        for Cv in range(1, 9):
            g = torch.Generator().manual_seed(100 * Cv + Hh)
            x0 = torch.randn(L, Hh, Ww, Cv, generator=g).to(dev)
            eps = torch.randn(L, Hh, Ww, Cv, generator=g).to(dev)
            vjp = torch.randn(L, Hh, Ww, Cv, generator=g).to(dev)
            y = torch.randn(-(-L // t), Cv, Hh // s, Ww // s, generator=g).to(dev)
            ystd2 = (0.05 + torch.rand(y.shape, generator=g)).to(dev)
            P = 50
            mask = torch.rand(4, Cv, P, generator=g) > 0.25
            op = PointObservation([9, 0, 3, 10], torch.randint(0, Hh, (P,), generator=g),
                                  torch.randint(0, Ww, (P,), generator=g), mask)
            py = torch.randn(4, Cv, P, generator=g)
            pstd = torch.where(torch.rand(4, Cv, P, generator=g) > 0.5, 0.1, 0.3)
            keep = []

            def plan(strip, max_pix, std=None, lo=1, hi=10, members=0, Lp=L):
                pl = point_plan(op, py, Lp, Cv, Hh, Ww, lo, hi, strip, max_pix, std, members=members)
                names = ("frame_slot", "strip_off", "pix", "ysum", "wsum") + (("std2",) if std is not None else ())
                d = {n: torch.as_tensor(pl[n]).to(dev) for n in names}
                for n in names[2:]:
                    if d[n].numel() == 0:
                        d[n] = torch.zeros(Cv, dtype=d[n].dtype, device=dev)
                keep.append(d)
                ob = _lib.PointObs()
                ob.frame_slot, ob.strip_off, ob.pix = (d[n].data_ptr() for n in ("frame_slot", "strip_off", "pix"))
                ob.ysum, ob.wsum, ob.n_slots, ob.strip_rows = d["ysum"].data_ptr(), d["wsum"].data_ptr(), \
                    pl["n_slots"], pl["strip_rows"]
                return ob, d, pl["n_strips"]

            pr, cr = point_strip_rows(Hh, Ww), combined_strip_rows(Hh, Ww, s)
            p_pts, _, ns_p = plan(pr, 2048)
            p_cmb, _, ns_c = plan(cr, 16384)
            p_pts_o, d_pts_o, _ = plan(pr, 2048, pstd)
            p_cmb_o, d_cmb_o, _ = plan(cr, 16384, pstd)
            # members: 2 members of L frames, every frame updated
            p_mem, _, _ = plan(cr, 16384, lo=0, hi=L, members=2)
            pstd2 = (C.c_float * Cv)(*[0.02 + 0.01 * c for c in range(Cv)])
            calls = {
                "coarse": (lambda gp: lib.c2w_guided_step(gp, st), True, Hh // s, 1),
                "points": (lambda gp: lib.c2w_guided_step_points(gp, C.byref(p_pts), st), False, ns_p, 1),
                "combined": (lambda gp: lib.c2w_guided_step_combined(gp, C.byref(p_cmb), pstd2, st), True, ns_c, 1),
                "obs_coarse": (lambda gp: lib.c2w_guided_step_obs_std(gp, None, ystd2.data_ptr(), None, st), True,
                               Hh // s, 1),
                "obs_points": (lambda gp: lib.c2w_guided_step_obs_std(gp, C.byref(p_pts_o), None,
                                                                      d_pts_o["std2"].data_ptr(), st), False, ns_p, 1),
                "obs_combined": (lambda gp: lib.c2w_guided_step_obs_std(gp, C.byref(p_cmb_o), ystd2.data_ptr(),
                                                                        d_cmb_o["std2"].data_ptr(), st), True, ns_c, 1),
                "members_combined": (lambda gp: lib.c2w_guided_step_members(gp, L, C.byref(p_mem), pstd2, None, None,
                                                                            None, st), True, ns_c, 2),
            }
            for name, (call, coarse, n_strips, members) in calls.items():
                for mode in (0, 1, 2):
                    for with_vjp in ((False, True) if mode != 2 else (False,)):
                        F = members * L
                        x = x0.repeat(members, 1, 1, 1)
                        e = eps.repeat(members, 1, 1, 1)
                        out = torch.zeros_like(x)
                        cot = torch.zeros_like(x)
                        own_lo, own_n = (0, F) if members > 1 else (1, 9)
                        parts = torch.zeros(own_n * n_strips, device=dev)
                        flag = torch.zeros(1, dtype=torch.int32, device=dev)
                        v = vjp.repeat(members, 1, 1, 1)
                        gp = _lib.Guide()
                        gp.x, gp.eps, gp.eps_out = x.data_ptr(), e.data_ptr(), out.data_ptr()
                        gp.y = y.data_ptr() if coarse else None
                        for c in range(Cv):
                            gp.std2[c], gp.gamma[c] = 0.01 * (c + 1), 7e-4 * (c + 1)
                        gp.mu, gp.sigma, gp.mu_next, gp.sigma_next = 0.8, 0.5, 0.9, 0.4
                        gp.t_step, gp.s_step, gp.H, gp.W = (t if coarse else 1), s, Hh, Ww
                        gp.frame_global0, gp.own_lo, gp.own_n = 0, own_lo, own_n
                        gp.mode, gp.partials, gp.nan_flag = mode, parts.data_ptr(), flag.data_ptr()
                        gp.vjp = v.data_ptr() if with_vjp else None
                        gp.cot_out = cot.data_ptr() if mode == 2 else None
                        gp.channels = Cv
                        rc = call(C.byref(gp))
                        if rc:
                            raise RuntimeError(f"{name}: {lib.c2w_last_error()}")
                        torch.cuda.synchronize()
                        for what, tns in (("x", x), ("eps_out", out), ("cot", cot), ("partials", parts), ("nan", flag)):
                            h = hashlib.sha256(tns.cpu().numpy().tobytes()).hexdigest()
                            print(f"{Hh}x{Ww} C={Cv} {name} mode={mode} vjp={int(with_vjp)} {what} {h}")


if __name__ == "__main__":
    main()
