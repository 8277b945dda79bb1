"""CPU tests of point observations (PointObservation): the operator against explicit indexing, the host plan the
guidance kernel reads (merged per frame and pixel, CSR by frame slot and strip) against autograd through the operator,
the validation errors, the observed-window selection for exact_grad, and the oracle's operator-generic guidance."""
import ctypes

import numpy as np
import pytest
import torch

from climate2weather_b200 import _lib
from climate2weather_b200.score import (CoarseGrain, PointObservation, observed_windows, point_plan,
                                        point_strip_rows)
from oracle import score_ref

import oracle_op


def _op(L, C, H, W, F, P, seed, masked=True, dup=True):
    g = torch.Generator().manual_seed(seed)
    frames = torch.randperm(L, generator=g)[:F]
    rows = torch.randint(0, H, (P,), generator=g)
    cols = torch.randint(0, W, (P,), generator=g)
    if dup and P >= 4:
        rows[1], cols[1] = rows[0], cols[0]                  # two points on one pixel
        rows[2], cols[2] = 0, 0                              # image corners
        rows[3], cols[3] = H - 1, W - 1
    mask = None
    if masked:
        mask = torch.rand(F, C, P, generator=g) > 0.3
        mask[:, :, min(4, P - 1)] = False                    # a fully masked point
    y = torch.randn(F, C, P, generator=g, dtype=torch.float64).float()
    return PointObservation(frames, rows, cols, mask), y


def _dense_from_plan(pl, x0, var, H, W, frame_lo, n_own):
    """What the kernel computes, in numpy: g[f, pix, c] = (ysum - wsum x0) / var at every entry, zero elsewhere."""
    C = x0.shape[1]
    out = np.zeros((n_own, C, H * W))
    ns, sr = pl["n_strips"], pl["strip_rows"]
    for i in range(n_own):
        s = pl["frame_slot"][i]
        if s < 0:
            continue
        for b in range(ns):
            for e in range(pl["strip_off"][s * ns + b], pl["strip_off"][s * ns + b + 1]):
                px = pl["pix"][e]
                assert b * sr * W <= px < min(H, (b + 1) * sr) * W  # the entry lies in its strip
                xv = x0[frame_lo + i].reshape(C, -1)[:, px].double().numpy()
                out[i, :, px] = (pl["ysum"][e].astype(np.float64) - pl["wsum"][e] * xv) / var
    return out.reshape(n_own, C, H, W)


def _autograd_cot(op, y, x0, var):
    """A^T((y - A x0)/var) by autograd through PointObservation.__call__ (masked y replaced by finite values)."""
    x0 = x0.double().clone().requires_grad_(True)
    yf = torch.where(op.mask_for(y.shape[1]), y, torch.zeros_like(y)).double()
    logp = -(((yf - op(x0)) ** 2) / var.reshape(1, -1, 1)).sum() / 2
    (gr,) = torch.autograd.grad(logp, x0)
    return gr


def test_operator_matches_explicit_indexing():
    L, C, H, W = 9, 3, 8, 12
    op, _ = _op(L, C, H, W, F=4, P=7, seed=1)
    x = torch.randn(L, C, H, W)
    got = op(x)
    assert got.shape == (4, C, 7)
    for m in range(4):
        for c in range(C):
            for p in range(7):
                want = x[op.frames[m], c, op.rows[p], op.cols[p]] * float(op.mask[m, c, p])
                assert got[m, c, p] == want


@pytest.mark.parametrize("L,C,H,W,F,P,seed", [(11, 4, 32, 32, 5, 40, 0), (7, 3, 24, 16, 7, 9, 1), (20, 1, 40, 8, 3, 60, 2),
                                              (6, 6, 33, 128, 2, 300, 3)])
def test_plan_equals_autograd_adjoint(L, C, H, W, F, P, seed):
    op, y = _op(L, C, H, W, F, P, seed)
    y[~op.mask] = float("nan")  # ignored under the mask
    x0 = torch.randn(L, C, H, W, generator=torch.Generator().manual_seed(seed + 9), dtype=torch.float64)
    var = torch.rand(C, dtype=torch.float64) + 0.05
    want = _autograd_cot(op, y, x0, var)
    strip = point_strip_rows(H, W)
    pl = point_plan(op, y, L, C, H, W, 0, L, strip)
    assert pl["n_slots"] == len(pl["frames"]) and pl["frames"] == op.observed_frames(C)
    assert np.all(np.diff(pl["strip_off"]) >= 0) and pl["strip_off"][-1] == pl["pix"].size
    got = _dense_from_plan(pl, x0, var.numpy(), H, W, 0, L)
    np.testing.assert_allclose(got, want.numpy(), rtol=1e-6, atol=1e-6)
    # entries are unique per (frame, pixel) and never fully masked
    assert (pl["wsum"] > 0).any(1).all()
    # a rank split: the per-rank plans keep only their frames and together give the whole
    for cuts in ([0, L // 2, L], [0, 1, L // 3 + 1, L - 1, L]):
        parts, n_entries = [], 0
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            pr = point_plan(op, y, L, C, H, W, lo, hi, strip)
            assert all(lo <= f < hi for f in pr["frames"])
            n_entries += pr["pix"].size
            parts.append(_dense_from_plan(pr, x0, var.numpy(), H, W, lo, hi - lo))
        assert n_entries == pl["pix"].size
        np.testing.assert_array_equal(np.concatenate(parts), got)


def test_plan_strips_of_one_row_and_strip_borders():
    """Points on every strip border row, with strips of 1 and of 3 rows."""
    L, C, H, W = 4, 4, 12, 16
    rows = torch.tensor([0, 2, 3, 5, 6, 11, 11, 3])
    cols = torch.tensor([0, 15, 0, 7, 8, 15, 0, 0])
    op = PointObservation([3, 1], rows, cols)
    y = torch.randn(2, C, 8)
    x0 = torch.randn(L, C, H, W, dtype=torch.float64)
    var = torch.full((C,), 0.3, dtype=torch.float64)
    want = _autograd_cot(op, y, x0, var).numpy()
    for strip in (1, 3, 12):
        pl = point_plan(op, y, L, C, H, W, 0, L, strip)
        assert pl["pix"].size == 2 * 7 and list(pl["frame_slot"]) == [-1, 0, -1, 1]
        np.testing.assert_allclose(_dense_from_plan(pl, x0, var.numpy(), H, W, 0, L), want, rtol=1e-6,
                                   atol=1e-6)


def test_duplicates_sum_exactly():
    op = PointObservation([0], [2, 2, 2], [1, 1, 1], mask=torch.tensor([[[True, False, True]]]))
    y = torch.tensor([[[1.5, float("nan"), 2.25]]])
    pl = point_plan(op, y, 1, 1, 4, 4, 0, 1, 4)
    assert pl["pix"].tolist() == [9] and pl["ysum"].tolist() == [[3.75]] and pl["wsum"].tolist() == [[2.0]]


@pytest.mark.parametrize("kw,call,match", [
    (dict(frames=[0, 2, 2], rows=[0], cols=[0]), None, "repeated frame"),
    (dict(frames=[0, -1], rows=[0], cols=[0]), None, "negative frame"),
    (dict(frames=[0], rows=[0, 1], cols=[0]), None, "rows but"),
    (dict(frames=[0, 1], rows=[0], cols=[0], mask=torch.ones(2, 4, 2, dtype=torch.bool)), None, "mask of shape"),
    (dict(frames=[0, 1], rows=[0], cols=[0], mask=torch.ones(2, 4, 1)), None, "bool"),
    (dict(frames=[0, 9], rows=[0], cols=[0]), "plan", "outside a trajectory"),
    (dict(frames=[0], rows=[8], cols=[0]), "plan", "outside the 8x8 grid"),
    (dict(frames=[0], rows=[0], cols=[-1]), "plan", "outside the 8x8 grid"),
    (dict(frames=[0], rows=[0], cols=[0], mask=torch.ones(1, 3, 1, dtype=torch.bool)), "plan", "mask of shape"),
    (dict(frames=[0, 1], rows=[0], cols=[0]), "y_shape", "y of shape"),
    (dict(frames=[0, 1], rows=[0], cols=[0]), "y_nan", "not finite"),
])
def test_validation_errors(kw, call, match):
    with pytest.raises(ValueError, match=match):
        op = PointObservation(**kw)
        y = torch.zeros(len(kw["frames"]), 4, len(kw["rows"]))
        if call == "plan":
            point_plan(op, y, 9, 4, 8, 8, 0, 9, 8)
        elif call == "y_shape":
            op.check_observation(torch.zeros(2, 4, 3))
        elif call == "y_nan":
            y[1, 2, 0] = float("inf")
            point_plan(op, y, 9, 4, 8, 8, 0, 9, 8)


def test_condition_on_rejects_non_finite_unmasked_y_and_accepts_masked_nan():
    import climate2weather_b200 as c2w
    net = c2w.ScoreUNet(channels=20, embedding_dim=64, hidden_channels=(64,), hidden_blocks=(1,), attention_levels=(),
                        activation=torch.nn.SiLU)
    sf = c2w.DefaultScoreFunction(net, markov_order=2, noise_process=c2w.SDAPipeline())
    mask = torch.ones(2, 4, 3, dtype=torch.bool)
    mask[0, 1, 2] = False
    op = c2w.PointObservation([0, 4], [1, 2, 3], [3, 2, 1], mask)
    y = torch.zeros(2, 4, 3)
    y[0, 1, 2] = float("nan")
    sf.condition_on(A=op, y=y, std=0.1, gamma=1e-2, exact_grad=False)  # masked NaN: fine
    y[1, 1, 2] = float("nan")
    with pytest.raises(ValueError, match="not finite"):
        sf.condition_on(A=op, y=y, std=0.1, gamma=1e-2, exact_grad=False)


def test_compat_exports_point_observation():
    import sys

    import climate2weather_b200 as c2w
    from climate2weather_b200 import compat
    compat.install()
    assert sys.modules["thor.score"].PointObservation is c2w.PointObservation


@pytest.mark.parametrize("L,k", [(13, 6), (25, 6), (40, 2), (31, 3), (168, 6)])
def test_observed_windows_with_a_frame_set(L, k):
    """With a set of observed frames, exactly the windows whose output (the fold of src/thor/score.py:76-88) contains
    an observed frame are selected; shards partition that selection; an int t_step keeps its old meaning."""
    from climate2weather_b200.sharding import make_plan
    nw = L - 2 * k
    f = score_ref.fold_index(L, k, 4)
    rng = np.random.default_rng(L + k)
    sets = [{0}, {L - 1}, set(range(L)), set(rng.choice(L, size=max(1, L // 5), replace=False).tolist()), {k, L - k - 1}]
    for frames in sets:
        # brute force: window j matters iff a frame taken from it is observed
        want = sorted({int(f[fr, 0, 0]) for fr in frames})
        assert observed_windows(0, nw, nw, L, k, frames) == want, frames
        assert observed_windows(0, nw, nw, L, k, sorted(frames)) == want
        for world in (2, 3):
            if nw // world < max(k, 1):
                continue
            got = []
            for r in range(world):
                p = make_plan(L, k, r, world)
                got += observed_windows(p.win_lo, p.win_hi, p.n_win_global, L, k, frames)
            assert got == want
    assert observed_windows(0, nw, nw, L, k, 3) == observed_windows(0, nw, nw, L, k, set(range(0, L, 3)))


def test_guided_score_op_with_coarse_grain_equals_guided_score():
    from oracle import unet_ref  # noqa: F401  (the oracle's window composition only needs a callable net)
    L, C, H, W, k = 9, 4, 16, 16, 2
    g = torch.Generator().manual_seed(4)
    lin = torch.randn(C * (2 * k + 1), C * (2 * k + 1), generator=g) * 0.2
    net = lambda u, t: torch.tanh(torch.einsum("oc,bchw->bohw", lin, u) * (1 + t))
    x = torch.randn(L, C, H, W, generator=g)
    y = score_ref.coarse_grain(torch.randn(L, C, H, W, generator=g), 3, 4)
    std = torch.tensor([0.1, 0.2, 0.3, 0.4]).reshape(1, C, 1, 1)
    t = torch.tensor(0.4)
    for exact in (False, True):
        want = score_ref.guided_score(net, x, t, k, y, std, 1e-3, 3, 4, exact_grad=exact)
        got = oracle_op.guided_score_op(net, x, t, k, y, std, 1e-3, CoarseGrain(3, 4), exact_grad=exact)
        assert ((got - want).abs().max() / want.abs().max()).item() <= 1e-6
    with torch.no_grad():
        eps = score_ref.window_score(net, x, t, k)
    want = score_ref.guided_score_closed_form(eps, x, t, y, std, 1e-3, 3, 4)
    got = oracle_op.guided_score_closed_form_op(eps, x, t, y, std, 1e-3, CoarseGrain(3, 4))
    assert ((got - want).abs().max() / want.abs().max()).item() <= 1e-6


def test_point_obs_struct_matches_library():
    lib = _lib.load()
    assert lib.c2w_abi_version() == 3
    assert lib.c2w_struct_size(4) == ctypes.sizeof(_lib.PointObs)
