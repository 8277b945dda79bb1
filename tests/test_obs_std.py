"""CPU tests of a noise std per observation: the std forms condition_on accepts for CoarseGrain, PointObservation and
CombinedObservation, their collapse to the per-variable path, every validation error; the point plan with std (runs of
entries per pixel, one per distinct std^2) against float64 autograd of the reference-form log-likelihood with the same
std tensor, over rank splits and strip geometries; and the combined per-observation split."""
import numpy as np
import pytest
import torch

import climate2weather_b200 as c2w
from climate2weather_b200 import score as S
from test_combined_obs import _conditioned_runtime
from test_point_obs import _op as _points_op

L, C, H, W = 13, 3, 32, 32


def _logp_grad(op, y, std, x0, gamma, r2):
    """d/dx0 of the reference's log p (src/thor/score.py:53-56: var = std^2 + gamma r^2 elementwise, err = y - A(x0))
    in float64; masked observations (NaN y or std there) contribute nothing."""
    x0 = x0.double().clone().requires_grad_(True)
    mask = op.mask_for(y.shape[1])
    var = std.double() ** 2 + torch.as_tensor(gamma, dtype=torch.float64).reshape(1, -1, 1) * r2
    err = torch.where(mask, y.double(), torch.zeros((), dtype=torch.float64)) - op(x0)
    term = torch.where(mask & torch.isfinite(var), err ** 2 / torch.where(mask, var, 1.0), 0.0)
    (gr,) = torch.autograd.grad(-term.sum() / 2, x0)
    return gr


def _dense_from_runs(pl, x0, gamma, r2, H_, W_, frame_lo, n_own):
    """What the per-observation kernel computes, in float64: per owned frame and pixel, the sum over the pixel's run
    of (ysum - wsum x0) / (std2 + gamma r^2); checks the run layout on the way."""
    C_ = x0.shape[1]
    out = np.zeros((n_own, C_, H_ * W_))
    ns, sr = pl["n_strips"], pl["strip_rows"]
    for i in range(n_own):
        s = pl["frame_slot"][i]
        if s < 0:
            continue
        for b in range(ns):
            e0, e1 = pl["strip_off"][s * ns + b], pl["strip_off"][s * ns + b + 1]
            assert np.all(np.diff(pl["pix"][e0:e1]) >= 0)  # sorted by pixel: a run is consecutive
            for e in range(e0, e1):
                px = pl["pix"][e]
                assert b * sr * W_ <= px < min(H_, (b + 1) * sr) * W_  # runs never cross a strip
                xv = x0[frame_lo + i].reshape(C_, -1)[:, px].double().numpy()
                var = pl["std2"][e].astype(np.float64) + np.asarray(gamma) * r2
                out[i, :, px] += (pl["ysum"][e].astype(np.float64) - pl["wsum"][e] * xv) / var
    return out.reshape(n_own, C_, H_, W_)


def _check_runs(pl):
    """Within a run: per variable, the used slots first, std^2 strictly ascending; unused slots wsum = ysum = 0,
    std2 = 1; every entry holds at least one observation."""
    pix, w, s2, ys = pl["pix"], pl["wsum"], pl["std2"], pl["ysum"]
    assert np.all((w > 0).any(1))
    e = 0
    while e < pix.size:
        k = e
        while k + 1 < pix.size and pix[k + 1] == pix[e] and k + 1 < _strip_end(pl, e):
            k += 1
        for c in range(w.shape[1]):
            used = w[e:k + 1, c] > 0
            n = int(used.sum())
            assert used[:n].all() and not used[n:].any()
            assert np.all(np.diff(s2[e:e + n, c]) > 0)
            assert np.all(s2[e + n:k + 1, c] == 1) and np.all(ys[e + n:k + 1, c] == 0)
        e = k + 1


def _strip_end(pl, e):
    off = pl["strip_off"]
    return int(off[np.searchsorted(off, e, side="right")])


def _station_std(op, C_, seed, classes=(0.05, 0.1, 0.2)):
    """A std [F, C, P] that takes up to len(classes) values per station, so that duplicated stations at one pixel
    hold runs of 2-3 classes; variable 0 has one class only, the others differ in number.  NaN under the mask."""
    g = torch.Generator().manual_seed(seed)
    F, P = op.n_frames, op.n_points
    idx = torch.randint(0, len(classes), (F, C_, P), generator=g)
    for c in range(C_):
        idx[:, c] = idx[:, c].clamp(max=min(c, len(classes) - 1))
    std = torch.tensor(classes)[idx]
    return torch.where(op.mask_for(C_), std, torch.tensor(float("nan")))


def _dup_op(C_, seed, H_=H, W_=W, L_=L):
    """Stations with three at one pixel and two at another, on top of _points_op's duplicates and corners."""
    op, y = _points_op(L_, C_, H_, W_, 5, 40, seed)
    rows, cols = op.rows.clone(), op.cols.clone()
    rows[5:8], cols[5:8] = 7, 9
    rows[8:10], cols[8:10] = H_ - 1, 0
    return c2w.PointObservation(op.frames, rows, cols, op.mask), y


# ------------------------------------------------------------------------------------------------ the plan
@pytest.mark.parametrize("strip", [1, 3, 16])
@pytest.mark.parametrize("seed", [0, 1])
def test_plan_with_std_matches_autograd_of_reference_log_p(strip, seed):
    """Every owned frame, for every partition into ranks: the plan's runs reproduce the fp64 gradient of the
    reference-form log p with the same std tensor; strips of one row, a ragged last strip and strip borders."""
    C_ = 3
    op, y = _dup_op(C_, seed)
    std = _station_std(op, C_, seed)
    gamma, r2 = [1e-2, 3e-3, 5e-2], 0.37
    x0 = torch.randn(L, C_, H, W, generator=torch.Generator().manual_seed(seed + 50), dtype=torch.float64).float()
    want = _logp_grad(op, y, std, x0, gamma, r2)
    for cuts in ((0, L), (0, 5, L), (0, 2, 7, 11, L)):
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            pl = S.point_plan(op, y, L, C_, H, W, lo, hi, strip, std=std)
            _check_runs(pl)
            got = _dense_from_runs(pl, x0, gamma, r2, H, W, lo, hi - lo)
            ref = want[lo:hi].numpy()
            assert np.abs(got - ref).max() <= 1e-6 * np.abs(want.numpy()).max(), (cuts, lo)
    pl = S.point_plan(op, y, L, C_, H, W, 0, L, strip, std=std)
    assert pl["pix"].size > np.unique(pl["frame_slot"][pl["frame_slot"] >= 0]).size  # there are runs
    run_len = np.diff(np.flatnonzero(np.r_[True, np.diff(pl["pix"]) != 0, True]))
    assert run_len.max() in (2, 3)


def test_plan_runs_split_classes_per_variable():
    """Three stations at one pixel of one frame with std (0.1, 0.2, 0.1) for variable 0 and (0.3, 0.3, 0.3) for
    variable 1: a run of two entries, classes ascending, variable 1 in the first slot only; sums in fp64."""
    op = c2w.PointObservation([2], [4, 4, 4], [5, 5, 5])
    y = torch.tensor([[[1.0, 2.0, 4.0], [0.5, 0.25, 0.125]]])
    std = torch.tensor([[[0.1, 0.2, 0.1], [0.3, 0.3, 0.3]]])
    pl = S.point_plan(op, y, 4, 2, 8, 8, 0, 4, 2, std=std)
    assert pl["pix"].tolist() == [4 * 8 + 5] * 2
    s01, s02, s03 = (np.float32(v) * np.float32(v) for v in (0.1, 0.2, 0.3))
    assert pl["std2"].tolist() == [[s01, s03], [s02, 1.0]]
    assert pl["ysum"].tolist() == [[5.0, 0.875], [2.0, 0.0]] and pl["wsum"].tolist() == [[2, 3], [1, 0]]


def test_plan_with_a_constant_std_is_the_plan_without():
    """A std constant per variable: the same entries, order and sums as the plan without std (one per pixel)."""
    op, y = _points_op(L, C, H, W, 5, 40, 3)
    std = torch.tensor([0.1, 0.2, 0.3]).reshape(1, C, 1).expand(op.n_frames, C, op.n_points)
    for lo, hi in ((0, L), (4, 9)):
        a = S.point_plan(op, y, L, C, H, W, lo, hi, 4)
        b = S.point_plan(op, y, L, C, H, W, lo, hi, 4, std=std)
        assert "std2" not in a
        for k in ("frame_slot", "strip_off", "pix", "ysum", "wsum"):
            assert a[k].dtype == b[k].dtype and np.array_equal(a[k], b[k]), k
        assert a["frames"] == b["frames"] and a["n_slots"] == b["n_slots"]
        used = b["wsum"] > 0
        assert np.array_equal(b["std2"][used], (np.float32([0.1, 0.2, 0.3]) ** 2)[np.nonzero(used)[1]])


def test_infinite_std_is_the_station_masked_out():
    """std = +inf at an observation: the plan is exactly the one with that observation masked."""
    op, y = _points_op(L, C, H, W, 5, 40, 4)
    std = torch.full((op.n_frames, C, op.n_points), 0.2)
    std[:, :, 3] = float("inf")
    std[1, 0, 6] = float("inf")
    std[2, 1, 7] = 0.4
    mask = op.mask_for(C).clone()
    mask[:, :, 3] = False
    mask[1, 0, 6] = False
    masked = c2w.PointObservation(op.frames, op.rows, op.cols, mask)
    a = S.point_plan(op, y, L, C, H, W, 0, L, 4, std=std)
    b = S.point_plan(masked, y, L, C, H, W, 0, L, 4, std=std)
    for k in ("frame_slot", "strip_off", "pix", "ysum", "wsum", "std2"):
        assert np.array_equal(a[k], b[k]), k


# ------------------------------------------------------------------------------------------------ accepted forms
def _cond(op, y, std, x_shape, monkeypatch):
    return _conditioned_runtime(op, y, std, x_shape, monkeypatch)


def test_coarse_std_forms(monkeypatch):
    """CoarseGrain: per frame, per tile and full std per observation; [1, C, 1, 1] and C values stay per variable;
    a per-observation std that is constant per variable collapses to it."""
    op = c2w.CoarseGrain(3, 8)
    want = (-(-L // 3), C, H // 8, W // 8)
    y = torch.randn(want)
    for std in (0.1, [0.1, 0.2, 0.3], torch.tensor([0.1, 0.2, 0.3]).reshape(1, C, 1, 1),
                torch.tensor([0.1, 0.2, 0.3]).reshape(1, C, 1, 1).expand(want)):
        seen = _cond(op, y, std, (L, C, H, W), monkeypatch)
        assert "obs_std" not in seen and len(seen["std"]) >= C
        assert seen["runtime"].coarse_std2_dev is None
    per_frame = torch.linspace(0.1, 0.5, want[0]).reshape(-1, 1, 1, 1)
    per_tile = torch.rand(1, C, want[2], want[3], generator=torch.Generator().manual_seed(0)) + 0.05
    full = torch.rand(want, generator=torch.Generator().manual_seed(1)) + 0.05
    for std in (per_frame, per_tile, full):
        seen = _cond(op, y, std, (L, C, H, W), monkeypatch)
        b = torch.broadcast_to(std, want).float()
        assert torch.equal(seen["obs_std"]["coarse_std2"], b * b) and seen["obs_std"]["point_std"] is None
        assert torch.equal(seen["runtime"].coarse_std2_dev, b * b)


def test_point_std_forms(monkeypatch):
    """PointObservation: per station [1, 1, P], per station and variable [1, C, P] and full [F, C, P]; a [1, 1, P]
    std with P == C is per variable; masked NaN is ignored."""
    op, y = _points_op(L, C, H, W, 5, 40, 5)
    F, P = op.n_frames, op.n_points
    g = torch.Generator().manual_seed(2)
    for std in (torch.rand(1, 1, P, generator=g) + 0.05, torch.rand(1, C, P, generator=g) + 0.05,
                torch.rand(F, C, P, generator=g) + 0.05):
        seen = _cond(op, y, std, (L, C, H, W), monkeypatch)
        assert torch.equal(seen["obs_std"]["point_std"], torch.broadcast_to(std, (F, C, P)))
        pl = S.point_plan(op, y, L, C, H, W, 0, L, S.point_strip_rows(H, W), std=seen["obs_std"]["point_std"])
        assert torch.equal(seen["runtime"].points["tensors"]["std2"], torch.as_tensor(pl["std2"]))
    nan_masked = torch.where(op.mask_for(C), torch.tensor(0.2), torch.tensor(float("nan"))).expand(F, C, P)
    seen = _cond(op, y, nan_masked, (L, C, H, W), monkeypatch)
    assert "obs_std" not in seen and seen["std"] == pytest.approx([0.2] * C)
    # P == C: a [1, 1, P] std reads as C per-variable values
    op3 = c2w.PointObservation([1, 4], [0, 3, 5], [2, 2, 2])
    y3 = torch.randn(2, C, 3)
    seen = _cond(op3, y3, torch.tensor([0.1, 0.2, 0.3]).reshape(1, 1, 3), (L, C, H, W), monkeypatch)
    assert "obs_std" not in seen and seen["std"][:C] == pytest.approx([0.1, 0.2, 0.3])


def test_combined_std_forms(monkeypatch):
    """CombinedObservation: a flat std that varies within a term takes the per-observation path; std_per_term keeps
    refusing it; constant per (term, variable) stays per term."""
    op = c2w.CombinedObservation(c2w.CoarseGrain(3, 8), _points_op(L, C, H, W, 4, 20, 6)[0])
    cs, ps = op.term_shapes((L, C, H, W))
    y = op.pack(torch.randn(cs), torch.randn(ps), (L, C, H, W))
    g = torch.Generator().manual_seed(3)
    cstd, pstd = torch.rand(cs, generator=g) + 0.05, torch.rand(ps, generator=g) + 0.05
    for c_part, p_part in ((cstd, 0.1), (0.2, pstd), (cstd, pstd)):
        std = op.pack(c_part, p_part, (L, C, H, W))
        with pytest.raises(ValueError, match="a std per observation is not supported"):
            op.std_per_term(std, (L, C, H, W))
        seen = _cond(op, y, std, (L, C, H, W), monkeypatch)
        c2, p = op.std_per_observation(std, (L, C, H, W))
        assert torch.equal(seen["obs_std"]["coarse_std2"], c2) and torch.equal(seen["obs_std"]["point_std"], p)
        assert torch.equal(seen["runtime"].coarse_std2_dev, c2) and "std2" in seen["runtime"].points["tensors"]
    seen = _cond(op, y, op.pack([0.1, 0.2, 0.3], 0.05, (L, C, H, W)), (L, C, H, W), monkeypatch)
    assert "obs_std" not in seen and seen["point_std"] == pytest.approx([0.05] * C)


def test_combined_std_per_observation_split():
    """The coarse std^2 block (fp32 std * std) and the point std, from a flat tensor, a scalar or C values."""
    op = c2w.CombinedObservation(c2w.CoarseGrain(4, 16), c2w.PointObservation([0, 5], [1, 2], [3, 4]))
    x_shape = (9, 2, 32, 32)
    cs, ps = op.term_shapes(x_shape)
    g = torch.Generator().manual_seed(4)
    cstd, pstd = torch.rand(cs, generator=g), torch.rand(ps, generator=g)
    c2, p = op.std_per_observation(op.pack(cstd, pstd, x_shape), x_shape)
    assert c2.shape == cs and c2.dtype == torch.float32 and torch.equal(c2, cstd * cstd)
    assert torch.equal(p, pstd)
    c2, p = op.std_per_observation([0.5, 0.25], x_shape)
    assert torch.equal(c2[:, 1], torch.full(c2[:, 1].shape, 0.0625)) and torch.equal(p[:, 0], torch.full((2, 2), 0.5))
    with pytest.raises(ValueError, match="std has 7 values"):
        op.std_per_observation(torch.ones(7), x_shape)


# ------------------------------------------------------------------------------------------------ errors
def test_std_errors(monkeypatch):
    op = c2w.CoarseGrain(3, 8)
    want = (-(-L // 3), C, H // 8, W // 8)
    y = torch.randn(want)
    with pytest.raises(ValueError, match=r"does not broadcast to A\(x\) of shape \(5, 3, 4, 4\)"):
        _cond(op, y, torch.ones(5, C, 4, 3), (L, C, H, W), monkeypatch)
    bad = torch.full(want, 0.1)
    bad[2, 1, 0, 0] = -0.1
    with pytest.raises(ValueError, match="negative or NaN"):
        _cond(op, y, bad, (L, C, H, W), monkeypatch)
    bad[2, 1, 0, 0] = float("nan")
    with pytest.raises(ValueError, match="negative or NaN"):
        _cond(op, y, bad, (L, C, H, W), monkeypatch)
    bad[2, 1, 0, 0] = float("inf")  # allowed
    assert "obs_std" in _cond(op, y, bad, (L, C, H, W), monkeypatch)
    with pytest.raises(ValueError, match="gamma: expected a scalar or 3 per-variable values"):
        S._per_channel(torch.full(want, 1e-2), C, "gamma")  # a per-observation gamma is still refused (runtime)
    # points: checked at condition_on, where the shape is known
    pop, py = _points_op(L, C, H, W, 5, 40, 7)
    sf = c2w.DefaultScoreFunction.__new__(c2w.DefaultScoreFunction)
    sf.likelihood, sf._runtimes = None, {}
    with pytest.raises(ValueError, match=r"does not broadcast to A\(x\) of shape \(5, 3, 40\)"):
        sf.condition_on(A=pop, y=py, std=torch.ones(1, 2, 40))
    bad = torch.full((5, C, 40), 0.1)
    unmasked = torch.nonzero(pop.mask_for(C))[0].tolist()
    masked = torch.nonzero(~pop.mask_for(C))[0].tolist()
    bad[tuple(masked)] = float("nan")
    sf.condition_on(A=pop, y=py, std=bad)  # NaN under the mask: ignored
    bad[tuple(masked)] = -1.0
    sf.condition_on(A=pop, y=py, std=bad)
    bad[tuple(unmasked)] = float("nan")
    with pytest.raises(ValueError, match="negative or NaN at an unmasked observation"):
        sf.condition_on(A=pop, y=py, std=bad)
    # combined: at runtime set-up, per term
    cop = c2w.CombinedObservation(op, pop)
    cs, ps = cop.term_shapes((L, C, H, W))
    yc = cop.pack(torch.randn(cs), torch.zeros(ps), (L, C, H, W))
    for part in ("coarse", "point"):
        cstd, pstd = torch.full(cs, 0.1), torch.where(pop.mask_for(C), 0.2, float("nan"))
        (cstd if part == "coarse" else pstd)[(0, 0, 0)] = -1.0
        if part == "point":
            pstd[tuple(unmasked)] = -1.0
        with pytest.raises(ValueError, match=f"{part} term: std .* is negative or NaN"):
            _cond(cop, yc, cop.pack(cstd, pstd, (L, C, H, W)), (L, C, H, W), monkeypatch)
