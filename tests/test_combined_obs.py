"""CPU tests of CombinedObservation (a coarse field and point observations in one likelihood): the operator, pack /
split / std_per_term, the reference-form likelihood against the sum of the two terms' own, the plan and upload split,
the strip height of the combined guidance kernel, every validation error, and exact-gradient window selection."""
import pytest
import torch

import climate2weather_b200 as c2w
from climate2weather_b200 import score as S

L, C, H, W = 13, 3, 32, 32


def _op(t=3, s=8, frames=(0, 4, 7, 12), P=20, seed=0, mask=True):
    g = torch.Generator().manual_seed(seed)
    rows, cols = torch.randint(0, H, (P,), generator=g), torch.randint(0, W, (P,), generator=g)
    m = torch.rand(len(frames), C, P, generator=g) > 0.3 if mask else None
    return c2w.CombinedObservation(c2w.CoarseGrain(t, s), c2w.PointObservation(list(frames), rows, cols, m))


def test_operator_is_the_concatenation_of_its_terms():
    op = _op()
    x = torch.randn(L, C, H, W, generator=torch.Generator().manual_seed(1))
    want = torch.cat([op.coarse(x).reshape(-1), op.points(x).reshape(-1)])
    assert torch.equal(op(x), want)
    cs, ps = op.term_shapes(x.shape)
    assert cs == (5, C, 4, 4) and ps == (4, C, 20) and op(x).numel() == 5 * C * 16 + 4 * C * 20


def test_pack_round_trips_and_expands_per_term_values():
    op = _op()
    cs, ps = op.term_shapes((L, C, H, W))
    a, b = torch.randn(cs), torch.randn(ps)
    flat = op.pack(a, b, (L, C, H, W))
    ga, gb = op.split(flat, (L, C, H, W))
    assert torch.equal(ga, a) and torch.equal(gb, b)
    std = op.pack(0.5, [0.1, 0.2, 0.3], (L, C, H, W))
    sa, sb = op.split(std, (L, C, H, W))
    assert torch.all(sa == 0.5)
    assert torch.equal(sb, torch.tensor([0.1, 0.2, 0.3]).reshape(1, C, 1).expand(ps))
    assert op.std_per_term(std, (L, C, H, W)) == ([0.5] * C, [float(torch.tensor(v)) for v in (0.1, 0.2, 0.3)])
    assert op.std_per_term([0.1, 0.2, 0.3], (L, C, H, W))[0] == op.std_per_term([0.1, 0.2, 0.3], (L, C, H, W))[1]
    with pytest.raises(ValueError, match="point part of shape"):
        op.pack(a, torch.randn(2, 2), (L, C, H, W))


def test_reference_log_p_is_the_sum_of_the_terms_own():
    """src/thor/score.py:44-60 with the flat y and flat std (var = std^2 + gamma (sigma/mu)^2 elementwise), by
    autograd in fp64, equals the sum of the two terms' own log-likelihoods with their own std."""
    op = _op(mask=False)
    g = torch.Generator().manual_seed(2)
    x = torch.randn(L, C, H, W, generator=g, dtype=torch.float64)
    cs, ps = op.term_shapes(x.shape)
    yc, yp = torch.randn(cs, generator=g, dtype=torch.float64), torch.randn(ps, generator=g, dtype=torch.float64)
    sc, sp = torch.tensor([0.3, 0.2, 0.5], dtype=torch.float64), torch.tensor([0.05, 0.07, 0.02], dtype=torch.float64)
    y = op.pack(yc, yp, x.shape).double()
    std = op.pack(sc, sp, x.shape).double()
    gamma, r2 = 0.01, 2.5

    def grad(fn):
        xg = x.clone().requires_grad_(True)
        (J,) = torch.autograd.grad(fn(xg), xg)
        return J

    flat = grad(lambda xx: -((y - op(xx)) ** 2 / (std ** 2 + gamma * r2)).sum() / 2)
    vc = (sc ** 2 + gamma * r2).reshape(1, C, 1, 1)
    vp = (sp ** 2 + gamma * r2).reshape(1, C, 1)
    terms = grad(lambda xx: -((yc - op.coarse(xx)) ** 2 / vc).sum() / 2 - ((yp - op.points(xx)) ** 2 / vp).sum() / 2)
    assert torch.allclose(flat, terms, rtol=1e-12, atol=1e-14)
    assert flat.abs().max() > 0


@pytest.mark.parametrize("H_,W_,s,R", [(32, 32, 4, 32), (32, 32, 8, 32), (32, 32, 32, 32), (48, 96, 3, 21),
                                       (128, 128, 16, 16), (128, 128, 64, 64), (128, 128, 128, 128)])
def test_combined_strip_rows(H_, W_, s, R):
    assert S.combined_strip_rows(H_, W_, s) == R
    assert R % s == 0 and R * W_ <= S.COMBINED_STRIP_PIX


def test_combined_strip_rows_refuses_a_map_beyond_the_kernel():
    with pytest.raises(NotImplementedError, match="exceeds the 16384 pixels"):
        S.combined_strip_rows(256, 256, 128)


def test_plan_and_upload_split():
    """The runtime's conditioning: the coarse block in A_c(x)'s shape, and this rank's point plan with strip_rows = R
    equal to point_plan at that strip (including a rank's slice)."""
    op = _op()
    cs, ps = op.term_shapes((L, C, H, W))
    g = torch.Generator().manual_seed(3)
    yc, yp = torch.randn(cs, generator=g), torch.randn(ps, generator=g)
    yp = yp.masked_fill(~op.points.mask, float("nan"))
    y = op.pack(yc, yp, (L, C, H, W))
    got_c, got_p = op.split(y, (L, C, H, W))
    assert torch.equal(got_c, yc) and got_c.shape == cs
    R = S.combined_strip_rows(H, W, op.coarse.s_step)
    for lo, hi in ((0, L), (3, 9)):
        a = S.point_plan(op.points, got_p, L, C, H, W, lo, hi, R, S.COMBINED_STRIP_PIX)
        b = S.point_plan(op.points, yp, L, C, H, W, lo, hi, R, S.COMBINED_STRIP_PIX)
        assert a["strip_rows"] == R and a["n_strips"] == -(-H // R)
        for k in ("frame_slot", "strip_off", "pix", "ysum", "wsum"):
            assert (a[k] == b[k]).all(), k


def test_constructor_limits():
    cg, pt = c2w.CoarseGrain(3, 8), _op().points
    with pytest.raises(NotImplementedError, match="cannot hold another set"):
        c2w.CombinedObservation(c2w.CombinedObservation(cg, pt), pt)
    with pytest.raises(NotImplementedError, match="at most one operator of each kind, got two CoarseGrain"):
        c2w.CombinedObservation(cg, c2w.CoarseGrain(2, 4))
    with pytest.raises(NotImplementedError, match="at most one operator of each kind, got two PointObservation"):
        c2w.CombinedObservation(pt, pt)


def test_split_length_and_std_errors():
    op = _op()
    cs, ps = op.term_shapes((L, C, H, W))
    n = 5 * C * 16 + 4 * C * 20
    with pytest.raises(ValueError, match=f"is not 1-D of length {n} \\({5 * C * 16} coarse"):
        op.split(torch.zeros(n - 1), (L, C, H, W))
    with pytest.raises(ValueError, match=f"is not 1-D of length {n}"):
        op.split(torch.zeros(5 * C * 16), (L, C, H, W))  # the coarse block is not broadcast
    std = op.pack(0.1, 0.2, (L, C, H, W)).clone()
    std[3] = 0.4
    with pytest.raises(ValueError, match="std varies within the coarse term"):
        op.std_per_term(std, (L, C, H, W))
    std = op.pack(0.1, 0.2, (L, C, H, W)).clone()
    std[-1] = 0.4
    with pytest.raises(ValueError, match="std varies within the point term"):
        op.std_per_term(std, (L, C, H, W))
    with pytest.raises(ValueError, match="std has 7 values"):
        op.std_per_term(torch.ones(7), (L, C, H, W))


def _score_fn():
    sf = c2w.DefaultScoreFunction.__new__(c2w.DefaultScoreFunction)
    sf.likelihood, sf._runtimes = None, {}
    return sf


def test_condition_on_requires_a_flat_y():
    op = _op()
    with pytest.raises(ValueError, match="y must be the flat tensor"):
        _score_fn().condition_on(A=op, y=torch.zeros(3, 4), std=0.1)
    _score_fn().condition_on(A=op, y=torch.zeros(10), std=0.1)  # the length is checked with the geometry


def _conditioned_runtime(op, y, std, x_shape, monkeypatch):
    """AbstractScoreFunction.runtime up to set_condition, with the device runtime replaced by a recorder."""
    seen = {}
    real = S._Runtime

    class Rt:  # the device-free part of _Runtime: its set_condition, which builds this rank's point plan
        def __init__(self, sf, L, C, H, W, device, plan, max_windows, exact=False):
            self.sf, self.L, self.C, self.H, self.W, self.device, self.plan, self.exact = sf, L, C, H, W, device, plan, exact

        def set_condition(self, cond):
            seen.update(cond)
            real.set_condition(self, cond)
            seen["runtime"] = self

    monkeypatch.setattr(S, "_Runtime", Rt)
    sf = _score_fn()
    sf.markov_order, sf.max_windows, sf.shard, sf.device = 2, None, None, None
    sf.condition_on(A=op, y=y, std=std, exact_grad=False)
    monkeypatch.setattr(sf, "_compute_device", lambda x: torch.device("cpu"))
    sf.runtime(torch.zeros(x_shape))
    return seen


def test_runtime_splits_y_and_std(monkeypatch):
    op = _op()
    cs, ps = op.term_shapes((L, C, H, W))
    yc, yp = torch.randn(cs), torch.randn(ps)
    seen = _conditioned_runtime(op, op.pack(yc, yp, (L, C, H, W)), op.pack([0.1, 0.2, 0.3], 0.05, (L, C, H, W)),
                                (L, C, H, W), monkeypatch)
    assert torch.equal(seen["y"], yc) and torch.equal(seen["point_y"], yp)
    assert seen["std"] == pytest.approx([0.1, 0.2, 0.3]) and seen["point_std"] == pytest.approx([0.05] * C)
    assert seen["op"] is op
    rt = seen["runtime"]  # the uploaded coarse block and the point plan at the combined kernel's strip
    assert torch.equal(rt.y_dev, yc)
    R = S.combined_strip_rows(H, W, op.coarse.s_step)
    want = S.point_plan(op.points, yp, L, C, H, W, 0, L, R, S.COMBINED_STRIP_PIX)
    assert rt.points["obs"].strip_rows == R and rt.points["n_strips"] == want["n_strips"]
    for k in ("frame_slot", "strip_off", "pix", "ysum", "wsum"):
        assert (rt.points["tensors"][k].numpy() == want[k]).all(), k


def test_runtime_checks_each_term(monkeypatch):
    """The coarse term's limits (NotImplementedError) with their own messages, then the flat length (ValueError naming
    both lengths), then the point term's geometry."""
    op = _op(s=5)
    with pytest.raises(NotImplementedError, match="s_step=5 must divide the 32x32 grid"):
        _conditioned_runtime(op, torch.zeros(10), 0.1, (L, C, H, W), monkeypatch)
    op = _op()
    with pytest.raises(ValueError, match="is not 1-D of length"):
        _conditioned_runtime(op, torch.zeros(10), 0.1, (L, C, H, W), monkeypatch)
    op = _op(frames=(0, 4, 7, 20))
    y = torch.zeros(sum(torch.Size(s).numel() for s in op.term_shapes((L, C, H, W))))
    with pytest.raises(ValueError, match="frame 20 outside a trajectory of 13 frames"):
        _conditioned_runtime(op, y, 0.1, (L, C, H, W), monkeypatch)


def test_observed_window_selection_is_the_fold_preimage_of_the_union():
    """observed_windows with the union of {f : f % t == 0} and the point term's observed frames selects exactly the
    windows whose composed output meets an observed frame, over every partition of the windows into shards."""
    k, Lt = 2, 23
    op = c2w.CombinedObservation(c2w.CoarseGrain(6, 8),
                                 c2w.PointObservation([1, 3, 9, 22], [0, 5], [1, 2],
                                                      torch.tensor([[[True, False]], [[False, False]], [[True, True]],
                                                                    [[False, True]]])))
    frames = op.observed_frames(Lt, 1)
    assert frames == [0, 1, 6, 9, 12, 18, 22]
    n_win = Lt - 2 * k
    owner = {}
    for j in range(n_win):
        outs = [j + k] + (list(range(k)) if j == 0 else []) + (list(range(Lt - k, Lt)) if j == n_win - 1 else [])
        for f in outs:
            owner[f] = j
    want = sorted({owner[f] for f in frames})
    assert S.observed_windows(0, n_win, n_win, Lt, k, frames) == want
    for cuts in ((0, 7, n_win), (0, 1, 10, 18, n_win)):
        got = []
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            got += S.observed_windows(lo, hi, n_win, Lt, k, frames)
        assert got == want
