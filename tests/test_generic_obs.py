"""CPU tests of the generic observation path (any differentiable observation operator A): which operators take it and
which keep their fused conditioning exactly as before, and its refusals — y, std or gamma not broadcasting to A(x),
time sharding, and mixing it with another operator family in a batch."""
import re

import pytest
import torch
import torch.distributed as dist
import torch.nn.functional as F

import climate2weather_b200 as c2w
from climate2weather_b200.score import (CoarseGrain, CombinedObservation, GenericObservation, PointObservation,
                                        _check_observation_shape, _combined_std, _per_channel, _recognise_operator,
                                        _single_std, coarse_grain_observation, condition_for, generic_operands)

L, C, H, W = 9, 4, 8, 8


def _net(k=2):
    return c2w.ScoreUNet(channels=C * (2 * k + 1), embedding_dim=64, hidden_channels=(64,), hidden_blocks=(1,),
                         attention_levels=(), activation=torch.nn.SiLU)


def _sf(net=None, **cond):
    sf = c2w.DefaultScoreFunction(net if net is not None else _net(), markov_order=2, noise_process=c2w.SDAPipeline())
    if cond:
        sf.condition_on(**cond)
    return sf


def _parent_condition_for(lk: dict, shape, members: int = 0) -> dict:
    """condition_for as it was before the generic path existed: the fused operators' conditioning must not move."""
    L, C, H, W = (int(v) for v in shape)
    if lk["op"] is None:
        if isinstance(lk["A"], (PointObservation, CombinedObservation)):
            lk["op"] = lk["A"]
        else:
            lk["op"] = _recognise_operator(lk["A"], L, C, H, W, lk["y"].shape)
        lk["gamma_c"] = _per_channel(lk["gamma"], C, "gamma")
    op, y = lk["op"], lk["y"]
    cond = dict(op=op, gamma=lk["gamma_c"])
    if members:
        cond["members"] = members
    if isinstance(op, CombinedObservation):
        _check_observation_shape(op.coarse, op.term_shapes(shape)[0], L, C, H, W)
        y, cond["point_y"] = op.split(y, shape)
        if torch.as_tensor(lk["std"]).numel() in (1, C):
            cond["std"], cond["point_std"] = op.std_per_term(lk["std"], shape)
        else:
            cond.update(_combined_std(op, lk["std"], shape))
    else:
        if isinstance(op, CoarseGrain):
            y = coarse_grain_observation(op, y, L, C, H, W)
        cond.update(_single_std(op, lk["std"], y.shape, C))
    return dict(cond, y=y)


def _same(a, b, path="cond"):
    if isinstance(a, dict):
        assert isinstance(b, dict) and a.keys() == b.keys(), (path, a.keys(), b.keys())
        for k in a:
            _same(a[k], b[k], f"{path}[{k!r}]")
    elif isinstance(a, torch.Tensor):
        assert isinstance(b, torch.Tensor) and a.dtype == b.dtype and torch.equal(a, b), path
    elif isinstance(a, CoarseGrain):
        assert type(b) is CoarseGrain and (a.t_step, a.s_step) == (b.t_step, b.s_step), path
    elif isinstance(a, (PointObservation, CombinedObservation)):
        assert a is b, path
    else:
        assert type(a) is type(b) and a == b, (path, a, b)


def _likelihood(A, y, std=0.1, gamma=1e-2):
    return dict(A=A, y=torch.as_tensor(y), std=std, gamma=gamma, op=None, exact=False)


def _route(A, y, std=0.1, gamma=1e-2, shape=(L, C, H, W)):
    return condition_for(_likelihood(A, y, std, gamma), shape)


# ------------------------------------------------------------------------------------------------ routing
def _fused_cases():
    g = torch.Generator().manual_seed(0)
    pts = PointObservation([0, 4, 7], torch.tensor([1, 5, 5]), torch.tensor([2, 6, 6]),
                           torch.rand(3, C, 3, generator=g) > 0.3)
    comb = CombinedObservation(CoarseGrain(3, 4), pts)
    yc = torch.randn(3, C, 2, 2, generator=g)
    yp = torch.randn(3, C, 3, generator=g)
    per_obs = 0.05 + torch.rand(3, C, 2, 2, generator=g)
    return [
        ("CoarseGrain", CoarseGrain(3, 4), yc, 0.1, 1e-2),
        ("CoarseGrain std per variable", CoarseGrain(3, 4), yc, [0.1, 0.2, 0.3, 0.4], [1e-2, 1e-3, 1e-4, 1e-5]),
        ("CoarseGrain std per observation", CoarseGrain(3, 4), yc, per_obs, 1e-2),
        ("CoarseGrain y broadcast", CoarseGrain(3, 4), yc[:1], 0.1, 1e-2),
        ("driver closure", lambda x: F.avg_pool2d(x[::3], 4), yc, 0.1, 1e-2),
        ("driver closure s=2", lambda x: torch.nn.AvgPool2d(2)(x[::2]), torch.randn(5, C, 4, 4, generator=g), 0.2,
         1e-3),
        ("PointObservation", pts, yp, 0.1, 1e-2),
        ("PointObservation std per observation", pts, yp, 0.05 + torch.rand(3, C, 3, generator=g), 1e-2),
        ("CombinedObservation", comb, comb.pack(yc, yp, (L, C, H, W)), 0.1, 1e-2),
        ("CombinedObservation std per term", comb, comb.pack(yc, yp, (L, C, H, W)),
         comb.pack(0.1, 0.3, (L, C, H, W)), 1e-2),
    ]


@pytest.mark.parametrize("case", _fused_cases(), ids=lambda c: c[0])
@pytest.mark.parametrize("members", [0, 3])
def test_fused_operators_keep_their_conditioning(case, members):
    _, A, y, std, gamma = case
    got = condition_for(_likelihood(A, y, std, gamma), (L, C, H, W), members)
    want = _parent_condition_for(_likelihood(A, y, std, gamma), (L, C, H, W), members)
    assert not isinstance(got["op"], GenericObservation)
    _same(got, want)


def test_fused_operators_keep_their_errors():
    # CoarseGrain's limits and y's shape raise as before; an explicit CoarseGrain never goes generic
    with pytest.raises(NotImplementedError, match="at most 32"):
        _route(CoarseGrain(1, 2), torch.randn(L, C, 64, 64), shape=(L, C, 128, 128))
    with pytest.raises(ValueError, match="does not broadcast to A"):
        _route(CoarseGrain(3, 4), torch.randn(2, C, 2, 2))
    with pytest.raises(ValueError, match="does not broadcast to A"):
        _route(CoarseGrain(3, 4), torch.randn(3, C, 4))


def _cuda_only(x):
    """What an operator holding CUDA tensors does with a CPU tensor."""
    if not x.is_cuda:
        raise RuntimeError("Expected all tensors to be on the same device")
    return x


def _matrix_op():
    M = torch.randn(5, H * W, generator=torch.Generator().manual_seed(1))
    return lambda x: torch.einsum("pk,lck->lcp", M, x.reshape(*x.shape[:2], -1))


@pytest.mark.parametrize("what,A,y", [
    ("y not 4-D (time mean of the field)", lambda x: x.mean(0), torch.randn(C, H, W)),
    ("time mean of tile means", lambda x: F.avg_pool2d(x, 4).reshape(3, 3, C, 2, 2).mean(1), torch.randn(3, C, 2, 2)),
    ("matrix operator", _matrix_op(), torch.randn(L, C, 5)),
    ("not a tile average (other channel count)", lambda x: x[:, :2, ::4, ::4], torch.randn(L, 2, 2, 2)),
    ("a tile average no (t, s) matches", lambda x: F.avg_pool2d(x[::3], 4) * 2, torch.randn(3, C, 2, 2)),
    ("fails on the CPU probe", lambda x: _cuda_only(x)[::3], torch.randn(3, C, H, W)),
])
def test_other_operators_go_generic(what, A, y):
    cond = _route(A, y)
    assert isinstance(cond["op"], GenericObservation) and cond["op"].A is A, what
    assert cond["y"] is not None and cond["std"] == 0.1 and cond["gamma"] == 1e-2


def test_recognised_closure_outside_the_kernel_limits_goes_generic():
    """avg_pool2d(x[::t], 2) at 128 x 128 (64 tiles per row) is the coarse family, but the fused kernel handles at most
    32 tiles per row: the closure goes generic, while CoarseGrain(t, 2) keeps its NotImplementedError."""
    Lb, Hb = 4, 128
    y = torch.randn(2, 1, 64, 64)
    cond = _route(lambda x: F.avg_pool2d(x[::2], 2), y, shape=(Lb, 1, Hb, Hb))
    assert isinstance(cond["op"], GenericObservation)
    with pytest.raises(NotImplementedError, match="at most 32"):
        _route(CoarseGrain(2, 2), y, shape=(Lb, 1, Hb, Hb))


# ------------------------------------------------------------------------------------------------ errors
def test_generic_operands_check_broadcasting():
    A = lambda x: F.avg_pool2d(x, 4).reshape(3, 3, C, 2, 2).mean(1)
    x = torch.zeros(L, C, H, W)
    ops = generic_operands(A, torch.randn(3, C, 2, 2), torch.tensor([0.1, 0.2, 0.3, 0.4]).reshape(1, C, 1, 1),
                           torch.full((3, 1, 2, 2), 1e-3), x)
    assert ops["shape"] == (3, C, 2, 2) and ops["y"].dtype == torch.float32
    assert torch.equal(ops["std2"], torch.tensor([0.1, 0.2, 0.3, 0.4]).reshape(1, C, 1, 1) ** 2)
    for name, bad in (("y", dict(y=torch.randn(2, C, 2, 2))), ("std", dict(std=torch.ones(C))),
                      ("gamma", dict(gamma=torch.ones(3, C, 2, 3)))):
        kw = {**dict(y=torch.randn(3, C, 2, 2), std=0.1, gamma=1e-2), **bad}
        shape = re.escape(str(tuple(torch.as_tensor(kw[name]).shape)))
        with pytest.raises(ValueError, match=rf"generic observation path: {name} of shape {shape} does not broadcast "
                                             rf"to A\(x\) of shape \(3, 4, 2, 2\)"):
            generic_operands(A, kw["y"], kw["std"], kw["gamma"], x)


def test_generic_operator_that_raises_names_the_path():
    def A(x):
        raise IndexError("no such station")
    with pytest.raises(RuntimeError, match="generic observation path: A raised IndexError.*no such station"):
        generic_operands(A, torch.zeros(1), 0.1, 1e-2, torch.zeros(L, C, H, W))


def test_time_sharding_is_refused(tmp_path):
    dist.init_process_group("gloo", init_method=f"file://{tmp_path / 'store'}", rank=0, world_size=1)
    try:
        sf = _sf(A=lambda x: x.mean(0), y=torch.randn(C, H, W), std=0.1, exact_grad=False).enable_time_sharding()
        with pytest.raises(NotImplementedError, match="generic observation path .* time-sharded score function"):
            c2w.SDAPipeline().sample(sf, torch.randn(L, C, H, W), steps=2, show_progressbar=False)
        # the fused operators keep running time-sharded up to the device
        fused = _sf(A=CoarseGrain(3, 4), y=torch.randn(3, C, 2, 2), std=0.1, exact_grad=False).enable_time_sharding()
        try:
            fused.runtime(torch.randn(L, C, H, W))
        except NotImplementedError as e:
            pytest.fail(f"a fused operator was refused: {e}")
        except Exception:
            pass  # no CUDA device here
    finally:
        dist.destroy_process_group()


def test_batch_family_mixing_names_the_member():
    net = _net()
    fused = _sf(net, A=CoarseGrain(3, 4), y=torch.randn(3, C, 2, 2), std=0.1, exact_grad=False)
    generic = _sf(net, A=lambda x: x.mean(0), y=torch.randn(C, H, W), std=0.1, exact_grad=False)
    run = lambda sfs: c2w.SDAPipeline().sample_batch(sfs, torch.randn(len(sfs), L, C, H, W), steps=2,
                                                     show_progressbar=False)
    with pytest.raises(NotImplementedError, match="member 1: operator family GenericObservation differs from member "
                                                  "0's CoarseGrain"):
        run([fused, generic])
    with pytest.raises(NotImplementedError, match="member 2: operator family CoarseGrain differs from member "
                                                  "0's GenericObservation"):
        run([generic, generic, fused])
