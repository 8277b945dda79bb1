"""CPU tests of batched sampling of independent problems (SDAPipeline.sample_batch): every refusal with its message
and member index, the concatenated point plan against each member's own plan, and the stacked coarse blocks and
[M, C] gamma / std^2 arrays against each member's own conditioning, fp32 bit for bit."""
import numpy as np
import pytest
import torch
import torch.distributed as dist

import climate2weather_b200 as c2w
from climate2weather_b200.score import (PointObservation, batch_condition, concat_point_plans, condition_for,
                                        point_plan)

L, C, H, W = 9, 4, 8, 8


def _net(k=2, C=C):
    return c2w.ScoreUNet(channels=C * (2 * k + 1), embedding_dim=64, hidden_channels=(64,), hidden_blocks=(1,),
                         attention_levels=(), activation=torch.nn.SiLU)


def _sf(net=None, k=2, **cond):
    sf = c2w.DefaultScoreFunction(net if net is not None else _net(k), markov_order=k, noise_process=c2w.SDAPipeline())
    if cond:
        sf.condition_on(**cond)
    return sf


def _coarse(t=3, s=4, **kw):
    return dict(A=c2w.CoarseGrain(t, s), y=torch.randn(-(-L // t), C, H // s, W // s), std=0.1, exact_grad=False, **kw)


def _run(sfs, noise=None, **kw):
    noise = torch.randn(len(sfs), L, C, H, W) if noise is None else noise
    return c2w.SDAPipeline().sample_batch(sfs, noise, steps=2, show_progressbar=False, **kw)


# ------------------------------------------------------------------------------------------------ refusals
def test_noise_must_be_five_dimensional():
    with pytest.raises(ValueError, match=r"noise must be \[M, L, C, H, W\], got shape \(9, 4, 8, 8\)"):
        c2w.SDAPipeline().sample_batch([_sf()], torch.randn(9, 4, 8, 8), steps=2)


def test_one_score_function_and_one_seed_per_member():
    net = _net()
    with pytest.raises(ValueError, match="3 score functions for 2 members"):
        _run([_sf(net)] * 3, torch.randn(2, L, C, H, W))
    with pytest.raises(ValueError, match="3 seeds for 2 members"):
        _run([_sf(net)] * 2, seeds=[1, 2, 3])


def test_score_functions_of_this_package_only():
    with pytest.raises(TypeError, match="member 1: .*got function"):
        _run([_sf(), lambda x, t: x])


def test_reference_rng_with_corrections_is_refused():
    pipe = c2w.SDAPipeline()
    pipe.rng = "reference"
    net = _net()
    with pytest.raises(NotImplementedError, match="rng='reference' with corrections"):
        pipe.sample_batch([_sf(net), _sf(net)], torch.randn(2, L, C, H, W), steps=2, corrections=1)


def test_members_share_one_network():
    net = _net()
    with pytest.raises(ValueError, match="member 2: its ScoreUNet is not member 0's"):
        _run([_sf(net), _sf(net), _sf(_net())])


def test_members_share_the_markov_order():
    net = _net(k=2)
    other = c2w.DefaultScoreFunction(net, markov_order=1, noise_process=c2w.SDAPipeline())
    with pytest.raises(ValueError, match="member 1: markov_order 1 differs from member 0's 2"):
        _run([_sf(net), other])


def test_members_share_the_windows_per_launch():
    net = _net()
    a, b = _sf(net), _sf(net)
    b.max_windows = 2
    with pytest.raises(ValueError, match="member 1: 2 windows per launch .* differ from member 0's 5"):
        _run([a, b])
    # an explicit setting equal to the class default is the same plan: b passes this check and fails the next one
    a.condition_on(**_coarse())
    b.max_windows = 5
    with pytest.raises(NotImplementedError, match="member 1: unconditioned while member 0 is conditioned"):
        _run([a, b])


def test_operator_families_must_agree():
    net = _net()
    P = 5
    pts = PointObservation([0, 4], torch.arange(P), torch.arange(P))
    a = _sf(net, **_coarse())
    b = _sf(net, A=pts, y=torch.randn(2, C, P), std=0.1, exact_grad=False)
    with pytest.raises(NotImplementedError, match="member 1: operator family PointObservation differs from member "
                                                  "0's CoarseGrain"):
        _run([a, b])
    comb = c2w.CombinedObservation(c2w.CoarseGrain(3, 4), pts)
    shape = (L, C, H, W)
    c = _sf(net, A=comb, y=comb.pack(torch.randn(3, C, 2, 2), torch.randn(2, C, P), shape), std=0.1, exact_grad=False)
    with pytest.raises(NotImplementedError, match="member 2: operator family CombinedObservation differs"):
        _run([b, b, c])


def test_coarse_steps_must_agree():
    net = _net()
    a = _sf(net, **_coarse(3, 4))
    with pytest.raises(NotImplementedError, match=r"member 1: coarse \(t_step, s_step\) = \(3, 2\) differs from "
                                                  r"member 0's \(3, 4\)"):
        _run([a, _sf(net, **_coarse(3, 2))])
    # an opaque closure recognised as AvgPool2d(4)(x[::2]): another t
    opaque = _sf(net, A=lambda x: torch.nn.functional.avg_pool2d(x[::2], 4), y=torch.randn(5, C, 2, 2), std=0.1,
                 exact_grad=False)
    with pytest.raises(NotImplementedError, match=r"member 2: coarse \(t_step, s_step\) = \(2, 4\) differs"):
        _run([a, a, opaque])


def test_conditioned_and_unconditioned_members_do_not_mix():
    net = _net()
    with pytest.raises(NotImplementedError, match="member 1: unconditioned while member 0 is conditioned; the "
                                                  "members are all conditioned or none"):
        _run([_sf(net, **_coarse()), _sf(net)])


def test_exact_grad_is_refused():
    net = _net()
    with pytest.raises(NotImplementedError, match="member 1: a batch runs closed-form guidance only.*exact_grad=False"):
        _run([_sf(net, **_coarse()), _sf(net, **dict(_coarse(), exact_grad=True))])


def test_time_sharding_is_refused(tmp_path):
    dist.init_process_group("gloo", init_method=f"file://{tmp_path / 'store'}", rank=0, world_size=1)
    try:
        net = _net()
        with pytest.raises(NotImplementedError, match="member 1: a batch does not run on a time-sharded"):
            _run([_sf(net), _sf(net).enable_time_sharding()])
    finally:
        dist.destroy_process_group()


def test_a_members_geometry_error_names_the_member():
    net = _net()
    bad = _sf(net, A=c2w.CoarseGrain(3, 4), y=torch.randn(2, C, 2, 2), std=0.1, exact_grad=False)
    with pytest.raises(ValueError, match=r"member 1: CoarseGrain\(t_step=3, s_step=4\): observation y of shape"):
        _run([_sf(net, **_coarse()), bad])


# ------------------------------------------------------------------------------------------------ the point plan
def _points(g, Lm, Cm, Hm, Wm, F, P, masked=0.3):
    frames = torch.randperm(Lm, generator=g)[:F]
    mask = torch.rand(F, Cm, P, generator=g) > masked
    op = PointObservation(frames, torch.randint(0, Hm, (P,), generator=g), torch.randint(0, Wm, (P,), generator=g),
                          mask)
    op.rows[1], op.cols[1] = op.rows[0], op.cols[0]  # two stations on one pixel
    return op, torch.randn(F, Cm, P, generator=g)


@pytest.mark.parametrize("strip", [1, 3, 16])
@pytest.mark.parametrize("per_obs", [False, True])
def test_concatenated_plan_is_each_members_own(strip, per_obs):
    g = torch.Generator().manual_seed(strip + 10 * per_obs)
    Lm, Cm, Hm, Wm = 11, 3, 32, 16
    members = []
    for m, (F, P) in enumerate([(4, 30), (2, 7), (5, 50), (3, 12)]):
        op, y = _points(g, Lm, Cm, Hm, Wm, F, P)
        if m == 2:  # a fully masked member
            op.mask[:] = False
        std = None
        if per_obs:  # runs: two std values per station
            std = torch.where(torch.rand(F, Cm, P, generator=g) > 0.5, 0.1, 0.2)
            std[..., ::7] = float("inf")
        members.append(point_plan(op, y, Lm, Cm, Hm, Wm, 0, Lm, strip, std=std))
    assert members[2]["n_slots"] == 0
    cat = concat_point_plans(members)
    assert cat["frame_slot"].shape == (4 * Lm,) and cat["frame_slot"].dtype == np.int32
    assert cat["strip_off"].dtype == np.int32 and cat["n_slots"] == sum(p["n_slots"] for p in members)
    slots = entries = 0
    n_strips = members[0]["n_strips"]
    for m, own in enumerate(members):
        fs = cat["frame_slot"][m * Lm:(m + 1) * Lm]
        assert np.array_equal(np.where(fs >= 0, fs - slots, fs), own["frame_slot"]), m
        off = cat["strip_off"][slots * n_strips:(slots + own["n_slots"]) * n_strips + 1]
        assert np.array_equal(off - entries, own["strip_off"]), m
        n = int(own["strip_off"][-1])
        for name in ("pix", "ysum", "wsum") + (("std2",) if per_obs else ()):
            got = cat[name][entries:entries + n]
            assert got.dtype == np.asarray(own[name]).dtype
            assert got.tobytes() == np.asarray(own[name]).tobytes(), (m, name)
        slots += own["n_slots"]
        entries += n
    assert entries == cat["pix"].size and int(cat["strip_off"][-1]) == entries


# ------------------------------------------------------------------------------------------------ stacked operands
def _own_std2(vals, Cm):
    """fp32(std^2) as a member's own run hands c2w_guide.std2 (a Python float squared, stored as a C float)."""
    import ctypes
    return np.array([(ctypes.c_float * 1)(float(v) ** 2)[0] for v in vals[:Cm]], dtype=np.float32)


def test_stacked_coarse_blocks_and_member_arrays_with_mixed_std_forms():
    g = torch.Generator().manual_seed(3)
    Cm, t, s = 3, 3, 4
    shape = (L, Cm, H, W)
    obs = (-(-L // t), Cm, H // s, W // s)
    lks = [
        dict(A=c2w.CoarseGrain(t, s), y=torch.randn(obs, generator=g), std=0.3, gamma=1e-2),
        dict(A=c2w.CoarseGrain(t, s), y=torch.randn(1, Cm, 1, W // s, generator=g).double(), std=[0.1, 0.2, 0.4],
             gamma=[1e-3, 2e-3, 3e-3]),
        dict(A=c2w.CoarseGrain(t, s), y=torch.randn(obs, generator=g), std=0.05 + torch.rand(1, 1, H // s, W // s,
                                                                                             generator=g), gamma=0.5),
    ]
    conds = []
    for lk in lks:
        conds.append(condition_for(dict(lk, op=None, y=torch.as_tensor(lk["y"]), exact=False), shape))
    b = batch_condition(conds, shape)
    assert b["per_obs"] and b["kind"] == "coarse" and b["std2"] is None
    assert b["y"].shape == (3 * obs[0],) + obs[1:] and b["y"].dtype == torch.float32
    for m, c in enumerate(conds):
        rows = slice(m * obs[0], (m + 1) * obs[0])
        own_y = c["y"].to(torch.float32).contiguous()
        assert b["y"][rows].numpy().tobytes() == own_y.numpy().tobytes(), m
        ob = c.get("obs_std")
        own = ob["coarse_std2"] if ob is not None else \
            torch.from_numpy(_own_std2(c["std"], Cm)).reshape(1, Cm, 1, 1).expand(obs)
        assert b["coarse_std2"][rows].numpy().tobytes() == own.to(torch.float32).contiguous().numpy().tobytes(), m
        assert b["gamma"][m].tobytes() == np.array(c["gamma"][:Cm], dtype=np.float32).tobytes(), m
    # per variable on every member: the [M, C] std^2 array, no tile block
    b2 = batch_condition(conds[:2], shape)
    assert not b2["per_obs"] and b2["coarse_std2"] is None
    for m, c in enumerate(conds[:2]):
        assert b2["std2"][m].tobytes() == _own_std2(c["std"], Cm).tobytes(), m


def test_combined_members_point_std_and_expanded_plans():
    g = torch.Generator().manual_seed(4)
    Cm = 2
    shape = (L, Cm, H, W)
    conds = []
    for m in range(3):
        op, py = _points(g, L, Cm, H, W, 3, 9)
        comb = c2w.CombinedObservation(c2w.CoarseGrain(2, 4), op)
        cy = torch.randn(-(-L // 2), Cm, 2, 2, generator=g)
        std = comb.pack(0.2 + 0.1 * m, torch.tensor([0.05, 0.07 + m]), shape) if m < 2 else \
            comb.pack(0.3, 0.05 + torch.rand(3, Cm, 9, generator=g), shape)
        lk = dict(A=comb, y=comb.pack(cy, py, shape), std=std, gamma=1e-2 * (m + 1), op=None, exact=False)
        conds.append(condition_for(lk, shape))
    b = batch_condition(conds[:2], shape)  # per (term, variable)
    assert not b["per_obs"] and b["kind"] == "combined"
    for m, c in enumerate(conds[:2]):
        assert b["std2"][m].tobytes() == _own_std2(c["std"], Cm).tobytes()
        assert b["point_std2"][m].tobytes() == _own_std2(c["point_std"], Cm).tobytes()
    b = batch_condition(conds, shape)  # member 2 per observation: all members on the per-observation kernels
    assert b["per_obs"] and b["point_std2"] is None and "std2" in b["plan"]
    strip = c2w.score.combined_strip_rows(H, W, 4)
    own = [point_plan(c["op"].points, c["point_y"], L, Cm, H, W, 0, L, strip, c2w.score.COMBINED_STRIP_PIX,
                      c["obs_std"]["point_std"]) for c in conds[2:]]
    n2 = int(own[0]["strip_off"][-1])
    for name in ("pix", "ysum", "wsum", "std2"):  # the last member's entries, byte for byte
        assert b["plan"][name][b["plan"][name].shape[0] - n2:].tobytes() == np.asarray(own[0][name]).tobytes(), name
    # a per-variable member's expanded plan has the entries of its own per-variable plan, with its std^2 on every
    # variable it observes (1.0, as the per-observation plans fill them, where an entry has none)
    plain = point_plan(conds[0]["op"].points, conds[0]["point_y"], L, Cm, H, W, 0, L, strip,
                       c2w.score.COMBINED_STRIP_PIX)
    n0 = int(plain["strip_off"][-1])
    for name in ("pix", "ysum", "wsum"):
        assert b["plan"][name][:n0].tobytes() == np.asarray(plain[name]).tobytes(), name
    assert np.array_equal(b["plan"]["frame_slot"][:L], plain["frame_slot"])
    want = np.where(plain["wsum"] > 0, _own_std2(conds[0]["point_std"], Cm)[None, :], np.float32(1.0))
    assert b["plan"]["std2"][:n0].tobytes() == want.astype(np.float32).tobytes()
