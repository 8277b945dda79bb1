"""CPU tests of ensemble sampling (SDAPipeline.sample_ensemble): the refusals and their messages, the member-major
window / frame layout against the reference's unfold / fold applied member by member, the point plan repeated per
member, and the default seeds drawn in member order."""
import numpy as np
import pytest
import torch
import torch.distributed as dist

import climate2weather_b200 as c2w
from climate2weather_b200.score import PointObservation, point_plan
from oracle import score_ref


def ensemble_windows(members: int, L: int, k: int) -> np.ndarray:
    """The member-major layout the kernels compute from the one integer Nw = L - 2k (K0's gather, the fold in K1's
    compose epilogue and compose_generic_kernel), restated: one row per ensemble window G in [0, members * Nw) of
    (member m = G div Nw, window j = G mod Nw, first frame G + 2k m = m L + j, head (j == 0), tail (j == Nw - 1))."""
    nw = L - 2 * k
    G = np.arange(members * nw)
    m, j = G // nw, G % nw
    return np.stack([m, j, G + 2 * k * m, j == 0, j == nw - 1], axis=1).astype(np.int64)


def _sf(k=2, C=4):
    net = c2w.ScoreUNet(channels=C * (2 * k + 1), embedding_dim=64, hidden_channels=(64,), hidden_blocks=(1,),
                        attention_levels=(), activation=torch.nn.SiLU)
    return c2w.DefaultScoreFunction(net, markov_order=k, noise_process=c2w.SDAPipeline())


def test_noise_must_be_five_dimensional():
    with pytest.raises(ValueError, match=r"noise must be \[M, L, C, H, W\], got shape \(9, 4, 8, 8\)"):
        c2w.SDAPipeline().sample_ensemble(_sf(), torch.randn(9, 4, 8, 8), steps=2)


def test_one_seed_per_member():
    with pytest.raises(ValueError, match="3 seeds for 2 members"):
        c2w.SDAPipeline().sample_ensemble(_sf(), torch.randn(2, 9, 4, 8, 8), steps=2, seeds=[1, 2, 3])


def test_reference_rng_with_corrections_is_refused():
    pipe = c2w.SDAPipeline()
    pipe.rng = "reference"
    with pytest.raises(NotImplementedError, match="rng='reference' with corrections"):
        pipe.sample_ensemble(_sf(), torch.randn(2, 9, 4, 8, 8), steps=2, corrections=1)


def test_exact_grad_is_refused():
    sf = _sf()
    sf.condition_on(A=c2w.CoarseGrain(3, 4), y=torch.randn(3, 4, 2, 2), std=0.1, exact_grad=True)
    with pytest.raises(NotImplementedError, match="closed-form guidance only.*exact_grad=False"):
        c2w.SDAPipeline().sample_ensemble(sf, torch.randn(2, 9, 4, 8, 8), steps=2)


def test_time_sharding_is_refused(tmp_path):
    dist.init_process_group("gloo", init_method=f"file://{tmp_path / 'store'}", rank=0, world_size=1)
    try:
        sf = _sf().enable_time_sharding()
        with pytest.raises(NotImplementedError, match="time-sharded score function"):
            c2w.SDAPipeline().sample_ensemble(sf, torch.randn(2, 9, 4, 8, 8), steps=2)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("M,L,k", [(1, 13, 6), (2, 13, 6), (3, 14, 6), (3, 26, 6), (4, 9, 2), (2, 5, 2), (3, 3, 1)])
def test_member_layout_matches_unfold_and_fold_per_member(M, L, k):
    """Every ensemble window reads the frames the reference's unfold gives its member's window, and the fold of all
    windows (centre slot, member-local head and tail) writes every frame of every member exactly once, from the
    (window, slot) the reference's fold names for that member alone."""
    w, nw = 2 * k + 1, L - 2 * k
    rows = ensemble_windows(M, L, k)
    assert rows.shape == (M * nw, 5)
    frames = torch.arange(M * L).reshape(M, L, 1, 1, 1).float()
    source = {}
    for G, (m, j, first, head, tail) in enumerate(rows.tolist()):
        assert (m, j) == (G // nw, G % nw)
        unfolded = c2w.score._window_view(frames[m], w)  # the reference's unfold of member m alone
        assert unfolded[j, :, 0, 0].tolist() == list(range(first, first + w))
        slots = ([*range(k)] if head else []) + [k] + ([*range(k + 1, w)] if tail else [])
        for tau in slots:
            f = first + tau
            assert f not in source, f"frame {f} written twice"
            source[f] = (m, j, tau)
    assert sorted(source) == list(range(M * L))
    ref = score_ref.fold_index(L, k, 1)  # [L, 1, (window, window-channel)] of one trajectory
    for m in range(M):
        for i in range(L):
            assert source[m * L + i] == (m, int(ref[i, 0, 0]), int(ref[i, 0, 1])), (m, i)


def test_point_plan_is_repeated_per_member():
    g = torch.Generator().manual_seed(5)
    L, C, H, W, P = 9, 3, 16, 16, 20
    mask = torch.rand(3, C, P, generator=g) > 0.3
    op = PointObservation([7, 0, 4], torch.randint(0, H, (P,), generator=g), torch.randint(0, W, (P,), generator=g),
                          mask)
    y = torch.randn(3, C, P, generator=g)
    std = torch.rand(3, C, P, generator=g) + 0.1
    for s in (None, std):
        one = point_plan(op, y, L, C, H, W, 0, L, 4, std=s)
        ens = point_plan(op, y, L, C, H, W, 0, L, 4, std=s, members=3)
        assert np.array_equal(ens["frame_slot"], np.tile(one["frame_slot"], 3))
        assert ens["frame_slot"].dtype == np.int32
        for name in one:
            if name != "frame_slot":
                assert np.array_equal(np.asarray(ens[name]), np.asarray(one[name])), name


def test_default_seeds_are_drawn_in_member_order():
    pipe = c2w.SDAPipeline()
    torch.manual_seed(11)
    sequential = [pipe._draw_seed(corrections=2) for _ in range(4)]  # what four sample() calls draw, one each
    torch.manual_seed(11)
    one = int(torch.empty((), dtype=torch.int64).random_().item())
    assert sequential[0] == one and len(set(sequential)) == 4
    torch.manual_seed(11)
    assert pipe._draw_seed(corrections=0) == 0  # no corrector, no draw
    assert int(torch.empty((), dtype=torch.int64).random_().item()) == one
    pipe.rng = "reference"
    assert pipe._draw_seed(corrections=2) == 0
