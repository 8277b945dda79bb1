"""Host-side mirror of `thor.score` (reference src/thor/score.py:7-185): AbstractScoreFunction,
DefaultScoreFunction, BatchedScoreFunction — same constructors, `condition_on`, `__call__`, `score_fn`.

What differs is where the work happens: the trajectory lives in HBM as fp32 [frames, H, W, C]; unfold, the UNet,
the centre-pick compose, the likelihood guidance and the predictor/corrector updates are CUDA kernels behind
include/c2w_b200.h.  Nothing here computes on the CPU and nothing falls back to torch ops; the one computation torch
runs is a user's own observation operator A and its VJP on the generic observation path (GenericObservation).
"""
from __future__ import annotations

import contextlib
import ctypes
import math
from typing import Callable, Optional, Sequence, Union

import numpy as np
import torch
import torch.distributed as dist
import torch.nn.functional as F
from torch import Tensor

from . import _lib
from .model import ScoreUNet, build_from_reference
from .sharding import PeerHalo, ShardPlan, exchange_halos, exchange_halos_adjoint, halo_transport, make_plan


class CoarseGrain:
    """The reference's observation operator (exp/downscaling.py:129-132): every `t_step`-th frame, mean over
    `s_step` x `s_step` tiles.  Passing an instance as `A=` lets `condition_on` skip operator recognition."""

    def __init__(self, t_step: int, s_step: int):
        self.t_step, self.s_step = int(t_step), int(s_step)

    def __call__(self, x: Tensor) -> Tensor:
        return F.avg_pool2d(x[..., ::self.t_step, :, :, :], self.s_step, stride=self.s_step)

    def __repr__(self):
        return f"CoarseGrain(t_step={self.t_step}, s_step={self.s_step})"


class PointObservation:
    """Variables observed at single grid points of chosen frames (weather stations, in-situ records with gaps, a
    variable measured at some sites only, fully observed frames):

        A(x)[m, c, p] = mask[m, c, p] * x[frames[m], c, rows[p], cols[p]]

    `frames`: F distinct global frame indices in any order; `rows`, `cols`: P pixel positions shared by every observed
    frame (several may name the same pixel; their contributions add); `mask`: bool [F, C, P], default all true — False
    marks a missing value or a variable not measured at that site, and the matching entries of y are ignored (they may
    be NaN).  Calling the object is the plain torch operator, so the same instance can condition the reference."""

    def __init__(self, frames, rows, cols, mask=None):
        self.frames = torch.as_tensor(frames, dtype=torch.long).reshape(-1).cpu()
        self.rows = torch.as_tensor(rows, dtype=torch.long).reshape(-1).cpu()
        self.cols = torch.as_tensor(cols, dtype=torch.long).reshape(-1).cpu()
        if self.rows.numel() != self.cols.numel():
            raise ValueError(f"PointObservation: {self.rows.numel()} rows but {self.cols.numel()} cols")
        if self.frames.numel() == 0 or self.rows.numel() == 0:
            raise ValueError("PointObservation: needs at least one frame and one point")
        if torch.unique(self.frames).numel() != self.frames.numel():
            raise ValueError(f"PointObservation: repeated frame in {self.frames.tolist()}")
        if bool((self.frames < 0).any()):
            raise ValueError(f"PointObservation: negative frame index in {self.frames.tolist()}")
        self.mask = None
        if mask is not None:
            self.mask = torch.as_tensor(mask).cpu()
            if self.mask.dtype != torch.bool:
                raise ValueError(f"PointObservation: mask must be a bool tensor, got {self.mask.dtype}")
            if self.mask.dim() != 3 or self.mask.shape[0] != self.n_frames or self.mask.shape[2] != self.n_points:
                raise ValueError(f"PointObservation: mask of shape {tuple(self.mask.shape)} is not "
                                 f"[{self.n_frames}, C, {self.n_points}]")

    @property
    def n_frames(self) -> int:
        return self.frames.numel()

    @property
    def n_points(self) -> int:
        return self.rows.numel()

    def mask_for(self, C: int) -> Tensor:
        """The mask as bool [F, C, P] (all true when none was given)."""
        if self.mask is None:
            return torch.ones(self.n_frames, C, self.n_points, dtype=torch.bool)
        if self.mask.shape[1] != C:
            raise ValueError(f"PointObservation: mask of shape {tuple(self.mask.shape)} does not match "
                             f"[{self.n_frames}, {C}, {self.n_points}]")
        return self.mask

    def __call__(self, x: Tensor) -> Tensor:
        dev = x.device
        out = x[self.frames.to(dev)][:, :, self.rows.to(dev), self.cols.to(dev)]
        if self.mask is not None:
            out = out * self.mask.to(device=dev, dtype=out.dtype)
        return out

    def check_observation(self, y: Tensor) -> None:
        """y must be [F, C, P], finite wherever the mask is set (conditioning time)."""
        if y.dim() != 3 or y.shape[0] != self.n_frames or y.shape[2] != self.n_points:
            raise ValueError(f"PointObservation: y of shape {tuple(y.shape)} is not [{self.n_frames}, C, {self.n_points}]")
        m = self.mask_for(y.shape[1])
        if not bool(torch.isfinite(y.cpu()[m]).all()):
            raise ValueError("PointObservation: y is not finite at an unmasked observation")

    def check_geometry(self, L: int, C: int, H: int, W: int) -> None:
        """Frames in [0, L), points inside the H x W grid, C variables (runtime build)."""
        if int(self.frames.max()) >= L:
            raise ValueError(f"PointObservation: frame {int(self.frames.max())} outside a trajectory of {L} frames")
        if int(self.rows.min()) < 0 or int(self.rows.max()) >= H or int(self.cols.min()) < 0 or int(self.cols.max()) >= W:
            raise ValueError(f"PointObservation: a point lies outside the {H}x{W} grid")
        self.mask_for(C)

    def observed_frames(self, C: int) -> list:
        """Global frames with at least one unmasked observation, ascending."""
        keep = self.mask_for(C).flatten(1).any(1)
        return sorted(int(f) for f in self.frames[keep])

    def __repr__(self):
        return f"PointObservation(frames={self.n_frames}, points={self.n_points}, masked={self.mask is not None})"


class CombinedObservation:
    """A coarse field and point observations in one likelihood (downscaling with station records):

        A(x) = cat([coarse(x).reshape(-1), points(x).reshape(-1)])

    The terms are independent, so log p(y | x) is the sum of the two terms' own.  Calling the object is the plain torch
    operator, so the same instance, a flat y and a flat std condition the reference unchanged.  Build y (and a std
    that differs between the terms) with `pack`; the point block may be NaN under the point mask.

    `condition_on(A=CombinedObservation(...), y=flat, std=..., gamma=...)`: std is a scalar or C per-variable values
    shared by both terms, or a flat tensor in y's layout (`pack` builds it from per-term parts): constant per (term,
    variable), or a std per observation (NaN allowed under the point mask, +inf for an observation that should not
    count); gamma is a scalar or C per-variable values shared by both terms."""

    def __init__(self, coarse: CoarseGrain, points: PointObservation):
        if isinstance(coarse, CombinedObservation) or isinstance(points, CombinedObservation):
            raise NotImplementedError("CombinedObservation: a set of observation operators cannot hold another set")
        if type(coarse) is type(points) and isinstance(coarse, (CoarseGrain, PointObservation)):
            raise NotImplementedError(f"CombinedObservation: at most one operator of each kind, got two "
                                      f"{type(coarse).__name__}")
        if not isinstance(coarse, CoarseGrain) or not isinstance(points, PointObservation):
            raise TypeError(f"CombinedObservation(coarse: CoarseGrain, points: PointObservation), got "
                            f"({type(coarse).__name__}, {type(points).__name__})")
        self.coarse, self.points = coarse, points

    def __call__(self, x: Tensor) -> Tensor:
        return torch.cat([self.coarse(x).reshape(-1), self.points(x).reshape(-1)])

    def term_shapes(self, x_shape) -> tuple:
        """Shapes of the two terms' observations for a trajectory of x_shape = (L, C, H, W)."""
        L, C, H, W = (int(v) for v in x_shape)
        s = self.coarse.s_step
        return (-(-L // self.coarse.t_step), C, H // s, W // s), (self.points.n_frames, C, self.points.n_points)

    def pack(self, coarse_part, point_part, x_shape) -> Tensor:
        """The flat tensor in y's layout from the per-term parts, for a trajectory of x_shape = (L, C, H, W).  Each part
        is a tensor of its term's shape ([ceil(L / t), C, H / s, W / s] and [F, C, P]), a scalar, or C per-variable
        values; the last two are expanded to the term's shape (an observation std per term)."""
        parts = []
        for part, shape, name in zip((coarse_part, point_part), self.term_shapes(x_shape), ("coarse", "point")):
            t = torch.as_tensor(part).cpu()
            t = t if t.is_floating_point() else t.float()
            C = shape[1]
            if t.numel() == 1:
                t = t.reshape(-1).expand(math.prod(shape))
            elif t.numel() == C and math.prod(shape) != C:
                t = t.reshape(1, C, *([1] * (len(shape) - 2))).expand(shape)
            elif tuple(t.shape) != shape:
                raise ValueError(f"{self}: {name} part of shape {tuple(t.shape)} is neither {shape}, a scalar nor "
                                 f"{C} per-variable values")
            parts.append(t.reshape(-1))
        return torch.cat(parts)

    def split(self, flat, x_shape) -> tuple:
        """The per-term parts (coarse [ceil(L / t), C, H / s, W / s], point [F, C, P]) of a flat tensor in y's layout.
        Its length must be exactly the sum of both terms' sizes (the coarse block is not broadcast)."""
        flat = torch.as_tensor(flat)
        cs, ps = self.term_shapes(x_shape)
        nc, n = math.prod(cs), math.prod(cs) + math.prod(ps)
        if flat.dim() != 1 or flat.numel() != n:
            raise ValueError(f"{self}: y of shape {tuple(flat.shape)} is not 1-D of length {n} ({nc} coarse "
                             f"{cs} + {n - nc} point {ps} entries) for a trajectory of {list(x_shape)}")
        return flat[:nc].reshape(cs), flat[nc:].reshape(ps)

    def std_per_term(self, std, x_shape) -> tuple:
        """(coarse std, point std), C floats each: a scalar or C per-variable values serve both terms; a flat tensor in
        y's layout must be constant per (term, variable)."""
        C = int(x_shape[1])
        t = torch.as_tensor(std, dtype=torch.float32).reshape(-1).cpu()
        if t.numel() in (1, C):
            v = _per_channel(t, C, "std")[:C]
            return v, list(v)
        cs, ps = self.term_shapes(x_shape)
        if t.numel() != math.prod(cs) + math.prod(ps):
            raise ValueError(f"{self}: std has {t.numel()} values; expected a scalar, {C} per-variable values or "
                             f"{math.prod(cs) + math.prod(ps)} in y's layout")
        out = []
        for name, block in zip(("coarse", "point"), self.split(t, x_shape)):
            per_var = block.transpose(0, 1).reshape(C, -1)
            if not bool((per_var == per_var[:, :1]).all()):
                raise ValueError(f"{self}: std varies within the {name} term of a variable; it must be constant per "
                                 f"(term, variable) (a std per observation is not supported)")
            out.append([float(v) for v in per_var[:, 0]])
        return out[0], out[1]

    def std_per_observation(self, std, x_shape) -> tuple:
        """(coarse std^2 [ceil(L / t), C, H / s, W / s], point std [F, C, P]), fp32, from a scalar, C per-variable values
        or a flat tensor in y's layout.  std^2 is fp32(std) * fp32(std) rounded to fp32, as the reference's `std ** 2`.
        A std that is negative or NaN at an observation (under the point mask it is ignored) raises ValueError."""
        C = int(x_shape[1])
        t = torch.as_tensor(std, dtype=torch.float32).reshape(-1).cpu()
        cs, ps = self.term_shapes(x_shape)
        if t.numel() in (1, C):
            t = self.pack(t, t, x_shape)
        elif t.numel() != math.prod(cs) + math.prod(ps):
            raise ValueError(f"{self}: std has {t.numel()} values; expected a scalar, {C} per-variable values or "
                             f"{math.prod(cs) + math.prod(ps)} in y's layout")
        coarse, point = (b.contiguous() for b in self.split(t, x_shape))
        _check_std_values(coarse, None, f"{self}: coarse term")
        _check_std_values(point, self.points.mask_for(C), f"{self}: point term")
        return coarse * coarse, point

    def observed_frames(self, L: int, C: int) -> list:
        """Global frames either term observes, ascending."""
        return sorted(set(range(0, L, self.coarse.t_step)) | set(self.points.observed_frames(C)))

    def __repr__(self):
        return f"CombinedObservation({self.coarse}, {self.points})"


def combined_strip_rows(H: int, W: int, s: int) -> int:
    """Rows per CTA of the combined guidance kernel: a multiple of s, so that every observation tile lies in one strip,
    and near POINT_STRIP_PIX pixels — s * max(1, min(H / s, floor(2048 / (s W)))), 16 rows at 128 x 128 with s = 16.
    The strip's pixel map must fit COMBINED_STRIP_PIX ints (c2w_b200.h: C2W_COMBINED_STRIP_PIX)."""
    R = s * max(1, min(H // s, POINT_STRIP_PIX // (s * W)))
    if R * W > COMBINED_STRIP_PIX:
        raise NotImplementedError(f"CombinedObservation: a strip of {R} rows of {W} pixels (s_step={s}) exceeds the "
                                  f"{COMBINED_STRIP_PIX} pixels the combined guidance kernel maps")
    return R


def point_strip_rows(H: int, W: int) -> int:
    """Rows per CTA of the point-guidance kernel: the strip's pixel -> entry map fits C2W_POINT_STRIP_PIX ints of static
    shared memory (c2w_b200.h) — 16 rows, 8 KB at 128 x 128."""
    if W > POINT_STRIP_PIX:
        raise NotImplementedError(f"PointObservation: a row of {W} pixels exceeds the {POINT_STRIP_PIX} pixels the point "
                                  "guidance kernel maps per strip")
    return max(1, min(H, POINT_STRIP_PIX // W))


def guidance_tile(H: int, W: int) -> int:
    """Tile side of the guidance and corrector kernels' per-CTA partial sums: divides H and W with at most 32 tiles per
    row (16 at 128 x 128 and 256 x 256).  Patches with no such side (e.g. 16 x 1024) are refused before device work."""
    for s in (16, 8, 32, 4, 64, 2, 128, 1):
        if H % s == 0 and W % s == 0 and W // s <= 32:
            return s
    raise NotImplementedError(f"guided sampling on a {H} x {W} patch: no tile side s dividing H and W with W / s <= 32 "
                              "(the guidance kernels' per-CTA partial sums)")


POINT_STRIP_PIX = 2048  # C2W_POINT_STRIP_PIX
COMBINED_STRIP_PIX = 16384  # C2W_COMBINED_STRIP_PIX


def point_plan(op: PointObservation, y, L: int, C: int, H: int, W: int, frame_lo: int, frame_hi: int, strip: int,
               max_strip_pix: int = POINT_STRIP_PIX, std=None, members: int = 0) -> dict:
    """The device form of a point observation for the owned global frames [frame_lo, frame_hi) (c2w_point_obs).

    Observations of one (frame, pixel) merge into one entry: per variable ysum = sum(mask * y), wsum = sum(mask), summed
    in fp64 in point order and rounded to fp32 once — exact, since sum_p mask_p (y_p - x0) / var = (ysum - wsum x0) / var.
    Entries with wsum = 0 for every variable are dropped.  Entries are sorted by (frame, strip, pixel); frame_slot maps
    owned frame i (global frame_lo + i) to its observed slot or -1, strip_off is the CSR over (slot, strip).  Frames
    outside [frame_lo, frame_hi) are not kept.

    With `std` (a std per observation, [F, C, P] or broadcasting to it), only observations of one (frame, pixel,
    variable) with the same fp32 std^2 merge: a pixel's distinct std^2 become a run of consecutive entries, entry j of
    the run holding the j-th smallest std^2 of every variable (wsum = ysum = 0, std2 = 1 in the slots of a variable
    with fewer).  An observation with std^2 = inf contributes exactly zero and is left out, as if masked.  The plan then
    also holds std2 [n_entries, C] fp32.

    `members` = M > 0: the plan of an ensemble of M trajectories stored member-major, all conditioned on y — one
    member's plan with frame_slot repeated M times, so that every member's frames point at the same entries."""
    y = torch.as_tensor(y)
    op.check_observation(y)
    op.check_geometry(L, C, H, W)
    if y.shape[1] != C:
        raise ValueError(f"PointObservation: y has {y.shape[1]} variables, the trajectory {C}")
    if strip < 1 or strip * W > max_strip_pix:
        raise ValueError(f"strip of {strip} rows of {W} pixels exceeds {max_strip_pix} pixels")
    n_own = frame_hi - frame_lo
    frames = op.frames.numpy()
    pix = (op.rows * W + op.cols).numpy()
    mask = op.mask_for(C).numpy()
    sel = np.nonzero((frames >= frame_lo) & (frames < frame_hi))[0]
    sel = sel[np.argsort(frames[sel], kind="stable")]
    yv = np.where(mask[sel], y.detach().cpu().double().numpy()[sel], 0.0)      # [n_sel, C, P]; NaN under the mask -> 0
    wv = mask[sel].astype(np.float64)
    key = ((frames[sel] - frame_lo)[:, None] * (H * W) + pix[None, :]).reshape(-1)  # (local frame, pixel)
    if std is None:
        uk, inv = np.unique(key, return_inverse=True)                              # sorted: frame, then pixel
        ysum = np.zeros((uk.size, C))
        wsum = np.zeros((uk.size, C))
        np.add.at(ysum, inv, yv.transpose(0, 2, 1).reshape(-1, C))
        np.add.at(wsum, inv, wv.transpose(0, 2, 1).reshape(-1, C))
        keep = (wsum > 0).any(1)
        uk, ysum, wsum = uk[keep], ysum[keep], wsum[keep]
    else:
        uk, ysum, wsum, std2 = _plan_runs(op, std, key, sel, mask, yv, C)
    fr, px = uk // (H * W), uk % (H * W)
    n_strips = -(-H // strip)
    obs_frames = np.unique(fr)
    frame_slot = np.full(n_own, -1, dtype=np.int32)
    frame_slot[obs_frames] = np.arange(obs_frames.size, dtype=np.int32)
    cell = frame_slot[fr].astype(np.int64) * n_strips + (px // W) // strip  # non-decreasing: the keys are sorted
    counts = np.bincount(cell, minlength=obs_frames.size * n_strips)
    strip_off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    out = dict(frame_slot=np.tile(frame_slot, members) if members else frame_slot, strip_off=strip_off,
               pix=px.astype(np.int32), ysum=ysum.astype(np.float32), wsum=wsum.astype(np.float32), n_slots=int(obs_frames.size), strip_rows=int(strip), n_strips=n_strips,
               frames=[int(frame_lo + f) for f in obs_frames])
    if std is not None:
        out["std2"] = std2
    return out


def _plan_runs(op: PointObservation, std, key, sel, mask, yv, C: int) -> tuple:
    """point_plan's entries with a std per observation: (entry keys, local frame * H W + pixel, repeated over a pixel's
    run; ysum, wsum (fp64) and std2 (fp32), each [n_entries, C]).  The sums run in point order, as without std."""
    s = torch.broadcast_to(torch.as_tensor(std, dtype=torch.float32).cpu(), (op.n_frames, C, op.n_points))
    s2 = (s * s).numpy()[sel].transpose(0, 2, 1).reshape(-1, C)      # fp32 std^2 per (observation, variable)
    live = mask[sel].transpose(0, 2, 1).reshape(-1, C) & np.isfinite(s2)  # std = inf: contributes exactly 0
    o, c = np.nonzero(live)                                            # point order, then variable
    k, v = key[o], s2[o, c]
    # the class of an observation: the rank of its std^2 among the distinct ones of its (frame, pixel, variable)
    order = np.lexsort((v, c, k))
    ks, cs, vs = k[order], c[order], v[order]
    new_group = np.ones(order.size, dtype=bool)
    new_group[1:] = (ks[1:] != ks[:-1]) | (cs[1:] != cs[:-1])
    new_value = new_group.copy()
    new_value[1:] |= vs[1:] != vs[:-1]
    value_id = np.cumsum(new_value) - 1
    cls = np.empty(order.size, dtype=np.int64)
    cls[order] = value_id - np.maximum.accumulate(np.where(new_group, value_id, 0))
    n_cls = int(cls.max()) + 1 if cls.size else 1
    uk, inv = np.unique(k * n_cls + cls, return_inverse=True)          # sorted: frame, pixel, then class
    ysum = np.zeros((uk.size, C))
    wsum = np.zeros((uk.size, C))
    std2 = np.ones((uk.size, C), dtype=np.float32)
    np.add.at(ysum, (inv, c), yv.transpose(0, 2, 1).reshape(-1, C)[o, c])
    np.add.at(wsum, (inv, c), 1.0)
    std2[inv, c] = v
    return uk // n_cls, ysum, wsum, std2


def concat_point_plans(plans: Sequence[dict]) -> dict:
    """One point plan of a batch of independent problems stored member-major from each member's own plan (point_plan
    over that member's frames [0, L)): member m's slots are offset by the slot count of the members before it, the
    frame_slot arrays (-1 kept) and the CSR strip_off (member m's entry offsets shifted by the entries before it) are
    concatenated, and so are the entries (pix, ysum, wsum, std2 where every plan has it).  A member's entries are then
    byte for byte those of its own plan; a member without an unmasked observation contributes no slot."""
    slots = entries = 0
    frame_slot, strip_off = [], [np.zeros(1, dtype=np.int32)]
    for pl in plans:
        fs = np.asarray(pl["frame_slot"], dtype=np.int32)
        frame_slot.append(np.where(fs >= 0, fs + slots, fs).astype(np.int32))
        strip_off.append((np.asarray(pl["strip_off"][1:], dtype=np.int64) + entries).astype(np.int32))
        slots += int(pl["n_slots"])
        entries += int(pl["strip_off"][-1])
    out = dict(frame_slot=np.concatenate(frame_slot), strip_off=np.concatenate(strip_off), n_slots=slots,
               strip_rows=plans[0]["strip_rows"], n_strips=plans[0]["n_strips"])
    names = ("pix", "ysum", "wsum") + (("std2",) if all("std2" in pl for pl in plans) else ())
    for n in names:
        out[n] = np.concatenate([np.asarray(pl[n]) for pl in plans])
    return out


def batch_condition(conds: Sequence[dict], shape) -> dict:
    """The device operands of a batch of independent problems (SDAPipeline.sample_batch) from each member's own
    conditioning (condition_for), as host arrays, each in the form the member's own run hands its kernel:

    - "y": the coarse term's observations stacked member-major, [M ceil(L / t), C, H / s, W / s] fp32 (None without a
      coarse term); "coarse_std2": a per-observation tile std^2 block in the same layout, or None;
    - "plan": the point term's plans, one per member over its frames [0, L), concatenated (concat_point_plans), or None;
    - "gamma", "std2", "point_std2": [M, C] fp32 per member and variable; the per-variable std^2 is fp32(std^2) as the
      member's own run rounds it (std2 / point_std2 None with a std per observation).

    When any member has a std per observation the batch runs the per-observation kernels: every other member's
    per-variable std is expanded to its observations (the same fp32 std^2, and with one std per (pixel, variable) the
    point entries merge exactly as without a std)."""
    L, C, H, W = (int(v) for v in shape)
    M = len(conds)
    op0 = conds[0]["op"]
    combined, points = isinstance(op0, CombinedObservation), isinstance(op0, PointObservation)
    per_obs = any(c.get("obs_std") is not None for c in conds)
    sq = lambda vals: np.array([np.float64(v) ** 2 for v in vals[:C]], dtype=np.float64).astype(np.float32)
    out = dict(per_obs=per_obs, kind="combined" if combined else "points" if points else "coarse",
               gamma=np.array([[float(v) for v in c["gamma"][:C]] for c in conds], dtype=np.float32),
               std2=None, point_std2=None, y=None, coarse_std2=None, plan=None)
    if not per_obs:
        out["std2"] = np.stack([sq(c["std"]) for c in conds])
        if combined:
            out["point_std2"] = np.stack([sq(c["point_std"]) for c in conds])
    if not points:
        out["y"] = torch.cat([c["y"].to(torch.float32).reshape(-1, C, *c["y"].shape[2:]) for c in conds]).contiguous()
        if per_obs:
            blocks = []
            for c in conds:
                ob = c.get("obs_std")
                if ob is not None:
                    blocks.append(ob["coarse_std2"].to(torch.float32))
                else:  # per variable: the same fp32 std^2 on each of the member's observation tiles
                    v = torch.tensor(c["std"][:C], dtype=torch.float32).reshape(1, C, 1, 1)
                    blocks.append((v * v).expand(c["y"].shape))
            out["coarse_std2"] = torch.cat(blocks).contiguous()
    if points or combined:
        plans = []
        for c in conds:
            op, y = (c["op"].points, c["point_y"]) if combined else (c["op"], c["y"])
            strip, max_pix = (combined_strip_rows(H, W, c["op"].coarse.s_step), COMBINED_STRIP_PIX) if combined \
                else (point_strip_rows(H, W), POINT_STRIP_PIX)
            std = None
            if per_obs:
                ob = c.get("obs_std")
                std = ob["point_std"] if ob is not None else \
                    torch.tensor((c["point_std"] if combined else c["std"])[:C], dtype=torch.float32).reshape(1, C, 1)
            plans.append(point_plan(op, y, L, C, H, W, 0, L, strip, max_pix, std))
        out["plan"] = concat_point_plans(plans)
    return out


def _per_channel(v, C: int, name: str):
    """float | Tensor[1,C,1,1] | sequence  ->  4 floats (exp/downscaling.py:218-234)."""
    t = torch.as_tensor(v, dtype=torch.float32).reshape(-1).cpu()
    if t.numel() == 1:
        t = t.expand(C)
    if t.numel() != C:
        raise ValueError(f"{name}: expected a scalar or {C} per-variable values, got {t.numel()}")
    out = [float(x) for x in t]
    return out + [1.0] * (4 - len(out))


def _check_std_values(std: Tensor, mask, what: str) -> None:
    """A std per observation is >= 0 (+inf allowed: that observation contributes exactly zero) and not NaN wherever
    mask is set (mask None: everywhere)."""
    v = std if mask is None else std[mask]
    if bool((torch.isnan(v) | (v < 0)).any()):
        raise ValueError(f"{what}: std (A(x)'s shape {tuple(std.shape)}) is negative or NaN at an unmasked observation")


def _std_per_observation(std, shape, C: int, mask, what: str) -> Optional[Tensor]:
    """A std given per observation, broadcast to A(x)'s `shape`, fp32 and contiguous, after its checks; None for the
    per-variable forms, a scalar or C values, which `_per_channel` reads.  So a [1, 1, P] std with P == C is per
    variable: expand it to [F, C, P] to give each of the P stations its own."""
    t = torch.as_tensor(std, dtype=torch.float32).cpu()
    if t.numel() in (1, C):
        return None
    try:
        b = torch.broadcast_to(t, tuple(shape)).contiguous()
    except RuntimeError:
        raise ValueError(f"{what}: std of shape {tuple(t.shape)} does not broadcast to A(x) of shape {tuple(shape)}; "
                         f"expected a scalar, {C} per-variable values or a tensor that broadcasts to {tuple(shape)}") \
            from None
    _check_std_values(b, mask, what)
    return b


def _collapse_per_variable(std: Tensor, mask) -> Optional[list]:
    """The C per-variable values of a std [M, C, ...] that is constant per variable over its observations (where mask
    is set; 1.0 for a variable without any), else None.  Such a std runs on the per-variable kernels."""
    C = std.shape[1]
    per_var = std.transpose(0, 1).reshape(C, -1)
    keep = None if mask is None else mask.transpose(0, 1).reshape(C, -1)
    out = []
    for c in range(C):
        v = per_var[c] if keep is None else per_var[c][keep[c]]
        if v.numel() and not bool((v == v[0]).all()):
            return None
        out.append(float(v[0]) if v.numel() else 1.0)
    return out


def _check_observation_shape(op: CoarseGrain, y_shape, L: int, C: int, H: int, W: int) -> tuple:
    """The shape of A(x) for x of [L, C, H, W], [ceil(L / t), C, H / s, W / s], after two checks.  A (t, s) the
    guidance kernel cannot run raises NotImplementedError: t or s below 1, s not dividing H and W, more than 32 tiles
    per row.  A y that does not broadcast to A(x) raises ValueError naming both shapes: the reference computes
    `y - A(x0)`, while the kernel would read y out of bounds or at the wrong offsets."""
    t, s = op.t_step, op.s_step
    if t < 1 or s < 1:
        raise NotImplementedError(f"{op}: t_step and s_step must be at least 1")
    if H % s or W % s:
        raise NotImplementedError(f"{op}: s_step={s} must divide the {H}x{W} grid")
    if W // s > 32:
        raise NotImplementedError(f"{op}: {W // s} tiles per row of a {H}x{W} grid; the guidance kernel handles at "
                                  f"most 32 (s_step >= {-(-W // 32)})")
    want = (-(-L // t), C, H // s, W // s)
    try:
        ok = torch.broadcast_shapes(tuple(y_shape), want) == want
    except RuntimeError:
        ok = False
    if not ok:
        raise ValueError(f"{op}: observation y of shape {tuple(y_shape)} does not broadcast to A(x) of shape {want} "
                         f"for a trajectory of [{L}, {C}, {H}, {W}]")
    return want


def coarse_grain_observation(op: CoarseGrain, y, L: int, C: int, H: int, W: int) -> Tensor:
    """y broadcast to the shape of A(x) and made contiguous: the tensor the guidance kernel reads."""
    y = torch.as_tensor(y)
    return torch.broadcast_to(y, _check_observation_shape(op, y.shape, L, C, H, W)).contiguous()


def _recognise_operator(A: Callable, L: int, C: int, H: int, W: int, y_shape) -> CoarseGrain:
    """`A` is an opaque Python callable in the reference API.  The fused path implements exactly one operator
    family (every t-th frame, s x s mean); identify (t, s) from the shapes and verify on a random probe.  A
    CoarseGrain is taken as it is.  Either way the operator's limits and y's shape are checked."""
    if isinstance(A, CoarseGrain):
        _check_observation_shape(A, y_shape, L, C, H, W)
        return A
    Lo, Cy, Hs, Ws = y_shape
    if Cy != C or H % Hs or W % Ws or H // Hs != W // Ws:
        raise NotImplementedError(f"observation of shape {tuple(y_shape)} is not a tile average of [{L},{C},{H},{W}]")
    s = H // Hs
    g = torch.Generator().manual_seed(1234)
    probe = torch.randn(L, C, H, W, generator=g)
    got = A(probe)
    for t in range(1, L + 1):
        if -(-L // t) != Lo:
            continue
        cand = CoarseGrain(t, s)
        ref = cand(probe)
        if ref.shape == got.shape and torch.allclose(ref, got, rtol=1e-5, atol=1e-6):
            _check_observation_shape(cand, y_shape, L, C, H, W)
            return cand
    raise NotImplementedError("observation operator A was not recognised as `AvgPool2d(s)(x[::t])`; the fused "
                              "guidance kernel supports only that family (pass climate2weather_b200.CoarseGrain)")


class GenericObservation:
    """The operator record of the generic observation path: a differentiable callable `A` that is none of the operators
    the fused guidance kernels implement.  Each score evaluation runs the reference's log_p through it
    (src/thor/score.py:44-60): x0 = (x - sigma eps)/mu, then A and its vector-Jacobian product in torch on the device,
    g = A^T((y - A x0)/var), then the fused guidance and state update on g (c2w_guided_step_dense)."""

    def __init__(self, A: Callable):
        self.A = A

    def __repr__(self):
        return f"GenericObservation({self.A!r})"


def _route_operator(A: Callable, L: int, C: int, H: int, W: int, y_shape):
    """The operator record of `A` for a trajectory [L, C, H, W] and an observation of y_shape.  PointObservation and
    CombinedObservation as they are, a CoarseGrain checked by `_recognise_operator` (its errors raise).  Any other
    callable is recognised as the coarse family if it can be and the fused kernel runs its (t, s); otherwise (y not
    4-D, not a tile average, no (t, s) matching, (t, s) outside the kernel's limits, or A failing on the CPU probe) it
    takes the generic path."""
    if isinstance(A, (PointObservation, CombinedObservation)):
        return A
    if isinstance(A, CoarseGrain):
        return _recognise_operator(A, L, C, H, W, y_shape)
    if len(y_shape) != 4:
        return GenericObservation(A)
    try:
        return _recognise_operator(A, L, C, H, W, y_shape)
    except Exception:  # not recognised, outside the kernel's limits, or A cannot run on a CPU tensor
        return GenericObservation(A)


def _generic_autograd() -> contextlib.ExitStack:
    """The mode A and its VJP run in: autograd on (also inside a caller's no_grad or inference_mode) and fp32 (also
    inside a caller's autocast, as the reference driver's `fabric.autocast()`)."""
    stack = contextlib.ExitStack()
    stack.enter_context(torch.inference_mode(False))
    stack.enter_context(torch.enable_grad())
    stack.enter_context(torch.autocast("cuda", enabled=False))
    return stack


def generic_operands(A: Callable, y, std, gamma, x: Tensor) -> dict:
    """The operands of the generic observation path for trajectories shaped like x ([L, C, H, W] fp32 on the compute
    device): A evaluated once on x for the shape of A(x); y, std^2 (fp32(std) * fp32(std)) and gamma as fp32 tensors on
    x's device that broadcast to that shape.  A raising is re-raised naming this path; y, std or gamma not broadcasting
    raises ValueError naming both shapes."""
    with _generic_autograd():
        try:
            out = A(x)
        except Exception as e:
            raise RuntimeError(f"generic observation path: A raised {type(e).__name__} on an fp32 tensor of shape "
                               f"{list(x.shape)} on {x.device}: {e}") from e
        if not isinstance(out, Tensor):
            raise TypeError(f"generic observation path: A returned {type(out).__name__}, not a tensor")
        shape = tuple(out.shape)
        ops = dict(A=A, shape=shape)
        for name, v in (("y", y), ("std", std), ("gamma", gamma)):
            t = torch.as_tensor(v).to(device=x.device, dtype=torch.float32)
            try:
                ok = torch.broadcast_shapes(tuple(t.shape), shape) == shape
            except RuntimeError:
                ok = False
            if not ok:
                raise ValueError(f"generic observation path: {name} of shape {tuple(t.shape)} does not broadcast to "
                                 f"A(x) of shape {shape} for a trajectory of {list(x.shape)}")
            ops[name] = t
        std = ops.pop("std")
        ops["std2"] = std * std
    return ops


def observed_windows(win_lo: int, win_hi: int, n_win_global: int, L: int, k: int, t_step) -> list:
    """Windows j in [win_lo, win_hi) whose part of the composed score meets an OBSERVED frame.  The likelihood's cotangent
    g = A^T((y - A x0)/var) (src/thor/score.py:53-56) is non-zero on observed frames only — frame f with f % t_step == 0
    (exp/downscaling.py:131), or f in the given set of frames (PointObservation: the frames with an unmasked value) —
    and window j contributes frame j + k to the composed score (plus frames 0..k-1 if it is the first window, L-k..L-1
    if it is the last, src/thor/score.py:76-88): every other window has an identically zero output cotangent, so its
    vector-Jacobian product vanishes and its backward pass is skipped."""
    if isinstance(t_step, int):
        observed = lambda f: f % t_step == 0
    else:
        frames = set(int(f) for f in t_step)
        observed = frames.__contains__
    out = []
    for j in range(win_lo, win_hi):
        need = observed(j + k)
        if j == 0:
            need = need or any(observed(f) for f in range(0, k))
        if j == n_win_global - 1:
            need = need or any(observed(f) for f in range(L - k, L))
        if need:
            out.append(j)
    return out


def _upload_point_plan(pl: dict, with_std: bool, device, C: int) -> dict:
    """A point plan on the device: its tensors and the c2w_point_obs that points at them."""
    names = ("frame_slot", "strip_off", "pix", "ysum", "wsum") + (("std2",) if with_std else ())
    dev = {n: torch.as_tensor(pl[n]).to(device) for n in names}
    for n in names[2:]:  # no entries on this rank: still a valid pointer
        if dev[n].numel() == 0:
            dev[n] = torch.zeros(max(1, C), dtype=dev[n].dtype, device=device)
    ob = _lib.PointObs()
    ob.frame_slot, ob.strip_off, ob.pix = (dev[n].data_ptr() for n in ("frame_slot", "strip_off", "pix"))
    ob.ysum, ob.wsum = dev["ysum"].data_ptr(), dev["wsum"].data_ptr()
    ob.n_slots, ob.strip_rows = pl["n_slots"], pl["strip_rows"]
    return dict(obs=ob, tensors=dev, n_strips=pl["n_strips"])


class _Runtime:
    """Device-resident state of one trajectory (or of this rank's time shard of it), or of an ensemble of `members`
    trajectories of L frames stored member-major in one state [members * L, H, W, C] (members = 0: one trajectory).
    An ensemble's plan is that of one member; every kernel call covers all members at once (the *_members entry
    points), and every member is conditioned on the same observation, or, for a batch of independent problems
    (set_condition with one conditioning per member), on its own (c2w_guided_step_batch)."""

    def __init__(self, sf: "AbstractScoreFunction", L: int, C: int, H: int, W: int, device: torch.device,
                 plan: ShardPlan, max_windows: int, exact: bool = False, members: int = 0):
        if not 1 <= C <= 8:
            raise NotImplementedError(f"1 to 8 variables per frame (c2w_b200.h: C2W_MAX_VARS); got C={C}")
        self.sf, self.L, self.C, self.H, self.W, self.device, self.plan = sf, L, C, H, W, device, plan
        self.members = int(members)
        self.lib = _lib.load()
        k = sf.markov_order
        self.exact = bool(exact)  # exact_grad=True: guidance through the UNet VJP (src/thor/score.py:28-33,51-52)
        self.cond = None
        self.points = None        # PointObservation: this rank's device plan (c2w_point_obs), see set_condition
        self.batch = None         # a batch of independent problems: its per-member operands, see set_condition
        self.generic = None       # GenericObservation: every member's operands (generic_operands), see set_condition
        self._x0 = self._grad = None  # the generic path's x0 and cotangent g, fp32 NCHW over the updated frames
        self._grad_ready = False      # g is that of the current score evaluation
        self._engine_args = (C, 2 * k + 1, H, W, device)
        self._engine_windows = min(max_windows, self.n_windows)
        # an ensemble's convs are planned as a member's own run plans them (its window count per launch): tile width,
        # CTA pair and main loop, and with them the order of the fp32 sums, match that run's, so each member is computed
        # bit for bit as alone
        self._tile_windows = min(sf.max_windows or sf._default_windows(plan.n_win_global), plan.n_win_global) \
            if self.members else 0
        self._engine = None
        self._engine_vjp = None   # exact_grad: the stashing engine for the windows that need a backward pass
        self._engine_epoch = None
        self._sel = None          # exact_grad: cached selection of those windows (per conditioning)
        self._rest = None         # exact_grad: the other local windows (int32 device list)
        self.s_tile = guidance_tile(H, W)  # refuses a patch the guidance kernels cannot tile, before device work
        self.refresh_engine()
        f32 = dict(dtype=torch.float32, device=device)
        self.x = torch.zeros(self.n_frames, H, W, C, **f32)
        self.eps = torch.zeros_like(self.x)
        self.eps_g: Optional[Tensor] = None
        self.vjp = torch.zeros_like(self.x) if self.exact else None   # J_eps^T g, accumulated per score evaluation
        self.cot = torch.zeros_like(self.x) if self.exact else None   # g = A^T((y - A x0)/var)
        self.nan_flag = torch.zeros(1, dtype=torch.int32, device=device)
        self.sumsq = torch.zeros(max(1, self.members), dtype=torch.float64, device=device)  # one per member
        self.partials: Optional[Tensor] = None
        self.cond = None
        self._peer_halo: Optional[PeerHalo] = None
        self._peer_halo_ok = True
        self._halo_pushed = False  # the last update kernel already stored the boundary frames into the neighbours' mailboxes

    @property
    def n_frames(self) -> int:
        """Frames of the resident state: this rank's (with halos), or every member's."""
        return self.members * self.L if self.members else self.plan.n_local

    @property
    def n_windows(self) -> int:
        """Windows one score evaluation runs: this rank's, or every member's (members x (L - 2k))."""
        p = self.plan
        return self.members * p.n_win_global if self.members else p.win_hi - p.win_lo

    @property
    def own(self) -> tuple:
        """(first local frame, frames) this runtime updates: this rank's owned frames, or every member's."""
        p = self.plan
        return (0, self.n_frames) if self.members else (p.own_lo - p.frame_lo, p.own_n)

    # ------------------------------------------------------------------------------------------------ engine
    def refresh_engine(self) -> None:
        """(Re)binds the packed-weight engine; `ScoreUNet.engine` re-packs if the parameters changed since (full
        fingerprint: data pointers, autograd versions, and the explicit epoch raw-pointer optimisers bump)."""
        self._engine = self.sf.unet.engine(*self._engine_args, max_windows=self._engine_windows, vjp=False,
                                           tile_windows=self._tile_windows)
        if self.exact and self.cond is not None:  # sized by the selection, so only once the operator is known
            nsel = max(1, len(self._selected_list()))
            self._engine_vjp = self.sf.unet.engine(*self._engine_args, max_windows=min(nsel, self._engine_windows), vjp=True)
        self._engine_epoch = getattr(self.sf.unet, "_weights_epoch", 0)

    @property
    def engine(self):
        if getattr(self.sf.unet, "_weights_epoch", 0) != self._engine_epoch:  # optimiser / EMA step since the last call
            self.refresh_engine()
        return self._engine

    @property
    def engine_vjp(self):
        _ = self.engine
        return self._engine_vjp

    def engines(self):
        """Every engine a score evaluation launches kernels on (bench.py's per-launch timing)."""
        return [e for e in (self.engine, self._engine_vjp) if e is not None]

    # ------------------------------------------------------------------------------------------------ exact_grad
    def _selected_list(self):
        """Global indices of this rank's windows whose OUTPUT carries a non-zero cotangent (see `observed_windows`)."""
        p = self.plan
        op = self.cond["op"]
        if isinstance(op, GenericObservation):  # an arbitrary A may read any frame: every window
            return list(range(p.win_lo, p.win_hi))
        if isinstance(op, CombinedObservation):
            obs = op.observed_frames(self.L, self.C)
        else:
            obs = op.observed_frames(self.C) if isinstance(op, PointObservation) else op.t_step
        return observed_windows(p.win_lo, p.win_hi, p.n_win_global, self.L, self.sf.markov_order, obs)

    def _selection(self):
        """(chunks of (win_list_dev, pos_dev), n_selected) for the current conditioning, cached."""
        if self._sel is None:
            sel = self._selected_list()
            step = max(1, self.engine_vjp.max_windows)
            chunks = []
            for i in range(0, len(sel), step):
                part = sel[i:i + step]
                pos = torch.full((self.plan.n_win_global,), -1, dtype=torch.int32)
                pos[torch.tensor(part, dtype=torch.long)] = torch.arange(len(part), dtype=torch.int32)
                chunks.append((torch.tensor(part, dtype=torch.int32, device=self.device), pos.to(self.device)))
            chosen = set(sel)
            rest = [j for j in range(self.plan.win_lo, self.plan.win_hi) if j not in chosen]
            self._rest = torch.tensor(rest, dtype=torch.int32, device=self.device)
            self._sel = (chunks, len(sel))
        return self._sel

    @property
    def n_selected(self) -> int:
        return self._selection()[1] if (self.exact and self.cond is not None) else 0

    @property
    def n_repeated(self) -> int:
        """Windows whose forward runs twice per score evaluation (selection larger than one stashing chunk)."""
        if not (self.exact and self.cond is not None):
            return 0
        chunks, n = self._selection()
        return 0 if len(chunks) == 1 else n

    # ------------------------------------------------------------------------------------------------ state io
    @property
    def stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def load(self, x_nchw: Tensor) -> None:
        """x_nchw: the FULL trajectory [L, C, H, W] (any device); keeps this rank's frames (with halos).  An ensemble:
        every member, [members, L, C, H, W]."""
        p = self.plan
        src = x_nchw.reshape(self.n_frames, self.C, self.H, self.W) if self.members else x_nchw[p.frame_lo:p.frame_hi]
        src = src.to(device=self.device, dtype=torch.float32, non_blocking=True).contiguous()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.c2w_traj_pack(src.data_ptr(), self.x.data_ptr(), self.n_frames, self.C, self.H * self.W,
                                              self.stream), "c2w_traj_pack")

    def unpack(self, buf: Tensor, lo: int, n: int) -> Tensor:
        out = torch.empty(n, self.C, self.H, self.W, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.c2w_traj_unpack(buf[lo:lo + n].data_ptr(), out.data_ptr(), n, self.C, self.H * self.W,
                                                self.stream), "c2w_traj_unpack")
        return out

    def owned(self, buf: Tensor) -> Tensor:
        """NCHW copy of this rank's owned frames of `buf` (an ensemble: every member's, [members * L, C, H, W])."""
        return self.unpack(buf, *self.own)

    # ------------------------------------------------------------------------------------------------ kernels
    def score(self, t: float, group=None) -> None:
        """eps <- composed window score of x at time t (src/thor/score.py:90-93 / :156-185).  With exact_grad the
        likelihood cotangent is pushed back through the same windows chunk by chunk: vjp <- J_eps^T g."""
        p = self.plan
        self._grad_ready = False
        if self.members:  # every member's windows, chunked by the workspace: a launch may hold several members'
            self.engine.window_score_members(self.x, self.members, self.L, 0, self.n_windows, t, self.eps)
            return
        if not (self.exact and self.cond is not None):
            self.engine.window_score(self.x, p.frame_lo, p.win_lo, p.win_hi - p.win_lo, p.n_win_global, t, self.eps)
            return
        mu, sigma = _mu_sigma(self.sf.noise_process, t)
        # J_eps^T g: only windows whose output meets an observed frame have a non-zero cotangent -> stashing forward +
        # input-gradient pass for that selection (~1/t_step of the windows)
        chunks, _ = self._selection()
        ev = self.engine_vjp
        if len(chunks) == 1:
            # the selection fits one stashing chunk: its forward also IS its part of the score, the other windows run
            # on the plain engine, both fold into eps by window list — no window is evaluated twice
            win_list, pos = chunks[0]
            if self._rest.numel():
                self.engine.window_score_sel(self.x, p.frame_lo, self._rest, t, p.n_win_global, self.eps)
            ev.window_score_sel(self.x, p.frame_lo, win_list, t, p.n_win_global, self.eps)
            # likelihood cotangent g = A^T((y - A x0)/var) on the owned frames (zero on unobserved frames)
            self._guide(2, mu, sigma, 0.0, 0.0)
            self.vjp.zero_()
            ev.window_score_backward_sel(self.cot, p.frame_lo, win_list, pos, p.n_win_global, self.vjp)
        else:
            # several stashing chunks (or none): the cotangent needs the whole score first, so every window runs on the
            # plain engine and each chunk of the selection repeats its forward, stashing, right before its backward
            self.engine.window_score(self.x, p.frame_lo, p.win_lo, p.win_hi - p.win_lo, p.n_win_global, t, self.eps)
            self._guide(2, mu, sigma, 0.0, 0.0)
            self.vjp.zero_()
            for win_list, pos in chunks:
                ev.window_score_sel(self.x, p.frame_lo, win_list, t)
                ev.window_score_backward_sel(self.cot, p.frame_lo, win_list, pos, p.n_win_global, self.vjp)
        exchange_halos_adjoint(self.vjp, p, group)

    def set_condition(self, cond) -> None:
        """One conditioning (condition_for), None, or for a batch of independent problems (members > 0) a list of
        every member's own conditioning."""
        self.batch = None
        if isinstance(cond, list):
            self._set_batch_condition(cond)
            return
        self.cond = cond
        self._sel = None
        self.points = None
        self.generic = None
        self._grad_ready = False
        if cond is not None and isinstance(cond["op"], GenericObservation):
            ops = self._generic_operands(cond)
            self.generic = [ops] * max(1, self.members)  # an ensemble: every member on the same observation
            if self.exact:
                self.refresh_engine()  # the stashing workspace is sized by the selection
            return
        # a std per observation (cond["obs_std"]): the coarse std^2 block next to y_dev, the point std in the plan
        obs_std = cond.get("obs_std") if cond is not None else None
        if cond is not None and isinstance(cond["op"], (PointObservation, CombinedObservation)):
            # this rank's owned frames only, built once per conditioning and trajectory geometry
            p = self.plan
            op, y, strip, max_pix = cond["op"], cond["y"], point_strip_rows(self.H, self.W), POINT_STRIP_PIX
            if isinstance(op, CombinedObservation):  # strips of whole observation tiles (guided_combined_kernel)
                op, y, max_pix = op.points, cond["point_y"], COMBINED_STRIP_PIX
                strip = combined_strip_rows(self.H, self.W, cond["op"].coarse.s_step)
            std = obs_std["point_std"] if obs_std is not None else None
            pl = point_plan(op, y, self.L, self.C, self.H, self.W, p.own_lo, p.own_lo + p.own_n, strip, max_pix, std,
                            members=cond.get("members", 0))
            self.points = _upload_point_plan(pl, std is not None, self.device, self.C)
        if cond is not None and self.exact:
            self.refresh_engine()  # the stashing workspace is sized by the selection
        if cond is not None and not isinstance(cond["op"], PointObservation):
            self.y_dev = cond["y"].to(device=self.device, dtype=torch.float32).contiguous()
        self.coarse_std2_dev = None
        if obs_std is not None and obs_std["coarse_std2"] is not None:
            self.coarse_std2_dev = obs_std["coarse_std2"].to(device=self.device, dtype=torch.float32).contiguous()

    def _set_batch_condition(self, conds: list) -> None:
        """A batch of independent problems: member m conditioned on conds[m] (condition_for of its own score function,
        one family, one coarse (t, s)).  Stacks the coarse blocks, concatenates the point plans and keeps the [M, C]
        gamma / std^2 arrays on the host (batch_condition), for c2w_guided_step_batch."""
        if not self.members or len(conds) != self.members:
            raise ValueError(f"a batch conditioning needs one conditioning per member ({self.members}), got {len(conds)}")
        self.generic, self._grad_ready = None, False
        if isinstance(conds[0]["op"], GenericObservation):  # one family: every member's own A, y, std and gamma
            ops = []
            for m, c in enumerate(conds):
                try:
                    ops.append(self._generic_operands(c))
                except (ValueError, RuntimeError, TypeError) as e:
                    raise type(e)(f"sample_batch: member {m}: {e}") from e
            self.cond, self._sel, self.points, self.generic = conds, None, None, ops
            return
        b = batch_condition(conds, (self.L, self.C, self.H, self.W))
        self.cond, self._sel = conds, None
        f32 = lambda a: None if a is None else \
            torch.as_tensor(a).to(device=self.device, dtype=torch.float32).contiguous()
        self.y_dev, self.coarse_std2_dev = f32(b["y"]), f32(b["coarse_std2"])
        self.points = _upload_point_plan(b["plan"], b["per_obs"], self.device, self.C) if b["plan"] is not None else None
        op0 = conds[0]["op"]
        cg = op0.coarse if isinstance(op0, CombinedObservation) else op0 if isinstance(op0, CoarseGrain) else None
        host = lambda a: None if a is None else (ctypes.c_float * a.size)(*a.reshape(-1).tolist())  # [M, C] fp32
        self.batch = dict(kind=b["kind"], per_obs=b["per_obs"], gamma=host(b["gamma"]), std2=host(b["std2"]),
                          point_std2=host(b["point_std2"]), t_step=cg.t_step if cg else 1,
                          s_step=cg.s_step if cg else None)

    def _generic_operands(self, cond: dict) -> dict:
        """generic_operands of a GenericObservation conditioning, A evaluated once on an [L, C, H, W] fp32 tensor of the
        compute device."""
        with torch.cuda.device(self.device), torch.inference_mode(False):
            probe = torch.zeros(self.L, self.C, self.H, self.W, dtype=torch.float32, device=self.device)
            return generic_operands(cond["op"].A, cond["y"], cond["std"], cond["gamma"], probe)

    def _generic_grad(self, mu: float, sigma: float) -> Tensor:
        """The generic path's likelihood cotangent g = A^T((y - A x0)/var) of the updated frames, fp32 NCHW, once per
        score evaluation: x0 by c2w_x0_nchw, then A and its VJP in torch on every member's [L, C, H, W] slice, gathered
        member-major.  var = std^2 + gamma (sigma/mu)^2 with sigma/mu rounded to fp32, as the reference computes it from
        fp32 schedule tensors.  Everything runs on the runtime's stream, without a host synchronisation."""
        if self._grad_ready:
            return self._grad
        lo, n = self.own
        with torch.cuda.device(self.device), _generic_autograd():
            if self._x0 is None:  # outside inference mode: A's backward may save it
                self._x0 = torch.empty(n, self.C, self.H, self.W, dtype=torch.float32, device=self.device)
                self._grad = torch.empty_like(self._x0)
            frame = self.H * self.W * self.C
            _lib.check(self.lib.c2w_x0_nchw(self.x.data_ptr() + 4 * lo * frame, self.eps.data_ptr() + 4 * lo * frame,
                                            mu, sigma, self._x0.data_ptr(), n, self.C, self.H * self.W, self.stream),
                       "c2w_x0_nchw")
            r2 = float((torch.tensor(sigma, dtype=torch.float32) / torch.tensor(mu, dtype=torch.float32)) ** 2)
            for m, ops in enumerate(self.generic):
                part = slice(m * self.L, (m + 1) * self.L) if self.members else slice(0, n)
                ax, pullback = torch.func.vjp(ops["A"], self._x0[part])
                (g,) = pullback((ops["y"] - ax) / (ops["std2"] + ops["gamma"] * r2))
                self._grad[part].copy_(g)
        self._grad_ready = True
        return self._grad

    def _guide(self, mode: int, mu: float, sigma: float, mu_next: float, sigma_next: float, frames=None) -> None:
        p = self.plan
        g = _lib.Guide()
        g.x, g.eps = self.x.data_ptr(), self.eps.data_ptr()
        s = self.s_tile
        pts = self.points if self.cond is not None else None
        bt = self.batch
        gen = self.generic
        if gen is not None and frames is not None:
            raise NotImplementedError("the generic observation path updates every owned frame at once")
        if gen is not None:
            combined = per_obs = False
        elif bt is not None:
            combined, per_obs = bt["kind"] == "combined", bt["per_obs"]
        else:
            combined = pts is not None and isinstance(self.cond["op"], CombinedObservation)
            per_obs = self.cond is not None and self.cond.get("obs_std") is not None  # g.std2 is not read
        if gen is not None:  # g is computed in torch (_generic_grad): y, std2, gamma, t_step and s_step are not read
            g.y, g.t_step = None, 1
        elif bt is not None:  # a batch: every member's y block, std^2 and gamma come from the batch's arrays
            g.y = self.y_dev.data_ptr() if self.y_dev is not None else None
            g.t_step = bt["t_step"]
            s = bt["s_step"] or s
        elif pts is not None and not combined:  # point observations: y, t_step and s_step are not read
            g.y, g.t_step = None, 1
            for i in range(self.C):
                g.std2[i] = 1.0 if per_obs else self.cond["std"][i] ** 2
                g.gamma[i] = self.cond["gamma"][i]
        elif self.cond is not None:  # the coarse term (of a CombinedObservation: the point term is in pts)
            cg: CoarseGrain = self.cond["op"].coarse if combined else self.cond["op"]
            s = cg.s_step
            g.y = self.y_dev.data_ptr()
            g.t_step = cg.t_step
            for i in range(self.C):
                g.std2[i] = 1.0 if per_obs else self.cond["std"][i] ** 2
                g.gamma[i] = self.cond["gamma"][i]
        else:
            g.y = None
            g.t_step = 1
        g.s_step, g.H, g.W = s, self.H, self.W
        g.mu, g.sigma, g.mu_next, g.sigma_next = mu, sigma, mu_next, sigma_next
        g.frame_global0, (g.own_lo, g.own_n) = p.frame_lo, self.own
        if frames is not None:
            g.own_lo, g.own_n = frames
        g.mode = mode
        g.channels = self.C
        g.nan_flag = self.nan_flag.data_ptr()
        g.vjp = self.vjp.data_ptr() if (self.exact and self.cond is not None and mode != 2) else None
        g.cot_out = self.cot.data_ptr() if mode == 2 else None
        g.halo, g.halo_k = None, self.sf.markov_order
        if mode == 0 and frames is None and p.world > 1:  # predictor update of the owned frames: fuse the halo push
            ph = self._ensure_peer_halo()
            if ph is not None:
                g.halo = ph.handle
                self._halo_pushed = True
        if mode == 1:
            strips = -(-self.H // point_strip_rows(self.H, self.W)) if gen is not None else \
                pts["n_strips"] if pts is not None else self.H // s
            n_part = g.own_n * strips
            if self.partials is None or self.partials.numel() < n_part:
                self.partials = torch.zeros(n_part, dtype=torch.float32, device=self.device)
            if self.eps_g is None:
                self.eps_g = torch.zeros_like(self.x)
            g.eps_out, g.partials = self.eps_g.data_ptr(), self.partials.data_ptr()
            self._n_part = n_part
        if gen is not None:
            grad = self._generic_grad(mu, sigma)
            with torch.cuda.device(self.device):
                if mode == 2:  # the cotangent fed to the UNet VJP is g itself, in the state layout
                    lo = g.own_lo * self.H * self.W * self.C
                    _lib.check(self.lib.c2w_traj_pack(grad.data_ptr(), self.cot.data_ptr() + 4 * lo, g.own_n, self.C,
                                                      self.H * self.W, self.stream), "c2w_traj_pack")
                else:
                    _lib.check(self.lib.c2w_guided_step_dense(ctypes.byref(g), grad.data_ptr(), self.stream),
                               "c2w_guided_step_dense")
            if mode == 0:  # x moved: the next g needs a new score evaluation
                self._grad_ready = False
            return
        with torch.cuda.device(self.device):
            if bt is not None:
                obs = ctypes.byref(pts["obs"]) if pts is not None else None
                entry = pts["tensors"]["std2"].data_ptr() if (per_obs and pts is not None) else None
                coarse = self.coarse_std2_dev.data_ptr() if self.coarse_std2_dev is not None else None
                _lib.check(self.lib.c2w_guided_step_batch(ctypes.byref(g), self.L, bt["gamma"], bt["std2"],
                                                          bt["point_std2"], obs, coarse, entry, self.stream),
                           "c2w_guided_step_batch")
            elif self.members:  # the same operands; the entry point observes every member's frames as one member's
                obs = ctypes.byref(pts["obs"]) if pts is not None else None
                pstd2 = (ctypes.c_float * self.C)(*(v ** 2 for v in self.cond["point_std"])) \
                    if (combined and not per_obs) else None
                entry = pts["tensors"]["std2"].data_ptr() if (per_obs and pts is not None) else None
                coarse = self.coarse_std2_dev.data_ptr() if (per_obs and self.coarse_std2_dev is not None) else None
                _lib.check(self.lib.c2w_guided_step_members(ctypes.byref(g), self.L, obs, pstd2, coarse, entry,
                                                            self.stream), "c2w_guided_step_members")
            elif per_obs:
                obs = ctypes.byref(pts["obs"]) if pts is not None else None
                entry = pts["tensors"]["std2"].data_ptr() if pts is not None else None
                coarse = self.coarse_std2_dev.data_ptr() if self.coarse_std2_dev is not None else None
                _lib.check(self.lib.c2w_guided_step_obs_std(ctypes.byref(g), obs, coarse, entry, self.stream),
                           "c2w_guided_step_obs_std")
            elif combined:
                pstd2 = (ctypes.c_float * self.C)(*(v ** 2 for v in self.cond["point_std"]))
                _lib.check(self.lib.c2w_guided_step_combined(ctypes.byref(g), ctypes.byref(pts["obs"]), pstd2, self.stream),
                           "c2w_guided_step_combined")
            elif pts is not None:
                _lib.check(self.lib.c2w_guided_step_points(ctypes.byref(g), ctypes.byref(pts["obs"]), self.stream),
                           "c2w_guided_step_points")
            else:
                _lib.check(self.lib.c2w_guided_step(ctypes.byref(g), self.stream), "c2w_guided_step")

    def predictor(self, mu: float, sigma: float, mu_next: float, sigma_next: float) -> None:
        """x <- mu' (x - sigma eps_g)/mu + sigma' eps_g on the owned frames (src/thor/pipelines.py:41-46)."""
        self._guide(0, mu, sigma, mu_next, sigma_next)

    def predictor_with_hook(self, mu: float, sigma: float, mu_next: float, sigma_next: float, proc_x0) -> None:
        """The predictor with a user `proc_x0` callable (src/thor/pipelines.py:43-45).  The fused update is split around
        the hook: the guided score comes from the kernel (mode 1); x0 = (x - sigma eps)/mu is handed to the callable as
        an NCHW device tensor and `mu' proc(x0) + sigma' eps` written back — elementwise torch ops on the resident
        tensors, because the hook itself is an arbitrary torch callable (no shipped config passes one).  An ensemble
        calls the hook once per member, on that member's [L, C, H, W], as a run of that member alone would."""
        self._guide(1, mu, sigma, 0.0, 0.0)
        lo, n = self.own
        parts = [(m * self.L, self.L) for m in range(self.members)] if self.members else [(lo, n)]
        for lo, n in parts:  # (first frame, frames) of each member, or of this rank's owned frames
            x_own, e_own = self.x[lo:lo + n], self.eps_g[lo:lo + n]
            x0 = proc_x0(((x_own - sigma * e_own) / mu).permute(0, 3, 1, 2))
            if tuple(x0.shape) != (n, self.C, self.H, self.W):
                raise ValueError(f"proc_x0 returned shape {tuple(x0.shape)}")
            x_own.copy_(mu_next * x0.permute(0, 2, 3, 1) + sigma_next * e_own)
            self.nan_flag |= (~torch.isfinite(x_own)).any().to(torch.int32)

    def guided_eps(self, mu: float, sigma: float) -> None:
        """eps_g <- eps - sigma * grad_x log p(y | x) (src/thor/score.py:24-35) and the partial sums of eps_g^2."""
        self._guide(1, mu, sigma, 0.0, 0.0)

    def corrector(self, tau: float, sigma_next: float, z: Optional[Tensor], seed, step_id: int,
                  group=None) -> None:
        """One Langevin correction with eps_g already computed (src/thor/pipelines.py:81-88).  An ensemble: `seed` is
        the members' seeds (int64 device tensor, `member_seeds`), each member has its own mean(eps^2) and noise."""
        p = self.plan
        hw = self.H * self.W
        if self.members:
            with torch.cuda.device(self.device):
                _lib.check(self.lib.c2w_reduce_partials_members(self.partials.data_ptr(), self.members,
                                                                self._n_part // self.members, self.sumsq.data_ptr(),
                                                                self.stream), "c2w_reduce_partials_members")
                _lib.check(self.lib.c2w_corrector_update_members(
                    self.x.data_ptr(), self.eps_g.data_ptr(), self.sumsq.data_ptr(), float(self.L * self.C * hw),
                    float(tau), float(sigma_next), self.members, self.L * hw, self.C, seed.data_ptr(), int(step_id),
                    self.nan_flag.data_ptr(), self.stream), "c2w_corrector_update_members")
            return
        with torch.cuda.device(self.device):
            _lib.check(self.lib.c2w_reduce_partials(self.partials.data_ptr(), self._n_part, self.sumsq.data_ptr(),
                                                    self.stream), "c2w_reduce_partials")
            if p.world > 1:
                dist.all_reduce(self.sumsq, group=group)  # trajectory-global mean(eps^2): one scalar per correction
            lo = p.own_lo - p.frame_lo
            zp = None
            if z is not None:
                zl = z[lo:lo + p.own_n]
                assert zl.is_contiguous()
                zp = zl.data_ptr()
            _lib.check(self.lib.c2w_corrector_update_c(
                self.x[lo:].data_ptr(), self.eps_g[lo:].data_ptr(), zp, self.sumsq.data_ptr(),
                float(self.L * self.C * hw), float(tau), float(sigma_next), p.own_lo * hw, p.own_n * hw, self.C, int(seed),
                int(step_id), self.nan_flag.data_ptr(), self.stream), "c2w_corrector_update_c")

    def member_seeds(self, seeds: Sequence[int]) -> Tensor:
        """The members' corrector seeds as the device array c2w_corrector_update_members reads: each taken modulo 2^64,
        as the single-trajectory call takes its uint64 seed."""
        u = np.array([int(s) & 0xFFFF_FFFF_FFFF_FFFF for s in seeds], dtype=np.uint64).view(np.int64)
        return torch.from_numpy(u).to(self.device)

    def _ensure_peer_halo(self) -> Optional[PeerHalo]:
        """The peer-memory mailboxes (set up collectively on first use by every rank at the same point)."""
        if self.plan.world == 1:
            return None
        if self.C != 4:  # the mailboxes and the fused push move one float4 per pixel
            return None
        if self._peer_halo is None and self._peer_halo_ok and halo_transport() != "nccl":
            group = self.sf.shard[2] if self.sf.shard else None
            try:
                self._peer_halo = PeerHalo(self.plan, self.x.shape[1:], self.device, group)
            except _lib.C2WError as e:  # no peer access between neighbours: say so once, use NCCL
                print(f"climate2weather_b200: peer-memory halo exchange unavailable ({e}); using NCCL send/recv")
                self._peer_halo_ok = False
        return self._peer_halo

    def halo(self, group=None) -> None:
        """Refresh the k halo frames of x from the neighbours (after every state update).  Over NVLink peer memory when
        the ranks' GPUs can map each other — the push half already happened inside the predictor kernel when that was
        the update (c2w_guided_step with g.halo), so only the pull remains; after a corrector update both halves run
        (c2w_halo_exchange).  torch.distributed send/recv pairs otherwise."""
        if self.plan.world == 1:
            return
        ph = self._ensure_peer_halo()
        if ph is None:
            exchange_halos(self.x, self.plan, group)
        elif self._halo_pushed:
            ph.pull(self.x)
        else:
            ph.exchange(self.x)
        self._halo_pushed = False

    def check_finite(self) -> None:
        if int(self.nan_flag.item()) != 0:
            raise ValueError("NaN detected in sample")  # same error as src/thor/pipelines.py:90-91

    def reset_finite_check(self) -> None:
        self.nan_flag.zero_()
        self._flag_n = 0

    def check_finite_lagged(self) -> None:
        """Per-step NaN check without stalling the launch queue: the flag is copied to pinned host memory every step
        (asynchronously, with an event) and the copy made ONE step earlier is inspected — by then it has long
        completed, so the host never waits for the step it has just enqueued.  A NaN raises the same error one step
        later than `check_finite()` would; the last step is covered by the final `check_finite()`."""
        if getattr(self, "_flag_host", None) is None:
            self._flag_host = [torch.zeros(1, dtype=self.nan_flag.dtype).pin_memory() for _ in range(2)]
            self._flag_event = [torch.cuda.Event() for _ in range(2)]
            self._flag_n = 0
        i = self._flag_n & 1
        if self._flag_n >= 1:
            j = (self._flag_n - 1) & 1
            self._flag_event[j].synchronize()
            if int(self._flag_host[j][0]) != 0:
                raise ValueError("NaN detected in sample")
        with torch.cuda.device(self.device):
            self._flag_host[i].copy_(self.nan_flag.reshape(-1)[:1], non_blocking=True)
            self._flag_event[i].record(torch.cuda.current_stream(self.device))
        self._flag_n += 1


class AbstractScoreFunction:
    """src/thor/score.py:7-60."""

    #: windows per UNet launch; None = the subclass default.  Results do not depend on it.
    max_windows: Optional[int] = None

    def __init__(self, unet, noise_process, unet_kwargs=None):
        if not isinstance(unet, ScoreUNet):
            # a reference `model.score.ScoreUNet` (e.g. snapshot["ema"]): take its architecture and weights
            unet = build_from_reference(unet)
        self.unet = unet
        self.noise_process = noise_process
        self.unet_kwargs = unet_kwargs if unet_kwargs is not None else {}
        self.likelihood = None
        self.device: Optional[torch.device] = None
        self.shard = None  # (rank, world, group) once enable_time_sharding() was called
        self.shard_gather = 0  # rank that receives the sampled trajectory ("all": every rank)
        self._runtimes = {}
        self.unet.eval()

    # ------------------------------------------------------------------------------------------------ reference API
    @property
    def is_conditioned(self):
        return self.likelihood is not None

    def net_forward(self, x: Tensor, t: Tensor) -> Tensor:
        return self.unet(x, t)

    def condition_on(self, *, A, y, std, gamma=1e-2, exact_grad=True):
        """src/thor/score.py:44-60.  `exact_grad=False` (every shipped config) is the closed-form guidance
        J = A^T((y - A x0)/var)/mu; `exact_grad=True` adds the term through the network,
        J = (g - sigma J_eps^T g)/mu with g = A^T((y - A x0)/var), computed by the UNet input-gradient kernels."""
        if isinstance(A, PointObservation):
            yt = torch.as_tensor(y)
            A.check_observation(yt)
            _std_per_observation(std, yt.shape, yt.shape[1], A.mask_for(yt.shape[1]), repr(A))
        if isinstance(A, CombinedObservation) and torch.as_tensor(y).dim() != 1:
            raise ValueError(f"{A}: y must be the flat tensor A(x) gives (CombinedObservation.pack), got shape "
                             f"{tuple(torch.as_tensor(y).shape)}")
        if self.likelihood is not None:
            print("Warning: Overwriting old conditioning")
        self.likelihood = dict(A=A, y=torch.as_tensor(y), std=std, gamma=gamma, op=None, exact=bool(exact_grad))
        for rt in self._runtimes.values():
            rt.set_condition(None)
        self._runtimes.clear()
        return self

    def __call__(self, x: Tensor, t: Tensor) -> Tensor:
        """src/thor/score.py:24-35: the (guided) noise prediction for the whole trajectory x[L, C, H, W]."""
        rt = self.runtime(x)
        rt.load(x)
        rt.score(float(t), self.shard[2] if self.shard else None)
        if not self.is_conditioned:
            out = rt.owned(rt.eps)
        else:
            mu, sigma = _mu_sigma(self.noise_process, t)
            rt.guided_eps(mu, sigma)
            out = rt.owned(rt.eps_g)
        return out.to(device=x.device, dtype=x.dtype)

    def score_fn(self, x: Tensor, t: Tensor) -> Tensor:
        """Unguided composed score (src/thor/score.py:90-93, :156-185)."""
        rt = self.runtime(x)
        rt.load(x)
        rt.score(float(t))
        return rt.owned(rt.eps).to(device=x.device, dtype=x.dtype)

    # ------------------------------------------------------------------------------------------------ runtime
    def enable_time_sharding(self, group=None, gather=0) -> "AbstractScoreFunction":
        """Partition trajectories along time over the ranks of `group` (default: the world group).  `gather`: the
        group rank on which `SDAPipeline.sample` assembles the result (the other ranks return None), or "all"."""
        if not dist.is_initialized():
            raise RuntimeError("torch.distributed is not initialised")
        self.shard = (dist.get_rank(group), dist.get_world_size(group), group)
        self.shard_gather = gather
        self._runtimes.clear()
        return self

    def _compute_device(self, x: Tensor) -> torch.device:
        if x.is_cuda:
            return x.device
        if self.device is not None and torch.device(self.device).type == "cuda":
            return torch.device(self.device)
        p = next(self.unet.parameters())
        if p.is_cuda:
            return p.device
        if torch.cuda.is_available():
            return torch.device("cuda", torch.cuda.current_device())
        raise _lib.C2WError("no CUDA device: climate2weather_b200 has no CPU path")

    #: Windows per UNet launch when nothing else is specified.  One launch over all windows of a one-week trajectory
    #: (156) keeps every level of the UNet at full machine occupancy: measured 20.9 ms/step vs 24.9 ms at 32 windows
    #: (profiles/r01_chunk_sweep.log).  The workspace is ~24 MiB per window.
    DEFAULT_WINDOWS = 192
    #: windows per forward+backward chunk with exact_grad=True
    VJP_WINDOWS = 192

    def _default_windows(self, n_win: int) -> int:
        return min(n_win, self.DEFAULT_WINDOWS)

    def runtime(self, x: Tensor, members: int = 0) -> _Runtime:
        """The device state for a trajectory x [L, C, H, W], or with members = M an ensemble x [M, L, C, H, W] (closed-
        form guidance only, not time-sharded; one plan over M L frames and M (L - 2k) windows)."""
        shape = tuple(x.shape[1:]) if members else tuple(x.shape)
        L, C, H, W = shape
        exact = bool(self.likelihood is not None and self.likelihood.get("exact"))
        if members and exact:
            raise NotImplementedError("ensemble sampling runs closed-form guidance only: condition_on(..., "
                                      "exact_grad=False); exact_grad=True needs member-aware window selection and "
                                      "adjoints, which are not implemented")
        if members and self.shard:
            raise NotImplementedError("ensemble sampling does not run on a time-sharded score function "
                                      "(enable_time_sharding); run one ensemble per rank instead")
        if self.shard and self.likelihood is not None and \
                isinstance(_operator_for(self.likelihood, L, C, H, W), GenericObservation):
            raise NotImplementedError(f"the generic observation path (A = {self.likelihood['A']!r}, an operator the "
                                      f"fused guidance kernels do not implement) does not run on a time-sharded score "
                                      f"function (enable_time_sharding): A sees the whole trajectory")
        dev = self._compute_device(x)
        rank, world = (self.shard[0], self.shard[1]) if self.shard else (0, 1)
        key = (L, C, H, W, str(dev), rank, world, exact, members)
        rt = self._runtimes.get(key)
        if rt is None:
            plan = make_plan(L, self.markov_order, rank, world)
            n_win = members * plan.n_win_global if members else plan.win_hi - plan.win_lo
            mw = self.max_windows or self._default_windows(n_win)
            if exact:
                mw = min(mw, self.VJP_WINDOWS)  # the stash costs ~110 MiB per window at the reference shapes
            args = (self, L, C, H, W, dev, plan, mw)
            rt = _Runtime(*args, exact=exact, members=members) if members else _Runtime(*args, exact=exact)
            if self.likelihood is not None:
                rt.set_condition(condition_for(self.likelihood, shape, members))
            self._runtimes = {key: rt}  # one live trajectory geometry at a time
        else:
            rt.refresh_engine()  # once per score call / sampling run: catches in-place parameter updates
        return rt


def condition_for(lk: dict, shape, members: int = 0) -> dict:
    """The conditioning of a trajectory of shape (L, C, H, W) from a score function's `likelihood` (condition_on): the
    operator recognised (cached in lk) and checked against the geometry, y in the form the guidance kernels read (a
    CombinedObservation's split into its terms), gamma and std per variable, or a std per observation ("obs_std").
    members = M: an ensemble's, whose point plan repeats its frame slots per member."""
    L, C, H, W = (int(v) for v in shape)
    op, y = _operator_for(lk, L, C, H, W), lk["y"]
    if isinstance(op, GenericObservation):  # y, std and gamma as given, checked against A(x) at runtime set-up
        return dict(op=op, y=y, std=lk["std"], gamma=lk["gamma"])
    cond = dict(op=op, gamma=lk["gamma_c"])
    if members:  # the point plan repeats its frame slots per member
        cond["members"] = members
    if isinstance(op, CombinedObservation):  # split and checked against this trajectory's geometry
        _check_observation_shape(op.coarse, op.term_shapes(shape)[0], L, C, H, W)
        y, cond["point_y"] = op.split(y, shape)
        if torch.as_tensor(lk["std"]).numel() in (1, C):
            cond["std"], cond["point_std"] = op.std_per_term(lk["std"], shape)
        else:
            cond.update(_combined_std(op, lk["std"], shape))
    else:
        if isinstance(op, CoarseGrain):  # checked against this trajectory's geometry, every time
            y = coarse_grain_observation(op, y, L, C, H, W)
        cond.update(_single_std(op, lk["std"], y.shape, C))
    return dict(cond, y=y)


def _operator_for(lk: dict, L: int, C: int, H: int, W: int):
    """The operator record of a score function's `likelihood` (`_route_operator`), cached in lk with the per-variable
    gamma of the fused operators."""
    if lk["op"] is None:
        # geometry checks run in point_plan (set_condition) and, for the coarse term, in condition_for
        lk["op"] = _route_operator(lk["A"], L, C, H, W, lk["y"].shape)
        if not isinstance(lk["op"], GenericObservation):
            lk["gamma_c"] = _per_channel(lk["gamma"], C, "gamma")
    return lk["op"]


def _single_std(op, std, obs_shape, C: int) -> dict:
    """The std entries of a CoarseGrain's or PointObservation's conditioning: per variable ({"std": C values}) when
    std is a scalar, C values or constant per variable, else per observation ({"obs_std": coarse std^2 block or
    point std, the other None})."""
    mask = op.mask_for(C) if isinstance(op, PointObservation) else None
    b = _std_per_observation(std, obs_shape, C, mask, repr(op))
    if b is None:
        return {"std": _per_channel(std, C, "std")}
    v = _collapse_per_variable(b, mask)
    if v is not None:
        return {"std": v}
    if mask is not None:
        return {"obs_std": dict(coarse_std2=None, point_std=b)}
    return {"obs_std": dict(coarse_std2=b * b, point_std=None)}


def _combined_std(op: CombinedObservation, std, x_shape) -> dict:
    """The std entries of a CombinedObservation's conditioning from a flat std in y's layout: per (term, variable)
    ({"std", "point_std"}) when each term's block is constant per variable, else per observation ({"obs_std"})."""
    coarse_std2, point_std = op.std_per_observation(std, x_shape)
    mask = op.points.mask_for(int(x_shape[1]))
    coarse = op.split(torch.as_tensor(std, dtype=torch.float32).reshape(-1).cpu(), x_shape)[0]
    cv, pv = _collapse_per_variable(coarse, None), _collapse_per_variable(point_std, mask)
    if cv is not None and pv is not None:
        return {"std": cv, "point_std": pv}
    return {"obs_std": dict(coarse_std2=coarse_std2, point_std=point_std)}


def _mu_sigma(noise_process, t) -> tuple:
    tt = torch.as_tensor(t, dtype=torch.float32).cpu()
    return float(noise_process.mu(tt)), float(noise_process.sigma(tt))


def _window_view(x: Tensor, w: int) -> Tensor:
    """[L, C, H, W] -> [L-w+1, w*C, H, W] with U[j, tau*C + c] = x[j + tau, c]: the zero-copy strided view the
    reference builds with unfold/movedim/flatten (src/thor/score.py:68-74, :143-152).  Layout helper only — the
    sampling path never materialises it (K0 gathers windows straight from the resident trajectory)."""
    L, C, H, W = x.shape
    if L < w:
        raise ValueError(f"trajectory of {L} frames is shorter than one window of {w}")
    x = x.contiguous()
    sL, sC, sH, sW = x.stride()
    return x.as_strided((L - w + 1, w * C, H, W), (sL, sC, sH, sW))  # channel tau*C + c sits tau*sL + c*sC == (tau*C + c)*sC


def _pick_slots(n: Tensor, k: int, head: bool, tail: bool) -> Tensor:
    """Centre-pick / edge-fill of a window batch n[B, w*C, H, W] (src/thor/score.py:76-88, :124-141): optional head
    slots 0..k-1 of the first window, the centre slot k of every window, optional tail slots k+1..2k of the last."""
    w = 2 * k + 1
    B = n.shape[0]
    v = n.reshape(B, w, n.shape[1] // w, *n.shape[2:])
    parts = []
    if head:
        parts.append(v[0, :k])
    parts.append(v[:, k])
    if tail:
        parts.append(v[B - 1, k + 1:])
    return torch.cat(parts, dim=0) if len(parts) > 1 else parts[0]


class DefaultScoreFunction(AbstractScoreFunction):
    """src/thor/score.py:63-93."""

    def __init__(self, unet, markov_order, **kwargs):
        super().__init__(unet=unet, **kwargs)
        self.markov_order = markov_order

    def unfold(self, x: Tensor) -> Tensor:
        """src/thor/score.py:68-74 (index map only; see `_window_view`)."""
        return _window_view(x, 2 * self.markov_order + 1)

    def fold(self, x: Tensor) -> Tensor:
        """src/thor/score.py:76-88 (index map only)."""
        return _pick_slots(x, self.markov_order, True, True)


class BatchedScoreFunction(AbstractScoreFunction):
    """src/thor/score.py:96-185.  `batch_size` windows go through the UNet per launch; `device` is where the
    trajectory is kept resident (the reference streams every batch host->device->host, :170-181)."""

    def __init__(self, unet, markov_order, batch_size=16, device=None, **kwargs):
        super().__init__(unet=unet, **kwargs)
        self.markov_order = markov_order
        self.batch_size = batch_size
        self.device = device if device is not None else torch.device("cuda")
        print(f">>> Initialized batched score function to use device: {self.device}")

    def _batch_noise(self, x: Tensor):
        """src/thor/score.py:143-154: the window view split into batches of `batch_size` (views, no copies)."""
        return _window_view(x, 2 * self.markov_order + 1).split(self.batch_size, 0)

    def _window_score(self, x: Tensor, t: Tensor, is_first: bool, is_last: bool) -> Tensor:
        """src/thor/score.py:111-141 for one explicit window batch x[B, w*C, H, W]: ScoreUNet forward on the device
        (c2w_unet_forward), then the slot selection.  `score_fn` / `__call__` do NOT go through this method — they run
        the fused gather -> UNet -> compose path on the resident trajectory."""
        dev = self._compute_device(x)
        out = self.net_forward(x.to(dev), t)
        return _pick_slots(out, self.markov_order, is_first, is_last)

    def _default_windows(self, n_win: int) -> int:
        # `batch_size` bounds device memory in the reference (src/thor/score.py:143-154); results do not depend on it.
        # Here it is a lower bound on the windows per launch: the resident workspace is small next to 180 GB of HBM.
        return min(n_win, max(int(self.batch_size), self.DEFAULT_WINDOWS))
