"""Host-side mirror of `thor.pipelines.SDAPipeline` (reference src/thor/pipelines.py:8-97): cosine VP schedule,
DSM loss, predictor-corrector sampler — same method names and signatures.

`sample()` with one of this package's score functions runs device-resident: the trajectory never leaves HBM
between steps, each step is  window score (K0/K1/K2/K4/K5)  ->  fused guidance + predictor (K6)  [-> corrector
(K7)]  [-> halo exchange when time-sharded].  The reference keeps x on the CPU and round-trips every window batch
(src/thor/score.py:170-181).
"""
from __future__ import annotations

import math
import time
from typing import Optional, Sequence

import torch
from torch import Tensor

from . import _lib
from .score import (AbstractScoreFunction, CoarseGrain, CombinedObservation, PointObservation, _mu_sigma, _Runtime,
                    condition_for)
from .sharding import all_gather_frames, gather_frames, make_plan


class SDAPipeline:
    #: corrector noise: "device" = on-chip Philox keyed by the global pixel index (default, sharding-invariant);
    #: "reference" = z.normal_() on a HOST tensor from the global CPU generator — what src/thor/pipelines.py:82 does when
    #: sample() runs on its default device (CPU, :59-60; the shipped driver calls it that way) — then uploaded (parity runs).
    rng: str = "device"
    #: read the device NaN flag every this many steps (0 = only at the end); the reference syncs every step (:90).
    #: The per-step read is asynchronous and inspected one check later, so a NaN raises one step after it appeared.
    nan_check_every: int = 0
    #: optional debugging / parity hook: sampler steps (1-based) after which the trajectory is copied out; the copies
    #: land in `self.traces[step]` (NCHW, host).  None = off (no copies, no synchronisation).
    trace_at = None

    def __init__(self, eta=1e-3):
        self.eta = eta  # src/thor/pipelines.py:9-11
        self.traces = {}

    # ---------------------------------------------------------------- schedule (src/thor/pipelines.py:13-20)
    def alpha(self, t):
        return torch.cos(math.acos(math.sqrt(self.eta)) * t) ** 2

    def mu(self, t):
        return self.alpha(t)

    def sigma(self, t):
        return (1 - self.alpha(t) ** 2 + self.eta ** 2).sqrt()

    # ---------------------------------------------------------------- training objective (:22-35)
    def forward(self, x, t):
        eps = torch.randn_like(x)
        # mu x + sigma eps in two passes over the batch instead of three (mul, then fused multiply-add)
        return torch.addcmul(self.mu(t) * x, self.sigma(t).expand_as(x), eps), eps

    def loss(self, net, x, forcing=None):
        t = torch.rand(x.shape[0], 1, 1, 1, dtype=x.dtype, device=x.device)
        xt, eps = self.forward(x, t)
        # (net(xt, t) - eps) ** 2, elementwise (:35), as ONE kernel forward and one backward
        return torch.nn.functional.mse_loss(net(xt, t, forcing=forcing), eps, reduction="none")

    def pred_eps(self, score_fn, x, t):
        return score_fn(x, t)

    def _sample_step(self, score_fn, x, t, dt, proc_x0=None):
        """:41-46, the reference's formula kept for API completeness (`sample` itself runs the fused kernels)."""
        eps_pred = self.pred_eps(score_fn, x, t)
        pred_x0 = (x - self.sigma(t) * eps_pred) / self.mu(t)
        if proc_x0 is not None:
            pred_x0 = proc_x0(pred_x0)
        return self.mu(t - dt) * pred_x0 + self.sigma(t - dt) * eps_pred

    # ---------------------------------------------------------------- sampler (:48-97)
    def sample(self, score_fn, noise, steps: int = 64, corrections: int = 0, tau: float = 1.0, proc_x0=None,
               device=None, show_progressbar=True, seed: Optional[int] = None):
        if not isinstance(score_fn, AbstractScoreFunction):
            raise TypeError("SDAPipeline.sample drives this package's score functions (Default/BatchedScoreFunction); "
                            f"got {type(score_fn).__name__}.  There is no generic torch-op sampling loop here.")
        return self._sample_resident(score_fn, noise, steps, corrections, tau, device, show_progressbar, seed, proc_x0)

    def sample_ensemble(self, score_fn, noise, steps: int = 64, corrections: int = 0, tau: float = 1.0, proc_x0=None,
                        device=None, show_progressbar=True, seeds: Optional[Sequence[int]] = None):
        """M members sampled together: noise [M, L, C, H, W] -> [M, L, C, H, W], every member conditioned on the score
        function's one `condition_on` (the reference's ensemble: the same observation, different noise).  The members
        share one device-resident state, so each UNet launch holds windows of several members.

        Member m is bit-identical to `sample(score_fn, noise[m], ..., seed=seeds[m])`, whatever `max_windows` is.
        `seeds`: M corrector seeds; by default M draws from the global generator in member order, as M sequential
        `sample` calls would make.  `proc_x0` is called once per member on its [L, C, H, W] x0; `trace_at` traces are
        [M, L, C, H, W].  Closed-form guidance only (exact_grad=False), not with time sharding, and not with
        `rng = "reference"` corrections."""
        if not isinstance(score_fn, AbstractScoreFunction):
            raise TypeError("SDAPipeline.sample_ensemble drives this package's score functions "
                            f"(Default/BatchedScoreFunction); got {type(score_fn).__name__}")
        if noise.dim() != 5:
            raise ValueError(f"sample_ensemble: noise must be [M, L, C, H, W], got shape {tuple(noise.shape)}")
        M = int(noise.shape[0])
        if M < 1:
            raise ValueError("sample_ensemble: noise holds no member (M = 0)")
        if seeds is not None:
            seeds = [int(v) for v in seeds]
            if len(seeds) != M:
                raise ValueError(f"sample_ensemble: {len(seeds)} seeds for {M} members (one per member)")
        if corrections > 0 and self.rng == "reference":
            raise NotImplementedError("sample_ensemble: rng='reference' with corrections draws z on the host from the "
                                      "global CPU generator, member after member; drawing it for all members step by "
                                      "step cannot reproduce that stream, so it is refused (use rng='device' or sample)")
        return self._sample_resident(score_fn, noise, steps, corrections, tau, device, show_progressbar, seeds, proc_x0,
                                     members=M)

    def sample_batch(self, score_fns, noise, steps: int = 64, corrections: int = 0, tau: float = 1.0, proc_x0=None,
                     device=None, show_progressbar=True, seeds: Optional[Sequence[int]] = None):
        """M independent problems sampled together: score_fns[m] (each conditioned by its own `condition_on`: its own
        y, std and gamma, for point terms its own stations, frames and mask) drives noise[m]; noise [M, L, C, H, W] ->
        [M, L, C, H, W].  The members share one device-resident state and one network, so each UNet launch holds
        windows of several members, as in `sample_ensemble`.

        Member m is bit-identical to `sample(score_fns[m], noise[m], ..., seed=seeds[m])`, whatever `max_windows` is
        (the same on every member).  `seeds`, `proc_x0`, `trace_at` and `nan_check_every` behave as in
        `sample_ensemble`, and `sample_batch([sf] * M, ...)` equals `sample_ensemble(sf, ...)`.  The members must share
        the ScoreUNet object, markov_order, the windows per launch, the operator family (all CoarseGrain, all
        PointObservation, all CombinedObservation, or all generic: each member then runs its own A, y, std and gamma
        through torch's VJP), the coarse term's (t_step, s_step), and whether they are
        conditioned at all; closed-form guidance only (exact_grad=False), not time-sharded, and not with
        `rng = "reference"` corrections.  A disagreement raises before any device work, naming the member."""
        score_fns = list(score_fns)
        for m, sf in enumerate(score_fns):
            if not isinstance(sf, AbstractScoreFunction):
                raise TypeError(f"sample_batch: member {m}: drives this package's score functions "
                                f"(Default/BatchedScoreFunction); got {type(sf).__name__}")
        if noise.dim() != 5:
            raise ValueError(f"sample_batch: noise must be [M, L, C, H, W], got shape {tuple(noise.shape)}")
        M = int(noise.shape[0])
        if M < 1:
            raise ValueError("sample_batch: noise holds no member (M = 0)")
        if len(score_fns) != M:
            raise ValueError(f"sample_batch: {len(score_fns)} score functions for {M} members (one per member)")
        if seeds is not None:
            seeds = [int(v) for v in seeds]
            if len(seeds) != M:
                raise ValueError(f"sample_batch: {len(seeds)} seeds for {M} members (one per member)")
        if corrections > 0 and self.rng == "reference":
            raise NotImplementedError("sample_batch: rng='reference' with corrections draws z on the host from the "
                                      "global CPU generator, member after member; drawing it for all members step by "
                                      "step cannot reproduce that stream, so it is refused (use rng='device' or sample)")
        if device is not None and torch.device(device).type == "cuda":
            for sf in score_fns:
                sf.device = torch.device(device)
        rt = self._batch_runtime(score_fns, noise)
        return self._sample_resident(score_fns[0], noise, steps, corrections, tau, device, show_progressbar, seeds,
                                     proc_x0, members=M, rt=rt)

    def _batch_runtime(self, score_fns: list, noise: Tensor) -> _Runtime:
        """The checks of sample_batch that need the members' score functions, then the batch's runtime: cached while the
        score functions, the geometry and every member's conditioning (its `likelihood` dict, by identity: condition_on
        replaces it) stay the same; a new conditioning of any member rebuilds the batch's conditioning only."""
        M = len(score_fns)
        shape = tuple(int(v) for v in noise.shape[1:])
        L = shape[0]
        sf0 = score_fns[0]
        k = sf0.markov_order
        nw = L - 2 * k

        def windows(sf):
            return min(sf.max_windows or sf._default_windows(nw), nw)

        for m, sf in enumerate(score_fns):
            lk = sf.likelihood
            if sf.unet is not sf0.unet:
                raise ValueError(f"sample_batch: member {m}: its ScoreUNet is not member 0's; the members share one "
                                 f"network (one engine)")
            if sf.markov_order != k:
                raise ValueError(f"sample_batch: member {m}: markov_order {sf.markov_order} differs from member 0's {k}")
            if windows(sf) != windows(sf0):
                raise ValueError(f"sample_batch: member {m}: {windows(sf)} windows per launch (max_windows or the class "
                                 f"default) differ from member 0's {windows(sf0)}; they decide each member's conv plan")
            if sf.shard:
                raise NotImplementedError(f"sample_batch: member {m}: a batch does not run on a time-sharded score "
                                          f"function (enable_time_sharding)")
            if lk is not None and lk.get("exact"):
                raise NotImplementedError(f"sample_batch: member {m}: a batch runs closed-form guidance only: "
                                          f"condition_on(..., exact_grad=False); exact_grad=True needs member-aware window "
                                          f"selection and adjoints, which are not implemented")
            if (lk is None) != (sf0.likelihood is None):
                state = lambda v: "unconditioned" if v is None else "conditioned"
                raise NotImplementedError(f"sample_batch: member {m}: {state(lk)} while member 0 is "
                                          f"{state(sf0.likelihood)}; the members are all conditioned or none")
        likes = tuple(sf.likelihood for sf in score_fns)
        ident = (tuple(id(sf) for sf in score_fns), shape)
        hit = getattr(self, "_batch_cache", None)
        same = hit is not None and hit[0][:2] == ident and all(a is b for a, b in zip(hit[1], likes))
        conds = None
        if sf0.likelihood is not None and not same:
            conds = []
            for m, lk in enumerate(likes):
                try:
                    conds.append(condition_for(lk, shape))
                except (ValueError, NotImplementedError) as e:
                    raise type(e)(f"sample_batch: member {m}: {e}") from None
            family = lambda op: type(op).__name__
            coarse = lambda op: op.coarse if isinstance(op, CombinedObservation) else op
            op0 = conds[0]["op"]
            for m, c in enumerate(conds):
                op = c["op"]
                if family(op) != family(op0):
                    raise NotImplementedError(f"sample_batch: member {m}: operator family {family(op)} differs from "
                                              f"member 0's {family(op0)}; a batch runs one guidance kernel")
                if isinstance(op, (CoarseGrain, CombinedObservation)) and \
                        (coarse(op).t_step, coarse(op).s_step) != (coarse(op0).t_step, coarse(op0).s_step):
                    raise NotImplementedError(f"sample_batch: member {m}: coarse (t_step, s_step) = "
                                              f"{(coarse(op).t_step, coarse(op).s_step)} differs from member 0's "
                                              f"{(coarse(op0).t_step, coarse(op0).s_step)}")
        dev = sf0._compute_device(noise)
        key = ident + (str(dev),)
        if same and hit[0] == key:
            hit[2].refresh_engine()  # catches in-place parameter updates, as AbstractScoreFunction.runtime does
            return hit[2]
        if sf0.likelihood is not None and conds is None:  # the same conditionings on another device
            conds = [condition_for(lk, shape) for lk in likes]
        rt = None
        if hit is not None and hit[0] == key:
            rt = hit[2]  # the same members and geometry: keep the runtime (and engine), rebuild the conditioning
            rt.refresh_engine()
        if rt is None:
            plan = make_plan(L, k, 0, 1)
            mw = sf0.max_windows or sf0._default_windows(M * plan.n_win_global)
            rt = _Runtime(sf0, *shape, dev, plan, mw, members=M)
        rt.set_condition(conds)
        self._batch_cache = (key, likes, rt, score_fns)  # the score functions stay alive: their ids stay theirs
        return rt

    def _draw_seed(self, corrections: int) -> int:
        """The corrector seed of a run without one: one draw from the global generator when the corrector draws its
        noise on chip, else 0.  rng == "reference" replays the reference's draws (z.normal_() only,
        src/thor/pipelines.py:82): nothing else may touch the global CPU generator, or the stream is shifted by one draw."""
        if corrections > 0 and self.rng != "reference":
            return int(torch.empty((), dtype=torch.int64).random_().item())
        return 0

    def _sample_resident(self, sf: AbstractScoreFunction, noise: Tensor, steps: int, corrections: int, tau: float,
                         device, show_progressbar: bool, seed, proc_x0=None, members: int = 0,
                         rt: Optional[_Runtime] = None) -> Optional[Tensor]:
        """The sampler on the resident state: one trajectory (`seed` an int or None), or an ensemble or batch of
        `members` (`seed` a list of M ints or None; a batch passes its runtime)."""
        if device is not None and torch.device(device).type == "cuda":
            sf.device = torch.device(device)
        if rt is None:
            rt = sf.runtime(noise, members=members)
        group = sf.shard[2] if sf.shard else None
        rt.reset_finite_check()
        rt.load(noise)
        time_steps = torch.linspace(1, 0, steps + 1).to(dtype=torch.float32)
        dt = 1 / steps
        z_dev = None
        if members:
            if seed is None:  # one draw per member, in member order: what M sequential sample() calls draw
                seed = [self._draw_seed(corrections) for _ in range(members)]
            seed = rt.member_seeds(seed)
        elif seed is None:
            seed = self._draw_seed(corrections)
            if sf.shard and corrections > 0 and self.rng != "reference":
                # the on-chip Philox stream is keyed by (seed, step, GLOBAL pixel): every rank must use rank 0's draw,
                # otherwise the result would depend on the sharding
                s_t = torch.tensor([seed], dtype=torch.int64, device=rt.device)
                torch.distributed.broadcast(s_t, src=torch.distributed.get_global_rank(group, 0) if group else 0,
                                            group=group)
                seed = int(s_t.item())
        self.traces = {}
        trace_at = set(int(v) for v in self.trace_at) if self.trace_at else ()
        iterator = time_steps[:-1]
        if show_progressbar:
            try:
                from tqdm.auto import tqdm
                iterator = tqdm(iterator, desc="Sampling")
            except Exception:  # pragma: no cover
                pass
        total_start_time = time.time()
        z_host = torch.empty(noise.shape, dtype=torch.float32) if (corrections > 0 and self.rng == "reference") else None
        for istep, t in enumerate(iterator):
            t_next = t - dt
            mu, sigma = _mu_sigma(self, t)
            mu_n, sigma_n = _mu_sigma(self, t_next)
            # predictor
            rt.score(float(t), group)
            if proc_x0 is None:
                rt.predictor(mu, sigma, mu_n, sigma_n)
            else:
                rt.predictor_with_hook(mu, sigma, mu_n, sigma_n, proc_x0)
            rt.halo(group)
            # corrector
            for ic in range(corrections):
                if z_host is not None:
                    z_host.normal_()
                    p = rt.plan
                    if z_dev is None:
                        z_dev = torch.empty_like(rt.x)
                    src = z_host[p.frame_lo:p.frame_hi].to(rt.device, non_blocking=False).contiguous()
                    with torch.cuda.device(rt.device):
                        _lib.check(rt.lib.c2w_traj_pack(src.data_ptr(), z_dev.data_ptr(), p.n_local, rt.C, rt.H * rt.W,
                                                        rt.stream), "c2w_traj_pack")
                rt.score(float(t_next), group)
                rt.guided_eps(mu_n, sigma_n)
                rt.corrector(tau, sigma_n, z_dev, seed, istep * max(corrections, 1) + ic, group)
                rt.halo(group)
            if self.nan_check_every and (istep + 1) % self.nan_check_every == 0:
                rt.check_finite_lagged()  # reads the flag every check, one check behind: no launch-queue stall
            if (istep + 1) in trace_at:
                tr = rt.owned(rt.x)
                if sf.shard:
                    tr = all_gather_frames(tr, rt.plan, group)
                self.traces[istep + 1] = tr.reshape(noise.shape).cpu() if members else tr.cpu()
        rt.check_finite()
        out = rt.owned(rt.x)
        if sf.shard:
            # time-sharded: the trajectory is assembled on the ranks that asked for it (default: rank 0 of the group;
            # `enable_time_sharding(gather="all")` for every rank) — the others return None
            if sf.shard_gather == "all":
                out = all_gather_frames(out, rt.plan, group)
            else:
                out = gather_frames(out, rt.plan, group, dst=int(sf.shard_gather))
        total_time = time.time() - total_start_time
        print(f"Total sampling time: {total_time:.2f} s  = {total_time / 60:.3f} min = {total_time / 3600:.4f} h")
        if out is None:
            return None
        target = noise.device if device is None else torch.device(device)
        if target.type == "cpu":
            # one asynchronous copy into pinned memory (a pageable destination makes the driver stage it in chunks)
            host = torch.empty(out.shape, dtype=noise.dtype, pin_memory=True)  # a fresh tensor per call: the caller owns it
            host.copy_(out.to(noise.dtype), non_blocking=True)
            torch.cuda.current_stream(rt.device).synchronize()
            return host.reshape(noise.shape)
        return out.to(device=target, dtype=noise.dtype).reshape(noise.shape)
