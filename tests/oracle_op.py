"""Guided score for an ARBITRARY observation operator A, restating src/thor/score.py:44-60 (log_p through A, autograd)
on top of the oracle's window composition and schedule (oracle/score_ref.py, whose coarse-graining functions
hard-code A = AvgPool2d(s)(x[::t])).  Test infrastructure only: the point-observation tests pin the CUDA path against
these with the same PointObservation object the package uses."""
from __future__ import annotations

from typing import Callable, Optional

import torch

from oracle.score_ref import mu_sigma, window_score

Tensor = torch.Tensor


def guided_score_op(net: Callable, x: Tensor, t: Tensor, k: int, y: Tensor, std, gamma, A: Callable, exact_grad: bool,
                    batch_size: Optional[int] = None, eta: float = 1e-3) -> Tensor:
    """AbstractScoreFunction.__call__ with a likelihood through any differentiable A, by autograd exactly as the
    reference does it."""
    mu, sigma = mu_sigma(t, eta)
    xg = x.detach().clone().requires_grad_(True)
    with torch.set_grad_enabled(exact_grad):
        eps = window_score(net, xg, t, k, batch_size)
    with torch.enable_grad():
        x0 = (xg - sigma * eps) / mu
        err = y - A(x0)
        var = std ** 2 + gamma * (sigma / mu) ** 2
        logp = -(err ** 2 / var).sum() / 2
        (J,) = torch.autograd.grad(logp, xg)
    return (eps - sigma * J).detach()


def guided_score_closed_form_op(eps: Tensor, x: Tensor, t: Tensor, y: Tensor, std, gamma, A: Callable,
                                eta: float = 1e-3) -> Tensor:
    """exact_grad=False for any A: J = A^T((y - A x0)/var) / mu, the adjoint by torch.func.vjp through A."""
    mu, sigma = mu_sigma(t, eta)
    x0 = (x - sigma * eps) / mu
    Ax0, pullback = torch.func.vjp(A, x0)
    var = std ** 2 + gamma * (sigma / mu) ** 2
    (g,) = pullback((y - Ax0) / var)
    return eps - sigma * g / mu
