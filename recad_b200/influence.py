"""Influence of training rows on an objective, from the victims' Hessian-vector products (loss_hvp) and per-row
directional derivatives (sample_directional_derivatives) -- the estimate -grad(obj)^T H^-1 grad(l_z) of influence-function
attacks and defenses (Fang et al., WWW 2020).  H is the Hessian of the training loss of the given rows taken as one batch,
at the victim's current tables.  Works with any victim that has those two methods (LightGCN, MF, NCF)."""
import math
from collections import namedtuple

import torch

from ._lib import RecadError

Influence = namedtuple("Influence", ["values", "s", "iterations", "residual"])


def conjugate_gradient(hvp, rhs, damping, max_iter=100, rtol=1e-6):
    """Solve (H + damping I) s = rhs by conjugate gradients on flat vectors.  hvp(x) returns H x for a vector shaped like
    rhs; the iteration runs in rhs's dtype.  `damping` has no default: H is indefinite away from a minimum, and CG needs
    H + damping I positive definite (RecadError when a search direction shows it is not).  Stops once
    ||r|| / ||rhs|| < rtol (r the recurrence residual) or after max_iter products.
    Returns (s, iterations, relative residual)."""
    damping = float(damping)
    if damping < 0 or max_iter < 1 or rtol <= 0:
        raise RecadError("conjugate_gradient: damping >= 0, max_iter >= 1 and rtol > 0 needed")
    x = torch.zeros_like(rhs)
    r = rhs.clone()
    p = r.clone()
    rs = float(r.dot(r))
    b_norm = math.sqrt(rs)
    if b_norm == 0.0:
        return x, 0, 0.0
    res = 1.0
    for k in range(1, max_iter + 1):
        Ap = hvp(p).to(rhs.dtype) + damping * p
        pAp = float(p.dot(Ap))
        if not pAp > 0.0:
            raise RecadError(f"conjugate_gradient: H + damping I is not positive definite (p^T A p = {pAp:.3e} at "
                             f"iteration {k}); increase damping")
        a = rs / pAp
        x.add_(p, alpha=a)
        r.add_(Ap, alpha=-a)
        rs_new = float(r.dot(r))
        res = math.sqrt(rs_new) / b_norm
        if res < rtol:
            return x, k, res
        p.mul_(rs_new / rs).add_(r)
        rs = rs_new
    return x, max_iter, res


def sample_influence(victim, batch, objective_grads, damping, max_iter=100, rtol=1e-6):
    """Influence of every row of `batch` on an objective.

    objective_grads: the objective's gradient with respect to the victim's trainable tables, one tensor per table in
    loss_hvp's order (parameters() order; MF without `mean`), e.g. the `.grad`s after `victim.requires_grad_(True)`,
    scoring the target pairs and `backward()`.  Solves (H + damping I) s = grad(obj) with conjugate_gradient (in float64,
    H from victim.loss_hvp) and returns Influence(values, s, iterations, residual) with values[b] = s^T grad(l_b)
    (float32 [n], victim.sample_directional_derivatives along s).

    Sign convention: with the loss L = (1/n) sum_b l_b, removing row b changes the trained tables by about
    +(1/n) H^-1 grad(l_b), so the predicted change of the objective when row b is removed is (1/n) values[b]
    (positive: removing the row raises the objective); up-weighting row b by eps changes it by -eps values[b]."""
    grads = [g.detach() for g in objective_grads]
    shapes = [g.shape for g in grads]
    sizes = [g.numel() for g in grads]

    def unflat(x):
        return tuple(c.view(s).float().contiguous() for c, s in zip(torch.split(x, sizes), shapes))

    def hvp(x):
        return torch.cat([h.reshape(-1) for h in victim.loss_hvp(batch, unflat(x))]).double()

    rhs = torch.cat([g.reshape(-1) for g in grads]).double()
    s, iters, res = conjugate_gradient(hvp, rhs, damping, max_iter, rtol)
    s_t = unflat(s)
    return Influence(victim.sample_directional_derivatives(batch, s_t), s_t, iters, res)
