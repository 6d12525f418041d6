"""Influence of training rows on an objective, from the victims' Hessian-vector products (loss_hvp) and per-row
directional derivatives (sample_directional_derivatives) -- the estimate -grad(obj)^T H^-1 grad(l_z) of influence-function
attacks and defenses (Fang et al., WWW 2020).  H is the Hessian of the training loss of the given rows taken as one batch,
at the victim's current tables.  Works with any victim that has those two methods (LightGCN, MF, NCF).

interaction_hypergradient: for LightGCN, whose training loss depends on the interactions both as training rows and as
graph edges, the derivative of an objective of the retrained tables with respect to every interaction weight;
candidate_hypergradient: the same derivative for chosen users against every item, at interactions not stored yet too."""
import math
from collections import namedtuple

import torch

from . import ops
from ._lib import RecadError

Influence = namedtuple("Influence", ["values", "s", "iterations", "residual"])
Hypergradient = namedtuple("Hypergradient", ["values", "direct", "implicit", "s", "iterations", "residual"])
CandidateHypergradient = namedtuple("CandidateHypergradient", ["values", "s", "iterations", "residual"])


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
    s_t, iters, res = _solve(victim, batch, objective_grads, damping, max_iter, rtol)
    return Influence(victim.sample_directional_derivatives(batch, s_t), s_t, iters, res)


def _solve(victim, batch, objective_grads, damping, max_iter, rtol):
    """s = (H + damping I)^-1 grad(obj) by conjugate_gradient in float64 over victim.loss_hvp: (s as float32 tensors shaped
    like objective_grads, iterations, relative residual)."""
    grads = [g.detach() for g in objective_grads]
    shapes = [g.shape for g in grads]
    sizes = [g.numel() for g in grads]

    def unflat(x):
        return tuple(c.view(s).float().contiguous() for c, s in zip(torch.split(x, sizes), shapes))

    def hvp(x):
        return torch.cat([h.reshape(-1) for h in victim.loss_hvp(batch, unflat(x))]).double()

    rhs = torch.cat([g.reshape(-1) for g in grads]).double()
    s, iters, res = conjugate_gradient(hvp, rhs, damping, max_iter, rtol)
    return unflat(s), iters, res


def interaction_hypergradient(victim, batch, objective, damping, max_iter=100, rtol=1e-6):
    """dJ/dw for every interaction weight w_k (one per stored entry of victim.Graph, CSR order, at the base point
    w = Graph.mult) of an objective J of the LightGCN tables trained on the BPR loss of `batch` (the rows as for
    loss_hvp, weighted by w_k(b) / mult_k(b) where k(b) is the entry (u_b, U + pos_b) when it is stored):

        dJ/dw = dJ/dw|_E - M^T s,   s = (H + damping I)^-1 grad_E J,   M^T s = d/dw [s^T grad_E L(E; w)]

    at the victim's current tables, taken as trained (grad_E L ~ 0).  objective(edge_values) returns a scalar tensor built
    from victim(users, items, edge_values=edge_values); it is evaluated at ops.normalized_values(Graph, w) with w and
    the tables requiring a gradient (their requires_grad flags are restored afterwards).  s is solved by
    conjugate_gradient in float64 over loss_hvp.  M^T s = N'(w)^T loss_mixed_values(batch, s) (the graph part) + the
    sample part, (1 / (n mult_k)) sum over the rows with k(b) = k of s^T grad l_b (rows whose positive pair is not stored
    have none).  Returns Hypergradient(values = direct - implicit, direct, implicit, s, iterations, residual), the first
    three float32 [nnz].  When both entries of an interaction carry one weight, its sensitivity is values[k] +
    values[T[k]] (k = Graph.entry_index(u, U + i), T = Graph.transpose_permutation()).  LightGCN only (DESIGN.md,
    "Second order"); deterministic; the tables are not changed."""
    from .victim.lightgcn import LightGCN
    if not isinstance(victim, LightGCN):
        raise RecadError(f"interaction_hypergradient: LightGCN victims only (got {type(victim).__name__})")
    victim._require_instance("interaction_hypergradient")
    g, U = victim.Graph, victim.num_users
    params = list(victim.parameters())
    flags = [p.requires_grad for p in params]
    w = g.mult.detach().clone().requires_grad_(True)
    try:
        for p in params:
            p.requires_grad_(True)
        with torch.enable_grad():
            J = objective(ops.normalized_values(g, w))
            if not isinstance(J, torch.Tensor) or J.numel() != 1:
                raise RecadError("interaction_hypergradient: the objective must return a scalar tensor")
            gw, *gE = torch.autograd.grad(J.reshape(()), [w] + params, allow_unused=True)
    finally:
        for p, f in zip(params, flags):
            p.requires_grad_(f)
    direct = torch.zeros_like(w) if gw is None else gw.detach()
    gE = [torch.zeros_like(p) if x is None else x for p, x in zip(params, gE)]
    s, iters, res = _solve(victim, batch, gE, damping, max_iter, rtol)

    gv = victim.loss_mixed_values(batch, s)
    w = g.mult.detach().clone().requires_grad_(True)
    with torch.enable_grad():
        graph_part, = torch.autograd.grad(ops.normalized_values(g, w), w, gv)
    dl = victim.sample_directional_derivatives(batch, s)
    k = g.entry_index(batch["users"], U + batch["positive_items"], missing=-1)
    sample_part = ops.index_sums(k, dl, g.nnz) / (dl.numel() * g.mult)
    implicit = graph_part + sample_part
    return Hypergradient(direct - implicit, direct, implicit, s, iters, res)


def candidate_hypergradient(victim, batch, objective, users, damping, max_iter=100, rtol=1e-6):
    """dJ/dW[r, i] for one weight W on both entries of the interaction (users[r], item i), for every item, stored or not
    (W = Graph.mult on stored pairs, 0 on the others), of an objective J of the LightGCN tables trained on the BPR loss of
    `batch` (rows weighted as for interaction_hypergradient):

        dJ/dW = dJ/dW|_E - M^T s,   s = (H + damping I)^-1 grad_E J

    at the victim's current tables, taken as trained.  objective(user_out, item_out) returns a scalar tensor built from
    the two outputs of computer(); its gradient gO comes from torch autograd on a fresh propagation, grad_E J =
    P^T gO, s is solved by conjugate_gradient in float64 over loss_hvp, and values =
    victim.candidate_weight_gradients(users, gO, batch, -s).  At a stored pair, values equals values[k] + values[T[k]] of
    interaction_hypergradient for the same objective.  Sign convention: a negative values[r, i] means that adding the
    interaction (users[r], i) -- raising its weight from 0 -- lowers J to first order (a positive one, that it raises J).
    Returns CandidateHypergradient(values float32 [len(users), num_items], s, iterations, residual).  LightGCN only
    (DESIGN.md, "Second order"); deterministic; the model is not changed."""
    from .victim.lightgcn import LightGCN
    if not isinstance(victim, LightGCN):
        raise RecadError(f"candidate_hypergradient: LightGCN victims only (got {type(victim).__name__})")
    victim._require_instance("candidate_hypergradient")
    if victim.dropout and victim.training:
        raise RecadError("candidate_hypergradient: not defined under graph dropout in training mode (call eval() first)")
    # the users and the batch are checked before the propagation and the solve, not after them
    victim._check_candidate_users(users, "candidate_hypergradient")
    if users.numel() and bool(((users < 0) | (users >= victim.num_users)).any()):
        raise RecadError("candidate_hypergradient: a user id is out of range")
    victim._loss_rows(batch, "candidate_hypergradient")
    U = victim.num_users
    with torch.cuda.device(victim._dev):
        O, _ = ops.lightgcn_propagate_layers(victim._st, victim.E, keep=False)
        uo = O[:U].clone().requires_grad_(True)
        io = O[U:].clone().requires_grad_(True)
        with torch.enable_grad():
            J = objective(uo, io)
            if not isinstance(J, torch.Tensor) or J.numel() != 1:
                raise RecadError("candidate_hypergradient: the objective must return a scalar tensor")
            gu, gi = torch.autograd.grad(J.reshape(()), [uo, io], allow_unused=True)
        gO = [torch.zeros_like(uo) if g is None else g.detach().float().contiguous() for g in (gu, gi)]
        gE = ops.lightgcn_backward(victim._st, torch.cat(gO))
    s, iters, res = _solve(victim, batch, [gE[:U], gE[U:]], damping, max_iter, rtol)
    values = victim.candidate_weight_gradients(users, gO, batch, [-x for x in s])
    return CandidateHypergradient(values, s, iters, res)
