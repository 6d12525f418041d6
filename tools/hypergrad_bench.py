"""One mixed second derivative of the LightGCN training loss with respect to the edge values against the same quantity in
stock torch, and one interaction hypergradient, on one GPU.

LightGCN at the synthetic size (1 M users x 200 k items x 50 M interactions, D = 64, L = 3) and a batch of 1 048 576
triples: victim.loss_mixed_values(batch, s) for a random direction s, against the float32 torch formulation -- the
propagation as index_add SpMMs over a value vector that requires a gradient (twice differentiable), the BPR loss with its
regulariser, torch.autograd.grad(create_graph=True) with respect to the tables, then the grad of <grad, s> with respect to
the values (double backward).  When torch runs out of memory the line says so instead of a time.  Then one
influence.interaction_hypergradient (objective: the scores of item 0 over the first 10 000 users) at a fixed count of
conjugate-gradient iterations (rtol 0), damping 0.01.

Both arms of the first part start from the same tables; times are CUDA-event medians after a warm-up call.  One JSON line
with the card's name, power limit and max SM clock, each arm's time and peak memory, the largest difference between the
two results relative to the largest magnitude of torch's, and the hypergradient's time and peak memory.
    python tools/hypergrad_bench.py [--reps 3] [--iters 3] [--cg 10] > profiles/hypergrad_r01.jsonl"""
import argparse
import json
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench import WORKLOADS, synth_edges  # noqa: E402
from edge_grad_bench import _Data, card, med, timed  # noqa: E402
from recad_b200 import influence, model, ops  # noqa: E402

DEV = torch.device("cuda:0")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--cg", type=int, default=10)
    ap.add_argument("--workload", default="synthetic", choices=sorted(WORKLOADS))
    args = ap.parse_args()
    w = WORKLOADS[args.workload]
    U, I, D, L, B = w["n_users"], w["n_items"], w["D"], w["L"], w["batch"]
    eu, ei = synth_edges(w, DEV)
    graph = ops.Graph.from_edges(eu, ei, U, I)
    del eu, ei
    m = model.from_config("victim", "lightgcn", latent_dim_rec=D, lightGCN_n_layers=L, init_on_device=True,
                          device=DEV).I(dataset=_Data(U, I, graph))
    lam = float(m.config["lambda"])
    gen = torch.Generator(device=DEV).manual_seed(1)
    us, ps, ns = (torch.randint(0, hi, (B,), device=DEV, generator=gen) for hi in (U, I, I))
    batch = {"users": us, "positive_items": ps, "negative_items": ns}
    s = torch.randn((U + I, D), device=DEV, generator=gen)
    vecs = (s[:U], s[U:])
    res = {}

    def ours():
        res["ours"] = m.loss_mixed_values(batch, vecs)

    N = U + I
    rows = torch.repeat_interleave(torch.arange(N, device=DEV), graph.rowptr[1:] - graph.rowptr[:-1])
    cols = graph.colidx.long()

    def stock():
        v = graph.vals.clone().requires_grad_(True)
        E = m.E.detach().clone().requires_grad_(True)
        X, acc = E, E
        for _ in range(L):
            X = torch.zeros_like(X).index_add(0, rows, v[:, None] * X[cols])
            acc = acc + X
        O = acc / (L + 1)
        u, p, q = O[us], O[U + ps], O[U + ns]
        reg = E[us].pow(2).sum() + E[U + ps].pow(2).sum() + E[U + ns].pow(2).sum()
        loss = F.softplus((u * q).sum(1) - (u * p).sum(1)).mean() + lam * 0.5 * reg / B
        g, = torch.autograd.grad(loss, E, create_graph=True)
        res["stock"], = torch.autograd.grad((g * s).sum(), v)

    out = dict(case=f"lightgcn_loss_mixed_values_D{D}", card=card(), n_users=U, n_items=I, nnz=graph.nnz, D=D, L=L, batch=B)
    ours()
    stock_note = None
    try:
        stock()
    except torch.OutOfMemoryError:
        stock_note = "stock torch ran out of device memory"
    except (RuntimeError, NotImplementedError) as e:
        stock_note = f"stock torch failed: {str(e).splitlines()[0][:200]}"
    if stock_note:
        res.pop("stock", None)
        torch.cuda.empty_cache()
    else:
        ref = res.pop("stock")
        out["max_diff_rel"] = (res["ours"] - ref).abs().max().item() / ref.abs().max().item()
        del ref
    t_o, t_s, m_o, m_s = [], [], 0.0, 0.0
    for _ in range(args.reps):
        t, mm = timed(ours, args.iters)
        t_o.append(t)
        m_o = max(m_o, mm)
        if not stock_note:
            t, mm = timed(stock, args.iters)
            res.pop("stock")
            t_s.append(t)
            m_s = max(m_s, mm)
    out.update(ours_ms=round(med(t_o), 3), ours_ms_all=[round(t, 3) for t in t_o], ours_peak_gb=round(m_o, 3))
    if stock_note:
        out.update(stock_ms=None, stock_note=stock_note)
    else:
        out.update(stock_ms=round(med(t_s), 3), stock_ms_all=[round(t, 3) for t in t_s], stock_peak_gb=round(m_s, 3),
                   speedup=round(med(t_s) / med(t_o), 3))
    res.clear()
    torch.cuda.empty_cache()

    obj_users = torch.arange(10_000, device=DEV)

    def objective(ev):
        return m(obj_users, torch.zeros_like(obj_users), edge_values=ev).sum()

    def hyper():
        res["hg"] = influence.interaction_hypergradient(m, batch, objective, 0.01, max_iter=args.cg, rtol=1e-300)

    hyper()                                                                      # warm-up
    t, mm = timed(hyper, 1)
    out.update(hypergradient_cg_iterations=res["hg"].iterations, hypergradient_ms=round(t, 3),
               hypergradient_peak_gb=round(mm, 3))
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
