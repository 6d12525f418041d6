"""One Hessian-vector product of the NCF training loss against the same product in stock torch, on one GPU.

NeuMF-end with the default tower (factor 32, 5 layers: 1024 -> 512 -> ... -> 32) at two table shapes, ml1m (5 950 users x
3 702 items) and yelp (54 632 x 34 474), and a batch of 1 048 576 random (user, item, label) rows: victim.loss_hvp(batch, v)
for a random direction v, in both tower precisions, against the float32 torch formulation -- an nn.Module built from the
victim's parameters (embeddings, Linear layers, ReLU), the mean BCE with logits, torch.autograd.grad(create_graph=True) and
a second grad of <grad, v> (double backward), TF32 off.  When torch runs out of memory, the line says so instead of a time.

Both arms start from the same parameters and run alternately in one process; times are CUDA-event medians after warm-up.
One JSON line per (shape, precision) with the card's name, power limit and max SM clock, each arm's time and peak memory,
the largest difference between the two products relative to the largest magnitude of torch's, and the time of one
victim.sample_directional_derivatives call on the same rows.
    python tools/ncf_hvp_bench.py [--reps 3] [--iters 3] > profiles/ncf_hvp_r01.jsonl"""
import argparse
import json
import os
import sys

import torch
import torch.nn.functional as F
from torch import nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from edge_grad_bench import _Data, card, med, timed  # noqa: E402
from recad_b200 import model  # noqa: E402

DEV = torch.device("cuda:0")
SHAPES = {"ml1m": (5950, 3702), "yelp": (54632, 34474)}


class StockNCF(nn.Module):
    """NeuMF-end (ncf.py:112-131) as plain torch modules, holding copies of a victim's parameters."""

    def __init__(self, views, L):
        super().__init__()
        self.L = L
        self.ps = nn.ParameterList([nn.Parameter(t.detach().clone()) for t in views])

    def forward(self, u, i):
        p = self.ps
        gmf = p[0][u] * p[1][i]
        h = torch.cat([p[2][u], p[3][i]], 1)
        for l in range(self.L):
            h = torch.relu(F.linear(h, p[4 + 2 * l], p[5 + 2 * l]))
        return F.linear(torch.cat([gmf, h], 1), p[-2], p[-1]).view(-1)


def case(shape, precision, n, reps, iters):
    U, I = SHAPES[shape]
    m = model.from_config("victim", "ncf", tower_precision=precision, device=DEV).I(dataset=_Data(U, I))
    gen = torch.Generator(device=DEV).manual_seed(1)
    batch = {"users": torch.randint(0, U, (n,), device=DEV, generator=gen),
             "items": torch.randint(0, I, (n,), device=DEV, generator=gen),
             "labels": torch.randint(0, 2, (n,), device=DEV, generator=gen)}
    views = m._param_views()
    vecs = tuple(torch.randn(t.shape, device=DEV, generator=gen) for t in views)
    stock_m = StockNCF(views, m.L)
    y = batch["labels"].float()
    res = {}

    def ours():
        res["ours"] = torch.cat([h.reshape(-1) for h in m.loss_hvp(batch, vecs)])

    def stock():
        ps = list(stock_m.ps)
        loss = F.binary_cross_entropy_with_logits(stock_m(batch["users"], batch["items"]), y)
        g = torch.autograd.grad(loss, ps, create_graph=True)
        hv = torch.autograd.grad(sum((a * v).sum() for a, v in zip(g, vecs)), ps)
        res["stock"] = torch.cat([h.reshape(-1) for h in hv])

    out = dict(case=f"ncf_loss_hvp_{shape}_{precision}", card=card(), n_users=U, n_items=I, factor=m.f, layers=m.L, rows=n,
               tower_precision=precision, n_params=sum(t.numel() for t in views))
    ours()
    stock_note = None
    try:
        stock()
    except torch.OutOfMemoryError:
        stock_note = "stock torch ran out of device memory"
    if stock_note:
        res.pop("stock", None)
        torch.cuda.empty_cache()
    else:
        ref = res.pop("stock")
        out["max_diff_rel"] = (res["ours"] - ref).abs().max().item() / ref.abs().max().item()
        del ref
    t_o, t_s, m_o, m_s = [], [], 0.0, 0.0
    for _ in range(reps):
        t, mm = timed(ours, iters)
        t_o.append(t)
        m_o = max(m_o, mm)
        if not stock_note:
            t, mm = timed(stock, iters)
            res.pop("stock")
            t_s.append(t)
            m_s = max(m_s, mm)
    t_d, _ = timed(lambda: m.sample_directional_derivatives(batch, vecs), iters)
    out.update(ours_ms=round(med(t_o), 3), ours_ms_all=[round(t, 3) for t in t_o], ours_peak_gb=round(m_o, 3),
               directional_ms=round(t_d, 3))
    if stock_note:
        out.update(stock_ms=None, stock_note=stock_note)
    else:
        out.update(stock_ms=round(med(t_s), 3), stock_ms_all=[round(t, 3) for t in t_s], stock_peak_gb=round(m_s, 3),
                   speedup=round(med(t_s) / med(t_o), 3))
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--rows", type=int, default=1 << 20)
    ap.add_argument("--shapes", nargs="+", default=["ml1m", "yelp"], choices=sorted(SHAPES))
    ap.add_argument("--precisions", nargs="+", default=["fp32", "tf32x3"], choices=["fp32", "tf32x3"])
    args = ap.parse_args()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    for shape in args.shapes:
        for precision in args.precisions:
            case(shape, precision, args.rows, args.reps, args.iters)
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
