"""Autograd through the victims against the same computation in stock torch, on one GPU.

LightGCN: forward + backward of a BPR-style loss built from torch ops on the victim's scores,
    s = victim(cat(users, users), cat(pos, neg)),  loss = softplus(s[B:] - s[:B]).mean(),
over a batch of 1 048 576 triples at the synthetic size (1 M users x 200 k items x 50 M interactions, L = 3), D = 64 and
D = 128.  Stock torch: the propagation as CSR torch.sparse.mm layers, gathers by indexing, autograd.
NCF: forward + backward of the mean BCE over a batch of 1024 pairs at the ml1m shape (5950 x 3702, the default tower:
factor 32, 5 layers, the default `tf32x3` tower), against the same network as torch ops in fp32.

Both arms start from the same tables and run alternately in one process; times are CUDA-event medians after warm-up.
Prints one JSON line per case with the card's name and power limit, the maximum gradient difference between the arms
(relative to the largest gradient magnitude) and each arm's peak memory.
    python tools/autograd_bench.py [--reps 5] [--iters 3] [--d 64 128] > profiles/autograd_r01.jsonl"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import WORKLOADS, synth_edges  # noqa: E402
from recad_b200 import model, ops  # noqa: E402

DEV = torch.device("cuda:0")


class _Data:
    def __init__(self, U, I, graph=None):
        self.U, self.I, self.graph = U, I, graph
        self.config = {"pairwise_batch_size": 1024, "pointwise_batch_size": 1024, "device": DEV}

    def info_describe(self):
        return {"n_users": self.U, "n_items": self.I, "graph": self.graph, "train_dict": None}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def timed(fn, iters):
    """Median over `iters` calls of fn, each bracketed by CUDA events (ms), and the peak memory of those calls (GB)."""
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(DEV)
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return sorted(ts)[len(ts) // 2], torch.cuda.max_memory_allocated(DEV) / 1e9


def compare(name, ours, stock, reps, iters, extra):
    ours(), stock()                           # warm-up: module loads, allocator, cuSPARSE / cuBLAS algorithm choice
    t_o, t_s, m_o, m_s = [], [], 0.0, 0.0
    for _ in range(reps):
        t, m = timed(ours, iters)
        t_o.append(t)
        m_o = max(m_o, m)
        t, m = timed(stock, iters)
        t_s.append(t)
        m_s = max(m_s, m)
    med = lambda v: sorted(v)[len(v) // 2]    # noqa: E731
    out = dict(case=name, card=card(), ours_ms=round(med(t_o), 3), stock_ms=round(med(t_s), 3),
               ours_ms_all=[round(t, 3) for t in t_o], stock_ms_all=[round(t, 3) for t in t_s],
               speedup=round(med(t_s) / med(t_o), 3), ours_peak_gb=round(m_o, 3), stock_peak_gb=round(m_s, 3), **extra)
    print(json.dumps(out), flush=True)


def lightgcn_case(graph, U, I, D, L, B, reps, iters):
    m = model.from_config("victim", "lightgcn", latent_dim_rec=D, lightGCN_n_layers=L, init_on_device=True,
                          device=DEV).I(dataset=_Data(U, I, graph))
    m.requires_grad_(True)
    gen = torch.Generator(device=DEV).manual_seed(1)
    us, ps, ns = (torch.randint(0, hi, (B,), device=DEV, generator=gen) for hi in (U, I, I))
    uu, ii = torch.cat([us, us]), torch.cat([ps, ns])

    def ours():
        m.zero_grad(set_to_none=True)
        s = m(uu, ii)
        F.softplus(s[B:] - s[:B]).mean().backward()

    N = U + I
    A = torch.sparse_csr_tensor(graph.rowptr, graph.colidx.long(), graph.vals, size=(N, N))
    E = torch.nn.Parameter(m.E.detach().clone())

    def stock():
        E.grad = None
        X, acc = E, E
        for _ in range(L):
            X = torch.sparse.mm(A, X)
            acc = acc + X
        O = acc / (L + 1)
        u, p, q = O[us], O[U + ps], O[U + ns]
        F.softplus((u * q).sum(1) - (u * p).sum(1)).mean().backward()

    ours()
    stock()
    g_ours = torch.cat([m.embedding_user.weight.grad, m.embedding_item.weight.grad])
    diff = (g_ours - E.grad).abs().max().item() / E.grad.abs().max().item()
    compare(f"lightgcn_D{D}", ours, stock, reps, iters,
            dict(n_users=U, n_items=I, nnz=graph.nnz, D=D, L=L, batch=B, max_grad_diff_rel=diff))
    del m, A, E


def ncf_case(reps, iters, B=1024):
    w = WORKLOADS["ml1m"]
    U, I = w["n_users"], w["n_items"]
    torch.manual_seed(2023)
    m = model.from_config("victim", "ncf", device=DEV).I(dataset=_Data(U, I))
    m.requires_grad_(True)
    gen = torch.Generator(device=DEV).manual_seed(2)
    us, its = torch.randint(0, U, (B,), device=DEV, generator=gen), torch.randint(0, I, (B,), device=DEV, generator=gen)
    y = torch.randint(0, 2, (B,), device=DEV, generator=gen).float()

    def ours():
        m.zero_grad(set_to_none=True)
        F.binary_cross_entropy_with_logits(m(us, its), y).backward()

    P = [torch.nn.Parameter(p.detach().clone()) for p in m._param_views()]
    n_lin = (len(P) - 6) // 2

    def stock():
        for p in P:
            p.grad = None
        gmf = P[0][us] * P[1][its]
        h = torch.cat([P[2][us], P[3][its]], 1)
        for k in range(n_lin):
            h = torch.relu(F.linear(h, P[4 + 2 * k], P[5 + 2 * k]))
        pred = F.linear(torch.cat([gmf, h], 1), P[-2], P[-1]).view(-1)
        F.binary_cross_entropy_with_logits(pred, y).backward()

    ours()
    stock()
    diff = max(((a.grad - b.grad).abs().max() / b.grad.abs().max().clamp_min(1e-30)).item()
               for a, b in zip(m._param_views(), P))
    compare("ncf_ml1m_b1024", ours, stock, reps, iters,
            dict(n_users=U, n_items=I, factor=m.f, layers=m.L, tower_precision=m.tower_precision, batch=B,
                 max_grad_diff_rel=diff))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--d", type=int, nargs="+", default=[64, 128])
    ap.add_argument("--workload", default="synthetic", choices=sorted(WORKLOADS))
    args = ap.parse_args()
    w = WORKLOADS[args.workload]
    U, I = w["n_users"], w["n_items"]
    eu, ei = synth_edges(w, DEV)
    graph = ops.Graph.from_edges(eu, ei, U, I)
    del eu, ei
    for D in args.d:
        lightgcn_case(graph, U, I, D, w["L"], w["batch"], args.reps, args.iters)
        torch.cuda.empty_cache()
    ncf_case(args.reps, 20 * args.iters)


if __name__ == "__main__":
    main()
