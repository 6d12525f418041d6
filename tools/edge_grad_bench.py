"""Gradients with respect to the graph's edge values against the same computation in stock torch, on one GPU.

LightGCN at the synthetic size (1 M users x 200 k items x 50 M interactions, L = 3), D = 64 and 128: forward + backward of a
BPR-style loss over 1 048 576 triples,
    s = victim(cat(users, users), cat(pos, neg), edge_values=v),  loss = softplus(s[B:] - s[:B]).mean(),
with respect to the edge values v (the graph's own values, CSR entry order) and both tables.  Stock torch (fp32): the
layers as index_add of vals[:, None] * X[cols], gathers by indexing, autograd.  The same call with the tables alone
requiring a gradient is timed too (the backward without the SDDMMs).

Both arms start from the same tables and run alternately in one process; times are CUDA-event medians after warm-up.
One JSON line per case with the card's name, power limit and max SM clock, the maximum gradient difference between the
arms (relative to each gradient's largest magnitude) and each arm's peak memory; then one line per D timing a single
SDDMM launch against a single SpMM launch on the same graph, with the no-reuse byte count (Graph.algorithmic_bytes).
    python tools/edge_grad_bench.py [--reps 3] [--iters 3] [--d 64 128] > profiles/edge_grad_r01.jsonl"""
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


def med(v):
    return sorted(v)[len(v) // 2]


def lightgcn_case(graph, U, I, D, L, B, reps, iters):
    m = model.from_config("victim", "lightgcn", latent_dim_rec=D, lightGCN_n_layers=L, init_on_device=True,
                          device=DEV).I(dataset=_Data(U, I, graph))
    gen = torch.Generator(device=DEV).manual_seed(1)
    us, ps, ns = (torch.randint(0, hi, (B,), device=DEV, generator=gen) for hi in (U, I, I))
    uu, ii = torch.cat([us, us]), torch.cat([ps, ns])
    v = graph.vals.clone().requires_grad_(True)
    v_const = graph.vals.clone()

    def ours():
        m.zero_grad(set_to_none=True)
        v.grad = None
        s = m(uu, ii, edge_values=v)
        F.softplus(s[B:] - s[:B]).mean().backward()

    def ours_tables_only():
        m.zero_grad(set_to_none=True)
        s = m(uu, ii, edge_values=v_const)
        F.softplus(s[B:] - s[:B]).mean().backward()

    rows = torch.repeat_interleave(torch.arange(U + I, device=DEV), graph.rowptr[1:] - graph.rowptr[:-1])
    cols = graph.colidx.long()
    E = torch.nn.Parameter(m.E.detach().clone())
    vs = torch.nn.Parameter(graph.vals.clone())

    def stock():
        E.grad = None
        vs.grad = None
        X, acc = E, E
        for _ in range(L):
            X = torch.zeros_like(X).index_add(0, rows, vs[:, None] * X[cols])
            acc = acc + X
        O = acc / (L + 1)
        u, p, q = O[us], O[U + ps], O[U + ns]
        F.softplus((u * q).sum(1) - (u * p).sum(1)).mean().backward()

    m.requires_grad_(True)
    ours()
    ours_tables_only()
    out = dict(case=f"lightgcn_edge_values_D{D}", card=card(), n_users=U, n_items=I, nnz=graph.nnz, D=D, L=L, batch=B)
    stock_ok = True
    try:
        stock()
    except torch.OutOfMemoryError:
        stock_ok = False
        E.grad = vs.grad = None
        torch.cuda.empty_cache()
    if stock_ok:
        g_ours = torch.cat([m.embedding_user.weight.grad, m.embedding_item.weight.grad])
        out["max_grad_diff_rel_tables"] = (g_ours - E.grad).abs().max().item() / E.grad.abs().max().item()
        out["max_grad_diff_rel_values"] = (v.grad - vs.grad).abs().max().item() / vs.grad.abs().max().item()
    t_o, t_t, t_s, m_o, m_t, m_s = [], [], [], 0.0, 0.0, 0.0
    for _ in range(reps):
        t, mm = timed(ours, iters)
        t_o.append(t)
        m_o = max(m_o, mm)
        t, mm = timed(ours_tables_only, iters)
        t_t.append(t)
        m_t = max(m_t, mm)
        if stock_ok:
            t, mm = timed(stock, iters)
            t_s.append(t)
            m_s = max(m_s, mm)
    out.update(ours_ms=round(med(t_o), 3), ours_ms_all=[round(t, 3) for t in t_o], ours_peak_gb=round(m_o, 3),
               tables_only_ms=round(med(t_t), 3), tables_only_ms_all=[round(t, 3) for t in t_t], tables_only_peak_gb=round(m_t, 3))
    if stock_ok:
        out.update(stock_ms=round(med(t_s), 3), stock_ms_all=[round(t, 3) for t in t_s], stock_peak_gb=round(m_s, 3),
                   speedup=round(med(t_s) / med(t_o), 3))
    else:
        out.update(stock_ms=None, stock_note="stock torch ran out of device memory")
    print(json.dumps(out), flush=True)
    del m, E, vs, v


def kernel_case(graph, D, launches=20):
    """One SDDMM launch against one SpMM launch over the same graph and table, CUDA events around `launches` launches."""
    N = graph.n_rows
    gen = torch.Generator(device=DEV).manual_seed(D)
    G = torch.randn((N, D), device=DEV, generator=gen)
    X = torch.randn((N, D), device=DEV, generator=gen)
    Y = torch.empty_like(X)
    out = torch.empty(graph.nnz, device=DEV)
    fns = {"sddmm": lambda: ops.sddmm(graph, G, X, out=out), "spmm": lambda: ops.spmm(graph, X, Y=Y)}
    res = {}
    for name, fn in fns.items():
        fn()
        ts = []
        for _ in range(3):
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(launches):
                fn()
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b) / launches)
        res[name] = med(ts)
    nbytes = graph.algorithmic_bytes(D)
    print(json.dumps(dict(case=f"sddmm_vs_spmm_D{D}", card=card(), nnz=graph.nnz, D=D, sddmm_ms=round(res["sddmm"], 4),
                          spmm_ms=round(res["spmm"], 4), no_reuse_bytes=nbytes,
                          sddmm_tb_s=round(nbytes / res["sddmm"] / 1e9, 3), spmm_tb_s=round(nbytes / res["spmm"] / 1e9, 3))),
          flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
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
        kernel_case(graph, D)
        torch.cuda.empty_cache()
    for D in args.d:
        lightgcn_case(graph, U, I, D, w["L"], w["batch"], args.reps, args.iters)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
