"""Weight gradients of candidate interactions (LightGCN.candidate_weight_gradients) and one candidate hypergradient
(influence.candidate_hypergradient), on one GPU.

LightGCN at the synthetic size (1 M users x 200 k items x 50 M interactions, D = 64, L = 3), 1024 fake users injected by
Graph.append_users with 50 filler items each, a batch of 1 048 576 triples, R = the 1024 fake users against every item.
  * one candidate_weight_gradients(R, gO, batch, S) call: CUDA-event median and peak memory; its kernels by torch.profiler
    in a run of its own, in four parts (kernel_part): gemm_tc_kernel (the [|R|, 4 L D + 1] x [I, 4 L D + 1]^T GEMM), the
    operand gather, the sample part's own kernels and the recurrence (width-2D SpMMs, seeds, pair pass and its sorts, the
    SDDMM, the normalisation row pass); and, by CUDA events, the d_inv host round trip the call starts with;
  * agreement with a float64 recomputation of the closed form (closed_form64) at 4096 sampled pairs, half of them stored
    pairs of R's rows and half random (mostly not stored);
  * the GEMM's algorithmic rate 2 |R| I (K + 1) over its kernel time, beside the 1125 TFLOP/s dense TF32 data-sheet
    figure (a data-sheet number, not a measured one), and torch.matmul in float32 with TF32 off on random operands of the
    same shapes;
  * one candidate_hypergradient (objective: the scores of item 0 over the first 10 000 users, damping 0.01, 10 CG
    iterations at rtol 0) and, for agreement, interaction_hypergradient on the same objective: at every stored pair of R the
    block against values[k] + values[T[k]], relative to the largest magnitude.
One JSON line with the card's name, power limit and max SM clock.
    python tools/candidate_hypergrad_bench.py [--iters 5] [--cg 10] > profiles/candidate_hypergrad_r01.jsonl"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench import WORKLOADS, synth_edges  # noqa: E402
from edge_grad_bench import _Data, card, timed  # noqa: E402
from recad_b200 import influence, model, ops  # noqa: E402

DEV = torch.device("cuda:0")
TF32_DATASHEET_TFLOPS = 1125.0      # HGX B200 data sheet, one GPU, dense


def kernel_part(name):
    """Which part of one candidate_weight_gradients call a kernel belongs to."""
    if "gemm_tc_kernel" in name:
        return "gemm"
    if "gather_split_kernel" in name or "tail_split_kernel" in name:
        return "gather"
    if any(k in name for k in ("positive_entry_kernel", "index_keys_kernel", "index_sums_kernel", "sample_part_kernel")):
        return "sample"
    if "Memcpy" in name or "Memset" in name:
        return "copies"
    return "recurrence"


def closed_form64(graph, m, batch, gO, S, pu, pi, chunk=1 << 19):
    """df/dW at the pairs (pu[j], item pi[j]) in float64, from the closed form of DESIGN.md ("Second order", candidate
    interactions), independently of the CUDA path: d from float64 row sums of Graph.mult, Y_l = A^l [E | S] and the Horner
    iterates t_j of the seed G = [H_O dO + gO | grad_O L_bpr] as float64 CSR products (torch.sparse), the seed by float64
    autograd, g_v gathered at the pairs and at every stored entry of their rows (for coef), and the sample part by a sorted
    match of the rows' positive pairs."""
    U, I, D, L = m.num_users, m.num_items, m.latent_dim, m.n_layers
    N, lam, n = U + I, float(m.config["lambda"]), batch["users"].numel()
    rowptr, col, w = graph.rowptr, graph.colidx.long(), graph.mult.double()
    rows = torch.repeat_interleave(torch.arange(N, device=DEV), rowptr[1:] - rowptr[:-1])
    d = (torch.zeros(N, dtype=torch.float64, device=DEV).index_add_(0, rows, w) + 1e-14) ** -0.5
    A = torch.sparse_csr_tensor(rowptr, col, d[rows] * w * d[col], (N, N))
    del rows
    E64, S64 = m.E.detach().double(), torch.cat(S).double()
    Y = [torch.cat([E64, S64], 1)]
    for _ in range(L - 1):
        Y.append(torch.sparse.mm(A, Y[-1]))
    OO = sum(Y)
    if L > 0:
        OO = OO + torch.sparse.mm(A, Y[-1])
    OO = OO / (L + 1)
    O, dO = OO[:, :D].contiguous(), OO[:, D:].contiguous()
    del OO
    u, p, q = batch["users"], batch["positive_items"], batch["negative_items"]
    Ol = O.clone().requires_grad_(True)
    with torch.enable_grad():
        x = (Ol[u] * Ol[U + q]).sum(1) - (Ol[u] * Ol[U + p]).sum(1)
        g, = torch.autograd.grad(torch.nn.functional.softplus(x).mean(), Ol, create_graph=True)
        GO, = torch.autograd.grad((g * dO).sum(), Ol)
    G = torch.cat([GO + torch.cat(gO).double(), g.detach()], 1)
    del Ol, g, GO
    t = [G]
    for _ in range(L - 1):
        t.append(G + torch.sparse.mm(A, t[-1]))

    def gv(r, c):                                         # (1 / (L + 1)) sum_j <t_j[r], Y_{L-1-j}[c]>, in chunks
        out = torch.empty(r.numel(), dtype=torch.float64, device=DEV)
        for a in range(0, r.numel(), chunk):
            rr, cc = r[a:a + chunk], c[a:a + chunk]
            out[a:a + chunk] = sum((t[j][rr] * Y[L - 1 - j][cc]).sum(1) for j in range(L)) / (L + 1)
        return out

    def pair(r, c):
        return gv(r, c) + gv(c, r)

    val = d[pu] * d[U + pi] * pair(pu, U + pi)
    # coef_r = -0.5 d_r^3 sum over row r's entries k of w_k d_c(k) (g_v(r, c) + g_v(c, r)) (w symmetric)
    rs = torch.unique(torch.cat([pu, U + pi]))
    cnt = rowptr[rs + 1] - rowptr[rs]
    ent = torch.repeat_interleave(rowptr[rs], cnt) + torch.arange(int(cnt.sum()), device=DEV) - \
        torch.repeat_interleave(torch.cumsum(cnt, 0) - cnt, cnt)
    er = torch.repeat_interleave(rs, cnt)
    P = torch.zeros(N, dtype=torch.float64, device=DEV).index_add_(0, er, w[ent] * d[col[ent]] * pair(er, col[ent]))
    coef = -0.5 * d ** 3 * P
    val = val + coef[pu] + coef[U + pi]
    # sample part: (1 / (n mult_k)) sum of the rows' directional derivatives over the rows with positive pair k
    dx = (dO[u] * (O[U + q] - O[U + p])).sum(1) + (O[u] * (dO[U + q] - dO[U + p])).sum(1)
    xb = (O[u] * O[U + q]).sum(1) - (O[u] * O[U + p]).sum(1)
    reg = (S64[u] * E64[u]).sum(1) + (S64[U + p] * E64[U + p]).sum(1) + (S64[U + q] * E64[U + q]).sum(1)
    dl = torch.sigmoid(xb) * dx + lam * reg
    bkey, order = torch.sort(u * I + p)
    csum = torch.cat([torch.zeros(1, dtype=torch.float64, device=DEV), torch.cumsum(dl[order], 0)])
    key = pu * I + pi
    sums = csum[torch.searchsorted(bkey, key, right=True)] - csum[torch.searchsorted(bkey, key)]
    k = graph.entry_index(pu, U + pi, missing=-1)
    mult_k = torch.where(k >= 0, w[k.clamp(min=0)], torch.ones_like(d[pu]))
    return val + torch.where(k >= 0, sums / (n * mult_k), torch.zeros_like(sums))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--cg", type=int, default=10)
    ap.add_argument("--fake", type=int, default=1024)
    ap.add_argument("--filler", type=int, default=50)
    ap.add_argument("--workload", default="synthetic", choices=sorted(WORKLOADS))
    args = ap.parse_args()
    w = WORKLOADS[args.workload]
    U0, I, D, L, B = w["n_users"], w["n_items"], w["D"], w["L"], w["batch"]
    F_ = args.fake
    eu, ei = synth_edges(w, DEV)
    graph = ops.Graph.from_edges(eu, ei, U0, I)
    del eu, ei
    gen = torch.Generator(device=DEV).manual_seed(1)
    filler = torch.argsort(torch.rand((F_, I), device=DEV, generator=gen), dim=1)[:, :args.filler].sort(dim=1).values
    fake_rowptr = torch.arange(F_ + 1, device=DEV) * args.filler
    graph = graph.append_users(U0, I, fake_rowptr, filler.reshape(-1).int())
    U = U0 + F_
    m = model.from_config("victim", "lightgcn", latent_dim_rec=D, lightGCN_n_layers=L, init_on_device=True,
                          device=DEV).I(dataset=_Data(U, I, graph))
    us, ns = (torch.randint(0, hi, (B,), device=DEV, generator=gen) for hi in (U, I))
    # positives: half stored pairs (k(b) exists), half random items
    rows = torch.repeat_interleave(torch.arange(U + I, device=DEV), graph.rowptr[1:] - graph.rowptr[:-1])
    user_side = torch.nonzero(rows < U).squeeze(1)
    pick = user_side[torch.randint(0, user_side.numel(), (B // 2,), device=DEV, generator=gen)]
    us[:B // 2] = rows[pick]
    ps = torch.randint(0, I, (B,), device=DEV, generator=gen)
    ps[:B // 2] = graph.colidx[pick].long() - U
    del rows, user_side, pick
    batch = {"users": us, "positive_items": ps, "negative_items": ns}
    R = torch.arange(U0, U, device=DEV)
    gO = tuple(torch.randn(s, device=DEV, generator=gen) for s in ((U, D), (I, D)))
    S = tuple(torch.randn(s, device=DEV, generator=gen) for s in ((U, D), (I, D)))
    K1 = 4 * L * D + 1
    out = dict(case=f"lightgcn_candidate_weight_grads_D{D}_L{L}", card=card(), n_users=U, n_fake=F_, n_items=I,
               nnz=graph.nnz, D=D, L=L, batch=B, n_sel=int(R.numel()), gemm_K=K1)
    res = {}

    def block():
        res["block"] = m.candidate_weight_gradients(R, gO, batch, S)

    block()                                                                      # warm-up
    t, mm = timed(block, args.iters)
    out.update(call_ms=round(t, 3), call_peak_gb=round(mm, 3))
    res.clear()
    torch.cuda.empty_cache()

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        block()
        torch.cuda.synchronize()
    part = {"gemm": 0.0, "gather": 0.0, "sample": 0.0, "recurrence": 0.0, "copies": 0.0}
    for e in prof.key_averages():
        if e.device_type.name != "CUDA" or e.device_time_total <= 0:
            continue
        part[kernel_part(e.key)] += e.device_time_total / 1e3
    flops = 2.0 * R.numel() * I * K1
    out.update(gemm_kernel_ms=round(part["gemm"], 3), gather_kernels_ms=round(part["gather"], 3),
               sample_part_kernels_ms=round(part["sample"], 3), recurrence_kernels_ms=round(part["recurrence"], 3),
               copies_ms=round(part["copies"], 3),
               gemm_tflops_algorithmic=round(flops / (part["gemm"] * 1e-3) / 1e12, 1),
               tf32_datasheet_tflops=TF32_DATASHEET_TFLOPS)
    res.clear()
    torch.cuda.empty_cache()

    def dinv():
        res["d_inv"] = ops.weights_d_inv(graph, graph.mult)

    dinv()
    t, _ = timed(dinv, args.iters)
    out.update(d_inv_host_round_trip_ms=round(t, 3))
    res.clear()

    # float64 recomputation of the closed form at 4096 sampled pairs: half stored pairs of R's rows, half random
    block()
    got_block = res.pop("block")
    lo, hi = int(graph.rowptr[U0]), int(graph.rowptr[U])
    r_all = torch.repeat_interleave(torch.arange(F_, device=DEV), graph.rowptr[U0 + 1:U + 1] - graph.rowptr[U0:U])
    pick = torch.randint(0, hi - lo, (2048,), device=DEV, generator=gen)
    pr = torch.cat([r_all[pick], torch.randint(0, F_, (2048,), device=DEV, generator=gen)])
    pi = torch.cat([graph.colidx[lo + pick].long() - U, torch.randint(0, I, (2048,), device=DEV, generator=gen)])
    stored = graph.entry_index(R[pr], U + pi, missing=-1) >= 0
    ref = closed_form64(graph, m, batch, gO, S, R[pr], pi)
    got = got_block[pr, pi].double()
    scale = ref.abs().max().item()
    out.update(f64_pairs=int(pr.numel()), f64_pairs_stored=int(stored.sum()), f64_pairs_unstored=int((~stored).sum()),
               f64_max_diff_rel=(got - ref).abs().max().item() / scale,
               f64_max_diff_rel_stored=(got - ref)[stored].abs().max().item() / scale,
               f64_max_diff_rel_unstored=(got - ref)[~stored].abs().max().item() / scale)
    del got_block, ref, got
    torch.cuda.empty_cache()

    A = torch.randn((R.numel(), K1), device=DEV, generator=gen)
    Bm = torch.randn((I, K1), device=DEV, generator=gen)
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False

    def mm_fp32():
        res["mm"] = torch.matmul(A, Bm.T)

    mm_fp32()
    t, _ = timed(mm_fp32, args.iters)
    torch.backends.cuda.matmul.allow_tf32 = prev
    out.update(torch_matmul_fp32_ms=round(t, 3), torch_matmul_fp32_tflops=round(flops / (t * 1e-3) / 1e12, 1))
    del A, Bm
    res.clear()
    torch.cuda.empty_cache()

    obj_users = torch.arange(10_000, device=DEV)

    def cand():
        res["ch"] = influence.candidate_hypergradient(m, batch, lambda uo, io: (uo[obj_users] * io[0]).sum(), R, 0.01,
                                                      max_iter=args.cg, rtol=1e-300)

    cand()                                                                       # warm-up
    t, mm = timed(cand, 1)
    out.update(hypergradient_cg_iterations=res["ch"].iterations, hypergradient_ms=round(t, 3),
               hypergradient_peak_gb=round(mm, 3))
    hg = influence.interaction_hypergradient(m, batch, lambda ev: m(obj_users, torch.zeros_like(obj_users),
                                                                    edge_values=ev).sum(),
                                             0.01, max_iter=args.cg, rtol=1e-300)
    lo, hi = int(graph.rowptr[U0]), int(graph.rowptr[U])
    k = torch.arange(lo, hi, device=DEV)
    r = torch.repeat_interleave(torch.arange(F_, device=DEV), graph.rowptr[U0 + 1:U + 1] - graph.rowptr[U0:U])
    T = graph.transpose_permutation()
    ref = hg.values[k] + hg.values[T[k]]
    got = res["ch"].values[r, graph.colidx[k].long() - U]
    out.update(stored_pairs_checked=int(k.numel()),
               stored_pairs_max_diff_rel=(got - ref).abs().max().item() / ref.abs().max().item())
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
