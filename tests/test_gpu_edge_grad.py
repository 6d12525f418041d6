"""Gradients with respect to the graph's edge values: the SDDMM (`ops.sddmm`), LightGCN scores differentiable with respect
to caller-supplied `edge_values`, and the weights -> values normalisation (`ops.normalized_values`).  Checked against torch
autograd in float64 on the same GPU, over the same CSR."""
import numpy as np
import pytest
import torch

from oracle import graph as og
from tests import util

pytestmark = pytest.mark.gpu
META = util.meta()
DEV = "cuda:0"
U, I = META["dev"]["n_users"], META["dev"]["n_items"]


class StubData:
    def __init__(self, graph, n_users=U, n_items=I):
        self.graph, self.n_users, self.n_items = graph, n_users, n_items
        self.config = {"pairwise_batch_size": 1024, "pointwise_batch_size": 1024, "device": torch.device(DEV)}

    def info_describe(self):
        return {"n_users": self.n_users, "n_items": self.n_items, "graph": self.graph, "train_dict": None}

    def generate_batch(self):
        return iter(())


def _dev_edges():
    tr, _, _ = util.dicts("dev")
    u, i, _, _ = og.flatten_dict(tr)
    return torch.as_tensor(u, device=DEV), torch.as_tensor(i, device=DEV)


@pytest.fixture(scope="module")
def dev_graph():
    from recad_b200 import ops
    return ops.Graph.from_edges(*_dev_edges(), U, I)


@pytest.fixture(scope="module")
def multiseg_graph():
    """700 users x 300 items x 20 000 draws with seg_len = 32: item rows (~60 entries) and user 0 (1 500 draws) are cut into
    several segments (the dev graph's rows hold at most 7 entries)."""
    from recad_b200 import ops
    rng = np.random.default_rng(7)
    u = np.concatenate([np.zeros(1500, np.int64), rng.integers(0, 700, 18500)])
    i = rng.integers(0, 300, 20000)
    g = ops.Graph.from_edges(torch.as_tensor(u, device=DEV), torch.as_tensor(i, device=DEV), 700, 300, seg_len=32)
    assert g.n_mrow > 0
    return g


def _rows(graph):
    return torch.repeat_interleave(torch.arange(graph.n_rows, device=DEV), graph.rowptr[1:] - graph.rowptr[:-1])


def _rel_close(got, ref, bar):
    """|got - ref| <= bar * max |ref|, on the whole tensor."""
    got, ref = got.detach().double(), ref.detach().double()
    assert got.shape == ref.shape
    err, scale = (got - ref).abs().max().item(), ref.abs().max().item()
    assert err <= bar * scale, f"max error {err:.3e} > {bar:g} x {scale:.3e}"


def _pairs(seed, B, n_users=U, n_items=I):
    rng = np.random.default_rng(seed)
    u = torch.as_tensor(rng.integers(0, n_users, B), device=DEV)
    i = torch.as_tensor(rng.integers(0, n_items, B), device=DEV)
    w = torch.as_tensor(rng.normal(size=B), dtype=torch.float32, device=DEV)
    return u, i, w


def _sddmm_ref(graph, G, X, chunk=1 << 18):
    rows, cols = _rows(graph), graph.colidx.long()
    out = torch.empty(graph.nnz, dtype=torch.float64, device=DEV)
    for s in range(0, graph.nnz, chunk):
        e = min(s + chunk, graph.nnz)
        out[s:e] = (G[rows[s:e]].double() * X[cols[s:e]].double()).sum(1)
    return out


# ------------------------------------------------------------------ SDDMM
@pytest.mark.parametrize("D", [4, 64, 128])
@pytest.mark.parametrize("which", ["dev", "multiseg"])
def test_sddmm_matches_float64(dev_graph, multiseg_graph, D, which):
    from recad_b200 import ops
    g = dev_graph if which == "dev" else multiseg_graph
    gen = torch.Generator(device=DEV).manual_seed(D)
    G = torch.randn((g.n_rows, D), device=DEV, generator=gen)
    X = torch.randn((g.n_cols, D), device=DEV, generator=gen)
    ref = _sddmm_ref(g, G, X)
    got = ops.sddmm(g, G, X, alpha=0.75)
    _rel_close(got, 0.75 * ref, 1e-5)
    assert torch.equal(ops.sddmm(g, G, X, alpha=0.75), got)                  # bit-stable
    base = torch.randn(g.nnz, device=DEV, generator=gen)
    acc = ops.sddmm(g, G, X, alpha=-2.0, out=base.clone(), accumulate=True)
    _rel_close(acc, base.double() - 2.0 * ref, 1e-5)


def test_sddmm_column_blocked_rows():
    """A user table the plan cuts into L2-sized column blocks (Graph._plan sizes them at 256 bytes per row: above 100 MB
    from ~400 k users): the item rows gather from it block by block, so they have several segments each."""
    from recad_b200 import ops
    nU, nI, nE, D = 600_000, 5_000, 1_000_000, 128
    gen = torch.Generator(device=DEV).manual_seed(3)
    eu = torch.randint(0, nU, (nE,), device=DEV, generator=gen)
    ei = torch.randint(0, nI, (nE,), device=DEV, generator=gen)
    g = ops.Graph.from_edges(eu, ei, nU, nI)
    assert ops.auto_col_blocks(nU) > 1 and g.n_mrow > 0
    G = torch.randn((g.n_rows, D), device=DEV, generator=gen)
    X = torch.randn((g.n_cols, D), device=DEV, generator=gen)
    got = ops.sddmm(g, G, X)
    _rel_close(got, _sddmm_ref(g, G, X), 1e-5)
    assert torch.equal(ops.sddmm(g, G, X), got)


# ------------------------------------------------------------------ LightGCN edge values
def _lightgcn(graph, D, L, seed=0, n_users=U, n_items=I, **kw):
    from recad_b200 import model
    m = model.from_config("victim", "lightgcn", latent_dim_rec=D, lightGCN_n_layers=L, device=torch.device(DEV), **kw).I(
        dataset=StubData(graph, n_users, n_items))
    rng = np.random.default_rng(seed)
    m.embedding_user.weight.data.copy_(torch.as_tensor(rng.normal(0, 0.1, (n_users, D)), dtype=torch.float32))
    m.embedding_item.weight.data.copy_(torch.as_tensor(rng.normal(0, 0.1, (n_items, D)), dtype=torch.float32))
    m.invalidate()
    return m


def _oracle(graph, m, L, u, i, w, vals):
    """float64 autograd: layers as index_add of vals[:, None] * X[cols], layer mean, dot scores, weighted sum.  Returns
    (scores, d vals, d user table, d item table); `vals` may be a float64 leaf of a longer chain (its .grad is left)."""
    nU = m.num_users
    rows, cols = _rows(graph), graph.colidx.long()
    v = vals if vals.dtype == torch.float64 else vals.detach().double().requires_grad_(True)
    eu = m.embedding_user.weight.detach().double().clone().requires_grad_(True)
    ei = m.embedding_item.weight.detach().double().clone().requires_grad_(True)
    x = torch.cat([eu, ei])
    acc = x
    for _ in range(L):
        x = torch.zeros_like(x).index_add(0, rows, v[:, None] * x[cols])
        acc = acc + x
    O = acc / (L + 1)
    s = (O[u] * O[nU + i]).sum(1)
    (w.double() * s).sum().backward()
    gv = v.grad if v.grad is not None else torch.zeros_like(v)
    return s.detach(), gv, eu.grad, ei.grad


@pytest.mark.parametrize("D", [4, 64, 128])
@pytest.mark.parametrize("L", [0, 1, 3])
def test_edge_value_gradient_matches_float64(dev_graph, D, L):
    m = _lightgcn(dev_graph, D, L, seed=D + L)
    u, i, w = _pairs(D * 10 + L, 10000)
    v = dev_graph.vals.clone().requires_grad_(True)
    s = m(u, i, edge_values=v)
    (w * s).sum().backward()
    s_ref, gv, _, _ = _oracle(dev_graph, m, L, u, i, w, v)
    _rel_close(s, s_ref, 1e-5)
    if L == 0:
        assert torch.equal(v.grad, torch.zeros_like(v))
    else:
        _rel_close(v.grad, gv, 1e-5)
    assert m.embedding_user.weight.grad is None                # the tables were not asked for


@pytest.mark.parametrize("L", [1, 2, 3])
@pytest.mark.parametrize("asymmetric", [False, True])
def test_edge_values_and_tables_together(dev_graph, L, asymmetric):
    """With the tables requiring grad too; asymmetric: each entry scaled by an independent factor in [0.5, 2], so that
    the backward must use values[T] for A^T."""
    m = _lightgcn(dev_graph, 64, L, seed=60 + L)
    m.requires_grad_(True)
    vals = dev_graph.vals.clone()
    if asymmetric:
        gen = torch.Generator(device=DEV).manual_seed(L)
        vals = vals * (0.5 + 1.5 * torch.rand(vals.shape, device=DEV, generator=gen))
    v = vals.requires_grad_(True)
    u, i, w = _pairs(70 + L, 10000)
    s = m(u, i, edge_values=v)
    (w * s).sum().backward()
    s_ref, gv, gu, gi = _oracle(dev_graph, m, L, u, i, w, v)
    _rel_close(s, s_ref, 1e-5)
    _rel_close(v.grad, gv, 1e-5)
    _rel_close(m.embedding_user.weight.grad, gu, 1e-5)
    _rel_close(m.embedding_item.weight.grad, gi, 1e-5)


def test_injected_fake_users_entries(dev_graph):
    """Fake users appended with append_users: the gradient of their interactions, read through entry_index at k and T[k]."""
    rng = np.random.default_rng(5)
    F = 4
    items = [np.sort(rng.choice(I, 12, replace=False)) for _ in range(F)]
    fake_rowptr = torch.as_tensor(np.concatenate([[0], np.cumsum([len(x) for x in items])]), device=DEV)
    fake_items = torch.as_tensor(np.concatenate(items), device=DEV)
    g = dev_graph.append_users(U, I, fake_rowptr, fake_items)
    nU = U + F
    m = _lightgcn(g, 32, 2, seed=9, n_users=nU)
    v = g.vals.clone().requires_grad_(True)
    u, i, w = _pairs(91, 10000, nU, I)
    (w * m(u, i, edge_values=v)).sum().backward()
    _, gv, _, _ = _oracle(g, m, 2, u, i, w, v)
    fu = torch.as_tensor(np.repeat(np.arange(U, nU), [len(x) for x in items]), device=DEV)
    k = g.entry_index(fu, nU + fake_items.long())
    kt = g.transpose_permutation()[k]
    assert torch.equal(g.entry_index(nU + fake_items.long(), fu), kt)
    _rel_close(v.grad[k], gv[k], 1e-5)
    _rel_close(v.grad[kt], gv[kt], 1e-5)
    _rel_close(v.grad, gv, 1e-5)
    assert v.grad[k].abs().sum() > 0


# ------------------------------------------------------------------ normalisation
def _norm_ref(graph, w64):
    rows, cols = _rows(graph), graph.colidx.long()
    s = torch.zeros(graph.n_rows, dtype=torch.float64, device=DEV).index_add(0, rows, w64)
    d = (s + 1e-14) ** -0.5
    return d[rows] * w64 * d[cols]


def test_normalized_values_forward_and_backward(dev_graph):
    from recad_b200 import ops
    g = dev_graph
    assert torch.equal(ops.normalized_values(g, g.mult), g.vals)
    gen = torch.Generator(device=DEV).manual_seed(11)
    w = (0.2 + 3.0 * torch.rand(g.nnz, device=DEV, generator=gen)).requires_grad_(True)
    vals = ops.normalized_values(g, w)
    w64 = w.detach().double().requires_grad_(True)
    ref = _norm_ref(g, w64)
    assert ((vals.detach().double() - ref).abs() <= 1e-6 * ref.abs()).all()
    gv = torch.randn(g.nnz, device=DEV, generator=gen)
    (gv * vals).sum().backward()
    (gv.double() * ref).sum().backward()
    _rel_close(w.grad, w64.grad, 1e-5)
    first = w.grad.clone()
    w.grad = None
    (gv * ops.normalized_values(g, w)).sum().backward()
    assert torch.equal(w.grad, first)                          # deterministic


def test_weights_through_normalisation_and_lightgcn(dev_graph):
    from recad_b200 import ops
    g, L = dev_graph, 3
    m = _lightgcn(g, 64, L, seed=12)
    gen = torch.Generator(device=DEV).manual_seed(12)
    w = (0.5 + 1.5 * torch.rand(g.nnz, device=DEV, generator=gen)).requires_grad_(True)
    u, i, wt = _pairs(121, 10000)
    (wt * m(u, i, edge_values=ops.normalized_values(g, w))).sum().backward()
    w64 = w.detach().double().requires_grad_(True)
    _oracle(g, m, L, u, i, wt, _norm_ref(g, w64))
    _rel_close(w.grad, w64.grad, 1e-5)


# ------------------------------------------------------------------ behaviour
def test_same_values_give_the_plain_forward_bit_for_bit(dev_graph):
    m = _lightgcn(dev_graph, 64, 3, seed=13)
    u, i, _ = _pairs(131, 5000)
    with torch.no_grad():
        plain = m(u, i)
        assert torch.equal(m(u, i, edge_values=dev_graph.vals.clone()), plain)
    s = m(u, i, edge_values=dev_graph.vals.clone().requires_grad_(True))
    assert s.grad_fn is not None and torch.equal(s.detach(), plain)
    ou, oi = m.computer(edge_values=dev_graph.vals.clone())
    assert ou.grad_fn is None and torch.equal(torch.cat([ou, oi]), m.O)


def test_no_grad_fn_without_a_gradient_to_compute(dev_graph):
    m = _lightgcn(dev_graph, 32, 2, seed=14)
    u, i, _ = _pairs(141, 100)
    assert m(u, i, edge_values=dev_graph.vals.clone()).grad_fn is None
    with torch.no_grad():
        assert m(u, i, edge_values=dev_graph.vals.clone().requires_grad_(True)).grad_fn is None
    assert m(u, i, edge_values=dev_graph.vals.clone().requires_grad_(True)).grad_fn is not None


def test_perturbed_forward_leaves_the_cached_propagation_alone(dev_graph):
    m = _lightgcn(dev_graph, 64, 3, seed=15)
    u, i, _ = _pairs(151, 3000)
    users = torch.arange(64, device=DEV)
    rowptr = torch.zeros(U + 1, dtype=torch.int64, device=DEV)
    col = torch.zeros(1, dtype=torch.int32, device=DEV)
    with torch.no_grad():
        before = m(u, i)
    rank_before = m.full_rank(users, [0, 1], 10, rowptr, col)
    v = (dev_graph.vals * 1.5).requires_grad_(True)
    pert = m(u, i, edge_values=v)
    pert.sum().backward()
    with torch.no_grad():
        assert not torch.equal(m(u, i, edge_values=v), before)
        after = m(u, i)
    rank_after = m.full_rank(users, [0, 1], 10, rowptr, col)
    assert torch.equal(after, before)
    assert all(torch.equal(a, b) for a, b in zip(rank_before[:4], rank_after[:4]))


def test_backward_is_bit_stable_accumulates_and_keeps_its_own_values(dev_graph):
    m = _lightgcn(dev_graph, 64, 3, seed=16)
    m.requires_grad_(True)
    u, i, w = _pairs(161, 20000)
    v = dev_graph.vals.clone().requires_grad_(True)
    (w * m(u, i, edge_values=v)).sum().backward()
    first_v, first_u = v.grad.clone(), m.embedding_user.weight.grad.clone()
    v.grad = None
    m.zero_grad()
    (w * m(u, i, edge_values=v)).sum().backward()
    assert torch.equal(v.grad, first_v) and torch.equal(m.embedding_user.weight.grad, first_u)
    (w * m(u, i, edge_values=v)).sum().backward()
    assert torch.equal(v.grad, 2 * first_v) and torch.equal(m.embedding_user.weight.grad, 2 * first_u)
    # a forward with other values between a forward and its backward
    v.grad = None
    m.zero_grad()
    s = m(u, i, edge_values=v)
    other = (dev_graph.vals * 0.5).requires_grad_(True)
    s_other = m(u, i, edge_values=other)
    (w * s).sum().backward()
    assert torch.equal(v.grad, first_v) and torch.equal(m.embedding_user.weight.grad, first_u)
    del s_other


# ------------------------------------------------------------------ errors
def test_bad_edge_values_raise(dev_graph):
    from recad_b200 import ops
    m = _lightgcn(dev_graph, 32, 2, seed=17)
    u, i, _ = _pairs(171, 10)
    bad = [dev_graph.vals[:-1].clone(), dev_graph.vals.double(), dev_graph.vals.cpu(), dev_graph.vals.view(-1, 1)]
    if torch.cuda.device_count() > 1:
        bad.append(dev_graph.vals.to("cuda:1"))
    for v in bad:
        with pytest.raises(ops.RecadError):
            m(u, i, edge_values=v)
        with pytest.raises(ops.RecadError):
            m.computer(edge_values=v)
    with pytest.raises(ops.RecadError):
        ops.normalized_values(dev_graph, dev_graph.mult.double())


def test_edge_values_under_training_dropout_raise(dev_graph):
    from recad_b200 import ops
    m = _lightgcn(dev_graph, 32, 2, seed=18, dropout=True, keep_prob=0.6)
    m.train()
    u, i, _ = _pairs(181, 10)
    with pytest.raises(ops.RecadError):
        m(u, i, edge_values=dev_graph.vals.clone())
    m.eval()
    with torch.no_grad():
        assert torch.equal(m(u, i, edge_values=dev_graph.vals.clone()), m(u, i))


def test_normalized_values_and_entry_index_errors(dev_graph):
    from recad_b200 import ops
    g = dev_graph
    rect = ops.Graph.from_csr(g.rowptr[:U + 1].clone(), g.colidx[:int(g.rowptr[U])].clone(), g.vals[:int(g.rowptr[U])].clone(),
                              g.n_cols)
    with pytest.raises(ops.RecadError):
        ops.normalized_values(rect, rect.vals)
    r = int(torch.nonzero(g.rowptr[1:] > g.rowptr[:-1])[0])   # first row with a stored entry
    lo, hi = int(g.rowptr[r]), int(g.rowptr[r + 1])
    stored_c = int(g.colidx[lo])
    assert int(g.entry_index([r], [stored_c])[0]) == lo
    row_cols = set(g.colidx[lo:hi].tolist())
    missing = next(c for c in range(g.n_cols) if c not in row_cols)
    with pytest.raises(ops.RecadError):
        g.entry_index([r], [missing])
    with pytest.raises(ops.RecadError):
        g.entry_index([0], [0])                               # user-user: never stored
    with pytest.raises(ops.RecadError):
        g.entry_index([g.n_rows], [0])
