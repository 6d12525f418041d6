"""Mixed second derivatives of the LightGCN training loss with respect to edge values (loss_mixed_values) and the
hypergradient of an objective with respect to interaction weights (influence.interaction_hypergradient).  Checked against
float64 torch autograd over an index_add SpMM of a leaf value vector (twice differentiable), a dense float64 solve, the
influence API's sign convention, and central finite differences of a retrained (Newton-minimised) float64 model."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.test_gpu_autograd import DEV, I, U, StubData, _lightgcn, _mf, _rel_close, dev_graph  # noqa: F401
from tests.test_gpu_edge_grad import _lightgcn as _lightgcn_n
from tests.test_gpu_edge_grad import _rows
from tests.test_gpu_hvp import _triples, _vectors

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------ float64 references
def _norm64(rows, cols, w, N):
    s = torch.zeros(N, dtype=torch.float64, device=w.device).index_add(0, rows, w)
    d = (s + 1e-14) ** -0.5
    return d[rows] * w * d[cols]


def _prop64(rows, cols, v, E, L):
    x, acc = E, E
    for _ in range(L):
        x = torch.zeros_like(x).index_add(0, rows, v[:, None] * x[cols])
        acc = acc + x
    return acc / (L + 1)


def _loss64(rows, cols, v, E, nu, L, u, p, q, lam, omega=None):
    """The weighted training loss (1/n) sum_b omega_b l_b(E; v) in float64."""
    O = _prop64(rows, cols, v, E, L)
    x = (O[u] * O[nu + q]).sum(1) - (O[u] * O[nu + p]).sum(1)
    reg = E[u].pow(2).sum(1) + E[nu + p].pow(2).sum(1) + E[nu + q].pow(2).sum(1)
    lb = F.softplus(x) + lam * 0.5 * reg
    return (lb if omega is None else omega * lb).mean()


def _batch_cols(batch):
    return batch["users"], batch["positive_items"], batch["negative_items"]


def _mixed64(graph, m, L, batch, S):
    """grad_v <grad_E L, S> with v a float64 leaf at the graph's values."""
    rows, cols = _rows(graph), graph.colidx.long()
    v = graph.vals.double().requires_grad_(True)
    E = torch.cat([m.embedding_user.weight, m.embedding_item.weight]).detach().double().requires_grad_(True)
    loss = _loss64(rows, cols, v, E, m.num_users, L, *_batch_cols(batch), float(m.config["lambda"]))
    gE, = torch.autograd.grad(loss, E, create_graph=True)
    return torch.autograd.grad((gE * torch.cat(S).double()).sum(), v)[0]


def _check_mixed(graph, m, L, batch, seed):
    S = _vectors(seed, [(m.num_users, m.latent_dim), (m.num_items, m.latent_dim)])
    got = m.loss_mixed_values(batch, S)
    assert got.dtype == torch.float32 and tuple(got.shape) == (graph.nnz,)
    if L == 0:
        assert torch.equal(got, torch.zeros_like(got))
        return
    ref = _mixed64(graph, m, L, batch, S)
    assert ref.abs().max() > 0
    _rel_close(got, ref, 1e-5)


# ------------------------------------------------------------------ loss_mixed_values
@pytest.mark.parametrize("D", [4, 64, 128])
@pytest.mark.parametrize("L", [0, 1, 3])
def test_loss_mixed_values_matches_float64_autograd(dev_graph, D, L):
    """10000 triples over 512 users / 511 items: every id repeats, as user, positive and negative."""
    m = _lightgcn(dev_graph, D, L, seed=D + L)
    _check_mixed(dev_graph, m, L, _triples(D * 10 + L, 10000), D + 7 * L)


def test_loss_mixed_values_where_margins_exceed_the_softplus_threshold(dev_graph):
    m = _lightgcn(dev_graph, 64, 1, seed=4)
    m.embedding_user.weight.data.mul_(30.0)
    m.embedding_item.weight.data.mul_(30.0)
    m.invalidate()
    batch = _triples(19, 10000)
    with torch.no_grad():
        O = _prop64(_rows(dev_graph), dev_graph.colidx.long(), dev_graph.vals.double(), m.E.double(), 1)
        u, p, q = _batch_cols(batch)
        x = (O[u] * O[U + q]).sum(1) - (O[u] * O[U + p]).sum(1)
    assert (x > 20).float().mean() > 0.2 and (x.abs() <= 20).float().mean() > 0.05
    _check_mixed(dev_graph, m, 1, batch, 20)


def test_loss_mixed_values_on_a_skewed_graph_with_a_million_triples():
    """The graph and batch of the HVP test: one item collects ~100 k pairs."""
    from recad_b200 import model, ops
    nu, ni, D, L, n = 40000, 4000, 64, 2, 1 << 20
    rng = np.random.default_rng(23)
    pop = 1.0 / np.arange(1, ni + 1) ** 1.1
    pop[0] = pop[1:].sum() / 4
    pop /= pop.sum()
    eu = np.repeat(np.arange(nu), 12)
    ei = rng.choice(ni, eu.size, p=pop)
    key = np.unique(eu.astype(np.int64) * ni + ei)
    eu, ei = key // ni, key % ni
    g = ops.Graph.from_edges(torch.as_tensor(eu, device=DEV), torch.as_tensor(ei, device=DEV), nu, ni)

    class Data(StubData):
        def info_describe(self):
            return {"n_users": nu, "n_items": ni, "graph": self.graph, "train_dict": None}

    m = model.from_config("victim", "lightgcn", latent_dim_rec=D, lightGCN_n_layers=L, device=torch.device(DEV)).I(
        dataset=Data(g))
    m.embedding_user.weight.data.copy_(torch.as_tensor(rng.normal(0, 0.1, (nu, D)), dtype=torch.float32))
    m.embedding_item.weight.data.copy_(torch.as_tensor(rng.normal(0, 0.1, (ni, D)), dtype=torch.float32))
    m.invalidate()
    pick = rng.integers(0, eu.size, n)
    batch = {"users": torch.as_tensor(eu[pick], device=DEV), "positive_items": torch.as_tensor(ei[pick], device=DEV),
             "negative_items": torch.as_tensor(rng.integers(0, ni, n), device=DEV)}
    assert int((batch["positive_items"] == 0).sum()) > 50_000
    _check_mixed(g, m, L, batch, 24)


def test_loss_mixed_values_on_multi_segment_rows_with_fake_users():
    """seg_len = 32 and fake users appended by append_users: item rows and user 0 span several SpMM segments."""
    from recad_b200 import ops
    rng = np.random.default_rng(7)
    nu, ni, F_ = 700, 300, 5
    u = np.concatenate([np.zeros(1500, np.int64), rng.integers(0, nu, 18500)])
    i = rng.integers(0, ni, 20000)
    g = ops.Graph.from_edges(torch.as_tensor(u, device=DEV), torch.as_tensor(i, device=DEV), nu, ni, seg_len=32)
    items = [np.sort(rng.choice(ni, 40, replace=False)) for _ in range(F_)]
    fake_rowptr = torch.as_tensor(np.concatenate([[0], np.cumsum([len(x) for x in items])]), device=DEV)
    g = g.append_users(nu, ni, fake_rowptr, torch.as_tensor(np.concatenate(items), device=DEV))
    assert g.n_mrow > 0
    m = _lightgcn_n(g, 32, 2, seed=9, n_users=nu + F_, n_items=ni)
    _check_mixed(g, m, 2, _triples(31, 10000, nu + F_, ni), 32)


# ------------------------------------------------------------------ hypergradient
def _stored_triples(graph, n_users, n_items, seed, n_stored, n_free):
    """Rows whose positive is a stored interaction (k(b) exists), then rows with random positives (mostly not stored)."""
    rng = np.random.default_rng(seed)
    rows = _rows(graph).cpu().numpy()
    cols = graph.colidx.long().cpu().numpy()
    user_side = np.nonzero(rows < n_users)[0]
    pick = rng.choice(user_side, n_stored)
    u = np.concatenate([rows[pick], rng.integers(0, n_users, n_free)])
    p = np.concatenate([cols[pick] - n_users, rng.integers(0, n_items, n_free)])
    q = rng.integers(0, n_items, n_stored + n_free)
    return {k: torch.as_tensor(c, device=DEV) for k, c in zip(("users", "positive_items", "negative_items"), (u, p, q))}


def _target_objective(m, item, n_users=64):
    users = torch.arange(n_users, device=DEV)
    return lambda ev: m(users, torch.full_like(users, item), edge_values=ev).sum()


def _row_entries(graph, batch, nu):
    return graph.entry_index(batch["users"], nu + batch["positive_items"], missing=-1)


def test_hypergradient_matches_a_dense_float64_solve(dev_graph):
    """D = 4 on the dev graph: 4092 parameters, a dense float64 Hessian from torch.autograd.functional.hessian, the same
    damping rule as the influence test; direct and M^T s by float64 autograd on the weighted loss."""
    from recad_b200 import influence
    D, L = 4, 2
    g = dev_graph
    m = _lightgcn(g, D, L, seed=12)
    lam = float(m.config["lambda"])
    batch = _stored_triples(g, U, I, 41, 1500, 500)
    rows, cols = _rows(g), g.colidx.long()
    u, p, q = _batch_cols(batch)
    kb = _row_entries(g, batch, U)
    assert int((kb >= 0).sum()) >= 1500 and int((kb < 0).sum()) > 0
    mult = g.mult.double()
    E0 = m.E.detach().double().reshape(-1)
    w0 = g.mult.double()

    def omega(w):
        return torch.where(kb >= 0, w[kb.clamp(min=0)] / mult[kb.clamp(min=0)], torch.ones_like(kb, dtype=torch.float64))

    def loss(flat, w):
        return _loss64(rows, cols, _norm64(rows, cols, w, U + I), flat.view(U + I, D), U, L, u, p, q, lam, omega(w))

    users = torch.arange(64, device=DEV)

    def J(flat, w):
        O = _prop64(rows, cols, _norm64(rows, cols, w, U + I), flat.view(U + I, D), L)
        return (O[users] * O[U + 7]).sum()

    H = torch.autograd.functional.hessian(lambda f: loss(f, w0), E0)
    H = 0.5 * (H + H.T)
    ev = torch.linalg.eigvalsh(H)
    damping = max(0.0, -float(ev[0])) + 0.1 * float(ev[-1])
    Ef, wl = E0.clone().requires_grad_(True), w0.clone().requires_grad_(True)
    gJ_E, direct_ref = torch.autograd.grad(J(Ef, wl), (Ef, wl))
    s_ref = torch.linalg.solve(H + damping * torch.eye(H.shape[0], dtype=H.dtype, device=DEV), gJ_E)
    Ef, wl = E0.clone().requires_grad_(True), w0.clone().requires_grad_(True)
    gE, = torch.autograd.grad(loss(Ef, wl), Ef, create_graph=True)
    mts_ref, = torch.autograd.grad((gE * s_ref).sum(), wl)
    values_ref = direct_ref - mts_ref

    hg = influence.interaction_hypergradient(m, batch, _target_objective(m, 7), damping, max_iter=1000, rtol=1e-7)
    assert hg.residual < 1e-7 and hg.iterations < 1000
    for t in (hg.values, hg.direct, hg.implicit):
        assert t.dtype == torch.float32 and tuple(t.shape) == (g.nnz,)
    assert torch.equal(hg.values, hg.direct - hg.implicit)
    _rel_close(torch.cat([x.reshape(-1) for x in hg.s]), s_ref, 1e-4)
    _rel_close(hg.direct, direct_ref, 1e-4)
    _rel_close(hg.implicit, mts_ref, 1e-4)
    _rel_close(hg.values, values_ref, 1e-4)
    # per interaction: both entries carry one weight
    k = torch.nonzero(rows < U).squeeze(1)
    T = g.transpose_permutation()
    _rel_close(hg.values[k] + hg.values[T[k]], values_ref[k] + values_ref[T[k]], 1e-4)


def test_sample_part_matches_the_influence_values(dev_graph):
    """values' sample part = -(1 / (n mult_k)) sum over the rows with k(b) = k of sample_influence values, from the same
    solve; rows whose positive pair is not stored contribute nothing and raise nothing."""
    from recad_b200 import influence, ops
    g = dev_graph
    m = _lightgcn(g, 16, 2, seed=13)
    batch = _stored_triples(g, U, I, 43, 3000, 3000)
    n = batch["users"].numel()
    kb = _row_entries(g, batch, U)
    assert int((kb < 0).sum()) > 1000
    obj = _target_objective(m, 11)
    damping = 1e-2
    hg = influence.interaction_hypergradient(m, batch, obj, damping, max_iter=50, rtol=1e-6)
    # the objective's table gradient exactly as interaction_hypergradient takes it, then the same solve
    w = g.mult.clone().requires_grad_(True)
    m.requires_grad_(True)
    gE = torch.autograd.grad(obj(ops.normalized_values(g, w)), list(m.parameters()))
    m.requires_grad_(False)
    inf = influence.sample_influence(m, batch, gE, damping, max_iter=50, rtol=1e-6)
    assert inf.iterations == hg.iterations and all(torch.equal(a, b) for a, b in zip(inf.s, hg.s))
    w = g.mult.clone().requires_grad_(True)
    graph_part, = torch.autograd.grad(ops.normalized_values(g, w), w, m.loss_mixed_values(batch, hg.s))
    sample_contribution = -(hg.implicit - graph_part)
    sums = torch.zeros(g.nnz, dtype=torch.float64).index_add(0, kb[kb >= 0].cpu(), inf.values[kb >= 0].double().cpu())
    ref = -(sums / (n * g.mult.double().cpu()))
    _rel_close(sample_contribution.cpu(), ref, 1e-5)
    assert torch.equal(ref[torch.isin(torch.arange(g.nnz), kb.cpu(), invert=True)],
                       torch.zeros(g.nnz - int(torch.unique(kb[kb >= 0]).numel()), dtype=torch.float64))


# ------------------------------------------------------------------ finite differences
def _newton(loss, E, tol=1e-13, lbfgs=False):
    """Minimise loss(flat E) in float64: L-BFGS to the basin (first call), then Newton steps with a least-squares solve (the
    rotations E -> E R leave the loss unchanged, so the Hessian has a null space)."""
    E = E.clone()
    if lbfgs:
        E.requires_grad_(True)
        opt = torch.optim.LBFGS([E], lr=1, max_iter=2000, tolerance_grad=1e-9, tolerance_change=1e-16, history_size=50,
                                line_search_fn="strong_wolfe")

        def closure():
            opt.zero_grad()
            f = loss(E)
            f.backward()
            return f
        opt.step(closure)
        E = E.detach()
    for _ in range(30):
        g = torch.autograd.functional.jacobian(loss, E)
        if float(g.norm()) < tol:
            return E
        H = torch.autograd.functional.hessian(loss, E)
        E = E - torch.linalg.lstsq(H, g, rcond=1e-9, driver="gelsd").solution
    raise AssertionError(f"Newton did not converge: |grad| = {float(g.norm()):.3e}")


def test_hypergradient_signs_by_finite_differences():
    """32 users x 20 items plus 2 fake users, D = 4, L = 2, lambda = 0.1 (a well-conditioned minimiser up to rotations).
    Retrain by Newton (|grad| < 1e-13) at w and w +- eps e_k; the central differences of J(E*(w), v(w)) match the closed form (damping 0,
    pseudo-inverse on the rotation null space), and the CUDA hypergradient at the minimiser matches both."""
    from recad_b200 import influence, ops
    rng = np.random.default_rng(3)
    nu, ni, D, L, lam, F_ = 32, 20, 4, 2, 0.1, 2
    eu, ei = rng.integers(0, nu, 150), rng.integers(0, ni, 150)
    g = ops.Graph.from_edges(torch.as_tensor(eu, device=DEV), torch.as_tensor(ei, device=DEV), nu, ni)
    fake = [np.array([1, 4, 9]), np.array([0, 4, 17, 19])]
    g = g.append_users(nu, ni, torch.as_tensor([0, 3, 7], device=DEV), torch.as_tensor(np.concatenate(fake), device=DEV))
    NU, N = nu + F_, nu + F_ + ni
    m = _lightgcn_n(g, D, L, seed=5, n_users=NU, n_items=ni)
    m.config["lambda"] = lam
    batch = _stored_triples(g, NU, ni, 44, 240, 60)
    batch["users"][:5] = nu + 1                                  # the second fake user's edge (nu + 1, item 17) is k(b)
    batch["positive_items"][:5] = 17

    cpu = torch.device("cpu")
    rows, cols = _rows(g).to(cpu), g.colidx.long().to(cpu)
    mult = g.mult.double().to(cpu)
    u, p, q = (t.to(cpu) for t in _batch_cols(batch))
    kb = _row_entries(g, batch, NU).to(cpu)
    users = torch.arange(16)

    def omega(w):
        return torch.where(kb >= 0, w[kb.clamp(min=0)] / mult[kb.clamp(min=0)], torch.ones_like(kb, dtype=torch.float64))

    def loss(flat, w):
        return _loss64(rows, cols, _norm64(rows, cols, w, N), flat.view(N, D), NU, L, u, p, q, lam, omega(w))

    def J(flat, w):
        O = _prop64(rows, cols, _norm64(rows, cols, w, N), flat.view(N, D), L)
        return (O[users] * O[NU + 4]).sum()

    w0 = mult.clone()
    E_star = _newton(lambda e: loss(e, w0), torch.as_tensor(rng.normal(0, 0.3, N * D)), lbfgs=True)
    # closed form, damping 0
    H = torch.autograd.functional.hessian(lambda e: loss(e, w0), E_star)
    ev = torch.linalg.eigvalsh(0.5 * (H + H.T))
    assert float(ev[6]) > 1e-3 * float(ev[-1]) and float(ev[0]) > -1e-9           # six rotations, then well conditioned
    Ef, wl = E_star.clone().requires_grad_(True), w0.clone().requires_grad_(True)
    gJ_E, direct = torch.autograd.grad(J(Ef, wl), (Ef, wl))
    s = torch.linalg.lstsq(H, gJ_E, rcond=1e-9, driver="gelsd").solution
    Ef, wl = E_star.clone().requires_grad_(True), w0.clone().requires_grad_(True)
    gE, = torch.autograd.grad(loss(Ef, wl), Ef, create_graph=True)
    closed = direct - torch.autograd.grad((gE * s).sum(), wl)[0]

    T = g.transpose_permutation().to(cpu)
    k_fake = int(g.entry_index(torch.tensor([nu + 1]), torch.tensor([NU + 17]))[0])
    k_row = int(kb[100])
    k_item = int(torch.nonzero(rows >= NU)[7])
    check = [k_fake, int(T[k_fake]), k_row, k_item]
    assert k_row >= 0 and k_fake in kb.tolist()
    eps = 1e-3
    for k in check:
        Js = []
        for sgn in (1, -1):
            w = w0.clone()
            w[k] += sgn * eps
            Js.append(float(J(_newton(lambda e: loss(e, w), E_star), w)))
        fd = (Js[0] - Js[1]) / (2 * eps)
        assert abs(fd - float(closed[k])) <= 1e-5 * float(closed.abs().max()), (k, fd, float(closed[k]))

    m.embedding_user.weight.data.copy_(E_star.view(N, D)[:NU].float())
    m.embedding_item.weight.data.copy_(E_star.view(N, D)[NU:].float())
    m.invalidate()
    obj_users = users.to(DEV)
    hg = influence.interaction_hypergradient(m, batch, lambda ev: m(obj_users, torch.full_like(obj_users, 4),
                                                                  edge_values=ev).sum(),
                                             damping=1e-6 * float(ev[-1]), max_iter=2000, rtol=1e-8)
    _rel_close(hg.values.cpu(), closed, 1e-3)


# ------------------------------------------------------------------ behaviour
def test_two_calls_give_the_same_bits_and_leave_the_model_alone(dev_graph):
    from recad_b200 import influence
    m = _lightgcn(dev_graph, 64, 3, seed=8)
    m.computer()
    m.embedding_item.weight.requires_grad_(True)                   # a flag the hypergradient must restore
    before = [t.clone() for t in (m.E, m.m, m.v, m.O, m.loss_acc)] + [m._steps, m._O_valid, m._O_version]
    batch = _stored_triples(dev_graph, U, I, 33, 10000, 10000)
    S = _vectors(34, [(U, 64), (I, 64)])
    assert torch.equal(m.loss_mixed_values(batch, S), m.loss_mixed_values(batch, S))
    obj = _target_objective(m, 3)
    a = influence.interaction_hypergradient(m, batch, obj, 0.05, max_iter=8, rtol=1e-30)
    b = influence.interaction_hypergradient(m, batch, obj, 0.05, max_iter=8, rtol=1e-30)
    assert a.iterations == b.iterations == 8
    assert all(torch.equal(x, y) for x, y in zip(a[:3], b[:3])) and all(torch.equal(x, y) for x, y in zip(a.s, b.s))
    assert not m.embedding_user.weight.requires_grad and m.embedding_item.weight.requires_grad
    m.embedding_item.weight.requires_grad_(False)
    after = [m.E, m.m, m.v, m.O, m.loss_acc, m._steps, m._O_valid, m._O_version]
    assert all(torch.equal(x, y) if isinstance(x, torch.Tensor) else x == y for x, y in zip(before, after))


def test_error_paths(dev_graph):
    from recad_b200 import influence
    from recad_b200.ops import RecadError
    m = _lightgcn(dev_graph, 16, 2, seed=10)
    batch = _triples(37, 100)
    v = _vectors(38, [(U, 16), (I, 16)])
    fn = m.loss_mixed_values
    with pytest.raises(RecadError):
        fn({k: t.cpu() for k, t in batch.items()}, v)                               # CPU ids
    with pytest.raises(RecadError):
        fn({k: t.int() for k, t in batch.items()}, v)                               # int32 ids
    with pytest.raises(RecadError):
        fn(dict(batch, users=batch["users"][:50]), v)                               # ragged columns
    with pytest.raises(RecadError):
        fn(batch, (v[0].cpu(), v[1]))                                               # CPU vector
    with pytest.raises(RecadError):
        fn(batch, (v[0].double(), v[1]))                                            # float64 vector
    with pytest.raises(RecadError):
        fn(batch, (v[0][:, :8].contiguous(), v[1]))                                 # wrong shape
    with pytest.raises(RecadError, match="out of range"):
        fn(dict(batch, negative_items=torch.full_like(batch["negative_items"], I)), v)
    with pytest.raises(RecadError, match="out of range"):
        fn(dict(batch, users=torch.full_like(batch["users"], -1)), v)
    with pytest.raises(RecadError, match="out of range"):
        influence.interaction_hypergradient(m, dict(batch, positive_items=torch.full_like(batch["users"], I)),
                                            _target_objective(m, 3), 0.1, max_iter=2)
    d = _lightgcn(dev_graph, 16, 2, seed=10, dropout=True, keep_prob=0.6)
    d.train()
    with pytest.raises(RecadError, match="dropout"):
        d.loss_mixed_values(batch, v)
    with pytest.raises(RecadError, match="dropout"):
        influence.interaction_hypergradient(d, batch, _target_objective(d, 3), 0.1, max_iter=2)
    assert not any(p.requires_grad for p in d.parameters())
    d.eval()
    d.loss_mixed_values(batch, v)                                                   # no mask in eval mode
    with pytest.raises(RecadError, match="LightGCN"):
        influence.interaction_hypergradient(_mf(16, seed=11), batch, lambda ev: ev.sum(), 0.1)
    with pytest.raises(RecadError, match="not a stored entry"):
        dev_graph.entry_index(torch.tensor([0], device=DEV), torch.tensor([1], device=DEV))   # the default still raises
    k = dev_graph.entry_index(torch.tensor([0], device=DEV), torch.tensor([1], device=DEV), missing=-1)
    assert k.tolist() == [-1]
