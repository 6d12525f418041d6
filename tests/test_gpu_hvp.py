"""Second order: Hessian-vector products of the LightGCN (BPR) and MF (BCE) training losses, per-row directional
derivatives, and the influence of training rows on an objective.  Checked against float64 torch autograd on the same GPU
(double backward through the graph's own normalised CSR) and, for influence, against a dense float64 Hessian."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.test_gpu_autograd import DEV, I, U, StubData, _lightgcn, _mf, _rel_close, dev_graph  # noqa: F401

pytestmark = pytest.mark.gpu


def _triples(seed, n, n_users=U, n_items=I):
    rng = np.random.default_rng(seed)
    cols = [rng.integers(0, k, n) for k in (n_users, n_items, n_items)]
    return {k: torch.as_tensor(c, device=DEV) for k, c in zip(("users", "positive_items", "negative_items"), cols)}


def _vectors(seed, shapes):
    rng = np.random.default_rng(seed)
    return tuple(torch.as_tensor(rng.normal(size=s), dtype=torch.float32, device=DEV) for s in shapes)


def _csr64(graph):
    N = graph.n_rows
    return torch.sparse_csr_tensor(graph.rowptr, graph.colidx.long(), graph.vals.double(), size=(N, N))


def _bpr_losses64(A, eu, ei, L, batch, lam):
    """The per-sample losses l_b = softplus(x_b) + lam * 0.5 * (|E_u|^2 + |E_p|^2 + |E_n|^2) in float64."""
    nu = eu.shape[0]
    x = torch.cat([eu, ei])
    acc = x
    for _ in range(L):
        x = torch.sparse.mm(A, x) if A.layout != torch.strided else A @ x
        acc = acc + x
    O = acc / (L + 1)
    u, p, q = batch["users"], batch["positive_items"], batch["negative_items"]
    xb = (O[u] * O[nu + q]).sum(1) - (O[u] * O[nu + p]).sum(1)
    reg = eu[u].pow(2).sum(1) + ei[p].pow(2).sum(1) + ei[q].pow(2).sum(1)
    return F.softplus(xb) + lam * 0.5 * reg, xb


def _leaves(*ts):
    return [t.detach().double().clone().requires_grad_(True) for t in ts]


def _hvp64(loss_fn, params, vectors):
    loss = loss_fn(*params)
    g = torch.autograd.grad(loss, params, create_graph=True)
    return torch.autograd.grad(sum((a * v.double()).sum() for a, v in zip(g, vectors)), params)


def _jvp64(losses_fn, params, vectors):
    """<grad l_b, v> for every b: the double-vjp trick (J^T w is linear in w; its derivative along v with respect to w is Jv)."""
    ls = losses_fn(*params)
    w = torch.zeros_like(ls, requires_grad=True)
    g = torch.autograd.grad(ls, params, grad_outputs=w, create_graph=True)
    return torch.autograd.grad(sum((a * v.double()).sum() for a, v in zip(g, vectors)), w)[0]


def _lgcn_params(m):
    return m.embedding_user.weight, m.embedding_item.weight


# ------------------------------------------------------------------ LightGCN
@pytest.mark.parametrize("D", [4, 64, 128])
@pytest.mark.parametrize("L", [0, 1, 3])
def test_lightgcn_hvp_matches_float64_autograd(dev_graph, D, L):
    """10000 triples over 512 users / 511 items: every id repeats, as user, positive and negative."""
    m = _lightgcn(dev_graph, D, L, seed=D + L)
    lam = float(m.config["lambda"])
    batch = _triples(D * 10 + L, 10000)
    v = _vectors(D + 7 * L, [(U, D), (I, D)])
    hu, hi = m.loss_hvp(batch, v)
    A = _csr64(dev_graph)
    ref = _hvp64(lambda a, b: _bpr_losses64(A, a, b, L, batch, lam)[0].mean(), _leaves(*_lgcn_params(m)), v)
    _rel_close(hu, ref[0], 1e-5)
    _rel_close(hi, ref[1], 1e-5)


def test_lightgcn_directional_derivatives_match_float64_autograd(dev_graph):
    m = _lightgcn(dev_graph, 64, 3, seed=3)
    lam = 0.5                            # large enough that the regulariser's share is visible at 1e-5
    m.config["lambda"] = lam
    batch = _triples(17, 10000)
    v = _vectors(18, [(U, 64), (I, 64)])
    d = m.sample_directional_derivatives(batch, v)
    ref = _jvp64(lambda a, b: _bpr_losses64(_csr64(dev_graph), a, b, 3, batch, lam)[0], _leaves(*_lgcn_params(m)), v)
    _rel_close(d, ref, 1e-5)


def test_lightgcn_hvp_where_margins_exceed_the_softplus_threshold(dev_graph):
    """Large tables: many x_b > 20 (l' = 1, l'' = 0), many in [-20, 20]."""
    m = _lightgcn(dev_graph, 64, 1, seed=4)
    m.embedding_user.weight.data.mul_(30.0)
    m.embedding_item.weight.data.mul_(30.0)
    m.invalidate()
    lam = float(m.config["lambda"])
    batch = _triples(19, 10000)
    A = _csr64(dev_graph)
    params = _leaves(*_lgcn_params(m))
    with torch.no_grad():
        x = _bpr_losses64(A, *params, 1, batch, lam)[1]
    assert (x > 20).float().mean() > 0.2 and (x.abs() <= 20).float().mean() > 0.05
    v = _vectors(20, [(U, 64), (I, 64)])
    hu, hi = m.loss_hvp(batch, v)
    ref = _hvp64(lambda a, b: _bpr_losses64(A, a, b, 1, batch, lam)[0].mean(), params, v)
    _rel_close(hu, ref[0], 1e-5)
    _rel_close(hi, ref[1], 1e-5)


def test_lightgcn_hvp_on_a_skewed_graph_with_a_million_triples():
    """One item takes a fifth of the interactions: its row collects ~100 k pairs, far above 8192."""
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
    v = _vectors(24, [(nu, D), (ni, D)])
    hu, hi = m.loss_hvp(batch, v)
    lam = float(m.config["lambda"])
    ref = _hvp64(lambda a, b: _bpr_losses64(_csr64(g), a, b, L, batch, lam)[0].mean(), _leaves(*_lgcn_params(m)), v)
    _rel_close(hu, ref[0], 1e-5)
    _rel_close(hi, ref[1], 1e-5)


# ------------------------------------------------------------------ MF
def _mf_batch(seed, n):
    rng = np.random.default_rng(seed)
    cols = [rng.integers(0, U, n), rng.integers(0, I, n), rng.integers(0, 2, n)]
    return {k: torch.as_tensor(c, device=DEV) for k, c in zip(("users", "items", "labels"), cols)}


def _mf_losses64(m, batch):
    mean = float(m.mean)

    def f(ue, ub, ie, ib):
        u, i = batch["users"], batch["items"]
        y = (ue[u] * ie[i]).sum(1) + ub[u, 0] + ib[i, 0] + mean
        return F.binary_cross_entropy_with_logits(y, batch["labels"].double(), reduction="none")
    return f


def _mf_params(m):
    return m.user_emb.weight, m.user_bias.weight, m.item_emb.weight, m.item_bias.weight


def _mf_shapes(D):
    return [(U, D), (U, 1), (I, D), (I, 1)]


def test_mf_hvp_and_directional_derivatives_match_float64_autograd():
    m = _mf(64, seed=5)
    with torch.no_grad():
        m.mean.zero_()                   # centre the logits: l'' is not small for most rows
    batch = _mf_batch(25, 10000)
    assert 0 < int(batch["labels"].sum()) < 10000
    v = _vectors(26, _mf_shapes(64))
    h = m.loss_hvp(batch, v)
    f = _mf_losses64(m, batch)
    ref = _hvp64(lambda *p: f(*p).mean(), _leaves(*_mf_params(m)), v)
    for a, r in zip(h, ref):
        _rel_close(a, r, 1e-5)
    d = m.sample_directional_derivatives(batch, v)
    _rel_close(d, _jvp64(f, _leaves(*_mf_params(m)), v), 1e-5)


# ------------------------------------------------------------------ properties
def _dot(a, b):
    return sum(float((x.double() * y.double()).sum()) for x, y in zip(a, b))


def test_hvp_is_symmetric(dev_graph):
    m = _lightgcn(dev_graph, 64, 3, seed=6)
    batch = _triples(27, 10000)
    a, b = _vectors(28, [(U, 64), (I, 64)]), _vectors(29, [(U, 64), (I, 64)])
    x, y = _dot(a, m.loss_hvp(batch, b)), _dot(b, m.loss_hvp(batch, a))
    assert abs(x - y) <= 1e-5 * max(abs(x), abs(y)), (x, y)
    mf = _mf(64, seed=7)
    mb = _mf_batch(30, 10000)
    a, b = _vectors(31, _mf_shapes(64)), _vectors(32, _mf_shapes(64))
    x, y = _dot(a, mf.loss_hvp(mb, b)), _dot(b, mf.loss_hvp(mb, a))
    assert abs(x - y) <= 1e-5 * max(abs(x), abs(y)), (x, y)


def test_two_calls_give_the_same_bits_and_leave_the_model_alone(dev_graph):
    m = _lightgcn(dev_graph, 64, 3, seed=8)
    m.computer()                                    # a cached propagation the calls must not touch
    before = [t.clone() for t in (m.E, m.m, m.v, m.O)] + [m._steps, m._O_valid, m._O_version]
    batch = _triples(33, 20000)
    v = _vectors(34, [(U, 64), (I, 64)])
    h1, h2 = m.loss_hvp(batch, v), m.loss_hvp(batch, v)
    d1, d2 = m.sample_directional_derivatives(batch, v), m.sample_directional_derivatives(batch, v)
    assert all(torch.equal(a, b) for a, b in zip(h1, h2)) and torch.equal(d1, d2)
    after = [m.E, m.m, m.v, m.O, m._steps, m._O_valid, m._O_version]
    assert all(torch.equal(a, b) if isinstance(a, torch.Tensor) else a == b for a, b in zip(before, after))

    mf = _mf(64, seed=9)
    before = [t.clone() for t in (mf.flat, mf.m, mf.v)] + [mf._steps]
    mb = _mf_batch(35, 20000)
    v = _vectors(36, _mf_shapes(64))
    h1, h2 = mf.loss_hvp(mb, v), mf.loss_hvp(mb, v)
    d1, d2 = mf.sample_directional_derivatives(mb, v), mf.sample_directional_derivatives(mb, v)
    assert all(torch.equal(a, b) for a, b in zip(h1, h2)) and torch.equal(d1, d2)
    assert all(torch.equal(a, b) for a, b in zip(before[:3], (mf.flat, mf.m, mf.v))) and mf._steps == before[3]


def test_error_paths(dev_graph):
    from recad_b200.ops import RecadError
    m = _lightgcn(dev_graph, 16, 2, seed=10)
    batch = _triples(37, 100)
    v = _vectors(38, [(U, 16), (I, 16)])
    for fn in (m.loss_hvp, m.sample_directional_derivatives):
        with pytest.raises(RecadError):
            fn({k: t.cpu() for k, t in batch.items()}, v)                           # CPU ids
        with pytest.raises(RecadError):
            fn({k: t.int() for k, t in batch.items()}, v)                           # int32 ids
        with pytest.raises(RecadError):
            fn({"users": batch["users"]}, v)                                        # missing keys
        with pytest.raises(RecadError):
            fn(dict(batch, users=batch["users"][:50]), v)                           # ragged columns
        with pytest.raises(RecadError):
            fn(batch, (v[0].cpu(), v[1]))                                           # CPU vector
        with pytest.raises(RecadError):
            fn(batch, (v[0].double(), v[1]))                                        # float64 vector
        with pytest.raises(RecadError):
            fn(batch, (v[0][:, :8].contiguous(), v[1]))                             # wrong shape
        with pytest.raises(RecadError, match="out of range"):
            fn(dict(batch, negative_items=torch.full_like(batch["negative_items"], I)), v)
        with pytest.raises(RecadError, match="out of range"):
            fn(dict(batch, users=torch.full_like(batch["users"], -1)), v)
    d = _lightgcn(dev_graph, 16, 2, seed=10, dropout=True, keep_prob=0.6)
    d.train()
    with pytest.raises(RecadError, match="dropout"):
        d.loss_hvp(batch, v)
    d.eval()
    d.loss_hvp(batch, v)                                                            # no mask in eval mode

    mf = _mf(16, seed=11)
    mb = _mf_batch(39, 100)
    mv = _vectors(40, _mf_shapes(16))
    for fn in (mf.loss_hvp, mf.sample_directional_derivatives):
        with pytest.raises(RecadError):
            fn(dict(mb, labels=mb["labels"].float()), mv)
        with pytest.raises(RecadError):
            fn(mb, mv[:3])
        with pytest.raises(RecadError, match="out of range"):
            fn(dict(mb, items=torch.full_like(mb["items"], I)), mv)
        with pytest.raises(RecadError, match="out of range"):
            fn(dict(mb, users=torch.full_like(mb["users"], U)), mv)


# ------------------------------------------------------------------ influence
def test_influence_matches_an_exact_dense_solve(dev_graph):
    """D = 4 on the dev graph: 4092 parameters, a dense float64 Hessian from torch.autograd.functional.hessian."""
    from recad_b200 import influence
    D, L = 4, 2
    m = _lightgcn(dev_graph, D, L, seed=12)
    lam = float(m.config["lambda"])
    batch = _triples(41, 2000)
    # objective: the scores of target item 7 over 64 users, differentiated by the first-order autograd
    m.requires_grad_(True)
    users = torch.arange(64, device=DEV)
    m(users, torch.full_like(users, 7)).sum().backward()
    grads = (m.embedding_user.weight.grad.clone(), m.embedding_item.weight.grad.clone())
    m.requires_grad_(False)

    A = _csr64(dev_graph).to_dense()
    E0 = torch.cat(_lgcn_params(m)).detach().double().reshape(-1)

    def losses(flat):
        E = flat.view(U + I, D)
        return _bpr_losses64(A, E[:U], E[U:], L, batch, lam)[0]

    H = torch.autograd.functional.hessian(lambda f: losses(f).mean(), E0)
    H = 0.5 * (H + H.T)
    ev = torch.linalg.eigvalsh(H)
    damping = max(0.0, -float(ev[0])) + 0.1 * float(ev[-1])
    g = torch.cat([t.reshape(-1) for t in grads]).double()
    s_ref = torch.linalg.solve(H + damping * torch.eye(H.shape[0], dtype=H.dtype, device=DEV), g)

    def hvp(x):
        xs = x.float().view(U + I, D)
        return torch.cat([h.reshape(-1) for h in m.loss_hvp(batch, (xs[:U].contiguous(), xs[U:].contiguous()))]).double()

    rtol = 1e-6
    s, iters, res = influence.conjugate_gradient(hvp, g, damping, max_iter=1000, rtol=rtol)
    assert res < rtol and iters < 1000
    _rel_close(s, s_ref, 1e-4)

    inf = influence.sample_influence(m, batch, grads, damping, max_iter=1000, rtol=rtol)
    assert inf.residual < rtol
    w = torch.zeros(2000, dtype=torch.float64, device=DEV, requires_grad=True)
    E = E0.clone().requires_grad_(True)
    gE = torch.autograd.grad(losses(E), E, grad_outputs=w, create_graph=True)[0]
    ref = torch.autograd.grad((gE * s_ref).sum(), w)[0]                             # s^T grad l_b for every b
    _rel_close(inf.values, ref, 1e-4)
