"""Weight gradients of LightGCN interactions that the graph may not hold yet (LightGCN.candidate_weight_gradients) and the
hypergradient of an objective with respect to them (influence.candidate_hypergradient), for chosen users against every item.
Checked against float64 torch autograd over one tied weight per interaction (stored ones at their multiplicity, candidates
at 0, both entries of each pair), the per-entry path of interaction_hypergradient, a dense float64 solve and central finite
differences of a retrained (Newton-minimised) float64 model."""
import numpy as np
import pytest
import torch

from tests.test_gpu_autograd import DEV, I, U, _lightgcn, _mf, _rel_close, dev_graph  # noqa: F401
from tests.test_gpu_edge_grad import _lightgcn as _lightgcn_n
from tests.test_gpu_edge_grad import _rows
from tests.test_gpu_hvp import _triples, _vectors
from tests.test_gpu_hypergrad import _loss64, _newton, _prop64, _stored_triples

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------ float64 reference
class _Interactions:
    """The graph's stored interactions (user rows of the CSR) followed by the candidate pairs not stored, each with one
    float64 weight put on both of its entries; `index(u, i)` gives a pair's position."""

    def __init__(self, g, nu, ni, cu, ci):
        rows, cols = _rows(g), g.colidx.long()
        us = rows < nu
        su, si = rows[us], cols[us] - nu
        self.nu, self.ni, self.n_stored = nu, ni, int(su.numel())
        self.mult = g.mult[us].double()
        skey = su * ni + si
        self.order = torch.argsort(skey)
        self.sk = skey[self.order]
        ckey = cu.long() * ni + ci.long()
        found = self._stored(ckey) >= 0
        self.new = torch.unique(ckey[~found])
        self.u = torch.cat([su, self.new // ni])
        self.i = torch.cat([si, self.new % ni])
        self.w0 = torch.cat([self.mult, torch.zeros(self.new.numel(), dtype=torch.float64, device=DEV)])

    def to(self, dev):
        for k in ("mult", "order", "sk", "new", "u", "i", "w0"):
            setattr(self, k, getattr(self, k).to(dev))
        return self

    def _stored(self, key):
        if self.sk.numel() == 0:
            return torch.full_like(key, -1)
        pos = torch.searchsorted(self.sk, key).clamp(max=self.sk.numel() - 1)
        return torch.where(self.sk[pos] == key, self.order[pos], torch.full_like(key, -1))

    def index(self, u, i):
        key = u.long() * self.ni + i.long()
        k = self._stored(key)
        pos = torch.searchsorted(self.new, key).clamp(max=max(self.new.numel() - 1, 0))
        return torch.where(k >= 0, k, self.n_stored + pos)

    def values(self, w):
        """Entry rows, columns and normalised values of the symmetric graph with interaction weights w."""
        N = self.nu + self.ni
        er = torch.cat([self.u, self.nu + self.i])
        ec = torch.cat([self.nu + self.i, self.u])
        wt = torch.cat([w, w])
        d = (torch.zeros(N, dtype=torch.float64, device=w.device).index_add(0, er, wt) + 1e-14) ** -0.5
        return er, ec, d[er] * wt * d[ec]

    def omega(self, w, batch):
        """w_k / mult_k for the rows whose positive pair k is stored, 1 for the others."""
        k = self._stored(batch["users"] * self.ni + batch["positive_items"])
        kc = k.clamp(min=0)
        return torch.where(k >= 0, w[kc] / self.mult[kc], torch.ones_like(k, dtype=torch.float64))


def _f64(ix, m, w, E, obj=None, batch=None, S=None):
    """f(W) = obj(O) + <S, grad_E L_batch(E; W)> in float64 (create_graph on the loss gradient)."""
    L, nu = m.n_layers, ix.nu
    er, ec, v = ix.values(w)
    f = torch.zeros((), dtype=torch.float64, device=DEV)
    if obj is not None:
        f = f + obj(_prop64(er, ec, v, E, L))
    if batch is not None:
        loss = _loss64(er, ec, v, E, nu, L, batch["users"], batch["positive_items"], batch["negative_items"],
                       float(m.config["lambda"]), ix.omega(w, batch))
        gE, = torch.autograd.grad(loss, E, create_graph=True)
        f = f + (gE * S).sum()
    return f


def _block64(g, m, users, obj=None, batch=None, S=None, pairs=None):
    """df/dW at the candidate pairs: (users x every item) as [R, I], or the pairs (u, i) given."""
    nu, ni = m.num_users, m.num_items
    if pairs is None:
        cu, ci = users.repeat_interleave(ni), torch.arange(ni, device=DEV).repeat(users.numel())
    else:
        cu, ci = pairs
    ix = _Interactions(g, nu, ni, cu, ci)
    w = ix.w0.clone().requires_grad_(True)
    E = m.E.detach().double().requires_grad_(True)
    f = _f64(ix, m, w, E, obj, batch, None if S is None else torch.cat([x.double() for x in S]))
    gw, = torch.autograd.grad(f, w, allow_unused=True) if f.requires_grad else (None,)
    gw = torch.zeros_like(w) if gw is None else gw
    out = gw[ix.index(cu, ci)]
    return out.view(users.numel(), ni) if pairs is None else out


def _dot_obj(gO):
    g64 = torch.cat([x.double() for x in gO])
    return lambda O: (O * g64).sum()


def _check_block(g, m, users, gO, batch, S, bar=1e-5):
    got = m.candidate_weight_gradients(users, gO, batch, S)
    assert got.dtype == torch.float32 and tuple(got.shape) == (users.numel(), m.num_items)
    ref = _block64(g, m, users, None if gO is None else _dot_obj(gO), batch, S)
    if float(ref.abs().max()) == 0.0:
        assert torch.equal(got, torch.zeros_like(got))
        return
    _rel_close(got, ref, bar)


# ------------------------------------------------------------------ against float64 autograd
@pytest.mark.parametrize("mode", ["gO", "loss", "both"])
@pytest.mark.parametrize("D", [4, 64, 128])
@pytest.mark.parametrize("L", [0, 1, 3])
def test_candidate_weight_gradients_match_float64_autograd(dev_graph, mode, D, L):
    """The dev graph (512 users x 511 items); R = every user, then a shuffled subset with a repeated id."""
    m = _lightgcn(dev_graph, D, L, seed=D + L)
    gO = _vectors(D + 3 * L, [(U, D), (I, D)]) if mode != "loss" else None
    batch = _stored_triples(dev_graph, U, I, D * 10 + L, 3000, 3000) if mode != "gO" else None
    S = _vectors(D + 5 * L + 1, [(U, D), (I, D)]) if mode != "gO" else None
    _check_block(dev_graph, m, torch.arange(U, device=DEV), gO, batch, S)
    rng = np.random.default_rng(D + L)
    sub = rng.permutation(U)[:77]
    sub = np.concatenate([sub, sub[3:4]])
    _check_block(dev_graph, m, torch.as_tensor(sub, device=DEV), gO, batch, S)


def _tile_graph():
    """700 users x 1000 items with seg_len = 32 (user 0 and item rows span several SpMM segments), plus 5 fake users."""
    from recad_b200 import ops
    rng = np.random.default_rng(17)
    nu, ni, F_ = 700, 1000, 5
    u = np.concatenate([np.zeros(1500, np.int64), rng.integers(0, nu, 18500)])
    i = rng.integers(0, ni, 20000)
    g = ops.Graph.from_edges(torch.as_tensor(u, device=DEV), torch.as_tensor(i, device=DEV), nu, ni, seg_len=32)
    items = [np.sort(rng.choice(ni, 40, replace=False)) for _ in range(F_)]
    fake_rowptr = torch.as_tensor(np.concatenate([[0], np.cumsum([len(x) for x in items])]), device=DEV)
    g = g.append_users(nu, ni, fake_rowptr, torch.as_tensor(np.concatenate(items), device=DEV))
    assert g.n_mrow > 0
    return g, nu + F_, ni


@pytest.mark.parametrize("R", [1, 127, 128, 129, 300])
def test_gemm_tile_edges_with_multi_segment_rows_and_fake_users(R):
    """|R| around the 128-row tile and 1000 items (not a multiple of the item tile); the fake users are among R."""
    g, nu, ni = _tile_graph()
    m = _lightgcn_n(g, 32, 2, seed=R, n_users=nu, n_items=ni)
    rng = np.random.default_rng(R)
    users = rng.integers(0, nu, R)
    users[0] = nu - 1
    if R > 2:
        users[1] = nu - 3
        users[2] = 0
    batch = _stored_triples(g, nu, ni, R + 1, 4000, 2000)
    batch["users"][:50] = nu - 1                                  # rows of a fake user's stored pairs
    k = int(g.rowptr[nu - 1])
    batch["positive_items"][:50] = g.colidx[k].long() - nu
    gO = _vectors(R + 2, [(nu, 32), (ni, 32)])
    S = _vectors(R + 3, [(nu, 32), (ni, 32)])
    _check_block(g, m, torch.as_tensor(users, device=DEV), gO, batch, S)


def test_a_block_with_enough_tiles_for_the_wide_gemm_tile(dev_graph):
    """|R| = 5000 (every dev-graph user about ten times) x 511 items: 40 x 4 tiles of 128 x 128, at least one per SM, so
    gemm_tc takes its BN = 128 tile -- the shape of production-sized blocks -- where the smaller tests take BN = 64."""
    sm = torch.cuda.get_device_properties(DEV).multi_processor_count
    R = 5000
    assert ((R + 127) // 128) * ((I + 127) // 128) >= sm and I > 64
    m = _lightgcn(dev_graph, 16, 2, seed=61)
    rng = np.random.default_rng(61)
    users = torch.as_tensor(rng.integers(0, U, R), device=DEV)
    gO = _vectors(62, [(U, 16), (I, 16)])
    batch = _stored_triples(dev_graph, U, I, 63, 3000, 3000)
    S = _vectors(64, [(U, 16), (I, 16)])
    got = m.candidate_weight_gradients(users, gO, batch, S)
    ref = _block64(dev_graph, m, torch.arange(U, device=DEV), _dot_obj(gO), batch, S)[users]
    _rel_close(got, ref, 1e-5)


def test_on_a_skewed_graph_with_a_million_triples():
    """The graph and batch of the HVP test (one item collects ~100 k positive pairs): 4096 sampled candidate pairs and every
    stored pair of R against float64 autograd."""
    from recad_b200 import model, ops
    from tests.test_gpu_autograd import StubData
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
    users = torch.as_tensor(rng.choice(nu, 200, replace=False), device=DEV)
    gO = _vectors(25, [(nu, D), (ni, D)])
    S = _vectors(26, [(nu, D), (ni, D)])
    got = m.candidate_weight_gradients(users, gO, batch, S)
    r = torch.as_tensor(rng.integers(0, 200, 4096), device=DEV)
    i = torch.as_tensor(rng.integers(0, ni, 4096), device=DEV)
    sel = torch.isin(torch.as_tensor(eu, device=DEV), users)
    su, si = torch.as_tensor(eu, device=DEV)[sel], torch.as_tensor(ei, device=DEV)[sel]
    row_of = torch.full((nu,), -1, dtype=torch.int64, device=DEV)
    row_of[users] = torch.arange(200, device=DEV)
    for rr, ii in ((r, i), (row_of[su], si)):
        ref = _block64(g, m, users, _dot_obj(gO), batch, S, pairs=(users[rr], ii))
        _rel_close(got[rr, ii], ref, 1e-5)


# ------------------------------------------------------------------ stored pairs and the per-entry path
def test_stored_pairs_match_the_entry_gradients(dev_graph):
    """At a stored pair, the block is normalized_values' backward of (the edge-value gradient of <gO, O> + loss_mixed_values)
    plus the sample part, summed over the pair's two entries; end to end, candidate_hypergradient equals
    interaction_hypergradient's values[k] + values[T[k]]."""
    from recad_b200 import influence, ops
    g = dev_graph
    m = _lightgcn(g, 16, 2, seed=21)
    batch = _stored_triples(g, U, I, 22, 3000, 1000)
    n = batch["users"].numel()
    gO = _vectors(23, [(U, 16), (I, 16)])
    S = _vectors(24, [(U, 16), (I, 16)])
    users = torch.arange(U, device=DEV)
    block = m.candidate_weight_gradients(users, gO, batch, S)
    ev = g.vals.clone().requires_grad_(True)
    with torch.enable_grad():
        uo, io = m.computer(edge_values=ev)
        gv, = torch.autograd.grad((uo * gO[0]).sum() + (io * gO[1]).sum(), ev)
    gv = gv + m.loss_mixed_values(batch, S)
    w = g.mult.clone().requires_grad_(True)
    with torch.enable_grad():
        gw, = torch.autograd.grad(ops.normalized_values(g, w), w, gv)
    kb = g.entry_index(batch["users"], U + batch["positive_items"], missing=-1)
    dl = m.sample_directional_derivatives(batch, S)
    per_entry = gw + ops.index_sums(kb, dl, g.nnz) / (n * g.mult)
    rows, cols = _rows(g), g.colidx.long()
    k = torch.nonzero(rows < U).squeeze(1)
    T = g.transpose_permutation()
    _rel_close(block[rows[k], cols[k] - U], per_entry[k] + per_entry[T[k]], 1e-5)

    obj_users = torch.arange(64, device=DEV)
    hg = influence.interaction_hypergradient(
        m, batch, lambda e: m(obj_users, torch.full_like(obj_users, 7), edge_values=e).sum(), 0.05, max_iter=300, rtol=1e-7)
    ch = influence.candidate_hypergradient(m, batch, lambda uo, io: (uo[obj_users] * io[7]).sum(), users, 0.05,
                                           max_iter=300, rtol=1e-7)
    assert ch.residual < 1e-7 and ch.values.shape == (U, I)
    _rel_close(ch.values[rows[k], cols[k] - U], hg.values[k] + hg.values[T[k]], 1e-4)


def test_hypergradient_matches_a_dense_float64_solve(dev_graph):
    """D = 4, L = 2 on the dev graph: s from a dense float64 Hessian, then the whole U x I block by float64 autograd."""
    from recad_b200 import influence
    D, L = 4, 2
    g = dev_graph
    m = _lightgcn(g, D, L, seed=12)
    batch = _stored_triples(g, U, I, 41, 1500, 500)
    users = torch.arange(U, device=DEV)
    ix = _Interactions(g, U, I, users.repeat_interleave(I), torch.arange(I, device=DEV).repeat(U))
    E0 = m.E.detach().double().reshape(-1)
    obj_users = torch.arange(64, device=DEV)

    def J(O):
        return (O[obj_users] * O[U + 7]).sum()

    def loss(flat):
        er, ec, v = ix.values(ix.w0)
        u, p, q = batch["users"], batch["positive_items"], batch["negative_items"]
        return _loss64(er, ec, v, flat.view(U + I, D), U, L, u, p, q, float(m.config["lambda"]), ix.omega(ix.w0, batch))

    H = torch.autograd.functional.hessian(loss, E0)
    H = 0.5 * (H + H.T)
    ev = torch.linalg.eigvalsh(H)
    damping = max(0.0, -float(ev[0])) + 0.1 * float(ev[-1])
    Ef = E0.clone().requires_grad_(True)
    er, ec, v = ix.values(ix.w0)
    gJ_E, = torch.autograd.grad(J(_prop64(er, ec, v, Ef.view(U + I, D), L)), Ef)
    s_ref = torch.linalg.solve(H + damping * torch.eye(H.shape[0], dtype=H.dtype, device=DEV), gJ_E).view(U + I, D)
    ref = _block64(g, m, users, J, batch, (-s_ref[:U], -s_ref[U:]))

    ch = influence.candidate_hypergradient(m, batch, lambda uo, io: (uo[obj_users] * io[7]).sum(), users, damping,
                                           max_iter=1000, rtol=1e-7)
    assert ch.residual < 1e-7 and ch.iterations < 1000
    _rel_close(torch.cat([x.reshape(-1) for x in ch.s]), s_ref.reshape(-1), 1e-4)
    _rel_close(ch.values, ref, 1e-4)


# ------------------------------------------------------------------ finite differences
def test_hypergradient_signs_by_finite_differences():
    """32 users x 20 items plus 2 fake users, D = 4, L = 2, lambda = 0.1.  Retrain by Newton at W and W +- eps on two pairs
    a fake user does not hold and on one stored pair; the central differences of J(E*(W), W) match the float64 closed form
    (damping 0, pseudo-inverse on the rotation null space), and the CUDA block at the minimiser matches it."""
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
    batch["users"][:5] = nu + 1
    batch["positive_items"][:5] = 17
    users = torch.arange(NU, device=DEV)
    cpu = torch.device("cpu")
    ix = _Interactions(g, NU, ni, users.repeat_interleave(ni), torch.arange(ni, device=DEV).repeat(NU)).to(cpu)
    cb = {k: t.to(cpu) for k, t in batch.items()}
    obj_users = torch.arange(16)

    def loss(flat, w):
        er, ec, v = ix.values(w)
        return _loss64(er, ec, v, flat.view(N, D), NU, L, cb["users"], cb["positive_items"], cb["negative_items"], lam,
                       ix.omega(w, cb))

    def Jf(flat, w):
        er, ec, v = ix.values(w)
        O = _prop64(er, ec, v, flat.view(N, D), L)
        return (O[obj_users] * O[NU + 4]).sum()

    w0 = ix.w0.clone()
    E_star = _newton(lambda e: loss(e, w0), torch.as_tensor(rng.normal(0, 0.3, N * D)), lbfgs=True)
    H = torch.autograd.functional.hessian(lambda e: loss(e, w0), E_star)
    ev = torch.linalg.eigvalsh(0.5 * (H + H.T))
    assert float(ev[6]) > 1e-3 * float(ev[-1]) and float(ev[0]) > -1e-9
    Ef, wl = E_star.clone().requires_grad_(True), w0.clone().requires_grad_(True)
    gJ_E, direct = torch.autograd.grad(Jf(Ef, wl), (Ef, wl))
    s = torch.linalg.lstsq(H, gJ_E, rcond=1e-9, driver="gelsd").solution
    Ef, wl = E_star.clone().requires_grad_(True), w0.clone().requires_grad_(True)
    gE, = torch.autograd.grad(loss(Ef, wl), Ef, create_graph=True)
    closed = direct - torch.autograd.grad((gE * s).sum(), wl)[0]

    fu = torch.tensor([nu + 1, nu + 1, nu + 1])
    fi = torch.tensor([2, 11, 17])                                      # (nu + 1, 17) is stored, the other two are not
    check = ix.index(fu, fi)
    assert int(check[0]) >= ix.n_stored and int(check[1]) >= ix.n_stored and int(check[2]) < ix.n_stored
    eps = 1e-3
    for k in check.tolist():
        Js = []
        for sgn in (1, -1):
            w = w0.clone()
            w[k] += sgn * eps
            Js.append(float(Jf(_newton(lambda e: loss(e, w), E_star), w)))
        fd = (Js[0] - Js[1]) / (2 * eps)
        assert abs(fd - float(closed[k])) <= 1e-5 * float(closed.abs().max()), (k, fd, float(closed[k]))

    m.embedding_user.weight.data.copy_(E_star.view(N, D)[:NU].float())
    m.embedding_item.weight.data.copy_(E_star.view(N, D)[NU:].float())
    m.invalidate()
    ch = influence.candidate_hypergradient(m, batch, lambda uo, io: (uo[:16] * io[4]).sum(), users,
                                           damping=1e-6 * float(ev[-1]), max_iter=2000, rtol=1e-8)
    ref = closed[ix.index(users.cpu().repeat_interleave(ni), torch.arange(ni).repeat(NU))].view(NU, ni)
    _rel_close(ch.values.cpu(), ref, 1e-3)


# ------------------------------------------------------------------ behaviour
def test_two_calls_give_the_same_bits_and_leave_the_model_alone(dev_graph):
    from recad_b200 import influence
    m = _lightgcn(dev_graph, 64, 3, seed=8)
    m.computer()
    before = [t.clone() for t in (m.E, m.m, m.v, m.O, m.loss_acc)] + [m._steps, m._O_valid, m._O_version]
    batch = _stored_triples(dev_graph, U, I, 33, 10000, 10000)
    gO = _vectors(35, [(U, 64), (I, 64)])
    S = _vectors(34, [(U, 64), (I, 64)])
    users = torch.arange(U, device=DEV)
    assert torch.equal(m.candidate_weight_gradients(users, gO, batch, S), m.candidate_weight_gradients(users, gO, batch, S))

    def obj(uo, io):
        return (uo[:32] * io[3]).sum()
    a = influence.candidate_hypergradient(m, batch, obj, users[:100], 0.05, max_iter=8, rtol=1e-30)
    b = influence.candidate_hypergradient(m, batch, obj, users[:100], 0.05, max_iter=8, rtol=1e-30)
    assert a.iterations == b.iterations == 8
    assert torch.equal(a.values, b.values) and all(torch.equal(x, y) for x, y in zip(a.s, b.s))
    assert not any(p.requires_grad for p in m.parameters())
    after = [m.E, m.m, m.v, m.O, m.loss_acc, m._steps, m._O_valid, m._O_version]
    assert all(torch.equal(x, y) if isinstance(x, torch.Tensor) else x == y for x, y in zip(before, after))
    assert m.candidate_weight_gradients(users[:0], gO, batch, S).shape == (0, I)


def test_zero_layers_give_exactly_the_sample_part(dev_graph):
    from recad_b200 import ops
    g = dev_graph
    m = _lightgcn(g, 16, 0, seed=30)
    batch = _stored_triples(g, U, I, 31, 4000, 1000)
    n = batch["users"].numel()
    S = _vectors(32, [(U, 16), (I, 16)])
    users = torch.arange(U, device=DEV)
    got = m.candidate_weight_gradients(users, _vectors(33, [(U, 16), (I, 16)]), batch, S)
    kb = g.entry_index(batch["users"], U + batch["positive_items"], missing=-1)
    sample = ops.index_sums(kb, m.sample_directional_derivatives(batch, S), g.nnz) / (n * g.mult)
    rows, cols = _rows(g), g.colidx.long()
    k = torch.nonzero(rows < U).squeeze(1)
    ref = torch.zeros(U, I, dtype=torch.float32, device=DEV)
    ref[rows[k], cols[k] - U] = sample[k]
    assert float(ref.abs().max()) > 0
    assert torch.equal(got, ref)


def test_error_paths(dev_graph):
    from recad_b200 import influence
    from recad_b200.ops import RecadError
    m = _lightgcn(dev_graph, 16, 2, seed=10)
    batch = _triples(37, 100)
    v = _vectors(38, [(U, 16), (I, 16)])
    users = torch.arange(10, device=DEV)
    fn = m.candidate_weight_gradients

    def obj(uo, io):
        return (uo[:4] * io[3]).sum()
    with pytest.raises(RecadError, match="LightGCN"):
        influence.candidate_hypergradient(_mf(16, seed=11), batch, obj, users, 0.1)
    with pytest.raises(RecadError, match="out of range"):
        fn(torch.tensor([0, U], device=DEV), v)
    with pytest.raises(RecadError, match="out of range"):
        fn(torch.tensor([-1], device=DEV), v, batch, v)
    with pytest.raises(RecadError, match="out of range"):
        fn(users, v, dict(batch, negative_items=torch.full_like(batch["negative_items"], I)), v)
    with pytest.raises(RecadError, match="out of range"):
        influence.candidate_hypergradient(m, batch, obj, torch.tensor([0, U], device=DEV), 0.1, max_iter=2)
    with pytest.raises(RecadError, match="CUDA"):
        influence.candidate_hypergradient(m, batch, obj, users.cpu(), 0.1, max_iter=2)
    with pytest.raises(RecadError):
        influence.candidate_hypergradient(m, batch, obj, users.float(), 0.1, max_iter=2)
    with pytest.raises(RecadError, match="scalar"):
        influence.candidate_hypergradient(m, batch, lambda uo, io: uo[:4] * io[3], users, 0.1, max_iter=2)
    with pytest.raises(RecadError):
        fn(users.cpu(), v)                                                         # CPU ids
    with pytest.raises(RecadError):
        fn(users, (v[0].cpu(), v[1]))                                              # CPU gO
    with pytest.raises(RecadError):
        fn(users, v, batch, (v[0].cpu(), v[1]))                                    # CPU vector
    with pytest.raises(RecadError):
        fn(users, (v[0][:, :8].contiguous(), v[1]))                                # wrong shape
    with pytest.raises(RecadError):
        fn(users.view(2, 5), v)                                                    # not [R]
    with pytest.raises(RecadError, match="together"):
        fn(users, v, batch)                                                        # batch without vectors
    d = _lightgcn(dev_graph, 16, 2, seed=10, dropout=True, keep_prob=0.6)
    d.train()
    with pytest.raises(RecadError, match="dropout"):
        d.candidate_weight_gradients(users, v)
    with pytest.raises(RecadError, match="dropout"):
        influence.candidate_hypergradient(d, batch, obj, users, 0.1, max_iter=2)
    d.eval()
    d.candidate_weight_gradients(users, v)                                         # no mask in eval mode
