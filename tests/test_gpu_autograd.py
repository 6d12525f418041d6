"""Autograd through the victims: LightGCN, MF and NCF scores are differentiable with respect to the victims' parameters
once grad mode is on and a parameter requires a gradient, with deterministic CUDA backward kernels.  Gradients are checked
against torch autograd in float64 on the same GPU."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import graph as og
from oracle import pointwise_models as opm
from tests import util

pytestmark = pytest.mark.gpu
META = util.meta()
DEV = "cuda:0"
U, I = META["dev"]["n_users"], META["dev"]["n_items"]


class StubData:
    def __init__(self, graph=None, bs=1024):
        self.graph = graph
        self.config = {"pairwise_batch_size": bs, "pointwise_batch_size": bs, "device": torch.device(DEV)}

    def info_describe(self):
        return {"n_users": U, "n_items": I, "graph": self.graph, "train_dict": None}

    def generate_batch(self):
        return iter(())


@pytest.fixture(scope="module")
def dev_graph():
    from recad_b200 import ops
    tr, _, _ = util.dicts("dev")
    u, i, _, _ = og.flatten_dict(tr)
    return ops.Graph.from_edges(torch.as_tensor(u, device=DEV), torch.as_tensor(i, device=DEV), U, I)


def _pairs(seed, B):
    rng = np.random.default_rng(seed)
    u = torch.as_tensor(rng.integers(0, U, B), device=DEV)
    i = torch.as_tensor(rng.integers(0, I, B), device=DEV)
    w = torch.as_tensor(rng.normal(size=B), dtype=torch.float32, device=DEV)      # random per-sample loss weights
    return u, i, w


def _rel_close(got, ref, bar):
    """|got - ref| <= bar * max |ref|, on the whole tensor."""
    got, ref = got.detach().double(), ref.detach().double()
    assert got.shape == ref.shape
    err, scale = (got - ref).abs().max().item(), ref.abs().max().item()
    assert err <= bar * scale, f"max error {err:.3e} > {bar:g} x {scale:.3e}"


def _close(got, ref, rtol=1e-4, atol=2e-6):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    assert got.shape == ref.shape
    bad = (got - ref).abs() > atol + rtol * ref.abs()
    assert not bad.any(), f"{int(bad.sum())} / {bad.numel()} differ, max abs {(got - ref).abs().max().item():.3e}"


# ------------------------------------------------------------------ LightGCN
def _lightgcn(graph, D, L, seed=0, **kw):
    from recad_b200 import model
    m = model.from_config("victim", "lightgcn", latent_dim_rec=D, lightGCN_n_layers=L, device=torch.device(DEV), **kw).I(
        dataset=StubData(graph))
    rng = np.random.default_rng(seed)
    m.embedding_user.weight.data.copy_(torch.as_tensor(rng.normal(0, 0.1, (U, D)), dtype=torch.float32))
    m.embedding_item.weight.data.copy_(torch.as_tensor(rng.normal(0, 0.1, (I, D)), dtype=torch.float32))
    m.invalidate()
    return m


def _lightgcn_oracle(graph, m, L, u, i, w, vals=None):
    """float64 torch autograd over the graph's own normalised CSR: layer mean, dot scores, weighted sum."""
    N = U + I
    A = torch.sparse_csr_tensor(graph.rowptr, graph.colidx.long(), (graph.vals if vals is None else vals).double(), size=(N, N))
    eu = m.embedding_user.weight.detach().double().clone().requires_grad_(True)
    ei = m.embedding_item.weight.detach().double().clone().requires_grad_(True)
    x = torch.cat([eu, ei])
    acc = x
    for _ in range(L):
        x = torch.sparse.mm(A, x)
        acc = acc + x
    O = acc / (L + 1)
    s = (O[u] * O[U + i]).sum(1)
    (w.double() * s).sum().backward()
    return s.detach(), eu.grad, ei.grad


@pytest.mark.parametrize("D", [4, 64, 128])
@pytest.mark.parametrize("L", [0, 1, 3])
def test_lightgcn_gradients_match_float64_autograd(dev_graph, D, L):
    """Batches of 10000 pairs over 512 users / 511 items: every id repeats, and the batch is above the 8192 pairs where
    the NCF scatter stops."""
    m = _lightgcn(dev_graph, D, L, seed=D + L)
    m.requires_grad_(True)
    u, i, w = _pairs(D * 10 + L, 10000)
    s = m(u, i)
    (w * s).sum().backward()
    s_ref, gu, gi = _lightgcn_oracle(dev_graph, m, L, u, i, w)
    _rel_close(s, s_ref, 1e-5)
    _rel_close(m.embedding_user.weight.grad, gu, 1e-5)
    _rel_close(m.embedding_item.weight.grad, gi, 1e-5)


def test_lightgcn_computer_and_get_users_rating_are_differentiable(dev_graph):
    m = _lightgcn(dev_graph, 64, 3, seed=5)
    m.requires_grad_(True)
    ou, oi = m.computer()
    assert ou.grad_fn is not None and oi.grad_fn is not None
    r = m.getUsersRating(torch.arange(7, device=DEV))
    r.sum().backward()
    assert m.embedding_user.weight.grad.abs().sum() > 0 and m.embedding_item.weight.grad.abs().sum() > 0


def test_lightgcn_dropout_backward_uses_its_own_forward_mask(dev_graph):
    m = _lightgcn(dev_graph, 32, 2, seed=7, dropout=True, keep_prob=0.6)
    m.train()
    m.requires_grad_(True)
    u, i, w = _pairs(11, 3000)
    torch.manual_seed(1234)
    s1 = m(u, i)
    vals1 = m._drop_graph.vals.clone()                 # the dropped matrix this forward used
    s2 = m(u, i)                                       # a second forward draws a new mask
    assert not torch.equal(vals1, m._drop_graph.vals)
    (w * s1).sum().backward()
    s_ref, gu, gi = _lightgcn_oracle(dev_graph, m, 2, u, i, w, vals=vals1)
    _rel_close(s1, s_ref, 1e-5)
    _rel_close(m.embedding_user.weight.grad, gu, 1e-5)
    _rel_close(m.embedding_item.weight.grad, gi, 1e-5)
    del s2


# ------------------------------------------------------------------ MF
def _mf(D=64, seed=0):
    from recad_b200 import model
    m = model.from_config("victim", "mf", embedding_size=D, device=torch.device(DEV)).I(dataset=StubData())
    rng = np.random.default_rng(seed)
    for t in (m.user_emb, m.user_bias, m.item_emb, m.item_bias):
        t.weight.data.copy_(torch.as_tensor(rng.normal(0, 0.3, tuple(t.weight.shape)), dtype=torch.float32))
    return m


def test_mf_gradients_match_float64_autograd():
    m = _mf(seed=3)
    m.requires_grad_(True)
    u, i, w = _pairs(21, 10000)
    s = m(u, i)
    (w * s).sum().backward()
    ref = [t.weight.detach().double().clone().requires_grad_(True) for t in (m.user_emb, m.user_bias, m.item_emb, m.item_bias)]
    mean = m.mean.detach().double().clone().requires_grad_(True)
    s_ref = (ref[0][u] * ref[2][i]).sum(1) + ref[1][u, 0] + ref[3][i, 0] + mean
    (w.double() * s_ref).sum().backward()
    _rel_close(s, s_ref, 1e-5)
    for t, r in zip((m.user_emb, m.user_bias, m.item_emb, m.item_bias), ref):
        _rel_close(t.weight.grad, r.grad, 1e-5)
    _rel_close(m.mean.grad, mean.grad, 1e-5)


# ------------------------------------------------------------------ NCF
F_, L_, B_NCF = 8, 3, 512
NCF_SEED = 15      # every ReLU pre-activation of this batch is at least 1e-4 away from zero (asserted below)


def _ncf_params(variant, seed=NCF_SEED):
    """Parameters in recad_ncf_layout order and a batch of 512 pairs, all from one numpy seed."""
    rng = np.random.default_rng(seed)
    w = F_ << (L_ - 1)
    p = [rng.normal(0, 0.5, (U, F_)), rng.normal(0, 0.5, (I, F_)), rng.normal(0, 0.5, (U, w)), rng.normal(0, 0.5, (I, w))]
    for l in range(L_):
        n_in = F_ << (L_ - l)
        lim = np.sqrt(6.0 / (n_in + n_in // 2))
        p += [rng.uniform(-lim, lim, (n_in // 2, n_in)), rng.normal(0, 0.1, n_in // 2)]
    p += [rng.normal(0, 0.3, (1, 2 * F_)), rng.normal(0, 0.1, 1)]
    u, i = rng.integers(0, U, B_NCF), rng.integers(0, I, B_NCF)
    p = [x.astype(np.float32) for x in p]
    if variant in ("GMF", "MLP"):
        p[-2] = p[-2][:, :F_].copy()
    return p, torch.as_tensor(u, device=DEV), torch.as_tensor(i, device=DEV)


def _ncf(variant, precision, params):
    from recad_b200 import model

    def build(name, **extra):
        return model.from_config("victim", "ncf", factor_num=F_, num_layers=L_, model=name, tower_precision=precision,
                                 device=torch.device(DEV), **extra).I(dataset=StubData())
    if variant == "NeuMF-pre":
        m = build(variant, GMF_model=build("GMF"), MLP_model=build("MLP"))
    else:
        m = build(variant)
    for t, a in zip(m._param_views(), params):
        t.data.copy_(torch.as_tensor(a))
    return m


def _ncf_f64(params, u, i, variant):
    """float64 restatement of ncf.py:112-131: the predict layer reads cat(gmf, tower) (NeuMF), gmf ('GMF') or the tower
    ('MLP')."""
    ug, ig, um, im = params[:4]
    gmf = ug[u] * ig[i]
    h = torch.cat([um[u], im[i]], 1)
    pre = []
    for l in range(L_):
        z = F.linear(h, params[4 + 2 * l], params[5 + 2 * l])
        pre.append(z)
        h = torch.relu(z)
    x = {"GMF": gmf, "MLP": h}.get(variant, torch.cat([gmf, h], 1))
    return F.linear(x, params[-2], params[-1]).view(-1), pre


def _ncf_ref_grads(params, u, i, w, variant):
    ref = [torch.as_tensor(a, dtype=torch.float64, device=DEV).requires_grad_(True) for a in params]
    pred, pre = _ncf_f64(ref, u, i, variant)
    (w.double() * pred).sum().backward()
    grads = [torch.zeros_like(r) if r.grad is None else r.grad for r in ref]      # the branch a variant does not read
    return pred.detach(), grads, min(z.abs().min().item() for z in pre)


def test_ncf_neumf_end_gradients_match_the_float64_oracle():
    params, u, i = _ncf_params("NeuMF-end")
    m = _ncf("NeuMF-end", "fp32", params)
    m.requires_grad_(True)
    w = _pairs(31, B_NCF)[2]
    s = m(u, i)
    (w * s).sum().backward()
    o = opm.NCFOracle({"ug": params[0], "ig": params[1], "um": params[2], "im": params[3], "W": params[4:-2:2],
                       "b": params[5:-2:2], "Wp": params[-2], "bp": params[-1]})
    plist = [o.ug, o.ig, o.um, o.im] + [x for wb in zip(o.W, o.b) for x in wb] + [o.Wp, o.bp]
    for p in plist:
        p.data = p.data.double()
    pred = o.forward(u.cpu().numpy(), i.cpu().numpy())
    (w.cpu().double() * pred).sum().backward()
    _close(s, pred)
    for t, p in zip(m._param_views(), plist):
        _close(t.grad, p.grad)


@pytest.mark.parametrize("variant", ["GMF", "MLP", "NeuMF-pre"])
def test_ncf_variant_gradients_match_a_float64_restatement(variant):
    params, u, i = _ncf_params(variant)
    m = _ncf(variant, "fp32", params)
    m.requires_grad_(True)
    w = _pairs(32, B_NCF)[2]
    s = m(u, i)
    (w * s).sum().backward()
    pred, grads, _ = _ncf_ref_grads(params, u, i, w, variant)
    _close(s, pred)
    for t, g in zip(m._param_views(), grads):
        _close(t.grad, g)


def test_ncf_tensor_core_tower_gradients():
    params, u, i = _ncf_params("NeuMF-end")
    w = _pairs(33, B_NCF)[2]
    pred, grads, margin = _ncf_ref_grads(params, u, i, w, "NeuMF-end")
    assert margin > 1e-6, f"a ReLU pre-activation lies {margin:.2e} from zero: choose another NCF_SEED"
    m = _ncf("NeuMF-end", "tf32x3", params)
    m.requires_grad_(True)
    s = m(u, i)
    (w * s).sum().backward()
    _rel_close(s, pred, 1e-3)
    for t, g in zip(m._param_views(), grads):
        _rel_close(t.grad, g, 1e-3)


@pytest.mark.parametrize("precision", ["fp32", "tf32x3"])
def test_ncf_bce_gradient_through_autograd_equals_the_fused_gradient(precision):
    import ctypes as C
    from recad_b200 import _lib, ops
    params, u, i = _ncf_params("NeuMF-end")
    y = torch.as_tensor(np.random.default_rng(34).integers(0, 2, B_NCF), device=DEV)
    m = _ncf("NeuMF-end", precision, params)
    m.requires_grad_(True)
    F.binary_cross_entropy_with_logits(m(u, i), y.float()).backward()
    samples = torch.stack([u, i, y], 1).contiguous()
    _lib.check(_lib.lib().recad_ncf_grad(C.byref(m._st), ops._ptr(samples), None, B_NCF, B_NCF, ops._stream()), "recad_ncf_grad")
    for t, (off, n, shape) in zip(m._param_views(), m._grad_slots):
        _rel_close(t.grad, m.g[off:off + n].view(shape), 1e-6)


# ------------------------------------------------------------------ behaviour
def _victims(dev_graph):
    return {"lightgcn": _lightgcn(dev_graph, 64, 3, seed=41), "mf": _mf(seed=42),
            "ncf": _ncf("NeuMF-end", "tf32x3", _ncf_params("NeuMF-end")[0])}


def test_graph_mode_forward_equals_the_plain_forward_bit_for_bit(dev_graph):
    u, i, _ = _pairs(51, 5000)
    for name, m in _victims(dev_graph).items():
        with torch.no_grad():
            plain = m(u, i)
        m.requires_grad_(True)
        s = m(u, i)
        assert s.grad_fn is not None, name
        assert torch.equal(s.detach(), plain), name


def test_no_grad_fn_under_no_grad_or_with_frozen_parameters(dev_graph):
    u, i, _ = _pairs(52, 100)
    for name, m in _victims(dev_graph).items():
        assert m(u, i).grad_fn is None, name                       # parameters frozen (the default)
        m.requires_grad_(True)
        with torch.no_grad():
            assert m(u, i).grad_fn is None, name
        assert m(u, i).grad_fn is not None, name
    m = _victims(dev_graph)["lightgcn"]
    assert all(t.grad_fn is None for t in m.computer())


@pytest.mark.parametrize("B", [3000, 20000])
def test_backward_is_bit_stable_and_grad_accumulates(dev_graph, B):
    u, i, w = _pairs(53, B)
    for name, m in _victims(dev_graph).items():
        if name == "ncf" and B > 8192:
            continue                         # NCF adds the embedding rows in a fixed order up to 8192 pairs per batch
        m.requires_grad_(True)
        (w * m(u, i)).sum().backward()
        first = [p.grad.clone() for p in m.parameters() if p.grad is not None]
        m.zero_grad()
        (w * m(u, i)).sum().backward()
        second = [p.grad.clone() for p in m.parameters() if p.grad is not None]
        assert len(first) == len(second) > 0
        assert all(torch.equal(a, b) for a, b in zip(first, second)), name
        (w * m(u, i)).sum().backward()
        assert all(torch.equal(p.grad, 2 * a) for p, a in zip([p for p in m.parameters() if p.grad is not None], first)), name


def test_out_of_range_ids_raise(dev_graph):
    from recad_b200 import ops
    good = torch.zeros(4, dtype=torch.int64, device=DEV)
    for name, m in _victims(dev_graph).items():
        m.requires_grad_(True)
        for bad_u, bad_i in ((torch.tensor([0, 1, U, 2], device=DEV), good), (good, torch.tensor([0, -1, 1, 2], device=DEV))):
            with pytest.raises(ops.RecadError):
                m(bad_u, bad_i)
    # the backward entries check their ids themselves
    X = torch.randn(U + I, 8, device=DEV)
    g = torch.ones(4, device=DEV)
    with pytest.raises(ops.RecadError):
        ops.pair_scores_backward(X[:U], X[U:], good, torch.tensor([0, 1, I, 2], device=DEV), g)
    with pytest.raises(ops.RecadError):
        ops.pair_scores_backward(X[:U], X[U:], torch.tensor([-3, 1, 2, 2], device=DEV), good, g, bias=True)
    m = _victims(dev_graph)["ncf"]
    with pytest.raises(ops.RecadError):
        ops.ncf_backward(m._st, torch.tensor([0, 1, U + 7, 2], device=DEV), good, g)


def test_torch_optimizer_steps_reach_forward_and_full_rank(dev_graph):
    from recad_b200 import ops
    u, i, w = _pairs(54, 2000)
    users = torch.arange(64, device=DEV)
    rowptr = torch.zeros(U + 1, dtype=torch.int64, device=DEV)
    col = torch.zeros(1, dtype=torch.int32, device=DEV)
    for name, m in _victims(dev_graph).items():
        with torch.no_grad():
            before = m(u, i)
        if name != "ncf":
            m.full_rank(users, [0, 1], 10, rowptr, col)       # fills the cached propagation
        m.requires_grad_(True)
        opt = torch.optim.SGD(m.parameters(), lr=0.5)
        (w * m(u, i)).sum().backward()
        opt.step()
        fresh = m(u, i).detach()                              # graph mode: computed from the live tables
        with torch.no_grad():
            after = m(u, i)
        assert not torch.equal(after, before), name
        assert torch.equal(after, fresh), name
        if name != "ncf":
            got = m.full_rank(users, [0, 1], 10, rowptr, col)
            if name == "lightgcn":
                with torch.no_grad():
                    O = torch.cat(m.computer())
                want = ops.fullrank_eval(O[:U], O[U:], users, rowptr, col, [0, 1], 10)
            else:
                want = ops.fullrank_eval(m.user_emb.weight.detach(), m.item_emb.weight.detach(), users, rowptr, col, [0, 1], 10,
                                         item_bias=m.item_bias.weight.detach().view(-1))
            assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]), name
