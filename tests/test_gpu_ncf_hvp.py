"""Second order for NCF: Hessian-vector products of the BCE training loss and per-row directional derivatives through the
tensor-core (3xTF32) and the exact CUDA-core towers, and the influence of training rows on NCF.  Checked against float64
torch double backward of the mean BCE on the same GPU and, for influence, against a dense float64 Hessian."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import util
from tests.test_gpu_autograd import DEV, I, U, StubData, _ncf_f64, _ncf_params, _rel_close
from tests.test_gpu_hvp import _dot, _hvp64, _jvp64, _leaves

pytestmark = pytest.mark.gpu

VARIANTS = ["NeuMF-end", "NeuMF-pre", "GMF", "MLP"]
BAR = {"fp32": 1e-5, "tf32x3": 1e-3}
MASK_GAP = {"fp32": 1e-5, "tf32x3": 1e-4}      # rows with a float64 pre-activation this close to zero are dropped


def _params(variant, f, L, seed):
    """Parameters in recad_ncf_layout order (f = 8, L = 3: the autograd tests' own generator)."""
    if (f, L) == (8, 3):
        return _ncf_params(variant, seed)[0]
    rng = np.random.default_rng(seed)
    w = f << (L - 1)
    # tower inputs at std 2: the deep tower's pre-activations stay clear of the ReLU kinks for most rows
    p = [rng.normal(0, 0.5, (U, f)), rng.normal(0, 0.5, (I, f)), rng.normal(0, 2.0, (U, w)), rng.normal(0, 2.0, (I, w))]
    for l in range(L):
        n_in = f << (L - l)
        lim = np.sqrt(6.0 / (n_in + n_in // 2))
        p += [rng.uniform(-lim, lim, (n_in // 2, n_in)), rng.normal(0, 0.1, n_in // 2)]
    p += [rng.normal(0, 0.3, (1, f if variant in ("GMF", "MLP") else 2 * f)), rng.normal(0, 0.1, 1)]
    return [x.astype(np.float32) for x in p]


def _model(variant, precision, params, f=8, L=3, data=None):
    from recad_b200 import model

    def build(name, **extra):
        return model.from_config("victim", "ncf", factor_num=f, num_layers=L, model=name, tower_precision=precision,
                                 device=torch.device(DEV), **extra).I(dataset=data or StubData())
    m = build(variant, GMF_model=build("GMF"), MLP_model=build("MLP")) if variant == "NeuMF-pre" else build(variant)
    for t, a in zip(m._param_views(), params):
        t.data.copy_(torch.as_tensor(a))
    return m


def _f64(p, u, i, variant, L):
    if L == 3:
        return _ncf_f64(p, u, i, variant)
    ug, ig, um, im = p[:4]
    gmf = ug[u] * ig[i]
    h = torch.cat([um[u], im[i]], 1)
    pre = []
    for l in range(L):
        z = F.linear(h, p[4 + 2 * l], p[5 + 2 * l])
        pre.append(z)
        h = torch.relu(z)
    x = {"GMF": gmf, "MLP": h}.get(variant, torch.cat([gmf, h], 1))
    return F.linear(x, p[-2], p[-1]).view(-1), pre


def _losses64(batch, variant, L):
    def f(*p):
        pred, _ = _f64(p, batch["users"], batch["items"], variant, L)
        return F.binary_cross_entropy_with_logits(pred, batch["labels"].double(), reduction="none")
    return f


def _used(variant, n):
    """Indices (parameters() order) of the parameters a variant reads."""
    if variant == "GMF":
        return [0, 1, n - 2, n - 1]
    if variant == "MLP":
        return list(range(2, n))
    return list(range(n))


def _ref_hvp(m, batch, variant, L, vectors):
    """float64 double backward of the mean BCE; exactly zero for the parameters the variant does not read."""
    views = m._param_views()
    keep = _used(variant, len(views))
    base = _leaves(*views)
    losses = _losses64(batch, variant, L)

    def loss(*used):
        p = list(base)
        for k, t in zip(keep, used):
            p[k] = t
        return losses(*p).mean()
    part = _hvp64(loss, [base[k] for k in keep], [vectors[k] for k in keep])
    out = [torch.zeros_like(b) for b in base]
    for k, t in zip(keep, part):
        out[k] = t
    return out


def _batch(seed, n, users=U, items=I):
    rng = np.random.default_rng(seed)
    cols = [rng.integers(0, users, n), rng.integers(0, items, n), rng.integers(0, 2, n)]
    return {k: torch.as_tensor(c, device=DEV) for k, c in zip(("users", "items", "labels"), cols)}


def _away_from_kinks(m, batch, variant, L, precision):
    """The rows whose float64 pre-activations all lie MASK_GAP away from zero (a ReLU whose mask float32 and float64 could
    disagree on makes the two Hessians different functions); at least 90 % of the rows must remain."""
    if variant == "GMF":
        return batch
    with torch.no_grad():
        p = [t.detach().double() for t in m._param_views()]
        _, pre = _f64(p, batch["users"], batch["items"], variant, L)
        gap = torch.stack([z.abs().min(1).values for z in pre], 1).min(1).values
    keep = gap > MASK_GAP[precision]
    assert float(keep.float().mean()) >= 0.9, f"only {float(keep.float().mean()):.3f} of the rows are away from the ReLU kinks"
    return {k: t[keep].contiguous() for k, t in batch.items()}


def _vectors(m, seed):
    rng = np.random.default_rng(seed)
    return tuple(torch.as_tensor(rng.normal(size=tuple(t.shape)), dtype=torch.float32, device=DEV) for t in m._param_views())


def _check_hvp(variant, precision, f, L, seed, n=4096):
    m = _model(variant, precision, _params(variant, f, L, seed), f, L)
    batch = _away_from_kinks(m, _batch(seed + 1, n), variant, L, precision)
    assert 0 < int(batch["labels"].sum()) < batch["labels"].numel()
    v = _vectors(m, seed + 2)
    h = m.loss_hvp(batch, v)
    ref = _ref_hvp(m, batch, variant, L, v)
    assert len(h) == len(ref) == 4 + 2 * L + 2
    for k, (a, r) in enumerate(zip(h, ref)):
        assert a.shape == r.shape and a.dtype == torch.float32
        if k not in _used(variant, len(ref)):
            assert not a.any(), f"parameter {k} is not read by {variant} but its product is not zero"
        else:
            _rel_close(a, r, BAR[precision])


# ------------------------------------------------------------------ H v
@pytest.mark.parametrize("precision", ["fp32", "tf32x3"])
@pytest.mark.parametrize("variant", VARIANTS)
def test_hvp_matches_float64_double_backward(variant, precision):
    """f = 8, L = 3, 4096 rows with both labels."""
    _check_hvp(variant, precision, 8, 3, seed=100 + VARIANTS.index(variant))


@pytest.mark.parametrize("precision", ["fp32", "tf32x3"])
def test_hvp_default_tower(precision):
    """f = 32, L = 5: the concatenated contractions reach K = 2048."""
    _check_hvp("NeuMF-end", precision, 32, 5, seed=200)


def test_hvp_exact_path_for_a_factor_off_the_tensor_core_alignment():
    """f = 6 is not a multiple of 4: the exact CUDA-core GEMMs run even though the tensor-core tower is asked for."""
    _check_hvp("NeuMF-end", "tf32x3", 6, 3, seed=300)
    m = _model("NeuMF-end", "tf32x3", _params("NeuMF-end", 6, 3, 300), 6, 3)
    assert m.tower_precision == "tf32x3"


def test_directional_derivatives_match_float64():
    m = _model("NeuMF-end", "fp32", _params("NeuMF-end", 8, 3, 400))
    batch = _away_from_kinks(m, _batch(401, 4096), "NeuMF-end", 3, "fp32")
    v = _vectors(m, 402)
    d = m.sample_directional_derivatives(batch, v)
    assert d.shape == (batch["users"].numel(),) and d.dtype == torch.float32
    _rel_close(d, _jvp64(_losses64(batch, "NeuMF-end", 3), _leaves(*m._param_views()), v), 1e-5)


def test_hvp_over_more_rows_than_max_batch():
    """40 000 rows: three chunks of max_batch = 16 384, the seeds normalised by the whole n."""
    m = _model("NeuMF-end", "fp32", _params("NeuMF-end", 8, 3, 500))
    assert m.max_batch == 16384
    batch = _away_from_kinks(m, _batch(501, 40000), "NeuMF-end", 3, "fp32")
    assert batch["users"].numel() > 2 * m.max_batch
    v = _vectors(m, 502)
    for a, r in zip(m.loss_hvp(batch, v), _ref_hvp(m, batch, "NeuMF-end", 3, v)):
        _rel_close(a, r, 1e-5)


def test_hvp_on_a_skewed_batch():
    """One item fills 40 % of the rows: its embedding rows collect one long group per chunk."""
    m = _model("NeuMF-end", "fp32", _params("NeuMF-end", 8, 3, 600))
    batch = _batch(601, 20000)
    rng = np.random.default_rng(602)
    hot = torch.as_tensor(rng.random(20000) < 0.4, device=DEV)
    batch["items"] = torch.where(hot, torch.full_like(batch["items"], 5), batch["items"])
    batch = _away_from_kinks(m, batch, "NeuMF-end", 3, "fp32")
    assert float((batch["items"] == 5).float().mean()) >= 0.3
    v = _vectors(m, 603)
    for a, r in zip(m.loss_hvp(batch, v), _ref_hvp(m, batch, "NeuMF-end", 3, v)):
        _rel_close(a, r, 1e-5)


# ------------------------------------------------------------------ properties
def test_hvp_is_symmetric():
    m = _model("NeuMF-end", "fp32", _params("NeuMF-end", 8, 3, 700))
    batch = _batch(701, 4096)
    a, b = _vectors(m, 702), _vectors(m, 703)
    x, y = _dot(a, m.loss_hvp(batch, b)), _dot(b, m.loss_hvp(batch, a))
    assert abs(x - y) <= 1e-5 * max(abs(x), abs(y)), (x, y)


@pytest.mark.parametrize("precision", ["fp32", "tf32x3"])
def test_two_calls_give_the_same_bits_and_leave_the_model_alone(precision):
    m = _model("NeuMF-end", precision, _params("NeuMF-end", 8, 3, 800))
    before = [t.clone() for t in (m.flat, m.m, m.v, m.loss_acc)] + [m._steps]
    batch = _batch(801, 20000)
    v = _vectors(m, 802)
    h1, h2 = m.loss_hvp(batch, v), m.loss_hvp(batch, v)
    d1, d2 = m.sample_directional_derivatives(batch, v), m.sample_directional_derivatives(batch, v)
    assert all(torch.equal(a, b) for a, b in zip(h1, h2)) and torch.equal(d1, d2)
    assert all(torch.equal(a, b) for a, b in zip(before[:4], (m.flat, m.m, m.v, m.loss_acc))) and m._steps == before[4]


@pytest.mark.parametrize("precision", ["fp32", "tf32x3"])
def test_later_training_is_unchanged(precision):
    """Two models built alike on the dev dataset; one first runs loss_hvp, sample_directional_derivatives and a call with
    an out-of-range id.  Their train_step losses and parameters stay bit-identical."""
    from recad_b200 import model
    from recad_b200.ops import RecadError
    from tests.test_gpu_models import StubData as Batches
    from tests.test_gpu_models import _load_ncf
    z = util.load("ncf_dev.npz")
    batches = util.split_batches(z, ("batch_users", "batch_items", "batch_labels"))
    runs = []
    for probe in (False, True):
        data = Batches(U, I, batches, ("users", "items", "labels"))
        data.per_epoch = len(batches) // 2
        m = model.from_config("victim", "ncf", factor_num=8, num_layers=3, tower_precision=precision,
                              device=torch.device(DEV)).I(dataset=data)
        _load_ncf(m, z, "init", 3)
        losses = [m.train_step()[0]]
        if probe:
            batch = _batch(901, 3000)
            v = _vectors(m, 902)
            m.loss_hvp(batch, v)
            m.sample_directional_derivatives(batch, v)
            with pytest.raises(RecadError, match="out of range"):
                m.loss_hvp(dict(batch, items=torch.full_like(batch["items"], I)), v)
        losses.append(m.train_step()[0])
        runs.append((losses, m.flat.clone()))
    assert runs[0][0] == runs[1][0]
    assert torch.equal(runs[0][1], runs[1][1])


def test_error_paths():
    from recad_b200.ops import RecadError
    m = _model("NeuMF-end", "fp32", _params("NeuMF-end", 8, 3, 1000))
    batch = _batch(1001, 100)
    v = _vectors(m, 1002)
    for fn in (m.loss_hvp, m.sample_directional_derivatives):
        with pytest.raises(RecadError):
            fn({k: t.cpu() for k, t in batch.items()}, v)                           # CPU ids
        with pytest.raises(RecadError):
            fn({k: t.int() for k, t in batch.items()}, v)                           # int32 ids
        with pytest.raises(RecadError):
            fn({"users": batch["users"], "items": batch["items"]}, v)               # missing key
        with pytest.raises(RecadError):
            fn(dict(batch, users=batch["users"][:50]), v)                           # ragged columns
        with pytest.raises(RecadError):
            fn(dict(batch, labels=batch["labels"].float()), v)                      # float labels
        with pytest.raises(RecadError):
            fn(batch, v[:-1])                                                       # a vector missing
        with pytest.raises(RecadError):
            fn(batch, (v[0][:, :4].contiguous(),) + v[1:])                          # wrong shape
        with pytest.raises(RecadError):
            fn(batch, (v[0].double(),) + v[1:])                                     # float64
        with pytest.raises(RecadError):
            fn(batch, (v[0].cpu(),) + v[1:])                                        # CPU vector
        with pytest.raises(RecadError, match="out of range"):
            fn(dict(batch, users=torch.full_like(batch["users"], U)), v)
        with pytest.raises(RecadError, match="out of range"):
            fn(dict(batch, items=torch.full_like(batch["items"], -1)), v)


# ------------------------------------------------------------------ influence
def test_influence_matches_an_exact_dense_solve():
    """64 users x 48 items, f = 4, L = 2, fp32 tower: 1 525 parameters, a dense float64 Hessian from
    torch.autograd.functional.hessian."""
    from recad_b200 import influence
    nu, ni, f, L, n = 64, 48, 4, 2, 2000

    class Small(StubData):
        def info_describe(self):
            return {"n_users": nu, "n_items": ni, "graph": None, "train_dict": None}

    rng = np.random.default_rng(1100)
    w = f << (L - 1)
    p = [rng.normal(0, 0.5, (nu, f)), rng.normal(0, 0.5, (ni, f)), rng.normal(0, 0.5, (nu, w)), rng.normal(0, 0.5, (ni, w))]
    for l in range(L):
        n_in = f << (L - l)
        p += [rng.uniform(-1, 1, (n_in // 2, n_in)), rng.normal(0, 0.1, n_in // 2)]
    p += [rng.normal(0, 0.5, (1, 2 * f)), rng.normal(0, 0.1, 1)]
    m = _model("NeuMF-end", "fp32", [x.astype(np.float32) for x in p], f, L, data=Small())
    views = m._param_views()
    n_params = sum(t.numel() for t in views)
    assert 1400 < n_params < 1600
    batch = _away_from_kinks(m, _batch(1101, n, nu, ni), "NeuMF-end", L, "fp32")
    n = batch["users"].numel()
    # objective: the scores of target item 7 over every user, differentiated by the first-order autograd
    m.requires_grad_(True)
    users = torch.arange(nu, device=DEV)
    m(users, torch.full_like(users, 7)).sum().backward()
    grads = tuple(t.grad.clone() for t in m._param_views())
    m.requires_grad_(False)

    shapes = [t.shape for t in views]
    sizes = [t.numel() for t in views]
    theta0 = torch.cat([t.detach().double().reshape(-1) for t in views])
    losses = _losses64(batch, "NeuMF-end", L)

    def per_row(flat):
        return losses(*[c.view(s) for c, s in zip(torch.split(flat, sizes), shapes)])

    H = torch.autograd.functional.hessian(lambda t: per_row(t).mean(), theta0)
    H = 0.5 * (H + H.T)
    ev = torch.linalg.eigvalsh(H)
    damping = max(0.0, -float(ev[0])) + 0.1 * float(ev[-1])
    g = torch.cat([t.reshape(-1) for t in grads]).double()
    s_ref = torch.linalg.solve(H + damping * torch.eye(H.shape[0], dtype=H.dtype, device=DEV), g)

    def hvp(x):
        xs = tuple(c.view(s).float().contiguous() for c, s in zip(torch.split(x, sizes), shapes))
        return torch.cat([h.reshape(-1) for h in m.loss_hvp(batch, xs)]).double()

    rtol = 1e-6
    s, iters, res = influence.conjugate_gradient(hvp, g, damping, max_iter=1000, rtol=rtol)
    assert res < rtol and iters < 1000
    _rel_close(s, s_ref, 1e-4)

    inf = influence.sample_influence(m, batch, grads, damping, max_iter=1000, rtol=rtol)
    assert inf.residual < rtol
    wv = torch.zeros(n, dtype=torch.float64, device=DEV, requires_grad=True)
    th = theta0.clone().requires_grad_(True)
    gth = torch.autograd.grad(per_row(th), th, grad_outputs=wv, create_graph=True)[0]
    ref = torch.autograd.grad((gth * s_ref).sum(), wv)[0]                            # s^T grad l_b for every b
    _rel_close(inf.values, ref, 1e-4)
    _rel_close(torch.cat([t.reshape(-1) for t in inf.s]).double(), s_ref, 1e-4)
