"""CPU: the oracle's float32 FMA chain (oracle/evaluate.py fmaf / fma_dot_rows) is correctly rounded, checked
against exact rational arithmetic, and the full-ranking restatement built on it is unchanged on the stored fixtures."""
from fractions import Fraction

import numpy as np

from oracle import evaluate as oev
from oracle import graph as og
from tests import util


def _round_f32(x):
    """Fraction -> nearest float32, ties to even (the IEEE default), with gradual underflow and overflow to inf."""
    if x == 0:
        return np.float32(0.0)
    sign = -1 if x < 0 else 1
    x = abs(x)
    e = x.numerator.bit_length() - x.denominator.bit_length()      # 2^e <= x < 2^(e + 2)
    if Fraction(2) ** e > x:
        e -= 1
    if Fraction(2) ** (e + 1) <= x:
        e += 1
    q = max(e - 23, -149)                                          # exponent of one ulp
    m = x / Fraction(2) ** q
    fl = m.numerator // m.denominator
    rem = m - fl
    if rem > Fraction(1, 2) or (rem == Fraction(1, 2) and fl % 2 == 1):
        fl += 1
    v = Fraction(fl) * Fraction(2) ** q
    if v >= Fraction(2) ** 128:
        return np.float32(sign * np.inf)
    return np.float32(sign * float(v))


def _exact_fma(a, b, c):
    return _round_f32(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c)))


def _fma_cast_once(a, b, c):
    """The emulation the oracle used before: float64 multiply-add, then one cast (two roundings)."""
    return (np.float64(a) * np.float64(b) + np.float64(c)).astype(np.float32)


def _same(x, y):
    return np.asarray(x, np.float32).view(np.uint32) == np.asarray(y, np.float32).view(np.uint32)


def test_fmaf_matches_rational_arithmetic_on_random_triples():
    rng = np.random.default_rng(0)
    n = 4000
    sig = rng.uniform(1.0, 2.0, (3, n)) * rng.choice([-1.0, 1.0], (3, n))
    ex = np.stack([rng.integers(-63, 63, n), rng.integers(-63, 63, n), rng.integers(-140, 126, n)])
    a, b, c = (np.ldexp(sig[k], ex[k]).astype(np.float32) for k in range(3))
    # a third with c close to -a*b: heavy cancellation, results down to the subnormal range
    m = n // 3
    c[:m] = (-(a[:m].astype(np.float64) * b[:m])).astype(np.float32)
    got = oev.fmaf(a, b, c)
    for k in range(n):
        assert _same(got[k], _exact_fma(a[k], b[k], c[k])), (a[k], b[k], c[k])


def _midpoint_triples():
    """(a, b, c) whose exact a * b + c lies within 2^-70 relative of a float32 rounding midpoint, on the side away
    from the even neighbour: c = (1 + odd * 2^-23) 2^k, a b = 2^(k - 24) (1 - 2^-46), so the float64 sum rounds onto
    the midpoint and a second rounding to float32 goes the wrong way."""
    out = []
    for odd in (1, 3, 5, 77, 2 ** 23 - 1):
        for k in (-60, -3, 0, 7, 90):
            for sg in (1.0, -1.0):
                c = np.float32(sg * np.ldexp(1.0 + odd * 2.0 ** -23, k))
                a = np.float32(sg * np.ldexp(1.0 + 2.0 ** -23, k - 24))
                b = np.float32(1.0 - 2.0 ** -23)
                out.append((a, b, c))
    return out


def test_fmaf_is_correct_on_float32_midpoints_where_double_rounding_is_not():
    trip = _midpoint_triples()
    a, b, c = (np.array(x, dtype=np.float32) for x in zip(*trip))
    want = np.array([_exact_fma(*t) for t in trip], dtype=np.float32)
    assert np.all(_same(oev.fmaf(a, b, c), want))
    assert not np.all(_same(_fma_cast_once(a, b, c), want))          # the old emulation gets these wrong
    # the same triples through the dot-product chain: acc = fma(1, c, 0) = c, then fma(a, b, c)
    u = np.stack([np.ones_like(a), a], 1)
    items = np.stack([c, b], 1)
    for r in range(len(trip)):
        assert _same(oev.fma_dot_rows(u[r], items[r:r + 1])[0], want[r])


def test_fmaf_special_values():
    inf, big = np.float32(np.inf), np.float32(3.0e38)
    a = np.array([0.0, -0.0, 1.0, big, big, 1.0, np.float32(2.0 ** -75)], dtype=np.float32)
    b = np.array([5.0, 5.0, inf, big, -big, 1.0, np.float32(2.0 ** -75)], dtype=np.float32)
    c = np.array([-0.0, -0.0, 1.0, 0.0, 0.0, -1.0, 0.0], dtype=np.float32)
    got = oev.fmaf(a, b, c)
    assert _same(got[0], np.float32(0.0)) and _same(got[1], np.float32(-0.0))
    assert got[2] == inf and got[3] == inf and got[4] == -inf
    assert _same(got[5], np.float32(0.0))                             # x - x is +0 under round-to-nearest
    assert _same(got[6], np.float32(0.0))                             # 2^-150: halfway to 2^-149, ties to even
    assert _same(got[6], _exact_fma(a[6], b[6], c[6]))


def _fma_dot_rows_old(u, items):
    acc = np.zeros(items.shape[0], dtype=np.float32)
    for d in range(items.shape[1]):
        acc = (np.float64(u[d]) * items[:, d].astype(np.float64) + acc.astype(np.float64)).astype(np.float32)
    return acc


def test_full_rank_batched_unchanged_on_the_mf_fixture(monkeypatch):
    """The exact FMA chain changes no bit of the restatement's output on the stored MF model (the half-way cases
    the old emulation mis-rounded do not occur there)."""
    tr, _, _ = util.dicts("dev")
    g = util.load("mf_dev.npz")
    meta = util.meta()
    U, I = meta["dev"]["n_users"], meta["dev"]["n_items"]
    ue = np.concatenate([g["final0"], g["final1"], np.ones((U, 1), np.float32)], 1)
    ie = np.concatenate([g["final2"], np.ones((I, 1), np.float32), g["final3"]], 1)
    u_tr, i_tr, _, _ = og.flatten_dict(tr)
    ptr, idx = og.all_pos(u_tr, i_tr, U, I)
    users = np.arange(U, dtype=np.int64)
    new = oev.full_rank_batched(ue, ie, users, ptr, idx, [5, 17], 50)
    monkeypatch.setattr(oev, "fma_dot_rows", _fma_dot_rows_old)
    old = oev.full_rank_batched(ue, ie, users, ptr, idx, [5, 17], 50)
    for x, y in zip(new, old):
        assert x.dtype == y.dtype and np.array_equal(x.view(np.uint32) if x.dtype == np.float32 else x,
                                                     y.view(np.uint32) if y.dtype == np.float32 else y)
