"""GPU: the full-ranking layer (exact CUDA-core kernel, tcgen05 kernel, rank_from_scores, recall_ndcg, eligible_users)
pinned bit for bit at every template tier, tile edge and tie.

Integer-lattice inputs make all three ranking paths exact: user and item entries are integers in [-15, 15] times 2^s,
item biases integers in [-255, 255] times 2^(2s).  Every score is then an integer below 136 * 225 + 255 < 2^24 times
2^(2s), so the fp32 FMA chain, the fp16 hi / lo split (lo = 0) and the tensor-core accumulation are all exact, and the
kernels must equal an int64 / fp64 reference exactly.  Equal scores are plentiful and some are placed on purpose.

The contract checked (oracle/evaluate.py states the tie rule):
  * top-K: eligible items (not train items, score not -inf) by score descending, then id ascending; empty slots are
    (-1, -inf);
  * target rank: non-train items that score higher, plus equal-scoring non-train items with a smaller id; -1 when
    the target is one of the user's train items.  For a target scoring -inf this counts the non-train -inf items with
    a smaller id (the oracle's rule, and rank_from_scores'); the two fused kernels mask train items by setting them to
    -inf, so for such a target they count those too: they are only checked on finite scores;
  * target score: the score of the target item, train item or not.
+0 and -0 are equal scores.  Rows with NaN scores have no defined ranking and are not tested."""
import numpy as np
import pytest
import torch

from oracle import evaluate as oev

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SCALES = (-50, 0, 40)


# ------------------------------------------------------------------ reference and case builders
def _csr(rows):
    ptr = np.zeros(len(rows) + 1, dtype=np.int64)
    ptr[1:] = np.cumsum([len(r) for r in rows])
    col = np.concatenate([np.asarray(sorted(set(r)), dtype=np.int32) for r in rows] + [np.zeros(0, np.int32)])
    return ptr, col


def _reference(S, masked, targets, K):
    """(topk_idx, topk_val, target_rank, target_score) of the score rows S (fp64 [n, I]) with train items `masked`."""
    n, I = S.shape
    ids = np.arange(I)
    valid = ~masked & (S != -np.inf)
    key = np.where(valid, -S, np.inf)
    order = np.lexsort((np.broadcast_to(ids, S.shape), key), axis=1)[:, :K]
    sel = np.take_along_axis(valid, order, 1)
    topi = -np.ones((n, K), dtype=np.int64)
    topv = np.full((n, K), -np.inf)
    kk = min(K, I)
    topi[:, :kk] = np.where(sel, order, -1)
    topv[:, :kk] = np.where(sel, np.take_along_axis(S, order, 1), -np.inf)
    T = len(targets)
    trank = np.zeros((n, T), dtype=np.int64)
    tscore = np.zeros((n, T))
    for j, t in enumerate(targets):
        st = S[:, t:t + 1]
        ok = ~masked
        trank[:, j] = np.sum(ok & ((S > st) | ((S == st) & (ids < t))), 1)
        trank[masked[:, t], j] = -1
        tscore[:, j] = S[:, t]
    return topi, topv, trank, tscore


def _assert_equal(got, ref, what):
    names = ("topk_idx", "topk_val", "target_rank", "target_score")
    for name, g, r in zip(names, got, ref):
        g = g.cpu().numpy()
        assert g.shape == r.shape, (what, name, g.shape, r.shape)
        # == compares +0 and -0 as equal and -inf as equal to itself; no tolerance
        ok = np.array_equal(g.astype(np.float64), r) if g.dtype == np.float32 else np.array_equal(g.astype(np.int64), r)
        if not ok:
            bad = np.argwhere(g != r)[:5].tolist()
            pytest.fail(f"{what}: {name} differs at {bad}: got {[g[tuple(b)] for b in bad]}, want {[r[tuple(b)] for b in bad]}")


class Lattice:
    """One lattice case: U user rows, I items, D dims, scale 2^s (or 2^su for users and 2^si for items when s is a pair),
    with the edge structure described inline."""

    def __init__(self, seed, U, I, D, s, bias, n_eval, T):
        rng = np.random.default_rng(seed)
        su, si = s if isinstance(s, tuple) else (s, s)
        self.I, self.D, self.s2 = I, D, su + si
        ni = rng.integers(-15, 16, (I, D))
        small = rng.integers(-1, 2, (I, D))
        if I > 64:
            ni[64:128] = small[64:128]          # a tile whose scale exponent differs from its neighbours'
        for i in (5, 15, 63):
            if i < I:
                ni[i] = small[i]
        if I > 256:
            ni[192:256] = 0                     # an all-zero 64-item tile
        nb = rng.integers(-255, 256, I) if bias else None
        # equal scores on purpose: across a 16-item block edge (15 | 16), a 64-item tile edge (63 | 64), and in tiles
        # with different scale exponents handled by different epilogue warpgroups (5: tile 0, 70: tile 1, 130: tile 2)
        for dst, src in ((16, 15), (64, 63), (70, 5), (130, 5)):
            if dst < I:
                ni[dst] = ni[src]
                if bias:
                    nb[dst] = nb[src]
        nu = rng.integers(-15, 16, (U, D))
        nu[4] = 0                               # an all-zero user row
        nu[5] = rng.integers(-1, 2, D)          # a user row with a small scale (large exponent), as `small` above
        self.ni, self.nu, self.nb = ni, nu, nb
        self.ue = np.ldexp(nu.astype(np.float64), su).astype(np.float32)
        self.ie = np.ldexp(ni.astype(np.float64), si).astype(np.float32)
        self.ib = None if nb is None else np.ldexp(nb.astype(np.float64), su + si).astype(np.float32)
        last = I - 1
        train = [sorted({p for p in (0, 15, 16, 63, 64, last) if p < I}),    # tile positions and the last item
                 sorted(set(range(I)) - {min(1, last), I // 2, max(last - 1, 0)}),   # fewer eligible items than K
                 [],                                                            # an empty row
                 list(range(I))]                                                # every item
        for _ in range(4, U):
            train.append(rng.choice(I, size=int(rng.integers(0, min(I, 40) + 1)), replace=False).tolist())
        self.train = train
        self.ptr, self.col = _csr(train)
        head = [5, 0, 1, 2, 3, 4, 0, 5]                                        # unsorted, repeated
        self.users = np.concatenate([head, rng.integers(0, U, max(n_eval - len(head), 0))])[:n_eval].astype(np.int64)
        cand = [0, last, 63, 64, 16, 15, 70, 0]                                 # T = 8 repeats target 0
        self.targets = [c % I for c in cand[:T]]

    def scores(self):
        """exact scores of the evaluated users, fp64 [n_eval, I] (integers times 2^(2s), all exact in fp32)"""
        S = self.nu[self.users].astype(np.int64) @ self.ni.T.astype(np.int64)
        if self.nb is not None:
            S = S + self.nb
        assert np.abs(S).max(initial=0) < 2 ** 24
        return np.ldexp(S.astype(np.float64), self.s2)

    def masked(self):
        m = np.zeros((len(self.users), self.I), dtype=bool)
        for r, u in enumerate(self.users):
            m[r, self.train[u]] = True
        return m

    def reference(self, K):
        return _reference(self.scores(), self.masked(), self.targets, K)

    def dev(self):
        t = lambda a: None if a is None else torch.as_tensor(a, device=DEV)   # noqa: E731
        return t(self.ue), t(self.ie), t(self.users), t(self.ptr), t(self.col), t(self.ib)

    def fullrank(self, K, precision, item_T=None):
        from recad_b200 import ops
        ue, ie, users, ptr, col, ib = self.dev()
        return ops.fullrank_eval(ue, ie, users, ptr, col, self.targets, K, item_T=item_T, item_bias=ib, precision=precision)

    def from_scores(self, K):
        from recad_b200 import ops
        _, _, users, ptr, col, _ = self.dev()
        S = torch.as_tensor(self.scores().astype(np.float32), device=DEV)
        return ops.rank_from_scores(S, users, ptr, col, self.targets, K)


# ------------------------------------------------------------------ exact CUDA-core kernel: every DP x TMAX tier
EXACT_D = (1, 3, 4, 16, 17, 32, 33, 64, 65, 72, 73, 128, 129, 136)
EXACT_K = (1, 31, 33, 128)
EXACT_T = (0, 1, 4, 5, 8)


@pytest.mark.parametrize("T", EXACT_T)
@pytest.mark.parametrize("D", EXACT_D)
def test_exact_kernel_lattice_tiers(D, T):
    """DP = 16 / 32 / 64 / 72 / 128 / 136 (and their edges) x TMAX = 0 / 1 / 4 / 8; K, bias and scale rotate over the
    cases so that each value meets several tiers."""
    i = EXACT_D.index(D) * len(EXACT_T) + EXACT_T.index(T)
    K = EXACT_K[i % len(EXACT_K)]
    s = SCALES[i % len(SCALES)]
    bias = (i // 2) % 2 == 1 and D < 136                  # the bias rides as dimension D + 1 <= 136
    c = Lattice(1000 + i, 40, 200, D, s, bias, 129, T)
    _assert_equal(c.fullrank(K, "exact"), c.reference(K), f"exact D={D} T={T} K={K} s={s} bias={bias}")


@pytest.mark.parametrize("K", EXACT_K)
def test_exact_kernel_explicit_item_table_with_wide_padded_stride(K):
    """A caller-provided transposed item table whose row stride is one tile wider than needed and whose padding
    columns hold NaN: they must never reach a score."""
    c = Lattice(7 + K, 40, 150, 20, 0, False, 129, 4)
    ld = (c.I + 63) // 64 * 64 + 64
    it = np.full((c.D, ld), np.nan, dtype=np.float32)
    it[:, :c.I] = c.ie.T
    _assert_equal(c.fullrank(K, "exact", item_T=torch.as_tensor(it, device=DEV)), c.reference(K), f"item_T K={K}")


def test_exact_kernel_rejects_unsupported_sizes():
    from recad_b200._lib import RecadError
    c = Lattice(3, 10, 100, 16, 0, False, 4, 1)
    with pytest.raises(RecadError):
        c.fullrank(129, "exact")
    with pytest.raises(RecadError):
        c.fullrank(128 + 1, "tf32x3")                     # K > 32 falls back to the exact kernel, which refuses
    c9 = Lattice(3, 10, 100, 16, 0, False, 4, 8)
    c9.targets = c9.targets + [1]
    with pytest.raises(RecadError):
        c9.fullrank(10, "exact")
    with pytest.raises(RecadError):
        c9.fullrank(10, "tf32x3")
    c137 = Lattice(3, 10, 100, 137, 0, False, 4, 1)
    with pytest.raises(RecadError):
        c137.fullrank(10, "exact")
    c136 = Lattice(3, 10, 100, 136, 0, True, 4, 1)        # the bias makes it 137 wide
    with pytest.raises(RecadError):
        c136.fullrank(10, "exact")


# ------------------------------------------------------------------ tensor-core kernel
TC_D = (1, 8, 16, 17, 33, 63, 64)
TC_T = (0, 1, 2, 4, 5, 8)


@pytest.mark.parametrize("T", TC_T)
@pytest.mark.parametrize("D", TC_D)
def test_tensor_core_kernel_lattice_is_exact(D, T):
    """TMAX = 0 / 1 / 2 / 4 / 8 at D from 1 to 64; an all-zero user row and an all-zero item tile, ties across
    tiles with different scale exponents and across the two epilogue warpgroups, and a user row and a tile with
    entries in {-1, 0, 1} times 2^-50, whose scale exponents add up to 128, beyond one fp32 power of two."""
    i = TC_D.index(D) * len(TC_T) + TC_T.index(T)
    K = (1, 32)[i % 2]
    s = SCALES[i % len(SCALES)]
    bias = (i // 2) % 2 == 1
    c = Lattice(2000 + i, 40, 333, D, s, bias, 129, T)
    what = f"tc D={D} T={T} K={K} s={s} bias={bias}"
    ref = c.reference(K)
    _assert_equal(c.fullrank(K, "tf32x3"), ref, what)
    _assert_equal(c.fullrank(K, "exact"), ref, what + " (exact)")
    _assert_equal(c.from_scores(K), ref, what + " (rank_from_scores)")


@pytest.mark.parametrize("s", [(-60, -60), (0, -125), (-125, 0)])
def test_tensor_core_kernel_tiny_operands(s):
    """Operands so small that the tiles' scale exponents ku + kt exceed 126 (every tile here, and the target tile), so
    that 2^(ku + kt) is no single fp32: the scores, biases included, must still come back exact, from both kernels."""
    for j, (D, T, K) in enumerate(((64, 8, 32), (5, 1, 1))):
        c = Lattice(90 + j, 40, 333, D, s, j == 0, 129, T)
        ref = c.reference(K)
        _assert_equal(c.fullrank(K, "tf32x3"), ref, f"tc s={s} D={D}")
        _assert_equal(c.fullrank(K, "exact"), ref, f"exact s={s} D={D}")


def _kernels_launched(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.key for e in prof.key_averages()}


@pytest.mark.parametrize("D,K,tc", [(64, 32, True), (65, 32, False), (64, 33, False), (1, 1, True)])
def test_dispatch_boundary(D, K, tc):
    """precision="tf32x3" takes the tensor cores exactly when D <= 64 and K <= 32, and on lattice data every output
    equals precision="exact"."""
    c = Lattice(300 + D + K, 40, 300, D, -50, True, 129, 2)
    got, names = _kernels_launched(lambda: c.fullrank(K, "tf32x3"))
    assert any("fullrank_tc_kernel" in n for n in names) == tc, names
    assert any("fullrank_kernel" in n and "fullrank_tc_kernel" not in n for n in names) == (not tc), names
    exact = c.fullrank(K, "exact")
    for a, b in zip(got, exact):
        assert torch.equal(a, b)
    _assert_equal(got, c.reference(K), f"dispatch D={D} K={K}")


# ------------------------------------------------------------------ shapes: n_items, n_eval, both kernels
@pytest.mark.parametrize("I", (1, 15, 16, 17, 63, 64, 65, 4097))
def test_both_kernels_item_counts(I):
    for j, (D, K, s) in enumerate(((16, 32, -50), (33, 1, 40), (64, 31, 0))):
        c = Lattice(40 + I + j, 30, I, D, s, j == 0, 129, 8)
        ref = c.reference(K)
        what = f"I={I} D={D} K={K} s={s}"
        _assert_equal(c.fullrank(K, "exact"), ref, what + " exact")
        _assert_equal(c.fullrank(K, "tf32x3"), ref, what + " tc")
        _assert_equal(c.from_scores(K), ref, what + " rank_from_scores")


@pytest.mark.parametrize("n_eval", (1, 127, 129, 257))
def test_both_kernels_eval_counts(n_eval):
    c = Lattice(60 + n_eval, 300, 517, 24, -50, True, n_eval, 5)
    for K in (1, 32):
        ref = c.reference(K)
        _assert_equal(c.fullrank(K, "exact"), ref, f"n_eval={n_eval} K={K} exact")
        _assert_equal(c.fullrank(K, "tf32x3"), ref, f"n_eval={n_eval} K={K} tc")
    _assert_equal(c.fullrank(128, "exact"), c.reference(128), f"n_eval={n_eval} K=128 exact")


# ------------------------------------------------------------------ random floats: exact kernel vs the FMA oracle
@pytest.mark.parametrize("D", (3, 17, 72, 73, 136))
def test_exact_kernel_random_floats_bit_exact(D):
    """Scores of random fp32 embeddings over many magnitudes are the ascending-d FMA chain, bit for bit."""
    from recad_b200 import ops
    rng = np.random.default_rng(D)
    U, I, K = 200, 300, 33
    ue = (rng.standard_normal((U, D)) * np.exp2(rng.integers(-20, 20, (U, 1)))).astype(np.float32)
    ie = (rng.standard_normal((I, D)) * np.exp2(rng.integers(-20, 20, (I, 1)))).astype(np.float32)
    train = [rng.choice(I, size=int(rng.integers(0, 50)), replace=False).tolist() for _ in range(U)]
    ptr, col = _csr(train)
    users = rng.integers(0, U, 131).astype(np.int64)
    targets = [0, 299, 64, 127, 128]
    got = ops.fullrank_eval(torch.as_tensor(ue, device=DEV), torch.as_tensor(ie, device=DEV), torch.as_tensor(users, device=DEV),
                            torch.as_tensor(ptr, device=DEV), torch.as_tensor(col, device=DEV), targets, K, precision="exact")
    S = np.stack([oev.fma_dot_rows(ue[u], ie) for u in users]).astype(np.float64)
    masked = np.zeros((len(users), I), dtype=bool)
    for r, u in enumerate(users):
        masked[r, train[u]] = True
    _assert_equal(got, _reference(S, masked, targets, K), f"random D={D}")


# ------------------------------------------------------------------ rank_from_scores
SPECIAL = np.array([-np.inf, -2.0, -1.0, -0.0, 0.0, 1.0, 2.0, np.inf], dtype=np.float32)


@pytest.mark.parametrize("K", (1, 32, 33, 1024))
@pytest.mark.parametrize("I", (1, 31, 33))
def test_rank_from_scores_special_values(I, K):
    """+-inf, -0 / +0 and long runs of equal scores; K up to 1024 (> n_items); T = 8."""
    from recad_b200 import ops
    rng = np.random.default_rng(I * 7 + K)
    n = 21
    S = SPECIAL[rng.integers(0, len(SPECIAL), (n, I))]
    S[0] = 0.0
    S[1] = np.where(np.arange(I) % 2 == 0, -0.0, 0.0)       # a run of +-0
    S[2] = np.inf
    S[3] = -np.inf
    S[4] = np.where(np.arange(I) < I // 2, np.inf, -np.inf)
    S[5] = 1.0
    users = rng.integers(0, 8, n).astype(np.int64)
    train = [[], list(range(I)), [0], [I - 1], list(range(0, I, 2)), [], [I // 2], list(range(I // 3))]
    ptr, col = _csr(train)
    targets = [0, I - 1, I // 2, 0, (I + 1) // 3 % I, 1 % I, I - 1, 2 % I]
    got = ops.rank_from_scores(torch.as_tensor(S, device=DEV), torch.as_tensor(users, device=DEV),
                               torch.as_tensor(ptr, device=DEV), torch.as_tensor(col, device=DEV), targets, K)
    masked = np.zeros((n, I), dtype=bool)
    for r, u in enumerate(users):
        masked[r, train[u]] = True
    _assert_equal(got, _reference(S.astype(np.float64), masked, targets, K), f"rank_from_scores I={I} K={K}")


def test_rank_from_scores_rejects_unsupported_sizes():
    from recad_b200 import ops
    from recad_b200._lib import RecadError
    S = torch.zeros((2, 40), device=DEV)
    users = torch.zeros(2, dtype=torch.int64, device=DEV)
    ptr = torch.zeros(2, dtype=torch.int64, device=DEV)
    col = torch.zeros(1, dtype=torch.int32, device=DEV)
    ops.rank_from_scores(S, users, ptr, col, [0] * 8, 1024)
    with pytest.raises(RecadError):
        ops.rank_from_scores(S, users, ptr, col, [0], 1025)
    with pytest.raises(RecadError):
        ops.rank_from_scores(S, users, ptr, col, [0] * 9, 10)


# ------------------------------------------------------------------ recall_ndcg
def _recall_ndcg_fp64(topi, users, gt_rows):
    """recall_ndcg_kernel's formula restated in fp64: per user with ground truth, hits / |gt| and
    sum_{hits at slot k} 1 / log2(k + 2) over sum_{k < min(|gt|, K)} 1 / log2(k + 2); -1 slots are no item."""
    K = topi.shape[1]
    disc = 1.0 / np.log2(np.arange(K) + 2.0)
    rec = ndcg = 0.0
    cnt = 0
    for row, u in zip(topi, users):
        gt = set(gt_rows[u])
        if not gt:
            continue
        hit = np.array([i >= 0 and int(i) in gt for i in row])
        rec += hit.sum() / len(gt)
        ndcg += disc[hit].sum() / disc[:min(len(gt), K)].sum()
        cnt += 1
    return rec, ndcg, cnt


@pytest.mark.parametrize("K", (1, 5, 20, 100))
def test_recall_ndcg_padding_and_long_ground_truth(K):
    from recad_b200 import ops
    rng = np.random.default_rng(K)
    U, I, n = 300, 500, 1000
    gt_rows = []
    for u in range(U):
        m = (0, 1, K, K + 7, 3 * K, int(rng.integers(0, 30)))[u % 6]    # none, one, exactly K, longer than K
        gt_rows.append(rng.choice(I, size=min(m, I), replace=False).tolist())
    ptr, col = _csr(gt_rows)
    users = rng.integers(0, U, n).astype(np.int64)
    topi = np.full((n, K), -1, dtype=np.int32)
    for r, u in enumerate(users):
        fill = int(rng.integers(0, K + 1)) if r % 3 else K           # some rows end in -1 padding
        pool = np.array(gt_rows[u] + rng.choice(I, size=K, replace=False).tolist())
        pick = list(dict.fromkeys(rng.permutation(pool).tolist()))[:fill]
        topi[r, :len(pick)] = pick
    got = ops.recall_ndcg(torch.as_tensor(topi, device=DEV), torch.as_tensor(users, device=DEV),
                          torch.as_tensor(ptr, device=DEV), torch.as_tensor(col, device=DEV)).cpu().numpy()
    rec, ndcg, cnt = _recall_ndcg_fp64(topi, users, gt_rows)
    assert got[2] == cnt
    assert got[0] == pytest.approx(rec, rel=1e-12) and got[1] == pytest.approx(ndcg, rel=1e-12)
    # and the oracle's own statement of the definition agrees
    o = oev.recall_ndcg_at_k(topi, [gt_rows[u] for u in users], K)
    assert o[2] == cnt and o[0] == pytest.approx(rec, rel=1e-12) and o[1] == pytest.approx(ndcg, rel=1e-12)


# ------------------------------------------------------------------ eligible_users across the multi-block scan
@pytest.mark.parametrize("with_keys", (False, True))
@pytest.mark.parametrize("n_users", (1, 8191, 8192, 8193, 3 * 8192 + 5))
def test_eligible_users_across_scan_tiles(n_users, with_keys):
    from recad_b200 import ops
    rng = np.random.default_rng(n_users + with_keys)
    I = 40
    targets = [3, 39]
    rows = []
    for u in range(n_users):
        kind = u % 7
        if kind == 0:
            rows.append([])
        elif kind == 1:
            rows.append(list(range(I)))                                  # every item: no candidate left
        elif kind == 2:
            rows.append([3, 10])                                         # holds a target
        else:
            rows.append(rng.choice(np.arange(4, 39), size=int(rng.integers(1, 6)), replace=False).tolist())
    ptr, col = _csr(rows)
    is_key = (rng.random(n_users) < 0.7).astype(np.uint8) if with_keys else None
    if is_key is not None:
        is_key[0] = 1                                                    # an empty row that is a key
    got = ops.eligible_users(torch.as_tensor(ptr, device=DEV), torch.as_tensor(col, device=DEV), n_users, I, targets,
                             None if is_key is None else torch.as_tensor(is_key, device=DEV)).cpu().numpy()
    keys = [u for u in range(n_users) if (is_key[u] if is_key is not None else len(rows[u]) > 0)]
    want = sorted(u for u in oev.eligible_users({u: rows[u] for u in keys}, targets) if len(rows[u]) < I)
    assert np.array_equal(got, np.asarray(want, dtype=np.int64))
