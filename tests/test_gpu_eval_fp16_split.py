"""Full-rank tensor-core evaluation, fp16 two-term split: the device split against a numpy emulation (bit for bit),
scores against fp64 truth on inputs that stress the power-of-two scales, the tie rule across the two epilogue
warpgroups, and the 16-row target path against the item path."""
import ctypes as C

import numpy as np
import pytest
import torch

DEV = "cuda:0"
TILE, WIDTH, TGT_ROWS = 64, 64, 16


def scale_exp(m):
    """f16_scale_exp: 2^k with max|x| 2^k < 2^15; 0 for an all-zero block."""
    m = np.float32(m)
    if not (m > 0) or not np.isfinite(m):
        return 0
    return 15 - int(np.frexp(m)[1])


def split_block(x, k):
    """hi = fp16_rn(x 2^k), lo = fp16_rn(x 2^k - hi); 2^k applied as 2^(k/2) 2^(k - k/2) in float32, like the kernel."""
    a = int(k / 2)                                    # C division: truncates toward zero
    xs = (x.astype(np.float32) * np.float32(2.0 ** a)) * np.float32(2.0 ** (k - a))
    hi = xs.astype(np.float16)
    lo = (xs - hi.astype(np.float32)).astype(np.float16)
    return hi, lo


def emulate_items(ie, targets):
    """(hi, lo) fp16 [ip, 64], (t_hi, t_lo) fp16 [16, 64], kexp int32 [ip / 64 + 1] as the kernel writes them."""
    I, D = ie.shape
    ip = (I + TILE - 1) // TILE * TILE
    pad = np.zeros((ip, WIDTH), np.float32)
    pad[:I, :D] = ie
    hi, lo = np.zeros((ip, WIDTH), np.float16), np.zeros((ip, WIDTH), np.float16)
    kexp = []
    for t in range(ip // TILE):
        blk = pad[t * TILE:(t + 1) * TILE]
        k = scale_exp(np.abs(blk).max())
        kexp.append(k)
        hi[t * TILE:(t + 1) * TILE], lo[t * TILE:(t + 1) * TILE] = split_block(blk, k)
    tg = np.zeros((TGT_ROWS, WIDTH), np.float32)
    tg[:len(targets), :D] = ie[targets]
    k = scale_exp(np.abs(tg).max())
    kexp.append(k)
    t_hi, t_lo = split_block(tg, k)
    return hi, lo, t_hi, t_lo, np.array(kexp, np.int32)


def emulated_scores(ue, ie):
    """fp64 value of the three-pass product the kernel accumulates (hi.hi + lo.hi + hi.lo), scaled back."""
    hi, lo, _, _, kexp = emulate_items(ie, [])
    I = ie.shape[0]
    out = np.zeros((ue.shape[0], I))
    for r, u in enumerate(ue):
        ku = scale_exp(np.abs(u).max())
        uh, ul = (np.pad(x, (0, WIDTH - u.shape[0])).astype(np.float64) for x in split_block(u, ku))
        s = hi.astype(np.float64) @ uh + hi.astype(np.float64) @ ul + lo.astype(np.float64) @ uh
        out[r] = s[:I] * 2.0 ** -(ku + np.repeat(kexp[:-1], TILE)[:I])
    return out


def stressed_tables(rng, U, I, D):
    ue = rng.standard_normal((U, D)).astype(np.float32)
    ue[1::7] *= np.float32(1e-20)
    ue[2::7] *= np.float32(1e20)
    ie = rng.standard_normal((I, D)).astype(np.float32)
    ie *= np.exp2(rng.uniform(-10, 10, (I, 1))).astype(np.float32)     # item norms span 2^20 inside every tile
    return ue, ie


def test_fp16_split_scheme_is_fp32_accurate():
    """CPU check of the numerical scheme itself: hi.hi + lo.hi + hi.lo of the scaled split is within the bar the
    tensor-core tests use, on the stressed tables."""
    rng = np.random.default_rng(5)
    ue, ie = stressed_tables(rng, 64, 300, 64)
    S = ue.astype(np.float64) @ ie.astype(np.float64).T
    mag = np.abs(ue).astype(np.float64) @ np.abs(ie).astype(np.float64).T
    err = np.abs(emulated_scores(ue, ie) - S)
    assert np.all(err <= 3e-6 * mag)


def _lib():
    from recad_b200 import _lib
    return _lib.lib()


@pytest.mark.gpu
def test_item_split_matches_numpy_bit_for_bit():
    from recad_b200 import ops
    rng = np.random.default_rng(11)
    I, D = 6 * TILE + 17, 50
    ie = rng.standard_normal((I, D)).astype(np.float32)
    ie[0:TILE] *= np.float32(1e30)
    ie[TILE:2 * TILE] *= np.float32(1e-30)
    ie[2 * TILE:3 * TILE] = 0.0
    ie[2 * TILE + 5, 7] = -0.0
    ie[3 * TILE:4 * TILE] = (rng.standard_normal((TILE, D)) * 1e-39).astype(np.float32)     # fp32 subnormals
    ie[4 * TILE + 3, 9] = np.float32(2.0 ** 20) * np.abs(ie[4 * TILE:5 * TILE]).max()        # one outlier
    targets = [5, TILE + 1, 3 * TILE + 2, 4 * TILE + 3, I - 1]
    U, K = 4, 5
    ue = torch.ones((U, D), device=DEV)
    ie_d = torch.as_tensor(ie, device=DEV)
    ptr = torch.zeros(U + 1, dtype=torch.int64, device=DEV)
    col = torch.zeros(1, dtype=torch.int32, device=DEV)
    tg = torch.as_tensor(targets, dtype=torch.int32, device=DEV)
    T = len(targets)
    outs = ops._eval_outputs(U, T, K, ue.device)
    L = _lib()
    nfl = L.recad_fullrank_tc_scratch_floats(U, I)
    scratch = torch.zeros(nfl, dtype=torch.float32, device=DEV)
    with torch.cuda.device(DEV):
        ops.check(L.recad_fullrank_eval_tc(ops._ptr(ue), ops._ptr(ie_d), I, D, ops._ptr(torch.arange(U, device=DEV)), U,
                                           ops._ptr(ptr), ops._ptr(col), ops._ptr(tg), T, K, None, *map(ops._ptr, outs),
                                           ops._ptr(scratch), C.c_int64(nfl), ops._stream(ue.device)), "fullrank_tc")
    torch.cuda.synchronize()
    hi, lo, t_hi, t_lo, kexp = emulate_items(ie, targets)
    ip = hi.shape[0]
    raw = scratch.cpu().numpy().view(np.uint16)
    n = ip * WIDTH
    got = [raw[:n], raw[n:2 * n], raw[2 * n:2 * n + TGT_ROWS * WIDTH], raw[2 * n + TGT_ROWS * WIDTH:2 * n + 2 * TGT_ROWS * WIDTH]]
    for g, want in zip(got, (hi, lo, t_hi, t_lo)):
        assert np.array_equal(g, want.view(np.uint16).ravel())
    kx = scratch.cpu().numpy().view(np.int32)[(2 * n + 2 * TGT_ROWS * WIDTH) // 2:][:ip // TILE + 1]
    assert np.array_equal(kx, kexp)
    assert kexp[2] == 0 and kexp[0] < 0 < kexp[1]


def _train_csr(train, U):
    ptr = np.zeros(U + 1, np.int64)
    for u in range(U):
        ptr[u + 1] = ptr[u] + len(train[u])
    idx = np.array([i for u in range(U) for i in train[u]] or [0], np.int32)
    return ptr, idx


@pytest.mark.gpu
@pytest.mark.parametrize("D,K,T,bias", [(16, 1, 1, False), (50, 20, 8, True), (64, 32, 5, True), (64, 20, 3, False)])
def test_scaled_scores_match_fp64_truth(D, K, T, bias):
    from recad_b200 import ops
    rng = np.random.default_rng(D * 13 + K + T)
    U, I = 300, 1000
    ue, ie = stressed_tables(rng, U, I, D)
    ib = rng.standard_normal(I).astype(np.float32) if bias else None
    train = {u: sorted(rng.choice(I, size=rng.integers(0, 80), replace=False).tolist()) for u in range(U)}
    ptr, idx = _train_csr(train, U)
    users = np.arange(U, dtype=np.int64)
    targets = [int(t) for t in rng.choice(I, size=T, replace=False)]
    topi, topv, trank, tscore = ops.fullrank_eval(
        torch.as_tensor(ue, device=DEV), torch.as_tensor(ie, device=DEV), torch.as_tensor(users, device=DEV),
        torch.as_tensor(ptr, device=DEV), torch.as_tensor(idx, device=DEV), targets, K,
        item_bias=None if ib is None else torch.as_tensor(ib, device=DEV), precision="tf32x3")
    S = ue.astype(np.float64) @ ie.astype(np.float64).T + (0 if ib is None else ib.astype(np.float64))
    mag = np.abs(ue).astype(np.float64) @ np.abs(ie).astype(np.float64).T + (0 if ib is None else np.abs(ib).astype(np.float64))
    ts = tscore.cpu().numpy().astype(np.float64)
    for j, t in enumerate(targets):
        assert np.all(np.abs(ts[:, j] - S[:, t]) <= 3e-6 * mag[:, t]), "target score not fp32-accurate"
    rk, ti, tv = trank.cpu().numpy(), topi.cpu().numpy(), topv.cpu().numpy().astype(np.float64)
    ids = np.arange(I)
    n_bad = 0
    for r in range(U):
        masked = np.zeros(I, bool)
        masked[train[r]] = True
        for j, t in enumerate(targets):
            if masked[t]:
                assert rk[r, j] == -1
                continue
            true_rank = int(np.sum(~masked & (S[r] > S[r, t])) + np.sum(~masked & (S[r] == S[r, t]) & (ids < t)))
            assert abs(rk[r, j] - true_rank) <= 2
            n_bad += rk[r, j] != true_rank
        sm = np.where(masked, -np.inf, S[r])
        order = np.lexsort((ids, -sm))[:K]
        n_bad += int(np.sum(ti[r] != order) > 2)
        assert np.all(np.abs(tv[r] - S[r, ti[r]]) <= 3e-6 * mag[r, ti[r]])
    assert n_bad <= 0.01 * U * (T + 1)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [20, 32])
def test_ties_across_both_warpgroups(K):
    """All scores equal: the two epilogue warpgroups rank alternate 64-item tiles; the merged list is the K lowest
    ids and the rank of a target counts the items with a smaller id in both warpgroups' tiles."""
    from recad_b200 import ops
    U, I, D = 4, 300, 64
    ue = torch.full((U, D), 3.0, device=DEV)
    ie = torch.full((I, D), 0.5, device=DEV)
    trains = [[], [3, 40, 90, 150], [], list(range(48))]     # user 1: train items in both warpgroups' tiles; user 3:
    ptr = torch.tensor(np.cumsum([0] + [len(t) for t in trains]), device=DEV)   # a top-K drawn from tiles 0 and 1
    col = torch.tensor(sum(trains, []), dtype=torch.int32, device=DEV)
    targets = [10, 40, 70, 100, 299]                                         # tiles 0, 0, 1, 1, 4: warpgroups 0, 0, 1, 1, 0
    topi, topv, trank, _ = ops.fullrank_eval(ue, ie, torch.arange(U, device=DEV), ptr, col, targets, K, precision="tf32x3")
    rk = trank.cpu().numpy()
    for u in range(U):
        train = set(trains[u])
        for j, t in enumerate(targets):
            want = -1 if t in train else sum(1 for i in range(t) if i not in train)
            assert rk[u, j] == want, (u, t)
        want_top = [i for i in range(I) if i not in train][:K]
        assert topi[u].tolist() == want_top
    assert torch.all(topv == 3.0 * 0.5 * D)


@pytest.mark.gpu
@pytest.mark.parametrize("bias", [False, True])
def test_target_path_equals_item_path(bias):
    """A target item's score from the 16-row target tile equals its score from its item tile: when the two tiles get
    the same scale the bits agree, otherwise they agree to fp32 accuracy."""
    from recad_b200 import ops
    rng = np.random.default_rng(3)
    U, I, D, K = 200, 5 * TILE, 64, 32
    ue = rng.uniform(0.5, 1.0, (U, D)).astype(np.float32)
    ie = rng.uniform(-1.0, 1.0, (I, D)).astype(np.float32)
    same = [2 * TILE + 1, 2 * TILE + 9, 2 * TILE + 40]          # tile 2: its largest |x| lies in a target row
    ie[same] = rng.uniform(2.0, 3.0, (3, D)).astype(np.float32)
    ib = rng.standard_normal(I).astype(np.float32) if bias else None
    ptr = np.zeros(U + 1, np.int64)
    topi, topv, trank, tscore = ops.fullrank_eval(
        torch.as_tensor(ue, device=DEV), torch.as_tensor(ie, device=DEV), torch.arange(U, device=DEV),
        torch.as_tensor(ptr, device=DEV), torch.zeros(1, dtype=torch.int32, device=DEV), same, K,
        item_bias=None if ib is None else torch.as_tensor(ib, device=DEV), precision="tf32x3")
    ti, tv, ts = topi.cpu().numpy(), topv.cpu().numpy(), tscore.cpu().numpy()
    for j, t in enumerate(same):
        pos = np.argmax(ti == t, axis=1)
        assert np.all(ti[np.arange(U), pos] == t), "target not in the top-K"
        assert np.array_equal(tv[np.arange(U), pos], ts[:, j])
    # the target tile and the target's item tile scaled differently: same score to fp32 accuracy
    ie2 = ie.copy()
    ie2[3 * TILE:4 * TILE] *= np.float32(0.25)
    ie2[3 * TILE + 5] = rng.uniform(2.0, 3.0, D).astype(np.float32)
    ie2[4 * TILE + 7] = rng.uniform(5.0, 6.0, D).astype(np.float32)        # the target tile's largest |x|
    t2 = [3 * TILE + 5, 4 * TILE + 7]
    topi, topv, _, tscore = ops.fullrank_eval(
        torch.as_tensor(ue, device=DEV), torch.as_tensor(ie2, device=DEV), torch.arange(U, device=DEV),
        torch.as_tensor(ptr, device=DEV), torch.zeros(1, dtype=torch.int32, device=DEV), t2, K, precision="tf32x3")
    ti, tv, ts = topi.cpu().numpy(), topv.cpu().numpy(), tscore.cpu().numpy()
    pos = np.argmax(ti == t2[0], axis=1)
    assert np.all(ti[np.arange(U), pos] == t2[0])
    assert np.allclose(tv[np.arange(U), pos], ts[:, 0], rtol=1e-6, atol=0)
