"""Oracle: full-ranking evaluation on CPU (numpy).

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Restates:
  * ``Normal.normal_evaluate``           recad/workflow/normal.py:111-160
  * ``Normal.user_item_model_generate``  recad/workflow/normal.py:57-93
  * test-mode batches (ground truth)     recad/dataset/implicit.py:461-476
  * ``LightGCN.getUsersRating``          recad/model/victim/lightgcn.py:115-120

HR@k / pred_shift are pinned against the live reference (tests/golden).
Recall/NDCG@20: PARITY UNPINNED -- the reference contains no Recall/NDCG code
(SURVEY.md section 0.2); the definition below is the upstream-LightGCN convention
built from the reference's own ingredients and is the only pin.

Tie rule (the reference's pandas quicksort is unspecified on ties, normal.py:86-88):
an item outranks the target iff score > s_t, or score == s_t and item_id < target.
Top-K lists order by (score desc, item id asc).
"""
import numpy as np


def eligible_users(train_dict, target_id_list):
    """normal.py:133-143: users of train_dict (dict order) that have NO target
    item in their train set."""
    tset = set(int(t) for t in target_id_list)
    return [u for u, v in train_dict.items() if not (tset & set(int(x) for x in v))]


def candidate_items(train_items, n_items):
    """normal.py:143: list(full_items - train_items); CPython iterates the small-int
    set ascending."""
    return np.setdiff1d(np.arange(n_items, dtype=np.int64), np.asarray(list(train_items), dtype=np.int64))


def target_rows_per_user(score_fn, train_dict, n_items, target_id_list, topks):
    """user_item_model_generate, user by user (slow, faithful): for each eligible
    user with a non-empty candidate list, score the candidates with
    ``score_fn(users[int64], items[int64]) -> float array``; row =
    [uid, score_target, 1[target in top-k] for k in topks].  One row per
    (user, target), users in ascending id order (pandas groupby sorts keys,
    normal.py:79)."""
    rows = []
    elig = sorted(eligible_users(train_dict, target_id_list))
    for u in elig:
        cand = candidate_items(train_dict[u], n_items)
        if len(cand) == 0:
            continue
        s = np.asarray(score_fn(np.full(len(cand), u, dtype=np.int64), cand), dtype=np.float64)
        for t in target_id_list:
            st = s[cand == t][0]
            rank = int(np.sum(s > st) + np.sum((s == st) & (cand < t)))
            rows.append([u, st] + [1 if rank < k else 0 for k in topks])
    return np.asarray(rows, dtype=np.float64).reshape(-1, 2 + len(topks))


def attack_table(rows_clean, rows_fake, topks):
    """normal.py:151-159: pred_shift and HR@k before / after attack."""
    assert np.allclose(rows_clean[:, 0], rows_fake[:, 0]), "Users are not aligned"
    out = {"pred_shift": float(np.mean(rows_fake[:, 1] - rows_clean[:, 1]))}
    for i, k in enumerate(topks):
        out[f"HR@{k}"] = float(np.mean(rows_clean[:, 2 + i]))
        out[f"HR@{k} after attack"] = float(np.mean(rows_fake[:, 2 + i]))
    return out


def full_rank_batched(user_emb, item_emb, user_ids, train_indptr, train_indices, targets, K):
    """Batched restatement for embedding-dot models: scores = U_b I^T in float32
    with a FIXED ascending-d summation order (matches the CUDA kernel's FMA order
    is not required: comparisons are made within one arithmetic), train items
    masked out.  Returns (topk_idx int64 [n, K] (-1 padded), topk_val float32,
    target_rank int64 [n, T] (-1 if the target is a train item), target_score)."""
    user_emb = np.asarray(user_emb, dtype=np.float32)
    item_emb = np.asarray(item_emb, dtype=np.float32)
    n, T, I = len(user_ids), len(targets), item_emb.shape[0]
    topi = -np.ones((n, K), dtype=np.int64)
    topv = np.full((n, K), -np.inf, dtype=np.float32)
    trank = -np.ones((n, T), dtype=np.int64)
    tscore = np.zeros((n, T), dtype=np.float32)
    ids = np.arange(I, dtype=np.int64)
    for r, u in enumerate(user_ids):
        s = fma_dot_rows(user_emb[u], item_emb)
        masked = np.zeros(I, dtype=bool)
        masked[train_indices[train_indptr[u]:train_indptr[u + 1]]] = True
        for j, t in enumerate(targets):
            tscore[r, j] = s[t]
            if not masked[t]:
                ok = ~masked
                trank[r, j] = int(np.sum(ok & (s > s[t])) + np.sum(ok & (s == s[t]) & (ids < t)))
        sm = np.where(masked, -np.inf, s).astype(np.float32)
        order = np.lexsort((ids, -sm.astype(np.float64)))[:K]
        order = order[~masked[order]]
        topi[r, :len(order)] = order
        topv[r, :len(order)] = sm[order]
    return topi, topv, trank, tscore


_F32_OVERFLOW_MID = 2.0 ** 128 - 2.0 ** 103      # halfway between FLT_MAX and 2^128: rounds to inf


def fmaf(a, b, c):
    """Correctly rounded float32 fused multiply-add a * b + c, elementwise (numpy broadcasting).
    The product of two float32 is exact in float64; the float64 sum s = p + c is not, and rounding it
    to float32 rounds twice.  That differs from one rounding of the exact sum only when s lies exactly
    on a float32 rounding midpoint while the exact sum does not, so the sum's rounding error e is
    recovered exactly (TwoSum) and, in that case, s is moved one float64 ulp toward e before the
    cast, which puts it on the same side of the midpoint as the exact sum."""
    p = np.asarray(a, dtype=np.float32).astype(np.float64) * np.asarray(b, dtype=np.float32).astype(np.float64)
    c = np.asarray(c, dtype=np.float32).astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        s = p + c
        bb = s - p
        e = (p - (s - bb)) + (c - bb)                       # TwoSum: p + c == s + e exactly (finite s)
        r32 = s.astype(np.float32)
        r = r32.astype(np.float64)
        # the other float32 neighbour of s; s is a midpoint iff it is the mean of the two (exact in float64)
        n = np.nextafter(r32, np.where(s > r, np.float32(np.inf), np.float32(-np.inf))).astype(np.float64)
        mid = (np.isfinite(r) & (s != r) & ((r + n) * 0.5 == s)) | (np.abs(s) == _F32_OVERFLOW_MID)
        mid &= e != 0
        s = np.where(mid, np.nextafter(s, np.where(e > 0, np.inf, -np.inf)), s)
        return s.astype(np.float32)


def fma_dot_rows(u, items):
    """Float32 dot of one user row against every item row, accumulated with a
    fused multiply-add per dimension in ascending d (acc = fma(u[d], i[d], acc)),
    each step correctly rounded as a hardware FMA is (fmaf above): bit for bit
    the exact CUDA-core kernel's chain."""
    acc = np.zeros(items.shape[0], dtype=np.float32)
    u = np.asarray(u, dtype=np.float32)
    items = np.asarray(items, dtype=np.float32)
    for d in range(items.shape[1]):
        acc = fmaf(u[d], items[:, d], acc)
    return acc


def recall_ndcg_at_k(topk_idx, ground_truth, K):
    """PARITY UNPINNED.  Upstream-LightGCN convention: per test user,
    recall = hits / |gt|; dcg = sum 1/log2(rank+2) over hits;
    idcg over min(|gt|, K); returns the SUMS over users and the user count
    (users with empty ground truth are skipped)."""
    rec, ndcg, cnt = 0.0, 0.0, 0
    for row, gt in zip(topk_idx, ground_truth):
        gt = set(int(g) for g in gt)
        if not gt:
            continue
        hits = np.array([1.0 if int(i) in gt else 0.0 for i in row[:K]])
        disc = 1.0 / np.log2(np.arange(2, K + 2))
        idcg = disc[:min(len(gt), K)].sum()
        rec += hits.sum() / len(gt)
        ndcg += (hits * disc).sum() / idcg
        cnt += 1
    return rec, ndcg, cnt
