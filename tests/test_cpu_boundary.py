"""CPU-only checks of the boundary: the shared library exports every symbol the header declares,
the host-side mirror of the reference interface behaves like the reference (lazy `.I()`, reset,
dataset flattening / sampling / injection bookkeeping), and the product fails LOUDLY without CUDA
(no CPU fallback).  No kernel is launched here."""
import os
import re

import numpy as np
import pytest
import torch

from oracle import graph as og
from recad_b200 import _lib, config, dataset, evaluate, model, ops
from tests import util

META = util.meta()
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CPU = torch.device("cpu")


def test_library_exports_every_header_symbol():
    header = open(os.path.join(ROOT, "include", "recad_b200.h")).read()
    declared = set(re.findall(r"\b(recad_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    lib = _lib.lib()                      # loads + binds every symbol of SIGNATURES
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    for name in declared:
        assert hasattr(lib, name)
    assert lib.recad_abi_version() == 2


def test_struct_layouts_match_header_sizes():
    # natural alignment, 8-byte pointers: catches a field added on one side only
    import ctypes as C
    assert C.sizeof(_lib.CSR) == 13 * 8
    assert C.sizeof(_lib.LightGCN) == 8 + 16 + 8 + 6 * 4 + 9 * 8 + 8
    assert C.sizeof(_lib.MF) == 16 + 6 * 4 + 17 * 8
    assert C.sizeof(_lib.NCF) == 16 + 8 + 16 + 8 + 4 * 8 + 8 + 8 + 8 + 8 + 8
    assert C.sizeof(_lib.Aush) == 8 + 2 * 4 + 4 * 4 + 9 * 8
    assert C.sizeof(_lib.AushEpoch) == 8 + 2 * 4 + 9 * 8


def test_host_error_paths_report_through_last_error():
    lib = _lib.lib()
    rc = lib.recad_mt19937_permutation(None, None, 5, None)
    assert rc == -1 and b"bad argument" in lib.recad_last_error()
    with pytest.raises(_lib.RecadError):
        _lib.check(rc, "recad_mt19937_permutation")
    # argument validation of the device entry points happens before any launch, so it is testable without a GPU
    assert lib.recad_spmm_scatter(None, None, None, 2, 10, 64, None) < 0 and b"spmm_scatter" in lib.recad_last_error()
    assert lib.recad_peer_reduce_bcast(None, 2, 8, 8, None, 2, 0, None) < 0 and b"peer_reduce_bcast" in lib.recad_last_error()
    assert lib.recad_mf_grad(None, None, None, 4, 4, None) < 0 and b"mf" in lib.recad_last_error()
    assert lib.recad_ncf_grad(None, None, None, 4, 4, None) < 0
    assert lib.recad_mt19937_permutation_draw(None, None, 5, None) < 0 and b"permutation_draw" in lib.recad_last_error()
    assert lib.recad_permutation_apply(5, None, None) < 0 and b"permutation_apply" in lib.recad_last_error()
    assert lib.recad_aush_train_epoch(None, None, 0, None, None) < 0 and b"aush_train_epoch" in lib.recad_last_error()
    assert lib.recad_aush_generate(None, None, None, 4, None, None) < 0 and lib.recad_aush_plan_columns(None, 4, 2, 3, 10, None, None) < 0
    assert lib.recad_mt19937_aush_batch(None, None, 4, None, None, None, None, 3, 1, None, 0.2, None, None, None) < 0
    assert lib.recad_fullrank_eval_tc(None, None, 10, 64, None, 4, None, None, None, 0, 20, None, None, None, None, None, None, 0,
                                      None) < 0 and b"fullrank_tc" in lib.recad_last_error()


def test_no_cpu_fallback_anywhere():
    tr, va, te = util.dicts("dev")
    with pytest.raises(ops.RecadError):
        dataset.from_config("implicit", "dev", train_dict=tr, valid_dict=va, test_dict=te, need_graph=True, device=CPU)
    data = dataset.from_config("implicit", "dev", train_dict=tr, valid_dict=va, test_dict=te, need_graph=False,
                               sample="pointwise", device=CPU)
    lazy = model.from_config("victim", "mf", embedding_size=64, device=CPU)
    with pytest.raises(config.InstantiateFail):
        lazy.I(dataset=data)
    with pytest.raises(ops.RecadError):
        ops.spmm(None, torch.zeros(4, 4))
    src = "".join(open(os.path.join(dp, f)).read() for dp, _, fs in os.walk(os.path.join(ROOT, "recad_b200"))
                  for f in fs if f.endswith(".py"))
    assert "import oracle" not in src and "from oracle" not in src, "the product must never import the oracle"


def test_lazy_contract_like_reference():
    lazy = model.from_config("victim", "lightgcn", latent_dim_rec=64, not_a_key=1)
    assert lazy.model_name == "lightgcn" and lazy._init_config["latent_dim_rec"] == 64
    assert "not_a_key" not in lazy._init_config                      # unknown keys dropped (model/base.py:41-47)
    with pytest.raises(config.NotInstantiatedError):
        lazy.train_step()
    with pytest.raises(config.NotInstantiatedError):
        lazy(torch.zeros(1), torch.zeros(1))
    again = lazy.reset(lr=0.01)
    assert again._init_config["lr"] == 0.01 and again._init_config["latent_dim_rec"] == 64 and not again._is_instantiate
    with pytest.raises(ValueError):
        lazy.reset(bogus=1)
    assert set(lazy.input_describe()["forward"]) == {"users", "items"}
    assert len(lazy.output_describe()["train_step"]) == 1


def test_dataset_host_side_matches_reference_bookkeeping():
    tr, va, te = util.dicts("dev")
    z = util.load("dev_graph.npz")
    d = dataset.from_config("implicit", "dev", train_dict=tr, valid_dict=va, test_dict=te, need_graph=False, device=CPU)
    m = META["dev"]
    assert (d.n_users, d.n_items, d.traindataSize, d.validDataSize, d.testDataSize) == \
        (m["n_users"], m["n_items"], m["train"], m["valid"], m["test"])
    # reference quirk (SURVEY 0.1): UserItemNet / allPos come from the LAST split read = test
    assert np.array_equal(d._allpos[0], z["allpos_indptr"]) and np.array_equal(d._allpos[1], z["allpos_indices"])
    assert len(d.trainUser) == m["test"]
    d2 = dataset.from_config("implicit", "dev", train_dict=tr, valid_dict=va, test_dict=te, need_graph=False, device=CPU,
                             graph_edges="train")
    assert np.array_equal(d2._allpos[0], z["allpos_indptr_train"]) and np.array_equal(d2._allpos[1], z["allpos_indices_train"])
    info = d.info_describe()
    assert info["train_dict"] is tr and info["n_users"] == m["n_users"] and "graph" not in info
    ptr, col = d.train_csr()
    rp, ri = og.all_pos(*og.flatten_dict(tr)[:2], d.n_users, d.n_items)
    assert np.array_equal(ptr, rp) and np.array_equal(col, ri)


def test_generate_batch_replays_reference_stream_on_host():
    tr, va, te = util.dicts("dev")
    g = util.load("samplers.npz")
    d = dataset.from_config("implicit", "dev", train_dict=tr, valid_dict=va, test_dict=te, need_graph=False, device=CPU)
    np.random.seed(2023)
    batches = list(d.generate_batch())
    S = g["dev_pairwise"][g["dev_perm"]]
    got = torch.stack([torch.cat([b[k] for b in batches]) for k in ("users", "positive_items", "negative_items")], 1).numpy()
    assert np.array_equal(got, S)
    assert [len(b["users"]) for b in batches] == [len(S)]              # 16 triples < 1024: one ragged batch
    dp = dataset.from_config("implicit", "dev", train_dict=tr, valid_dict=va, test_dict=te, need_graph=False, device=CPU,
                             sample="pointwise", pointwise_batch_size=1000)
    st = ("MT19937", g["dev_state_key_after_pairwise"], int(g["dev_state_pos_after_pairwise"]), 0, 0.0)
    np.random.set_state(st)
    ops.mt_permutation(len(g["dev_pairwise"]))
    P = g["dev_pointwise"]
    batches = list(dp.generate_batch())
    assert [len(b["users"]) for b in batches] == [1000, 1000, len(P) - 2000]
    got = torch.stack([torch.cat([b[k] for b in batches]) for k in ("users", "items", "labels")], 1).numpy()
    assert sorted(map(tuple, got.tolist())) == sorted(map(tuple, P.tolist()))      # same multiset (then shuffled)
    assert np.array_equal(np.random.get_state()[1], np.random.get_state()[1])
    d.switch_mode("test")
    tb = list(d.generate_batch())
    assert sum(len(b["users"]) for b in tb) == len(te) and tb[0]["ground_truth"][0] == te[int(tb[0]["users"][0])]


def test_inject_and_delete_bookkeeping():
    tr, va, te = util.dicts("dev")
    d = dataset.from_config("implicit", "dev", train_dict=tr, valid_dict=va, test_dict=te, need_graph=False, device=CPU,
                            sample="pointwise")
    fake = np.zeros((50, d.n_items))
    fake[:, 0] = 5
    fake[3, 7] = 4          # == filter_num: dropped (strict >)
    fake[3, 9] = 4.5
    new = d.inject_data("explicit", fake, filter_num=4)
    assert new is not d and new.n_users == d.n_users + 50 and new.traindataSize == d.traindataSize + 51
    assert new.train_dict[d.n_users + 3] == [0, 9] and d.n_users + 3 not in d.train_dict
    assert new.train_dict == og.inject(tr, fake, d.n_users, 4)
    again = new.inject_data("explicit", fake[:2], filter_num=4)      # a second injection stacks on top
    assert again.n_users == new.n_users + 2
    with pytest.raises(NotImplementedError):
        d.inject_data("implicit", fake)
    kept = d.delete_data("explicit", [d.n_users + 1, 0], fake, filter_num=4)
    assert d.n_users + 1 not in kept.train_dict and 0 not in kept.train_dict and d.n_users + 2 in kept.train_dict
    sub = d.partial_sample(user_ratio=0.5)
    assert len(sub.train_dict) == len(tr) // 2 and d.partial_sample(user_ratio=1) is d


def test_eligible_users_like_reference():
    tr, va, te = util.dicts("dev")
    d = dataset.from_config("implicit", "dev", train_dict=tr, valid_dict=va, test_dict=te, need_graph=False, device=CPU)
    from oracle import evaluate as oev
    for tg in ([0], [5], [0, 5, 62]):
        assert evaluate.eligible_users(d, tg).tolist() == sorted(oev.eligible_users(tr, tg))


def test_fast_filter_sampler_is_bit_identical_to_the_plain_one():
    """The filter-based parser used for large epochs draws exactly the same samples and leaves exactly the same
    RNG state as the plain one (and hence as the reference), including heavy users (> 96 positives)."""
    tr, va, te = util.dicts("game")
    m = META["game"]
    U, I = m["n_users"], m["n_items"]
    u, i, _, _ = og.flatten_dict(tr)
    ptr, idx = og.all_pos(u, i, U, I)
    ptr, idx = np.ascontiguousarray(ptr), np.ascontiguousarray(idx, dtype=np.int32)
    assert np.diff(ptr).max() > 96
    old = ops.FAST_SAMPLER_MIN
    try:
        outs = []
        for thr in (1 << 60, 0):
            ops.FAST_SAMPLER_MIN = thr
            np.random.seed(7)
            S = ops.mt_pairwise(U, I, 200_000, ptr, idx)
            outs.append((S.copy(), np.random.get_state()[1].copy(), np.random.get_state()[2]))
    finally:
        ops.FAST_SAMPLER_MIN = old
    assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1]) and outs[0][2] == outs[1][2]
    from oracle import sampler as osm
    np.random.seed(7)
    ref = osm.pairwise_sample_numpy(U, I, 3000, ptr, idx)
    ops.FAST_SAMPLER_MIN = 0
    try:
        np.random.seed(7)
        assert np.array_equal(ops.mt_pairwise(U, I, 3000, ptr, idx), ref)
    finally:
        ops.FAST_SAMPLER_MIN = old


def test_workflow_registry_mirrors_reference():
    """recad/workflow/__init__.py:4-7: both workflows, the required user arguments raise a TypeError when missing."""
    import pytest
    from recad_b200 import config, workflow
    assert set(workflow.factories) == {"no defense", "defense"}
    assert config.WORKFLOW["defense"]["defense_epoch"] == 1 and config.WORKFLOW["no defense"]["topks"] == [10, 20, 50, 100]
    with pytest.raises(TypeError):
        workflow.from_config("defense", victim_data=None, attack_data=None, victim=None, attacker=None)
    with pytest.raises(TypeError):
        workflow.from_config("no defense", victim_data=None)


def test_prefetched_epochs_equal_synchronous_epochs():
    """The depth-2 prefetch queue (sampler chained epoch to epoch, swaps applied on the side) hands out exactly the
    epochs a synchronous draw produces, leaves np.random where the reference would, and steps aside (same stream!)
    when somebody else consumes np.random between two epochs."""
    tr, va, te = util.dicts("game")
    mk = lambda pf: dataset.from_config("implicit", "game", train_dict=tr, valid_dict=va, test_dict=te, need_graph=False,  # noqa: E731
                                        device=CPU, prefetch=pf)
    runs = []
    for pf in (False, True):
        d = mk(pf)
        np.random.seed(11)
        seq = []
        for e in range(5):
            if e == 3:
                np.random.randint(0, 10, 7)          # a foreign consumer: queued epochs no longer match the stream
            s, p = d.epoch_samples(CPU)
            seq.append((s.numpy().copy(), p.numpy().copy(), np.random.get_state()[1].copy(), int(np.random.get_state()[2])))
        if pf:
            assert d._pipe.prefetch and len(d._pipe.queue) == d._pipe.DEPTH
            d._pipe._flush()
        runs.append(seq)
    for a, b in zip(*runs):
        assert all(np.array_equal(x, y) for x, y in zip(a[:3], b[:3])) and a[3] == b[3]
    # and the synchronous epoch is the reference's: sampler then np.random.shuffle on the same stream
    np.random.seed(11)
    S, P = runs[0][0][0], runs[0][0][1]
    ptr, col = mk(False)._allpos
    ref = ops.mt_pairwise(META["game"]["n_users"], META["game"]["n_items"], mk(False).traindataSize, ptr, col)
    idx = np.arange(len(ref))
    np.random.shuffle(idx)
    assert np.array_equal(S, ref) and np.array_equal(P, idx)


def test_fast_sampler_rewinds_are_exact_on_a_dense_dataset():
    """Worst case for the optimistic block parser: 64 items, users holding 0..40 of them -- a third of the first
    negative candidates ARE positives, so nearly every block is rewound several times (and users without positives
    are dropped).  Samples and generator state must still equal the plain loop's, whatever the number of helper threads
    (RECAD_SAMPLER_HELPERS=0 runs one)."""
    import os
    rng = np.random.default_rng(3)
    U, I, n = 5000, 64, 300_000
    lens = rng.integers(0, 41, size=U)
    lens[rng.integers(0, U, 200)] = 0
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col = np.concatenate([np.sort(rng.choice(I, size=k, replace=False)) for k in lens] + [np.zeros(0, np.int64)]).astype(np.int32)
    old = ops.FAST_SAMPLER_MIN
    outs = []
    try:
        for thr, helpers in ((1 << 60, None), (0, "0"), (0, "3"), (0, None)):
            ops.FAST_SAMPLER_MIN = thr
            if helpers is None:
                os.environ.pop("RECAD_SAMPLER_HELPERS", None)
            else:
                os.environ["RECAD_SAMPLER_HELPERS"] = helpers
            np.random.seed(21)
            S = ops.mt_pairwise(U, I, n, ptr, col)
            outs.append((S.copy(), np.random.get_state()[1].copy(), int(np.random.get_state()[2])))
    finally:
        ops.FAST_SAMPLER_MIN = old
        os.environ.pop("RECAD_SAMPLER_HELPERS", None)
    assert len(outs[0][0]) < n                                   # the users without positives were dropped
    for o in outs[1:]:
        assert np.array_equal(o[0], outs[0][0]) and np.array_equal(o[1], outs[0][1]) and o[2] == outs[0][2]
    pos_sets = [set(col[ptr[u]:ptr[u + 1]].tolist()) for u in range(U)]
    S = outs[0][0]
    assert all(int(p) in pos_sets[int(u)] and int(q) not in pos_sets[int(u)] for u, p, q in S[:5000])


def test_sampler_caches_do_not_mix_datasets():
    """The filter blocks / sorted lists derived from a dataset's positives are cached per dataset: alternating between
    two datasets of identical shape (the clean and the attacked one of a workflow, whose epochs are drawn by different
    threads) must give each its own results."""
    rng = np.random.default_rng(8)
    U, I, n = 400, 300, 20_000

    def make():
        lens = rng.integers(1, 30, size=U)
        ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        col = np.concatenate([np.sort(rng.choice(I, size=k, replace=False)) for k in lens]).astype(np.int32)
        return ptr, col
    sets = [make(), make()]
    old = ops.FAST_SAMPLER_MIN
    try:
        want = []
        ops.FAST_SAMPLER_MIN = 1 << 60
        for ptr, col in sets:
            np.random.seed(4)
            want.append(ops.mt_pairwise(U, I, n, ptr, col).copy())
        ops.FAST_SAMPLER_MIN = 0
        for _ in range(2):
            for k, (ptr, col) in enumerate(sets):
                np.random.seed(4)
                assert np.array_equal(ops.mt_pairwise(U, I, n, ptr, col), want[k])
    finally:
        ops.FAST_SAMPLER_MIN = old
    # pointwise: per-user sorted lists are cached per (items, rowptr) pair
    keys = np.arange(U, dtype=np.int64)
    outs = []
    for rnd in range(2):
        for ptr, col in sets:
            np.random.seed(9)
            st, key, pos = ops._np_state()
            outs.append(ops.mt_pointwise_raw(key, pos, keys, ptr, col.astype(np.int64), I, 2).copy())
    assert np.array_equal(outs[0], outs[2]) and np.array_equal(outs[1], outs[3]) and not np.array_equal(outs[0], outs[1])


def test_csv_loader_and_dict_cache(tmp_path):
    """csv2dict (implicit.py:94-104): time order, rating >= filter, first occurrence kept; the .npy dict cache of
    implicit.py:153-164 is written and read back under the reference's file names."""
    import os
    from recad_b200.dataset import csv2dict
    rows = [(0, 7, 3, 5, 50), (1, 7, 9, 4, 10), (2, 7, 3, 5, 60), (3, 2, 1, 3, 5), (4, 2, 8, 5, 7), (5, 7, 4, 2, 20), (6, 5, 0, 4, 1)]
    for split in ("train", "valid", "test"):
        with open(tmp_path / f"toy_{split}.csv", "w") as f:
            f.write(",user_id,item_id,rating,timestamp\n" + "".join(f"{a},{u},{i},{r},{t}\n" for a, u, i, r, t in rows))
    d = csv2dict(str(tmp_path / "toy_train.csv"), filter=4)
    assert d == {5: [0], 2: [8], 7: [9, 3]} and list(d) == [5, 2, 7]          # dict order = first appearance in time
    kw = dict(path_train=str(tmp_path / "toy_train.csv"), path_valid=str(tmp_path / "toy_valid.csv"),
              path_test=str(tmp_path / "toy_test.csv"), need_graph=False, device=CPU, if_cache=True, cache_dir=str(tmp_path / "gen"))
    a = dataset.from_config("implicit", "toy", **kw)
    assert sorted(os.listdir(tmp_path / "gen")) == [f"toy_implicit_{s}_dict.npy" for s in ("test", "train", "valid")]
    for split in ("train", "valid", "test"):
        os.remove(tmp_path / f"toy_{split}.csv")                                  # second load must come from the cache
    b = dataset.from_config("implicit", "toy", **kw)
    assert b.train_dict == a.train_dict == d and (b.n_users, b.n_items) == (8, 10)


@pytest.mark.reference
def test_csv_loader_reproduces_the_golden_dev_dicts():
    import os
    from recad_b200.dataset import csv2dict
    root = os.path.join(util.REFERENCE, "data", "dev")
    tr, va, te = util.dicts("dev")
    for split, want in (("train", tr), ("valid", va), ("test", te)):
        got = csv2dict(os.path.join(root, f"dev_{split}.csv"), filter=4)
        assert got == want and list(got) == list(want)


def test_pointwise_sampler_dense_users_follow_cpython_set_order():
    """implicit.py:86 `list(full_items - set(iids))` is ascending only while CPython copies the full set and discards;
    from len(set(iids)) >= n_items / 4 the difference is rebuilt into a smaller hash table and the list follows its
    slot order.  The C++ replay emulates that table: same negatives, same generator state as the reference's Python."""
    def ref_pointwise(train_dict, n_items, ratio):          # implicit.py:77-91 verbatim in behaviour
        data = []
        full_items = set(range(n_items))
        for uid, iids in train_dict.items():
            data.extend([(uid, iid, 1) for iid in iids])
            left_set = list(full_items - set(iids))
            negs = np.random.choice(left_set, size=len(iids) * ratio)
            data.extend([(uid, ni, 0) for ni in negs])
        return np.array(data)
    rng = np.random.default_rng(3)
    for n_items, fracs in [(1000, [0.1, 0.24, 0.25, 0.26, 0.7, 0.99]), (3706, [0.2, 0.8]), (10000, [0.55]), (17, [0.5, 0.9])]:
        d = {u: [int(x) for x in rng.permutation(n_items)[:max(1, min(n_items - 1, int(n_items * f)))]] for u, f in enumerate(fracs)}
        d[len(fracs)] = [5, 5, 7, 5]                         # duplicated positives
        np.random.seed(11)
        ref = ref_pointwise(d, n_items, 2)
        st_ref = np.random.get_state()
        np.random.seed(11)
        keys = np.array(list(d), np.int64)
        ptr = np.concatenate([[0], np.cumsum([len(v) for v in d.values()])]).astype(np.int64)
        items = np.concatenate([np.array(v, np.int64) for v in d.values()])
        got = ops.mt_pointwise(keys, ptr, items, n_items, 2)
        st = np.random.get_state()
        assert np.array_equal(got, ref), n_items
        assert np.array_equal(st[1], st_ref[1]) and st[2] == st_ref[2]


def test_soa_epoch_sampler_equals_plain_sampler_and_shuffle():
    """recad_mt19937_pairwise_soa (stream producer thread, pre-gathered lengths, optimistic parse with exact redo and
    re-convergence, 32-bit arrays) == recad_mt19937_pairwise + recad_mt19937_permutation_draw: users, positives
    (through the row index), negatives, shuffle draws, generator state -- including users without positives, a
    one-user dataset and a dataset where nearly every optimistic candidate is a positive."""
    import ctypes as C
    rng = np.random.default_rng(1)
    for U, I, deg, n, empty in [(2000, 64, 20, 60000, 0.0), (3000, 3000, 40, 300000, 0.01), (1, 7, 3, 3000, 0.0), (40, 16, 15, 20000, 0.1)]:
        ptr, cols = [0], []
        for u in range(U):
            d = 0 if rng.random() < empty else int(min(I - 1, max(1, rng.poisson(deg))))
            cols.append(np.sort(rng.choice(I, d, replace=False)).astype(np.int32))
            ptr.append(ptr[-1] + d)
        ptr, col = np.array(ptr, np.int64), np.concatenate(cols)
        for seed in (0, 5):
            np.random.seed(seed)
            _, key, pos = ops._np_state()
            pos = [(pos[0] + seed * 100) % 625]
            key2, pos2 = key.copy(), [pos[0]]
            out, n_out, cpos = np.empty((n, 3), np.int64), C.c_int64(), C.c_int32(pos[0])
            _lib.check(_lib.lib().recad_mt19937_pairwise(key.ctypes.data, C.byref(cpos), U, I, n, ptr.ctypes.data, col.ctypes.data,
                                                         out.ctypes.data, C.byref(n_out)), "recad_mt19937_pairwise")
            S, pos = out[:n_out.value], [cpos.value]
            j_ref = ops.mt_permutation_draw_raw(key, pos, len(S))
            users, rel, negs, j = (np.empty(n, np.uint32) for _ in range(4))
            m = ops.mt_pairwise_soa_raw(key2, pos2, U, I, n, ptr, col, users, rel, negs, j)
            assert m == len(S)
            assert np.array_equal(users[:m], S[:, 0]) and np.array_equal(col[ptr[users[:m]] + rel[:m]], S[:, 1])
            assert np.array_equal(negs[:m], S[:, 2]) and np.array_equal(j[:m], j_ref)
            assert np.array_equal(key2, key) and pos2[0] == pos[0]
            perm32 = ops.permutation_apply32(j[:m], np.empty(max(m, 1), np.int32))
            assert np.array_equal(perm32, ops.permutation_apply(j_ref))


def test_scalar_and_avx512_stream_parse_agree(monkeypatch):
    """The AVX-512 window parse (csrc/sampler_avx512.cpp, taken when the CPU has it) and the scalar parse produce the same
    samples, shuffle draws and generator state."""
    rng = np.random.default_rng(3)
    U, I, n = 4000, 500, 200000
    lens = rng.integers(0, 70, U)
    lens[::97] = 0                                           # users without positives are dropped (implicit.py:63-64)
    ptr = np.zeros(U + 1, np.int64)
    np.cumsum(lens, out=ptr[1:])
    col = np.concatenate([np.sort(rng.choice(I, l, replace=False)) for l in lens]).astype(np.int32)
    outs = []
    for scalar in ("1", "0"):
        monkeypatch.setenv("RECAD_SAMPLER_SCALAR", scalar)
        np.random.seed(12)
        _, key, pos = ops._np_state()
        users, rel, negs, j = (np.empty(n, np.uint32) for _ in range(4))
        m = ops.mt_pairwise_soa_raw(key, pos, U, I, n, ptr, col, users, rel, negs, j)
        outs.append((m, users[:m].copy(), rel[:m].copy(), negs[:m].copy(), j[:m].copy(), key.copy(), pos[0]))
    a, b = outs
    assert a[0] == b[0] and all(np.array_equal(x, y) for x, y in zip(a[1:6], b[1:6])) and a[6] == b[6]


def test_injected_dataset_reuses_the_parents_sampler_filter():
    """ops.filter_parent_hint: the per-user filter blocks of a dataset derived by appending rows equal a build from scratch."""
    rng = np.random.default_rng(0)
    U, I, F = 5000, 800, 7
    lens = rng.integers(0, 60, U)
    ptr = np.zeros(U + 1, np.int64)
    np.cumsum(lens, out=ptr[1:])
    col = np.concatenate([np.sort(rng.choice(I, l, replace=False)) for l in lens]).astype(np.int32)
    ops.pairwise_filter(ptr, col, U)
    fl = rng.integers(1, 40, F)
    fptr = np.concatenate([[0], np.cumsum(fl)])
    fcol = np.concatenate([np.sort(rng.choice(I, l, replace=False)) for l in fl]).astype(np.int32)
    nptr = np.concatenate([ptr, ptr[-1] + fptr[1:]]).astype(np.int64)
    ncol = np.concatenate([col, fcol]).astype(np.int32)
    ops.filter_parent_hint(nptr, ncol, ptr, col, U)
    f1, e1 = ops.pairwise_filter(nptr, ncol, U + F)
    nptr2, ncol2 = nptr.copy(), ncol.copy()
    f2, e2 = ops.pairwise_filter(nptr2, ncol2, U + F)
    assert np.array_equal(f1, f2) and np.array_equal(e1, e2)


def test_aush_host_draws_and_column_plan_match_the_oracle():
    """Host half of the AUSH step: recad_mt19937_aush_batch consumes np.random exactly as the reference's sample_fillers +
    ZR-pool shuffle (restated in oracle/aush.py, which the golden run pins), and recad_aush_plan_columns groups the sparse
    discriminator inputs by column in row order.  No kernel is launched: the attacker object is assembled without its
    device state."""
    import ctypes as C
    from oracle import aush as oa
    from recad_b200 import attacker
    mat, _, _, kw, batch, targets, _ = util.aush_case("b")
    a = attacker.Aush.__new__(attacker.Aush)
    a._mat, a.n_items, a.selected_ids, a._sel = mat, mat.shape[1], kw["selected_ids"], np.unique(np.asarray(kw["selected_ids"]))
    a.filler_num, a.ZR_ratio, a._cand = kw["filler_num"], kw["ZR_ratio"], {}
    np.random.seed(5)
    elig = oa.eligible_rows(mat, a.selected_ids, targets, a.filler_num)
    assert np.array_equal(elig, attacker.filler_filter_mat(mat, targets, a.selected_ids, a.filler_num))
    users = np.random.permutation(elig)[:batch]
    st = np.random.get_state()
    real = mat[users]
    fill = oa.draw_fillers(real, a.n_items, a.selected_ids, targets, a.filler_num)
    sel = np.zeros_like(fill)
    sel[:, a.selected_ids] = 1
    zr = oa.draw_zr(real, sel, a.ZR_ratio)
    after = np.random.get_state()
    np.random.set_state(st)
    cols, tval, zr2 = a._draw_batch(users, targets)
    mine = np.random.get_state()
    assert np.array_equal(after[1], mine[1]) and after[2] == mine[2]
    f2 = np.zeros_like(fill)
    f2[np.arange(len(users))[:, None], cols] = 1
    assert np.array_equal(fill, f2) and np.array_equal(zr[:, a._sel], zr2)
    dense = np.zeros_like(fill)
    np.add.at(dense, (np.arange(len(users))[:, None], cols), tval)           # repeats carry 0: the sum IS the template
    assert np.array_equal(dense, real * fill)
    # column plan of two ragged batches
    F, S, I, n = a.filler_num, len(a._sel), a.n_items, len(users)
    b2 = 64
    nb = (n + b2 - 1) // b2
    colptr, ent = np.empty((nb, I + 1), dtype=np.int32), np.empty(n * F, dtype=np.int32)
    vp = lambda x: C.c_void_p(x.ctypes.data)
    _lib.check(_lib.lib().recad_aush_plan_columns(vp(cols), n, b2, F, I, vp(colptr), vp(ent)), "plan")
    for k in range(nb):
        lo, hi = k * b2, min(n, (k + 1) * b2)
        order = np.argsort(cols[lo:hi].ravel(), kind="stable")
        assert np.array_equal(ent[lo * F:hi * F], order)
        assert np.array_equal(colptr[k], np.concatenate([[0], np.cumsum(np.bincount(cols[lo:hi].ravel(), minlength=I))]))


def test_explicit_dataset_batches_are_lazy_and_sum_repeated_rows():
    """explicit.py:110-119 builds the rating matrix with scipy's csr (repeated (user, item) rows add up); the batch dict
    makes `users_mat` only when a consumer asks for it."""
    from recad_b200 import explicit
    ex = util.load("dev_explicit.npz")
    d = explicit.ExplicitData.from_config("dev", device=CPU, train_dict=ex["train"].copy(), valid_dict=ex["valid"].copy(),
                                          test_dict=ex["test"].copy())
    assert (d.n_users, d.n_items) == (int(ex["n_users"]), int(ex["n_items"]))
    kvr = np.array([[0, 1, 3], [0, 1, 2], [2, 0, 5]], dtype=np.float64)
    assert np.array_equal(explicit.ExplicitData.to_matrix(kvr, 3, 2), np.array([[0, 5], [0, 0], [5, 0]], dtype=np.float32))
    np.random.seed(0)
    batches = list(d.generate_batch())
    assert len(batches) == (d.n_users + 255) // 256 and sum(len(b["users"]) for b in batches) == d.n_users
    b = batches[0]
    assert not dict.__contains__(b, "users_mat") and "users_mat" in b and set(b.keys()) == {"users", "users_mat"}
    assert np.array_equal(b["users_mat"].numpy(), d.train_mat[b["users"].numpy()])
    with pytest.raises(KeyError):
        b["nope"]


def test_csv_loader_index_arithmetic_equals_the_row_loop(tmp_path):
    """csv2dict (implicit.py:94-104) on a CSV with timestamp ties, repeated (user, item) pairs and ratings below the filter:
    the vectorised form must give the dict of the reference's row loop -- same key order, same item order."""
    import pandas as pd
    rng = np.random.default_rng(5)
    n = 20000
    df = pd.DataFrame({"user_id": rng.integers(0, 300, n), "item_id": (rng.random(n) ** 2 * 200).astype(int),
                       "rating": rng.integers(1, 6, n), "timestamp": rng.integers(0, 500, n)})
    path = tmp_path / "x.csv"
    df.to_csv(path, index=False)
    got = dataset.csv2dict(str(path), 4)
    want = {}
    d = pd.read_csv(path).sort_values("timestamp")
    for u, i in zip(d[d["rating"] >= 4]["user_id"], d[d["rating"] >= 4]["item_id"]):
        lst = want.setdefault(int(u), [])
        if int(i) not in lst:
            lst.append(int(i))
    assert list(got) == list(want) and all(got[k] == want[k] for k in want)
    assert all(type(k) is int and all(type(x) is int for x in v) for k, v in got.items())
    (tmp_path / "empty.csv").write_text("user_id,item_id,rating,timestamp\n1,2,1,5\n")
    assert dataset.csv2dict(str(tmp_path / "empty.csv"), 4) == {}
