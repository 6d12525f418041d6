"""Drop-in for the reference's implicit-feedback dataset (recad/dataset/implicit.py)
with the graph built and kept on the device and the samplers replayed in C++.

Same public surface as `recad.dataset.implicit.ImplicitData` (SURVEY.md 8-b1):
``from_config(name, **kw)``, ``info_describe()``, ``batch_describe()``,
``generate_batch()``, ``mode()/switch_mode()``, ``inject_data()``,
``delete_data()``, ``partial_sample()``, ``reset()``, ``dataset_name``,
``print_help()``; plus ``epoch_samples()`` (the whole shuffled epoch as device
arrays, consumed by the C epoch drivers) and ``train_csr()`` (evaluation masks).
"""
import os
import random
from copy import copy
from pprint import pprint

import numpy as np
import torch

from . import ops
from .config import get_logger, implicit_defaults, merge_config


# --------------------------------------------------------------------------- #
# loading (implicit.py:94-127)
# --------------------------------------------------------------------------- #
def csv2dict(file, filter=4):
    """implicit.py:94-104: rows sorted by timestamp (pandas' default sort, as the reference: ties keep ITS order),
    rating >= filter, then per user the items in time order without repeats; users in order of first appearance.
    The reference does the last step with a Python loop and a linear `i not in list` scan per row (quadratic for heavy
    users); here it is index arithmetic on the sorted columns."""
    import pandas as pd
    df = pd.read_csv(file)
    df = df.sort_values("timestamp")
    df = df[df["rating"] >= filter]
    u = df["user_id"].to_numpy().astype(np.int64)
    i = df["item_id"].to_numpy().astype(np.int64)
    if len(u) == 0:
        return {}
    lo = int(i.min())
    key = u * (int(i.max()) - lo + 1) + (i - lo)
    first = np.sort(np.unique(key, return_index=True)[1])          # first occurrence of every (user, item) pair, in time order
    u, i = u[first], i[first]
    uniq, ufirst, inv = np.unique(u, return_index=True, return_inverse=True)
    rank = np.empty(len(uniq), dtype=np.int64)
    rank[np.argsort(ufirst)] = np.arange(len(uniq))                # a user's position in the dict = order of first appearance
    order = np.argsort(rank[inv], kind="stable")                   # stable: time order inside a user
    u, i = u[order], i[order]
    cut = np.flatnonzero(u[1:] != u[:-1]) + 1
    return {int(k): v.tolist() for k, v in zip(u[np.concatenate([[0], cut])], np.split(i, cut))}


def convert2dict(file, filter_num):
    if file.endswith(".csv"):
        return csv2dict(file, filter=filter_num)
    if file.endswith(".npy"):
        return np.load(file, allow_pickle=True).item()
    raise ValueError(f"Expect data file ends witg [csv/npy], but got {file}")


def fake_array2dict(fake_array, n_users, filter_num=4):
    """implicit.py:107-114: row r -> user n_users + r, columns with rating STRICTLY > filter_num."""
    fake_array = np.asarray(fake_array)
    assert len(fake_array.shape) == 2, "Expect a user-item 2D rating matrix"
    uids, iids = np.where(fake_array > filter_num)
    result = {}
    for u, i in zip((uids + n_users).tolist(), iids.tolist()):
        result.setdefault(u, []).append(i)
    return result


def flatten(data_dict):
    """read_data (implicit.py:221-241) as arrays: keys with a non-empty list (dict order),
    indptr, items (stored order)."""
    keys, lens, items = [], [], []
    for uid, iids in data_dict.items():
        if len(iids) != 0:
            keys.append(int(uid))
            lens.append(len(iids))
            items.extend(iids)
    indptr = np.zeros(len(keys) + 1, dtype=np.int64)
    if keys:
        np.cumsum(lens, out=indptr[1:])
    return np.asarray(keys, dtype=np.int64), indptr, np.asarray(items, dtype=np.int64)


def _sorted_distinct_csr(users, items, n_rows, n_cols):
    """Per-row ascending distinct columns (what `UserItemNet[u].nonzero()[1]` returns, implicit.py:339-343)."""
    if len(users) == 0:
        return np.zeros(n_rows + 1, dtype=np.int64), np.zeros(0, dtype=np.int64)
    key = np.unique(users.astype(np.int64) * np.int64(n_cols) + items.astype(np.int64))
    u, i = key // n_cols, key % n_cols
    indptr = np.zeros(n_rows + 1, dtype=np.int64)
    np.cumsum(np.bincount(u, minlength=n_rows), out=indptr[1:])
    return indptr, i


class _EpochJob:
    """One prefetched epoch.  Its generator-dependent part (sampler, then the draws of the shuffle) runs as soon as
    the previous job's generator-dependent part is finished -- it starts from that job's end state -- while the
    previous job may still be applying its swaps."""

    def __init__(self, slot, prev=None, key=None, pos=None):
        import threading
        self.slot, self.prev = slot, prev
        self.start_key, self.start_pos = key, pos          # known now, or once prev.rng_done fires
        self.end_key = self.end_pos = self.out = self.error = None
        self.rng_done, self.done = threading.Event(), threading.Event()


class _EpochPipe:
    """Host side of an epoch: draw (samples, perm) with the exact MT19937 replay into PINNED buffers and
    ship them to the device with one asynchronous copy each.

    Speculative prefetch: the sampler is a sequential state machine on numpy's global stream (seconds for
    50 M samples), so while the GPU trains epoch e background threads draw epochs e+1 and e+2, each from a
    COPY of the state the previous one ended with.  Only the stream-consuming work is chained (sampler, then
    the draws of the shuffle); applying the swaps needs no generator and overlaps the next epoch's sampler.
    At the next call the head of the queue is used only if np.random's state still equals its starting state
    (nobody else consumed the stream, the case inside normal_train's epoch loop, normal.py:95-109); then the
    global state is advanced to where that epoch ended.  Otherwise the queue is discarded and the epoch is drawn
    synchronously -- the stream seen by every consumer is identical to the reference's in both cases."""

    DEPTH = 2

    def __init__(self, data):
        from collections import deque
        import weakref
        # a weak reference: dataset <-> pipe would be a cycle, and a cycle is only freed by the garbage collector's next
        # pass -- the pinned epoch buffers of a dropped dataset (one per attack iteration) would then miss the pool and
        # the next dataset would page-lock 0.8 GB again (0.46 s at the synthetic size)
        self._data_ref = weakref.ref(data)
        self.bufs = [None] * (self.DEPTH + 1)
        self.queue = deque()
        self.last_slot = -1          # its buffers may still be the source of an asynchronous H2D copy
        self.calls = 0
        pf = data.config.get("prefetch")
        # default: on from ~10^5 interactions (ml1m-sized), where an epoch draw costs 0.05-0.2 s -- as much as the device
        # epoch of MF or LightGCN at that size
        self.prefetch = bool(pf) if pf is not None else data.traindataSize >= (1 << 17)
        # speculative epochs still being drawn at interpreter exit write into pinned buffers that the CUDA runtime
        # frees during its own teardown: wait for them first
        import atexit
        import weakref
        ref = weakref.ref(self)
        atexit.register(lambda: ref() is not None and ref()._flush())

    @property
    def data(self):
        d = self._data_ref()
        if d is None:
            raise ops.RecadError("the dataset of this epoch pipe was dropped")
        return d

    def _soa(self, cuda):
        """Large pairwise epochs take the 32-bit structure-of-arrays path: the host sampler emits (user, index of the
        positive, negative) as uint32, the positive ITEM is gathered on the device, rows and permutation stay int32."""
        d = self.data
        return cuda and d.config["sample"] == "pairwise" and ops.fits_soa_sampler(d.n_users, d.n_items, d.traindataSize)

    _POOL = []          # pinned 32-bit buffer sets of pipes that were garbage collected (page-locking 0.8 GB costs ~0.3 s)

    def __del__(self):
        try:
            for b in self.bufs:
                if b is not None and b[0] and len(_EpochPipe._POOL) < 4 and not self.queue:
                    _EpochPipe._POOL.append(b)
        except Exception:   # noqa: BLE001 -- interpreter teardown
            pass

    def _buffers(self, slot, cuda):
        n = self.data.traindataSize * (1 if self.data.config["sample"] == "pairwise" else 1 + self.data.config["negative_ratio"])
        soa = self._soa(cuda)
        if self.bufs[slot] is None or self.bufs[slot][-1].shape[0] < n or self.bufs[slot][0] != soa:
            if soa:
                for k, b in enumerate(_EpochPipe._POOL):        # a dataset derived by injection is a few hundred samples larger
                    if b[-1].shape[0] >= n:
                        self.bufs[slot] = _EpochPipe._POOL.pop(k)
                        torch.cuda.current_stream().synchronize()      # the previous owner's H2D copies out of these buffers
                        return self.bufs[slot]
                cap = max(n + (n >> 8), 1)                      # head-room so that the next injected dataset fits the same buffers
                host = [torch.empty(cap, dtype=torch.int32).pin_memory() for _ in range(4)]   # users, rel, negs, perm
                self.bufs[slot] = (True, *host, ops.host_empty(cap, np.uint32))
            else:
                s, p = torch.empty((max(n, 1), 3), dtype=torch.int64), torch.empty(max(n, 1), dtype=torch.int64)
                if cuda:
                    s, p = s.pin_memory(), p.pin_memory()
                self.bufs[slot] = (False, s, p, ops.host_empty(max(n, 1), np.uint32))
        return self.bufs[slot]

    def _draw_into(self, slot, cuda, key, pos, after_rng=None):
        """Sampler + shuffle of one epoch from an explicit generator state into the slot's host buffers."""
        d = self.data
        buf = self._buffers(slot, cuda)
        if buf[0]:
            _, u, r, g, p, jb = buf
            un, rn, gn = (t.numpy().view(np.uint32) for t in (u, r, g))
            m = ops.mt_pairwise_soa_raw(key, pos, d.n_users, d.n_items, d.traindataSize, *d._allpos, un, rn, gn, jb)
            if after_rng is not None:
                after_rng()
            ops.permutation_apply32(jb[:m], p.numpy())
            return ("soa", u[:m], r[:m], g[:m], p[:m])
        _, s, p, jb = buf
        S = d._draw_samples(key, pos, s.numpy())
        j = ops.mt_permutation_draw_raw(key, pos, len(S), jb)
        if after_rng is not None:
            after_rng()
        perm = ops.permutation_apply(j, p.numpy())
        return ("rows", s[:len(S)], p[:len(perm)])

    def _to_device(self, got, device):
        if got[0] == "soa":
            _, u, r, g, p = got
            if getattr(self, "raw_soa", False):       # sharded path: the host arrays themselves (each rank expands its own users)
                return u, r, g, p
            ud, rd, gd, pd = (t.to(device, non_blocking=True) for t in (u, r, g, p))
            rows = torch.empty((int(u.shape[0]), 3), dtype=torch.int32, device=device)
            ops.samples_expand(*self.data.allpos_device(device), ud, rd, gd, rows)
            return rows, pd
        _, s, p = got
        if device.type == "cuda":
            return s.to(device, non_blocking=True), p.to(device, non_blocking=True)
        return s.clone(), p.clone()           # host "device" (CPU-only tests): detach from the reusable buffers

    def _free_slot(self):
        used = {j.slot for j in self.queue} | {self.last_slot}
        return next(k for k in range(self.DEPTH + 1) if k not in used)

    def _run(self, job, cuda):
        try:
            if job.prev is not None:
                job.prev.rng_done.wait()
                if job.prev.error is not None:
                    raise RuntimeError("the previous prefetched epoch failed")
                job.start_key, job.start_pos = job.prev.end_key.copy(), int(job.prev.end_pos)
                job.prev = None
            key, pos = job.start_key.copy(), [int(job.start_pos)]

            def rng_done():
                job.end_key, job.end_pos = key, int(pos[0])
                job.rng_done.set()                              # the next epoch's sampler may start now
            job.out = self._draw_into(job.slot, cuda, key, pos, after_rng=rng_done)
        except BaseException as e:   # noqa: BLE001 -- reported by falling back to the synchronous draw
            job.error = e
        finally:
            job.rng_done.set()
            job.done.set()

    def _spawn(self, cuda, prev=None, key=None, pos=None):
        import threading
        job = _EpochJob(self._free_slot(), prev, key, pos)
        self.queue.append(job)
        threading.Thread(target=self._run, args=(job, cuda), daemon=True).start()

    def _flush(self):
        for job in self.queue:
            job.done.wait()
        self.queue.clear()

    def next(self, device):
        cuda = device.type == "cuda"
        st = np.random.get_state()
        if st[0] != "MT19937":
            raise ops.RecadError("np.random global state is not MT19937")
        got = None
        if self.queue:
            head = self.queue[0]
            head.rng_done.wait()
            if head.error is None and head.start_pos == int(st[2]) and np.array_equal(head.start_key, st[1]):
                head.done.wait()
                if head.error is None:
                    self.queue.popleft()
                    got, key, pos, self.last_slot = head.out, head.end_key, [head.end_pos], head.slot
            if got is None:
                self._flush()
        if got is None:
            key, pos = np.ascontiguousarray(st[1], dtype=np.uint32).copy(), [int(st[2])]
            slot = self._free_slot()
            got, self.last_slot = self._draw_into(slot, cuda, key, pos), slot
        np.random.set_state((st[0], key, int(pos[0]), st[3], st[4]))
        on_dev = self._to_device(got, device)
        self.calls += 1
        # speculate only once the caller has come back for a second epoch: a dataset that lives for ONE epoch (the
        # attacked copy of an attack iteration) would otherwise leave two useless epochs running in the background,
        # and the next dataset's sampler queues up behind them
        if self.prefetch and self.calls >= 2:
            while len(self.queue) < self.DEPTH:
                if self.queue:
                    self._spawn(cuda, prev=self.queue[-1])
                else:
                    self._spawn(cuda, key=key.copy(), pos=int(pos[0]))
        return on_dev


class ImplicitData:
    def __init__(self, **config):
        self.config = config
        self.logger = get_logger(f"{__name__}:{self.dataset_name}", level=config["logging_level"])
        self._mode = "train"
        self._load_data()
        self._init_data()

    # ---------------------------------------------------------------- factory / reset
    @classmethod
    def from_config(cls, name, **user_config):
        defaults = implicit_defaults(name)
        cfg = merge_config(defaults, {k: v for k, v in user_config.items() if k != "download"}, logger=None)
        for k in user_config:
            if k not in defaults and k != "download":
                get_logger(__name__).debug(f"Unexpected key [{k}] for {cls}")
        inst = object.__new__(cls)
        inst._dataset_name = name
        inst._init_config = cfg
        inst.__init__(**cfg)
        return inst

    @property
    def dataset_name(self):
        return getattr(self, "_dataset_name", type(self).__name__)

    def reset(self, **kwargs):
        """base.py:108-118: same config with some keys replaced -> a NEW dataset."""
        if not hasattr(self, "_init_config"):
            raise ValueError("reset method is only for datasets instantiated from_config")
        config = copy(self._init_config)
        for k, v in kwargs.items():
            if k not in config:
                raise ValueError(f"reset arg {k} should be in {list(config)}")
            config[k] = v
        return type(self).from_config(self.dataset_name, **config)

    # ---------------------------------------------------------------- loading
    def _load_data(self):
        """implicit.py:140-164 (dict passed in > .npy cache > csv)."""
        for attr, path in (("train_dict", "path_train"), ("valid_dict", "path_valid"), ("test_dict", "path_test")):
            if self.config[attr] is not None:
                setattr(self, attr, self.config[attr])
                continue
            cache = os.path.join(self.config["cache_dir"], f"{self.dataset_name}_implicit_{attr}.npy")
            if os.path.exists(cache) and self.config["if_cache"]:
                self.logger.info(f"loading cached {attr}")
                setattr(self, attr, np.load(cache, allow_pickle=True).item())
            else:
                setattr(self, attr, convert2dict(self.config[path], self.config["rating_filter"]))
                if self.config["if_cache"]:
                    os.makedirs(self.config["cache_dir"], exist_ok=True)
                    np.save(cache, getattr(self, attr))

    def _init_data(self):
        """implicit.py:166-219, vectorised; the graph goes to the device (ops.Graph)."""
        if self.config["A_split"]:
            raise ValueError("A_split is not supported (the reference's LightGCN rejects it too, lightgcn.py:38-39)")
        self._tr = flatten(self.train_dict)
        self._va = flatten(self.valid_dict)
        self._te = flatten(self.test_dict)
        max_u, max_i = 0, 0            # running max starts at 0 (implicit.py:167-168)
        for keys, _, items in (self._tr, self._va, self._te):
            if len(keys):
                max_u, max_i = max(max_u, int(keys.max())), max(max_i, int(items.max()))
        self.n_users, self.n_items = max_u + 1, max_i + 1
        self.traindataSize = int(self._tr[1][-1])
        self.validDataSize = int(self._va[1][-1])
        self.testDataSize = int(self._te[1][-1])
        self.trainUniqueUsers = self._tr[0]
        # flat (user, item) of each split
        self._flat = {}
        for nm, (keys, indptr, items) in (("train", self._tr), ("valid", self._va), ("test", self._te)):
            self._flat[nm] = (np.repeat(keys, np.diff(indptr)), items)
        # which interactions feed UserItemNet / allPos / the graph (SURVEY.md 0.1)
        which = self.config.get("graph_edges", "reference")
        if which not in ("reference", "train"):
            raise ValueError("graph_edges must be 'reference' or 'train'")
        self.trainUser, self.trainItem = self._flat["test" if which == "reference" else "train"]
        ptr, idx = _sorted_distinct_csr(self.trainUser, self.trainItem, self.n_users, self.n_items)
        self._allpos = (ptr, idx.astype(np.int32))
        self._train_csr = None
        self.Graph = None
        if self.config["need_graph"]:
            self.getSparseGraph()

    # ---------------------------------------------------------------- graph (implicit.py:243-298)
    def getSparseGraph(self):
        if self.Graph is None:
            dev = torch.device(self.config["device"])
            if dev.type != "cuda":
                raise ops.RecadError("recad_b200 builds the graph on a CUDA device; config['device'] is " + str(dev))
            # the reference's on-disk cache (implicit.py:246-256, 279-289): same file name, same scipy .npz of the
            # normalised CSR, so either implementation reads what the other wrote
            cache = os.path.join(self.config["cache_dir"], f"adj_mat_{self.dataset_name}_{self.n_users}_{self.n_items}.npz")
            if self.config.get("if_cache") and os.path.exists(cache):
                import scipy.sparse as sp
                m = sp.load_npz(cache).tocsr()
                m.sort_indices()
                N = self.n_users + self.n_items
                if m.shape != (N, N):
                    raise ValueError(f"{cache}: cached adjacency is {m.shape}, the dataset needs {(N, N)}")
                self.logger.info(f"successfully loaded adj_mat from {cache}, this could cause the inconsistency of the dataset")
                self.Graph = ops.Graph.from_csr(torch.from_numpy(m.indptr.astype(np.int64)).to(dev),
                                                torch.from_numpy(m.indices.astype(np.int32)).to(dev),
                                                torch.from_numpy(m.data.astype(np.float32)).to(dev), n_cols=N, split=self.n_users)
                return self.Graph
            u = torch.from_numpy(self.trainUser).to(dev)
            i = torch.from_numpy(self.trainItem).to(dev)
            self.Graph = ops.Graph.from_edges(u, i, self.n_users, self.n_items)
            if self.config.get("if_cache"):
                import scipy.sparse as sp
                os.makedirs(self.config["cache_dir"], exist_ok=True)
                ptr, col, val = self.Graph.to_numpy()
                N = self.n_users + self.n_items
                sp.save_npz(cache, sp.csr_matrix((val, col, ptr), shape=(N, N)))
        return self.Graph

    @property
    def allPos(self):
        """List of per-user positive arrays (implicit.py:300-302); built on demand."""
        ptr, idx = self._allpos
        return [idx[ptr[u]:ptr[u + 1]] for u in range(self.n_users)]

    def getUserPosItems(self, users):
        ptr, idx = self._allpos
        return [idx[ptr[u]:ptr[u + 1]] for u in users]

    def allpos_device(self, device):
        """allPos (implicit.py:300-302) as a CSR on the device: (rowptr int64 [n_users + 1], col int32)."""
        if getattr(self, "_allpos_dev", None) is None or self._allpos_dev[0].device != device:
            self._allpos_dev = tuple(torch.from_numpy(np.ascontiguousarray(a)).to(device) for a in self._allpos)
        return self._allpos_dev

    def train_csr(self, device=None):
        """Sorted distinct train items per user id (mask of normal_evaluate, normal.py:133-143):
        (rowptr int64 [n_users + 1], col int32) on `device`."""
        if self._train_csr is None:
            ptr, idx = _sorted_distinct_csr(*self._flat["train"], self.n_users, self.n_items)
            self._train_csr = (ptr, idx.astype(np.int32))
        if device is None:
            return self._train_csr
        return tuple(torch.from_numpy(a).to(device) for a in self._train_csr)

    def ground_truth_csr(self, split="test", device=None):
        ptr, idx = _sorted_distinct_csr(*self._flat[split], self.n_users, self.n_items)
        out = (ptr, idx.astype(np.int32))
        return out if device is None else tuple(torch.from_numpy(a).to(device) for a in out)

    # ---------------------------------------------------------------- describe
    def batch_describe(self):
        c = self.config
        if c["sample"] == "pairwise" and self.mode() == "train":
            return {k: (torch.int64, f"batch[0~{c['pairwise_batch_size']}]") for k in ("users", "positive_items", "negative_items")}
        if c["sample"] == "pointwise" and self.mode() == "train":
            return {k: (torch.int64, f"batch[0~{c['pointwise_batch_size']}]") for k in ("users", "items", "labels")}
        if self.mode() in ("validate", "test"):
            return {"users": (torch.int64, f"batch[0~{c['test_batch_size']}]"), "positive_items": (list, "batch"),
                    "ground_truth": (list, "batch")}

    def info_describe(self):
        infos = {
            "n_users": self.n_users, "n_items": self.n_items,
            "train_interactions": self.traindataSize, "valid_interactions": self.validDataSize,
            "test_interactions": self.testDataSize,
            "train_dict": self.train_dict, "valid_dict": self.valid_dict, "test_dict": self.test_dict,
            "batch_describe": self.batch_describe(),
        }
        if self.config["need_graph"]:
            infos["graph"] = self.Graph
        return infos

    def print_help(self, **kwargs):
        info = self.info_describe()
        info["dataset_name"] = self.dataset_name
        pprint({k: (v if len(str(v)) < 30 else f"{type(v)}") for k, v in info.items() if k != "batch_describe"})

    def mode(self):
        return self._mode

    def switch_mode(self, mode):
        assert mode in ["train", "test", "validate"]
        self._mode = mode

    # ---------------------------------------------------------------- sampling (implicit.py:18-91, 416-476)
    def epoch_samples(self, device=None):
        """One epoch of training rows for the C epoch drivers: (samples, perm) on the device.
        samples int64 [n, 3] = (user, pos, neg) or (user, item, label) in SAMPLER order; perm int64 [n] =
        the epoch shuffle (implicit.py:18-35), applied by the kernels as an index indirection.
        Consumes the global np.random stream exactly as `generate_batch` of the reference does (sampler,
        then shuffle).  With config['prefetch'] the NEXT epoch is drawn on a background thread while the
        GPU trains (see _EpochPipe)."""
        if self.mode() != "train":
            raise NotImplementedError("epoch_samples is for train mode")
        if getattr(self, "_pipe", None) is None:
            self._pipe = _EpochPipe(self)
        return self._pipe.next(torch.device(device or self.config["device"]))

    def _draw_samples(self, key, pos, out=None):
        """The sampler from an EXPLICIT MT19937 state (key, pos are advanced in place)."""
        if self.config["sample"] == "pairwise":
            return ops.mt_pairwise_raw(key, pos, self.n_users, self.n_items, self.traindataSize, *self._allpos, out=out)
        if self.config["sample"] == "pointwise":
            return ops.mt_pointwise_raw(key, pos, *self._tr, self.n_items, self.config["negative_ratio"], out=out)
        raise NotImplementedError("Not implemented yet")

    def generate_batch(self, **config):
        c = self.config
        if self.mode() == "train":
            samples, perm = self.epoch_samples()
            S = samples[perm.long()].long()                # compatibility path only: materialise the shuffle
            if c["sample"] == "pairwise":
                names, bs = ("users", "positive_items", "negative_items"), c["pairwise_batch_size"]
            else:
                names, bs = ("users", "items", "labels"), c["pointwise_batch_size"]
            for s in range(0, len(S), bs):                 # minibatch (implicit.py:38-47)
                yield {names[0]: S[s:s + bs, 0], names[1]: S[s:s + bs, 1], names[2]: S[s:s + bs, 2]}
        elif self.mode() in ("validate", "test"):
            test_dict = self.valid_dict if self.mode() == "validate" else self.test_dict
            users = list(test_dict.keys())
            bs = c["test_batch_size"]
            for s in range(0, len(users), bs):
                batch_users = users[s:s + bs]
                yield {
                    "users": torch.tensor(batch_users, dtype=torch.int64).to(c["device"]),
                    "positive_items": self.getUserPosItems(batch_users),
                    "ground_truth": [test_dict[u] for u in batch_users],
                }

    # ---------------------------------------------------------------- injection (implicit.py:482-525)
    def inject_data(self, data_mode, data, **kwargs):
        if data_mode != "explicit":
            raise NotImplementedError(f"Injection not supported in {data_mode} mode")
        new_train_dict = copy(self.train_dict)
        inject_dict = fake_array2dict(data, self.n_users, filter_num=kwargs["filter_num"])
        for k, v in inject_dict.items():
            assert k not in new_train_dict, f"Injection to a exist user {k} is not allowed"
            new_train_dict[k] = v
        return self._derive_injected(new_train_dict, inject_dict)

    def _derive_injected(self, new_train_dict, inject_dict):
        """What `reset(train_dict=..., if_cache=False)` produces (implicit.py:493), but the device graph
        is EXTENDED in place (rows appended, no re-sort, valid/test not re-read)."""
        config = copy(self._init_config)
        config.update(train_dict=new_train_dict, valid_dict=self.valid_dict, test_dict=self.test_dict,
                      if_cache=False, need_graph=False)
        new = type(self).from_config(self.dataset_name, **config)
        new.config["need_graph"] = new._init_config["need_graph"] = self.config["need_graph"]
        if self.config["need_graph"]:
            F = new.n_users - self.n_users
            if self.config.get("graph_edges", "reference") == "train" and new.n_items == self.n_items:
                rows = [sorted(set(inject_dict.get(self.n_users + r, []))) for r in range(F)]
            elif new.n_items == self.n_items:
                rows = [[] for _ in range(F)]   # reference quirk: fake users add rows but NO edges (SURVEY.md 0.1)
            else:
                rows = None                     # item universe grew: rebuild from scratch
            if rows is not None and self.Graph is not None and self.Graph.mult is not None:   # a graph read from the cache carries no multiplicities
                fake_rowptr = torch.tensor(np.concatenate([[0], np.cumsum([len(r) for r in rows])]), dtype=torch.int64)
                fake_items = torch.tensor([i for r in rows for i in r], dtype=torch.int32)
                new.Graph = self.Graph.append_users(self.n_users, self.n_items, fake_rowptr, fake_items)
            else:
                new.getSparseGraph()
        return new

    def delete_data(self, data_mode, user_id, data, **kwargs):
        """implicit.py:496-513 (defense workflow): inject, then drop the flagged users; full rebuild."""
        if data_mode != "explicit":
            raise NotImplementedError(f"Injection not supported in {data_mode} mode")
        new_train_dict = copy(self.train_dict)
        inject_dict = fake_array2dict(data, self.n_users, filter_num=kwargs["filter_num"])
        for k, v in inject_dict.items():
            assert k not in new_train_dict, f"Injection to a exist user {k} is not allowed"
            new_train_dict[k] = v
        for key in list(new_train_dict.keys()):
            if key in user_id:
                del new_train_dict[key]
        return self.reset(train_dict=new_train_dict, if_cache=False)

    def partial_sample(self, **kwargs):
        assert "user_ratio" in kwargs, "Expect to have [user_ratio]"
        user_ratio = kwargs["user_ratio"]
        if abs(user_ratio - 1) < 1e-9:
            return self
        users = list(self.train_dict)
        random.shuffle(users)
        left_users = users[: int(len(users) * user_ratio)]
        return self.reset(train_dict={u: self.train_dict[u] for u in left_users})


class ArrayImplicitData:
    """Array-backed dataset for graphs too large for Python dicts (the synthetic 1M x 200k x 50M
    configuration): the same sampler / epoch pipe / graph code as ImplicitData, but everything is derived
    from the DEVICE graph -- the user rows of the symmetric CSR already are every user's sorted distinct
    positives (allPos / the evaluation mask), so no host-side sort of the interactions is ever done.
    `train_dict` is not materialised; the evaluator uses `train_csr()`.

    train: (users, items) CUDA int64 tensors of distinct pairs, or None when `graph` is given.
    test:  optional (users, items) host arrays of held-out pairs (ground truth for Recall/NDCG)."""

    def __init__(self, name, n_users, n_items, train, device, test=None, sample="pairwise", batch_size=1024,
                 negative_ratio=4, need_graph=True, graph=None, prefetch=None, allpos_host=None):
        self._dataset_name = name
        self.n_users, self.n_items = int(n_users), int(n_items)
        dev = torch.device(device)
        self.config = {"device": dev, "sample": sample, "pairwise_batch_size": batch_size,
                       "pointwise_batch_size": batch_size, "negative_ratio": negative_ratio, "need_graph": need_graph,
                       "graph_edges": "train"}
        if prefetch is not None:
            self.config["prefetch"] = prefetch
        if graph is None:
            tu, ti = (torch.as_tensor(a).to(dev).long() for a in train)
            graph = ops.Graph.from_edges(tu, ti, n_users, n_items)
        self.Graph = graph
        U = self.n_users
        rowptr_u = graph.rowptr[:U + 1].contiguous()
        n_train = int(rowptr_u[-1])
        col_u = (graph.colidx[:n_train] - U).contiguous()                 # int32 item ids, ascending per user
        self._train_csr_dev = (rowptr_u, col_u)
        # host copy (huge pages) of the positives for the C++ sampler; an injected dataset gets it from its parent
        self._allpos = allpos_host if allpos_host is not None else (ops.to_host(rowptr_u), ops.to_host(col_u))
        self._train_csr = self._allpos
        self.traindataSize = n_train
        # pointwise sampler: dict order = users ascending, each list ascending
        lens = np.diff(self._allpos[0])
        keys = np.flatnonzero(lens > 0).astype(np.int64)
        self._tr = (keys, np.concatenate([[0], np.cumsum(lens[keys])]).astype(np.int64), self._allpos[1].astype(np.int64)) \
            if sample == "pointwise" else None
        self._test = test
        self._gt = {}
        self._mode = "train"

    dataset_name = ImplicitData.dataset_name
    mode = ImplicitData.mode
    switch_mode = ImplicitData.switch_mode
    epoch_samples = ImplicitData.epoch_samples
    _draw_samples = ImplicitData._draw_samples
    generate_batch = ImplicitData.generate_batch

    def allpos_device(self, device):
        return tuple(t.to(device) for t in self._train_csr_dev)

    def train_csr(self, device=None):
        if device is None:
            return self._train_csr
        return tuple(t.to(device) for t in self._train_csr_dev)

    def ground_truth_csr(self, split="test", device=None):
        if split not in self._gt:
            if split != "test" or self._test is None:
                raise ValueError(f"ArrayImplicitData has no '{split}' ground truth")
            ptr, idx = _sorted_distinct_csr(np.asarray(self._test[0], np.int64), np.asarray(self._test[1], np.int64),
                                            self.n_users, self.n_items)
            self._gt[split] = (ptr, idx.astype(np.int32))
        out = self._gt[split]
        return out if device is None else tuple(torch.from_numpy(a).to(device) for a in out)

    # ---------------------------------------------------------------- injection (implicit.py:482-494)
    @staticmethod
    def fake_rows(data, filter_num=4):
        """fake_array2dict (implicit.py:107-114) as CSR: row r keeps the columns rated STRICTLY above
        filter_num; n_users = max uid + 1 (implicit.py:194), so trailing rows with nothing left do not
        become users.  -> (rowptr int64 [F + 1], items int32 ascending per row)"""
        data = np.asarray(data)
        assert len(data.shape) == 2, "Expect a user-item 2D rating matrix"
        r, c = np.nonzero(data > filter_num)
        F = int(r.max()) + 1 if r.size else 0
        rowptr = np.zeros(F + 1, dtype=np.int64)
        np.cumsum(np.bincount(r, minlength=F), out=rowptr[1:])
        return rowptr, c.astype(np.int32)

    def inject_data(self, data_mode, data, **kwargs):
        """New, independent dataset with the fake users appended.  The device graph is EXTENDED (rows
        appended, touched items re-normalised, no re-sort); the reference rebuilds everything from dicts
        (implicit.py:493, base.py:108-118)."""
        if data_mode != "explicit":
            raise NotImplementedError(f"Injection not supported in {data_mode} mode")
        rowptr, items = self.fake_rows(data, kwargs["filter_num"])
        assert data.shape[1] <= self.n_items, "fake profiles rate items outside the item universe"
        F = len(rowptr) - 1
        graph = self.Graph.append_users(self.n_users, self.n_items, torch.from_numpy(rowptr), torch.from_numpy(items))
        c = self.config
        batch = c["pairwise_batch_size"] if c["sample"] == "pairwise" else c["pointwise_batch_size"]
        # the positives of the attacked dataset = the parent's with F rows appended: a host concatenation instead of a
        # device -> host copy, and the sampler's per-user filter blocks of the genuine users are reused (ops.pairwise_filter)
        old_ptr, old_col = self._allpos
        new_ptr = ops.host_empty(len(old_ptr) + F, np.int64)
        new_ptr[:len(old_ptr)] = old_ptr
        new_ptr[len(old_ptr):] = old_ptr[-1] + rowptr[1:]
        new_col = ops.host_empty(len(old_col) + len(items), np.int32)
        new_col[:len(old_col)] = old_col
        new_col[len(old_col):] = items
        ops.filter_parent_hint(new_ptr, new_col, old_ptr, old_col, self.n_users)
        return ArrayImplicitData(self._dataset_name, self.n_users + F, self.n_items, None, c["device"], test=self._test,
                                 sample=c["sample"], batch_size=batch, negative_ratio=c["negative_ratio"],
                                 need_graph=c["need_graph"], graph=graph, prefetch=c.get("prefetch"), allpos_host=(new_ptr, new_col))

    def info_describe(self):
        infos = {"n_users": self.n_users, "n_items": self.n_items, "train_interactions": self.traindataSize,
                 "train_dict": None}
        if self.config["need_graph"]:
            infos["graph"] = self.Graph
        return infos


from .explicit import ExplicitData  # noqa: E402

factories = {"implicit": ImplicitData, "explicit": ExplicitData}    # recad/dataset/__init__.py:13


def from_config(scope, *args, **kwargs):
    return factories[scope].from_config(*args, **kwargs)
