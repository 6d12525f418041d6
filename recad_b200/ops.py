"""Tensor-level wrappers over the C ABI (include/recad_b200.h).

PyTorch is used here for device memory and the current CUDA stream only; every
computation is a kernel of librecad_b200.so.  All functions raise RecadError on
failure -- there is no fallback path.
"""
import ctypes as C
import os

import numpy as np
import torch
from torch.autograd.function import once_differentiable

from . import _lib
from ._lib import RecadError, check

SEG_LEN = None  # SpMM plan: max stored entries one warp walks (multiple of 32); None = by size (auto_seg_len)


def auto_seg_len(nnz):
    """Measured on B200 (profiles/spmm_variant_sweep_r01.jsonl, spmm_sweep_ml1m_r01.jsonl): long segments
    amortise the per-segment prologue when there are far more segments than resident warps (synthetic,
    100 M entries: 256 is fastest); an L2-resident graph with ~1 segment per warp slot is latency-bound and
    wants more, shorter chains (ml1m-shaped, 0.94 M entries: 64 is 25 % faster than 256)."""
    return 64 if nnz <= 8_000_000 else 256


def _ptr(t):
    if t is None:
        return None
    assert t.is_contiguous(), "recad_b200 ops need contiguous tensors"
    return C.c_void_p(t.data_ptr())


def _stream(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _need_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RecadError("recad_b200 runs on CUDA tensors only (no CPU path); got a CPU tensor")


def device_info():
    sm, a, b = C.c_int(), C.c_int(), C.c_int()
    check(_lib.lib().recad_device_info(C.byref(sm), C.byref(a), C.byref(b)), "recad_device_info")
    return sm.value, a.value, b.value


# --------------------------------------------------------------------------- #
# graph
# --------------------------------------------------------------------------- #
def d_inv_from_degree(degree):
    """The reference's own host expression (recad/dataset/implicit.py:269-272):
    float32 rowsum as an (N, 1) array, ``np.power(rowsum + 1e-14, -0.5)``.  It is
    evaluated on the host with numpy on purpose: numpy's float32 pow is not
    correctly rounded and no device expression reproduces its bits."""
    rowsum = np.asarray(degree).astype(np.float32).reshape(-1, 1)
    d_inv = np.power(rowsum + 1e-14, -0.5).flatten()
    d_inv[np.isinf(d_inv)] = 0.0
    return d_inv


def auto_col_blocks(n_cols, row_bytes=256):
    """Column blocks for rows that gather from a table of n_cols rows: one block while the table fits the 126 MB L2
    next to the streamed matrix, else ~80 MB blocks (measured on B200: 2-4 blocks of the 256 MB user table are equally
    fast, profiles/spmm2_sweep_r02.jsonl)."""
    nbytes = int(n_cols) * row_bytes
    return 1 if nbytes <= 100e6 else max(2, int(round(nbytes / 80e6)))


class PackedPlan:
    """Work list of the SpMM (csrc/spmm.cu): one 16-byte entry per SEGMENT {lo (64 bit), row, (slot + 1) << 11 | count}.
    `groups` = [(row_lo, row_hi, col_lo, col_hi, n_blocks)] partitions the rows; the rows of a group gather columns in
    [col_lo, col_hi) and are cut at n_blocks equal column blocks, their segments ordered block by block, so that the
    gathered slice of X (an L2-sized block of the user table) stays cache resident while it is in use; inside a
    (group, block) the segments go longest first (no straggler warps at the tail of the persistent kernel).  A row
    with more than one segment gets consecutive partial-sum slots in (row, first entry) order; its last-arriving warp
    adds them in that order (deterministic).
    Plain index arithmetic on torch tensors (runs wherever the row pointer lives): executed once per graph, the hot
    path only reads its output."""

    MAX_SEG = 1024

    def __init__(self, meta, row_mseg, n_mrow, n_slot, group_segs):
        self.meta, self.row_mseg, self.n_mrow, self.n_slot, self.group_segs = meta, row_mseg, int(n_mrow), int(n_slot), group_segs
        self.n_seg = int(meta.shape[0])

    @classmethod
    def build(cls, rowptr, colidx, n_rows, seg_len, groups=None):
        if not (0 < seg_len <= cls.MAX_SEG):
            raise RecadError(f"PackedPlan: seg_len must be in (0, {cls.MAX_SEG}]")
        dev = rowptr.device
        i64 = dict(dtype=torch.int64, device=dev)
        rowptr = rowptr.long()
        if groups is None:
            groups = [(0, n_rows, 0, 1 << 31, 1)]
        assert groups[0][0] == 0 and groups[-1][1] == n_rows and all(a[1] == b[0] for a, b in zip(groups, groups[1:]))
        # pieces = (row, lo, hi, order key): one piece per (row, column block)
        p_row, p_lo, p_hi, p_grp = [], [], [], []
        gkey = 0
        for (r0, r1, c0, c1, nb) in groups:
            rows = torch.arange(r0, r1, **i64)
            if nb <= 1 or r1 == r0:
                p_row.append(rows); p_lo.append(rowptr[r0:r1]); p_hi.append(rowptr[r0 + 1:r1 + 1])
                p_grp.append(torch.full((r1 - r0,), gkey, **i64))
                gkey += 1
                continue
            e0, e1 = int(rowptr[r0]), int(rowptr[r1])
            erow = torch.repeat_interleave(rows, rowptr[r0 + 1:r1 + 1] - rowptr[r0:r1])
            key = (erow << 32) | colidx[e0:e1].long()                       # ascending: CSR is (row, col) sorted
            bounds = torch.tensor([c0 + (b * (c1 - c0)) // nb for b in range(1, nb)], **i64)
            q = (rows[:, None] << 32) | bounds[None, :]
            cut = torch.searchsorted(key, q.reshape(-1)).reshape(-1, nb - 1) + e0
            edges = torch.cat([rowptr[r0:r1, None], cut, rowptr[r0 + 1:r1 + 1, None]], 1)   # [rows, nb + 1]
            lo_b, hi_b = edges[:, :-1], edges[:, 1:]
            keep = hi_b > lo_b
            keep[:, 0] |= ~keep.any(1)                                       # an empty row is still written once
            grp_b = (gkey + torch.arange(nb, **i64))[None, :].expand_as(lo_b)
            p_row.append(rows[:, None].expand_as(lo_b)[keep]); p_lo.append(lo_b[keep]); p_hi.append(hi_b[keep])
            p_grp.append(grp_b[keep])
            gkey += nb
        p_row, p_lo, p_hi, p_grp = (torch.cat(x) for x in (p_row, p_lo, p_hi, p_grp))
        # pieces -> segments of at most seg_len entries
        nch = torch.clamp((p_hi - p_lo + seg_len - 1) // seg_len, min=1)
        first = torch.cumsum(nch, 0) - nch
        n_seg = int(nch.sum())
        piece = torch.repeat_interleave(torch.arange(p_row.numel(), **i64), nch)
        k = torch.arange(n_seg, **i64) - first[piece]
        s_row, s_grp = p_row[piece], p_grp[piece]
        s_lo = p_lo[piece] + k * seg_len
        s_cnt = torch.minimum(p_hi[piece] - s_lo, torch.full_like(s_lo, seg_len))
        # partial-sum slots of the rows with more than one segment, in (row, lo) order
        per_row = torch.bincount(s_row, minlength=n_rows)
        multi = per_row > 1
        slots_of = torch.where(multi, per_row, torch.zeros_like(per_row))
        slot0 = torch.cumsum(slots_of, 0) - slots_of
        n_slot, n_mrow = int(slots_of.sum()), int(multi.sum())
        if n_slot + 1 >= (1 << 21):
            raise RecadError(f"PackedPlan: {n_slot} partial slots exceed the packed field; use a longer seg_len")
        by_row = torch.argsort(s_row * (1 << 40) + s_lo)                    # lo < 2^40
        row_first = torch.cumsum(per_row, 0) - per_row
        rank = torch.empty(n_seg, **i64)
        rank[by_row] = torch.arange(n_seg, **i64) - row_first[s_row[by_row]]
        s_slot = torch.where(multi[s_row], slot0[s_row] + rank, torch.full_like(rank, -1))
        # execution order: group by group, block by block, longest first
        ex = torch.argsort(s_grp * (1 << 44) + (cls.MAX_SEG - s_cnt) * (1 << 32) + s_row, stable=True)
        meta = torch.stack([s_lo & 0xffffffff, s_lo >> 32, s_row, ((s_slot + 1) << 11) | s_cnt], 1)[ex]
        meta = torch.where(meta >= (1 << 31), meta - (1 << 32), meta).to(torch.int32).contiguous()
        row_mseg = torch.stack([slot0, per_row], 1).to(torch.int32).contiguous()
        # segment ranges of the caller's groups (profiling tools time them separately)
        g_of_key, gk = [], 0
        for gi, (r0, r1, c0, c1, nb) in enumerate(groups):
            n_keys = 1 if (nb <= 1 or r1 == r0) else nb
            g_of_key += [gi] * n_keys
            gk += n_keys
        cnt_key = torch.bincount(s_grp, minlength=gk).tolist()
        group_segs, at = [], 0
        for gi in range(len(groups)):
            n = sum(c for c, g in zip(cnt_key, g_of_key) if g == gi)
            group_segs.append((at, at + n))
            at += n
        return cls(meta, row_mseg, n_mrow, n_slot, group_segs)


class Graph:
    """Device-resident CSR of a (normalised) adjacency + its SpMM work plan."""

    def __init__(self, n_rows, n_cols, rowptr, colidx, vals, mult=None, degree=None, seg_len=SEG_LEN, split=None):
        """split = n_users for the symmetric bipartite adjacency (rows < split gather item rows of X, rows >= split
        gather user rows): the two halves become separate plan groups, each column-blocked when its gathered table
        exceeds L2 (PackedPlan)."""
        self.n_rows, self.n_cols = int(n_rows), int(n_cols)
        self.rowptr, self.colidx, self.vals, self.mult, self.degree = rowptr, colidx, vals, mult, degree
        self.nnz = int(colidx.numel())
        self.device = rowptr.device
        self.seg_len = seg_len or auto_seg_len(self.nnz)
        self.split = None if split is None else int(split)
        self._partials = {}
        self._structs = {}
        self._plan()

    # -- construction ------------------------------------------------------ #
    @classmethod
    def from_edges(cls, users, items, n_users, n_items, seg_len=SEG_LEN, degree_hook=None):
        """Symmetric-normalised bipartite adjacency (implicit.py:243-298) from an
        edge list on the device.  users / items: int64 CUDA tensors.
        degree_hook(degree int32 [N]) may complete the degrees in place before normalisation (the sharded
        path all-reduces the item block: a rank's rows hold only its own users' edges)."""
        _need_cuda(users, items)
        L = _lib.lib()
        dev = users.device
        users, items = users.contiguous().long(), items.contiguous().long()
        E, N = int(users.numel()), int(n_users) + int(n_items)
        with torch.cuda.device(dev):
            rowptr = torch.empty(N + 1, dtype=torch.int64, device=dev)
            colidx = torch.empty(max(2 * E, 1), dtype=torch.int32, device=dev)
            mult = torch.empty(max(2 * E, 1), dtype=torch.float32, device=dev)
            degree = torch.empty(N, dtype=torch.int32, device=dev)
            nbytes = L.recad_csr_build_scratch_bytes(E, n_users, n_items)
            scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            nnz = C.c_int64()
            check(L.recad_csr_build_structure(_ptr(users), _ptr(items), E, n_users, n_items, _ptr(rowptr), _ptr(colidx),
                                              _ptr(mult), _ptr(degree), C.byref(nnz), _ptr(scratch), nbytes, _stream(dev)),
                  "recad_csr_build_structure")
            del scratch
            colidx, mult = colidx[:nnz.value].clone(), mult[:nnz.value].clone()
            if degree_hook is not None:
                degree_hook(degree)
            vals = cls._normalize(rowptr, colidx, mult, degree, N)
        return cls(N, N, rowptr, colidx, vals, mult, degree, seg_len, split=n_users)

    @staticmethod
    def _normalize(rowptr, colidx, mult, degree, N):
        dev = rowptr.device
        d_inv = torch.from_numpy(d_inv_from_degree(degree.cpu().numpy())).to(dev)
        vals = torch.empty(colidx.numel(), dtype=torch.float32, device=dev)
        check(_lib.lib().recad_csr_normalize(_ptr(rowptr), _ptr(colidx), _ptr(mult), _ptr(d_inv), N, _ptr(vals), _stream(dev)),
              "recad_csr_normalize")
        return vals

    def append_users(self, n_users, n_items, fake_rowptr, fake_items, degree_hook=None):
        """In-place injection (implicit.py:482-494): returns the graph over
        n_users + F users with the fake rows appended; no sort, no Python dict.
        degree_hook: as in from_edges (a shard completes its item degrees before normalisation)."""
        L = _lib.lib()
        dev = self.device
        F = int(fake_rowptr.numel()) - 1
        nf = int(fake_items.numel())
        Nn = n_users + F + n_items
        with torch.cuda.device(dev):
            fake_rowptr = fake_rowptr.to(dev, torch.int64).contiguous()
            fake_items = fake_items.to(dev, torch.int32).contiguous()
            rowptr = torch.empty(Nn + 1, dtype=torch.int64, device=dev)
            colidx = torch.empty(max(self.nnz + 2 * nf, 1), dtype=torch.int32, device=dev)
            mult = torch.empty(max(self.nnz + 2 * nf, 1), dtype=torch.float32, device=dev)
            degree = torch.empty(Nn, dtype=torch.int32, device=dev)
            nbytes = L.recad_csr_append_scratch_bytes(n_users, n_items, F, nf)
            scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            check(L.recad_csr_append_users(_ptr(self.rowptr), _ptr(self.colidx), _ptr(self.mult), n_users, n_items, F,
                                           _ptr(fake_rowptr), _ptr(fake_items), nf, _ptr(rowptr), _ptr(colidx), _ptr(mult),
                                           _ptr(degree), _ptr(scratch), nbytes, _stream(dev)), "recad_csr_append_users")
            colidx, mult = colidx[:self.nnz + 2 * nf], mult[:self.nnz + 2 * nf]
            if degree_hook is not None:
                degree_hook(degree)
            vals = self._normalize(rowptr, colidx, mult, degree, Nn)
        return Graph(Nn, Nn, rowptr, colidx, vals, mult, degree, self.seg_len, split=n_users + F)

    def renormalized(self, degree):
        """The same structure with values recomputed from new degrees (a shard whose own rows did not
        change while fake users elsewhere changed the item degrees)."""
        with torch.cuda.device(self.device):
            vals = self._normalize(self.rowptr, self.colidx, self.mult, degree, self.n_rows)
        return Graph(self.n_rows, self.n_cols, self.rowptr, self.colidx, vals, self.mult, degree, self.seg_len, split=self.split)

    @classmethod
    def from_csr(cls, rowptr, colidx, vals, n_cols, seg_len=SEG_LEN, split=None):
        """Wrap an existing (possibly rectangular) CSR, e.g. a user-row shard or a cached adjacency (split = n_users for
        the symmetric bipartite matrix).  Without multiplicities / degrees such a graph cannot be extended in place."""
        _need_cuda(rowptr, colidx, vals)
        return cls(rowptr.numel() - 1, n_cols, rowptr.contiguous().long(), colidx.contiguous().int(),
                   vals.contiguous().float(), None, None, seg_len, split=split)

    # -- plan ---------------------------------------------------------------- #
    def _plan(self):
        if self.split is not None and 0 < self.split < self.n_rows:
            U = self.split
            groups = [(0, U, U, self.n_cols, auto_col_blocks(self.n_cols - U)), (U, self.n_rows, 0, U, auto_col_blocks(U))]
        else:
            groups = [(0, self.n_rows, 0, self.n_cols, auto_col_blocks(self.n_cols))]
        self.plan = PackedPlan.build(self.rowptr, self.colidx, self.n_rows, self.seg_len, groups)
        self.n_seg, self.n_mrow, self.n_slot = self.plan.n_seg, self.plan.n_mrow, self.plan.n_slot
        with torch.cuda.device(self.device):
            self.cv = torch.empty((max(self.nnz, 1), 2), dtype=torch.int32, device=self.device)
            check(_lib.lib().recad_spmm_pack_cv(_ptr(self.colidx), _ptr(self.vals), self.nnz, _ptr(self.cv), _stream(self.device)),
                  "recad_spmm_pack_cv")
            self.row_cnt = torch.zeros(self.n_rows, dtype=torch.int32, device=self.device)

    def struct(self, D):
        """ctypes recad_csr for embedding width D.  The partial-sum scratch is per D and is never freed while a
        struct handed out for that D may still be referenced by a victim."""
        if D not in self._structs:
            self._partials[D] = torch.empty(max(self.n_slot, 1) * D, dtype=torch.float32, device=self.device)
            s = _lib.CSR()
            s.n_rows, s.n_cols, s.nnz = self.n_rows, self.n_cols, self.nnz
            s.rowptr, s.colidx, s.vals, s.cv = self.rowptr.data_ptr(), self.colidx.data_ptr(), self.vals.data_ptr(), self.cv.data_ptr()
            s.n_seg, s.seg_meta = self.n_seg, self.plan.meta.data_ptr()
            s.n_mrow, s.row_mseg, s.row_cnt = self.n_mrow, self.plan.row_mseg.data_ptr(), self.row_cnt.data_ptr()
            s.partials = self._partials[D].data_ptr()
            self._structs[D] = s
        return self._structs[D]

    def with_values(self, vals=None):
        """A matrix with this one's structure and PLAN but values of its own (graph dropout: the kept entries rescaled, the
        dropped ones zero).  Only vals / cv and the partial-sum scratch are new; call `set_values` to refill them in place
        (the structs handed out stay valid).  Shares row_cnt with its parent: never launch both at the same time."""
        g = object.__new__(Graph)
        g.__dict__.update(self.__dict__)
        g._partials, g._structs = {}, {}
        with torch.cuda.device(self.device):
            g.vals = torch.empty_like(self.vals)
            g.cv = torch.empty_like(self.cv)
        g.set_values(self.vals if vals is None else vals)
        return g

    def transpose_permutation(self):
        """T with entry k = (r, c) -> the position of (c, r): vals[T] are the values of the transposed matrix on the SAME
        structure (square, structurally symmetric matrices only -- the bipartite adjacency).  Cached."""
        if getattr(self, "_tperm", None) is None:
            if self.n_rows != self.n_cols:
                raise RecadError("transpose_permutation: the matrix is not square")
            with torch.cuda.device(self.device):
                rows = torch.repeat_interleave(torch.arange(self.n_rows, device=self.device), self.rowptr[1:] - self.rowptr[:-1])
                cols = self.colidx.long()
                keys = rows * self.n_cols + cols                              # ascending: CSR order with sorted columns
                T = torch.searchsorted(keys, cols * self.n_cols + rows)
                if self.nnz and not bool((keys[T.clamp_(max=self.nnz - 1)] == cols * self.n_cols + rows).all()):
                    raise RecadError("transpose_permutation: the structure is not symmetric")
            self._tperm = T
        return self._tperm

    def entry_index(self, rows, cols, missing=None):
        """int64 positions (CSR entry order) of the stored entries (rows[j], cols[j]); RecadError if a pair is not stored,
        unless `missing` is given: an int returned at the pairs that are not stored (out-of-range ids still raise).
        With transpose_permutation, entry_index(r, c) and T[entry_index(r, c)] are the two entries of one interaction."""
        with torch.cuda.device(self.device):
            rows = torch.as_tensor(rows, device=self.device).long()
            cols = torch.as_tensor(cols, device=self.device).long()
            if rows.shape != cols.shape:
                raise RecadError(f"entry_index: {tuple(rows.shape)} rows but {tuple(cols.shape)} columns")
            if rows.numel() and bool(((rows < 0) | (rows >= self.n_rows) | (cols < 0) | (cols >= self.n_cols)).any()):
                raise RecadError("entry_index: a row or column is out of range")
            if getattr(self, "_ekeys", None) is None:
                r = torch.repeat_interleave(torch.arange(self.n_rows, device=self.device), self.rowptr[1:] - self.rowptr[:-1])
                self._ekeys = r * self.n_cols + self.colidx.long()              # ascending: CSR order with sorted columns
            q = rows * self.n_cols + cols
            k = torch.searchsorted(self._ekeys, q.reshape(-1)).clamp_(max=max(self.nnz - 1, 0)).reshape(q.shape)
            if missing is not None:
                found = self._ekeys[k] == q if self.nnz else torch.zeros_like(q, dtype=torch.bool)
                return torch.where(found, k, torch.full_like(k, int(missing)))
            if q.numel() and (self.nnz == 0 or not bool((self._ekeys[k] == q).all())):
                raise RecadError("entry_index: a (row, column) pair is not a stored entry")
        return k

    def set_values(self, vals):
        with torch.cuda.device(self.device):
            self.vals.copy_(vals)
            check(_lib.lib().recad_spmm_pack_cv(_ptr(self.colidx), _ptr(self.vals), self.nnz, _ptr(self.cv), _stream(self.device)),
                  "recad_spmm_pack_cv")

    # -- export --------------------------------------------------------------- #
    def to_numpy(self):
        return (self.rowptr.cpu().numpy(), self.colidx.cpu().numpy().astype(np.int64), self.vals.cpu().numpy())

    def to_torch_sparse(self):
        """torch sparse COO view with the reference's layout (implicit.py:295-296)."""
        rows = torch.repeat_interleave(torch.arange(self.n_rows, device=self.device), self.rowptr[1:] - self.rowptr[:-1])
        return torch.sparse_coo_tensor(torch.stack([rows, self.colidx.long()]), self.vals, (self.n_rows, self.n_cols)).coalesce()

    def algorithmic_bytes(self, D):
        """SURVEY.md section 8(d) no-reuse gather model for one SpMM over this matrix."""
        return self.nnz * (8 + 4 * D) + self.n_rows * 4 * D + (self.n_rows + 1) * 4


def spmm(graph, X, Y=None, C_=None, Z=None, alpha=1.0):
    """Y = A X; Z = alpha * (C + A X).  Returns (Y, Z)."""
    _need_cuda(X, Y, C_, Z)
    D = X.shape[1]
    with torch.cuda.device(X.device):
        check(_lib.lib().recad_spmm(C.byref(graph.struct(D)), _ptr(X), _ptr(Y), _ptr(C_), _ptr(Z), float(alpha), D,
                                    _stream(X.device)), "recad_spmm")
    return Y, Z


def sddmm(graph, G, X, alpha=1.0, out=None, accumulate=False):
    """out[k] = alpha * <G[r_k], X[c_k]> for every stored entry k = (r_k, c_k), in CSR entry order (recad_csr_sddmm); with
    `accumulate`, out[k] += ... into the given `out`.  The gradient of sum(gY * (A X)) with respect to A's values for
    G = gY.  Returns out (float32 [nnz])."""
    _need_cuda(G, X, out)
    D = int(X.shape[1]) if X.dim() == 2 else -1
    if G.dtype != torch.float32 or X.dtype != torch.float32 or tuple(G.shape) != (graph.n_rows, D) or \
            tuple(X.shape) != (graph.n_cols, D):
        raise RecadError(f"sddmm: G must be float32 [{graph.n_rows}, D] and X float32 [{graph.n_cols}, D]")
    if accumulate and out is None:
        raise RecadError("sddmm: accumulate needs out")
    if out is not None and (out.dtype != torch.float32 or out.numel() != graph.nnz or not out.is_contiguous()):
        raise RecadError(f"sddmm: out must be a contiguous float32 tensor of {graph.nnz} entries")
    with torch.cuda.device(X.device):
        if out is None:
            out = torch.empty(graph.nnz, dtype=torch.float32, device=X.device)
        check(_lib.lib().recad_csr_sddmm(C.byref(graph.struct(D)), _ptr(G.contiguous()), _ptr(X.contiguous()), D, float(alpha),
                                         int(bool(accumulate)), _ptr(out), _stream(X.device)), "recad_csr_sddmm")
    return out


def axpby(z, a, x, b, y):
    """z = a * x + b * y (z may alias x or y)."""
    _need_cuda(z, x, y)
    with torch.cuda.device(z.device):
        check(_lib.lib().recad_axpby(_ptr(z), float(a), _ptr(x), float(b), _ptr(y), z.numel(), _stream(z.device)), "recad_axpby")
    return z


def bpr_fwd_bwd(O, E, n_users, n_items, samples, perm, grad_scale, gO, cnt, loss_acc, B_norm=None):
    """samples: int64 [n, 3] (user, pos, neg); perm: int64 [B] rows of this batch or None (= all rows in order).
    B_norm: batch size used for the 1/B normalisation (default: the number of rows processed)."""
    _need_cuda(O, E, samples, perm, gO, cnt, loss_acc)
    B = perm.numel() if perm is not None else samples.shape[0]
    with torch.cuda.device(O.device):
        check(_lib.lib().recad_bpr_fwd_bwd(_ptr(O), _ptr(E), n_users, n_items, _ptr(samples), _ptr(perm), B,
                                           int(B_norm or B), float(grad_scale), _ptr(gO), _ptr(cnt), _ptr(loss_acc), O.shape[1], _stream(O.device)),
              "recad_bpr_fwd_bwd")


def adam(p, g, m, v, step, lr=1e-3, b1=0.9, b2=0.999, eps=1e-8, cnt=None, reg_scale=0.0):
    _need_cuda(p, g, m, v, cnt)
    D = p.shape[1] if p.dim() == 2 else 1
    with torch.cuda.device(p.device):
        check(_lib.lib().recad_adam(_ptr(p), _ptr(g), _ptr(cnt), float(reg_scale), _ptr(m), _ptr(v), p.numel(), D, lr, b1, b2, eps,
                                    int(step), _stream(p.device)), "recad_adam")


def gemm_tn(A, B, bias=None, relu=False):
    """C = A @ B.T (+ bias) (relu) on the tensor cores (tcgen05, 3xTF32 = fp32-accurate).  A [M, K], B [N, K]."""
    _need_cuda(A, B, bias)
    M, K = A.shape
    N = B.shape[0]
    ld = (K + 3) // 4 * 4
    out = torch.empty((M, N), dtype=torch.float32, device=A.device)
    with torch.cuda.device(A.device):
        scratch = torch.empty(2 * (M + N) * ld, dtype=torch.float32, device=A.device)
        check(_lib.lib().recad_gemm_tn_tf32x3(_ptr(A.contiguous()), _ptr(B.contiguous()), M, N, K, _ptr(bias), int(relu), _ptr(out),
                                              _ptr(scratch), _stream(A.device)), "recad_gemm_tn_tf32x3")
    return out


def dot_scores(O, n_users, users, items):
    _need_cuda(O, users, items)
    out = torch.empty(users.numel(), dtype=torch.float32, device=O.device)
    with torch.cuda.device(O.device):
        check(_lib.lib().recad_dot_scores(_ptr(O), n_users, _ptr(users), _ptr(items), users.numel(), O.shape[1], _ptr(out),
                                          _stream(O.device)), "recad_dot_scores")
    return out


def mf_forward(st, users, items):
    """recad_mf_forward over the tables of an MF state: <Ue[u], Ie[i]> + Ub[u] + Ib[i] + mean."""
    dev = users.device
    out = torch.empty(users.numel(), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        check(_lib.lib().recad_mf_forward(C.byref(st), _ptr(users), _ptr(items), users.numel(), _ptr(out), _stream(dev)),
              "recad_mf_forward")
    return out


def ncf_forward(st, users, items):
    """recad_ncf_forward in slices of st.max_batch pairs."""
    dev = users.device
    n = users.numel()
    out = torch.empty(n, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        for s in range(0, n, st.max_batch):
            e = min(s + st.max_batch, n)
            check(_lib.lib().recad_ncf_forward(C.byref(st), _ptr(users[s:e]), _ptr(items[s:e]), e - s, _ptr(out[s:e]), _stream(dev)),
                  "recad_ncf_forward")
    return out


# --------------------------------------------------------------------------- #
# autograd: backward passes of the victims' scores
# --------------------------------------------------------------------------- #
def pair_scores_backward(Xa, Xb, ia, ib, g, bias=False):
    """Gradient of s_b = <Xa[ia_b], Xb[ib_b]> (+ ba[ia_b] + bb[ib_b]) for the upstream gradient g (recad_pair_scores_backward):
    (dX [n_a + n_b, D] with the rows of Xa first, dba [n_a], dbb [n_b]); the bias gradients are None unless `bias`.
    Atomic-free: the same bits on every run at any batch size.  An id out of range raises RecadError."""
    return pair_scores_hvp(Xa, None, Xb, None, ia, ib, g, None, bias)


def pair_scores_hvp(Xa, Va, Xb, Vb, ia, ib, alpha, beta, bias=False):
    """out[r] = sum over the b with ia_b = r of (alpha_b Xb[ib_b] + beta_b Vb[ib_b]) for the rows of A, and the same with
    Xa / Va for the rows of B (recad_pair_scores_hvp): (out [n_a + n_b, D] with the rows of A first, dba [n_a], dbb [n_b] =
    the sums of alpha per row, None unless `bias`).  beta None: the pair backward, and Va / Vb are not read.  Atomic-free and
    bit-stable; an id out of range raises RecadError."""
    _need_cuda(Xa, Va, Xb, Vb, ia, ib, alpha, beta)
    dev = Xa.device
    (n_a, D), n_b, B = Xa.shape, Xb.shape[0], ia.numel()
    L = _lib.lib()
    with torch.cuda.device(dev):
        out = torch.empty((n_a + n_b, D), dtype=torch.float32, device=dev)
        dba = torch.empty(n_a, dtype=torch.float32, device=dev) if bias else None
        dbb = torch.empty(n_b, dtype=torch.float32, device=dev) if bias else None
        nbytes = int(L.recad_pair_scores_backward_scratch_bytes(B))
        scratch = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=dev)
        if beta is None:
            check(L.recad_pair_scores_backward(_ptr(Xa), n_a, _ptr(Xb), n_b, D, _ptr(ia), _ptr(ib), B, _ptr(alpha),
                                               _ptr(out[:n_a]), _ptr(out[n_a:]), _ptr(dba), _ptr(dbb), _ptr(scratch), nbytes,
                                               _stream(dev)), "recad_pair_scores_backward")
        else:
            check(L.recad_pair_scores_hvp(_ptr(Xa), _ptr(Va), n_a, _ptr(Xb), _ptr(Vb), n_b, D, _ptr(ia), _ptr(ib), B, _ptr(alpha),
                                          _ptr(beta), _ptr(out[:n_a]), _ptr(out[n_a:]), _ptr(dba), _ptr(dbb), _ptr(scratch), nbytes,
                                          _stream(dev)), "recad_pair_scores_hvp")
    return out, dba, dbb


def bpr_hvp_seeds(O, dO, n_users, samples, lam=0.0, E=None, V=None, dloss=False):
    """Seeds of the BPR loss's Hessian-vector product over the rows samples int64 [n, 3] (recad_bpr_hvp_seeds, B = n):
    (alpha [2n], beta [2n], dloss [n] or None) for the pairs (u, neg) then (u, pos).  With `dloss`, each sample's derivative
    along V, l'(x_b) dx_b + lam (<V_u, E_u> + <V_p, E_p> + <V_n, E_n>), where dO = P V."""
    _need_cuda(O, dO, samples, E, V)
    dev = O.device
    N, D = O.shape
    n = samples.shape[0]
    with torch.cuda.device(dev):
        alpha = torch.empty(2 * n, dtype=torch.float32, device=dev)
        beta = torch.empty(2 * n, dtype=torch.float32, device=dev)
        dl = torch.empty(n, dtype=torch.float32, device=dev) if dloss else None
        bad = torch.empty(1, dtype=torch.int32, device=dev)
        check(_lib.lib().recad_bpr_hvp_seeds(_ptr(O), _ptr(dO), n_users, N - n_users, _ptr(samples), n, n, D,
                                             _ptr(E if dloss else None), _ptr(V if dloss else None), float(lam), _ptr(alpha),
                                             _ptr(beta), _ptr(dl), _ptr(bad), _stream(dev)), "recad_bpr_hvp_seeds")
    return alpha, beta, dl


def lightgcn_loss_mixed_values(st, graph, S, samples):
    """recad_lightgcn_loss_mixed_values: d/dv <S, grad_E L> (float32 [nnz], the graph's entry order) for the BPR loss of the
    rows samples int64 [n, 3] at a LightGCN state over `graph` (its own values), S float32 [N, D].  Fresh buffers only."""
    _need_cuda(S, samples)
    dev = S.device
    N, D = S.shape
    n = samples.shape[0]
    L = _lib.lib()
    with torch.cuda.device(dev):
        nbytes = int(L.recad_lightgcn_loss_mixed_values_work_bytes(N, D, st.n_layers, n))
        work = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=dev)
        out = torch.empty(graph.nnz, dtype=torch.float32, device=dev)
        check(L.recad_lightgcn_loss_mixed_values(C.byref(st), C.byref(graph.struct(2 * D)), _ptr(S), _ptr(samples), n, _ptr(out),
                                                 _ptr(work), nbytes, _stream(dev)), "recad_lightgcn_loss_mixed_values")
    return out


def lightgcn_candidate_weight_grads(st, graph, users, gO=None, S=None, samples=None, lam=0.0):
    """recad_lightgcn_candidate_weight_grads: float32 [len(users), n_items], the gradient of <gO, O> + <S, grad_E L> with
    respect to one weight on both entries of every interaction (users[r], item i), stored or not, at the base point
    W = graph.mult (0 where not stored), for a LightGCN state over `graph` (its own values).  users int64 [R]; gO, S float32
    [N, D] or None; samples int64 [n, 3] (with S) or None; lam the regulariser's weight in the rows' losses.  d_inv is
    weights_d_inv(graph, graph.mult), so the base point's values are normalized_values(graph, graph.mult) bit for bit.
    Fresh buffers only."""
    _need_cuda(users, gO, S, samples)
    if (S is None) != (samples is None):
        raise RecadError("lightgcn_candidate_weight_grads: S and samples go together")
    if graph.mult is None:
        raise RecadError("lightgcn_candidate_weight_grads: the graph carries no interaction weights (mult)")
    dev = users.device
    U, I, D = st.n_users, st.n_items, st.D
    n = 0 if samples is None else int(samples.shape[0])
    R = int(users.numel())
    L = _lib.lib()
    with torch.cuda.device(dev):
        out = torch.empty((R, I), dtype=torch.float32, device=dev)
        if R == 0:
            return out
        users = users.contiguous().long()
        d_inv = weights_d_inv(graph, graph.mult)
        nbytes = int(L.recad_lightgcn_candidate_weight_grads_work_bytes(U, I, D, st.n_layers, n, graph.nnz, R))
        work = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=dev)
        check(L.recad_lightgcn_candidate_weight_grads(
            C.byref(st), C.byref(graph.struct(2 * D)), _ptr(graph.mult), _ptr(graph.transpose_permutation()), _ptr(d_inv),
            _ptr(gO), _ptr(S), _ptr(samples), n, float(lam), _ptr(users), R, _ptr(out), _ptr(work), nbytes, _stream(dev)),
            "recad_lightgcn_candidate_weight_grads")
    return out


def index_sums(idx, x, n_out):
    """out[r] = sum of x[b] over the b with idx[b] = r (float32 [n_out]; entries of idx below 0 are skipped), atomic-free and
    bit-stable (recad_index_sums: one stable sort, one writer per output, summed in double).  An index >= n_out raises."""
    _need_cuda(idx, x)
    dev = x.device
    n = int(x.numel())
    L = _lib.lib()
    with torch.cuda.device(dev):
        out = torch.zeros(n_out, dtype=torch.float32, device=dev)
        if n == 0:
            return out
        nbytes = int(L.recad_pair_scores_backward_scratch_bytes(n))
        scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        check(L.recad_index_sums(_ptr(idx.contiguous().long()), _ptr(x.contiguous().float()), n, int(n_out), _ptr(out),
                                 _ptr(scratch), nbytes, _stream(dev)), "recad_index_sums")
    return out


def mf_hvp_seeds(st, dUe, dUb, dIe, dIb, samples, dloss=False):
    """Seeds of the BCE loss's Hessian-vector product over the (user, item, label) rows samples int64 [n, 3] of an MF state
    along (dUe, dUb, dIe, dIb) (recad_mf_hvp_seeds, B = n): (alpha [n], beta [n], dloss [n] or None)."""
    _need_cuda(dUe, dUb, dIe, dIb, samples)
    dev = samples.device
    n = samples.shape[0]
    with torch.cuda.device(dev):
        alpha = torch.empty(n, dtype=torch.float32, device=dev)
        beta = torch.empty(n, dtype=torch.float32, device=dev)
        dl = torch.empty(n, dtype=torch.float32, device=dev) if dloss else None
        bad = torch.empty(1, dtype=torch.int32, device=dev)
        check(_lib.lib().recad_mf_hvp_seeds(C.byref(st), _ptr(dUe), _ptr(dUb), _ptr(dIe), _ptr(dIb), _ptr(samples), n, n,
                                            _ptr(alpha), _ptr(beta), _ptr(dl), _ptr(bad), _stream(dev)), "recad_mf_hvp_seeds")
    return alpha, beta, dl


def ncf_hvp(st, samples, vec_flat, out=True, dloss=False):
    """Hessian-vector product of an NCF state's BCE training loss over the (user, item, label) rows samples int64 [n, 3] taken
    as one batch, along vec_flat float32 [n_params] (recad_ncf_layout order) (recad_ncf_hvp): (H v [n_params] or None,
    dloss [n] or None), dloss[b] = <grad l_b, v>.  Deterministic; the state's parameters, moments and loss accumulator are not
    touched.  An id out of range raises RecadError."""
    _need_cuda(samples, vec_flat)
    dev = samples.device
    n = samples.shape[0]
    L = _lib.lib()
    with torch.cuda.device(dev):
        hv = torch.empty(st.n_params, dtype=torch.float32, device=dev) if out else None
        dl = torch.empty(n, dtype=torch.float32, device=dev) if dloss else None
        wf = int(L.recad_ncf_hvp_work_floats(st.factor, st.n_layers, st.max_batch))
        work = torch.empty(max(wf, 1), dtype=torch.float32, device=dev)
        check(L.recad_ncf_hvp(C.byref(st), _ptr(samples), n, _ptr(vec_flat), _ptr(hv), _ptr(dl), _ptr(work), wf, _stream(dev)),
              "recad_ncf_hvp")
    return hv, dl


def lightgcn_backward(st, gO):
    """gE = (1 / (L + 1)) sum_l (A^T)^l gO (recad_lightgcn_backward) for a LightGCN state; the Horner loop runs through work
    buffers of its own, so the state's X0 / X1 are left alone."""
    _need_cuda(gO)
    dev = gO.device
    with torch.cuda.device(dev):
        gE = torch.empty_like(gO)
        work = [torch.empty_like(gO) for _ in range(min(max(st.n_layers - 1, 0), 2))]
        sb = _lib.LightGCN()
        C.memmove(C.byref(sb), C.byref(st), C.sizeof(sb))
        sb.X0 = work[0].data_ptr() if len(work) > 0 else None
        sb.X1 = work[1].data_ptr() if len(work) > 1 else None
        check(_lib.lib().recad_lightgcn_backward(C.byref(sb), _ptr(gO), _ptr(gE), _stream(dev)), "recad_lightgcn_backward")
    return gE


def ncf_backward(st, users, items, dpred):
    """Flat gradient (recad_ncf_layout order) of sum_b dpred[b] pred[b] for an NCF state (recad_ncf_backward), in slices of
    st.max_batch pairs."""
    _need_cuda(users, items, dpred)
    dev = dpred.device
    n = users.numel()
    with torch.cuda.device(dev):
        grads = torch.empty(st.n_params, dtype=torch.float32, device=dev)
        part = torch.empty_like(grads) if n > st.max_batch else None
        for s in range(0, n, st.max_batch):
            e = min(s + st.max_batch, n)
            dst = grads if s == 0 else part
            check(_lib.lib().recad_ncf_backward(C.byref(st), _ptr(users[s:e]), _ptr(items[s:e]), e - s, _ptr(dpred[s:e]), _ptr(dst),
                                                _stream(dev)), "recad_ncf_backward")
            if s:
                grads += part
    return grads


class LightGCNPropagate(torch.autograd.Function):
    """O = mean_l A^l E (lightgcn.py:82-113) into a fresh [N, D] buffer; backward by recad_lightgcn_backward.  graph_t /
    vals_t: the transposed matrix of a dropped graph and the values this propagation drew for it -- restored before the
    backward, so that it uses this forward's mask even if a later forward drew another."""

    @staticmethod
    def forward(ctx, st, graph_t, vals_t, user_w, item_w):
        N = st.n_users + st.n_items
        dev = user_w.device
        with torch.cuda.device(dev):
            O = torch.empty((N, st.D), dtype=torch.float32, device=dev)
            sf = _lib.LightGCN()
            C.memmove(C.byref(sf), C.byref(st), C.sizeof(sf))
            sf.O = O.data_ptr()
            check(_lib.lib().recad_lightgcn_propagate(C.byref(sf), _stream(dev)), "recad_lightgcn_propagate")
        ctx.st, ctx.graph_t, ctx.vals_t = sf, graph_t, vals_t
        return O

    @staticmethod
    @once_differentiable
    def backward(ctx, gO):
        if ctx.graph_t is not None:
            ctx.graph_t.set_values(ctx.vals_t)
        gE = lightgcn_backward(ctx.st, gO.contiguous())
        U = ctx.st.n_users
        return None, None, None, gE[:U], gE[U:]


def check_values(graph, values, what):
    """RecadError unless `values` is a float32 CUDA tensor [graph.nnz] on the graph's device."""
    if not isinstance(values, torch.Tensor) or not values.is_cuda:
        raise RecadError(f"{what}: a float32 CUDA tensor [{graph.nnz}] is needed (got {type(values).__name__}"
                         f"{' on the CPU' if isinstance(values, torch.Tensor) else ''})")
    if values.dtype != torch.float32 or tuple(values.shape) != (graph.nnz,) or values.device != graph.device:
        raise RecadError(f"{what}: float32 [{graph.nnz}] on {graph.device} needed, got {values.dtype} "
                         f"{list(values.shape)} on {values.device}")


class ValueGraphs:
    """A LightGCN state whose propagation runs over caller-supplied values instead of its graph's: a value copy of the graph
    and of its transpose (the same structure and plan, values[T]), made by Graph.with_values on the first `load` and
    refilled in place by set_values after that.  A victim keeps one, as it keeps its dropped graph."""

    def __init__(self, graph, st):
        self.graph, self.base, self.g, self.g_t, self.st = graph, st, None, None, None

    def load(self, values):
        """Fill both matrices with `values` / values[T] and return the state that propagates over them."""
        with torch.cuda.device(self.graph.device):
            values = values.detach()
            vals_t = values[self.graph.transpose_permutation()]
            if self.g is None:
                self.g, self.g_t = self.graph.with_values(values), self.graph.with_values(vals_t)
                st = _lib.LightGCN()
                C.memmove(C.byref(st), C.byref(self.base), C.sizeof(st))
                st.graph = C.pointer(self.g.struct(st.D))
                st.graph_t = C.pointer(self.g_t.struct(st.D))
                self.st = st
            else:
                self.g.set_values(values)
                self.g_t.set_values(vals_t)
        return self.st


def lightgcn_propagate_layers(st, E, keep):
    """O = mean_l A^l E over st.graph into a fresh [N, D] buffer, layer by layer with recad_spmm (the calls
    recad_lightgcn_propagate makes, so the bits are the same), and the layers [E, X_1, .., X_{L-1}] when `keep`."""
    N, D, L = st.n_users + st.n_items, st.D, st.n_layers
    dev = E.device
    lib = _lib.lib()
    with torch.cuda.device(dev):
        O = torch.empty((N, D), dtype=torch.float32, device=dev)
        if L == 0:
            O.copy_(E)
            return O, [E]
        layers, x = [E], E
        work = [torch.empty_like(O) for _ in range(min(L - 1, 2))] if not keep else []
        for k in range(L):
            last = k == L - 1
            y = None if last else (torch.empty_like(O) if keep else work[k & 1])
            check(lib.recad_spmm(st.graph, _ptr(x), _ptr(y), _ptr(E if k == 0 else O), _ptr(O),
                                 1.0 / (L + 1) if last else 1.0, D, _stream(dev)), "recad_spmm")
            if keep and y is not None:
                layers.append(y)
            x = y
    return O, (layers if keep else None)


class LightGCNPropagateValues(torch.autograd.Function):
    """O = mean_l A^l E with A's values given as a tensor [nnz] (CSR entry order), differentiable with respect to those
    values and both tables.  `vg` is the victim's ValueGraphs; E is the victim's table, of which user_w / item_w are the
    views.  The layers X_1 .. X_{L-1} are kept for the backward, which first restores its own forward's values into the
    value graphs (a later forward may have loaded others) and then runs recad_lightgcn_backward_values (edge values
    wanted) or recad_lightgcn_backward."""

    @staticmethod
    def forward(ctx, vg, E, values, user_w, item_w):
        st = vg.load(values)
        O, layers = lightgcn_propagate_layers(st, E, keep=True)
        ctx.vg, ctx.E, ctx.layers = vg, E, layers
        ctx.save_for_backward(values, user_w, item_w)
        return O

    @staticmethod
    @once_differentiable
    def backward(ctx, gO):
        values, _, _ = ctx.saved_tensors
        need_v, need_u, need_i = ctx.needs_input_grad[2:5]
        st = ctx.vg.load(values)
        gO = gO.contiguous()
        dev, U, L = gO.device, st.n_users, st.n_layers
        lib = _lib.lib()
        with torch.cuda.device(dev):
            gE = torch.empty_like(gO) if (need_u or need_i) else None
            work = [torch.empty_like(gO) for _ in range(min(max(L - 1, 0), 2))]
            sb = _lib.LightGCN()
            C.memmove(C.byref(sb), C.byref(st), C.sizeof(sb))
            sb.X0 = work[0].data_ptr() if len(work) > 0 else None
            sb.X1 = work[1].data_ptr() if len(work) > 1 else None
            gvals = None
            if need_v:
                gvals = torch.empty(values.numel(), dtype=torch.float32, device=dev)
                X = (_lib.vp * max(L, 1))(*[x.data_ptr() for x in ctx.layers[:L]])
                check(lib.recad_lightgcn_backward_values(C.byref(sb), _ptr(gO), X, _ptr(gE), _ptr(gvals), _stream(dev)),
                      "recad_lightgcn_backward_values")
            else:
                check(lib.recad_lightgcn_backward(C.byref(sb), _ptr(gO), _ptr(gE), _stream(dev)), "recad_lightgcn_backward")
        return (None, None, gvals, gE[:U] if need_u else None, gE[U:] if need_i else None)


def lightgcn_propagate_values(st_vals, E):
    """recad_lightgcn_propagate over a value-graph state into fresh buffers (no autograd)."""
    O, _ = lightgcn_propagate_layers(st_vals, E, keep=False)
    return O


def weights_d_inv(graph, weights):
    """d_r = (s_r + 1e-14)^(-1/2) of the row sums s_r of per-entry weights [nnz] (recad_csr_row_sums, then the host
    expression d_inv_from_degree): the normalisation factors normalized_values uses."""
    dev = graph.device
    with torch.cuda.device(dev):
        sums = torch.empty(graph.n_rows, dtype=torch.float32, device=dev)
        check(_lib.lib().recad_csr_row_sums(_ptr(graph.rowptr), _ptr(weights), graph.n_rows, graph.nnz, _ptr(sums),
                                            _stream(dev)), "recad_csr_row_sums")
        return torch.from_numpy(d_inv_from_degree(sums.cpu().numpy())).to(dev)


class NormalizedValues(torch.autograd.Function):
    """vals_k = d_r w_k d_c from per-entry weights (recad_csr_row_sums, the host d_inv, recad_csr_normalize); backward by
    recad_csr_normalize_backward."""

    @staticmethod
    def forward(ctx, graph, weights):
        dev = graph.device
        lib = _lib.lib()
        with torch.cuda.device(dev):
            d_inv = weights_d_inv(graph, weights)
            vals = torch.empty(graph.nnz, dtype=torch.float32, device=dev)
            check(lib.recad_csr_normalize(_ptr(graph.rowptr), _ptr(graph.colidx), _ptr(weights), _ptr(d_inv), graph.n_rows,
                                          _ptr(vals), _stream(dev)), "recad_csr_normalize")
        ctx.graph, ctx.d_inv = graph, d_inv
        ctx.save_for_backward(weights)
        return vals

    @staticmethod
    @once_differentiable
    def backward(ctx, gv):
        weights, = ctx.saved_tensors
        g = ctx.graph
        dev = g.device
        with torch.cuda.device(dev):
            gv = gv.contiguous().float()
            coef = torch.empty(g.n_rows, dtype=torch.float32, device=dev)
            gw = torch.empty(g.nnz, dtype=torch.float32, device=dev)
            check(_lib.lib().recad_csr_normalize_backward(_ptr(g.rowptr), _ptr(g.colidx), _ptr(g.transpose_permutation()),
                                                          _ptr(weights), _ptr(ctx.d_inv), _ptr(gv), g.n_rows, g.nnz, _ptr(coef),
                                                          _ptr(gw), _stream(dev)), "recad_csr_normalize_backward")
        return None, gw


def normalized_values(graph, weights):
    """The symmetric normalisation (implicit.py:269-276) as a differentiable map from per-entry weights [nnz] (CSR entry
    order) to values: vals_k = d_r w_k d_c, d_r = (sum of row r's weights + 1e-14)^(-1/2), d_inv evaluated on the host
    exactly as for the dataset's graph, so normalized_values(g, g.mult) equals g.vals.  For a square, structurally
    symmetric graph; the weights need not be symmetric."""
    if graph.n_rows != graph.n_cols:
        raise RecadError("normalized_values: the matrix is not square")
    check_values(graph, weights, "normalized_values")
    graph.transpose_permutation()                 # RecadError unless the structure is symmetric
    return NormalizedValues.apply(graph, weights.contiguous())


class DotScores(torch.autograd.Function):
    """scores[b] = <O[users[b]], O[n_users + items[b]]> (lightgcn.py:174-183); backward by recad_pair_scores_backward."""

    @staticmethod
    def forward(ctx, O, n_users, users, items):
        ctx.save_for_backward(O, users, items)
        ctx.n_users = n_users
        return dot_scores(O, n_users, users, items)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        O, users, items = ctx.saved_tensors
        U = ctx.n_users
        dO, _, _ = pair_scores_backward(O[:U], O[U:], users, items, g.contiguous().float())
        return dO, None, None, None


class MFScores(torch.autograd.Function):
    """pred = <Ue[u], Ie[i]> + Ub[u] + Ib[i] + mean (mf.py:40-47) over the tables of an MF state (the four tables and mean are
    passed so that autograd routes their gradients); backward by recad_pair_scores_backward."""

    @staticmethod
    def forward(ctx, st, users, items, Ue, Ub, Ie, Ib, mean):
        ctx.save_for_backward(users, items, Ue, Ie)
        return mf_forward(st, users, items)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        users, items, Ue, Ie = ctx.saved_tensors
        U, I = Ue.shape[0], Ie.shape[0]
        g = g.contiguous().float()
        dX, dUb, dIb = pair_scores_backward(Ue, Ie, users, items, g, bias=True)
        dmean = g.sum().view(1) if ctx.needs_input_grad[7] else None
        return None, None, None, dX[:U], dUb.view(U, 1), dX[U:], dIb.view(I, 1), dmean


class NCFScores(torch.autograd.Function):
    """pred = NCF(users, items) (ncf.py:112-131) over the flat parameter buffer of an NCF state; `params` are the parameter
    views in recad_ncf_layout order at float offsets `offs`, so that autograd routes the flat gradient back onto them."""

    @staticmethod
    def forward(ctx, st, offs, users, items, *params):
        ctx.st, ctx.offs = st, offs
        ctx.save_for_backward(users, items, *params)     # the backward recomputes the forward: in-place edits must fail it
        return ncf_forward(st, users, items)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        users, items = ctx.saved_tensors[:2]
        flat = ncf_backward(ctx.st, users, items, g.contiguous().float())
        grads = tuple(flat[o:o + n].view(s) for o, n, s in ctx.offs)
        return (None, None, None, None) + grads


# --------------------------------------------------------------------------- #
# evaluation
# --------------------------------------------------------------------------- #
def transpose_items(item_emb):
    """[I, D] -> [D, ld] with ld = I rounded up to 64, zero padded."""
    _need_cuda(item_emb)
    I, D = item_emb.shape
    ld = (I + 63) // 64 * 64
    out = torch.zeros((D, ld), dtype=torch.float32, device=item_emb.device)
    with torch.cuda.device(item_emb.device):
        check(_lib.lib().recad_transpose_items(_ptr(item_emb.contiguous()), I, D, _ptr(out), ld, _stream(item_emb.device)),
              "recad_transpose_items")
    return out


def _eval_outputs(n, T, K, dev):
    return (torch.empty((n, K), dtype=torch.int32, device=dev), torch.empty((n, K), dtype=torch.float32, device=dev),
            torch.empty((n, max(T, 1)), dtype=torch.int32, device=dev), torch.empty((n, max(T, 1)), dtype=torch.float32, device=dev))


EVAL_PRECISION = os.environ.get("RECAD_EVAL_PRECISION", "tf32x3")   # "tf32x3" (tensor cores) | "exact" (fp32 FMA chain)


def fullrank_eval(user_emb, item_emb, user_ids, train_rowptr, train_col, targets, K, item_T=None, item_bias=None,
                  precision=None):
    """Fused score + mask + top-K + target rank (normal.py:57-93 without the score matrix).
    score(u, i) = <user_emb[u], item_emb[i]> (+ item_bias[i]).  Returns (topk_idx, topk_val, target_rank,
    target_score).  precision "tf32x3" (the name is kept for RECAD_EVAL_PRECISION and existing callers): tcgen05
    tensor-core kernel, three-pass split, ~2^-21 accuracy (power-of-two scaled fp16 hi / lo operands; needs D <= 64,
    K <= 32; ranks may differ from "exact" between near-tied items only); "exact": CUDA-core kernel whose scores are
    the bit-exact ascending-d FMA chain."""
    _need_cuda(user_emb, item_emb, user_ids, train_rowptr, train_col, item_bias)
    dev = user_emb.device
    I, D = item_emb.shape
    targets_t = torch.as_tensor(list(targets), dtype=torch.int32, device=dev)
    T = int(targets_t.numel())
    if T and (int(targets_t.min()) < 0 or int(targets_t.max()) >= I):
        raise RecadError(f"target item id out of range [0, {I})")
    n = int(user_ids.numel())
    topi, topv, trank, tscore = _eval_outputs(n, T, K, dev)
    precision = precision or EVAL_PRECISION
    if precision not in ("tf32x3", "exact"):
        raise RecadError(f"unknown evaluation precision {precision!r}")
    if precision == "tf32x3" and D <= 64 and K <= 32:
        L = _lib.lib()
        nfl = L.recad_fullrank_tc_scratch_floats(n, I)
        with torch.cuda.device(dev):
            scratch = torch.empty(nfl, dtype=torch.float32, device=dev)
            check(L.recad_fullrank_eval_tc(_ptr(user_emb.contiguous()), _ptr(item_emb.contiguous()), I, D,
                                           _ptr(user_ids.contiguous().long()), n, _ptr(train_rowptr), _ptr(train_col),
                                           _ptr(targets_t), T, K, _ptr(item_bias), _ptr(topi), _ptr(topv), _ptr(trank),
                                           _ptr(tscore), _ptr(scratch), nfl, _stream(dev)), "recad_fullrank_eval_tc")
        return topi, topv, trank[:, :T], tscore[:, :T]
    if item_bias is not None:        # exact kernel: the bias rides along as one more embedding dimension
        user_emb = torch.cat([user_emb, torch.ones((user_emb.shape[0], 1), device=dev)], 1)
        item_emb = torch.cat([item_emb, item_bias.view(-1, 1)], 1)
        D, item_T = D + 1, None
    if item_T is None:
        item_T = transpose_items(item_emb)
    with torch.cuda.device(dev):
        check(_lib.lib().recad_fullrank_eval(_ptr(user_emb.contiguous()), _ptr(item_T), item_T.shape[1], I, D,
                                             _ptr(user_ids.contiguous().long()), n, _ptr(train_rowptr), _ptr(train_col),
                                             _ptr(targets_t), T, K, _ptr(topi), _ptr(topv), _ptr(trank), _ptr(tscore),
                                             _stream(dev)), "recad_fullrank_eval")
    return topi, topv, trank[:, :T], tscore[:, :T]


def rank_from_scores(scores, user_ids, train_rowptr, train_col, targets, K):
    _need_cuda(scores, user_ids, train_rowptr, train_col)
    dev = scores.device
    n, I = scores.shape
    targets_t = torch.as_tensor(list(targets), dtype=torch.int32, device=dev)
    T = int(targets_t.numel())
    if T and (int(targets_t.min()) < 0 or int(targets_t.max()) >= I):
        raise RecadError(f"target item id out of range [0, {I})")
    topi, topv, trank, tscore = _eval_outputs(n, T, K, dev)
    with torch.cuda.device(dev):
        check(_lib.lib().recad_rank_from_scores(_ptr(scores.contiguous()), n, I, _ptr(user_ids.contiguous().long()),
                                                _ptr(train_rowptr), _ptr(train_col), _ptr(targets_t), T, K, _ptr(topi),
                                                _ptr(topv), _ptr(trank), _ptr(tscore), _stream(dev)), "recad_rank_from_scores")
    return topi, topv, trank[:, :T], tscore[:, :T]


def eligible_users(train_rowptr, train_col, n_users, n_items, targets, is_key=None):
    """Candidate users of the evaluation (normal.py:133-143) as an ascending int64 device tensor."""
    _need_cuda(train_rowptr, train_col, is_key)
    dev = train_rowptr.device
    L = _lib.lib()
    with torch.cuda.device(dev):
        t = torch.as_tensor(list(targets), dtype=torch.int32, device=dev)
        out = torch.empty(n_users, dtype=torch.int64, device=dev)
        nbytes = L.recad_eligible_users_scratch_bytes(n_users)
        scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        n = C.c_int64()
        check(L.recad_eligible_users(_ptr(train_rowptr), _ptr(train_col), n_users, n_items, _ptr(t), int(t.numel()), _ptr(is_key),
                                     _ptr(out), C.byref(n), _ptr(scratch), nbytes, _stream(dev)), "recad_eligible_users")
    return out[:n.value]


def recall_ndcg(topk_idx, user_ids, gt_rowptr, gt_col):
    """Sums of Recall@K / NDCG@K and the number of users with ground truth."""
    _need_cuda(topk_idx, user_ids, gt_rowptr, gt_col)
    out = torch.zeros(3, dtype=torch.float64, device=topk_idx.device)
    with torch.cuda.device(topk_idx.device):
        check(_lib.lib().recad_recall_ndcg(_ptr(topk_idx), topk_idx.shape[0], topk_idx.shape[1], _ptr(user_ids.contiguous().long()),
                                           _ptr(gt_rowptr), _ptr(gt_col), _ptr(out), _stream(topk_idx.device)), "recad_recall_ndcg")
    return out


# --------------------------------------------------------------------------- #
# samplers (host; advance numpy's legacy global MT19937 state in place)
# --------------------------------------------------------------------------- #
def _np_state():
    st = np.random.get_state()
    if st[0] != "MT19937":
        raise RecadError("np.random global state is not MT19937")
    return st, np.ascontiguousarray(st[1], dtype=np.uint32).copy(), [int(st[2])]


def _np_state_commit(st, key, pos):
    np.random.set_state((st[0], key, int(pos[0]), st[3], st[4]))


def _np(a, dtype=np.int64):
    return np.ascontiguousarray(a, dtype=dtype)


# *_raw: explicit MT19937 state -- key: uint32[624] (advanced in place), pos: one-element list.
# The ctypes calls release the GIL, so a raw sampler can run on a background thread.
def mt_pairwise_raw(key, pos, n_users, n_items, train_size, allpos_rowptr, allpos_col, out=None):
    """pairwise_sample (implicit.py:50-74) as int64 rows (user, positive, negative).  A large epoch is drawn by
    mt_pairwise_soa_raw and its positive items are gathered here; any other by the plain sampler."""
    rp, col = _np(allpos_rowptr), _np(allpos_col, np.int32)
    if out is None:
        out = np.empty((max(train_size, 1), 3), dtype=np.int64)
    assert out.dtype == np.int64 and out.flags.c_contiguous and out.shape[0] >= train_size
    if fits_soa_sampler(n_users, n_items, train_size):
        users, rel, negs = (host_empty(train_size, np.uint32) for _ in range(3))
        m = mt_pairwise_soa_raw(key, pos, n_users, n_items, train_size, rp, col, users, rel, negs)
        out[:m, 0] = users[:m]
        out[:m, 1] = col[rp[users[:m]] + rel[:m]]
        out[:m, 2] = negs[:m]
        return out[:m]
    n_out, cpos = C.c_int64(), C.c_int32(pos[0])
    check(_lib.lib().recad_mt19937_pairwise(key.ctypes.data, C.byref(cpos), n_users, n_items, train_size, rp.ctypes.data,
                                            col.ctypes.data, out.ctypes.data, C.byref(n_out)), "recad_mt19937_pairwise")
    pos[0] = cpos.value
    return out[:n_out.value]


def mt_pairwise_soa_raw(key, pos, n_users, n_items, train_size, allpos_rowptr, allpos_col, users, rel, negs, j_out=None):
    """The large-epoch sampler (csrc/sampler.cpp, recad_mt19937_pairwise_soa): same samples and stream consumption as
    mt_pairwise_raw (+ mt_permutation_draw_raw when j_out is given), written as three uint32 arrays
    (user, index of the positive inside the user's row, negative).  -> number of samples."""
    rp, col = _np(allpos_rowptr), _np(allpos_col, np.int32)
    for a in (users, rel, negs) + ((j_out,) if j_out is not None else ()):
        assert a.dtype == np.uint32 and a.flags.c_contiguous and a.shape[0] >= train_size
    filt, ext = pairwise_filter(rp, col, n_users)
    n_out, cpos = C.c_int64(), C.c_int32(pos[0])
    check(_lib.lib().recad_mt19937_pairwise_soa(key.ctypes.data, C.byref(cpos), n_users, n_items, train_size, rp.ctypes.data,
                                                col.ctypes.data, filt.ctypes.data, ext.ctypes.data, min(os.cpu_count() or 1, 32),
                                                users.ctypes.data, rel.ctypes.data, negs.ctypes.data, C.byref(n_out),
                                                j_out.ctypes.data if j_out is not None else None), "recad_mt19937_pairwise_soa")
    pos[0] = cpos.value
    return n_out.value


def permutation_apply32(j, out):
    n = int(j.shape[0])
    assert out.dtype == np.int32 and out.flags.c_contiguous and out.shape[0] >= n
    check(_lib.lib().recad_permutation_apply32(n, j.ctypes.data, out.ctypes.data), "recad_permutation_apply32")
    return out[:n]


def samples_expand(allpos_rowptr, allpos_col, users, rel, negs, rows):
    """rows[k] = (users[k], allpos_col[allpos_rowptr[users[k]] + rel[k]], negs[k]) on the device (int32 [n, 3])."""
    _need_cuda(allpos_rowptr, allpos_col, users, rel, negs, rows)
    n = int(users.shape[0])
    assert rows.dtype == torch.int32 and rows.shape[0] >= n and allpos_rowptr.dtype == torch.int64 and allpos_col.dtype == torch.int32
    with torch.cuda.device(rows.device):
        check(_lib.lib().recad_samples_expand(_ptr(allpos_rowptr), _ptr(allpos_col), _ptr(users), _ptr(rel), _ptr(negs), n,
                                              _ptr(rows), _stream(rows.device)), "recad_samples_expand")
    return rows


def host_empty(shape, dtype):
    """np.empty whose pages are requested as transparent huge pages (must be called before first touch)."""
    a = np.empty(shape, dtype=dtype)
    if a.nbytes >= (8 << 20):
        _lib.lib().recad_host_advise_huge(a.ctypes.data, a.nbytes)
    return a


def to_host(t, dtype=None):
    """Device tensor -> numpy array backed by huge pages (for arrays the samplers access at random)."""
    out = host_empty(tuple(t.shape), dtype or {torch.int64: np.int64, torch.int32: np.int32, torch.float32: np.float32}[t.dtype])
    torch.from_numpy(out).copy_(t)
    return out


FAST_SAMPLER_MIN = 1 << 20      # samples per epoch from which the filter-based parser pays off


def fits_soa_sampler(n_users, n_items, train_size):
    """Whether a pairwise epoch is drawn by mt_pairwise_soa_raw: large enough for its filter to pay off, and every id
    and count within the sampler's 32-bit arrays."""
    return FAST_SAMPLER_MIN <= train_size < (1 << 31) and n_users < (1 << 31) and n_items < (1 << 31)


class _DerivedCache:
    """Per-dataset host structures derived from the positives (filter blocks, sorted lists), keyed by the identity of
    the source arrays.  The entry keeps those arrays alive, so an address can never be reused by another dataset while
    its derived data is cached; a lock makes lookup-or-build atomic (the epochs of two datasets -- the clean one's
    speculative prefetch and the attacked one's first draw -- do run concurrently)."""

    def __init__(self, capacity):
        import threading
        from collections import OrderedDict
        self.capacity, self.lock, self.entries = capacity, threading.Lock(), OrderedDict()

    def get(self, key, keepalive, build):
        with self.lock:
            if key in self.entries:
                self.entries.move_to_end(key)
                return self.entries[key][0]
            value = build()
            self.entries[key] = (value, keepalive)
            while len(self.entries) > self.capacity:
                self.entries.popitem(last=False)
            return value


_filters = _DerivedCache(3)
_sorted_lists = _DerivedCache(4)


_filter_parents = {}     # (new col address, new rowptr address) -> (parent rowptr, parent col, parent n_users): injected datasets


def filter_parent_hint(new_rowptr, new_col, old_rowptr, old_col, n_users_old):
    """The positives (new_rowptr, new_col) are (old_rowptr, old_col) with rows APPENDED (dataset injection): the sampler's
    filter blocks of the old users can be copied instead of rebuilt."""
    if len(_filter_parents) > 8:
        _filter_parents.clear()
    _filter_parents[(new_col.ctypes.data, new_rowptr.ctypes.data)] = (old_rowptr, old_col, int(n_users_old))


def _filter_key(rowptr, col, n_users):
    return (col.ctypes.data, rowptr.ctypes.data, len(col), int(n_users))


def pairwise_filter(allpos_rowptr, allpos_col, n_users):
    """Per-user 128-byte blocks (row bounds + two-level membership filter, first line decisive) for mt_pairwise_soa_raw;
    built once per positives array -- or, for a dataset derived by injection from one whose blocks are still cached,
    copied from the parent and completed for the appended users only."""
    def build():
        filt = host_empty(int(n_users) * 16, np.uint64)
        ext = host_empty(max(len(allpos_col), 1), np.uint32)
        u_lo = 0
        parent = _filter_parents.pop((allpos_col.ctypes.data, allpos_rowptr.ctypes.data), None)
        if parent is not None:
            prp, pcol, pn = parent
            got = _filters.entries.get(_filter_key(prp, pcol, pn))        # build() runs under the cache's lock
            if got is not None and pn <= n_users:
                _filters.entries.move_to_end(_filter_key(prp, pcol, pn))    # a parent in use is not the eviction candidate
                (pf, pe), _ = got
                filt[:pn * 16] = pf[:pn * 16]
                ext[:len(pe)] = pe
                u_lo = pn
        check(_lib.lib().recad_pairwise_filter_build_range(allpos_rowptr.ctypes.data, allpos_col.ctypes.data, u_lo, n_users,
                                                           filt.ctypes.data, ext.ctypes.data, os.cpu_count() or 1),
              "recad_pairwise_filter_build_range")
        return filt, ext
    return _filters.get(_filter_key(allpos_rowptr, allpos_col, n_users), (allpos_rowptr, allpos_col), build)


def mt_pointwise_raw(key, pos, user_ids, pos_rowptr, pos_items, n_items, ratio, out=None):
    uid, rp, items = _np(user_ids), _np(pos_rowptr), _np(pos_items)

    def build():                                # once per dataset, not once per epoch (a 0.1 s lexsort at ml1m size)
        rows = np.repeat(np.arange(len(uid), dtype=np.int64), np.diff(rp))
        return items[np.lexsort((items, rows))]   # each user's list sorted ascending, lists kept in place
    srt = _sorted_lists.get((items.ctypes.data, rp.ctypes.data, len(items)), (items, rp), build)
    n = len(items) * (1 + ratio)
    if out is None:
        out = np.empty((max(n, 1), 3), dtype=np.int64)
    assert out.dtype == np.int64 and out.flags.c_contiguous and out.shape[0] >= n
    cpos = C.c_int32(pos[0])
    check(_lib.lib().recad_mt19937_pointwise(key.ctypes.data, C.byref(cpos), len(uid), uid.ctypes.data, rp.ctypes.data,
                                             items.ctypes.data, srt.ctypes.data, n_items, ratio, out.ctypes.data),
          "recad_mt19937_pointwise")
    pos[0] = cpos.value
    return out[:n]


def mt_permutation_raw(key, pos, n, out=None):
    perm = np.empty(max(n, 1), dtype=np.int64) if out is None else out
    assert perm.dtype == np.int64 and perm.flags.c_contiguous and perm.shape[0] >= n
    cpos = C.c_int32(pos[0])
    check(_lib.lib().recad_mt19937_permutation(key.ctypes.data, C.byref(cpos), n, perm.ctypes.data), "recad_mt19937_permutation")
    pos[0] = cpos.value
    return perm[:n]


def mt_permutation_draw_raw(key, pos, n, j_out=None):
    """The stream-consuming half of the shuffle: j[i] = random_interval(i), i = n-1 .. 1 (uint32 [n])."""
    j = host_empty(max(n, 1), np.uint32) if j_out is None else j_out
    assert j.dtype == np.uint32 and j.flags.c_contiguous and j.shape[0] >= n
    cpos = C.c_int32(pos[0])
    check(_lib.lib().recad_mt19937_permutation_draw(key.ctypes.data, C.byref(cpos), n, j.ctypes.data), "recad_mt19937_permutation_draw")
    pos[0] = cpos.value
    return j[:n]


def permutation_apply(j, out=None):
    """The generator-free half: perm = arange(n) with swap(perm[i], perm[j[i]]) applied for i = n-1 .. 1."""
    n = int(j.shape[0])
    perm = np.empty(max(n, 1), dtype=np.int64) if out is None else out
    assert perm.dtype == np.int64 and perm.flags.c_contiguous and perm.shape[0] >= n
    check(_lib.lib().recad_permutation_apply(n, j.ctypes.data, perm.ctypes.data), "recad_permutation_apply")
    return perm[:n]


def mt_pairwise(n_users, n_items, train_size, allpos_rowptr, allpos_col, out=None):
    """== pairwise_sample (implicit.py:50-74) on the global np.random stream."""
    st, key, pos = _np_state()
    S = mt_pairwise_raw(key, pos, n_users, n_items, train_size, allpos_rowptr, allpos_col, out)
    _np_state_commit(st, key, pos)
    return S


def mt_pointwise(user_ids, pos_rowptr, pos_items, n_items, ratio, out=None):
    """== pointwise_sample (implicit.py:77-91) on the global np.random stream."""
    st, key, pos = _np_state()
    S = mt_pointwise_raw(key, pos, user_ids, pos_rowptr, pos_items, n_items, ratio, out)
    _np_state_commit(st, key, pos)
    return S


def mt_permutation(n, out=None):
    """== np.random.shuffle(np.arange(n)) (implicit.py:24-25)."""
    st, key, pos = _np_state()
    perm = mt_permutation_raw(key, pos, n, out)
    _np_state_commit(st, key, pos)
    return perm
