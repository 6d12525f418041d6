"""User-row sharded LightGCN over torch.distributed: one process per GPU, NCCL over NVLink.

Partitioning (SURVEY.md 8e, "scheme B"): rank g owns the users [lo, hi).  It holds
  * the rows of its users of the normalised adjacency and the transposed block, stored as ONE local
    matrix over the local index space [own users ; ALL items]:   A_g = [[0, R_g], [R_g^T, 0]]
    (values use the GLOBAL degrees: the item degrees are all-reduced once at build time);
  * one table [U_g + I, D]: its user rows (+ Adam state) and a REPLICA of the item rows.
One local SpMM Y = A_g X then yields the rank's user rows (complete) and a PARTIAL sum for every item
row; the item block Y[U_g:] (I x D floats, 51 MB at I = 200 k) is all-reduced -- the only exchange of a
layer.  BPR rows go to the owner of their user; the item block of the gradient (and of the batch
multiplicities) is all-reduced once per batch; Adam then updates the user rows locally and the item
replica identically on every rank.  Evaluation shards the users and exchanges nothing but metric sums.
Results equal the single-GPU path up to fp32 summation order.
"""
import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from . import _lib, ops


def user_range(n_users, rank, world):
    """Contiguous, balanced split of [0, n_users)."""
    base, rem = divmod(int(n_users), int(world))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def route_epoch(samples, perm, batch, lo, hi):
    """Rows of every GLOBAL batch whose user lives in [lo, hi), in batch order.
    samples int64 [n, 3] (sampler order), perm int64 [n] (epoch shuffle) -> (local rows int64 [m, 3] with
    LOCAL user ids, batch_ptr python list [n_batches + 1])."""
    S = samples[perm]
    n = int(S.shape[0])
    n_batches = (n + batch - 1) // batch
    idx = torch.nonzero((S[:, 0] >= lo) & (S[:, 0] < hi)).flatten()
    local = S[idx].contiguous()
    local[:, 0] -= lo
    counts = torch.bincount(idx // batch, minlength=n_batches)
    ptr = [0] + torch.cumsum(counts, 0).cpu().tolist()
    return local, ptr


class _PeerBlock:
    """Peer-memory plumbing of the C-driven sharded epoch (csrc/shard.cu): ONE NVLink-mapped symmetric block per rank
    (torch symmetric memory) holding every buffer a peer reads or writes -- the layer buffers X0 / X1, the propagated
    mean O, the gradient g (each [n_max, D]), the batch multiplicities cnt [n_max], the staging slots
    [2, world, slice, D] (slot s receives rank s's partial rows of the items this rank owns, slice = ceil(I / world)) and
    the barrier pad -- at the same byte offsets on every rank."""

    def __init__(self, Ug, I, D, dev, group):
        import os
        import torch.distributed._symmetric_memory as symm
        self.group = group if group is not None else dist.group.WORLD
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        if self.world > 16:
            raise ops.RecadError("the peer-memory exchange supports at most 16 ranks")
        ugs = torch.zeros(self.world, dtype=torch.int64, device=dev)
        ugs[self.rank] = Ug
        dist.all_reduce(ugs, group=group)
        self.Ugs = [int(x) for x in ugs.tolist()]
        self.I, self.D, self.dev = I, D, dev
        self.slice = (I + self.world - 1) // self.world
        n_max = max(self.Ugs) + I
        al = lambda x: (x + 255) // 256 * 256     # noqa: E731
        off, self.off = 0, {}
        for name, nbytes in (("X0", n_max * D * 4), ("X1", n_max * D * 4), ("O", n_max * D * 4), ("g", n_max * D * 4),
                             ("cnt", n_max * 4), ("stage", 2 * self.world * self.slice * D * 4), ("signal", 256)):
            self.off[name] = off
            off = al(off + nbytes)
        self.block = symm.empty((off,), dtype=torch.uint8, device=dev)
        self.block.zero_()
        self.handle = symm.rendezvous(self.block, self.group)
        self.handle.barrier(channel=0)                 # every pad is zero before anybody signals
        self.peer_base = (C.c_void_p * self.world)(*[int(p) for p in self.handle.buffer_ptrs])
        self.peer_users = (C.c_int64 * self.world)(*self.Ugs)
        mc = int(getattr(self.handle, "multicast_ptr", 0) or 0)
        self.multicast = bool(len(set(self.Ugs)) == 1 and mc and os.environ.get("RECAD_DIST_MULTICAST", "1") != "0")
        self.mc_base = mc if self.multicast else None

    def view(self, name, rows, cols=None):
        n = rows * (cols or 1) * 4
        t = self.block[self.off[name]:self.off[name] + n].view(torch.float32)
        return t.view(rows, cols) if cols else t


class ShardedLightGCN:
    def __init__(self, n_users, n_items, edges, D=64, n_layers=3, lam=1e-4, lr=1e-3, batch=1024, device=None,
                 init_user=None, init_item=None, group=None, graph=None, bounds=None, fused=None):
        """edges: (users, items) int64 CUDA tensors of the GLOBAL edge list (every rank passes the same), or
        None with `graph` = this rank's prebuilt local matrix and `bounds` = its user range (inject())."""
        self.group = group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.dev = torch.device(device)
        self.U, self.I, self.D, self.L, self.lam, self.lr, self.batch = int(n_users), int(n_items), D, n_layers, lam, lr, batch
        self.lo, self.hi = bounds if bounds is not None else user_range(n_users, self.rank, self.world)
        self.Ug = self.hi - self.lo
        Ug = self.Ug
        if graph is None:
            eu, ei = edges
            mine = (eu >= self.lo) & (eu < self.hi)

            def complete_item_degrees(degree):        # users' degrees are complete locally, items' are partial
                block = degree[Ug:].clone()
                dist.all_reduce(block, group=group)
                degree[Ug:] = block
            graph = ops.Graph.from_edges((eu[mine] - self.lo).contiguous(), ei[mine].contiguous(), Ug, self.I,
                                         degree_hook=complete_item_degrees)
        self.graph = graph
        # the same matrix as two row blocks, so that the item rows (whose result must be all-reduced) can be
        # multiplied FIRST and their all-reduce overlapped with the multiplication of the user rows
        g = self.graph
        nnz_u = int(g.rowptr[Ug])
        self.g_user = ops.Graph.from_csr(g.rowptr[:Ug + 1], g.colidx[:nnz_u] - Ug, g.vals[:nnz_u], n_cols=self.I)
        self.g_item = ops.Graph.from_csr(g.rowptr[Ug:] - nnz_u, g.colidx[nnz_u:], g.vals[nnz_u:], n_cols=Ug)
        self.overlap = True
        N = Ug + self.I
        with torch.cuda.device(self.dev):
            self.E = torch.empty((N, D), dtype=torch.float32, device=self.dev)
            if init_user is None:                     # N(0, 0.1) like lightgcn.py:52-53; same item replica on every rank
                gen = torch.Generator(device=self.dev).manual_seed(2023)
                init_item = torch.randn(self.I, D, device=self.dev, generator=gen) * 0.1
                gen.manual_seed(2024 + self.rank)
                self.E[:Ug].copy_(torch.randn(Ug, D, device=self.dev, generator=gen) * 0.1)
            else:
                self.E[:Ug].copy_(init_user[self.lo:self.hi])
            self.E[Ug:].copy_(init_item)
            self.m, self.v = torch.zeros_like(self.E), torch.zeros_like(self.E)
            self.peer = self._make_peer(fused)
            if self.peer is not None:                 # everything a peer touches lives in the NVLink-mapped block
                self.X0, self.X1, self.O, self.g = (self.peer.view(k, N, D) for k in ("X0", "X1", "O", "g"))
                self.cnt = self.peer.view("cnt", N)
            else:
                self.O, self.g = torch.empty_like(self.E), torch.empty_like(self.E)
                self.X0, self.X1 = torch.empty_like(self.E), torch.empty_like(self.E)
                self.cnt = torch.empty(N, dtype=torch.float32, device=self.dev)
            self.loss_acc = torch.zeros(4, dtype=torch.float64, device=self.dev)
            self._st = self._shard_struct() if self.peer is not None else None
        self.steps = 0
        self._O_valid = False
        self.n_allreduce = 0
        self.n_fused = 0

    def _make_peer(self, fused):
        """fused=None: use the peer-memory exchange when every rank can set it up (RECAD_DIST_FUSED=0 disables);
        True: require it; False: NCCL all-reduce."""
        import os
        if fused is None and os.environ.get("RECAD_DIST_FUSED", "1") == "0":
            fused = False
        if fused is False or self.world == 1 or self.D not in (32, 64, 128) or self.L < 1:
            return None
        peer, err = None, None
        try:
            peer = _PeerBlock(self.Ug, self.I, self.D, self.dev, self.group)
        except Exception as e:   # noqa: BLE001 -- no symmetric memory on this system
            err = e
        ok = torch.tensor([0 if peer is None else 1], device=self.dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)
        if int(ok.item()) == 0:
            if fused:
                raise ops.RecadError(f"fused exchange requested but symmetric memory is unavailable: {err}")
            return None
        return peer

    # ------------------------------------------------------------------ C-driven path (csrc/shard.cu)
    def _shard_struct(self):
        p, g = self.peer, self.graph
        st = _lib.LightGCNShard()
        st.rank, st.world, st.D, st.n_layers = self.rank, self.world, self.D, self.L
        st.n_users_local, st.n_items, st.user_lo, st.slice = self.Ug, self.I, self.lo, p.slice
        st.lam, st.lr, st.beta1, st.beta2, st.eps = self.lam, self.lr, 0.9, 0.999, 1e-8
        self._csr_user, self._csr_item = self.g_user.struct(self.D), self.g_item.struct(self.D)
        st.g_user, st.g_item = C.pointer(self._csr_user), C.pointer(self._csr_item)
        # the rank's own users' sorted distinct items = its user rows of the matrix (columns carry the Ug offset)
        st.pos_rowptr, st.pos_col, st.pos_col_offset = g.rowptr.data_ptr(), g.colidx.data_ptr(), self.Ug
        st.E, st.m, st.v, st.loss_acc = self.E.data_ptr(), self.m.data_ptr(), self.v.data_ptr(), self.loss_acc.data_ptr()
        st.peer_base, st.mc_base, st.peer_users = p.peer_base, p.mc_base, p.peer_users
        for k in ("X0", "X1", "O", "g", "cnt", "stage", "signal"):
            setattr(st, "off_" + k, p.off[k])
        return st

    def _check_barriers(self):
        state = (C.c_uint32 * 2)()
        with torch.cuda.device(self.dev):
            _lib.check(_lib.lib().recad_lightgcn_shard_barrier_state(C.byref(self._st), state, ops._stream(self.dev)), "barrier_state")
        if state[1]:
            raise ops.RecadError("ShardedLightGCN: a cross-device barrier timed out (a peer rank never arrived)")

    def _epoch_c(self, ep, n, trace=None):
        """The whole epoch enqueued by ONE call: no collective library, no host synchronisation inside."""
        n_batches = (n + self.batch - 1) // self.batch
        tr = (C.c_double * 8)() if trace is not None else None
        with torch.cuda.device(self.dev):
            _lib.check(_lib.lib().recad_lightgcn_shard_train_epoch(C.byref(self._st), C.byref(ep), self.batch, self.steps, tr,
                                                                   ops._stream(self.dev)), "recad_lightgcn_shard_train_epoch")
        self.steps += n_batches
        self.n_fused += n_batches * (2 * self.L + 1)
        self._O_valid = False
        if trace is not None:
            trace.update(dict(zip(("item_spmm_push", "user_spmm", "barriers", "slice_reduce_store", "zeroing", "bpr",
                                   "gradient_exchange", "adam"), [round(float(x), 3) for x in tr])))
        # [2] = this rank's part of the sum of batch losses, [3] = out-of-range flag (an int in the slot's bits)
        out = torch.stack([self.loss_acc[2], (self.loss_acc[3:4].view(torch.int64) != 0).double()[0]])
        dist.all_reduce(out, group=self.group)                   # ONE collective per epoch
        loss, bad = out.tolist()
        if bad:
            raise ops.RecadError("ShardedLightGCN.train_epoch: a sample id is out of range")
        self._check_barriers()
        return loss / n_batches

    def train_epoch_soa(self, users, rel, negs, perm=None, trace=None):
        """One epoch from the host sampler's 32-bit arrays (GLOBAL user id, index of the positive inside the user's row,
        negative; recad_mt19937_pairwise_soa) + the int32 epoch permutation, every rank holding the whole epoch."""
        if self._st is None:
            raise ops.RecadError("train_epoch_soa needs the peer-memory path (symmetric memory)")
        ep = _lib.EpochSamples()
        ep.n_samples = int(users.numel())
        ep.users, ep.rel, ep.negs = users.data_ptr(), rel.data_ptr(), negs.data_ptr()
        ep.perm32 = perm.data_ptr() if perm is not None else None
        assert users.dtype == rel.dtype == negs.dtype == torch.int32 and (perm is None or perm.dtype == torch.int32)
        return self._epoch_c(ep, ep.n_samples, trace)

    # ------------------------------------------------------------------ pieces (NCCL path)
    def _allreduce_items(self, t):
        dist.all_reduce(t[self.Ug:], group=self.group)          # contiguous [I, D] (or [I]) block, in place
        self.n_allreduce += 1

    def _spmm_exchange(self, x, y):
        """y = A_g x with the item block of y summed over ranks (NCCL)."""
        Ug = self.Ug
        if not self.overlap:
            ops.spmm(self.graph, x, y)
            self._allreduce_items(y)
            return
        ops.spmm(self.g_item, x[:Ug], y[Ug:])                       # partial item rows (gathers own users)
        work = dist.all_reduce(y[Ug:], group=self.group, async_op=True)
        self.n_allreduce += 1
        ops.spmm(self.g_user, x[Ug:], y[:Ug])                       # own user rows (gathers the item replica)
        work.wait()

    def propagate(self):
        """O = mean_k A^k E (lightgcn.py:82-113), L local SpMMs + L exchanges of the item block."""
        L = self.L
        if self._st is not None:
            with torch.cuda.device(self.dev):
                _lib.check(_lib.lib().recad_lightgcn_shard_propagate(C.byref(self._st), ops._stream(self.dev)),
                           "recad_lightgcn_shard_propagate")
            self.n_fused += L
            self._O_valid = True
            return self.O[:self.Ug], self.O[self.Ug:]
        if L == 0:
            self.O.copy_(self.E)
        x = self.E
        for k in range(L):
            y = self.X1 if k & 1 else self.X0
            self._spmm_exchange(x, y)
            s = 1.0 / (L + 1) if k == L - 1 else 1.0
            ops.axpby(self.O, s, self.E if k == 0 else self.O, s, y)
            x = y
        self._O_valid = True
        return self.O[:self.Ug], self.O[self.Ug:]

    def train_epoch(self, samples, perm=None, trace=None):
        """One epoch (lightgcn.py:132-172) over the GLOBAL sample list (int64 [n, 3] rows of GLOBAL ids, perm int64 [n]);
        returns the mean batch loss."""
        n = int(samples.shape[0])
        if self._st is not None:
            ep = _lib.EpochSamples()
            ep.n_samples, ep.rows = n, samples.data_ptr()
            ep.perm64 = perm.data_ptr() if perm is not None else None
            assert samples.dtype == torch.int64 and samples.is_contiguous() and (perm is None or perm.dtype == torch.int64)
            return self._epoch_c(ep, n, trace)
        if perm is None:
            perm = torch.arange(samples.shape[0], device=samples.device)
        local, ptr = route_epoch(samples, perm, self.batch, self.lo, self.hi)
        n_batches = len(ptr) - 1
        B_of = [min(self.batch, n - b * self.batch) for b in range(n_batches)]
        parts = torch.zeros((n_batches, 2), dtype=torch.float64, device=self.dev)
        L = self.L
        self.loss_acc.zero_()
        for b in range(n_batches):
            self.steps += 1
            self.propagate()
            self.g.zero_()
            self.cnt.zero_()
            self.loss_acc[:2].zero_()                # [3] keeps the out-of-range flag of the whole epoch
            rows = local[ptr[b]:ptr[b + 1]]
            if rows.shape[0]:
                ops.bpr_fwd_bwd(self.O, self.E, self.Ug, self.I, rows, None, 1.0 / (L + 1), self.g, self.cnt, self.loss_acc,
                                B_norm=B_of[b])
            parts[b].copy_(self.loss_acc[:2])
            self._allreduce_items(self.g)
            self._allreduce_items(self.cnt)
            t = self.g
            for k in range(L):                       # Horner: t <- g + A t
                y = self.X1 if k & 1 else self.X0
                self._spmm_exchange(t, y)
                ops.axpby(y, 1.0, self.g, 1.0, y)
                t = y
            ops.adam(self.E, t, self.m, self.v, self.steps, lr=self.lr, cnt=self.cnt, reg_scale=self.lam / B_of[b])
        self._O_valid = False
        bad = self.loss_acc[3:4].view(torch.int64).clone()
        dist.all_reduce(parts, group=self.group)
        dist.all_reduce(bad, group=self.group)
        if int(bad.item()):
            raise ops.RecadError("ShardedLightGCN.train_epoch: a sample id is out of range")
        p = parts.cpu().numpy()
        Bs = np.asarray(B_of, dtype=np.float64)
        return float(np.mean(p[:, 0] / Bs + self.lam * 0.5 * p[:, 1] / Bs))

    def full_rank(self, targets, K=20, users_local=None):
        """Fused evaluation of this rank's users (no exchange): outputs for users lo + users_local."""
        if not self._O_valid:
            self.propagate()
        Ug = self.Ug
        uid = torch.arange(Ug, device=self.dev) if users_local is None else users_local
        if getattr(self, "_eval_csr", None) is None:        # the users' train rows = the mask of the evaluation; built once
            rowptr = self.graph.rowptr[:Ug + 1].contiguous()
            self._eval_csr = (rowptr, (self.graph.colidx[:int(rowptr[-1])] - Ug).contiguous())
        rowptr, col = self._eval_csr
        return ops.fullrank_eval(self.O[:Ug], self.O[Ug:], uid, rowptr, col, targets, K)

    def gather_tables(self):
        """(user table [U, D], item table [I, D]) assembled on every rank (tests / checkpoints)."""
        sizes = torch.zeros(self.world, dtype=torch.int64, device=self.dev)
        sizes[self.rank] = self.Ug
        dist.all_reduce(sizes, group=self.group)
        parts = [torch.empty((int(n), self.D), dtype=torch.float32, device=self.dev) for n in sizes.tolist()]
        dist.all_gather(parts, self.E[:self.Ug].contiguous(), group=self.group)
        return torch.cat(parts), self.E[self.Ug:].clone()

    def inject(self, fake_rowptr, fake_items, init_user=None, init_item=None):
        """The attacked model of normal.py:198-206 on the sharded path: a NEW, freshly initialised model
        over U + F users.  The fake users' rows are appended to the LAST rank's shard (no re-sort); every
        rank knows the fake rows, adds their item counts to its copy of the global item degrees and
        re-normalises its values -- no exchange at all.
        fake_rowptr int64 [F + 1], fake_items int32 (ascending, distinct per row): identical on every rank."""
        fake_rowptr = torch.as_tensor(fake_rowptr).to(self.dev, torch.int64)
        fake_items = torch.as_tensor(fake_items).to(self.dev, torch.int32)
        F = int(fake_rowptr.numel()) - 1
        delta = torch.bincount(fake_items.long(), minlength=self.I).to(torch.int32)
        item_degree = self.graph.degree[self.Ug:] + delta
        last = self.rank == self.world - 1
        if last:
            def complete(degree):
                degree[self.Ug + F:] = item_degree
            graph = self.graph.append_users(self.Ug, self.I, fake_rowptr, fake_items, degree_hook=complete)
        else:
            degree = self.graph.degree.clone()
            degree[self.Ug:] = item_degree
            graph = self.graph.renormalized(degree)
        bounds = (self.lo, self.hi + F) if last else (self.lo, self.hi)
        return ShardedLightGCN(self.U + F, self.I, None, D=self.D, n_layers=self.L, lam=self.lam, lr=self.lr, batch=self.batch,
                               device=self.dev, init_user=init_user, init_item=init_item, group=self.group, graph=graph,
                               bounds=bounds, fused=self.peer is not None)


def batch_rows(perm, b0, B, rank, world):
    """This rank's rows of the global batch perm[b0 : b0 + B]: every world-th row starting at `rank`
    (an even split whatever the user ids are; any split gives the same sum)."""
    return perm[b0 + rank:b0 + B:world].contiguous()


class DataParallelVictim:
    """Plain data parallelism for the pointwise victims (MF, NCF; SURVEY.md 8e): every rank holds a full
    replica (same seed -> same init), takes every world-th row of each global batch, computes its part of
    the batch gradient with the 1/B of the GLOBAL batch (recad_mf_grad / recad_ncf_grad), the flat gradient
    is all-reduced over NCCL and every rank applies the same dense Adam step (recad_adam).  Equal to the
    single-GPU epoch up to fp32 summation order."""

    def __init__(self, victim, group=None):
        from .victim.mf import MF
        from .victim.ncf import NCF
        if not isinstance(victim, (MF, NCF)):
            raise TypeError("DataParallelVictim wraps an instantiated recad_b200 MF or NCF victim")
        victim._require_instance("DataParallelVictim")
        self.victim, self.group = victim, group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self._grad = _lib.lib().recad_mf_grad if isinstance(victim, MF) else _lib.lib().recad_ncf_grad
        self._name = "recad_mf_grad" if isinstance(victim, MF) else "recad_ncf_grad"
        # replicas must start identical: rank 0's tables win (a no-op when every rank used the same seed)
        dist.broadcast(victim.flat, 0, group=group)
        self.n_allreduce = 0

    def train_epoch(self, samples, perm=None, batch=None):
        """One epoch over the GLOBAL (samples [n, 3] int64 = user, item, label; perm [n]) on the device;
        returns the mean batch loss (mf.py:49-69 / ncf.py:131-153)."""
        v = self.victim
        dev = v._dev
        n = int(samples.shape[0])
        if perm is None:
            perm = torch.arange(n, device=dev)
        B = int(batch or (v.dataset.config["pointwise_batch_size"] if hasattr(v.dataset, "config") else 1024))
        n_batches = (n + B - 1) // B
        parts = torch.zeros(n_batches, dtype=torch.float64, device=dev)
        cfg = v.config
        with torch.cuda.device(dev):
            v.loss_acc.zero_()
            for b in range(n_batches):
                b0 = b * B
                Bg = min(B, n - b0)
                rows = batch_rows(perm, b0, Bg, self.rank, self.world)
                v.loss_acc[0:1].zero_()                 # [3] keeps the out-of-range flag of the whole epoch
                _lib.check(self._grad(C.byref(v._st), v._vp(samples), v._vp(rows) if rows.numel() else None, int(rows.numel()), Bg,
                                      ops._stream(dev)), self._name)
                parts[b] = v.loss_acc[0] / Bg
                dist.all_reduce(v.g, group=self.group)
                self.n_allreduce += 1
                v._steps += 1
                ops.adam(v.flat, v.g, v.m, v.v, v._steps, lr=cfg["lr"])
            bad = v.loss_acc[3:4].view(torch.int64).clone()
            dist.all_reduce(parts, group=self.group)
            dist.all_reduce(bad, group=self.group)
        if int(bad.item()):
            raise ops.RecadError("DataParallelVictim.train_epoch: a sample id is out of range")
        return float(parts.mean().item())


class _Rank0Epochs:
    """The slice of the dataset interface dataset._EpochPipe needs, over rank 0's host copy of the positives: lets the
    sharded bench draw epochs with the same background pipeline as the single-GPU path."""

    def __init__(self, n_users, n_items, allpos_rowptr, allpos_col):
        from .dataset import ImplicitData
        self.config = {"prefetch": True, "sample": "pairwise", "negative_ratio": 4}
        self.n_users, self.n_items, self.traindataSize = int(n_users), int(n_items), int(len(allpos_col))
        self._allpos = (allpos_rowptr, allpos_col)
        self._draw_samples = ImplicitData._draw_samples.__get__(self)


# ---------------------------------------------------------------------------------------------- bench.py --gpus N
def parity_check(dev, rank, world):
    """Small-graph epoch + evaluation on the sharded path against the single-GPU path (rank 0), before anything is timed."""
    from . import dataset, model, synthetic
    U, I, E, D, L, B, n = 6000, 1500, 90_000, 64, 3, 8192, 40_000
    u, i = synthetic.make_edges(U, I, E, seed=5)
    eu, ei = torch.as_tensor(u, device=dev), torch.as_tensor(i, device=dev)
    g = torch.Generator().manual_seed(7)
    init_u, init_i = torch.randn(U, D, generator=g) * 0.1, torch.randn(I, D, generator=g) * 0.1
    samples = torch.stack([torch.randint(0, U, (n,), generator=g), torch.randint(0, I, (n,), generator=g),
                           torch.randint(0, I, (n,), generator=g)], 1).to(dev)
    perm = torch.randperm(n, generator=g).to(dev)
    m = ShardedLightGCN(U, I, (eu, ei), D=D, n_layers=L, batch=B, device=dev, init_user=init_u.to(dev), init_item=init_i.to(dev))
    losses = [m.train_epoch(samples, perm) for _ in range(2)]
    tu, ti = m.gather_tables()
    res = torch.zeros(4, dtype=torch.float64, device=dev)
    if rank == 0:
        data = dataset.ArrayImplicitData("parity", U, I, (eu, ei), dev, batch_size=B, prefetch=False)
        ref = model.from_config("victim", "lightgcn", latent_dim_rec=D, lightGCN_n_layers=L, device=dev).I(dataset=data)
        ref.embedding_user.weight.data.copy_(init_u)
        ref.embedding_item.weight.data.copy_(init_i)
        data.epoch_samples = lambda device=None: (samples, perm)
        ref_losses = [ref.train_step()[0] for _ in range(2)]
        rel = lambda a, b: float(((a - b).abs() / (b.abs() + 2e-2 * b.abs().max())).max())     # noqa: E731
        res[0] = max(abs(a - b) / abs(b) for a, b in zip(losses, ref_losses))
        res[1], res[2] = rel(tu, ref.embedding_user.weight), rel(ti, ref.embedding_item.weight)
        res[3] = 1.0 if (res[0] <= 1e-5 and res[1] <= 1e-4 and res[2] <= 1e-4) else 0.0
    dist.broadcast(res, 0)
    out = {"parity_checked": bool(res[3].item()), "loss_rel_err": float(res[0]), "user_table_rel_err": float(res[1]),
           "item_table_rel_err": float(res[2]), "path": "peer-memory C driver" if m.peer is not None else "NCCL",
           "case": f"{U} users x {I} items x {E} edges, 2 epochs of {n} samples (batch {B}) vs the single-GPU path on rank 0"}
    del m
    return out


def bench_sharded(args, w, dev, rank, world, metric, synth_edges, ClockSampler, peaks, workload):
    import time
    U, I, D, L, B = w["n_users"], w["n_items"], w["D"], w["L"], args.batch or w["batch"]
    ev = lambda: torch.cuda.Event(enable_timing=True)     # noqa: E731
    parity = parity_check(dev, rank, world)
    if not parity["parity_checked"]:
        raise ops.RecadError(f"sharded path does not reproduce the single-GPU path: {parity}")
    eu, ei = synth_edges(w, dev)                           # same seed on every rank: identical global edge list
    torch.manual_seed(2023)
    init_u = (torch.randn(U, D) * 0.1)
    init_i = (torch.randn(I, D) * 0.1)
    t0 = time.time()
    m = ShardedLightGCN(U, I, (eu, ei), D=D, n_layers=L, batch=B, device=dev, init_user=init_u.to(dev), init_item=init_i.to(dev))
    torch.cuda.synchronize()
    t_graph = time.time() - t0
    if m.peer is None:
        raise ops.RecadError("bench --gpus N needs the peer-memory path (torch symmetric memory over NVLink)")
    # rank 0 draws the epoch with the exact MT19937 sampler (needs every user's positives) and broadcasts it:
    # four 32-bit arrays (user, index of the positive, negative, permutation), 16 bytes per sample
    n = int(eu.numel())
    epoch = torch.empty((4, n), dtype=torch.int32, device=dev)
    pipe = None
    if rank == 0:
        keys = torch.unique(eu * I + ei)
        ap_ptr = torch.zeros(U + 1, dtype=torch.int64, device=dev)
        ap_ptr[1:] = torch.cumsum(torch.bincount(keys // I, minlength=U), 0)
        ap = (ap_ptr.cpu().numpy(), (keys % I).int().cpu().numpy())
        del keys
        from .dataset import _EpochPipe
        np.random.seed(2023)
        pipe = _EpochPipe(_Rank0Epochs(U, I, *ap))
        pipe.raw_soa = True
    del eu, ei

    def fetch_epoch():                                      # host sampler -> pinned H2D (rank 0) -> NVLink broadcast
        if rank == 0:
            got = pipe.next(dev)
            assert len(got) == 4 and int(got[0].numel()) == n, "the synthetic graph has no user without positives"
            for k in range(4):
                epoch[k].copy_(got[k], non_blocking=True)
        dist.broadcast(epoch, 0)

    t0 = time.time()
    fetch_epoch()
    torch.cuda.synchronize()
    t_sampler = time.time() - t0
    n_batches = (n + B - 1) // B

    marks = []

    def step(trace=None):
        e0, e1, e2 = ev(), ev(), ev()
        e0.record()
        loss = m.train_epoch_soa(epoch[0], epoch[1], epoch[2], epoch[3], trace=trace)
        e1.record()
        topi, topv, rank_, score = m.full_rank([0], 20)
        hits = (rank_[:, 0] < 20).sum().double().view(1)
        dist.all_reduce(hits)
        e2.record()
        marks.append((e0, e1, e2))
        return loss, float(hits.item()) / U

    for _ in range(args.warmup):
        step()
    dist.barrier()
    torch.cuda.synchronize()
    a, b = ev(), ev()
    with ClockSampler(dev.index) as clocks:
        a.record()
        for _ in range(args.steps):
            loss, hr = step()
        b.record()
        torch.cuda.synchronize()
    dist.barrier()
    timed = marks[-args.steps:]
    ms = torch.tensor([a.elapsed_time(b) / args.steps, float(np.mean([x.elapsed_time(y) for x, y, _ in timed])),
                       float(np.mean([y.elapsed_time(z) for _, y, z in timed]))], dtype=torch.float64, device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)            # device time, max over ranks
    step_ms, epoch_ms, eval_ms = (float(x) for x in ms.tolist())
    # per-phase device timeline of one epoch (CUDA events inside the C driver), max over ranks per phase
    trace = {}
    step(trace)
    tr = torch.tensor([trace[k] for k in sorted(trace)], dtype=torch.float64, device=dev)
    dist.all_reduce(tr, op=dist.ReduceOp.MAX)
    trace = {k: round(float(v), 2) for k, v in zip(sorted(trace), tr.tolist())}
    # end to end: rank 0 draws the epoch on the host (exact sampler, background threads), ships 16 B / sample over PCIe,
    # broadcasts it over NVLink; all ranks: sharded epoch + evaluation; steady state of an epoch loop
    e2e = []
    prime = 4                                               # untimed: fill the prefetch queue
    for it in range(prime + max(1, args.steps)):
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.time()
        fetch_epoch()
        step()
        torch.cuda.synchronize()
        dist.barrier()
        if it >= prime:
            e2e.append(time.time() - t0)
    if pipe is not None:
        pipe._flush()
    e2e_t = torch.tensor([float(np.mean(e2e))], dtype=torch.float64, device=dev)
    dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    if rank != 0:
        return None
    pk, pk_src = peaks()
    return {
        "metric": metric, "value": round(step_ms / 1e3, 6), "unit": "s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(step_ms, 3), "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload,
                   "l2": "inputs exceed L2 (graph + tables > 126 MB)",
                   "parallelism": (f"user rows sharded over {world} GPUs, whole epoch enqueued by one C call per rank, no collective "
                                   f"library inside: per layer / Horner step the partial item rows [{I} x {D}] fp32 go to their owner "
                                   f"from the SpMM epilogue over NVLink peer memory, the owner reduces and stores into every replica "
                                   f"({'multimem.st' if m.peer.multicast else 'peer stores'}); gradient block pulled by its owners; "
                                   f"{2 * L + 1} exchanges per batch, 1 NCCL all-reduce per epoch (loss)")},
        "epoch_s": round(epoch_ms / 1e3, 6), "eval_s": round(eval_ms / 1e3, 6), "eval_users_per_s": round(U / (eval_ms / 1e3), 1),
        "epoch_loss": loss, "HR@20(target 0)": hr, "graph_build_s": round(t_graph, 4), "host_sampler_s": round(t_sampler, 3),
        "parity": parity, "phase_ms_per_epoch": trace,
        "roofline": {"bound": "hbm", "achieved": None, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": None, "traffic": None,
                     "note": "per-kernel roofline is reported by the 1-GPU run; this line is the sharded whole-step time"},
        "e2e": {"value": round(float(e2e_t.item()), 6), "unit": "s", "h2d_bytes_per_step": n * 16, "d2h_bytes_per_step": 60,
                "per_step_s": [round(t, 3) for t in e2e],
                "includes": "steady state of an epoch loop: rank 0 draws the next epochs with the exact C++ MT19937 sampler + shuffle on "
                            "background threads, pinned H2D of 16 B / sample, NCCL broadcast; all ranks: sharded epoch + "
                            "evaluation, metric all-reduce and D2H"},
        "gpu_launches": args.steps * (n_batches * ((2 * L) * 5 + 9) + 3),
        "clocks": clocks.summary(),
    }
