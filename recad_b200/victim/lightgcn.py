"""LightGCN victim (drop-in for recad/model/victim/lightgcn.py) on the CUDA kernels.

State layout in HBM: ONE table E [N, D] fp32 with the user rows first, then the item rows
(the `torch.cat([users_emb, items_emb])` of lightgcn.py:86-88 is free), Adam moments m, v of
the same shape, and five work buffers of N*D floats.  `embedding_user.weight` /
`embedding_item.weight` are Parameter views into E, so `parameters()` / `state_dict()` see the
live values.
"""
import ctypes as C

import torch
from torch import nn

from .. import _lib, ops
from ..config import get_logger
from .base import BaseVictim


class LightGCN(BaseVictim):
    name = "lightgcn"
    user_args = ("dataset", "user_emb", "item_emb")

    def _construct(self, **config):
        self.config = config
        self.dataset = config["dataset"]
        self.logger = get_logger(__name__, config["logging_level"])
        if config["A_split"]:
            raise ValueError("A_split is not support in LightGCN yet")          # lightgcn.py:38-39
        # graph dropout (lightgcn.py:62-80, off by default): every computer() call of a model in training mode -- one per
        # batch, and, since the reference never calls eval(), one per forward -- draws a fresh mask over the nnz entries
        self.dropout, self.keep_prob = bool(config["dropout"]), float(config["keep_prob"])
        self._drop_graph = self._drop_graph_t = self._st_drop = None
        if str(config["optim"]).lower() != "adam":
            raise ValueError("optimizer not supported")                          # only Adam is on the hot path
        info = self.dataset.info_describe()
        self.num_users, self.num_items = info["n_users"], info["n_items"]
        self.Graph = info["graph"]
        if not isinstance(self.Graph, ops.Graph):
            raise TypeError("recad_b200.LightGCN needs the device-resident graph of recad_b200.dataset.ImplicitData "
                            f"(got {type(self.Graph)})")
        self.latent_dim = config["latent_dim_rec"]
        self.n_layers = config["lightGCN_n_layers"]
        if self.latent_dim % 4:
            raise ValueError("latent_dim_rec must be a multiple of 4")
        # initialisation on the CPU generator, call for call as the reference (lightgcn.py:40-48):
        # nn.Embedding draws N(0,1) at construction, then normal_(std=0.1) overwrites
        if config.get("init_on_device") and not config["pretrain"]:
            # NEW, off by default: N(0, 0.1) drawn by the CUDA generator (seeded by torch.manual_seed as well) instead of
            # replaying the reference's CPU stream -- 2 x 77 M CPU draws cost 0.6 s per fresh model at the synthetic size,
            # which an attack loop pays every iteration.  Same distribution, different numbers than the reference.
            dev = self._device()
            with torch.cuda.device(dev):
                w = torch.randn((self.num_users + self.num_items, self.latent_dim), device=dev) * 0.1
            self._alloc(dev, w[:self.num_users], w[self.num_users:])
            self._steps = 0
            self._O_valid = False
            return
        eu = nn.Embedding(self.num_users, self.latent_dim)
        ei = nn.Embedding(self.num_items, self.latent_dim)
        if not config["pretrain"]:
            nn.init.normal_(eu.weight, std=0.1)
            nn.init.normal_(ei.weight, std=0.1)
        else:
            eu.weight.data.copy_(torch.from_numpy(config["user_emb"]))
            ei.weight.data.copy_(torch.from_numpy(config["item_emb"]))
        self._alloc(self._device(), eu.weight.data, ei.weight.data)
        self._steps = 0
        self._O_valid = False

    # ------------------------------------------------------------------ buffers
    def _alloc(self, dev, user_w, item_w, m=None, v=None):
        U, I, D = self.num_users, self.num_items, self.latent_dim
        N = U + I
        self._dev = dev
        with torch.cuda.device(dev):
            self.E = torch.empty((N, D), dtype=torch.float32, device=dev)
            self.E[:U].copy_(user_w)
            self.E[U:].copy_(item_w)
            self.m = torch.zeros_like(self.E) if m is None else m.to(dev)
            self.v = torch.zeros_like(self.E) if v is None else v.to(dev)
            self.O, self.X0, self.X1, self.g = (torch.empty_like(self.E) for _ in range(4))
            self.cnt = torch.empty(N, dtype=torch.float32, device=dev)
            self.loss_acc = torch.zeros(4, dtype=torch.float64, device=dev)
        self.embedding_user = nn.Embedding(U, D, _weight=self.E[:U])
        self.embedding_item = nn.Embedding(I, D, _weight=self.E[U:])
        for p in self.parameters():
            p.requires_grad_(False)
        self.optimizer = None     # Adam is fused into the epoch driver; its moments are self.m / self.v
        st = _lib.LightGCN()
        st.graph = C.pointer(self.Graph.struct(D))
        st.n_users, st.n_items, st.D, st.n_layers = U, I, D, self.n_layers
        st.lam, st.lr, st.beta1, st.beta2, st.eps = self.config["lambda"], self.config["lr"], 0.9, 0.999, 1e-8
        for k in ("E", "m", "v", "O", "X0", "X1", "g", "cnt", "loss_acc"):
            setattr(st, k, getattr(self, k).data_ptr())
        self._st = st
        self._drop_graph = self._drop_graph_t = self._st_drop = None
        self._value_graphs = None  # ops.ValueGraphs for caller-supplied edge values, made on first use
        self._O_valid = False      # O was just (re)allocated: never score from it before a propagate
        self._O_version = -1

    def load_state_dict(self, *args, **kwargs):
        out = super().load_state_dict(*args, **kwargs)
        self._O_valid = False      # the tables changed under the cached propagation
        return out

    def invalidate(self):
        """Call after editing embedding_*.weight.data in place: forward() / full_rank() reuse the cached propagation
        until a train_step, load_state_dict or device move says the tables changed (the reference re-propagates on
        every forward, lightgcn.py:174-176)."""
        self._O_valid = False

    def _move(self, dev):
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        if dev != self._dev:
            if self.Graph.device != dev:
                raise ops.RecadError("the dataset graph lives on another device")
            self._alloc(dev, self.E[:self.num_users], self.E[self.num_users:], self.m, self.v)

    # ------------------------------------------------------------------ graph dropout
    def _dropped_state(self, with_vals_t=False):
        """lightgcn.py:62-80 `__dropout_x`: keep an entry when int(rand + keep_prob) is 1, rescale the kept values by
        1 / keep_prob.  The mask is drawn exactly as the reference draws it -- torch.rand(nnz) on the CPU generator, in the
        coalesced (row-major) entry order, which is the CSR order -- so a seeded run drops the same entries.  Dropped
        entries keep their place in the structure with value 0 (the plan and both SpMM directions are unchanged): the
        state returned is this model's with the graph swapped for that matrix (and, with_vals_t, the transposed values,
        which an autograd backward restores)."""
        g = self.Graph
        keep = (torch.rand(g.nnz) + self.keep_prob).int().bool()
        with torch.cuda.device(self._dev):
            keep = keep.to(self._dev)
            vals = torch.where(keep, g.vals / self.keep_prob, torch.zeros((), dtype=g.vals.dtype, device=self._dev))
            # (u, i) and (i, u) are dropped independently: the dropped matrix is not symmetric and autograd's backward
            # multiplies by its TRANSPOSE -- the same structure with the values permuted
            vals_t = vals[g.transpose_permutation()]
            if self._drop_graph is None:
                self._drop_graph, self._drop_graph_t = g.with_values(vals), g.with_values(vals_t)
                st = _lib.LightGCN()
                C.memmove(C.byref(st), C.byref(self._st), C.sizeof(st))
                st.graph = C.pointer(self._drop_graph.struct(self.latent_dim))
                st.graph_t = C.pointer(self._drop_graph_t.struct(self.latent_dim))
                self._st_drop = st
            else:
                self._drop_graph.set_values(vals)
                self._drop_graph_t.set_values(vals_t)
        return (self._st_drop, vals_t) if with_vals_t else self._st_drop

    # ------------------------------------------------------------------ compute
    def _propagate_graph(self):
        """The propagation as an autograd node: a fresh [N, D] output differentiable with respect to both tables."""
        if self.dropout and self.training:
            st, vals_t = self._dropped_state(with_vals_t=True)
            graph_t = self._drop_graph_t
        else:
            st, graph_t, vals_t = self._st, None, None
        return ops.LightGCNPropagate.apply(st, graph_t, vals_t, self.embedding_user.weight, self.embedding_item.weight)

    def _propagate_values(self, edge_values):
        """The propagation over caller-supplied edge values (float32 CUDA [Graph.nnz], CSR entry order) into a fresh buffer:
        differentiable with respect to them and to the tables when grad mode is on and one of them requires a gradient.
        The cached propagation (self.O) is neither read nor written."""
        ops.check_values(self.Graph, edge_values, "LightGCN edge_values")
        if self.dropout and self.training:
            raise ops.RecadError("LightGCN: edge_values cannot be combined with graph dropout in training mode")
        if self._value_graphs is None:
            self._value_graphs = ops.ValueGraphs(self.Graph, self._st)
        w_u, w_i = self.embedding_user.weight, self.embedding_item.weight
        if torch.is_grad_enabled() and (edge_values.requires_grad or w_u.requires_grad or w_i.requires_grad):
            return ops.LightGCNPropagateValues.apply(self._value_graphs, self.E, edge_values.contiguous(), w_u, w_i)
        st = self._value_graphs.load(edge_values)
        return ops.lightgcn_propagate_values(st, self.E)

    def _cached_O(self):
        """self.O, propagated again unless it is current: the tables have not changed since (train_step, load_state_dict,
        in-place updates such as a torch optimizer's step, which bump the tables' version) and no dropout mask applies."""
        if not self._O_valid or self._O_version != self.E._version or (self.dropout and self.training):
            self.computer()
        return self.O

    def computer(self, edge_values=None):
        """lightgcn.py:82-113: (users, items) propagated embeddings = mean of the layer outputs (over a freshly dropped
        graph when dropout is on and the module is in training mode).  Differentiable with respect to the two tables when
        grad mode is on and one of them requires a gradient.
        edge_values: float32 CUDA tensor [Graph.nnz] in the graph's CSR entry order, propagated over instead of the graph's
        values (and differentiable with respect to when it requires a gradient); not with graph dropout in training mode."""
        self._require_instance("computer")
        if edge_values is not None:
            O = self._propagate_values(edge_values)
            return O[:self.num_users], O[self.num_users:]
        if self._graph_mode():
            O = self._propagate_graph()
            return O[:self.num_users], O[self.num_users:]
        dropped = self.dropout and self.training
        st = self._dropped_state() if dropped else self._st
        with torch.cuda.device(self._dev):
            self._check(_lib.lib().recad_lightgcn_propagate(C.byref(st), ops._stream(self._dev)), "recad_lightgcn_propagate")
        self._O_valid = not dropped      # a dropped propagation is never reused: the next call draws a new mask
        self._O_version = self.E._version
        return self.O[:self.num_users], self.O[self.num_users:]

    def getUsersRating(self, users):
        """lightgcn.py:115-120 (unused by the reference's workflows; kept for API parity)."""
        all_users, all_items = self.computer()
        return torch.sigmoid(all_users[users.long()] @ all_items.t())

    def train_step(self, **config):
        """One epoch (lightgcn.py:132-172): returns (mean batch loss,)."""
        self._require_instance("train_step")
        self.train()
        samples, perm = self._epoch_arrays(("users", "positive_items", "negative_items"))
        n = int(samples.shape[0])
        if n == 0:
            raise ops.RecadError("LightGCN.train_step: the sampler produced no training triple")
        B = int(self.dataset.config["pairwise_batch_size"]) if hasattr(self.dataset, "config") else 1024
        n_batches = (n + B - 1) // B
        if self.dropout:
            # one mask per batch (lightgcn.py:90-92 inside getEmbedding): the epoch driver runs batch by batch, each over its
            # own dropped graph; loss and the out-of-range flag are summed on the device
            total = torch.zeros_like(self.loss_acc)
            for k in range(n_batches):
                lo, hi = k * B, min(n, (k + 1) * B)
                rows, order = (samples, perm[lo:hi]) if perm is not None else (samples[lo:hi], None)
                self.run_epoch(rows, order, B, st=self._dropped_state(), n=hi - lo, step0=self._steps + k)
                total[2] += self.loss_acc[2]
                total[3:4].view(torch.int64).bitwise_or_(self.loss_acc[3:4].view(torch.int64))
            self.loss_acc.copy_(total)
        else:
            self.run_epoch(samples, perm, B)
        self._steps += n_batches
        self._O_valid = False
        pbar = config.get("progress_bar", None)
        out = self._read_loss(self.loss_acc, n_batches)
        if pbar:
            pbar.set_description(f"loss {out[0]:.5f}")
        return out

    def run_epoch(self, samples, perm, B, st=None, n=None, step0=None):
        """Enqueue one epoch over device-resident rows (int64 or int32 [n, 3]) visited in the order perm (same dtype).
        st / n / step0: another state (the dropped graph), the number of rows to visit and the Adam steps taken so far."""
        L = _lib.lib()
        i32 = samples.dtype == torch.int32
        if perm is not None and perm.dtype != samples.dtype:
            perm = perm.to(samples.dtype)
        fn, name = (L.recad_lightgcn_train_epoch_i32, "recad_lightgcn_train_epoch_i32") if i32 else \
            (L.recad_lightgcn_train_epoch, "recad_lightgcn_train_epoch")
        with torch.cuda.device(self._dev):
            self._check(fn(C.byref(self._st if st is None else st), self._vp(samples), self._vp(perm),
                           int(samples.shape[0]) if n is None else int(n), B, self._steps if step0 is None else int(step0),
                           ops._stream(self._dev)), name)

    def forward(self, users, items, edge_values=None):
        """lightgcn.py:174-183: <O_u, O_i>.  The propagation is redone only when the tables changed
        (the reference redoes it on every call, i.e. once per evaluated user).  In autograd (grad mode on and a table
        that requires a gradient) every call propagates again, as the reference does, and the scores are differentiable
        with respect to both tables.
        edge_values: see `computer`; such a call always propagates again, and its scores are differentiable with respect
        to edge_values when it requires a gradient."""
        self._require_instance("forward")
        users = users.to(self._dev).long().contiguous()
        items = items.to(self._dev).long().contiguous()
        if edge_values is not None:
            O = self._propagate_values(edge_values)
            if O.requires_grad:
                self._check_ids(users, self.num_users, items, self.num_items)
                return ops.DotScores.apply(O, self.num_users, users, items)
            return ops.dot_scores(O, self.num_users, users, items)
        if self._graph_mode():
            self._check_ids(users, self.num_users, items, self.num_items)
            return ops.DotScores.apply(self._propagate_graph(), self.num_users, users, items)
        return ops.dot_scores(self._cached_O(), self.num_users, users, items)

    def full_rank(self, user_ids, targets, K, train_rowptr, train_col):
        """Batched evaluation entry used by recad_b200.evaluate (fused score/mask/top-K kernel)."""
        self._require_instance("full_rank")
        with torch.no_grad():
            O = self._cached_O()
        U = self.num_users
        return ops.fullrank_eval(O[:U], O[U:], user_ids, train_rowptr, train_col, targets, K) + (0.0,)

    # ------------------------------------------------------------------ second order
    def _loss_inputs(self, batch, vectors, what):
        """The rows of `batch` as int64 [n, 3] and the direction V [N, D], checked."""
        self._require_instance(what)
        if self.dropout and self.training:
            raise ops.RecadError(f"LightGCN.{what}: not defined under graph dropout in training mode (call eval() first)")
        samples = self._loss_rows(batch, f"LightGCN.{what}")
        U, I, D = self.num_users, self.num_items, self.latent_dim
        vu, vi = self._check_vectors(vectors, [(U, D), (I, D)], f"LightGCN.{what}")
        with torch.cuda.device(self._dev):
            return samples, torch.cat([vu, vi])

    def _loss_directions(self, batch, vectors, what):
        """Rows, the direction V [N, D], O = P E and dO = P V for the training loss of `batch` (fresh buffers: the model's
        tables, moments and cached propagation are not touched)."""
        samples, V = self._loss_inputs(batch, vectors, what)
        with torch.cuda.device(self._dev):
            O, _ = ops.lightgcn_propagate_layers(self._st, self.E, keep=False)
            dO, _ = ops.lightgcn_propagate_layers(self._st, V, keep=False)
        return samples, V, O, dO

    def loss_hvp(self, batch, vectors):
        """H v for the BPR training loss of `batch` taken as one batch (what train_step minimises for it: mean softplus +
        lambda * 0.5 * sum of the squared rows / n), H its Hessian with respect to (embedding_user.weight,
        embedding_item.weight) at the current tables.  batch: dict of int64 CUDA [n] users / positive_items /
        negative_items; vectors: (v_user [U, D], v_item [I, D]) float32.  Returns (Hv_user, Hv_item).  Deterministic; the
        model is not changed.  H v = P^T H_O (P v) + (lambda / n) cnt * v (DESIGN.md, "Second order")."""
        samples, V, O, dO = self._loss_directions(batch, vectors, "loss_hvp")
        U, N, n = self.num_users, self.num_users + self.num_items, samples.shape[0]
        lam = float(self.config["lambda"])
        with torch.cuda.device(self._dev):
            alpha, beta, _ = ops.bpr_hvp_seeds(O, dO, U, samples)
            u, p, q = samples.unbind(1)
            HO, _, _ = ops.pair_scores_hvp(O[:U], dO[:U], O[U:], dO[U:], torch.cat([u, u]), torch.cat([q, p]), alpha, beta)
            hv = ops.lightgcn_backward(self._st, HO)
            cnt = torch.bincount(torch.cat([u, p + U, q + U]), minlength=N)       # exact integer multiplicities
            hv.addcmul_(V, (cnt.float() * (lam / n)).unsqueeze(1))
        return hv[:U], hv[U:]

    def sample_directional_derivatives(self, batch, vectors):
        """For every row b of `batch`, the derivative of its own loss l_b = softplus(x_b) + lambda * 0.5 * (|E_u|^2 + |E_p|^2 +
        |E_n|^2) along `vectors` (shaped as for loss_hvp): <grad l_b, v>, float32 [n], unnormalised (the batch loss is the
        mean of the l_b).  Deterministic; the model is not changed."""
        samples, V, O, dO = self._loss_directions(batch, vectors, "sample_directional_derivatives")
        with torch.cuda.device(self._dev):
            _, _, dloss = ops.bpr_hvp_seeds(O, dO, self.num_users, samples, float(self.config["lambda"]), self.E, V, dloss=True)
        return dloss

    def loss_mixed_values(self, batch, vectors):
        """g_v = d/dv <v_vec, grad_E L>: the mixed second derivative of the BPR training loss of `batch` (as for loss_hvp)
        with respect to the graph's edge values v, along `vectors` (shaped as for loss_hvp), at the current tables and the
        graph's own values.  Float32 [Graph.nnz] in CSR entry order; zeros for n_layers = 0 (the regulariser does not
        depend on v).  Chain it through ops.normalized_values for interaction weights.  Deterministic; the model is not
        changed.  One recurrence over the interleaved [E | v_vec] rows at width 2D (DESIGN.md, "Second order")."""
        samples, V = self._loss_inputs(batch, vectors, "loss_mixed_values")
        with torch.cuda.device(self._dev):
            return ops.lightgcn_loss_mixed_values(self._st, self.Graph, V, samples)

    def _check_candidate_users(self, users, what):
        """RecadError unless `users` is an int64 / int32 CUDA tensor [R] on the model's device (ids are range-checked by the
        kernel)."""
        if not isinstance(users, torch.Tensor) or not users.is_cuda or users.device != self._dev:
            raise ops.RecadError(f"{what}: users must be a CUDA tensor on {self._dev}")
        if users.dim() != 1 or users.dtype not in (torch.int64, torch.int32):
            raise ops.RecadError(f"{what}: users must be int64 [R], got {users.dtype} {list(users.shape)}")

    def candidate_weight_gradients(self, users, gO=None, batch=None, vectors=None):
        """df/dW[r, i] for f(W) = <gO, O(W)> + <v_vec, grad_E L_batch(E; W)>, W one weight on both entries (users[r], U + i)
        and (U + i, users[r]) of an interaction, for every item i, stored or not: float32 [len(users), num_items].  The base
        point is W = Graph.mult on stored pairs and 0 elsewhere, at the current tables; O = (users_out, items_out) of
        computer().  gO: (g_user [U, D], g_item [I, D]) float32 or None; batch and vectors (shaped as for loss_hvp) go
        together or are both None; L_batch weights row b by w_k / mult_k when its positive pair k is stored.  users: int64
        CUDA ids (repeats allowed; empty gives [0, num_items]).  At a stored pair the value is the sum over the pair's two
        entries of normalized_values' backward of the edge-value gradient, plus the sample part of interaction_hypergradient.
        Deterministic; the model is not changed.  One width-2D recurrence and one tensor-core GEMM (DESIGN.md, "Second
        order")."""
        what = "LightGCN.candidate_weight_gradients"
        self._require_instance("candidate_weight_gradients")
        if self.dropout and self.training:
            raise ops.RecadError(f"{what}: not defined under graph dropout in training mode (call eval() first)")
        if (batch is None) != (vectors is None):
            raise ops.RecadError(f"{what}: batch and vectors go together")
        self._check_candidate_users(users, what)
        U, I, D = self.num_users, self.num_items, self.latent_dim
        G = S = samples = None
        with torch.cuda.device(self._dev):
            if gO is not None:
                G = torch.cat(self._check_vectors(gO, [(U, D), (I, D)], what))
            if batch is not None:
                samples, S = self._loss_inputs(batch, vectors, "candidate_weight_gradients")
            return ops.lightgcn_candidate_weight_grads(self._st, self.Graph, users.long(), G, S, samples,
                                                       float(self.config["lambda"]))

    def input_describe(self):
        return {
            "train_step": {"users": (torch.int64, "batch"), "positive_items": (torch.int64, "batch"),
                           "negative_items": (torch.int64, "batch")},
            "forward": {"users": (torch.int64, "batch"), "items": (torch.int64, "batch")},
        }

    def output_describe(self):
        return {"train_step": {"loss": (float, [])}, "forward": {"unnormalized_scores": (torch.float32, "batch")}}
