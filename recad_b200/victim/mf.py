"""Biased-MF victim (drop-in for recad/model/victim/mf.py) on the CUDA kernels.

All four tables live back to back in one flat fp32 buffer [Ue | Ie | Ub | Ib] (so the dense Adam
of every step is one launch); `user_emb.weight` etc. are Parameter views.
"""
import ctypes as C

import torch
from torch import nn

from .. import _lib, ops
from .base import BaseVictim


class MF(BaseVictim):
    name = "mf"

    def _construct(self, factor_num, embedding_size, dropout, **config):
        self.config = dict(config, factor_num=factor_num, embedding_size=embedding_size, dropout=dropout)
        self.dataset = config["dataset"]
        if dropout:
            raise NotImplementedError("MF dropout (mf.py:27) is 0 by default and not implemented")
        if str(config["optim"]).lower() != "adam":
            raise ValueError("optimizer not supported")
        if embedding_size % 4:
            raise ValueError("embedding_size must be a multiple of 4")
        info = self.dataset.info_describe()
        self.num_users, self.num_items, self.D = info["n_users"], info["n_items"], embedding_size
        # same constructor / init sequence as mf.py:16-24 on the CPU generator
        tabs = [nn.Embedding(self.num_users, embedding_size), nn.Embedding(self.num_users, 1),
                nn.Embedding(self.num_items, embedding_size), nn.Embedding(self.num_items, 1)]
        tabs[0].weight.data.uniform_(0, 0.005)
        tabs[1].weight.data.uniform_(-0.01, 0.01)
        tabs[2].weight.data.uniform_(0, 0.005)
        tabs[3].weight.data.uniform_(-0.01, 0.01)
        self.mean_value = float(factor_num)                     # mf.py:26: `mean` is the constant factor_num
        self._alloc(self._device(), [t.weight.data for t in tabs])
        self._steps = 0

    def _alloc(self, dev, tabs, m=None, v=None):
        U, I, D = self.num_users, self.num_items, self.D
        sizes = [U * D, I * D, U, I]           # flat order: Ue, Ie, Ub, Ib
        offs = [0, U * D, U * D + I * D, U * D + I * D + U]
        total = sum(sizes)
        self._dev = dev
        with torch.cuda.device(dev):
            self.flat = torch.empty(total, dtype=torch.float32, device=dev)
            self.m = torch.zeros(total, dtype=torch.float32, device=dev) if m is None else m.to(dev)
            self.v = torch.zeros(total, dtype=torch.float32, device=dev) if v is None else v.to(dev)
            self.g = torch.empty(total, dtype=torch.float32, device=dev)
            self.loss_acc = torch.zeros(4, dtype=torch.float64, device=dev)

        def view(buf, k):
            return buf[offs[k]:offs[k] + sizes[k]]
        Ue, Ie, Ub, Ib = (view(self.flat, k) for k in range(4))
        Ue.view(U, D).copy_(tabs[0]); Ub.view(U, 1).copy_(tabs[1]); Ie.view(I, D).copy_(tabs[2]); Ib.view(I, 1).copy_(tabs[3])
        self.user_emb = nn.Embedding(U, D, _weight=Ue.view(U, D))
        self.user_bias = nn.Embedding(U, 1, _weight=Ub.view(U, 1))
        self.item_emb = nn.Embedding(I, D, _weight=Ie.view(I, D))
        self.item_bias = nn.Embedding(I, 1, _weight=Ib.view(I, 1))
        self.mean = nn.Parameter(torch.tensor([self.mean_value], device=dev), False)
        self._mean_version = self.mean._version
        for p in self.parameters():
            p.requires_grad_(False)
        self.optimizer = None
        st = _lib.MF()
        st.n_users, st.n_items, st.D, st.mean = U, I, D, self.mean_value
        st.lr, st.beta1, st.beta2, st.eps = self.config["lr"], 0.9, 0.999, 1e-8
        for prefix, buf in (("", self.flat), ("m", self.m), ("v", self.v), ("g", self.g)):
            for k, nm in enumerate(("Ue", "Ie", "Ub", "Ib")):
                setattr(st, prefix + nm, view(buf, k).data_ptr())
        st.loss_acc = self.loss_acc.data_ptr()
        self._st = st

    def _move(self, dev):
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        if dev != self._dev:
            self._alloc(dev, [self.user_emb.weight.data, self.user_bias.weight.data, self.item_emb.weight.data,
                              self.item_bias.weight.data], self.m, self.v)

    def _sync_mean(self):
        """The kernels read `mean` from the state: take over an in-place update of the parameter (a torch optimizer's step
        once the user made it trainable)."""
        if self.mean._version != self._mean_version:
            self.mean_value = float(self.mean.detach().view(-1)[0])
            self._st.mean = self.mean_value
            self._mean_version = self.mean._version

    def forward(self, users, items):
        """mf.py:40-47.  Differentiable with respect to the four tables (and `mean` once it requires a gradient) when grad
        mode is on and a parameter requires a gradient."""
        self._require_instance("forward")
        users = users.to(self._dev).long().contiguous()
        items = items.to(self._dev).long().contiguous()
        self._sync_mean()
        if self._graph_mode():
            self._check_ids(users, self.num_users, items, self.num_items)
            return ops.MFScores.apply(self._st, users, items, self.user_emb.weight, self.user_bias.weight, self.item_emb.weight,
                                      self.item_bias.weight, self.mean)
        return ops.mf_forward(self._st, users, items)

    def train_step(self, **config):
        """One epoch (mf.py:49-69): returns (mean batch loss,)."""
        self._require_instance("train_step")
        self.train()
        samples, perm = self._epoch_arrays(("users", "items", "labels"))
        n = int(samples.shape[0])
        if n == 0:
            raise ops.RecadError("MF.train_step: the sampler produced no training row")
        B = int(self.dataset.config["pointwise_batch_size"]) if hasattr(self.dataset, "config") else 1024
        with torch.cuda.device(self._dev):
            self._check(_lib.lib().recad_mf_train_epoch(C.byref(self._st), self._vp(samples), self._vp(perm),
                                                        n, B, self._steps, ops._stream(self._dev)), "recad_mf_train_epoch")
        n_batches = (n + B - 1) // B
        self._steps += n_batches
        out = self._read_loss(self.loss_acc, n_batches)
        pbar = config.get("progress_bar", None)
        if pbar:
            pbar.set_description(f"loss: {out[0]:.4f}")
        return out

    def full_rank(self, user_ids, targets, K, train_rowptr, train_col):
        """score = <U_u, V_i> + b_i (+ b_u + mean, constant per user): the item bias is added inside the
        fused full-rank kernel, the per-user constants afterwards."""
        self._require_instance("full_rank")
        self._sync_mean()
        with torch.no_grad():
            topi, topv, rank, score = ops.fullrank_eval(self.user_emb.weight, self.item_emb.weight, user_ids, train_rowptr,
                                                        train_col, targets, K, item_bias=self.item_bias.weight.view(-1))
            # b_u and the mean shift every score of a user equally: they never change a rank, only the reported score
            score = score + self.user_bias.weight.view(-1)[user_ids].unsqueeze(1)
        return topi, topv, rank, score, self.mean_value

    # ------------------------------------------------------------------ second order
    def _loss_seeds(self, batch, vectors, what, dloss):
        self._require_instance(what)
        samples = self._loss_rows(batch, f"MF.{what}")
        U, I, D = self.num_users, self.num_items, self.D
        vecs = self._check_vectors(vectors, [(U, D), (U, 1), (I, D), (I, 1)], f"MF.{what}")
        self._sync_mean()
        with torch.cuda.device(self._dev):
            alpha, beta, dl = ops.mf_hvp_seeds(self._st, *vecs, samples, dloss=dloss)
        return samples, vecs, alpha, beta, dl

    def loss_hvp(self, batch, vectors):
        """H v for the BCE training loss of `batch` taken as one batch (what train_step minimises for it), H its Hessian
        with respect to (user_emb, user_bias, item_emb, item_bias) at the current tables, `mean` held constant.
        batch: dict of int64 CUDA [n] users / items / labels; vectors: (v_Ue [U, D], v_Ub [U, 1], v_Ie [I, D], v_Ib [I, 1])
        float32.  Returns the four products shaped likewise.  Deterministic; the model is not changed."""
        samples, (vUe, _, vIe, _), alpha, beta, _ = self._loss_seeds(batch, vectors, "loss_hvp", False)
        U, I = self.num_users, self.num_items
        with torch.cuda.device(self._dev):
            out, hUb, hIb = ops.pair_scores_hvp(self.user_emb.weight.detach(), vUe, self.item_emb.weight.detach(), vIe,
                                                samples[:, 0].contiguous(), samples[:, 1].contiguous(), alpha, beta, bias=True)
        return out[:U], hUb.view(U, 1), out[U:], hIb.view(I, 1)

    def sample_directional_derivatives(self, batch, vectors):
        """For every row b of `batch`, the derivative of its own BCE loss along `vectors` (shaped as for loss_hvp):
        <grad l_b, v>, float32 [n], unnormalised (the batch loss is the mean of the l_b).  Deterministic; the model is not
        changed."""
        return self._loss_seeds(batch, vectors, "sample_directional_derivatives", True)[4]

    def input_describe(self):
        return {
            "train_step": {"users": (torch.int64, "batch"), "items": (torch.int64, "batch"), "labels": (torch.int64, "batch")},
            "forward": {"users": (torch.int64, "batch"), "items": (torch.int64, "batch")},
        }

    def output_describe(self):
        return {"train_step": {"loss": (float, [])}, "forward": {"unnormalized_scores": (torch.float32, "batch")}}
