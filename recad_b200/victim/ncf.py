"""NCF victim (drop-in for recad/model/victim/ncf.py: 'NeuMF-end', 'NeuMF-pre', 'GMF', 'MLP') on the CUDA kernels.

Every parameter lives in one flat fp32 buffer laid out by `recad_ncf_layout`; the module
attributes of the reference (`embed_user_GMF`, `MLP_layers`, `predict_layer`, ...) are rebuilt as
Parameter views into it.
"""
import ctypes as C
import os

import torch
from torch import nn

from .. import _lib, ops
from .base import BaseVictim

EVAL_CHUNK = 1 << 20   # (user, item) pairs scored per forward call during full-rank evaluation
RANK_PAIRS = 1 << 19   # pairs per block of the factored full-rank path (its workspace: 8.3 KB per pair at the default tower)


def _linear_view(weight, bias):
    """An nn.Linear whose parameters ARE the given views; built without running
    reset_parameters so the global torch generator is not consumed (the reference draws
    nothing here either)."""
    lin = nn.Linear.__new__(nn.Linear)
    nn.Module.__init__(lin)
    lin.out_features, lin.in_features = weight.shape
    lin.weight = nn.Parameter(weight, False)
    lin.bias = nn.Parameter(bias, False)
    return lin


class NCF(BaseVictim):
    name = "ncf"

    def _construct(self, factor_num, num_layers, dropout, model, GMF_model, MLP_model, **config):
        self.config = dict(config, factor_num=factor_num, num_layers=num_layers, dropout=dropout, model=model,
                           GMF_model=GMF_model, MLP_model=MLP_model)
        self.dataset = config["dataset"]
        if dropout:
            raise NotImplementedError("NCF dropout is 0 by default and not implemented")
        if model not in ("NeuMF-end", "NeuMF-pre", "GMF", "MLP"):
            raise ValueError(f"unknown NCF model {model!r}")
        if model == "NeuMF-pre" and (GMF_model is None or MLP_model is None):
            raise ValueError("'NeuMF-pre' needs GMF_model and MLP_model (ncf.py:79-104)")
        if str(config["optim"]).lower() != "adam":
            raise ValueError("optimizer not supported")
        self.tower_precision = config.get("tower_precision", "tf32x3")
        if self.tower_precision not in ("tf32x3", "fp32"):
            raise ValueError("tower_precision must be 'tf32x3' (tensor cores) or 'fp32' (exact CUDA-core GEMMs)")
        info = self.dataset.info_describe()
        U, I = info["n_users"], info["n_items"]
        self.num_users, self.num_items, self.f, self.L = U, I, factor_num, num_layers
        self.variant = {"GMF": 1, "MLP": 2}.get(model, 0)
        w = factor_num * (2 ** (num_layers - 1))
        # constructor + _init_weight_ sequence of ncf.py:32-104 on the CPU generator (the constructors draw their default
        # initialisation for every variant; 'NeuMF-pre' then copies the trained GMF / MLP parts instead of re-drawing)
        ug, ig = nn.Embedding(U, factor_num), nn.Embedding(I, factor_num)
        um, im = nn.Embedding(U, w), nn.Embedding(I, w)
        lins = []
        for i in range(num_layers):
            size = factor_num * (2 ** (num_layers - i))
            lins.append(nn.Linear(size, size // 2))
        pred = nn.Linear(factor_num if self.variant else factor_num * 2, 1)
        if model != "NeuMF-pre":
            nn.init.normal_(ug.weight, std=0.01)
            nn.init.normal_(um.weight, std=0.01)
            nn.init.normal_(ig.weight, std=0.01)
            nn.init.normal_(im.weight, std=0.01)
            for m in lins:
                nn.init.xavier_uniform_(m.weight)
            nn.init.kaiming_uniform_(pred.weight, a=1, nonlinearity="sigmoid")
            for m in lins + [pred]:
                m.bias.data.zero_()
        else:
            cpu = lambda t: t.detach().to("cpu", torch.float32)      # noqa: E731
            ug.weight.data.copy_(cpu(GMF_model.embed_user_GMF.weight))
            ig.weight.data.copy_(cpu(GMF_model.embed_item_GMF.weight))
            um.weight.data.copy_(cpu(MLP_model.embed_user_MLP.weight))
            im.weight.data.copy_(cpu(MLP_model.embed_item_MLP.weight))
            theirs = [x for x in MLP_model.MLP_layers if isinstance(x, nn.Linear)]
            for m1, m2 in zip(lins, theirs):
                m1.weight.data.copy_(cpu(m2.weight))
                m1.bias.data.copy_(cpu(m2.bias))
            pw = torch.cat([cpu(GMF_model.predict_layer.weight), cpu(MLP_model.predict_layer.weight)], dim=1)
            pb = cpu(GMF_model.predict_layer.bias) + cpu(MLP_model.predict_layer.bias)
            pred.weight.data.copy_(0.5 * pw)
            pred.bias.data.copy_(0.5 * pb)
        pieces = [ug.weight.data, ig.weight.data, um.weight.data, im.weight.data]
        for m in lins:
            pieces += [m.weight.data, m.bias.data]
        pieces += [pred.weight.data, pred.bias.data]
        self._alloc(self._device(), pieces)
        self._steps = 0

    def _alloc(self, dev, pieces, m=None, v=None):
        L = _lib.lib()
        offs = (C.c_int64 * (4 + 2 * self.L + 3))()
        self._check(L.recad_ncf_layout(self.f, self.L, self.num_users, self.num_items, offs), "recad_ncf_layout")
        offs = list(offs)
        total = offs[-1]
        self._dev = dev
        # the activation workspace is sized for evaluation-time forward batches (~17 KB per row at the default tower)
        self.max_batch = max(int(self.dataset.config["pointwise_batch_size"]) if hasattr(self.dataset, "config") else 1024, 16384)
        work_floats = L.recad_ncf_work_floats(self.f, self.L, self.max_batch)
        with torch.cuda.device(dev):
            self.flat = torch.zeros(total, dtype=torch.float32, device=dev)
            self.m = torch.zeros(total, dtype=torch.float32, device=dev) if m is None else m.to(dev)
            self.v = torch.zeros(total, dtype=torch.float32, device=dev) if v is None else v.to(dev)
            self.g = torch.empty(total, dtype=torch.float32, device=dev)
            self.work = torch.empty(work_floats, dtype=torch.float32, device=dev)
            self.loss_acc = torch.zeros(4, dtype=torch.float64, device=dev)
        views = []
        for off, src in zip(offs[:-1], pieces):
            vw = self.flat[off:off + src.numel()].view(src.shape)
            vw.copy_(src)
            views.append(vw)
        self._grad_slots = tuple((off, src.numel(), src.shape) for off, src in zip(offs[:-1], pieces))
        U, I, f, w = self.num_users, self.num_items, self.f, self.f * (2 ** (self.L - 1))
        self.embed_user_GMF = nn.Embedding(U, f, _weight=views[0])
        self.embed_item_GMF = nn.Embedding(I, f, _weight=views[1])
        self.embed_user_MLP = nn.Embedding(U, w, _weight=views[2])
        self.embed_item_MLP = nn.Embedding(I, w, _weight=views[3])
        mods = []
        for l in range(self.L):
            mods += [nn.Dropout(p=0.0), _linear_view(views[4 + 2 * l], views[5 + 2 * l]), nn.ReLU()]
        self.MLP_layers = nn.Sequential(*mods)
        self.predict_layer = _linear_view(views[-2], views[-1])
        for p in self.parameters():
            p.requires_grad_(False)
        self.optimizer = None
        st = _lib.NCF()
        st.n_users, st.n_items, st.factor, st.n_layers = U, I, f, self.L
        st.lr, st.beta1, st.beta2, st.eps = self.config["lr"], 0.9, 0.999, 1e-8
        st.tower_fp32 = 1 if self.tower_precision == "fp32" else 0
        st.variant = self.variant
        st.params, st.m, st.v, st.grads, st.n_params = (self.flat.data_ptr(), self.m.data_ptr(), self.v.data_ptr(),
                                                        self.g.data_ptr(), total)
        st.work, st.work_floats, st.max_batch, st.loss_acc = self.work.data_ptr(), work_floats, self.max_batch, self.loss_acc.data_ptr()
        self._st = st

    def _param_views(self):
        """The parameters in recad_ncf_layout order."""
        out = [self.embed_user_GMF.weight, self.embed_item_GMF.weight, self.embed_user_MLP.weight, self.embed_item_MLP.weight]
        for mod in self.MLP_layers:
            if isinstance(mod, nn.Linear):
                out += [mod.weight, mod.bias]
        return out + [self.predict_layer.weight, self.predict_layer.bias]

    def _pieces(self):
        return [p.data for p in self._param_views()]

    def _move(self, dev):
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        if dev != self._dev:
            self._alloc(dev, [p.clone() for p in self._pieces()], self.m, self.v)

    def forward(self, user, item):
        """ncf.py:112-131 (NeuMF-end).  Differentiable with respect to every parameter when grad mode is on and a parameter
        requires a gradient."""
        self._require_instance("forward")
        user = user.to(self._dev).long().contiguous()
        item = item.to(self._dev).long().contiguous()
        if self._graph_mode():
            self._check_ids(user, self.num_users, item, self.num_items)
            return ops.NCFScores.apply(self._st, self._grad_slots, user, item, *self._param_views())
        return ops.ncf_forward(self._st, user, item)

    def train_step(self, **config):
        """One epoch (ncf.py:133-153): returns (mean batch loss,)."""
        self._require_instance("train_step")
        self.train()
        samples, perm = self._epoch_arrays(("users", "items", "labels"))
        n = int(samples.shape[0])
        if n == 0:
            raise ops.RecadError("NCF.train_step: the sampler produced no training row")
        B = int(self.dataset.config["pointwise_batch_size"]) if hasattr(self.dataset, "config") else 1024
        with torch.cuda.device(self._dev):
            self._check(_lib.lib().recad_ncf_train_epoch(C.byref(self._st), self._vp(samples), self._vp(perm),
                                                         n, B, self._steps, ops._stream(self._dev)), "recad_ncf_train_epoch")
        n_batches = (n + B - 1) // B
        self._steps += n_batches
        out = self._read_loss(self.loss_acc, n_batches)
        pbar = config.get("progress_bar", None)
        if pbar:
            pbar.set_description(f"loss: {out[0]:.5f}")
        return out

    def _rank_work(self):
        """Workspace of the factored full-rank path: blocks of RANK_PAIRS (user, item) pairs, 8.3 KB per pair at the default
        tower (recad_ncf_rank_work_floats)."""
        mb = max(RANK_PAIRS, self.num_items)
        if getattr(self, "_rank_ws", None) is None or self._rank_ws[1] != mb:
            wf = int(_lib.lib().recad_ncf_rank_work_floats(self.f, self.L, mb))
            with torch.cuda.device(self._dev):
                self._rank_ws = (torch.empty(wf, dtype=torch.float32, device=self._dev), mb, wf)
        return self._rank_ws

    def full_rank(self, user_ids, targets, K, train_rowptr, train_col):
        """NCF scores are not an inner product: score blocks [users x all items] are materialised block by block and ranked
        by recad_rank_from_scores.  The first tower layer is evaluated once per user and once per item
        (recad_ncf_rank_prepare), a block then costs the remaining layers only; models the factored path does not cover
        (exact fp32 tower, a single layer) go through forward() pair by pair."""
        self._require_instance("full_rank")
        I, dev = self.num_items, self._dev
        n = int(user_ids.numel())
        L = _lib.lib()
        factored = (self.variant == 1 or (self.tower_precision != "fp32" and self.L >= 2 and self.f % 4 == 0)) \
            and not os.environ.get("RECAD_NCF_EXACT") and os.environ.get("RECAD_NCF_RANK_FACTORED", "1") != "0" and n > 0
        outs = []
        if factored:
            st = self._st
            work, mb, wf = self._rank_work()
            users = user_ids.to(dev).long().contiguous()
            with torch.cuda.device(dev):
                pui = torch.empty(max(int(L.recad_ncf_rank_floats(C.byref(st), n)), 1), dtype=torch.float32, device=dev)
                self._check(L.recad_ncf_rank_prepare(C.byref(st), self._vp(users), n, self._vp(pui), self._vp(work), wf, mb,
                                                     ops._stream(dev)), "recad_ncf_rank_prepare")
                per = max(1, mb // I)
                scores = torch.empty((per, I), dtype=torch.float32, device=dev)
                for s in range(0, n, per):
                    nu = min(per, n - s)
                    self._check(L.recad_ncf_rank_block(C.byref(st), self._vp(pui), self._vp(users), n, s, nu, self._vp(scores),
                                                       self._vp(work), wf, mb, ops._stream(dev)), "recad_ncf_rank_block")
                    outs.append(ops.rank_from_scores(scores[:nu], users[s:s + nu], train_rowptr, train_col, targets, K))
            bad = self.loss_acc[3:4].view(torch.int64)
            if int(bad.item()):
                bad.zero_()
                raise ops.RecadError("NCF.full_rank: a user id is out of range")
        else:
            per = max(1, EVAL_CHUNK // I)
            all_items = torch.arange(I, device=dev)
            for s in range(0, n, per):
                ub = user_ids[s:s + per]
                uu = ub.repeat_interleave(I)
                ii = all_items.repeat(ub.numel())
                with torch.no_grad():
                    scores = self.forward(uu, ii).view(ub.numel(), I)
                outs.append(ops.rank_from_scores(scores, ub, train_rowptr, train_col, targets, K))
        return tuple(torch.cat([o[k] for o in outs]) for k in range(4)) + (0.0,)

    # ------------------------------------------------------------------ second order
    def _hvp(self, batch, vectors, what, out, dloss):
        self._require_instance(what)
        samples = self._loss_rows(batch, f"NCF.{what}")
        vecs = self._check_vectors(vectors, [s for _, _, s in self._grad_slots], f"NCF.{what}")
        with torch.cuda.device(self._dev):
            flat = torch.zeros(self._st.n_params, dtype=torch.float32, device=self._dev)    # layout padding stays zero
            for (off, n, _), v in zip(self._grad_slots, vecs):
                flat[off:off + n] = v.view(-1)
            return ops.ncf_hvp(self._st, samples, flat, out=out, dloss=dloss)

    def loss_hvp(self, batch, vectors):
        """H v for the BCE training loss of `batch` taken as one batch (what train_step minimises for it; no regulariser),
        H its Hessian with respect to every parameter at the current values, in the model's tower precision.
        batch: dict of int64 CUDA [n] users / items / labels; vectors: one float32 tensor per parameter, shaped as
        parameters() (embed_user_GMF, embed_item_GMF, embed_user_MLP, embed_item_MLP, each MLP layer's weight and bias,
        predict weight and bias).  Returns the product shaped the same way; parameters the variant does not read get exactly
        zero.  Deterministic; the model is not changed."""
        hv, _ = self._hvp(batch, vectors, "loss_hvp", True, False)
        return tuple(hv[off:off + n].view(shape) for off, n, shape in self._grad_slots)

    def sample_directional_derivatives(self, batch, vectors):
        """For every row b of `batch`, the derivative of its own BCE loss along `vectors` (shaped as for loss_hvp):
        <grad l_b, v>, float32 [n], unnormalised (the batch loss is the mean of the l_b).  Deterministic; the model is not
        changed."""
        return self._hvp(batch, vectors, "sample_directional_derivatives", False, True)[1]

    def input_describe(self):
        return {
            "train_step": {"users": (torch.int64, "batch"), "items": (torch.int64, "batch"), "labels": (torch.int64, "batch")},
            "forward": {"users": (torch.int64, "batch"), "items": (torch.int64, "batch")},
        }

    def output_describe(self):
        return {"train_step": {"loss": (float, [])}, "forward": {"unnormalized_scores": (torch.float32, "batch")}}
