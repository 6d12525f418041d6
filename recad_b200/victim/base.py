"""Victim base: the reference's BaseModel / BaseVictim contract (recad/model/base.py:21-104,
recad/model/victim/base.py) for models whose state lives in flat device buffers driven by
librecad_b200.so."""
import ctypes as C

import torch

from .. import _lib, ops
from ..config import MODEL, LazyMixin, get_logger, merge_config


class BaseVictim(LazyMixin, torch.nn.Module):
    name = None            # key in MODEL['victim']
    user_args = ("dataset",)

    @classmethod
    def from_config(cls, **kwargs):
        """model.from_config('victim', name, **kw) (model/base.py:27-53): lazy shell; `.I(dataset=...)` builds."""
        logger = get_logger(__name__)
        cfg = merge_config(MODEL["victim"][cls.name], kwargs, cls.user_args, logger, owner=str(cls))
        return cls._shell(cfg, cls.name)

    @property
    def model_name(self):
        return getattr(self, "_model_name", type(self).__name__)

    def reset(self, **kwargs):
        """model/base.py:94-104: a fresh LAZY model with the original hyper-parameters."""
        if not hasattr(self, "_init_config"):
            raise ValueError("reset method is only for datasets instantiated from_config")
        config = dict(self._init_config)
        for k, v in kwargs.items():
            if k not in config:
                raise ValueError(f"reset arg {k} should be in {list(config)}")
            config[k] = v
        return type(self).from_config(**config)

    def info_describe(self):
        return {"input_describe": self.input_describe(), "output_describe": self.output_describe()}

    def print_help(self, **kwargs):
        from pprint import pprint
        pprint({"model_name": self.model_name, **{k: str(v)[:60] for k, v in self.config.items() if k != "dataset"}})

    # ------------------------------------------------------------------ device handling
    def _device(self):
        dev = torch.device(self.config["device"])
        if dev.type != "cuda":
            raise ops.RecadError(
                f"{type(self).__name__}: recad_b200 victims compute on a CUDA device only (config device = {dev}); "
                "there is no CPU fallback")
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        return dev

    def to(self, device=None, *args, **kwargs):
        """workflow: `victim.to(self.c['device'])` (normal.py:167, 206).  State is created on the
        config device at construction; a different CUDA device moves it."""
        self._require_instance("to")
        if device is not None and torch.device(device).type == "cuda" and hasattr(self, "_move"):
            self._move(torch.device(device))
        return self

    def _epoch_arrays(self, names):
        """The epoch's training rows for the C epoch driver: (samples int64 [n, 3], perm int64 [n] or None)
        on the device.  recad_b200 datasets hand over sampler-order rows + the shuffle permutation; for any
        other BaseData the reference-style batch generator is drained (its rows are already shuffled)."""
        ds = self.dataset
        # a pairwise victim on a pointwise dataset (or the reverse) would read (user, item, label) rows as
        # (user, pos, neg): the reference fails on the missing batch key, so does this
        want = "pairwise" if names[1] == "positive_items" else "pointwise"
        have = getattr(ds, "config", {}).get("sample") if isinstance(getattr(ds, "config", None), dict) else None
        if have is not None and have != want:
            raise KeyError(f"{names[1]}: {type(self).__name__} trains on {want} batches but the dataset samples {have}")
        if hasattr(ds, "epoch_samples"):
            return ds.epoch_samples(self._dev)
        cols = [[] for _ in names]
        for batch in ds.generate_batch():
            for c, n in zip(cols, names):
                c.append(batch[n].to(self._dev).long())
        if not cols[0]:
            return torch.zeros((0, 3), dtype=torch.int64, device=self._dev), None
        return torch.stack([torch.cat(c) for c in cols], 1).contiguous(), None

    def _read_loss(self, loss_acc, n_batches):
        """One device->host copy per epoch (the reference syncs every batch, lightgcn.py:169)."""
        acc = loss_acc.cpu()
        if acc[3:4].view(torch.int64).item() != 0:
            raise ops.RecadError(f"{type(self).__name__}.train_step: a sample id is out of range")
        return (float(acc[2]) / n_batches,)

    def _graph_mode(self):
        """Autograd applies to this call (the usual torch rule): grad mode is on and a parameter requires a gradient.
        Otherwise the victim runs its plain kernels and returns tensors without a grad_fn."""
        return torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())

    @staticmethod
    def _check_ids(users, n_users, items, n_items):
        """RecadError unless every id lies inside its table (one device->host copy)."""
        if users.numel() != items.numel():
            raise ops.RecadError(f"{users.numel()} users but {items.numel()} items")
        if users.numel() and bool(((users < 0) | (users >= n_users)).any() | ((items < 0) | (items >= n_items)).any()):
            raise ops.RecadError("a user or item id is out of range")

    def _loss_rows(self, batch, what):
        """The train_step rows of a caller's batch dict (keys of input_describe()["train_step"], int64 CUDA [n] each on
        the model's device) as one int64 [n, 3] tensor; RecadError otherwise.  Ids are range-checked by the kernels."""
        names = tuple(self.input_describe()["train_step"])
        if not isinstance(batch, dict) or set(names) - set(batch):
            raise ops.RecadError(f"{what}: batch must be a dict with the keys {names}")
        cols = [batch[k] for k in names]
        for k, c in zip(names, cols):
            if not isinstance(c, torch.Tensor) or not c.is_cuda or c.device != self._dev:
                raise ops.RecadError(f"{what}: batch[{k!r}] must be a CUDA tensor on {self._dev}")
            if c.dtype != torch.int64 or c.dim() != 1:
                raise ops.RecadError(f"{what}: batch[{k!r}] must be int64 [n], got {c.dtype} {list(c.shape)}")
        n = cols[0].numel()
        if n == 0 or any(c.numel() != n for c in cols):
            raise ops.RecadError(f"{what}: the batch columns must have the same positive length")
        return torch.stack([c.detach() for c in cols], 1).contiguous()

    def _check_vectors(self, vectors, shapes, what):
        """RecadError unless `vectors` is a sequence of float32 CUDA tensors on the model's device with the given shapes
        (the trainable tables in parameters() order); returns them detached and contiguous."""
        if not isinstance(vectors, (tuple, list)) or len(vectors) != len(shapes):
            raise ops.RecadError(f"{what}: vectors must be a tuple of {len(shapes)} tensors shaped {shapes}")
        out = []
        for v, shp in zip(vectors, shapes):
            if not isinstance(v, torch.Tensor) or not v.is_cuda or v.device != self._dev:
                raise ops.RecadError(f"{what}: vectors must be CUDA tensors on {self._dev}")
            if v.dtype != torch.float32 or tuple(v.shape) != tuple(shp):
                raise ops.RecadError(f"{what}: float32 {list(shp)} needed, got {v.dtype} {list(v.shape)}")
            out.append(v.detach().contiguous())
        return out

    @staticmethod
    def _vp(t):
        return C.c_void_p(t.data_ptr()) if t is not None else None

    @staticmethod
    def _check(rc, what):
        _lib.check(rc, what)
