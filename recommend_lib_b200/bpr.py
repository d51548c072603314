"""BPR-MF behind Daisy's surface, computed by libdaisy_b200.so on a B200.

Reference surface mirrored here (file:line relative to the reference root):

* ``BPR(user_num, item_num, factor_num)`` with ``embed_user`` / ``embed_item`` (``nn.Embedding``, N(0, 0.01^2) init)
  and ``forward(user, item_i, item_j) -> (pred_i, pred_j)``                      BPRMFRecommender.py:28-50
* ``optim.SGD(model.parameters(), lr=, weight_decay=)`` + the five calls of one step
  (zero_grad, forward, loss, backward, step)                                      BPRMFRecommender.py:154,172-176
  -> ``BPRSGD(model, lr=, weight_decay=).step(user, item_i, item_j)``: one fused device step
* the epoch loop of the script body                                               BPRMFRecommender.py:157-181
  -> ``BPRMFRecommender.fit`` (the convenience wrapper the north star names)

The tables stay ordinary ``nn.Embedding`` weights on the CUDA device, so ``torch.save(model)``, ``state_dict`` and
``.cpu()`` keep working; the library updates them in place.  While training, the L2 decay of *untouched* rows is
carried by one scalar (``model.decay_scale``; exact, see DESIGN.md) and folded into the weights by
``model.materialize()`` -- called automatically by ``state_dict``/pickling/``BPRMFRecommender`` epoch ends.
There is no CPU path: without the built library or a CUDA device every call raises.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from ._lib import c_vp


def _as_triples(user, item_i, item_j, device):
    """int32 [B,3] device tensor from the reference's three index tensors (any int dtype / device)."""
    t = torch.stack([torch.as_tensor(user).reshape(-1), torch.as_tensor(item_i).reshape(-1),
                     torch.as_tensor(item_j).reshape(-1)], dim=1)
    return t.to(device=device, dtype=torch.int32, non_blocking=True).contiguous()


class BPR(_lib.HandleOwner, nn.Module):
    """Drop-in for ``class BPR`` (BPRMFRecommender.py:28-50)."""

    _batch_grows = True
    _cpu_error = "BPR tables are on the CPU: call model.cuda() first (no CPU fallback)"

    def __init__(self, user_num, item_num, factor_num, max_batch=4096, eager_decay=False):
        super().__init__()
        self.embed_user = nn.Embedding(user_num, factor_num)
        self.embed_item = nn.Embedding(item_num, factor_num)
        nn.init.normal_(self.embed_user.weight, std=0.01)
        nn.init.normal_(self.embed_item.weight, std=0.01)
        self.user_num, self.item_num, self.factor_num = int(user_num), int(item_num), int(factor_num)
        self._max_batch = int(max_batch)
        self._eager = bool(eager_decay)
        self._pending_scale = 1.0

    # -- library plumbing ---------------------------------------------------------------------
    def _weight(self):
        # straight from _modules: the attribute route (__getattr__ below) would fold the lazy decay in on every step
        return self._modules["embed_user"].weight

    def _handle_dims(self):
        return self.user_num, self.item_num, self.factor_num

    @property
    def _handle_flags(self):
        return _lib.FLAG_EAGER_DECAY if self._eager else 0

    def _tables(self):
        self._device()
        return self._modules["embed_user"].weight, self._modules["embed_item"].weight

    def rank_tables(self):
        return (*self._tables(), None)

    def handle(self, batch=None):
        """The library handle for the tables' current device; re-created when a larger batch arrives, with the lazy
        decay scale of the handle it replaces."""
        h = self._handle
        new = super().handle(batch)
        if new is not h:
            new.scale = self._pending_scale
        return new

    def _close_handle(self):
        if self._handle is not None:
            self._pending_scale = self._handle.scale
        super()._close_handle()

    @property
    def decay_scale(self):
        """c of the lazy L2 decay: true weights = c * stored weights (1.0 after ``materialize``)."""
        return self._handle.scale if self._handle is not None else self._pending_scale

    def materialize(self):
        """Fold the lazy decay scale into the weights (one pass over both tables)."""
        if self._handle is None or self._handle.scale == 1.0:
            return self
        P, Q = self._tables()
        h = self._handle
        _lib.check(h.L.daisy_materialize(h.ptr, c_vp(P.data_ptr()), c_vp(Q.data_ptr()),
                                         _lib.stream_ptr(torch, P.device)))
        return self

    def pin_hot_items(self, n_rows=None, hit_ratio=1.0):
        """Pin rows [0, n_rows) of the item table in L2 through an access-policy window on the current stream
        (``daisy_set_l2_window``): with a popularity-ordered catalogue these are the hot items of the Zipf head.
        ``n_rows=None`` pins the whole item table (as much as the device's persisting-L2 carve-out allows);
        ``n_rows=0`` clears the window."""
        P, Q = self._tables()
        h = self.handle()
        n = self.item_num if n_rows is None else int(n_rows)
        _lib.check(h.L.daisy_set_l2_window(h.ptr, c_vp(Q.data_ptr()), n, float(hit_ratio),
                                           _lib.stream_ptr(torch, P.device)))
        return self

    # -- reference surface --------------------------------------------------------------------
    def forward(self, user, item_i, item_j):
        """(pred_i, pred_j) = (<P[u],Q[i]>, <P[u],Q[j]>)  -- BPRMFRecommender.py:42-50.  Inference only:
        training goes through ``BPRSGD.step`` (one fused kernel pipeline), not autograd."""
        P, Q = self._tables()
        tri = _as_triples(user, item_i, item_j, P.device)
        B = tri.shape[0]
        h = self.handle()
        pred_i = torch.empty(B, dtype=torch.float32, device=P.device)
        pred_j = torch.empty(B, dtype=torch.float32, device=P.device)
        _lib.check(h.L.daisy_bpr_forward(h.ptr, c_vp(P.data_ptr()), c_vp(Q.data_ptr()), c_vp(tri.data_ptr()), B,
                                         c_vp(pred_i.data_ptr()), c_vp(pred_j.data_ptr()),
                                         _lib.stream_ptr(torch, P.device)))
        shape = torch.as_tensor(user).shape
        return pred_i.reshape(shape), pred_j.reshape(shape)

    # State leaving the library's control must carry true weights.  Between two steps the tables hold W / c; every
    # route by which reference-style code reaches them -- ``model.embed_user.weight``, ``parameters()``,
    # ``state_dict()``, pickling, ``.cpu()`` -- folds c in first (one pass over the tables, and only when c != 1).
    # A tensor obtained EARLIER and kept across later steps is the one thing this cannot cover: re-read it.
    def __getattr__(self, name):
        if name in ("embed_user", "embed_item"):
            d = self.__dict__
            h = d.get("_handle")
            if h is not None and h.scale != 1.0:
                self.materialize()
        return super().__getattr__(name)

    def state_dict(self, *args, **kwargs):
        self.materialize()
        return super().state_dict(*args, **kwargs)

    def named_parameters(self, *args, **kwargs):      # parameters() is built on this
        self.materialize()
        return super().named_parameters(*args, **kwargs)

    def load_state_dict(self, state_dict, *args, **kwargs):
        """Loaded weights are TRUE weights: the pending decay scale of whatever the tables held is dropped (the
        reference's restore-the-best-checkpoint pattern after some steps with weight_decay > 0)."""
        out = super().load_state_dict(state_dict, *args, **kwargs)
        if self._handle is not None:
            self._handle.scale = 1.0
        self._pending_scale = 1.0
        return out

    def __getstate__(self):
        self.materialize()
        d = super().__getstate__()
        d["_pending_scale"] = 1.0
        return d

    def _apply(self, fn, *a, **k):
        self.materialize()
        return super()._apply(fn, *a, **k)


class BPRSGD:
    """``optim.SGD(model.parameters(), lr, weight_decay)`` + the training step, fused.

    ``step(user, item_i, item_j)`` == ``model.zero_grad(); pi, pj = model(u, i, j);
    loss = -(pi - pj).sigmoid().log().sum(); loss.backward(); optimizer.step()``  (BPRMFRecommender.py:172-176).
    The batch loss is accumulated on the device; ``loss_sum()`` reads (and optionally clears) it.
    """

    def __init__(self, model: BPR, lr=0.01, weight_decay=0.0):
        self.model = model
        self.lr = float(lr)
        self.weight_decay = float(weight_decay)
        self._loss = None

    def _loss_buf(self, device):
        if self._loss is None or self._loss.device != device:
            self._loss = torch.zeros(1, dtype=torch.float64, device=device)
        return self._loss

    def step(self, user, item_i=None, item_j=None, loss_out=None, ready=False):
        """One fused step.  ``user`` may also be a packed int32 [B,3] tensor: on the device it is used in place;
        on the host (pinned for an asynchronous copy) it goes through ``daisy_bpr_step_host``.
        ``ready=True`` declares that a packed DEVICE tensor is complete at call time (uploaded and synchronised
        earlier), which lets the library overlap this step's bookkeeping with the previous step's kernels
        (``daisy_set_inputs_ready``); host tensors always overlap."""
        m = self.model
        P, Q = m._tables()
        packed = item_i is None
        tri = user if packed else _as_triples(user, item_i, item_j, P.device)
        if packed and (tri.dtype != torch.int32 or tri.dim() != 2 or tri.shape[1] != 3 or not tri.is_contiguous()):
            raise ValueError("packed triples must be a contiguous int32 [B, 3] tensor")
        B = tri.shape[0]
        h = m.handle(B)
        ready = bool(ready and packed and tri.is_cuda)
        if getattr(h, "_ready", False) != ready:
            h.set_inputs_ready(ready)
            h._ready = ready
        loss = self._loss_buf(P.device) if loss_out is None else loss_out
        fn = h.L.daisy_bpr_step if tri.is_cuda else h.L.daisy_bpr_step_host
        _lib.check(fn(h.ptr, c_vp(P.data_ptr()), c_vp(Q.data_ptr()), c_vp(tri.data_ptr()), B, self.lr,
                      self.weight_decay, c_vp(loss.data_ptr()), _lib.stream_ptr(torch, P.device)))

    def epoch(self, triples, batch_size, loss_out=None):
        """Every step of one epoch in ONE library call (``daisy_bpr_epoch``): ``triples`` is the epoch's packed
        int32 [n,3] tensor (device, or pinned host), consumed in consecutive batches of ``batch_size`` -- the loop
        ``for user, item_i, item_j in train_loader`` of BPRMFRecommender.py:162-178.  Same result as calling
        ``step`` per batch; what it saves is the per-call cost of Python, which at the reference's default batch of
        4 096 triples is larger than the ~20 us the step takes on the device."""
        m = self.model
        P, Q = m._tables()
        tri = triples
        if tri.dtype != torch.int32 or tri.dim() != 2 or tri.shape[1] != 3 or not tri.is_contiguous():
            raise ValueError("packed triples must be a contiguous int32 [n, 3] tensor")
        n, batch = tri.shape[0], int(batch_size)
        h = m.handle(min(batch, max(n, 1)))
        loss = self._loss_buf(P.device) if loss_out is None else loss_out
        _lib.check(h.L.daisy_bpr_epoch(h.ptr, c_vp(P.data_ptr()), c_vp(Q.data_ptr()), c_vp(tri.data_ptr()), n, batch,
                                       0 if tri.is_cuda else 1, self.lr, self.weight_decay, c_vp(loss.data_ptr()),
                                       _lib.stream_ptr(torch, P.device)))

    def loss_sum(self, reset=True):
        if self._loss is None:
            return 0.0
        v = float(self._loss.item())
        if reset:
            self._loss.zero_()
        return v

    def zero_grad(self):        # kept so reference-shaped loops still run; there is no dense gradient buffer
        pass


class BPRAdam:
    """Lazy sparse Adam on the BPR loss (only rows present in the batch move; torch.optim.SparseAdam semantics)."""

    def __init__(self, model: BPR, lr=1e-3, betas=(0.9, 0.999), eps=1e-8):
        self.model, self.lr, self.betas, self.eps = model, float(lr), betas, float(eps)
        self.t = 0
        self._loss = None
        self.state = None

    def step(self, user, item_i=None, item_j=None):
        m = self.model
        P, Q = m._tables()
        tri = user if item_i is None else _as_triples(user, item_i, item_j, P.device)
        tri = tri.to(P.device)
        if self.state is None:
            self.state = [torch.zeros_like(P), torch.zeros_like(P), torch.zeros_like(Q), torch.zeros_like(Q)]
            self._loss = torch.zeros(1, dtype=torch.float64, device=P.device)
        m.materialize()
        self.t += 1
        h = m.handle(tri.shape[0])
        mP, vP, mQ, vQ = self.state
        _lib.check(h.L.daisy_bpr_adam_step(h.ptr, c_vp(P.data_ptr()), c_vp(Q.data_ptr()), c_vp(mP.data_ptr()),
                                           c_vp(vP.data_ptr()), c_vp(mQ.data_ptr()), c_vp(vQ.data_ptr()),
                                           c_vp(tri.data_ptr()), tri.shape[0], self.lr, self.betas[0], self.betas[1],
                                           self.eps, self.t, c_vp(self._loss.data_ptr()),
                                           _lib.stream_ptr(torch, P.device)))

    def loss_sum(self, reset=True):
        v = float(self._loss.item()) if self._loss is not None else 0.0
        if reset and self._loss is not None:
            self._loss.zero_()
        return v


class BPRMFRecommender:
    """``fit()/predict()`` wrapper around the script body of BPRMFRecommender.py (argparse defaults :53-116).

    ``fit(train_pairs, eval_users=None, eval_cands=None)`` runs ``epochs`` x [deterministic negative sampling
    (replaces ``ng_sample`` :160), fused steps over shuffled batches of ``batch_size`` (:162-176), optional
    ``metric_eval`` (:181)] and records ``history`` = [{epoch, loss, hr, ndcg, triples_per_s}].
    """

    def __init__(self, user_num, item_num, factor_num=32, lr=0.01, wd=0.001, batch_size=4096, epochs=20, num_ng=4,
                 topk=10, seed=2019, device="cuda", optimizer="sgd", sampler="host"):
        _lib.require_cuda()
        self.user_num, self.item_num, self.factor_num = int(user_num), int(item_num), int(factor_num)
        self.lr, self.wd, self.batch_size, self.epochs = float(lr), float(wd), int(batch_size), int(epochs)
        self.num_ng, self.topk, self.seed = int(num_ng), int(topk), int(seed)
        self.device = torch.device(device)
        torch.manual_seed(self.seed)
        self.model = BPR(user_num, item_num, factor_num, max_batch=batch_size).to(self.device)
        self.optimizer = (BPRSGD(self.model, lr=self.lr, weight_decay=self.wd) if optimizer == "sgd"
                          else BPRAdam(self.model, lr=self.lr))
        self.history = []
        assert sampler in ("host", "device")
        self.sampler = sampler     # "device": negatives drawn on the GPU (daisy_sample_triples), no H2D of triples

    def fit(self, train_pairs, eval_users=None, eval_cands=None, verbose=False):
        import time
        from .metrics import topk_candidates, hr_ndcg
        from .sampler import TripleSampler, DeviceTripleSampler
        on_device = self.sampler == "device"
        if on_device:
            sampler = DeviceTripleSampler(train_pairs, self.item_num, self.user_num, num_ng=self.num_ng,
                                          seed=self.seed, device=self.device)
            n = len(sampler)
            epoch_triples = torch.empty((n, 3), dtype=torch.int32, device=self.device)
        else:
            sampler = TripleSampler(train_pairs, self.item_num, num_ng=self.num_ng, seed=self.seed)
            n = len(sampler)
            epoch_triples = torch.empty((n, 3), dtype=torch.int32).pin_memory()
        for ep in range(self.epochs):
            t0 = time.time()
            if on_device:
                sampler.sample_epoch(ep, out=epoch_triples)
            else:
                epoch_triples.numpy()[:] = sampler.sample_epoch(ep)
            torch.cuda.synchronize(self.device)
            t1 = time.time()
            if isinstance(self.optimizer, BPRSGD):
                self.optimizer.epoch(epoch_triples, self.batch_size)
            else:
                for s in range(0, n, self.batch_size):
                    self.optimizer.step(epoch_triples[s:s + self.batch_size])
            self.model.materialize()
            loss = self.optimizer.loss_sum()          # synchronises
            self.model.check()
            dt = time.time() - t1
            rec = dict(epoch=ep + 1, loss=loss, triples_per_s=n / dt, sample_s=t1 - t0, train_s=dt)
            if eval_users is not None:
                pos, items, _ = topk_candidates(self.model, eval_users, eval_cands, self.topk)
                rec["hr"], rec["ndcg"] = hr_ndcg(pos)
            self.history.append(rec)
            if verbose:
                print(rec, flush=True)
        return self

    def predict(self, user, item):
        """Score(s) <P[u], Q[i]> for scalar or array-like ids (the call of BPRMFRecommender.py:204)."""
        u = torch.as_tensor(np.asarray(user)).reshape(-1)
        i = torch.as_tensor(np.asarray(item)).reshape(-1)
        pi, _ = self.model(u, i, i)
        self.model.check()
        out = pi.cpu().numpy()
        return float(out[0]) if np.ndim(user) == 0 else out

    def recommend(self, users, k=None, exclude=None):
        from .metrics import topk_full
        return topk_full(self.model, users, k or self.topk, exclude)
