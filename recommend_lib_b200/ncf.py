"""Drop-in for ``class NCF`` of the reference in its GMF variant (NCFRecommender.py:28-125) and for the training step
of its script (:255-287), on the C-ABI library (``daisy_gmf_forward`` / ``daisy_gmf_step``, csrc/gmf.cu).

Only ``model='GMF'`` is on the accelerated path (SURVEY.md section 8f, row N3): 'MLP' / 'NeuMF-*' raise.  Host code is
PyTorch for device memory and streams only; there is no CPU fallback.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch
import torch.nn as nn

from . import _lib

c_vp = ctypes.c_void_p


def _samples(user, item, label, device):
    """Pack (user, item[, label]) into the int32 [B,3] layout the library takes (label column 0 when absent)."""
    u = torch.as_tensor(user).reshape(-1)
    i = torch.as_tensor(item).reshape(-1)
    y = torch.zeros_like(u) if label is None else torch.as_tensor(label).reshape(-1)
    if not (u.shape == i.shape == y.shape):
        raise ValueError("user, item and label must have the same length")
    s = torch.stack([u.to(torch.int64), i.to(torch.int64), y.to(torch.float32).round().to(torch.int64)], 1)
    return s.to(device=device, dtype=torch.int32).contiguous()


class NCF(_lib.HandleOwner, nn.Module):
    """``NCF(user_num, item_num, factor_num, num_layers, dropout, model)`` with ``model == 'GMF'``.

    Attributes as in the reference: ``embed_user_GMF``, ``embed_item_GMF`` (``nn.Embedding``, N(0, 0.01^2)) and
    ``predict_layer`` (``nn.Linear(factor_num, 1)``, Kaiming-uniform weight, zero bias; NCFRecommender.py:66-84).
    ``forward(user, item) -> prediction`` (:105-125) runs ``daisy_gmf_forward``; training goes through
    ``GMFAdam.step`` (one fused pipeline), not autograd.
    """

    _batch_grows = True
    _cpu_error = "NCF tables are on the CPU: call model.cuda() first (no CPU fallback)"

    def __init__(self, user_num, item_num, factor_num, num_layers=3, dropout=0.0, model="GMF", GMF_model=None,
                 MLP_model=None, max_batch=256):
        super().__init__()
        if model != "GMF":
            raise NotImplementedError("only model='GMF' is on this (GPU-verified) path; 'MLP' / 'NeuMF-end' are "
                                      "ncf_mlp.NeuMF / NeuMFAdam")
        if factor_num % 4:
            raise ValueError("factor_num must be a multiple of 4 (rows move as 128-bit vectors)")
        self.dropout, self.model = dropout, model
        self.user_num, self.item_num, self.factor_num = int(user_num), int(item_num), int(factor_num)
        self.embed_user_GMF = nn.Embedding(user_num, factor_num)
        self.embed_item_GMF = nn.Embedding(item_num, factor_num)
        self.predict_layer = nn.Linear(factor_num, 1)
        nn.init.normal_(self.embed_user_GMF.weight, std=0.01)
        nn.init.normal_(self.embed_item_GMF.weight, std=0.01)
        nn.init.kaiming_uniform_(self.predict_layer.weight, a=1, nonlinearity="sigmoid")
        self.predict_layer.bias.data.zero_()
        for p in self.parameters():
            p.requires_grad_(False)
        self._max_batch = int(max_batch)

    def _weight(self):
        return self.embed_user_GMF.weight

    def _handle_dims(self):
        return self.user_num, self.item_num, self.factor_num

    def _tensors(self):
        self._device()
        return self.embed_user_GMF.weight, self.embed_item_GMF.weight, self.predict_layer.weight, self.predict_layer.bias

    def _tables(self):
        """(P * w, Q): what the candidate top-K kernel ranks with -- <P[u] * w, Q[i]> = logit - b, and the bias does not
        change a ranking (metrics.metric_eval(..., algo='ncf'), util/metrics.py:68-86)."""
        P, Q, w, _ = self._tensors()
        return (P * w.reshape(1, -1)).contiguous(), Q

    def rank_tables(self):
        return (*self._tables(), None)

    def forward(self, user, item):
        P, Q, w, b = self._tensors()
        s = _samples(user, item, None, P.device)
        B = s.shape[0]
        h = self.handle()
        pred = torch.empty(B, dtype=torch.float32, device=P.device)
        _lib.check(h.L.daisy_gmf_forward(h.ptr, c_vp(P.data_ptr()), c_vp(Q.data_ptr()), c_vp(w.data_ptr()),
                                         c_vp(b.data_ptr()), c_vp(s.data_ptr()), B, c_vp(pred.data_ptr()),
                                         _lib.stream_ptr(torch, P.device)))
        return pred.view(-1)


class GMFAdam:
    """``optim.Adam(model.parameters(), lr)`` + ``BCEWithLogitsLoss`` + the step of NCFRecommender.py:283-287, fused:
    ``step(user, item, label)``.  Torch-default betas / eps; dense Adam over every row (as the reference does).
    ``last_loss()`` reads the mean BCE of the most recent batch."""

    def __init__(self, model: NCF, lr=1e-3, betas=(0.9, 0.999), eps=1e-8):
        self.model, self.lr, self.betas, self.eps = model, float(lr), betas, float(eps)
        self.t = 0
        self.state = None
        self._loss = None

    def step(self, user, item=None, label=None):
        """``step(user, item, label)`` as in the reference loop, or ``step(samples)`` with a packed int32 [B,3] tensor
        (user, item, label) -- on the device it is used in place, from (pinned) host memory it is copied first."""
        m = self.model
        P, Q, w, b = m._tensors()
        if item is None:
            s = user
            if s.dtype != torch.int32 or s.dim() != 2 or s.shape[1] != 3 or not s.is_contiguous():
                raise ValueError("packed samples must be a contiguous int32 [B, 3] tensor")
            if not s.is_cuda:
                s = s.to(P.device, non_blocking=True)
        else:
            s = _samples(user, item, label, P.device)
        B = s.shape[0]
        if self.state is None:
            D = m.factor_num
            self.state = [torch.zeros_like(P), torch.zeros_like(P), torch.zeros_like(Q), torch.zeros_like(Q),
                          torch.zeros(2 * (D + 1), dtype=torch.float32, device=P.device)]
            self._loss = torch.zeros(1, dtype=torch.float64, device=P.device)
        if B == 0:
            return
        self.t += 1
        self._loss.zero_()
        h = m.handle(B)
        mP, vP, mQ, vQ, mwb = self.state
        _lib.check(h.L.daisy_gmf_step(h.ptr, c_vp(P.data_ptr()), c_vp(Q.data_ptr()), c_vp(w.data_ptr()), c_vp(b.data_ptr()),
                                      c_vp(mP.data_ptr()), c_vp(vP.data_ptr()), c_vp(mQ.data_ptr()), c_vp(vQ.data_ptr()),
                                      c_vp(mwb.data_ptr()), c_vp(s.data_ptr()), B, self.lr, self.betas[0], self.betas[1],
                                      self.eps, self.t, c_vp(self._loss.data_ptr()), _lib.stream_ptr(torch, P.device)))

    def epoch(self, samples, batch_size):
        """All steps of one epoch in ONE library call (``daisy_gmf_epoch``): ``samples`` is the epoch's packed int32
        [n,3] tensor (device or pinned host), consumed in consecutive batches -- the loop of NCFRecommender.py:268-288.
        ``last_loss()`` then returns the SUM of the batches' mean losses."""
        m = self.model
        P, Q, w, b = m._tensors()
        s = samples
        if s.dtype != torch.int32 or s.dim() != 2 or s.shape[1] != 3 or not s.is_contiguous():
            raise ValueError("packed samples must be a contiguous int32 [n, 3] tensor")
        n, batch = s.shape[0], int(batch_size)
        if self.state is None:
            D = m.factor_num
            self.state = [torch.zeros_like(P), torch.zeros_like(P), torch.zeros_like(Q), torch.zeros_like(Q),
                          torch.zeros(2 * (D + 1), dtype=torch.float32, device=P.device)]
            self._loss = torch.zeros(1, dtype=torch.float64, device=P.device)
        if n == 0:
            return
        self._loss.zero_()
        h = m.handle(min(batch, n))
        mP, vP, mQ, vQ, mwb = self.state
        _lib.check(h.L.daisy_gmf_epoch(h.ptr, c_vp(P.data_ptr()), c_vp(Q.data_ptr()), c_vp(w.data_ptr()), c_vp(b.data_ptr()),
                                       c_vp(mP.data_ptr()), c_vp(vP.data_ptr()), c_vp(mQ.data_ptr()), c_vp(vQ.data_ptr()),
                                       c_vp(mwb.data_ptr()), c_vp(s.data_ptr()), n, batch, 0 if s.is_cuda else 1, self.lr,
                                       self.betas[0], self.betas[1], self.eps, self.t + 1, c_vp(self._loss.data_ptr()),
                                       _lib.stream_ptr(torch, P.device)))
        self.t += (n + batch - 1) // batch

    def last_loss(self):
        return float(self._loss.item()) if self._loss is not None else 0.0

    def zero_grad(self):
        pass
