"""Drop-in for ``class BPRFM`` of the reference (BPRFMRecommender.py:29-80) with two one-hot features per example and
for the training step of its script (:191-193, 214-219), on the C-ABI library (``daisy_bprfm_adagrad_step``,
``daisy_bpr_forward``).  SURVEY.md section 8f, row N3.

Accelerated configuration: ``batch_norm=False``, ``drop_prob=[0, 0]`` (dropout draws from torch's global generator inside
``forward``, so no two runs of the reference agree either; batch-norm is outside the gather/score/scatter path) and the
feature layout the script builds: ``features = [user, user_num + item]``, ``feature_values = [1, 1]``
(util/data_loader.py:159-172, 595-614).  Anything else raises.  No CPU fallback.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch
import torch.nn as nn

from . import _lib

c_vp = ctypes.c_void_p


class BPRFM(_lib.HandleOwner, nn.Module):
    """``BPRFM(num_features, num_factors, batch_norm, drop_prob, user_num=...)``: attributes ``embeddings``, ``biases``,
    ``bias_`` as in the reference (:45-55).  ``user_num`` (features ``[0, user_num)`` are users, the rest items) is the
    one extra argument the accelerated path needs.

    The library trains on AUGMENTED rows ``[e_0 .. e_{F-1}, x, 0, 0, 0]`` (x = 1 for users, the item bias for items), so
    that the bias term and its gradient ride through the BPR kernels; ``embeddings.weight`` / ``biases.weight`` are
    refreshed from that buffer whenever they are read through ``forward``, ``state_dict`` or ``sync()``.
    """

    _batch_grows = True
    _cpu_error = "BPRFM tables are on the CPU: call model.cuda() first (no CPU fallback)"

    def __new__(cls, num_features=None, num_factors=None, batch_norm=False, drop_prob=(0.0, 0.0), *args, **kwargs):
        # the reference has ONE class (BPRFMRecommender.py:29-55) and the script's defaults are batch_norm=True,
        # drop_prob=[0.5, 0.2] (:116-125): that configuration is the batch-norm + dropout step of csrc/fmbn.cu
        if cls is BPRFM and batch_norm:
            from .bprfm_bn import BPRFMBN
            return BPRFMBN(num_features, num_factors, True, drop_prob, *args, **kwargs)
        return super().__new__(cls)

    def __init__(self, num_features, num_factors, batch_norm=False, drop_prob=(0.0, 0.0), user_num=None, max_batch=4096):
        super().__init__()
        if batch_norm or any(float(p) != 0.0 for p in drop_prob):
            raise NotImplementedError("dropout without batch norm is not on an accelerated path (the script cannot select "
                                      "it: --batch_norm is on by default and has no off switch, BPRFMRecommender.py:116-125)")
        if user_num is None or not (0 < int(user_num) < int(num_features)):
            raise ValueError("user_num (features [0, user_num) are users, the rest items) is required")
        if num_factors % 4:
            raise ValueError("num_factors must be a multiple of 4 (rows move as 128-bit vectors)")
        self.num_features, self.num_factors = int(num_features), int(num_factors)
        self.user_num, self.item_num = int(user_num), int(num_features) - int(user_num)
        self.batch_norm, self.drop_prob = False, list(drop_prob)
        self.embeddings = nn.Embedding(num_features, num_factors)
        self.biases = nn.Embedding(num_features, 1)
        self.bias_ = nn.Parameter(torch.tensor([0.0]))
        nn.init.normal_(self.embeddings.weight, std=0.01)
        nn.init.constant_(self.biases.weight, 0.0)
        for p in self.parameters():
            p.requires_grad_(False)
        self._max_batch = int(max_batch)
        self._aug = None        # [num_features, F + 4] device buffer the library trains on
        self._dirty = False     # _aug is newer than embeddings / biases

    def _weight(self):
        return self.embeddings.weight

    def _handle_dims(self):
        return self.user_num, self.item_num, self.num_factors + 4

    # -- augmented layout ---------------------------------------------------------------------------------------------
    def pack(self):
        """Build the augmented buffer from embeddings / biases (after the weights were set from outside)."""
        dev = self._device()
        F, U = self.num_factors, self.user_num
        aug = torch.zeros((self.num_features, F + 4), dtype=torch.float32, device=dev)
        aug[:, :F] = self.embeddings.weight
        aug[:U, F] = 1.0
        aug[U:, F] = self.biases.weight[U:, 0]
        self._aug, self._dirty = aug, False
        return aug

    def sync(self):
        """Write the trained rows back into embeddings.weight / biases.weight (item biases; user biases never move)."""
        if self._aug is not None and self._dirty:
            F, U = self.num_factors, self.user_num
            with torch.no_grad():
                self.embeddings.weight.copy_(self._aug[:, :F])
                self.biases.weight[U:, 0] = self._aug[U:, F]
            self._dirty = False
        return self

    def triples(self, features_i, feature_values_i, features_j, feature_values_j):
        """(user, item_i, item_j) int32 [B,3] on the device from the loader's tensors; validates the feature layout."""
        fi, fj = torch.as_tensor(features_i), torch.as_tensor(features_j)
        if fi.dim() != 2 or fi.shape[1] != 2 or fj.shape != fi.shape:
            raise ValueError("features must be [B, 2]: (user feature, item feature)")
        for v in (feature_values_i, feature_values_j):
            if v is not None and not bool((torch.as_tensor(v) == 1).all()):
                raise NotImplementedError("feature values other than 1 are not on the accelerated path")
        dev = self._device()
        t = torch.stack([fi[:, 0], fi[:, 1] - self.user_num, fj[:, 1] - self.user_num], 1)
        return t.to(device=dev, dtype=torch.int32).contiguous()

    # -- reference surface --------------------------------------------------------------------------------------------
    def forward(self, features_i, feature_values_i, features_j, feature_values_j):
        """(pred_i, pred_j)  -- BPRFMRecommender.py:57-80."""
        dev = self._device()
        if self._aug is None:
            self.pack()
        tri = self.triples(features_i, feature_values_i, features_j, feature_values_j)
        B = tri.shape[0]
        h = self.handle()
        P = self._aug
        Q = self._aug[self.user_num:]
        pi = torch.empty(B, dtype=torch.float32, device=dev)
        pj = torch.empty(B, dtype=torch.float32, device=dev)
        _lib.check(h.L.daisy_bpr_forward(h.ptr, c_vp(P.data_ptr()), c_vp(Q.data_ptr()), c_vp(tri.data_ptr()), B,
                                         c_vp(pi.data_ptr()), c_vp(pj.data_ptr()), _lib.stream_ptr(torch, dev)))
        extra = self.biases.weight[tri[:, 0].long(), 0] + self.bias_          # user bias + global bias: the same in both
        return (pi + extra).view(-1), (pj + extra).view(-1)

    def rank_tables(self):
        """(P, Q, None): the augmented rows the library trains on, so that ``forward()``'s score is
        <P[u], Q[i]> + b_u + bias_.  Views of the training buffer: no copy, and unsynced training is included."""
        if self._aug is None:
            self.pack()
        return self._aug, self._aug[self.user_num:], None

    def user_term(self, users, c0):
        """b_u + bias_ (+ c0) per ranked user: what ``forward()`` adds to every item of a user (c0: the batch-norm model's
        share, ``BPRFMBN.rank_tables``).  Gathers by user id, so call it only after ``check()``."""
        off = self.biases.weight[users.long(), 0] + self.bias_
        return off if c0 is None else off + c0

    def state_dict(self, *args, **kwargs):
        self.sync()
        return super().state_dict(*args, **kwargs)

    def __getstate__(self):
        self.sync()
        d = super().__getstate__()
        d["_aug"], d["_dirty"] = None, False
        return d

    def _apply(self, fn, *a, **k):
        self.sync()
        self._aug = None
        return super()._apply(fn, *a, **k)


class FMAdagrad:
    """``optim.Adagrad(model.parameters(), lr, initial_accumulator_value=1e-8)`` + the step of
    BPRFMRecommender.py:214-219, fused: ``step(features_i, feature_values_i, features_j, feature_values_j)``.
    Adagrad moves only elements with a gradient, so the fused sparse step equals the reference's dense one."""

    def __new__(cls, model=None, *args, **kwargs):
        from .bprfm_bn import BPRFMBN, FMBNAdagrad
        if cls is FMAdagrad and isinstance(model, BPRFMBN):        # BPRFM(batch_norm=True) built a BPRFMBN
            return FMBNAdagrad(model, *args, **kwargs)
        return super().__new__(cls)

    def __init__(self, model: BPRFM, lr=0.05, initial_accumulator_value=1e-8, eps=1e-10):
        self.model, self.lr, self.eps = model, float(lr), float(eps)
        self.init_acc = float(initial_accumulator_value)
        self.acc = None
        self._loss = None

    def step(self, features_i, feature_values_i=None, features_j=None, feature_values_j=None):
        m = self.model
        dev = m._device()
        if m._aug is None:
            m.pack()
        if self.acc is None or self.acc.shape != m._aug.shape or self.acc.device != m._aug.device:
            self.acc = torch.full_like(m._aug, self.init_acc)
            self._loss = torch.zeros(1, dtype=torch.float64, device=dev)
        if features_j is None and torch.is_tensor(features_i) and features_i.dtype == torch.int32 and features_i.is_cuda:
            tri = features_i                          # packed (user, item_i, item_j) int32 [B,3], item ids relative
            if tri.dim() != 2 or tri.shape[1] != 3 or not tri.is_contiguous():
                raise ValueError("packed triples must be a contiguous int32 [B, 3] device tensor")
        else:
            tri = m.triples(features_i, feature_values_i, features_j, feature_values_j)
        B = tri.shape[0]
        h = m.handle(B)
        _lib.check(h.L.daisy_bprfm_adagrad_step(h.ptr, c_vp(m._aug.data_ptr()), c_vp(self.acc.data_ptr()),
                                                c_vp(tri.data_ptr()), B, self.lr, self.eps, c_vp(self._loss.data_ptr()),
                                                _lib.stream_ptr(torch, dev)))
        m._dirty = True

    def loss_sum(self, reset=True):
        if self._loss is None:
            return 0.0
        v = float(self._loss.item())
        if reset:
            self._loss.zero_()
        return v

    def zero_grad(self):
        pass
