"""BPR-FM at the reference script's DEFAULTS -- batch norm + dropout on the FM vector (BPRFMRecommender.py:45-80, 116-125)
-- on the C-ABI library (``daisy_fmbn_step`` / ``daisy_fmbn_forward``, and ``daisy_fmbn_rank_tables`` for ranking;
csrc/fmbn.cu).  SURVEY.md section 8f, row N3.

``bprfm.BPRFM(batch_norm=True, ...)`` builds this class (and ``FMAdagrad`` on it the optimiser below), so the reference's
one constructor covers both configurations.  Parity: tests/test_bprfm_bn_gpu.py against the golden run of the unmodified
reference class and ``oracle/bprfm_oracle.py: BPRFMFull``.

Same module structure as the reference class, so ``state_dict()`` / ``torch.save(model)`` carry the same keys:
``embeddings``, ``biases``, ``bias_``, ``FM_layers = Sequential(BatchNorm1d(num_factors), Dropout(drop_prob[0]))``.
The library updates those tensors in place.  Feature layout of the script: ``features = [user, user_num + item]``,
``feature_values = [1, 1]`` (util/data_loader.py:159-172, 595-614); anything else raises.  No CPU fallback.
"""
from __future__ import annotations

import ctypes

import torch
import torch.nn as nn

from . import _lib
from .bprfm import BPRFM

c_vp = ctypes.c_void_p


class BPRFMBN(_lib.HandleOwner, nn.Module):
    """``BPRFM(num_features, num_factors, batch_norm=True, drop_prob, user_num=...)`` (BPRFMRecommender.py:29-55)."""

    _cpu_error = "BPRFMBN tables are on the CPU: call model.cuda() first (no CPU fallback)"
    user_term = BPRFM.user_term

    def __init__(self, num_features, num_factors, batch_norm=True, drop_prob=(0.5, 0.2), user_num=None, max_batch=4096):
        super().__init__()
        if not batch_norm:
            raise NotImplementedError("batch_norm=False is bprfm.BPRFM (dropout 0) -- this class is the batch-norm path")
        if user_num is None or not (0 < int(user_num) < int(num_features)):
            raise ValueError("user_num (features [0, user_num) are users, the rest items) is required")
        if not (1 <= int(num_factors) <= 255):
            raise ValueError("num_factors must be in 1..255")
        if not (0.0 <= float(drop_prob[0]) < 1.0):
            raise ValueError("drop_prob[0] must be in [0, 1)")
        self.num_features, self.num_factors = int(num_features), int(num_factors)
        self.user_num, self.item_num = int(user_num), int(num_features) - int(user_num)
        self.batch_norm, self.drop_prob = True, list(drop_prob)
        self.embeddings = nn.Embedding(num_features, num_factors)
        self.biases = nn.Embedding(num_features, 1)
        self.bias_ = nn.Parameter(torch.tensor([0.0]))
        self.FM_layers = nn.Sequential(nn.BatchNorm1d(num_factors), nn.Dropout(float(drop_prob[0])))   # :47-52
        nn.init.normal_(self.embeddings.weight, std=0.01)
        nn.init.constant_(self.biases.weight, 0.0)
        for p in self.parameters():
            p.requires_grad_(False)

    # -- plumbing -----------------------------------------------------------------------------------------------------
    def _weight(self):
        return self.embeddings.weight

    def _handle_dims(self):
        # the step and the forward read the device, the error flag and the launch counter; the ranking entry points
        # also read the row width of the folded tables (rank_tables)
        return self.user_num, self.item_num, self.rank_width

    def params(self, lr=0.0, eps=1e-10, state=None):
        """The ``daisy_fmbn_params`` block over this module's tensors (+ an optimizer's state_sum tensors)."""
        bn = self.FM_layers[0]
        for t in (self.embeddings.weight, self.biases.weight, bn.weight, bn.bias, bn.running_mean, bn.running_var):
            if t.dtype != torch.float32 or not t.is_contiguous():
                raise _lib.DaisyError("BPRFMBN tensors must be contiguous float32")
        ptr = lambda t: c_vp(t.data_ptr()) if t is not None else None
        st = state or {}
        return _lib.FMBNParams(ptr(self.embeddings.weight), ptr(self.biases.weight), ptr(st.get("accE")), ptr(st.get("accb")),
                               ptr(bn.weight), ptr(bn.bias), ptr(st.get("acc_gamma")), ptr(st.get("acc_beta")),
                               ptr(bn.running_mean), ptr(bn.running_var), float(lr), float(eps), float(bn.eps),
                               float(bn.momentum if bn.momentum is not None else 0.1), self.user_num, self.num_features,
                               self.num_factors)

    def triples(self, features_i, feature_values_i, features_j, feature_values_j):
        """(user, item_i, item_j) int32 [B,3] on the device from the loader's tensors; validates the feature layout."""
        fi, fj = torch.as_tensor(features_i), torch.as_tensor(features_j)
        if fi.dim() != 2 or fi.shape[1] != 2 or fj.shape != fi.shape:
            raise ValueError("features must be [B, 2]: (user feature, item feature)")
        if not bool((fi[:, 0] == fj[:, 0]).all()):
            raise ValueError("features_i and features_j must carry the same user feature")
        for v in (feature_values_i, feature_values_j):
            if v is not None and not bool((torch.as_tensor(v) == 1).all()):
                raise NotImplementedError("feature values other than 1 are not on the accelerated path")
        t = torch.stack([fi[:, 0], fi[:, 1] - self.user_num, fj[:, 1] - self.user_num], 1)
        return t.to(device=self._device(), dtype=torch.int32).contiguous()

    # -- reference surface --------------------------------------------------------------------------------------------
    def forward(self, features_i, feature_values_i, features_j, feature_values_j):
        """(pred_i, pred_j) in evaluation mode (running statistics, no dropout) -- BPRFMRecommender.py:57-80 after
        ``model.eval()``.  Training goes through ``FMBNAdagrad.step`` (the fused step); a training-mode forward raises."""
        if self.training:
            raise RuntimeError("training-mode forward is fused into FMBNAdagrad.step; call model.eval() to predict")
        dev = self._device()
        tri = self.triples(features_i, feature_values_i, features_j, feature_values_j)
        B = tri.shape[0]
        h = self.handle()
        pi = torch.empty(B, dtype=torch.float32, device=dev)
        pj = torch.empty(B, dtype=torch.float32, device=dev)
        prm = self.params()
        _lib.check(h.L.daisy_fmbn_forward(h.ptr, ctypes.byref(prm), c_vp(tri.data_ptr()), B, c_vp(pi.data_ptr()),
                                          c_vp(pj.data_ptr()), _lib.stream_ptr(torch, dev)))
        extra = self.biases.weight[tri[:, 0].long(), 0] + self.bias_          # user bias + global bias: the same in both
        return (pi + extra).view(-1), (pj + extra).view(-1)

    @property
    def rank_width(self):
        """Row width W of the ranking tables: F + 1 rounded up to a multiple of 4 (the ranking kernels read 16-byte rows)."""
        return (self.num_factors + 4) // 4 * 4

    def rank_tables(self):
        """(P [user_num, W], Q [item_num, W], c0 [1]): the evaluation-mode score folded into a dot product,
        ``forward()``'s score = <P[u], Q[i]> + b_u + bias_ + c0 (``daisy_fmbn_rank_tables``).  Folded anew on every call,
        since training moves the weights and the running statistics."""
        if self.training:
            raise RuntimeError("training-mode forward is fused into FMBNAdagrad.step; call model.eval() to predict")
        dev = self._device()
        h = self.handle()
        W = self.rank_width
        P = torch.empty((self.user_num, W), dtype=torch.float32, device=dev)
        Q = torch.empty((self.item_num, W), dtype=torch.float32, device=dev)
        c0 = torch.empty(1, dtype=torch.float32, device=dev)
        prm = self.params()
        _lib.check(h.L.daisy_fmbn_rank_tables(h.ptr, ctypes.byref(prm), W, c_vp(P.data_ptr()), c_vp(Q.data_ptr()),
                                              c_vp(c0.data_ptr()), _lib.stream_ptr(torch, dev)))
        return P, Q, c0


class FMBNAdagrad:
    """``optim.Adagrad(model.parameters(), lr, initial_accumulator_value=1e-8)`` + the step of
    BPRFMRecommender.py:214-219, fused: ``step(features_i, feature_values_i, features_j, feature_values_j)``.

    ``mask_i`` / ``mask_j`` ([B, F], kept elements already scaled by 1 / (1 - p)) replace the dropout draw -- that is how
    the parity tests feed the masks the reference drew; without them and with ``drop_prob[0] > 0`` the masks are drawn
    on the device from torch's CUDA generator (seed it with ``torch.manual_seed`` for reproducible runs)."""

    def __init__(self, model: BPRFMBN, lr=0.05, initial_accumulator_value=1e-8, eps=1e-10):
        self.model, self.lr, self.eps = model, float(lr), float(eps)
        self.init_acc = float(initial_accumulator_value)
        self.state = None
        self._scratch = None
        self._loss = None

    def _ensure(self, B):
        m = self.model
        dev = m._device()
        bn = m.FM_layers[0]
        if self.state is None or self.state["accE"].device != dev:
            full = lambda t: torch.full_like(t, self.init_acc)
            self.state = dict(accE=full(m.embeddings.weight), accb=full(m.biases.weight), acc_gamma=full(bn.weight),
                              acc_beta=full(bn.bias))
            self._loss = torch.zeros(1, dtype=torch.float64, device=dev)
            self._scratch = None
        need = ctypes.c_int64()
        _lib.check(m.handle().L.daisy_fmbn_scratch_bytes(int(B), m.num_factors, ctypes.byref(need)))
        if self._scratch is None or self._scratch.numel() < need.value or self._scratch.device != dev:
            self._scratch = torch.empty(need.value, dtype=torch.uint8, device=dev)     # torch allocations are 512-B aligned
        return need.value

    def step(self, features_i, feature_values_i=None, features_j=None, feature_values_j=None, mask_i=None, mask_j=None):
        m = self.model
        dev = m._device()
        if features_j is None and torch.is_tensor(features_i) and features_i.dtype == torch.int32 and features_i.device == dev:
            tri = features_i                          # packed (user, item_i, item_j) int32 [B,3], item ids relative
            if tri.dim() != 2 or tri.shape[1] != 3 or not tri.is_contiguous():
                raise ValueError("packed triples must be a contiguous int32 [B, 3] device tensor")
        else:
            tri = m.triples(features_i, feature_values_i, features_j, feature_values_j)
        B, F = tri.shape[0], m.num_factors
        if B == 0:
            return
        p = float(m.drop_prob[0])
        if (mask_i is None) != (mask_j is None):
            raise ValueError("give both dropout masks or neither")
        if mask_i is None and p > 0.0:
            keep = torch.full((2, B, F), 1.0 - p, dtype=torch.float32, device=dev)
            masks = torch.bernoulli(keep).div_(1.0 - p)
            mask_i, mask_j = masks[0], masks[1]
        if mask_i is not None:
            mask_i = torch.as_tensor(mask_i).to(device=dev, dtype=torch.float32).contiguous()
            mask_j = torch.as_tensor(mask_j).to(device=dev, dtype=torch.float32).contiguous()
            if mask_i.shape != (B, F) or mask_j.shape != (B, F):
                raise ValueError(f"dropout masks must be [{B}, {F}]")
        nbytes = self._ensure(B)
        h = m.handle()
        prm = m.params(self.lr, self.eps, self.state)
        _lib.check(h.L.daisy_fmbn_step(h.ptr, ctypes.byref(prm), c_vp(tri.data_ptr()), B,
                                       c_vp(mask_i.data_ptr()) if mask_i is not None else None,
                                       c_vp(mask_j.data_ptr()) if mask_j is not None else None,
                                       c_vp(self._scratch.data_ptr()), nbytes, c_vp(self._loss.data_ptr()),
                                       _lib.stream_ptr(torch, dev)))
        m.FM_layers[0].num_batches_tracked += 2      # two _out calls per step (:57-59), one update each

    def loss_sum(self, reset=True):
        if self._loss is None:
            return 0.0
        v = float(self._loss.item())
        if reset:
            self._loss.zero_()
        return v

    def zero_grad(self):
        pass
