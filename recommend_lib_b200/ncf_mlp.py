"""Drop-in for ``class NCF`` of the reference with an MLP tower -- ``model='MLP'`` and the script's default
``model='NeuMF-end'`` (NCFRecommender.py:28-125, 175-178), dropout 0 -- and for the training step of its script
(:255-260, 283-287), on the C-ABI library (``daisy_neumf_forward`` / ``daisy_neumf_step``, csrc/neumf.cu).
SURVEY.md section 8f, row N3.  The GMF variant is ``ncf.NCF`` / ``GMFAdam``.

GPU-verified in round 2 (tests/test_neumf_gpu.py, part of the default ``-m gpu`` suite); outside the scope table
(SURVEY 2 #13), kept because it exists.  The checker is the NeuMF checker under ``oracle/``, pinned to the unmodified
reference class; the same translation unit passes it under the host emulation of tests/emu.

Same module structure as the reference (all four embedding tables, ``MLP_layers = Sequential(Dropout, Linear, ReLU, ...)``,
``predict_layer``), so ``state_dict()`` / ``torch.save(model)`` carry the same keys.  No CPU fallback.
"""
from __future__ import annotations

import ctypes

import torch
import torch.nn as nn

from . import _lib
from .ncf import _samples

c_vp = ctypes.c_void_p


class NeuMF(_lib.HandleOwner, nn.Module):
    """``NCF(user_num, item_num, factor_num, num_layers, dropout, model)`` with ``model in ('MLP', 'NeuMF-end')``;
    initialisation as ``_init_weight_`` (:68-84).  ``forward(user, item) -> prediction`` (:105-125)."""

    _cpu_error = "NCF tables are on the CPU: call model.cuda() first (no CPU fallback)"
    bpr_topk = False        # _bpr_topk calls model(user, item_i, item_j), which NCF does not take

    def __init__(self, user_num, item_num, factor_num, num_layers=3, dropout=0.0, model="NeuMF-end", GMF_model=None,
                 MLP_model=None):
        super().__init__()
        if model not in ("MLP", "NeuMF-end"):
            raise NotImplementedError("model must be 'MLP' or 'NeuMF-end' here ('GMF' is ncf.NCF; 'NeuMF-pre' only differs "
                                      "in its initialisation from pre-trained models and is not wired)")
        if float(dropout) != 0.0:
            raise NotImplementedError("dropout other than 0 (the script's default) is not on the accelerated path")
        if not (1 <= int(num_layers) <= _lib.NEUMF_MAX_LAYERS) or int(factor_num) * 2 ** int(num_layers) > 1024:
            raise ValueError("num_layers must be in 1..6 and factor_num * 2^num_layers <= 1024")
        self.dropout, self.model = dropout, model
        self.user_num, self.item_num = int(user_num), int(item_num)
        self.factor_num, self.num_layers = int(factor_num), int(num_layers)
        self.embed_user_GMF = nn.Embedding(user_num, factor_num)
        self.embed_item_GMF = nn.Embedding(item_num, factor_num)
        self.embed_user_MLP = nn.Embedding(user_num, factor_num * (2 ** (num_layers - 1)))
        self.embed_item_MLP = nn.Embedding(item_num, factor_num * (2 ** (num_layers - 1)))
        mods = []
        for i in range(num_layers):                                        # :51-57
            input_size = factor_num * (2 ** (num_layers - i))
            mods += [nn.Dropout(p=self.dropout), nn.Linear(input_size, input_size // 2), nn.ReLU()]
        self.MLP_layers = nn.Sequential(*mods)
        self.predict_layer = nn.Linear(factor_num if model == "MLP" else factor_num * 2, 1)
        for e in (self.embed_user_GMF, self.embed_item_GMF, self.embed_user_MLP, self.embed_item_MLP):
            nn.init.normal_(e.weight, std=0.01)
        for m in self.MLP_layers:
            if isinstance(m, nn.Linear):
                nn.init.xavier_uniform_(m.weight)
        nn.init.kaiming_uniform_(self.predict_layer.weight, a=1, nonlinearity="sigmoid")
        for m in self.modules():
            if isinstance(m, nn.Linear) and m.bias is not None:
                m.bias.data.zero_()
        for p in self.parameters():
            p.requires_grad_(False)

    # -- plumbing -----------------------------------------------------------------------------------------------------
    def _weight(self):
        return self.embed_user_MLP.weight

    def _handle_dims(self):
        return self.user_num, self.item_num, 4          # device, error flag, launch counter

    def linears(self):
        return [m for m in self.MLP_layers if isinstance(m, nn.Linear)]

    def tensors(self):
        """Every parameter the step touches, in the optimizer's order: name -> tensor."""
        t = {}
        if self.model != "MLP":
            t["Pg"], t["Qg"] = self.embed_user_GMF.weight, self.embed_item_GMF.weight
        t["Pm"], t["Qm"] = self.embed_user_MLP.weight, self.embed_item_MLP.weight
        for l, m in enumerate(self.linears()):
            t[f"W{l}"], t[f"b{l}"] = m.weight, m.bias
        t["wp"], t["bp"] = self.predict_layer.weight, self.predict_layer.bias
        return t

    def params(self, lr=0.0, betas=(0.9, 0.999), eps=1e-8, moments=None):
        """The ``daisy_neumf_params`` block over this module's tensors (+ an optimizer's moment tensors)."""
        t = self.tensors()
        for v in t.values():
            if v.dtype != torch.float32 or not v.is_contiguous():
                raise _lib.DaisyError("NCF tensors must be contiguous float32")
        mo = moments or {}
        L = self.num_layers
        ptr = lambda x: c_vp(x.data_ptr()) if x is not None else None
        arr = lambda xs: (c_vp * _lib.NEUMF_MAX_LAYERS)(*[x.data_ptr() if x is not None else None for x in xs],
                                                        *([None] * (_lib.NEUMF_MAX_LAYERS - L)))
        mv = lambda k, j: mo[k][j] if k in mo else None
        return _lib.NeuMFParams(
            int(self.model != "MLP"), L, self.factor_num, self.user_num, self.item_num,
            ptr(t.get("Pg")), ptr(t.get("Qg")), ptr(t["Pm"]), ptr(t["Qm"]),
            arr([t[f"W{l}"] for l in range(L)]), arr([t[f"b{l}"] for l in range(L)]), ptr(t["wp"]), ptr(t["bp"]),
            ptr(mv("Pg", 0)), ptr(mv("Pg", 1)), ptr(mv("Qg", 0)), ptr(mv("Qg", 1)), ptr(mv("Pm", 0)), ptr(mv("Pm", 1)),
            ptr(mv("Qm", 0)), ptr(mv("Qm", 1)),
            arr([mv(f"W{l}", 0) for l in range(L)]), arr([mv(f"W{l}", 1) for l in range(L)]),
            arr([mv(f"b{l}", 0) for l in range(L)]), arr([mv(f"b{l}", 1) for l in range(L)]),
            ptr(mv("wp", 0)), ptr(mv("wp", 1)), ptr(mv("bp", 0)), ptr(mv("bp", 1)),
            float(lr), float(betas[0]), float(betas[1]), float(eps))

    # -- reference surface --------------------------------------------------------------------------------------------
    def forward(self, user, item):
        dev = self._device()
        s = _samples(user, item, None, dev)
        B = s.shape[0]
        h = self.handle()
        pred = torch.empty(B, dtype=torch.float32, device=dev)
        prm = self.params()
        _lib.check(h.L.daisy_neumf_forward(h.ptr, ctypes.byref(prm), c_vp(s.data_ptr()), B, c_vp(pred.data_ptr()),
                                           _lib.stream_ptr(torch, dev)))
        return pred.view(-1)

    # -- ranking: the tower's scores through daisy_neumf_topk_candidates / daisy_neumf_topk_full ----------------------
    def rank_candidates(self, users, cands, top_k):
        h = self.handle()
        N, C = cands.shape
        dev = users.device
        pos = torch.empty((N, top_k), dtype=torch.int32, device=dev)
        items = torch.empty((N, top_k), dtype=torch.int32, device=dev)
        scores = torch.empty((N, top_k), dtype=torch.float32, device=dev)
        prm = self.params()
        _lib.check(h.L.daisy_neumf_topk_candidates(h.ptr, ctypes.byref(prm), c_vp(users.data_ptr()), c_vp(cands.data_ptr()),
                                                   N, C, int(top_k), c_vp(pos.data_ptr()), c_vp(items.data_ptr()),
                                                   c_vp(scores.data_ptr()), _lib.stream_ptr(torch, dev)))
        self.check()
        return pos, items, scores

    def rank_full(self, users, k, excl):
        h = self.handle()
        N = users.shape[0]
        dev = users.device
        ptr, idx = excl
        items = torch.empty((N, k), dtype=torch.int32, device=dev)
        scores = torch.empty((N, k), dtype=torch.float32, device=dev)
        prm = self.params()
        _lib.check(h.L.daisy_neumf_topk_full(h.ptr, ctypes.byref(prm), c_vp(users.data_ptr()), N, int(k),
                                             c_vp(ptr.data_ptr()) if ptr is not None else None,
                                             c_vp(idx.data_ptr()) if idx is not None and idx.numel() else None,
                                             c_vp(items.data_ptr()), c_vp(scores.data_ptr()), _lib.stream_ptr(torch, dev)))
        self.check()
        return items, scores


class NeuMFAdam:
    """``optim.Adam(model.parameters(), lr)`` (:260) + the step of :283-287 with ``nn.BCEWithLogitsLoss()`` (:255), fused:
    ``step(user, item, label)``.  Parameters without a gradient (the GMF tables of model 'MLP') are left alone, as torch's
    Adam leaves parameters whose ``.grad`` is None."""

    def __init__(self, model: NeuMF, lr=1e-3, betas=(0.9, 0.999), eps=1e-8):
        self.model, self.lr, self.betas, self.eps = model, float(lr), (float(betas[0]), float(betas[1])), float(eps)
        self.t = 0
        self.moments = None
        self._scratch = None
        self._loss = None

    def step(self, user, item, label):
        m = self.model
        dev = m._device()
        s = _samples(user, item, label, dev)
        B = s.shape[0]
        if B == 0:
            return
        if self.moments is None or next(iter(self.moments.values()))[0].device != dev:
            self.moments = {k: (torch.zeros_like(v), torch.zeros_like(v)) for k, v in m.tensors().items()}
            self._loss = torch.zeros(1, dtype=torch.float64, device=dev)
            self._scratch = None
        h = m.handle()
        prm = m.params(self.lr, self.betas, self.eps, self.moments)
        need = ctypes.c_int64()
        _lib.check(h.L.daisy_neumf_scratch_bytes(ctypes.byref(prm), B, ctypes.byref(need)))
        if self._scratch is None or self._scratch.numel() < need.value:
            self._scratch = torch.empty(need.value, dtype=torch.uint8, device=dev)
        self.t += 1
        _lib.check(h.L.daisy_neumf_step(h.ptr, ctypes.byref(prm), c_vp(s.data_ptr()), B, self.t, c_vp(self._scratch.data_ptr()),
                                        need.value, c_vp(self._loss.data_ptr()), _lib.stream_ptr(torch, dev)))

    def loss_sum(self, reset=True):
        """Sum of the batches' mean BCE losses since the last reset."""
        if self._loss is None:
            return 0.0
        v = float(self._loss.item())
        if reset:
            self._loss.zero_()
        return v

    def zero_grad(self):
        pass
