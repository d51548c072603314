"""Drop-ins for ``class Item2Vec`` and ``class SGNS`` of the reference (Item2VecRecommender.py:37-97) and for the training
step of its script (:266, 274-277), on the C-ABI library (``daisy_sgns_step``, csrc/sgns.cu).  SURVEY.md section 8f, N4.

GPU-verified in round 2 (tests/test_sgns_gpu.py, part of the default ``-m gpu`` suite).  The checker is
``oracle/sgns_oracle.py``, pinned to the unmodified reference classes.  No CPU fallback.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch
import torch.nn as nn

from . import _lib

c_vp = ctypes.c_void_p


class Item2Vec(nn.Module):
    """``Item2Vec(vocab_size, embedding_size, padding_idx=0)``: ``ivectors`` / ``ovectors`` initialised as the reference
    does (:40-52: row 0 zero, the rest U(-0.5 / D, 0.5 / D)); ``forward`` / ``forward_i`` / ``forward_o`` are row gathers."""

    def __init__(self, vocab_size=20000, embedding_size=100, padding_idx=0):
        super().__init__()
        self.vocab_size, self.embedding_size = int(vocab_size), int(embedding_size)
        self.ivectors = nn.Embedding(self.vocab_size, self.embedding_size, padding_idx=padding_idx)
        self.ovectors = nn.Embedding(self.vocab_size, self.embedding_size, padding_idx=padding_idx)
        bound = 0.5 / self.embedding_size
        for emb in (self.ivectors, self.ovectors):
            w = torch.cat([torch.zeros(1, self.embedding_size),
                           torch.empty(self.vocab_size - 1, self.embedding_size).uniform_(-bound, bound)])
            emb.weight = nn.Parameter(w, requires_grad=False)

    def forward(self, data):
        return self.forward_i(data)

    def forward_i(self, data):
        v = torch.as_tensor(data, dtype=torch.long, device=self.ivectors.weight.device)
        return self.ivectors.weight[v]

    def forward_o(self, data):
        v = torch.as_tensor(data, dtype=torch.long, device=self.ovectors.weight.device)
        return self.ovectors.weight[v]


class SGNS(nn.Module):
    """``SGNS(embedding, vocab_size, n_negs, weights)`` (:70-80).  Training is the fused step of ``SGNSAdam``; ``forward``
    (which in the reference builds the autograd graph of the loss) raises and says so."""

    def __init__(self, embedding, vocab_size=20000, n_negs=20, weights=None):
        super().__init__()
        self.embedding = embedding
        self.vocab_size, self.n_negs = int(vocab_size), int(n_negs)
        self.weights = None
        if weights is not None:
            wf = np.power(weights, 0.75)
            wf = wf / wf.sum()
            self.weights = torch.FloatTensor(wf)

    def draw_negatives(self, batch_size, context_size, device):
        """The draw of :86-91 (unigram^0.75 table, or uniform over [0, vocab_size - 1)), on ``device``."""
        n = context_size * self.n_negs
        if self.weights is not None:
            w = self.weights.to(device)
            return torch.multinomial(w, batch_size * n, replacement=True).view(batch_size, -1)
        return torch.empty(batch_size, n, device=device).uniform_(0, self.vocab_size - 1).long()

    def forward(self, iword, owords):
        raise RuntimeError("the SGNS loss, its backward and the Adam step are fused: use SGNSAdam(sgns).step(iword, owords)")


class SGNSAdam(_lib.HandleOwner):
    """``optim.Adam(sgns.parameters())`` (:266) + the step of :274-277, fused: ``step(iword, owords, nwords=None)``.
    ``nwords`` ([B, C * n_negs]) replaces the draw inside the reference's forward -- that is how the parity tests feed the
    negatives the reference drew; without it they are drawn on the device (``SGNS.draw_negatives``)."""

    _cpu_error = "Item2Vec tables are on the CPU: call sgns.cuda() first (no CPU fallback)"

    def __init__(self, sgns: SGNS, lr=1e-3, betas=(0.9, 0.999), eps=1e-8):
        self.sgns, self.lr, self.betas, self.eps = sgns, float(lr), (float(betas[0]), float(betas[1])), float(eps)
        self.t = 0
        self.state = None
        self._scratch = None
        self._loss = None

    def _weight(self):
        return self.sgns.embedding.ivectors.weight

    def _handle_dims(self):
        V = self.sgns.embedding.vocab_size
        return V, V, 4                                  # carries the device, the error flag and the launch counter

    def step(self, iword, owords, nwords=None):
        emb = self.sgns.embedding
        dev = self._device()
        iv, ov = emb.ivectors.weight, emb.ovectors.weight
        for t in (iv, ov):
            if t.dtype != torch.float32 or not t.is_contiguous():
                raise _lib.DaisyError("Item2Vec tables must be contiguous float32")
        i32 = lambda a: torch.as_tensor(a).to(device=dev, dtype=torch.int32).contiguous()
        iword, owords = i32(iword), i32(owords)
        if iword.dim() != 1 or owords.dim() != 2 or owords.shape[0] != iword.shape[0]:
            raise ValueError("iword must be [B] and owords [B, C]")
        B, C, N = iword.shape[0], owords.shape[1], self.sgns.n_negs
        if nwords is None:
            nwords = self.sgns.draw_negatives(B, C, dev)
        nwords = i32(nwords)
        if tuple(nwords.shape) != (B, C * N):
            raise ValueError(f"nwords must be [{B}, {C * N}]")
        if self.state is None or self.state[0].device != dev:
            self.state = [torch.zeros_like(iv), torch.zeros_like(iv), torch.zeros_like(ov), torch.zeros_like(ov)]
            self._loss = torch.zeros(1, dtype=torch.float64, device=dev)
            self._scratch = None
        h = self.handle()
        need = ctypes.c_int64()
        _lib.check(h.L.daisy_sgns_scratch_bytes(B, C, N, emb.vocab_size, emb.embedding_size, ctypes.byref(need)))
        if self._scratch is None or self._scratch.numel() < need.value:
            self._scratch = torch.empty(need.value, dtype=torch.uint8, device=dev)
        pad = emb.ivectors.padding_idx
        m_iv, v_iv, m_ov, v_ov = self.state
        p = lambda t: c_vp(t.data_ptr())
        prm = _lib.SGNSParams(p(iv), p(ov), p(m_iv), p(v_iv), p(m_ov), p(v_ov), self.lr, self.betas[0], self.betas[1],
                              self.eps, emb.vocab_size, emb.embedding_size, -1 if pad is None else int(pad))
        self.t += 1
        _lib.check(h.L.daisy_sgns_step(h.ptr, ctypes.byref(prm), p(iword), p(owords), p(nwords) if N else None, B, C, N,
                                       self.t, p(self._scratch), need.value, p(self._loss), _lib.stream_ptr(torch, dev)))

    def loss_sum(self, reset=True):
        """Sum of the batch losses (:97) since the last reset."""
        if self._loss is None:
            return 0.0
        v = float(self._loss.item())
        if reset:
            self._loss.zero_()
        return v

    def zero_grad(self):
        pass
