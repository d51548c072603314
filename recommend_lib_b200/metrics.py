"""HR@K / NDCG@K evaluation on the device (replaces util/metrics.py:35-66,88-94 and BPRMFRecommender.py:196-210).

``metric_eval(model, test_loader, top_k)`` keeps the reference signature: ``test_loader`` yields
``(user, item_i, item_j)`` batches, one batch per evaluated user, positive first
(``BPRMFRecommender.py:143-146``).  All groups are scored and ranked by ONE ``daisy_topk_candidates``
launch instead of one forward + topk + ``.item()`` sync per user.
Ranking order is (score desc, candidate position asc) -- ``torch.topk`` leaves ties unspecified.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib


def _i32(x, device):
    return torch.as_tensor(np.asarray(x) if not torch.is_tensor(x) else x).to(device=device, dtype=torch.int32).contiguous()


def topk_candidates(model, users, cands, top_k):
    """users [N], cands [N, C] -> (pos [N,K] candidate positions, items [N,K], scores [N,K]) as device tensors.
    ``model``: a dot-product model (BPR, NCF(model='GMF')), a BPR-FM model (``BPRFM``, and ``BPRFM(batch_norm=True)`` in
    evaluation mode), whose score is folded into one, or a ``NeuMF`` ('MLP' / 'NeuMF-end'), whose tower scores rank
    through ``daisy_neumf_topk_candidates``; each ranks itself (``rank_candidates``)."""
    dev = model._device()
    users = _i32(users, dev).reshape(-1)
    cands = _i32(cands, dev)
    N, _ = cands.shape
    if users.shape[0] != N:
        raise ValueError("users and cands disagree on the number of groups")
    return model.rank_candidates(users, cands, top_k)


def hr_ndcg(pos):
    """_hit / _ndcg (util/metrics.py:35-44) for groups whose ground truth is candidate position 0."""
    pos = pos.cpu().numpy() if torch.is_tensor(pos) else np.asarray(pos)
    hit = pos == 0
    hr = hit.any(axis=1).astype(np.float64)
    rank = hit.argmax(axis=1)
    ndcg = np.where(hr > 0, 1.0 / np.log2(rank + 2.0), 0.0)
    return float(hr.mean()), float(ndcg.mean())


def metric_eval(model, test_loader, top_k, algo="bpr"):
    """Drop-in for ``metric_eval`` (util/metrics.py:88-94); returns (HR, NDCG).  ``algo='bpr'`` (``_bpr_topk``) with a
    ``BPR`` model, ``algo='ncf'`` (``_ncf_topk``, :68-86) with an ``NCF(model='GMF')`` or a ``NeuMF`` model; a BPR-FM model
    (``BPRFM``, or ``BPRFM(batch_norm=True)`` after ``model.eval()``) with either: both loaders yield (user, candidates, _)
    groups whose first candidate is the ground truth."""
    if algo not in ("bpr", "ncf"):
        raise ValueError("algo must be 'bpr' or 'ncf'")
    if algo == "bpr" and not model.bpr_topk:
        raise ValueError("algo='bpr' needs a BPR model; rank an NCF model with algo='ncf'")
    groups = {}
    order = []
    for user, item_i, _ in test_loader:
        u = torch.as_tensor(user).reshape(-1)
        it = torch.as_tensor(item_i).reshape(-1)
        groups.setdefault(int(it.shape[0]), []).append((len(order), u[:1], it))
        order.append(None)
    hrs = np.zeros(len(order))
    ndcgs = np.zeros(len(order))
    for C, lst in groups.items():
        users = torch.cat([g[1] for g in lst])
        cands = torch.stack([g[2] for g in lst])
        k = min(int(top_k), C)
        pos, items, _ = topk_candidates(model, users, cands, k)
        items = items.cpu().numpy()
        gt = cands[:, 0].cpu().numpy()
        hit = items == gt[:, None]                     # `gt_item in recommends`
        h = hit.any(axis=1)
        r = hit.argmax(axis=1)
        for n, g in enumerate(lst):
            hrs[g[0]] = float(h[n])
            ndcgs[g[0]] = 1.0 / np.log2(r[n] + 2.0) if h[n] else 0.0
    return np.mean(hrs), np.mean(ndcgs)


def topk_full(model, users, k, exclude=None):
    """Full-catalogue top-k for ``users``: (items [N,k] int32, scores [N,k]) device tensors, order (score desc, item asc).
    ``model``: BPR, NCF(model='GMF'), a BPR-FM model or a ``NeuMF``, as for ``topk_candidates``.
    ``exclude``: optional per-user lists of item ids to mask (training positives)."""
    dev = model._device()
    users = _i32(users, dev).reshape(-1)
    return model.rank_full(users, k, _lib.exclusion_csr(exclude, users.shape[0], dev))


# ----------------------------------------------------------------------------------------------------------------
# final test-set KPIs (SURVEY.md section 8f row N2): the ranking loop BPRMFRecommender.py:196-210 as ONE
# daisy_topk_candidates launch, then the six numpy metrics of util/metrics.py:99-195 vectorised over users
# ----------------------------------------------------------------------------------------------------------------
def rank_metrics(rel, gt_len, top_k=None):
    """Precision / Recall / MAP / NDCG / HR / MRR @k exactly as the reference computes them from per-user relevance
    lists in rank order (``rel`` [N, k] of 0/1, ``gt_len`` [N] = len(test_ur[u])):

    * precision_at_k = sum(r) / k, recall_at_k = sum(r) / len(ground truth) (0 when empty)      util/metrics.py:99-125
    * average_precision = sum over hits of precision@(rank) / **len(r)** (not the number of hits)  :136-149
    * ndcg_at_k = dcg(r) / dcg(sorted(r)), dcg = sum(r / log2(rank + 1)); ``np.asfarray`` there is the NumPy-2
      casualty of SURVEY D3 -- restated with plain float arrays                                     :171-195
    * hr_at_k = total hits / total ground-truth size (a micro average)                              :161-169
    * mrr_at_k adds 1/rank for EVERY hit, not only the first                                        :127-134
    """
    rel = (np.asarray(rel) != 0).astype(np.float64)
    if rel.ndim != 2:
        raise ValueError("rel must be [users, k]")
    n, k = rel.shape
    if top_k is not None and int(top_k) != k:
        raise ValueError("Relevance score length < k")          # the reference's ValueError (:113, :122)
    gt_len = np.asarray(gt_len, dtype=np.float64).reshape(-1)
    hits = rel.sum(axis=1)
    ranks = np.arange(1, k + 1, dtype=np.float64)
    prec_at = np.cumsum(rel, axis=1) / ranks                    # precision_at_k(r, j + 1) for every prefix
    disc = 1.0 / np.log2(ranks + 1.0)
    dcg = (rel * disc).sum(axis=1)
    idcg = (-np.sort(-rel, axis=1) * disc).sum(axis=1)
    with np.errstate(divide="ignore", invalid="ignore"):
        recall = np.where(gt_len != 0, hits / gt_len, 0.0)
        ndcg = np.where(idcg != 0, dcg / idcg, 0.0)
    return {"precision": float((hits / k).mean()), "recall": float(recall.mean()),
            "map": float(((prec_at * rel).sum(axis=1) / k).mean()), "ndcg": float(ndcg.mean()),
            "hr": float(hits.sum() / gt_len.sum()) if gt_len.sum() else 0.0,
            "mrr": float((rel / ranks).sum() / n)}


def final_kpi(model, test_users, test_cands, test_ur, top_k=10):
    """The final KPI block of the script (BPRMFRecommender.py:196-229): rank every test user's candidate items with the
    model, mark the top-k that are in the user's ground truth ``test_ur[u]`` (a dict of sets, or a list aligned with
    ``test_users``) and return the six metrics.  One device launch for all users instead of one scalar forward per
    (user, candidate).  Ranking order: (score desc, candidate position asc); the reference's
    ``np.argsort(...)[::-1]`` leaves ties unspecified."""
    test_users = np.asarray(test_users).reshape(-1)
    cands = np.asarray(test_cands)
    k = min(int(top_k), cands.shape[1])
    _, items, _ = topk_candidates(model, test_users, cands, k)
    items = items.cpu().numpy()
    get = (lambda n, u: test_ur[int(u)]) if isinstance(test_ur, dict) else (lambda n, u: test_ur[n])
    rel = np.zeros(items.shape, dtype=np.int8)
    gt_len = np.zeros(len(test_users), dtype=np.int64)
    for n, u in enumerate(test_users):
        gt = get(n, u)
        gt_len[n] = len(gt)
        rel[n] = [1 if int(e) in gt else 0 for e in items[n]]
    return rank_metrics(rel, gt_len, k)
