"""Golden vectors for the final-KPI ranking metrics, produced by RUNNING THE UNMODIFIED REFERENCE functions
(util/metrics.py:99-195: precision_at_k, recall_at_k, mrr_at_k, map_at_k, hr_at_k, ndcg_at_k) and the ranking rule of
BPRMFRecommender.py:204-210 (np.argsort(pred_rates)[::-1][:topk]) on seeded random inputs.

Runs only in the build container (needs /root/reference).  `np.asfarray` (removed in NumPy 2, SURVEY D3) is provided
as the alias it used to be (np.asarray(..., dtype=float)) for the duration of the run -- the reference source is not
touched.

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_rank_metrics_golden.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True
sys.path.insert(0, "/root/reference")
if not hasattr(np, "asfarray"):
    np.asfarray = lambda a, dtype=float: np.asarray(a, dtype=dtype)      # what NumPy < 2 provided

from util.metrics import (hr_at_k, map_at_k, mrr_at_k, ndcg_at_k, precision_at_k, recall_at_k)  # noqa: E402

rng = np.random.default_rng(2019)
out = {}
for case, (n_users, n_cand, k, n_pos_max) in enumerate([(50, 100, 10, 3), (7, 20, 5, 8), (200, 1000, 10, 1)]):
    scores = rng.standard_normal((n_users, n_cand)).astype(np.float32)
    scores[:, ::7] = np.round(scores[:, ::7], 1)                          # some exact ties
    cands = np.stack([rng.permutation(5000)[:n_cand] for _ in range(n_users)]).astype(np.int64)
    users = rng.permutation(10_000)[:n_users]
    test_ur = {int(u): set(rng.choice(c, size=rng.integers(1, n_pos_max + 1), replace=False).tolist())
               for u, c in zip(users, cands)}
    preds = {}
    for n, u in enumerate(users):                                          # BPRMFRecommender.py:204-210
        rec_idx = np.argsort(scores[n])[::-1][:k]
        top_n = cands[n][rec_idx]
        preds[int(u)] = [1 if e in test_ur[int(u)] else 0 for e in top_n]
    kpi = dict(
        precision=np.mean([precision_at_k(r, k) for r in preds.values()]),
        recall=np.mean([recall_at_k(r, len(test_ur[u]), k) for u, r in preds.items()]),
        map=map_at_k(list(preds.values())),
        ndcg=np.mean([ndcg_at_k(r, k) for r in preds.values()]),
        hr=hr_at_k(list(preds.values()), list(preds.keys()), test_ur),
        mrr=mrr_at_k(list(preds.values())))
    # scores and candidates are not stored (case 2's alone are over 1 MB): the test reads the relevance rows the
    # ranking produced, and the seeded generator above draws the inputs again
    out[f"c{case}_users"] = users
    out[f"c{case}_k"] = k
    out[f"c{case}_ur_ptr"] = np.cumsum([0] + [len(test_ur[int(u)]) for u in users])
    out[f"c{case}_ur_idx"] = np.concatenate([sorted(test_ur[int(u)]) for u in users])
    out[f"c{case}_rel"] = np.array([preds[int(u)] for u in users], dtype=np.int8)
    out[f"c{case}_kpi"] = np.array([kpi[m] for m in ("precision", "recall", "map", "ndcg", "hr", "mrr")], dtype=np.float64)
    print(case, kpi)
np.savez_compressed(os.path.join(HERE, "rank_metrics.npz"), **out)
