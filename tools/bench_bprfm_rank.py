"""Measure ranking with BPR-FM models (metrics.topk_candidates / topk_full: the batch-norm model's fold
daisy_fmbn_rank_tables, then daisy_topk_candidates / daisy_topk_full) against the path it replaces, the model's own
forward() over the same (user, item) pairs followed by torch.topk, in the same process.

    python tools/bench_bprfm_rank.py [--out FILE] [--cases script,ml100k_full,large_tc,large_simt]

Cases (DESIGN.md section 6f): the script's evaluation (941 users x 1 + 999 candidates, hidden_factor 64, top 10), with
and without batch norm; the ml-100k full catalogue (943 x 1 682, training positives excluded, top 10), with and without
batch norm; 16 384 users x 2 M items, F 64, top 100 (W = 68: the tensor-core filter); the same at F 255 (W = 256: the
CUDA-core filter).  The batch-norm model is in evaluation mode.  Weights are seeded draws with the spread of a trained
model (embeddings N(0, 0.1^2), item and user biases N(0, 0.05^2), gamma, beta, running mean and variance away from their
initial 1 / 0 / 0 / 1), so that scores are distinct.
Times are CUDA events around whole ranking calls, fold included, after a warm-up call, over windows of at least 1 s;
the fold alone (BPRFMBN.rank_tables) is timed the same way and reported as a share of the call.  forward() scores a
pair twice (pred_i and pred_j of the same item), as a caller ranking with it does.  The baseline of the two large cases
runs on a prefix of the users (all of them would take minutes); its time is scaled to all users and the JSON says so.
The card's name, power limit and clocks are read (nvidia-smi --query-gpu, read-only) in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from recommend_lib_b200.bprfm import BPRFM  # noqa: E402
from recommend_lib_b200.metrics import topk_candidates, topk_full  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,temperature.gpu"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        return dict(zip(q.split(","), [x.strip() for x in out[0].split(",")])) if out else {}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def timed(fn, min_s=1.0, min_reps=3):
    """ms per call: one warm-up call, then calls until the window holds >= min_s of device time."""
    fn()
    torch.cuda.synchronize()
    reps, total = 0, 0.0
    while total < min_s * 1e3 or reps < min_reps:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        total += a.elapsed_time(b)
        reps += 1
    return total / reps, reps


def make_model(U, I, F, bn, seed, dev):
    m = BPRFM(U + I, F, bn, [0.5, 0.2] if bn else [0.0, 0.0], user_num=U).to(dev)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    with torch.no_grad():
        m.embeddings.weight.normal_(0.0, 0.1, generator=g)
        m.biases.weight.normal_(0.0, 0.05, generator=g)
        m.bias_.fill_(0.1)
        if bn:
            layer = m.FM_layers[0]
            layer.weight.normal_(1.0, 0.3, generator=g)
            layer.bias.normal_(0.0, 0.1, generator=g)
            layer.running_mean.normal_(0.0, 0.002, generator=g)
            layer.running_var.uniform_(5e-5, 2e-4, generator=g)      # the variance of e_u * e_i at this spread: 1e-4
    if bn:
        m.eval()
    return m


def run_case(name, U, I, F, bn, N, K, C=None, exclude=None, base_users=None, seed=2019):
    dev = torch.device("cuda:0")
    m = make_model(U, I, F, bn, seed, dev)
    rng = np.random.default_rng(seed)
    users = (rng.choice(U, N, replace=False) if N <= U else rng.integers(0, U, N)).astype(np.int32)
    users_d = torch.from_numpy(users).to(dev)
    if C is not None:
        cands = np.stack([rng.choice(I, C, replace=False) for _ in range(N)]).astype(np.int32)
        cands_d = torch.from_numpy(cands).to(dev)
        fn = lambda: topk_candidates(m, users_d, cands_d, K)
        cols = C
    else:
        excl = [exclude[u] for u in users] if exclude is not None else None
        fn = lambda: topk_full(m, users_d, K, exclude=excl)
        cols = I
    ms, reps = timed(fn)
    fold_ms, fold_reps = timed(m.rank_tables) if bn else (0.0, 0)
    new_out = fn()
    new_items = (new_out[1] if C is not None else new_out[0]).cpu().numpy()
    path = m.handle().topk_full_path()[0] if C is None else "candidates"
    pairs = N * cols
    # baseline: forward over every pair of the (first nb) users + torch.topk; the same masking for exclusions
    nb = N if base_users is None else min(base_users, N)
    bu = torch.from_numpy(np.repeat(users[:nb], cols).astype(np.int64)).to(dev)
    bi = torch.from_numpy((cands[:nb] if C is not None else np.tile(np.arange(I), (nb, 1))).reshape(-1).astype(np.int64)).to(dev)
    feats = torch.stack([bu, bi + U], 1)
    mask = None
    if C is None and exclude is not None:
        mk = np.zeros((nb, I), bool)
        for n in range(nb):
            mk[n, exclude[users[n]]] = True
        mask = torch.from_numpy(mk).to(dev)
    step = 1 << 20                                    # forward() takes up to 2^31 / 3 / (F + 1) triples per call

    def base():
        s = torch.cat([m(feats[a:a + step], None, feats[a:a + step], None)[0] for a in range(0, feats.shape[0], step)])
        s = s.view(nb, cols)
        if mask is not None:
            s = s.masked_fill(mask, float("-inf"))
        return torch.topk(s, K, dim=1)
    bms, breps = timed(base, min_reps=2)
    bt = base()
    bidx = bt.indices.cpu().numpy()
    base_items = np.take_along_axis(cands[:nb], bidx, 1) if C is not None else bidx
    same = [set(a.tolist()) == set(b.tolist()) for a, b in zip(new_items[:nb], base_items)]
    base_ms_all = bms * N / nb
    return {
        "case": name, "batch_norm": bn, "users": N, "items_per_user": cols, "catalogue": I,
        "mode": "candidate" if C is not None else "full", "topk_path": path, "exclusions": exclude is not None, "K": K,
        "factors": F, "row_width": (F + 4) // 4 * 4 if bn else F + 4,
        "ms": round(ms, 4), "reps": reps, "pairs": pairs, "pairs_per_s": pairs / (ms * 1e-3),
        "fold_ms": round(fold_ms, 4), "fold_reps": fold_reps, "fold_share": fold_ms / ms,
        "baseline": {"what": "forward() over the pairs + torch.topk" + (" (+ masked_fill of the exclusions)" if mask is not None else ""),
                     "users_measured": nb, "ms_measured": round(bms, 4), "reps": breps,
                     "pairs_per_s": nb * cols / (bms * 1e-3), "ms_all_users": round(base_ms_all, 4),
                     "scaled_from_prefix": nb < N},
        "speedup": base_ms_all / ms,
        "topk_item_sets_equal_baseline": bool(all(same)), "users_compared": nb,
        "users_with_equal_item_sets": int(sum(same)),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--cases", default="script,ml100k_full,large_tc,large_simt")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU; there is nothing to measure without one"
    split = np.load(os.path.join(ROOT, "tests", "golden", "ml100k_split.npz"))
    U, I = int(split["user_num"]), int(split["item_num"])
    tr = split["train_pairs"].astype(np.int64)
    pos = [[] for _ in range(U)]
    for u, i in tr:
        pos[u].append(i)
    pos = [np.asarray(p, np.int32) for p in pos]
    res = {"gpu_before": gpu_info(), "torch": torch.__version__, "cases": []}
    want = a.cases.split(",")
    t0 = time.time()

    def add(case):                                    # saved after every case, so a later failure keeps the earlier ones
        res["cases"].append(case)
        save(res, a.out)

    for bn in (True, False):
        if "script" in want:
            add(run_case("script shape", U, I, 64, bn, 941, 10, C=1000))
        if "ml100k_full" in want:
            add(run_case("ml-100k full", U, I, 64, bn, U, 10, exclude=pos))
    if "large_tc" in want:
        add(run_case("16k users x 2M items, F 64", 16384, 1 << 21, 64, True, 16384, 100, base_users=64))
    if "large_simt" in want:
        add(run_case("16k users x 2M items, F 255", 16384, 1 << 21, 255, True, 16384, 100, base_users=64))
    res["gpu_after"] = gpu_info()
    res["wall_s"] = round(time.time() - t0, 1)
    print(json.dumps(res))
    save(res, a.out)


def save(res, out):
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
