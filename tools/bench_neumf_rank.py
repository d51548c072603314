"""Measure ranking with the NeuMF tower (daisy_neumf_topk_candidates / daisy_neumf_topk_full) against the path it replaces,
NeuMF.forward over the same (user, item) pairs followed by torch.topk, in the same process.

    python tools/bench_neumf_rank.py [--out FILE] [--cases script,ml100k_full,ml20m_full,wide]

Cases (DESIGN.md section 6e): the script's evaluation (941 users x 1 + 999 candidates, top 10); ml-100k full catalogue
(943 x 1 682, training positives excluded, top 10); an ml-20m-sized catalogue (a 16 384-user sample x 27 278 items, top
100); the widest tower (factor 64, 4 layers) on the ml-100k catalogue.  Weights are NeuMF's own initialisation (seeded).
Times are CUDA events around whole calls after a warm-up call, over windows of at least 1 s.  The forward baseline of
the two largest cases runs on a prefix of the users (it takes minutes on all of them); its rate is reported per pair and
its time scaled to all pairs, and the JSON says so.  Achieved FLOP/s use the algorithmic count of the split tower:
2 * (sum over layers l >= 1 of in_l * out_l + predict + GMF) per pair, plus 2 * Dm * Dm per user and per catalogue item.
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

from recommend_lib_b200.metrics import topk_candidates, topk_full  # noqa: E402
from recommend_lib_b200.ncf_mlp import NeuMF  # noqa: E402


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


def flops(F, L, neumf, pairs, n_users, n_items):
    Dm = F << (L - 1)
    per_pair = sum((Dm >> (l - 1)) * (Dm >> l) for l in range(1, L)) + (2 * F if neumf else F) + (F if neumf else 0)
    return 2.0 * (per_pair * pairs + Dm * Dm * (n_users + n_items))


def run_case(name, U, I, F, L, N, K, C=None, exclude=None, base_users=None, seed=2019):
    dev = torch.device("cuda:0")
    torch.manual_seed(seed)
    m = NeuMF(U, I, F, L, 0.0, "NeuMF-end").to(dev)
    rng = np.random.default_rng(seed)
    users = (rng.choice(U, N, replace=False) if N <= U else rng.integers(0, U, N)).astype(np.int32)
    if C is not None:
        cands = np.stack([rng.choice(I, C, replace=False) for _ in range(N)]).astype(np.int32)
        cands_d = torch.from_numpy(cands).to(dev)
        users_d = torch.from_numpy(users).to(dev)
        fn = lambda: topk_candidates(m, users_d, cands_d, K)
        cols = C
    else:
        users_d = torch.from_numpy(users).to(dev)
        excl = [exclude[u] for u in users] if exclude is not None else None
        fn = lambda: topk_full(m, users_d, K, exclude=excl)
        cols = I
    ms, reps = timed(fn)
    new_out = fn()
    new_items = (new_out[1] if C is not None else new_out[0]).cpu().numpy()
    pairs = N * cols
    fl = flops(F, L, True, pairs, N, I)
    # baseline: forward over every pair of the (first nb) users + torch.topk; the same masking for exclusions
    nb = N if base_users is None else min(base_users, N)
    bu = torch.from_numpy(np.repeat(users[:nb], cols).astype(np.int64)).to(dev)
    bi = torch.from_numpy((cands[:nb] if C is not None else np.tile(np.arange(I), (nb, 1))).reshape(-1).astype(np.int64)).to(dev)
    mask = None
    if C is None and exclude is not None:
        mk = np.zeros((nb, I), bool)
        for n in range(nb):
            mk[n, exclude[users[n]]] = True
        mask = torch.from_numpy(mk).to(dev)

    step = 1 << 19                                    # forward() takes batches of at most ~1 M samples

    def base():
        s = torch.cat([m(bu[a:a + step], bi[a:a + step]) for a in range(0, bu.shape[0], step)]).view(nb, cols)
        if mask is not None:
            s = s.masked_fill(mask, float("-inf"))
        return torch.topk(s, K, dim=1)
    bms, breps = timed(base, min_reps=2)
    bt = base()
    bidx = bt.indices.cpu().numpy()
    base_items = np.take_along_axis(cands[:nb], bidx, 1) if C is not None else bidx
    agree = float(np.mean([len(set(a) & set(b)) / K for a, b in zip(new_items[:nb], base_items)]))
    base_ms_all = bms * N / nb
    return {
        "case": name, "users": N, "items_per_user": cols, "catalogue": I, "mode": "candidate" if C is not None else "full",
        "exclusions": exclude is not None, "K": K, "factor": F, "layers": L, "model": "NeuMF-end",
        "ms": round(ms, 4), "reps": reps, "pairs": pairs, "pairs_per_s": pairs / (ms * 1e-3),
        "algorithmic_flop": fl, "tflop_per_s": fl / (ms * 1e-3) / 1e12,
        "baseline": {"what": "NeuMF.forward over the pairs + torch.topk" + (" (+ masked_fill of the exclusions)" if mask is not None else ""),
                     "users_measured": nb, "ms_measured": round(bms, 4), "reps": breps,
                     "pairs_per_s": nb * cols / (bms * 1e-3), "ms_all_users": round(base_ms_all, 4),
                     "scaled_from_prefix": nb < N},
        "speedup": base_ms_all / ms,
        "topk_item_overlap_with_baseline": agree,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--cases", default="script,ml100k_full,ml20m_full,wide")
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
    if "script" in want:
        res["cases"].append(run_case("script shape", U, I, 32, 3, 941, 10, C=1000))
    if "ml100k_full" in want:
        res["cases"].append(run_case("ml-100k full", U, I, 32, 3, U, 10, exclude=pos))
    if "ml20m_full" in want:
        res["cases"].append(run_case("ml-20m full", 138493, 27278, 32, 3, 16384, 100, base_users=128))
    if "wide" in want:
        res["cases"].append(run_case("wide tower", U, I, 64, 4, U, 10, exclude=pos, base_users=64))
    res["gpu_after"] = gpu_info()
    res["wall_s"] = round(time.time() - t0, 1)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
