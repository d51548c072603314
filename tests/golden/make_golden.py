"""Generate the golden fixtures under tests/golden/ by RUNNING THE UNMODIFIED REFERENCE.

Runs only in the build container (needs /root/reference); the fixtures it writes are
committed and are what the GPU box sees.  Nothing here is imported by the product.

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py [--skip-trajectory]

Fixtures
--------
ml100k_split.npz     train / test pairs of config 1: leave-one-out by latest timestamp, restated
                     with pandas exactly as util/data_loader.py:447-448 (codes), :412-414 (split);
                     the numpy restatement in recommend_lib_b200/data.py is asserted equal.
bpr_small.npz        3 steps of the reference BPR + optim.SGD on a tiny table with heavy in-batch
                     duplicates (BPRMFRecommender.py:28-50,154,172-176).
bpr_config1_step.npz first step of config 1 (943 x 1682, D 64, B 4096, lr .01, wd .001): tables
                     before the step, the batch and the loss; bpr_config1_step_after.npz: the tables after it.
bpr_eval_small.npz   reference metric_eval (util/metrics.py:46-66,88-94) on a tiny model.
bpr_ml100k_traj.json 20-epoch config-1 trajectory of the reference loop fed by the
                     deterministic sampler: epoch loss, HR@10, NDCG@10.
mf_small.npz         SVD (biased / unbiased) and RSVD (v1 / v2) fits by the reference's compiled
                     Cython extension (oracle/_ref), util/matrix_factorization.pyx.
"""
import contextlib
import hashlib
import io
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(1, REF)

import pandas as pd  # noqa: E402
import torch  # noqa: E402

from BPRMFRecommender import BPR  # noqa: E402  (reference, unmodified)
from util.data_loader import BPRData  # noqa: E402  (reference, unmodified)
from util.metrics import metric_eval  # noqa: E402  (reference, unmodified)

from recommend_lib_b200 import data as hostdata  # noqa: E402
from recommend_lib_b200.sampler import TripleSampler, _rng  # noqa: E402
from oracle.build_ref import load_ref  # noqa: E402


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def ref_steps(model, batches, lr, wd):
    """BPRMFRecommender.py:154,172-176 driven verbatim as calls."""
    opt = torch.optim.SGD(model.parameters(), lr=lr, weight_decay=wd)
    losses = []
    for b in batches:
        t = torch.from_numpy(np.asarray(b)).long()
        user, item_i, item_j = t[:, 0], t[:, 1], t[:, 2]
        model.zero_grad()
        pred_i, pred_j = model(user, item_i, item_j)
        loss = -(pred_i - pred_j).sigmoid().log().sum()
        loss.backward()
        opt.step()
        losses.append(float(loss))
    return losses


def tables(model):
    return (model.embed_user.weight.detach().numpy().copy(),
            model.embed_item.weight.detach().numpy().copy())


def ref_eval(model, users, cands, top_k):
    """metric_eval through the reference's own BPRData + DataLoader (BPRMFRecommender.py:138-146,181)."""
    feats = [[int(u), int(c)] for u, row in zip(users, cands) for c in row]
    ds = BPRData(feats, 0, None, 0, False)
    loader = torch.utils.data.DataLoader(ds, batch_size=cands.shape[1], shuffle=False, num_workers=0)
    model.eval()
    with torch.no_grad():
        hr, ndcg = metric_eval(model, loader, top_k)
    return float(hr), float(ndcg)


def make_split():
    df = pd.read_csv(f"{REF}/data/ml-100k/u.data", sep="\t", header=None,
                     names=["user", "item", "rating", "timestamp"], engine="python")
    df.sort_values(["user", "item", "timestamp"], inplace=True)            # load_rate :117
    df["user"] = pd.Categorical(df.user).codes                             # load_mat :447-448
    df["item"] = pd.Categorical(df.item).codes
    user_num, item_num = int(df.user.max() + 1), int(df.item.max() + 1)
    df["rank_latest"] = df.groupby(["user"])["timestamp"].rank(method="first", ascending=False)   # :412
    train = df[df["rank_latest"] > 1]
    test = df[df["rank_latest"] == 1]
    train_pairs = train[["user", "item"]].values.astype(np.int64)
    test_pairs = test[["user", "item"]].values.astype(np.int64)

    # pin the numpy restatement used by the product's host code
    raw = hostdata.load_ml100k(f"{REF}/data/ml-100k/u.data")
    u, nu = hostdata.encode_ids(raw[:, 0])
    i, ni = hostdata.encode_ids(raw[:, 1])
    tr, te = hostdata.split_loo_by_time(u, i, raw[:, 3])
    assert (nu, ni) == (user_num, item_num)
    assert np.array_equal(np.stack([u[tr], i[tr]], 1), train_pairs)
    assert np.array_equal(np.stack([u[te], i[te]], 1), test_pairs)

    np.savez_compressed(f"{HERE}/ml100k_split.npz", train_pairs=train_pairs.astype(np.uint16),
                        test_pairs=test_pairs.astype(np.uint16), user_num=user_num, item_num=item_num,
                        ratings=train["rating"].values.astype(np.uint8))
    print("split:", user_num, item_num, train_pairs.shape, test_pairs.shape)
    return train_pairs, test_pairs, user_num, item_num


def make_bpr_small():
    torch.manual_seed(7)
    U, I, D, B = 60, 50, 16, 200
    model = BPR(U, I, D)
    with torch.no_grad():                       # larger weights than std .01 so that sigma is not ~0.5 everywhere
        model.embed_user.weight.mul_(40.0)
        model.embed_item.weight.mul_(40.0)
    P0, Q0 = tables(model)
    g = _rng(7, 99)
    batches = [np.stack([g.integers(0, U, B), g.integers(0, I, B), g.integers(0, I, B)], 1).astype(np.int32)
               for _ in range(3)]
    batches[1][:40, 1] = 3                      # a very hot positive item
    batches[1][10:30, 0] = 5                    # a hot user
    batches[2][:5, 2] = batches[2][:5, 1]       # i == j: contributions cancel
    snaps = []
    losses = []
    opt_losses = None
    lr, wd = 0.05, 0.01
    opt = torch.optim.SGD(model.parameters(), lr=lr, weight_decay=wd)
    for b in batches:
        t = torch.from_numpy(b).long()
        model.zero_grad()
        pi, pj = model(t[:, 0], t[:, 1], t[:, 2])
        loss = -(pi - pj).sigmoid().log().sum()
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
        snaps.append(tables(model))
    t = torch.from_numpy(batches[0]).long()
    with torch.no_grad():
        pi, pj = model(t[:, 0], t[:, 1], t[:, 2])
    np.savez_compressed(f"{HERE}/bpr_small.npz", P0=P0, Q0=Q0, batches=np.stack(batches), lr=lr, wd=wd,
                        losses=np.array(losses), P=np.stack([s[0] for s in snaps]), Q=np.stack([s[1] for s in snaps]),
                        fwd_pred_i=pi.numpy(), fwd_pred_j=pj.numpy())
    print("bpr_small losses", losses)


def make_config1_step(train_pairs, user_num, item_num):
    torch.manual_seed(2019)
    model = BPR(user_num, item_num, 64)
    P0, Q0 = tables(model)
    sampler = TripleSampler(train_pairs, item_num, num_ng=4, seed=2019)
    batch = next(iter(sampler.batches(0, 4096)))
    losses = ref_steps(model, [batch], 0.01, 0.001)
    P1, Q1 = tables(model)
    # two files keep each fixture under 1 MB (the tables before and after the step are 1.3 MB together)
    np.savez_compressed(f"{HERE}/bpr_config1_step.npz", P0=P0, Q0=Q0, loss=losses[0], batch=batch, batch_sha=sha(batch))
    np.savez_compressed(f"{HERE}/bpr_config1_step_after.npz", P1=P1, Q1=Q1)
    print("config1 step loss", losses[0], "batch sha", sha(batch))


def make_eval_small():
    torch.manual_seed(11)
    U, I, D, C, K = 64, 300, 32, 100, 10
    model = BPR(U, I, D)
    g = _rng(11, 5)
    users = np.arange(U, dtype=np.int32)
    cands = np.stack([g.choice(I, C, replace=False) for _ in range(U)]).astype(np.int32)
    with torch.no_grad():                       # pull some users towards their held-out item so HR/NDCG are not ~0
        for u in range(0, U, 2):
            w = float(g.random()) * 0.6
            model.embed_user.weight[u] += w * model.embed_item.weight[int(cands[u, 0])]
    hr, ndcg = ref_eval(model, users, cands, K)
    P, Q = tables(model)
    np.savez_compressed(f"{HERE}/bpr_eval_small.npz", P=P, Q=Q, users=users, cands=cands, top_k=K, hr=hr, ndcg=ndcg)
    print("eval small", hr, ndcg)


def make_trajectory(train_pairs, test_pairs, user_num, item_num, epochs=20):
    torch.manual_seed(2019)
    torch.set_num_threads(os.cpu_count())
    model = BPR(user_num, item_num, 64)
    opt = torch.optim.SGD(model.parameters(), lr=0.01, weight_decay=0.001)
    sampler = TripleSampler(train_pairs, item_num, num_ng=4, seed=2019)
    allp = np.concatenate([train_pairs, test_pairs])
    eu, ec = hostdata.eval_candidates(allp[:, 0], allp[:, 1], test_pairs[:, 0], test_pairs[:, 1], item_num, 999, 2019)
    out = dict(config="ml-100k D64 B4096 lr.01 wd.001 num_ng4 seed2019", eval_users=int(len(eu)),
               cand_sha=sha(ec), epochs=[])
    for ep in range(epochs):
        t0 = time.time()
        model.train()
        tot = 0.0
        for b in sampler.batches(ep, 4096):
            t = torch.from_numpy(b).long()
            model.zero_grad()
            pi, pj = model(t[:, 0], t[:, 1], t[:, 2])
            loss = -(pi - pj).sigmoid().log().sum()
            loss.backward()
            opt.step()
            tot += float(loss)
        hr, ndcg = ref_eval(model, eu, ec, 10)
        out["epochs"].append(dict(epoch=ep + 1, loss=tot, hr=hr, ndcg=ndcg))
        print(f"epoch {ep + 1}: loss {tot:.1f} HR {hr:.4f} NDCG {ndcg:.4f}  ({time.time() - t0:.1f}s)", flush=True)
    with open(f"{HERE}/bpr_ml100k_traj.json", "w") as f:
        json.dump(out, f, indent=1)


def make_mf_small():
    m = load_ref()
    assert m is not None, "oracle/_ref could not be built"
    g = _rng(3, 1)
    U, I, D, N, E = 40, 30, 12, 600, 3
    users = g.integers(0, U, N).astype(np.int64)
    items = g.integers(0, I, N).astype(np.int64)
    ratings = g.integers(1, 6, N).astype(np.float64)
    df = pd.DataFrame({"user": users, "item": items, "rating": ratings})
    out = dict(users=users.astype(np.int32), items=items.astype(np.int32), ratings=ratings, U=U, I=I, D=D, E=E)
    for name, kw in (("svd_b", dict(biased=True)), ("svd_u", dict(biased=False, lr_all=0.01, reg_all=0.05))):
        np.random.seed(2019)
        st = np.random.get_state()
        a = m.SVD(U, I, n_factors=D, n_epochs=E, verbose=False, **kw)
        a.fit(df)
        np.random.set_state(st)
        pu0 = np.random.normal(0, .1, size=(U, D))
        qi0 = np.random.normal(0, .1, size=(I, D))
        out.update({f"{name}_pu0": pu0, f"{name}_qi0": qi0, f"{name}_pu": a.pu, f"{name}_qi": a.qi,
                    f"{name}_bu": a.bu, f"{name}_bi": a.bi, f"{name}_mu": a.global_mean,
                    f"{name}_pred": np.array([a.predict(int(u), int(i)) for u, i in zip(users[:20], items[:20])])})
    for name, ver in (("rsvd_1", 1), ("rsvd_2", 2)):
        np.random.seed(2020)
        st = np.random.get_state()
        a = m.RSVD(U, I, n_factors=D, n_epochs=E, version=ver, lr=0.005, verbose=True)    # D5: verbose must be True
        with contextlib.redirect_stdout(io.StringIO()):
            a.fit(df)
        np.random.set_state(st)
        ui0 = np.random.normal(0, .1, size=(U, D))
        vj0 = np.random.normal(0, .1, size=(I, D))
        out.update({f"{name}_ui0": ui0, f"{name}_vj0": vj0, f"{name}_ui": a.ui, f"{name}_vj": a.vj,
                    f"{name}_ci": a.ci, f"{name}_dj": a.dj,
                    f"{name}_pred": np.array([a.predict(int(u), int(i)) for u, i in zip(users[:20], items[:20])])})
    np.savez_compressed(f"{HERE}/mf_small.npz", **out)
    print("mf_small written")


if __name__ == "__main__":
    os.chdir(HERE)
    tp, te, un, inum = make_split()
    make_bpr_small()
    make_config1_step(tp, un, inum)
    make_eval_small()
    make_mf_small()
    if "--skip-trajectory" not in sys.argv:
        make_trajectory(tp, te, un, inum)
