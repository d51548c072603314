"""GPU tests of ranking with NCF's MLP / NeuMF towers (daisy_neumf_topk_candidates / daisy_neumf_topk_full through
metrics.topk_candidates, topk_full, metric_eval(algo='ncf') and final_kpi) against the float64 NeuMF oracle.

Ranking criterion (neumf_rank_testing.check_ranking), with eps(s) = 1e-4 |s| + 1e-5 as for forward() in
tests/test_neumf_gpu.py: returned scores within eps of the oracle's, ranks equal wherever the oracle's neighbouring
scores are more than 2 eps apart, nothing returned below the oracle's K-th score minus 2 eps."""
import numpy as np
import pytest

from neumf_rank_testing import check_ranking, oracle_scores, random_tower
from test_neumf_gpu import make, state

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (there is no CPU fallback to test)"
    return torch.device("cuda:0")


def tower(dev, model, U, I, F, L, seed):
    init = random_tower(np.random.default_rng(seed), U, I, F, L, model)
    return make(model, init, U, I, F, L, dev)[0], init


def bits(t):
    return t.cpu().numpy().view(np.int32)


# (model, U, I, F, L, N, C, K, repeated users)
CASES = [
    ("NeuMF-end", 943, 1682, 32, 3, 64, 1000, 10, False),   # the script's shape: 1 + 999 candidates, top 10
    ("MLP", 100, 300, 8, 1, 40, 200, 10, False),            # no hidden layer
    ("NeuMF-end", 50, 400, 128, 3, 12, 300, 10, False),     # the widest tower: factor * 2^L = 1024, W1 256 x 512
    ("NeuMF-end", 200, 700, 16, 4, 33, 333, 7, False),      # odd C, 4 layers
    ("MLP", 60, 80, 16, 2, 20, 17, 17, False),              # K = C
    ("NeuMF-end", 80, 900, 32, 3, 10, 500, 128, False),     # K = 128
    ("NeuMF-end", 20, 9000, 32, 3, 6, 8192, 50, True),      # C = 8192, the same user in several groups
]


@pytest.mark.parametrize("model,U,I,F,L,N,C,K,rep", CASES)
def test_neumf_topk_candidates_against_oracle(dev, model, U, I, F, L, N, C, K, rep):
    from recommend_lib_b200.metrics import topk_candidates
    m, init = tower(dev, model, U, I, F, L, U + C)
    rng = np.random.default_rng(C)
    users = rng.integers(0, U, N).astype(np.int32)
    if rep:
        users[:] = users[0]
        users[-1] = (users[0] + 1) % U
    cands = np.stack([rng.permutation(I)[:C] for _ in range(N)]).astype(np.int32)
    pos, items, scores = topk_candidates(m, users, cands, K)
    pos, items, scores = pos.cpu().numpy(), items.cpu().numpy(), scores.cpu().numpy()
    assert np.array_equal(items, np.take_along_axis(cands, pos, 1))
    check_ranking(pos, scores, oracle_scores(init, model, L, users, cands))


@pytest.mark.parametrize("exclude", [False, True])
def test_neumf_topk_full_against_oracle(dev, exclude):
    from recommend_lib_b200.metrics import topk_full
    U, I, F, L, N, K = 943, 1682, 32, 3, 77, 10              # N and I multiples of no tile size
    m, init = tower(dev, "NeuMF-end", U, I, F, L, 7)
    rng = np.random.default_rng(8)
    users = rng.choice(U, N, replace=False).astype(np.int32)
    excl = [rng.choice(I, int(rng.integers(0, 60)), replace=False) for _ in range(N)] if exclude else None
    items, scores = topk_full(m, users, K, exclude=excl)
    ora = oracle_scores(init, "NeuMF-end", L, users, np.tile(np.arange(I), (N, 1)))
    if exclude:
        for n in range(N):
            ora[n, excl[n]] = -np.inf
    check_ranking(items.cpu().numpy(), scores.cpu().numpy(), ora)


@pytest.mark.parametrize("model,F,L", [("NeuMF-end", 32, 3), ("MLP", 8, 1)])
def test_neumf_rank_invariants_bit_for_bit(dev, model, F, L):
    """Candidate mode on C = I candidates in item order == full mode; a user alone == the same user in a batch; two
    calls == each other."""
    from recommend_lib_b200.metrics import topk_candidates, topk_full
    U, I, N, K = 300, 1682, 200, 20
    m, _ = tower(dev, model, U, I, F, L, 3)
    users = np.random.default_rng(9).integers(0, U, N).astype(np.int32)
    fi, fs = topk_full(m, users, K)
    _, ci, cs = topk_candidates(m, users, np.tile(np.arange(I, dtype=np.int32), (N, 1)), K)
    assert torch.equal(fi, ci) and np.array_equal(bits(fs), bits(cs))
    fi2, fs2 = topk_full(m, users, K)
    assert torch.equal(fi, fi2) and np.array_equal(bits(fs), bits(fs2))
    for n in (0, 137, N - 1):
        ai, as_ = topk_full(m, users[n:n + 1], K)
        assert torch.equal(ai[0], fi[n]) and np.array_equal(bits(as_[0]), bits(fs[n]))
        _, bi, bs = topk_candidates(m, users[n:n + 1], np.arange(I, dtype=np.int32)[None], K)
        assert torch.equal(bi[0], fi[n]) and np.array_equal(bits(bs[0]), bits(fs[n]))


def test_neumf_metric_eval_and_final_kpi(dev):
    """metric_eval(model, loader, K, algo='ncf') == the reference's rule applied to forward() scores (as
    test_gmf_metric_eval checks for GMF); final_kpi == a CPU ranking of the same scores; algo='bpr' is refused."""
    from recommend_lib_b200.metrics import final_kpi, metric_eval, rank_metrics
    rng = np.random.default_rng(5)
    U, I, N, C, K = 80, 300, 60, 50, 10
    m, _ = tower(dev, "NeuMF-end", U, I, 16, 3, 5)
    users = rng.integers(0, U, N)
    cands = np.stack([rng.permutation(I)[:C] for _ in range(N)])
    loader = [(torch.full((C,), int(u)), torch.from_numpy(c.astype(np.int64)), torch.zeros(C)) for u, c in zip(users, cands)]
    hr, ndcg = metric_eval(m, loader, K, algo="ncf")
    want_hr, want_ndcg, tops = [], [], []
    for u, c in zip(users, cands):
        pred = m(torch.full((C,), int(u)), torch.from_numpy(c.astype(np.int64))).cpu().numpy()
        top = list(c[np.argsort(-pred, kind="stable")[:K]])
        tops.append(top)
        want_hr.append(1.0 if c[0] in top else 0.0)
        want_ndcg.append(1.0 / np.log2(top.index(c[0]) + 2.0) if c[0] in top else 0.0)
    assert hr == pytest.approx(np.mean(want_hr), abs=1e-12) and ndcg == pytest.approx(np.mean(want_ndcg), abs=1e-9)
    test_ur = [set(int(x) for x in rng.choice(c, 5, replace=False)) for c in cands]
    got = final_kpi(m, users, cands, test_ur, K)
    rel = np.array([[1 if int(e) in gt else 0 for e in top] for top, gt in zip(tops, test_ur)])
    want = rank_metrics(rel, [len(g) for g in test_ur], K)
    assert got == pytest.approx(want, abs=1e-12)
    with pytest.raises(ValueError):
        metric_eval(m, loader, K, algo="bpr")


def test_neumf_script_loop_hr_ndcg_match_the_oracle_ranking(golden, dev):
    """The script's loop at its defaults: ml-100k split, 4 negatives, NeuMF-end (factor 32, 3 layers), Adam at batch 256,
    two epochs, metric_eval(algo='ncf') on 1 + 999 candidates after each; HR@10 / NDCG@10 within one user of the float64
    oracle's ranking of the same weights."""
    from recommend_lib_b200 import data
    from recommend_lib_b200.metrics import metric_eval
    from recommend_lib_b200.ncf_mlp import NeuMF, NeuMFAdam
    from recommend_lib_b200.sampler import SampleSampler
    s = golden("ml100k_split.npz")
    tr, te = s["train_pairs"].astype(np.int64), s["test_pairs"].astype(np.int64)
    U, I = int(s["user_num"]), int(s["item_num"])
    allp = np.concatenate([tr, te])
    eu, ec = data.eval_candidates(allp[:, 0], allp[:, 1], te[:, 0], te[:, 1], I, 999, 2019)
    torch.manual_seed(2019)
    m = NeuMF(U, I, 32, 3, 0.0, "NeuMF-end").to(dev)
    opt = NeuMFAdam(m, lr=1e-3)
    sampler = SampleSampler(tr, I, num_ng=4, seed=2019)
    loader = [(torch.full((ec.shape[1],), int(u)), torch.from_numpy(c.astype(np.int64)), torch.zeros(ec.shape[1]))
              for u, c in zip(eu, ec)]
    for epoch in range(2):
        smp = torch.from_numpy(sampler.sample_epoch(epoch).astype(np.int64))
        for b in range(0, smp.shape[0], 256):
            opt.step(smp[b:b + 256, 0], smp[b:b + 256, 1], smp[b:b + 256, 2])
        hr, ndcg = metric_eval(m, loader, 10, algo="ncf")
        st = state(m)
        hits, gains = [], []
        for a in range(0, len(eu), 128):
            sc = oracle_scores(st, "NeuMF-end", 3, eu[a:a + 128], ec[a:a + 128])
            order = np.argsort(-sc, axis=1, kind="stable")[:, :10]      # (score desc, position asc)
            hit = order == 0
            hits += list(hit.any(1))
            gains += [1.0 / np.log2(r.argmax() + 2.0) if r.any() else 0.0 for r in hit]
        tol = 1.0 / len(eu) + 1e-12
        assert abs(hr - np.mean(hits)) <= tol and abs(ndcg - np.mean(gains)) <= tol, (epoch, hr, np.mean(hits), ndcg)
    m.check()


@pytest.mark.parametrize("what", ["user", "candidate", "exclusion"])
def test_neumf_rank_bad_ids_raise_index_error(dev, what):
    from recommend_lib_b200.metrics import topk_candidates, topk_full
    U, I = 50, 120
    m, _ = tower(dev, "NeuMF-end", U, I, 8, 3, 11)
    users = np.array([1, 2, 3], np.int32)
    cands = np.stack([np.arange(40)] * 3).astype(np.int32)
    with pytest.raises(IndexError):
        if what == "user":
            users[1] = U
            topk_candidates(m, users, cands, 5)
        elif what == "candidate":
            cands[2, 7] = I
            topk_candidates(m, users, cands, 5)
        else:
            topk_full(m, users, 5, exclude=[[1], [I + 3], []])
    items, _ = topk_full(m, users[:1], 5)                                 # the handle is usable afterwards
    assert items.shape == (1, 5)
