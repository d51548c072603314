"""GPU tests of ranking with BPR-FM models, with and without batch norm: metrics.topk_candidates, topk_full,
metric_eval and final_kpi over BPRFM(batch_norm=False) (its augmented training rows) and BPRFM(batch_norm=True) in
evaluation mode (tables folded by daisy_fmbn_rank_tables), against the float64 oracle (oracle/bprfm_oracle.py).

Ranking criterion (bprfm_rank_testing.check_ranking) with the per-pair tolerance of bprfm_rank_testing: returned scores
within eps of the oracle's, ranks equal wherever the oracle's neighbouring scores are further apart than their
tolerances, nothing returned below the oracle's K-th score minus twice its tolerance."""
import numpy as np
import pytest

from bprfm_rank_testing import check_ranking, oracle_scores, random_state

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (there is no CPU fallback to test)"
    return torch.device("cuda:0")


def make(st, U, dev):
    """BPRFM(batch_norm=st['bn']) holding the state st, on dev; a batch-norm model is put in evaluation mode."""
    from recommend_lib_b200.bprfm import BPRFM
    n, F = st["E"].shape
    bn = st["bn"]
    m = BPRFM(n, F, bn, [0.5, 0.2] if bn else [0.0, 0.0], user_num=U)
    with torch.no_grad():
        m.embeddings.weight.copy_(torch.from_numpy(st["E"]))
        m.biases.weight.copy_(torch.from_numpy(st["b"].reshape(-1, 1)))
        m.bias_.fill_(float(st["bias_"]))
        if bn:
            layer = m.FM_layers[0]
            for t, k in ((layer.weight, "gamma"), (layer.bias, "beta"), (layer.running_mean, "rm"), (layer.running_var, "rv")):
                t.copy_(torch.from_numpy(st[k]))
    m = m.to(dev)
    if bn:
        m.eval()
    return m


def model(dev, U, I, F, bn, seed):
    st = random_state(np.random.default_rng(seed), U, I, F, bn)
    return make(st, U, dev), st


def state(m):
    """The model's current state in the layout of bprfm_rank_testing.random_state (the plain model's rows read from the
    training buffer, which may be newer than embeddings / biases)."""
    c = lambda t: t.detach().cpu().numpy().astype(np.float32)
    st = dict(E=c(m.embeddings.weight), b=c(m.biases.weight).reshape(-1), bias_=np.float32(c(m.bias_)[0]), bn=m.batch_norm)
    if m.batch_norm:
        layer = m.FM_layers[0]
        st.update(gamma=c(layer.weight), beta=c(layer.bias), rm=c(layer.running_mean), rv=c(layer.running_var))
    elif m._aug is not None:
        F, U = m.num_factors, m.user_num
        st["E"] = c(m._aug[:, :F])
        st["b"][U:] = c(m._aug[U:, F])
    return st


def bits(t):
    return t.cpu().numpy().view(np.int32)


# (batch norm, U, I, F, N, C, K, repeated users)
CASES = [
    (True, 943, 1682, 64, 943, 1000, 10, False),    # the script's shape: hidden_factor 64, 1 + 999 candidates, top 10
    (False, 943, 1682, 64, 943, 1000, 10, False),
    (True, 100, 300, 1, 40, 200, 10, False),        # F = 1: W = 4
    (True, 100, 300, 7, 40, 200, 10, False),        # F = 7: W = 8, no padding beyond the bias column
    (True, 50, 400, 255, 12, 300, 10, False),       # F = 255: W = 256, the widest row
    (True, 60, 80, 16, 20, 17, 17, False),          # K = C
    (False, 60, 80, 16, 20, 17, 17, False),
    (True, 20, 9000, 32, 6, 8192, 50, True),        # C = 8192, the same user in several groups
    (False, 20, 9000, 32, 6, 8192, 50, True),
]


@pytest.mark.parametrize("bn,U,I,F,N,C,K,rep", CASES)
def test_bprfm_topk_candidates_against_oracle(dev, bn, U, I, F, N, C, K, rep):
    from recommend_lib_b200.metrics import topk_candidates
    m, st = model(dev, U, I, F, bn, U + C + F)
    rng = np.random.default_rng(C + F)
    users = (rng.permutation(U)[:N] if N <= U else rng.integers(0, U, N)).astype(np.int32)
    if rep:
        users[:] = users[0]
        users[-1] = (users[0] + 1) % U
    cands = np.stack([rng.permutation(I)[:C] for _ in range(N)]).astype(np.int32)
    pos, items, scores = topk_candidates(m, users, cands, K)
    pos, items, scores = pos.cpu().numpy(), items.cpu().numpy(), scores.cpu().numpy()
    assert np.array_equal(items, np.take_along_axis(cands, pos, 1))
    check_ranking(pos, scores, *oracle_scores(st, U, users, cands))


@pytest.mark.parametrize("bn", [True, False])
@pytest.mark.parametrize("exclude", [False, True])
def test_bprfm_topk_full_against_oracle(dev, bn, exclude):
    from recommend_lib_b200.metrics import topk_full
    U, I, F, N, K = 943, 1682, 64, 77, 10
    m, st = model(dev, U, I, F, bn, 7)
    rng = np.random.default_rng(8)
    users = rng.choice(U, N, replace=False).astype(np.int32)
    excl = [rng.choice(I, int(rng.integers(0, 60)), replace=False) for _ in range(N)] if exclude else None
    items, scores = topk_full(m, users, K, exclude=excl)
    ora, eps = oracle_scores(st, U, users, np.tile(np.arange(I), (N, 1)))
    if exclude:
        for n in range(N):
            ora[n, excl[n]] = -np.inf
    check_ranking(items.cpu().numpy(), scores.cpu().numpy(), ora, eps)


@pytest.mark.parametrize("bn", [True, False])
def test_bprfm_rank_invariants_bit_for_bit(dev, bn):
    """Within each mode a user alone == the same user in a batch, and two calls == each other; two folds of the same
    weights == each other.  Candidate mode on C = I candidates in item order returns full mode's items, and its scores
    within a few ulps: the two modes' unchanged kernels sum a dot product in different orders (k_topk_cand: per-lane
    float4 dots, then a warp tree; k_score_tile: one fma chain), as they do for every dot-product model."""
    from recommend_lib_b200.metrics import topk_candidates, topk_full
    U, I, F, N, K = 300, 1682, 64, 200, 20
    m, _ = model(dev, U, I, F, bn, 3)
    users = np.random.default_rng(9).integers(0, U, N).astype(np.int32)
    every = lambda n: np.tile(np.arange(I, dtype=np.int32), (n, 1))
    fi, fs = topk_full(m, users, K)
    _, ci, cs = topk_candidates(m, users, every(N), K)
    assert torch.equal(fi, ci)
    assert torch.allclose(fs, cs, rtol=1e-6, atol=0)
    fi2, fs2 = topk_full(m, users, K)
    _, ci2, cs2 = topk_candidates(m, users, every(N), K)
    assert torch.equal(fi, fi2) and np.array_equal(bits(fs), bits(fs2))
    assert torch.equal(ci, ci2) and np.array_equal(bits(cs), bits(cs2))
    for n in (0, 137, N - 1):
        ai, as_ = topk_full(m, users[n:n + 1], K)
        assert torch.equal(ai[0], fi[n]) and np.array_equal(bits(as_[0]), bits(fs[n]))
        _, bi, bs = topk_candidates(m, users[n:n + 1], every(1), K)
        assert torch.equal(bi[0], ci[n]) and np.array_equal(bits(bs[0]), bits(cs[n]))
    a, b = m.rank_tables(), m.rank_tables()
    for x, y in zip(a, b):
        assert (x is None and y is None) or np.array_equal(bits(x), bits(y))
    if bn:
        W = m.rank_width
        assert W == 68 and a[0].shape == (U, W) and a[1].shape == (I, W)
        assert bits(a[0][:, F + 1:]).max() == 0 and bits(a[1][:, F + 1:]).max() == 0 and (a[0][:, F] == 1).all()


@pytest.mark.parametrize("F,path", [(64, "filter-tc"), (255, "filter-simt")])
def test_bprfm_large_catalogue_filter_equals_exact(dev, monkeypatch, F, path):
    """At I >= 131 072 daisy_topk_full serves the folded tables through a candidate filter: the tensor-core one at
    F = 64 (W = 68 <= 128), the CUDA-core one at F = 255 (W = 256).  Its items and scores equal the exact path's bit for
    bit, and a few users are checked against the oracle."""
    from recommend_lib_b200.metrics import topk_full
    U, I, N, K = 300, 131072, 96, 100
    m, st = model(dev, U, I, F, True, F)
    rng = np.random.default_rng(F)
    users = rng.choice(U, N, replace=False).astype(np.int32)
    excl = [rng.choice(I, int(rng.integers(0, 40)), replace=False) for _ in range(N)]
    out = {}
    for p in ("exact", path):
        monkeypatch.setenv("DAISY_TOPK_PATH", "exact" if p == "exact" else "filter")
        monkeypatch.setenv("DAISY_TOPK_TC", "1")
        items, scores = topk_full(m, users, K, exclude=excl)
        out[p] = items.cpu().numpy(), scores.cpu().numpy()
        served, filtered, redone = m.handle().topk_full_path()
        assert served == p and filtered + redone == (N if p != "exact" else 0), (p, served, filtered, redone)
    assert np.array_equal(out["exact"][0], out[path][0])
    assert np.array_equal(out["exact"][1].view(np.int32), out[path][1].view(np.int32))
    few = np.arange(0, N, 24)
    ora, eps = oracle_scores(st, U, users[few], np.tile(np.arange(I), (len(few), 1)))
    for r, n in enumerate(few):
        ora[r, excl[n]] = -np.inf
    check_ranking(out[path][0][few], out[path][1][few], ora, eps)


def test_bprfm_bn_rankings_follow_training(dev):
    """After FMBNAdagrad steps (weights, gamma / beta and running statistics all move) the ranking in evaluation mode is
    within eps of the oracle fed the updated state."""
    from recommend_lib_b200.bprfm_bn import FMBNAdagrad
    from recommend_lib_b200.metrics import topk_candidates, topk_full
    U, I, F, B, N, C, K = 200, 500, 32, 1024, 50, 300, 10
    m, st0 = model(dev, U, I, F, True, 21)
    m.train()
    opt = FMBNAdagrad(m, lr=0.05)
    rng = np.random.default_rng(22)
    for _ in range(3):
        tri = np.stack([rng.integers(0, U, B), rng.integers(0, I, B), rng.integers(0, I, B)], 1).astype(np.int32)
        opt.step(torch.from_numpy(tri).to(dev))
    m.check()
    m.eval()
    st = state(m)
    assert not np.array_equal(st["rm"], st0["rm"]) and not np.array_equal(st["rv"], st0["rv"])
    users = rng.choice(U, N, replace=False).astype(np.int32)
    cands = np.stack([rng.permutation(I)[:C] for _ in range(N)]).astype(np.int32)
    pos, _, scores = topk_candidates(m, users, cands, K)
    check_ranking(pos.cpu().numpy(), scores.cpu().numpy(), *oracle_scores(st, U, users, cands))
    items, scores = topk_full(m, users, K)
    check_ranking(items.cpu().numpy(), scores.cpu().numpy(), *oracle_scores(st, U, users, np.tile(np.arange(I), (N, 1))))


def test_bprfm_rankings_use_unsynced_training_rows(dev):
    """The plain model ranks its augmented training rows: after FMAdagrad steps that were not sync()ed, embeddings /
    biases are stale and the ranking follows the trained rows."""
    from recommend_lib_b200.bprfm import FMAdagrad
    from recommend_lib_b200.metrics import topk_candidates, topk_full
    U, I, F, B, N, C, K = 200, 500, 32, 1024, 50, 300, 10
    m, _ = model(dev, U, I, F, False, 31)
    opt = FMAdagrad(m, lr=0.05, initial_accumulator_value=0.1)
    rng = np.random.default_rng(32)
    for _ in range(3):
        tri = np.stack([rng.integers(0, U, B), rng.integers(0, I, B), rng.integers(0, I, B)], 1).astype(np.int32)
        opt.step(torch.from_numpy(tri).to(dev))
    m.check()
    assert m._dirty
    st = state(m)
    assert not np.allclose(st["E"], m.embeddings.weight.cpu().numpy(), rtol=0, atol=1e-4)     # not synced yet
    users = rng.choice(U, N, replace=False).astype(np.int32)
    cands = np.stack([rng.permutation(I)[:C] for _ in range(N)]).astype(np.int32)
    pos, _, scores = topk_candidates(m, users, cands, K)
    check_ranking(pos.cpu().numpy(), scores.cpu().numpy(), *oracle_scores(st, U, users, cands))
    items, scores = topk_full(m, users, K)
    check_ranking(items.cpu().numpy(), scores.cpu().numpy(), *oracle_scores(st, U, users, np.tile(np.arange(I), (N, 1))))
    assert m._dirty


@pytest.mark.parametrize("bn", [True, False])
def test_bprfm_metric_eval_and_final_kpi(dev, bn):
    """metric_eval(model, loader, K) with either algo == HR / NDCG of the oracle's (score desc, position asc) ranking of
    the same groups; final_kpi == the six metrics of a CPU ranking of the oracle's scores."""
    from recommend_lib_b200.metrics import final_kpi, metric_eval, rank_metrics
    rng = np.random.default_rng(5)
    U, I, F, N, C, K = 80, 300, 16, 60, 50, 10
    m, st = model(dev, U, I, F, bn, 5)
    users = rng.integers(0, U, N)
    cands = np.stack([rng.permutation(I)[:C] for _ in range(N)])
    loader = [(torch.full((C,), int(u)), torch.from_numpy(c.astype(np.int64)), torch.zeros(C)) for u, c in zip(users, cands)]
    ora, _ = oracle_scores(st, U, users, cands)
    order = np.argsort(-ora, axis=1, kind="stable")[:, :K]
    tops = np.take_along_axis(cands, order, 1)
    hit = order == 0
    want_hr = hit.any(1).mean()
    want_ndcg = np.mean([1.0 / np.log2(r.argmax() + 2.0) if r.any() else 0.0 for r in hit])
    for algo in ("bpr", "ncf"):
        hr, ndcg = metric_eval(m, loader, K, algo=algo)
        assert hr == pytest.approx(want_hr, abs=1e-12) and ndcg == pytest.approx(want_ndcg, abs=1e-12), algo
    test_ur = [set(int(x) for x in rng.choice(c, 5, replace=False)) for c in cands]
    got = final_kpi(m, users, cands, test_ur, K)
    rel = np.array([[1 if int(e) in gt else 0 for e in top] for top, gt in zip(tops, test_ur)])
    want = rank_metrics(rel, [len(g) for g in test_ur], K)
    assert got == pytest.approx(want, abs=1e-12)


@pytest.mark.parametrize("bn", [True, False])
@pytest.mark.parametrize("what", ["user", "candidate", "exclusion"])
def test_bprfm_rank_bad_ids_raise_index_error(dev, bn, what):
    from recommend_lib_b200.metrics import topk_candidates, topk_full
    U, I = 50, 120
    m, _ = model(dev, U, I, 8, bn, 11)
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
    m.check()


def test_bprfm_bn_ranking_in_training_mode_raises(dev):
    from recommend_lib_b200.metrics import topk_candidates, topk_full
    m, _ = model(dev, 50, 120, 8, True, 12)
    m.train()
    with pytest.raises(RuntimeError, match="model.eval"):
        m.rank_tables()
    with pytest.raises(RuntimeError, match="model.eval"):
        topk_candidates(m, np.array([1], np.int32), np.arange(40, dtype=np.int32)[None], 5)
    with pytest.raises(RuntimeError, match="model.eval"):
        topk_full(m, np.array([1], np.int32), 5)
