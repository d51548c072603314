"""Full-catalogue top-K (daisy_topk_full) on each of the paths that can serve it, with the path that ran asserted
through daisy_topk_full_path: the exact path (materialised fp32 scores + radix select), the CUDA-core candidate filter
and the tensor-core (BF16 tcgen05) candidate filter.  Every filter result must equal the exact path's items AND scores
bit for bit; on at most 64 users per shape both are also checked against float64 scores.

Reference tolerance: the fp32 fma chain of a D-term dot product is off by at most gamma_D |p_u| |q_i| with
gamma_D = D 2^-24 / (1 - D 2^-24), so every item whose float64 score beats the K-th by more than the two items' bounds
must be returned, and no returned item may sit more than that below the K-th.

Which path a call takes (topk_full.cu): catalogues of >= 131 072 items take a filter (the sample threshold's rank r is
then <= 128), the tensor-core one when dim <= 128 unless DAISY_TOPK_TC=0; DAISY_TOPK_PATH=exact forces the exact path.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

PATHS = ("exact", "filter-simt", "filter-tc")


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (there is no CPU fallback to test)"
    return torch.device("cuda:0")


def make_model(P0, Q0, dev):
    from recommend_lib_b200.bpr import BPR
    m = BPR(P0.shape[0], Q0.shape[0], P0.shape[1], max_batch=1024)
    with torch.no_grad():
        m.embed_user.weight.copy_(torch.from_numpy(np.asarray(P0, dtype=np.float32)))
        m.embed_item.weight.copy_(torch.from_numpy(np.asarray(Q0, dtype=np.float32)))
    return m.to(dev)


def run(m, monkeypatch, path, users, K, excl=None):
    """(items, scores) of one daisy_topk_full call on `path` (one of PATHS)."""
    from recommend_lib_b200.metrics import topk_full
    monkeypatch.setenv("DAISY_TOPK_PATH", "exact" if path == "exact" else "filter")
    monkeypatch.setenv("DAISY_TOPK_TC", "0" if path == "filter-simt" else "1")
    items, scores = topk_full(m, users, K, exclude=excl)
    return items.cpu().numpy(), scores.cpu().numpy()


def served(m):
    """(path, users the filter served, users the exact fallback redid) of the model's last daisy_topk_full call."""
    return m.handle().topk_full_path()


def random_exclusions(rng, N, I, most):
    lens = rng.integers(0, most, N)
    return np.split(rng.integers(0, I, int(lens.sum())).astype(np.int32), np.cumsum(lens)[:-1])


def assert_same(a, b, what):
    assert np.array_equal(a[0], b[0]), f"{what}: items differ in rows {np.nonzero((a[0] != b[0]).any(1))[0][:10]}"
    assert np.array_equal(a[1], b[1]), f"{what}: scores differ in rows {np.nonzero((a[1] != b[1]).any(1))[0][:10]}"


def check_against_float64(P0, Q0, users, K, got, excl=None):
    """The exact path's answer against float64 scores, with the per-item fp32 error bound of the module docstring."""
    items, scores = got
    N, D = len(users), P0.shape[1]
    gamma = D * 2.0 ** -24 / (1 - D * 2.0 ** -24)
    Q64 = Q0.astype(np.float64)
    qn = np.linalg.norm(Q64, axis=1)
    for n in np.unique(np.linspace(0, N - 1, min(N, 64)).astype(np.int64)):
        p = P0[users[n]].astype(np.float64)
        ref = Q64 @ p
        bound = gamma * np.linalg.norm(p) * qn
        if excl is not None and len(excl[n]):
            ref[excl[n]] = -np.inf
        it, sc = items[n], scores[n]
        assert len(np.unique(it)) == K and np.isfinite(ref[it]).all(), n            # distinct, none excluded
        assert (np.abs(sc.astype(np.float64) - ref[it]) <= bound[it]).all(), n
        assert (np.diff(sc) <= 0).all() and (np.diff(it)[np.diff(sc) == 0] > 0).all(), n   # score desc, ties item asc
        k = np.argsort(-ref, kind="stable")[K - 1]
        must = np.nonzero(ref - ref[k] > bound + bound[k])[0]
        assert np.isin(must, it).all(), n
        assert (ref[it] >= ref[k] - bound[it] - bound[k]).all(), n


# ---------------------------------------------------------------------------------------------------------------------
# the BF16 error bound of the tensor-core filter
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [64, 128])
def test_tensor_core_filter_keeps_items_that_bf16_rounding_pulls_down(dev, monkeypatch, D):
    """BF16 keeps 8 significant bits: 1 + 2^-8 rounds to 1, so a product can lose 2^-7 of itself.  The user row holds
    D/2 coordinates of 1 + 2^-8 and D/2 of 1.  300 sampled items (ids 16 j; 16 = I / 8192 is the sample stride) carry
    1 + 2^-7 on the second half: exact score D/2 (1 + 2^-7), exactly representable in BF16, so they set the threshold.
    Ten unsampled items carry 1 + 2^-8 on the first half: exact score D/2 (1 + 2^-7 + 2^-16), the true top 10, but BF16
    score D/2.  A threshold widened for a 2^-8 relative error per product drops all ten (and the call then returns
    the sampled items); the bound for 2^-7 keeps them.  300 users: enough for the filter to serve them all."""
    I, K, N, h = 131072, 10, 300, D // 2
    P0 = np.ones((N, D), np.float32)
    P0[:, :h] = 1 + 2.0 ** -8
    Q0 = np.zeros((I, D), np.float32)
    Q0[16 * np.arange(300), h:] = 1 + 2.0 ** -7
    top = 16 * np.arange(1000, 1010) + 8
    Q0[top, :h] = 1 + 2.0 ** -8
    m = make_model(P0, Q0, dev)
    users = np.arange(N, dtype=np.int32)
    exact = run(m, monkeypatch, "exact", users, K)
    assert (exact[0] == top).all() and (exact[1] == np.float32(h * (1 + 2.0 ** -7 + 2.0 ** -16))).all()
    check_against_float64(P0, Q0, users, K, exact)
    for path in ("filter-tc", "filter-simt"):
        got = run(m, monkeypatch, path, users, K)
        assert_same(exact, got, path)
        assert served(m) == (path, N, 0)


# ---------------------------------------------------------------------------------------------------------------------
# the tensor-core filter across dims (padding to 64 / 128 columns), user counts (partial and extra 256-user groups,
# a second 16 384-user tile), K and catalogue sizes (a multiple of the 128-item tile and not)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D,N,K,I", [(4, 1, 1, 131072), (4, 16385, 128, 300001), (32, 255, 20, 300001),
                                     (32, 257, 128, 131072), (64, 256, 128, 131072), (64, 1, 20, 300001),
                                     (68, 257, 1, 300001), (68, 255, 20, 131072), (100, 16385, 20, 131072),
                                     (100, 256, 1, 300001), (128, 1, 128, 300001), (128, 257, 20, 131072)])
def test_tensor_core_filter_is_bit_identical_to_exact_path(dev, monkeypatch, D, N, K, I):
    rng = np.random.default_rng(D * 1000 + N + K)
    U = max(N, 300)
    P0 = rng.standard_normal((U, D)).astype(np.float32)
    Q0 = rng.standard_normal((I, D)).astype(np.float32)
    Q0[rng.integers(0, I, I // 20)] = Q0[rng.integers(0, I, I // 20)]               # exactly tied scores
    users = rng.integers(0, U, N).astype(np.int32)
    m = make_model(P0, Q0, dev)
    exact = run(m, monkeypatch, "exact", users, K)
    assert served(m) == ("exact", 0, 0)
    got = run(m, monkeypatch, "filter-tc", users, K)
    assert served(m) == ("filter-tc", N, 0)
    assert_same(exact, got, "filter-tc")
    check_against_float64(P0, Q0, users, K, exact)


# ---------------------------------------------------------------------------------------------------------------------
# more than one user tile on each path, with exclusion lists (k_mask / k_select_topk / k_select_cand offsets)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path,N,I,D", [("exact", 2000, 300001, 32),        # exact tile: 2^30 / (4 I) = 894 users
                                        ("filter-simt", 4200, 131072, 32),  # CUDA-core filter tile: 4 096 users
                                        ("filter-tc", 16500, 131072, 64)])  # tensor-core filter tile: 16 384 users
def test_several_user_tiles_with_exclusions(dev, monkeypatch, path, N, I, D):
    rng = np.random.default_rng(N)
    U, K = 5000, 50
    P0 = rng.standard_normal((U, D)).astype(np.float32)
    Q0 = rng.standard_normal((I, D)).astype(np.float32)
    users = rng.integers(0, U, N).astype(np.int32)
    excl = random_exclusions(rng, N, I, 40)
    for n in range(0, N, 97):                    # and the user's own best items, so that the exclusions matter
        excl[n] = np.concatenate([excl[n], np.argpartition(Q0 @ P0[users[n]], -20)[-20:].astype(np.int32)])
    m = make_model(P0, Q0, dev)
    got = run(m, monkeypatch, path, users, K, excl)
    assert served(m) == ((path, N, 0) if path != "exact" else ("exact", 0, 0))
    # each user's answer does not depend on the tile it was computed in: users from every tile, alone
    pick = np.array([0, 1, 893, 894, 1788, 4095, 4096, 16383, 16384, N - 1])
    pick = pick[pick < N]
    alone = run(m, monkeypatch, "exact", users[pick], K, [excl[n] for n in pick])
    assert_same((got[0][pick], got[1][pick]), alone, "rows computed alone")
    if path == "exact":
        check_against_float64(P0, Q0, users, K, got, excl)
    else:
        assert_same(run(m, monkeypatch, "exact", users, K, excl), got, path)


# ---------------------------------------------------------------------------------------------------------------------
# fallbacks: a user whose candidate list cannot give K admissible items, or overflows, is redone by the exact path
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["filter-simt", "filter-tc"])
def test_user_whose_exclusions_remove_the_candidates_is_redone(dev, monkeypatch, path):
    rng = np.random.default_rng(3)
    U, I, D, N, K = 300, 131072, 32, 300, 20
    P0 = rng.standard_normal((U, D)).astype(np.float32)
    Q0 = rng.standard_normal((I, D)).astype(np.float32)
    users = np.arange(N, dtype=np.int32)
    excl = random_exclusions(rng, N, I, 10)
    excl[5] = np.argsort(Q0 @ P0[5])[-3000:].astype(np.int32)                       # more than the ~2 048 candidates
    m = make_model(P0, Q0, dev)
    got = run(m, monkeypatch, path, users, K, excl)
    path_run, filtered, redone = served(m)
    assert path_run == path and redone >= 1 and filtered + redone == N
    exact = run(m, monkeypatch, "exact", users, K, excl)
    assert_same(exact, got, path)
    check_against_float64(P0, Q0, users[:8], K, (exact[0][:8], exact[1][:8]), excl[:8])


@pytest.mark.parametrize("path", ["filter-simt", "filter-tc"])
def test_tie_of_more_than_the_candidate_cap_is_redone(dev, monkeypatch, path):
    """10 000 identical item rows score above everything else for every user: all of them reach the threshold, the
    candidate list (8 192 slots) overflows, and the exact path must take the 10 lowest ids of the tie."""
    rng = np.random.default_rng(4)
    U, I, D, N, K = 300, 131072, 32, 300, 10
    P0 = (1 + 0.1 * rng.standard_normal((U, D))).astype(np.float32)
    Q0 = (0.1 * rng.standard_normal((I, D))).astype(np.float32)
    tied = np.sort(rng.choice(I, 10000, replace=False))
    Q0[tied] = 1.0
    users = np.arange(N, dtype=np.int32)
    m = make_model(P0, Q0, dev)
    got = run(m, monkeypatch, path, users, K)
    path_run, filtered, redone = served(m)
    assert path_run == path and redone >= 1 and filtered + redone == N
    exact = run(m, monkeypatch, "exact", users, K)
    assert_same(exact, got, path)
    assert (exact[0] == tied[:K]).all()


# ---------------------------------------------------------------------------------------------------------------------
# candidates clustered in a few item tiles (a popularity-ordered catalogue): the reserved slots must not overflow
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [1, 200, 16384])
def test_clustered_candidates_need_no_fallback(dev, monkeypatch, N):
    """All items that can reach a user's top K sit in the first 2 % of the ids.  Each epilogue thread of the tensor-core
    filter reserves slots per chunk of item tiles up front; those reservations must leave room for the candidates,
    however they are spread over the chunks, at the user counts that split the catalogue finely (<= 256 users: one
    group, many chunks for balance) and coarsely (16 384)."""
    rng = np.random.default_rng(N)
    I, D, K = 131072, 64, 100
    U = max(N, 300)
    v = np.ones(D, np.float32)
    P0 = (v + 0.3 * rng.standard_normal((U, D))).astype(np.float32)
    Q0 = (0.3 * rng.standard_normal((I, D))).astype(np.float32)
    Q0[: I // 50] += v
    users = rng.integers(0, U, N).astype(np.int32)
    m = make_model(P0, Q0, dev)
    got = run(m, monkeypatch, "filter-tc", users, K)
    assert served(m) == ("filter-tc", N, 0)
    assert (got[0] < I // 50).all()
    exact = run(m, monkeypatch, "exact", users, K)
    assert_same(exact, got, "filter-tc")


# ---------------------------------------------------------------------------------------------------------------------
# negative thresholds
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["filter-simt", "filter-tc"])
def test_users_whose_scores_are_almost_all_negative(dev, monkeypatch, path):
    rng = np.random.default_rng(6)
    U, I, D, N, K = 300, 131072, 64, 300, 50
    v = np.ones(D, np.float32)
    P0 = (-v + 0.3 * rng.standard_normal((U, D))).astype(np.float32)
    Q0 = (v + 0.3 * rng.standard_normal((I, D))).astype(np.float32)
    users = np.arange(N, dtype=np.int32)
    m = make_model(P0, Q0, dev)
    got = run(m, monkeypatch, path, users, K)
    assert served(m) == (path, N, 0)
    assert (got[1] < 0).all()                                  # the whole top K, so the threshold, is below zero
    exact = run(m, monkeypatch, "exact", users, K)
    assert_same(exact, got, path)
    check_against_float64(P0, Q0, users, K, exact)


# ---------------------------------------------------------------------------------------------------------------------
# bad ids raise on every path
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", PATHS)
def test_bad_user_and_exclusion_ids_raise(dev, monkeypatch, path):
    rng = np.random.default_rng(8)
    U, I, D, N, K = 300, 131072, 32, 300, 10
    P0 = rng.standard_normal((U, D)).astype(np.float32)
    Q0 = rng.standard_normal((I, D)).astype(np.float32)
    users = np.arange(N, dtype=np.int32)
    m = make_model(P0, Q0, dev)
    bad_users = users.copy()
    bad_users[123] = U
    with pytest.raises(IndexError):
        run(m, monkeypatch, path, bad_users, K)
    for bad_item in (I, -1):
        excl = random_exclusions(rng, N, I, 10)
        excl[77] = np.array([3, bad_item, 5], np.int32)
        with pytest.raises(IndexError):
            run(m, monkeypatch, path, users, K, excl)
        assert served(m)[0] == path
    good = run(m, monkeypatch, path, users, K)                 # the error is reported once, the handle stays usable
    assert served(m) == ((path, N, 0) if path != "exact" else ("exact", 0, 0))
    assert_same(run(m, monkeypatch, "exact", users, K), good, path)
