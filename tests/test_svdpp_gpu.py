"""GPU parity tests of SVD++ (SURVEY.md section 8f, row N4): daisy_svdpp_fit / daisy_svdpp_user_factors through the
drop-in SVDpp class against the golden run of the reference's own compiled Cython class (tests/golden/svdpp_small.npz)
and the C oracle (oracle/mf_oracle.c: mf_oracle_svdpp_fit, bit-identical to that class).

First run on a B200 in round 2 (profiles/r02a_*).
float64 on both sides; two sums are re-associated on the device (history rows over warps, factors over lanes), so
agreement is to rounding (1e-9 relative, as for funk-SVD), the sequential update ORDER is the reference's."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
pd = pytest.importorskip("pandas")

TOL = dict(rtol=1e-9, atol=1e-12)


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (there is no CPU fallback to test)"


def frame(users, items, ratings):
    return pd.DataFrame({"user": np.asarray(users, np.int64), "item": np.asarray(items, np.int64), "rating": ratings})


def fit_from(a, users, items, ratings, pu0, qi0, yj0):
    """fit() on given start tables (the reference draws them from numpy's global RNG inside fit)."""
    a.global_mean = float(np.asarray(ratings, np.float64).mean())
    pu, qi, yj = (np.array(x, dtype=np.float64) for x in (pu0, qi0, yj0))
    a._fit_arrays(np.ascontiguousarray(users, np.int32), np.ascontiguousarray(items, np.int32),
                  np.ascontiguousarray(ratings, np.float64), pu, qi, yj, np.zeros(a.user_num), np.zeros(a.item_num))
    return a


@pytest.mark.parametrize("threads", ["1024", "64"])
def test_svdpp_golden(golden, monkeypatch, threads):
    from recommend_lib_b200.svdpp import SVDpp
    monkeypatch.setenv("DAISY_SVDPP_THREADS", threads)
    g = golden("svdpp_small.npz")
    a = SVDpp(int(g["U"]), int(g["I"]), n_factors=int(g["D"]), n_epochs=int(g["E"]), verbose=False)
    fit_from(a, g["users"], g["items"], g["ratings"], g["pu0"], g["qi0"], g["yj0"])
    for k in ("pu", "qi", "yj", "bu", "bi"):
        assert np.allclose(getattr(a, k), g[k], **TOL), k
    assert np.isclose(a.global_mean, float(g["mu"]))
    pred = np.array([a.predict(int(u), int(i)) for u, i in zip(g["users"][:15], g["items"][:15])])
    assert np.allclose(pred, g["pred"], **TOL)
    assert np.allclose(a.predict_many(g["users"][:15], g["items"][:15]), g["pred"], **TOL)
    u0 = int(g["users"][0])
    assert [j for j, _ in a.ur[u0]] == g["items"][g["users"] == u0].tolist()
    with pytest.raises(ValueError, match="Invalid user code"):
        a.predict(int(g["U"]), 0)
    with pytest.raises(ValueError, match="Invalid item code"):
        a.predict(0, int(g["I"]))


def test_svdpp_fit_seeds_like_the_reference(golden):
    """np.random.seed reproduces the reference's start tables (pu, qi, yj drawn in that order, :221-224)."""
    from recommend_lib_b200.svdpp import SVDpp
    g = golden("svdpp_small.npz")
    U, I, D = int(g["U"]), int(g["I"]), int(g["D"])
    np.random.seed(7)
    a = SVDpp(U, I, n_factors=D, n_epochs=1, verbose=False)
    a.fit(frame(g["users"], g["items"], g["ratings"]))
    np.random.seed(7)
    pu0, qi0, yj0 = (np.random.normal(0, .1, size=s) for s in ((U, D), (I, D), (I, D)))
    b = fit_from(SVDpp(U, I, n_factors=D, n_epochs=1, verbose=False), g["users"], g["items"], g["ratings"], pu0, qi0, yj0)
    for k in ("pu", "qi", "yj", "bu", "bi"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k          # same kernel, same inputs: bit-identical


@pytest.mark.parametrize("U,I,D,n,E", [(300, 200, 128, 6000, 2),     # the script's width; histories of ~20 items
                                       (40, 500, 20, 5000, 1),       # the class default n_factors; histories > 32 rows
                                       (3, 60, 300, 7000, 1)])       # histories longer than the shared-memory list (2048)
def test_svdpp_against_c_oracle(U, I, D, n, E):
    from oracle import mf_oracle
    from recommend_lib_b200.svdpp import SVDpp
    rng = np.random.default_rng(D)
    users, items = rng.integers(0, U, n), rng.integers(0, I, n)
    ratings = rng.integers(1, 6, n).astype(np.float64)
    pu0, qi0, yj0 = (rng.normal(0, .1, s) for s in ((U, D), (I, D), (I, D)))
    ref = mf_oracle.svdpp_fit(users, items, ratings, pu0, qi0, yj0, n_epochs=E)
    a = fit_from(SVDpp(U, I, n_factors=D, n_epochs=E, verbose=False), users, items, ratings, pu0, qi0, yj0)
    for k in ("pu", "qi", "yj", "bu", "bi"):
        assert np.allclose(getattr(a, k), ref[k], **TOL), k
    assert np.isclose(a.sse_[E - 1], ref["sse"], rtol=1e-9)
    b = fit_from(SVDpp(U, I, n_factors=D, n_epochs=E, verbose=False), users, items, ratings, pu0, qi0, yj0)
    assert np.array_equal(a.yj, b.yj) and np.array_equal(a.pu, b.pu)      # run-to-run bit-reproducible


def test_svdpp_bad_item_raises_and_leaves_no_partial_state():
    from recommend_lib_b200.svdpp import SVDpp
    a = SVDpp(5, 4, n_factors=8, n_epochs=1, verbose=False)
    with pytest.raises(ValueError, match="Invalid item code"):
        a.fit(frame([0, 1, 2], [0, 4, 1], np.array([3., 4., 5.])))
    with pytest.raises(ValueError, match="Invalid user code"):
        a.fit(frame([0, 5, 2], [0, 1, 1], np.array([3., 4., 5.])))
