"""GPU parity tests of the funk-SVD / RSVD path against the reference's compiled Cython extension (golden fixtures)
and the C oracle.  float64 on both sides; the device computes the dot product with a warp tree instead of a
left-to-right loop, so agreement is to rounding (1e-9 relative stated here), not bit-exact; the sequential update ORDER
is the reference's."""
import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
pd = pytest.importorskip("pandas")

TOL = 1e-9


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"


@pytest.fixture(params=["owner", "ticket"], autouse=True)
def _schedule(request, monkeypatch):
    """Both dataflow schedules of daisy_mf_fit (csrc/mf.cu): item-owner warps (default) and the ticket schedule."""
    monkeypatch.setenv("DAISY_MF_SCHEDULE", request.param)
    return request.param


def frame(g):
    return pd.DataFrame({"user": g["users"].astype(np.int64), "item": g["items"].astype(np.int64),
                         "rating": g["ratings"]})


@pytest.mark.parametrize("name,kw", [("svd_b", dict(biased=True)), ("svd_u", dict(biased=False, lr_all=0.01, reg_all=0.05))])
def test_svd_golden(golden, name, kw):
    from recommend_lib_b200.mf import SVD
    g = golden("mf_small.npz")
    np.random.seed(2019)                                   # the fixture was produced under this seed
    a = SVD(int(g["U"]), int(g["I"]), n_factors=int(g["D"]), n_epochs=int(g["E"]), verbose=False, **kw)
    assert a.fit(frame(g)) is None
    for k in ("pu", "qi", "bu", "bi"):
        ref = g[f"{name}_{k}"]
        if np.abs(ref).max() > 0:
            assert rel_err(getattr(a, k), ref) <= TOL, k
        else:
            assert np.abs(getattr(a, k)).max() == 0, k
    assert a.global_mean == pytest.approx(float(g[f"{name}_mu"]), abs=1e-15)
    pred = np.array([a.predict(int(u), int(i)) for u, i in zip(g["users"][:20], g["items"][:20])])
    assert np.allclose(pred, g[f"{name}_pred"], rtol=1e-9, atol=1e-12)
    assert np.allclose(a.predict_many(g["users"][:20], g["items"][:20]), g[f"{name}_pred"], rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("name,version", [("rsvd_1", 1), ("rsvd_2", 2)])
def test_rsvd_golden(golden, name, version):
    from recommend_lib_b200.mf import RSVD
    g = golden("mf_small.npz")
    np.random.seed(2020)
    a = RSVD(int(g["U"]), int(g["I"]), n_factors=int(g["D"]), n_epochs=int(g["E"]), version=version, lr=0.005,
             verbose=False)
    a.fit(frame(g))
    for k in ("ui", "vj", "ci", "dj"):
        ref = g[f"{name}_{k}"]
        if np.abs(ref).max() > 0:
            assert rel_err(getattr(a, k), ref) <= TOL, k
        else:
            assert np.abs(getattr(a, k)).max() == 0, k
    pred = np.array([a.predict(int(u), int(i)) for u, i in zip(g["users"][:20], g["items"][:20])])
    assert np.allclose(pred, g[f"{name}_pred"], rtol=1e-9, atol=1e-12)


def test_predict_errors(golden):
    from recommend_lib_b200.mf import SVD
    g = golden("mf_small.npz")
    np.random.seed(1)
    a = SVD(int(g["U"]), int(g["I"]), n_factors=int(g["D"]), n_epochs=1, verbose=False)
    a.fit(frame(g))
    with pytest.raises(ValueError, match="Invalid user code"):
        a.predict(int(g["U"]), 0)
    with pytest.raises(ValueError, match="Invalid item code"):
        a.predict(0, int(g["I"]))
    with pytest.raises(ValueError, match="Invalid user code"):
        a.predict_many([0, int(g["U"])], [0, 0])
    with pytest.raises(ValueError, match="Invalid item code"):
        a.predict_many([0, 1], [0, int(g["I"])])
    bad = frame(g)
    bad.loc[3, "item"] = int(g["I"]) + 5
    with pytest.raises(IndexError):
        a.fit(bad)


@pytest.mark.parametrize("variant", ["svd", "rsvd2"])
def test_config2_shape_against_c_oracle(variant):
    """ml-1m shape (6040 x 3706, D 128), Zipf items: long dependency chains through the hot items."""
    from oracle import mf_oracle
    from recommend_lib_b200.mf import SVD, RSVD
    from recommend_lib_b200.sampler import synthetic_ratings
    U, I, D, N, E = 6040, 3706, 128, 200_000, 2
    users, items, ratings = synthetic_ratings(N, U, I, seed=2019)
    df = pd.DataFrame({"user": users, "item": items, "rating": ratings})
    np.random.seed(5)
    st = np.random.get_state()
    if variant == "svd":
        a = SVD(U, I, n_factors=D, n_epochs=E, verbose=False)
        a.fit(df)
        np.random.set_state(st)
        p0, q0 = mf_oracle.draw_init(U, I, D)
        o = mf_oracle.svd_fit(users, items, ratings, p0, q0, n_epochs=E)
        got = (a.pu, a.qi, a.bu, a.bi)
        want = (o["pu"], o["qi"], o["bu"], o["bi"])
    else:
        a = RSVD(U, I, n_factors=D, n_epochs=E, version=2, verbose=False)
        a.fit(df)
        np.random.set_state(st)
        p0, q0 = mf_oracle.draw_init(U, I, D)
        o = mf_oracle.rsvd_fit(users, items, ratings, p0, q0, n_epochs=E, version=2)
        got = (a.ui, a.vj, a.ci, a.dj)
        want = (o["ui"], o["vj"], o["ci"], o["dj"])
    for x, y in zip(got, want):
        assert rel_err(x, y) <= 1e-8
    assert a.sse_[-1] == pytest.approx(o["sse"], rel=1e-9)          # epoch loss, last epoch
    assert a.sse_[0] > a.sse_[-1]


def test_single_hot_row_chain_and_determinism():
    """Every rating shares one item: the schedule degenerates to a pure chain and must still finish, twice the same."""
    from oracle import mf_oracle
    from recommend_lib_b200.mf import SVD
    rng = np.random.default_rng(0)
    U, I, D, N = 500, 7, 16, 20000
    users = rng.integers(0, U, N).astype(np.int32)
    items = np.full(N, 3, dtype=np.int32)
    ratings = rng.integers(1, 6, N).astype(np.float64)
    df = pd.DataFrame({"user": users, "item": items, "rating": ratings})
    outs = []
    for _ in range(2):
        np.random.seed(9)
        a = SVD(U, I, n_factors=D, n_epochs=2, verbose=False)
        a.fit(df)
        outs.append((a.pu.copy(), a.qi.copy()))
    assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1])
    np.random.seed(9)
    p0, q0 = mf_oracle.draw_init(U, I, D)
    o = mf_oracle.svd_fit(users, items, ratings, p0, q0, n_epochs=2)
    assert rel_err(outs[0][0], o["pu"]) <= 1e-9 and rel_err(outs[0][1], o["qi"]) <= 1e-9


def test_batched_groups_match_the_link_by_link_schedule_and_are_reproducible(monkeypatch, _schedule):
    """k_mf_owner takes a full group of 8 links on one item with distinct users through the batched form (all dot
    products at once, scalar recurrence for the chain).  Which groups are batched follows from the rating list alone,
    and the batched arithmetic is the same whether or not every row was ready -- so two runs agree bit for bit even
    with warps racing each other -- and the result agrees with the link-by-link schedule (DAISY_MF_BATCH=0) and the C
    oracle to rounding.  Hot items (Zipf) and all three bias variants."""
    if _schedule != "owner":
        pytest.skip("item-owner schedule only")
    from oracle import mf_oracle
    from recommend_lib_b200.mf import SVD, RSVD
    from recommend_lib_b200.sampler import synthetic_ratings
    U, I, D, N, E = 2000, 300, 128, 120_000, 3
    users, items, ratings = synthetic_ratings(N, U, I, seed=77)
    df = pd.DataFrame({"user": users, "item": items, "rating": ratings})
    for make, names, ofit in ((lambda: SVD(U, I, n_factors=D, n_epochs=E, verbose=False), ("pu", "qi", "bu", "bi"),
                               lambda p0, q0: mf_oracle.svd_fit(users, items, ratings, p0, q0, n_epochs=E)),
                              (lambda: RSVD(U, I, n_factors=D, n_epochs=E, version=1, verbose=False), ("ui", "vj", "ci", "dj"),
                               lambda p0, q0: mf_oracle.rsvd_fit(users, items, ratings, p0, q0, n_epochs=E, version=1)),
                              (lambda: RSVD(U, I, n_factors=D, n_epochs=E, version=2, verbose=False), ("ui", "vj", "ci", "dj"),
                               lambda p0, q0: mf_oracle.rsvd_fit(users, items, ratings, p0, q0, n_epochs=E, version=2))):
        runs = {}
        for tag, env in (("b1", "1"), ("b2", "1"), ("seq", "0")):
            monkeypatch.setenv("DAISY_MF_BATCH", env)
            np.random.seed(11)
            a = make()
            a.fit(df)
            runs[tag] = [np.array(getattr(a, k)).copy() for k in names]
        for x, y in zip(runs["b1"], runs["b2"]):
            assert np.array_equal(x, y)
        for x, y in zip(runs["b1"], runs["seq"]):
            assert rel_err(x, y) <= 1e-10
        np.random.seed(11)
        p0, q0 = mf_oracle.draw_init(U, I, D)
        o = ofit(p0, q0)
        for x, k in zip(runs["b1"], names):
            assert rel_err(x, o[k]) <= TOL, k


def test_many_items_per_warp_and_wide_rows():
    """More items than resident warps (every warp multiplexes several items) and D = 200 (7 doubles per lane)."""
    from oracle import mf_oracle
    from recommend_lib_b200.mf import SVD
    rng = np.random.default_rng(1)
    U, I, D, N = 3000, 60000, 200, 150_000
    users = rng.integers(0, U, N).astype(np.int32)
    items = (rng.zipf(1.3, N) % I).astype(np.int32)
    ratings = rng.integers(1, 6, N).astype(np.float64)
    df = pd.DataFrame({"user": users, "item": items, "rating": ratings})
    np.random.seed(11)
    a = SVD(U, I, n_factors=D, n_epochs=2, verbose=False)
    a.fit(df)
    np.random.seed(11)
    p0, q0 = mf_oracle.draw_init(U, I, D)
    o = mf_oracle.svd_fit(users, items, ratings, p0, q0, n_epochs=2)
    for x, y in zip((a.pu, a.qi, a.bu, a.bi), (o["pu"], o["qi"], o["bu"], o["bi"])):
        assert rel_err(x, y) <= 1e-8
