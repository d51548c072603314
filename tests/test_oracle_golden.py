"""Pin the CPU oracle against fixtures produced by the UNMODIFIED reference (tests/golden/make_golden.py)."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, rel_err
from oracle import bpr_oracle, mf_oracle


# ---------------------------------------------------------------- BPR step
def test_closed_form_matches_reference_small(golden):
    g = golden("bpr_small.npz")
    P, Q = g["P0"], g["Q0"]
    for k, batch in enumerate(g["batches"]):
        P, Q, loss = bpr_oracle.bpr_step_closed_form(P, Q, batch, float(g["lr"]), float(g["wd"]), np.float64)
        assert rel_err(P, g["P"][k]) < 2e-6, k
        assert rel_err(Q, g["Q"][k]) < 2e-6, k
        assert abs(loss - g["losses"][k]) / g["losses"][k] < 1e-5


def test_closed_form_fp32_matches_reference_small(golden):
    g = golden("bpr_small.npz")
    P, Q = g["P0"], g["Q0"]
    for k, batch in enumerate(g["batches"]):
        P, Q, _ = bpr_oracle.bpr_step_closed_form(P, Q, batch, float(g["lr"]), float(g["wd"]), np.float32)
        assert rel_err(P, g["P"][k]) < 1e-5 and rel_err(Q, g["Q"][k]) < 1e-5


def test_torch_port_is_bit_identical_to_reference_small(golden):
    g = golden("bpr_small.npz")
    port = bpr_oracle.TorchPort(g["P0"], g["Q0"], float(g["lr"]), float(g["wd"]))
    for k, batch in enumerate(g["batches"]):
        loss = port.step(batch)
        P, Q = port.tables()
        assert np.array_equal(P, g["P"][k]) and np.array_equal(Q, g["Q"][k])
        assert loss == pytest.approx(float(g["losses"][k]), rel=1e-6)


def test_sparse_adam_closed_form_is_pinned_to_torch_sparse_adam():
    """Lazy sparse Adam has no Daisy counterpart (BPRMFRecommender.py:154 is optim.SGD): its stated oracle is
    torch.optim.SparseAdam on nn.Embedding(sparse=True) under the reference's loss (BPRMFRecommender.py:172-176).
    Four steps with repeated rows, rows that skip steps (their moments must stay put), float64 and float32."""
    import torch
    rng = np.random.default_rng(5)
    U, I, D, B = 40, 30, 16, 200
    P0 = (rng.standard_normal((U, D)) * 0.3)
    Q0 = (rng.standard_normal((I, D)) * 0.3)
    batches = []
    for k in range(4):
        t = np.stack([rng.integers(0, U - 5 * (k % 2), B), rng.integers(0, I // 2, B), rng.integers(0, I, B)], 1)
        t[:40, 1] = 3                                     # a hot positive item
        batches.append(t.astype(np.int32))
    for dtype, tdtype, tol in ((np.float64, torch.float64, 1e-12), (np.float32, torch.float32, 1e-5)):
        eu = torch.nn.Embedding(U, D, sparse=True, dtype=tdtype)
        ei = torch.nn.Embedding(I, D, sparse=True, dtype=tdtype)
        with torch.no_grad():
            eu.weight.copy_(torch.from_numpy(P0))
            ei.weight.copy_(torch.from_numpy(Q0))
        opt = torch.optim.SparseAdam(list(eu.parameters()) + list(ei.parameters()), lr=0.01)
        P, Q = P0.astype(dtype), Q0.astype(dtype)
        st = [np.zeros_like(P), np.zeros_like(P), np.zeros_like(Q), np.zeros_like(Q)]
        for k, b in enumerate(batches):
            u, i, j = (torch.from_numpy(b[:, c].astype(np.int64)) for c in range(3))
            opt.zero_grad()
            pu = eu(u)
            loss_t = -((pu * ei(i)).sum(-1) - (pu * ei(j)).sum(-1)).sigmoid().log().sum()
            loss_t.backward()
            opt.step()
            P, Q, st[0], st[1], st[2], st[3], loss = bpr_oracle.bpr_adam_step_closed_form(P, Q, *st, b, k + 1, 0.01,
                                                                                          dtype=dtype)
            assert abs(loss - float(loss_t.detach())) / float(loss_t.detach()) < 1e-6
            assert rel_err(P, eu.weight.detach().numpy()) <= tol, (dtype, k)
            assert rel_err(Q, ei.weight.detach().numpy()) <= tol, (dtype, k)
        sP, sQ = opt.state[eu.weight], opt.state[ei.weight]
        assert rel_err(st[0], sP["exp_avg"].numpy()) <= tol and rel_err(st[1], sP["exp_avg_sq"].numpy()) <= tol
        assert rel_err(st[2], sQ["exp_avg"].numpy()) <= tol and rel_err(st[3], sQ["exp_avg_sq"].numpy()) <= tol


def test_forward_matches_reference(golden):
    g = golden("bpr_small.npz")
    b = g["batches"][0]
    pi, pj = bpr_oracle.bpr_scores(g["P"][-1], g["Q"][-1], b[:, 0], b[:, 1], b[:, 2])
    assert np.allclose(pi, g["fwd_pred_i"], rtol=1e-5, atol=1e-7)
    assert np.allclose(pj, g["fwd_pred_j"], rtol=1e-5, atol=1e-7)


def test_config1_first_step(golden):
    g = {**golden("bpr_config1_step.npz"), **golden("bpr_config1_step_after.npz")}
    P1, Q1, loss = bpr_oracle.bpr_step_closed_form(g["P0"], g["Q0"], g["batch"], 0.01, 0.001, np.float64)
    assert rel_err(P1, g["P1"]) < 1e-6 and rel_err(Q1, g["Q1"]) < 1e-6
    assert abs(loss - float(g["loss"])) / float(g["loss"]) < 1e-6
    # untouched rows shrink by exactly 1 - lr*wd (dense decay, SURVEY 3.2)
    untouched = np.setdiff1d(np.arange(g["P0"].shape[0]), g["batch"][:, 0])
    if untouched.size:
        assert np.allclose(g["P1"][untouched], g["P0"][untouched] * (1 - 1e-5), rtol=2e-7, atol=0)
    port = bpr_oracle.TorchPort(g["P0"], g["Q0"], 0.01, 0.001)
    port.step(g["batch"])
    P, Q = port.tables()
    assert np.array_equal(P, g["P1"]) and np.array_equal(Q, g["Q1"])


def test_sampler_reproduces_golden_batch(golden):
    """The fixture's batch came from TripleSampler(seed 2019): the sampler must be reproducible."""
    from recommend_lib_b200.sampler import TripleSampler
    g = golden("bpr_config1_step.npz")
    s = golden("ml100k_split.npz")
    sampler = TripleSampler(s["train_pairs"].astype(np.int64), int(s["item_num"]), num_ng=4, seed=2019)
    batch = next(iter(sampler.batches(0, 4096)))
    assert np.array_equal(batch, g["batch"])


# ---------------------------------------------------------------- eval
def test_eval_matches_reference_metric_eval(golden):
    g = golden("bpr_eval_small.npz")
    hr, ndcg, top = bpr_oracle.bpr_topk_eval(g["P"], g["Q"], g["users"], g["cands"], int(g["top_k"]))
    assert hr == pytest.approx(float(g["hr"]), abs=1e-12)
    assert ndcg == pytest.approx(float(g["ndcg"]), abs=1e-9)
    assert 0.0 < hr < 1.0


def test_topk_order_ties():
    assert list(bpr_oracle.topk_order(np.array([1., 3., 3., 2., 3., 0.]), 3)) == [1, 2, 4]


def test_trajectory_fixture_is_sane():
    path = os.path.join(GOLDEN, "bpr_ml100k_traj.json")
    if not os.path.exists(path):
        pytest.skip("trajectory fixture not generated")
    t = json.load(open(path))
    ep = t["epochs"]
    assert len(ep) == 20 and ep[0]["loss"] > ep[-1]["loss"]
    assert abs(ep[0]["loss"] - 396228 * np.log(2)) / ep[0]["loss"] < 0.01     # BASELINE.md: epoch 1 ~ N ln 2
    assert 0.15 < ep[-1]["hr"] < 0.25                                         # BASELINE.md: HR@10 ~ 0.204


# ---------------------------------------------------------------- funk-SVD / RSVD
@pytest.mark.parametrize("name,biased,kw", [("svd_b", True, {}), ("svd_u", False, dict(lr_all=0.01, reg_all=0.05))])
def test_svd_c_oracle_bit_identical_to_cython_reference(golden, name, biased, kw):
    g = golden("mf_small.npz")
    o = mf_oracle.svd_fit(g["users"], g["items"], g["ratings"], g[f"{name}_pu0"], g[f"{name}_qi0"],
                          n_epochs=int(g["E"]), biased=biased, **kw)
    for k in ("pu", "qi", "bu", "bi"):
        assert np.array_equal(o[k], g[f"{name}_{k}"]), k
    assert o["global_mean"] == float(g[f"{name}_mu"])
    for n in range(20):
        est = mf_oracle.predict(g["users"][n], g["items"][n], o["pu"], o["qi"], o["bu"], o["bi"], biased, o["global_mean"])
        assert est == pytest.approx(g[f"{name}_pred"][n], rel=1e-12, abs=1e-14)


@pytest.mark.parametrize("name,version", [("rsvd_1", 1), ("rsvd_2", 2)])
def test_rsvd_c_oracle_bit_identical_to_cython_reference(golden, name, version):
    g = golden("mf_small.npz")
    o = mf_oracle.rsvd_fit(g["users"], g["items"], g["ratings"], g[f"{name}_ui0"], g[f"{name}_vj0"],
                           n_epochs=int(g["E"]), version=version, lr=0.005)
    for k in ("ui", "vj", "ci", "dj"):
        assert np.array_equal(o[k], g[f"{name}_{k}"]), k
    for n in range(20):
        est = mf_oracle.predict(g["users"][n], g["items"][n], o["ui"], o["vj"], o["ci"], o["dj"], version == 2)
        assert est == pytest.approx(g[f"{name}_pred"][n], rel=1e-12, abs=1e-14)


def test_predict_rejects_invalid_codes(golden):
    g = golden("mf_small.npz")
    z = np.zeros(1)
    with pytest.raises(ValueError, match="Invalid user code"):
        mf_oracle.predict(int(g["U"]), 0, g["svd_b_pu"], g["svd_b_qi"], g["svd_b_bu"], g["svd_b_bi"], True)
    with pytest.raises(ValueError, match="Invalid item code"):
        mf_oracle.predict(0, int(g["I"]), g["svd_b_pu"], g["svd_b_qi"], g["svd_b_bu"], g["svd_b_bi"], True)


def test_seeded_draw_and_fit_match_the_reference_extension_golden(golden):
    """The reference's SVD.fit draws its start from the global numpy RNG: draw_init under the seed of the fixture's run,
    then svd_fit, ends bit for bit where the compiled reference ended (mf_small.npz, seed 2019)."""
    g = golden("mf_small.npz")
    np.random.seed(2019)
    pu0, qi0 = mf_oracle.draw_init(int(g["U"]), int(g["I"]), int(g["D"]))
    assert np.array_equal(pu0, g["svd_b_pu0"]) and np.array_equal(qi0, g["svd_b_qi0"])
    o = mf_oracle.svd_fit(g["users"], g["items"], g["ratings"], pu0, qi0, n_epochs=int(g["E"]))
    assert np.array_equal(o["pu"], g["svd_b_pu"]) and np.array_equal(o["qi"], g["svd_b_qi"])


# ------------------------------------------------------------------------------------------------
# device sampler rule (oracle/sampler_oracle.py): the generator against published known answers, the rule's
# semantics against util/data_loader.py:680-690
# ------------------------------------------------------------------------------------------------
def test_philox4x32_10_known_answers():
    """Random123 (Salmon et al., SC'11) kat_vectors for philox4x32-10."""
    from oracle.sampler_oracle import philox4x32_10
    a = lambda *v: tuple(np.array([x], dtype=np.uint64) for x in v)
    kat = [((0, 0), a(0, 0, 0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
           ((0xffffffff, 0xffffffff), a(0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff),
            (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
           ((0xa4093822, 0x299f31d0), a(0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344),
            (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for key, ctr, want in kat:
        got = tuple(int(x[0]) for x in philox4x32_10(key, ctr))
        assert got == want


def test_sampler_rule_semantics():
    from oracle.sampler_oracle import sample_epoch
    rng = np.random.default_rng(0)
    U, I, num_ng = 60, 50, 4
    pairs = np.unique(np.stack([rng.integers(0, U, 1500), rng.integers(0, I, 1500)], 1), axis=0)
    flat = sample_epoch(pairs, I, num_ng, 2019, 0, shuffle=False)
    assert np.array_equal(flat[:, :2], np.repeat(pairs, num_ng, axis=0))          # features_fill order (:684-690)
    pos = set(map(tuple, pairs.tolist()))
    assert not any((int(u), int(j)) in pos for u, _, j in flat)                    # re-drawn while (u, j) in train_mat
    assert flat[:, 2].min() >= 0 and flat[:, 2].max() < I
    sh = sample_epoch(pairs, I, num_ng, 2019, 0, shuffle=True)
    assert sorted(map(tuple, sh.tolist())) == sorted(map(tuple, flat.tolist()))
    assert not np.array_equal(sample_epoch(pairs, I, num_ng, 2019, 1, shuffle=False), flat)
    # negatives of one user are uniform over its non-positives
    big = sample_epoch(np.array([[0, 1], [0, 2]] * 1), 10, 4000, 5, 0, shuffle=False)
    c = np.bincount(big[:, 2], minlength=10)
    assert c[1] == 0 and c[2] == 0 and c[[0, 3, 4, 5, 6, 7, 8, 9]].min() > 0.8 * 8000 / 8


# ------------------------------------------------------------------------------------------------
# next row (SURVEY 8f N3, NCF-GMF): the oracle is pinned before any kernel is built on it
# ------------------------------------------------------------------------------------------------
def test_gmf_oracle_matches_reference_ncf_with_adam(golden):
    """oracle/gmf_oracle.py (closed-form forward / BCE / dense gradients / torch-default Adam over EVERY row) against
    5 steps of the unmodified reference NCF(model='GMF') + nn.BCEWithLogitsLoss + optim.Adam
    (tests/golden/make_ncf_golden.py).  float64 closed form vs the reference's fp32: 2e-6 relative on the tables."""
    from oracle import gmf_oracle
    g = golden("gmf_small.npz")
    st = gmf_oracle.GMFAdam(g["P0"], g["Q0"], g["w0"], g["b0"], lr=float(g["lr"]))
    for k in range(len(g["losses"])):
        loss = st.step(g["users"][k], g["items"][k], g["labels"][k])
        assert abs(loss - g["losses"][k]) < 2e-6 * abs(g["losses"][k]) + 1e-7, (k, loss, g["losses"][k])
        for got, want in ((st.P, g["P"][k]), (st.Q, g["Q"][k]), (st.w, g["w"][k]), (st.b, g["b"][k])):
            assert rel_err(got, want) <= 2e-6, (k, rel_err(got, want))
    # untouched rows keep moving under dense Adam: users >= U/2 get no gradient on odd steps, yet step 1 -> 2 moves them
    U = g["P0"].shape[0]
    quiet = np.setdiff1d(np.arange(U // 2, U), g["users"][1])
    assert quiet.size > 0 and np.abs(g["P"][1][quiet] - g["P"][0][quiet]).max() > 0
    fwd = gmf_oracle.gmf_forward(st.P, st.Q, st.w, st.b[0], g["users"][0], g["items"][0])
    assert np.allclose(fwd, g["fwd_last"], rtol=1e-5, atol=1e-6)


def test_bprfm_oracle_matches_reference_with_adagrad(golden):
    """oracle/bprfm_oracle.py against 4 steps of the unmodified reference BPRFM(batch_norm=False, drop_prob=[0, 0]) +
    optim.Adagrad(lr=0.05, initial_accumulator_value=1e-8) (tests/golden/make_bprfm_golden.py).  Biases within 1e-6;
    embeddings within 5e-5: with state_sum starting at 1e-8, an element whose gradient nearly cancels to |g| ~ 1e-4 turns
    the fp32 rounding of the reference's own gradient (1e-8 absolute) into 2e-5 of its value -- the float64 closed
    form and the reference differ by that much, on exactly such an element."""
    from oracle import bprfm_oracle
    g = golden("bprfm_small.npz")
    E, b = g["E0"].astype(np.float64), g["b0"].astype(np.float64)
    aE, ab = np.full_like(E, 1e-8), np.full_like(b, 1e-8)
    for k in range(len(g["losses"])):
        loss = bprfm_oracle.bprfm_adagrad_step(E, b, float(g["bias_"]), aE, ab, g["feats_i"][k], g["feats_j"][k], lr=float(g["lr"]))
        assert abs(loss - g["losses"][k]) <= 1e-6 * g["losses"][k], k
        assert rel_err(E, g["E"][k]) <= 5e-5 and rel_err(b, g["b"][k]) <= 1e-6, (k, rel_err(E, g["E"][k]), rel_err(b, g["b"][k]))
    U = int(g["user_num"])
    assert np.array_equal(g["b"][-1][:U], g["b0"][:U])          # user biases never move (their gradient is +g - g)
    pi = bprfm_oracle.pred(E, b, float(g["bias_"]), g["feats_i"][0])
    assert np.allclose(pi, g["fwd_i"], rtol=1e-4, atol=1e-5)


# ---------------------------------------------------------------- next row N4: Item2Vec / SGNS
@pytest.mark.parametrize("branch", ["w", "u"])       # negatives from the unigram^0.75 table / uniform (:86-91)
def test_sgns_oracle_matches_reference_item2vec_with_adam(golden, branch):
    """oracle/sgns_oracle.py (closed-form SGNS loss for given negatives, dense gradients with the padding row masked,
    torch-default Adam over EVERY row) against 5 steps of the reference's own Item2Vec + SGNS classes and
    torch.optim.Adam (tests/golden/make_sgns_golden.py)."""
    from oracle import sgns_oracle
    g = golden("sgns_small.npz")
    k = lambda name: g[f"{branch}_{name}"]
    st = sgns_oracle.SGNSAdam(k("iv0"), k("ov0"))
    for s in range(len(k("losses"))):
        loss = st.step(k("iword")[s], k("owords")[s], k("nwords")[s])
        assert loss == pytest.approx(float(k("losses")[s]), rel=1e-6), s
        assert rel_err(st.iv, k("iv")[s]) < 1e-6, s
        assert rel_err(st.ov, k("ov")[s]) < 1e-6, s
        assert np.abs(st.iv[0]).max() == 0 and np.abs(st.ov[0]).max() == 0        # the padding row never moves
    # rows without a gradient in a step still move under dense Adam once they have a first moment
    assert rel_err(st.iv, k("iv0")) > 1e-3


# ---------------------------------------------------------------- row N3, the script's defaults: batch norm + dropout
@pytest.mark.parametrize("branch,tol_b,tol_fwd", [("cond", 1e-6, 1e-6), ("script", 2e-4, 2e-5)])
def test_bprfm_full_oracle_matches_reference_with_batch_norm_and_dropout(golden, branch, tol_b, tol_fwd):
    """oracle/bprfm_oracle.py: BPRFMFull (bi-interaction, BatchNorm1d in training mode incl. running statistics,
    dropout with the RECORDED masks, Adagrad over every parameter) against 4 steps of the unmodified reference
    BPRFM(batch_norm=True, drop_prob=[0.5, 0.2]) (tests/golden/make_bprfm_bn_golden.py).  'cond': accumulator 0.1,
    everything within 1e-6.  'script': the script's 1e-8 -- the user bias gradient is +g - g = rounding noise, which an
    accumulator of 1e-8 turns into 5e-5 of the bias scale (same effect as in the batch_norm=False fixture)."""
    from oracle import bprfm_oracle
    g = golden("bprfm_bn_small.npz")
    k = lambda name: g[f"{branch}_{name}"]
    st = bprfm_oracle.BPRFMFull(k("E0"), k("b0"), float(k("g0")), True, lr=float(k("lr")),
                                initial_accumulator_value=float(k("acc0")))
    ones = np.ones((k("fi").shape[1], 2))
    for s in range(len(k("loss"))):
        loss = st.step(k("fi")[s], ones, k("fj")[s], ones, k("mi")[s], k("mj")[s])
        assert loss == pytest.approx(float(k("loss")[s]), rel=1e-6), s
        assert rel_err(st.E, k("E")[s]) < 1e-6, s
        assert rel_err(st.bias, k("b")[s]) < tol_b, s
        assert abs(st.bias_[0] - float(k("g")[s])) < 1e-6, s
        assert rel_err(st.gamma, k("gamma")[s]) < 1e-6 and rel_err(st.beta, k("beta")[s]) < 2e-6, s
        assert rel_err(st.running_mean, k("rm")[s]) < 1e-6 and rel_err(st.running_var, k("rv")[s]) < 1e-6, s
    pi, pj = st.forward(k("fi")[0], ones, k("fj")[0], ones)          # eval mode: running statistics, no dropout
    assert rel_err(pi, k("fwd_i")) < tol_fwd and rel_err(pj, k("fwd_j")) < tol_fwd
    assert (k("mi")[0] == 0).mean() == pytest.approx(float(k("p")), abs=0.1)        # the recorded masks are masks


def test_bprfm_full_oracle_reduces_to_the_two_feature_closed_form(golden):
    """With batch_norm off and no mask BPRFMFull is the oracle the CUDA path is checked against (bprfm_adagrad_step)."""
    from oracle import bprfm_oracle
    g = golden("bprfm_small.npz")
    E, b = g["E0"].astype(np.float64), g["b0"].astype(np.float64)
    aE, ab = np.full_like(E, 1e-8), np.full_like(b, 1e-8)
    full = bprfm_oracle.BPRFMFull(g["E0"], g["b0"], float(g["bias_"]), False, lr=float(g["lr"]))
    ones = np.ones((g["feats_i"].shape[1], 2))
    for s in range(len(g["losses"])):
        l0 = bprfm_oracle.bprfm_adagrad_step(E, b, float(g["bias_"]), aE, ab, g["feats_i"][s], g["feats_j"][s], lr=float(g["lr"]))
        l1 = full.step(g["feats_i"][s], ones, g["feats_j"][s], ones)
        assert l1 == pytest.approx(l0, rel=1e-12)
        # the general form gives the user bias a gradient of -s + s that is zero only up to rounding; with the script's
        # 1e-8 accumulator that is visible on the biases, not on the embeddings
        assert rel_err(full.E, E) < 1e-9 and rel_err(full.bias, b) < 2e-4


# ---------------------------------------------------------------- row N3: NCF with an MLP tower (MLP, NeuMF-end)
def _neumf_oracle(g, tag, name):
    from oracle import neumf_oracle
    k = lambda n: g[f"{tag}_{n}"]
    L = int(k("num_layers"))
    return k, L, neumf_oracle.NeuMFAdam(name, k("Pg_0"), k("Qg_0"), k("Pm_0"), k("Qm_0"), [k(f"W{l}_0") for l in range(L)],
                                        [k(f"b{l}_0") for l in range(L)], k("wp_0"), k("bp_0"), lr=float(k("lr")))


@pytest.mark.parametrize("tag,name", [("mlp", "MLP"), ("neumf", "NeuMF-end")])
def test_neumf_oracle_matches_reference_ncf_with_adam(golden, tag, name):
    """oracle/neumf_oracle.py (closed-form MLP tower + GMF branch, BCE, dense gradients, torch-default Adam over every
    parameter that has a gradient) against 4 steps of the reference's own NCF class with model 'MLP' and the script's
    default 'NeuMF-end', dropout 0 (tests/golden/make_neumf_golden.py)."""
    k, L, st = _neumf_oracle(golden("neumf_small.npz"), tag, name)
    for s in range(len(k("loss"))):
        loss = st.step(k("users")[s], k("items")[s], k("labels")[s])
        assert loss == pytest.approx(float(k("loss")[s]), rel=1e-6), s
        for mine, key in ((st.Pg, "Pg"), (st.Qg, "Qg"), (st.Pm, "Pm"), (st.Qm, "Qm"), (st.wp, "wp")):
            assert rel_err(mine, k(key)[s]) < 1e-6, (s, key)
        assert abs(st.bp[0] - float(k("bp")[s][0])) < 1e-8
        for l in range(L):
            assert rel_err(st.Ws[l], k(f"W{l}")[s]) < 1e-6 and rel_err(st.bs[l], k(f"b{l}")[s]) < 2e-6, (s, l)
    assert rel_err(st.forward(k("users")[0], k("items")[0]), k("fwd_last")) < 2e-6
    if tag == "mlp":                                       # no gradient ever reaches the GMF tables: torch's Adam skips them
        assert np.array_equal(st.Pg, k("Pg_0").astype(np.float64))


# ---------------------------------------------------------------- row N4: SVD++
def test_svdpp_c_oracle_is_bit_identical_to_the_reference_extension(golden):
    """oracle/mf_oracle.c: mf_oracle_svdpp_fit against the reference's own compiled SVDpp
    (util/matrix_factorization.pyx:169-288; tests/golden/make_svdpp_golden.py): all five arrays bit for bit, predictions
    to the last ulp (the reference sums the implicit rows with Python's sum, the oracle in the same order)."""
    g = golden("svdpp_small.npz")
    o = mf_oracle.svdpp_fit(g["users"], g["items"], g["ratings"], g["pu0"], g["qi0"], g["yj0"], n_epochs=int(g["E"]))
    for k in ("pu", "qi", "yj", "bu", "bi"):
        assert np.array_equal(o[k], g[k]), k
    assert o["global_mean"] == float(g["mu"])
    pred = np.array([mf_oracle.svdpp_predict(int(u), int(i), o) for u, i in zip(g["users"][:15], g["items"][:15])])
    assert np.allclose(pred, g["pred"], rtol=0, atol=1e-14)
    with pytest.raises(ValueError, match="Invalid user code"):
        mf_oracle.svdpp_predict(int(g["U"]), 0, o)
    with pytest.raises(ValueError, match="Invalid item code"):
        mf_oracle.svdpp_predict(0, int(g["I"]), o)
