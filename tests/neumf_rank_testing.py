"""Shared by the NeuMF ranking tests (emulated and on the GPU): random towers, float64 oracle scores and the ranking
criterion.  Tolerance eps(s) = 1e-4 |s| + 1e-5, the one tests/test_neumf_gpu.py uses for forward()."""
import numpy as np


def random_tower(rng, U, I, F, L, model):
    """Weights of NeuMF(U, I, F, L, 0.0, model) with enough spread that scores are distinct: dict like test_neumf_gpu.make."""
    Dm = F << (L - 1)
    rnd = lambda *sh: (rng.standard_normal(sh) * 0.3).astype(np.float32)
    init = dict(Pg=rnd(U, F), Qg=rnd(I, F), Pm=rnd(U, Dm), Qm=rnd(I, Dm), wp=rnd(F if model == "MLP" else 2 * F),
                bp=rnd(1))
    n_in = 2 * Dm
    for l in range(L):
        init[f"W{l}"] = rnd(n_in // 2, n_in) * np.float32(2.0 / np.sqrt(n_in))
        init[f"b{l}"] = rnd(n_in // 2) * np.float32(0.3)
        n_in //= 2
    return init


def oracle_scores(init, model, L, users, items):
    """float64 logits of NCF.forward for every (users[n], items[n, c]) -> [N, C]."""
    from oracle import neumf_oracle
    ora = neumf_oracle.NeuMFAdam(model, init["Pg"], init["Qg"], init["Pm"], init["Qm"], [init[f"W{l}"] for l in range(L)],
                                 [init[f"b{l}"] for l in range(L)], init["wp"], init["bp"])
    items = np.asarray(items, np.int64)
    uu = np.repeat(np.asarray(users, np.int64)[:, None], items.shape[1], 1)
    return ora.forward(uu.reshape(-1), items.reshape(-1)).reshape(items.shape)


def eps(s):
    return 1e-4 * np.abs(s) + 1e-5


def check_ranking(got_idx, got_score, ora):
    """got_idx [N, K]: candidate positions (or items) in returned order, got_score [N, K]; ora [N, C]: float64 oracle
    scores by position (-inf = excluded).  Checks, per row:
      * every returned score is within eps of the oracle's score of what it returned;
      * ranks equal the oracle's (score desc, index asc) ranks wherever the oracle's neighbouring scores are > 2 eps apart;
      * no returned entry's oracle score lies below the oracle's K-th score minus 2 eps."""
    N, K = got_idx.shape
    for n in range(N):
        o = ora[n]
        order = np.lexsort((np.arange(o.shape[0]), -o))
        so = o[order]
        g = got_idx[n].astype(np.int64)
        assert (g >= 0).all(), (n, g)
        og = o[g]
        assert np.all(np.abs(got_score[n].astype(np.float64) - og) <= eps(og)), (n, got_score[n], og)
        kth = so[K - 1]
        assert np.all(og >= kth - 2 * eps(kth)), (n, og, kth)
        for r in range(K):
            sep_prev = r == 0 or so[r - 1] - so[r] > 2 * eps(so[r])
            sep_next = r + 1 >= so.shape[0] or so[r] - so[r + 1] > 2 * eps(so[r])
            if sep_prev and sep_next:
                assert g[r] == order[r], (n, r, g, order[:K])
