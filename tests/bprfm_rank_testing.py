"""Shared by the BPR-FM ranking tests (emulated and on the GPU): random model states, float64 oracle scores with their
per-pair tolerance, and the ranking criterion.

Tolerance of a score s(u, i) (fp32 fold + fp32 dot product + the per-user term, against oracle/bprfm_oracle.py in float64):
    eps = 1e-5 (sum_f |a_f e_u,f e_i,f| + sum_f |beta_f - a_f mu_f| + |b_i| + |b_u| + |bias_|) + 1e-6,
a_f = gamma_f / sqrt(running_var_f + bn_eps); without batch norm a = 1 and beta = mu = 0."""
import numpy as np

BN_EPS = 1e-5


def random_state(rng, U, I, F, bn):
    """Weights of a BPR-FM model over U users and I items with F factors; with ``bn`` a batch-norm state away from its
    initial values (gamma, beta, running mean and variance), and non-zero user, item and global biases."""
    st = dict(E=(rng.standard_normal((U + I, F)) * 0.3).astype(np.float32),
              b=(rng.standard_normal(U + I) * 0.2).astype(np.float32), bias_=np.float32(0.37), bn=bn)
    if bn:
        st.update(gamma=(1.0 + 0.5 * rng.standard_normal(F)).astype(np.float32),
                  beta=(0.2 * rng.standard_normal(F)).astype(np.float32),
                  rm=(0.05 * rng.standard_normal(F)).astype(np.float32),
                  rv=rng.uniform(0.02, 0.3, F).astype(np.float32))
    return st


def _fold64(st):
    """(a [F], sum_f |beta_f - a_f mu_f|) in float64."""
    F = st["E"].shape[1]
    if not st["bn"]:
        return np.ones(F), 0.0
    a = st["gamma"].astype(np.float64) / np.sqrt(st["rv"].astype(np.float64) + BN_EPS)
    return a, float(np.abs(st["beta"].astype(np.float64) - a * st["rm"].astype(np.float64)).sum())


def oracle_scores(st, U, users, items, chunk=1 << 16):
    """float64 scores of the evaluation-mode forward for every (users[n], items[n, c]) -> (score [N, C], eps [N, C]).
    The batch-norm model is oracle/bprfm_oracle.py: BPRFMFull.forward with the state's running statistics; the plain
    model is bprfm_oracle.pred."""
    from oracle import bprfm_oracle
    items = np.asarray(items, np.int64)
    users = np.asarray(users, np.int64)
    uu = np.repeat(users[:, None], items.shape[1], 1).reshape(-1)
    feats = np.stack([uu, U + items.reshape(-1)], 1)
    E, b = st["E"].astype(np.float64), st["b"].astype(np.float64)
    if st["bn"]:
        ora = bprfm_oracle.BPRFMFull(E, b, float(st["bias_"]), True)
        ora.gamma[:], ora.beta[:] = st["gamma"], st["beta"]
        ora.running_mean[:], ora.running_var[:] = st["rm"], st["rv"]
        ones = np.ones((min(chunk, len(feats)), 2))
        fwd = lambda f: ora.forward(f, ones[:len(f)], f, ones[:len(f)])[0]
    else:
        fwd = lambda f: bprfm_oracle.pred(E, b, float(st["bias_"]), f)
    score = np.concatenate([fwd(f) for f in np.split(feats, np.arange(chunk, len(feats), chunk))])
    a, cterm = _fold64(st)
    dots = np.abs(E[users] * a) @ np.abs(E[U:]).T                        # [N, I]: sum_f |a_f e_u,f e_i,f|
    dots = np.take_along_axis(dots, items, 1)
    mag = dots + cterm + np.abs(b[U + items]) + np.abs(b[users])[:, None] + abs(float(st["bias_"]))
    return score.reshape(items.shape), 1e-5 * mag + 1e-6


def check_ranking(got_idx, got_score, ora, eps):
    """got_idx [N, K]: candidate positions (or items) in returned order, got_score [N, K]; ora [N, C]: float64 oracle
    scores by position (-inf = excluded), eps [N, C] their tolerances.  Per row:
      * every returned score is within eps of the oracle's score of what it returned;
      * ranks equal the oracle's (score desc, index asc) ranks wherever the oracle's neighbouring scores are further
        apart than the two tolerances;
      * no returned entry's oracle score lies below the oracle's K-th score minus twice its tolerance."""
    N, K = got_idx.shape
    for n in range(N):
        o, e = ora[n], eps[n]
        order = np.lexsort((np.arange(o.shape[0]), -o))
        so, se = o[order], e[order]
        g = got_idx[n].astype(np.int64)
        assert (g >= 0).all() and len(np.unique(g)) == K, (n, g)
        og = o[g]
        assert np.isfinite(og).all(), (n, g)
        assert np.all(np.abs(got_score[n].astype(np.float64) - og) <= e[g]), (n, got_score[n], og, e[g])
        assert np.all(og >= so[K - 1] - 2 * se[K - 1]), (n, og, so[K - 1])
        for r in range(K):
            sep_prev = r == 0 or so[r - 1] - so[r] > se[r - 1] + se[r]
            sep_next = r + 1 >= so.shape[0] or so[r] - so[r + 1] > se[r] + se[r + 1]
            if sep_prev and sep_next:
                assert g[r] == order[r], (n, r, g, order[:K])
