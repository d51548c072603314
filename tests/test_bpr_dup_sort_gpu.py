"""GPU tests of the general bookkeeping path's merged sort, which sorts only the refs of repeated rows (DESIGN.md
section 4): k_refs marks every row in two bitmaps, the compaction settles the refs of rows referenced once as DIRECT,
and csrc/ref_sort.cuh sorts the rest with a count that stays on the device; k_seg_all reads both counts from there.

The refs of a row keep their order, so every row is summed in the same order as with two full sorts: the default path
must give the bits of DAISY_MERGED_SORT=0 -- tables, decay scale and losses -- for SGD, sparse Adam and BPR-FM Adagrad,
with the graph-replayed chain (B <= 262 144) and the directly launched one.  Every shape here takes the merged sort by
default (the key space of U + I costs no extra radix pass).
"""
import numpy as np
import pytest

from test_bpr_gpu import rand_problem
from test_bpr_pipeline_gpu import assert_bit_identical, hot_edges, lr_for, run

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

WD = 0.001


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (there is no CPU fallback to test)"
    return torch.device("cuda:0")


def both(monkeypatch, fn):
    """fn() with the default bookkeeping, then with two full sorts (DAISY_MERGED_SORT=0)."""
    monkeypatch.delenv("DAISY_MERGED_SORT", raising=False)
    a = fn()
    monkeypatch.setenv("DAISY_MERGED_SORT", "0")
    b = fn()
    monkeypatch.delenv("DAISY_MERGED_SORT", raising=False)
    return a, b


def unique_batch(B, U, I, seed):
    """Every user, positive and negative row of the batch is referenced once."""
    rng = np.random.default_rng(seed)
    items = rng.permutation(I)[: 2 * B]
    return np.stack([rng.permutation(U)[:B], items[:B], items[B:]], 1).astype(np.int32)


@pytest.mark.parametrize("B", [100000, 300000])
def test_sgd_matches_two_sorts(dev, monkeypatch, B):
    U, I, D = 70000, 70000, 32
    P0, Q0, batches = rand_problem(U, I, D, B, 4, seed=B)
    batches = [hot_edges(b, U, I) for b in batches]          # rows longer than DAISY_HEAVY_LEN, the largest keys
    lr = lr_for(B) / 10
    a, b = both(monkeypatch, lambda: run("ready", P0, Q0, batches, lr, WD, dev))
    assert_bit_identical(a, b, "merged sort of repeated rows")


@pytest.mark.parametrize("B", [100000, 300000])
def test_every_ref_unique_or_every_ref_repeated(dev, monkeypatch, B):
    """A batch whose refs are all unique (nothing to sort), one with a row seen once as a negative and once as a run
    head, one where every triple is the same (u, i, j), and one where every triple is (u, i, i)."""
    U, I, D = 3 * B, 3 * B, 16
    rng = np.random.default_rng(B + 1)
    P0 = (rng.standard_normal((U, D)) * 0.3).astype(np.float32)
    Q0 = (rng.standard_normal((I, D)) * 0.3).astype(np.float32)
    uniq = unique_batch(B, U, I, B)
    neg_and_head = uniq.copy()
    neg_and_head[7, 2] = neg_and_head[B // 2, 1]            # row once a negative, once a positive (a run head)
    same = np.tile(np.array([[5, 9, 11]], np.int32), (B, 1))
    same_ij = np.tile(np.array([[U - 1, I - 1, I - 1]], np.int32), (B, 1))
    batches = [uniq, neg_and_head, same, same_ij, uniq]
    a, b = both(monkeypatch, lambda: run("ready", P0, Q0, batches, 1e-4, WD, dev))
    assert_bit_identical(a, b, "unique / repeated refs")


def test_back_to_back_steps_of_different_sizes(dev, monkeypatch):
    U, I, D = 70000, 70000, 32
    P0, Q0, pool = rand_problem(U, I, D, 300000, 2, seed=3)
    sizes = [300000, 100000, 70000, 250000, 300000, 131072, 100000]
    rng = np.random.default_rng(4)
    batches = [pool[k % 2][rng.permutation(300000)[:n]] for k, n in enumerate(sizes)]
    a, b = both(monkeypatch, lambda: run("ready", P0, Q0, batches, 1e-4, WD, dev, max_batch=300000))
    assert_bit_identical(a, b, "mixed sizes")


def test_bad_id_raises_the_flag(dev, monkeypatch):
    from recommend_lib_b200._lib import DaisyError
    from recommend_lib_b200.bpr import BPR, BPRSGD
    U, I, D, B = 70000, 70000, 32, 100000
    _, _, batches = rand_problem(U, I, D, B, 1, seed=5)
    bad = batches[0].copy()
    bad[B // 3, 2] = I                                      # a negative item past the table
    for forced in (None, "0"):
        if forced is None:
            monkeypatch.delenv("DAISY_MERGED_SORT", raising=False)
        else:
            monkeypatch.setenv("DAISY_MERGED_SORT", forced)
        m = BPR(U, I, D, max_batch=B).to(dev)
        opt = BPRSGD(m, lr=0.01)
        opt.step(torch.from_numpy(bad).to(dev))
        with pytest.raises((IndexError, DaisyError)):
            m.check()


def test_adam_matches_two_sorts(dev, monkeypatch):
    from recommend_lib_b200.bpr import BPR, BPRAdam
    U, I, D, B = 70000, 70000, 32, 100000
    P0, Q0, batches = rand_problem(U, I, D, B, 3, seed=6)

    def go():
        m = BPR(U, I, D, max_batch=B)
        with torch.no_grad():
            m.embed_user.weight.copy_(torch.from_numpy(P0))
            m.embed_item.weight.copy_(torch.from_numpy(Q0))
        m = m.to(dev)
        opt = BPRAdam(m, lr=0.001)
        losses = []
        for bt in batches:
            opt.step(torch.from_numpy(bt).to(dev))
            losses.append(opt.loss_sum())
        m.check()
        m.materialize()
        return ([m.embed_user.weight.detach().cpu().numpy(), m.embed_item.weight.detach().cpu().numpy()]
                + [s.cpu().numpy() for s in opt.state], losses)

    (ta, la), (tb, lb) = both(monkeypatch, go)
    assert la == lb
    for x, y in zip(ta, tb):
        assert np.array_equal(x, y)


def test_bprfm_adagrad_matches_two_sorts(dev, monkeypatch):
    from recommend_lib_b200.bprfm import BPRFM, FMAdagrad
    U, I, F, B = 70000, 70000, 16, 100000
    rng = np.random.default_rng(7)
    E0 = (rng.standard_normal((U + I, F)) * 0.3).astype(np.float32)
    b0 = (rng.standard_normal(U + I) * 0.05).astype(np.float32)
    steps = []
    for _ in range(3):
        u, i, j = rng.integers(0, U, B), rng.integers(0, I, B), rng.integers(0, I, B)
        u[: B // 4] = 2
        i[B // 2: B // 2 + B // 6] = 1
        j[-B // 8:] = 1
        steps.append((np.stack([u, U + i], 1), np.stack([u, U + j], 1)))

    def go():
        m = BPRFM(U + I, F, False, [0.0, 0.0], user_num=U, max_batch=B)
        with torch.no_grad():
            m.embeddings.weight.copy_(torch.from_numpy(E0))
            m.biases.weight.copy_(torch.from_numpy(b0.reshape(-1, 1)))
            m.bias_.fill_(0.25)
        m = m.to(dev)
        opt = FMAdagrad(m, lr=0.05, initial_accumulator_value=1e-2)
        losses = []
        for fi, fj in steps:
            opt.step(torch.from_numpy(fi), None, torch.from_numpy(fj), None)
            losses.append(opt.loss_sum())
        m.check()
        m.sync()
        return m.embeddings.weight.detach().cpu().numpy(), m.biases.weight.detach().cpu().numpy(), losses

    a, b = both(monkeypatch, go)
    assert a[2] == b[2]
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_config4_shape(dev, monkeypatch):
    """bench.py's configuration: 10 M users x 2 M items, D 128, 1 M triples per step, steps issued back to back."""
    from recommend_lib_b200.bpr import BPR, BPRSGD
    U, I, D, B, K = 10_000_000, 2_000_000, 128, 1_000_000, 3
    rng = np.random.default_rng(8)
    batches = []
    for _ in range(K):
        b = np.stack([rng.integers(0, U, B), rng.integers(0, I, B), rng.integers(0, I, B)], 1).astype(np.int32)
        b[: B // 50, 1] = 3                                 # a hot positive item and a hot user
        b[B // 2: B // 2 + B // 100, 0] = U - 1
        rng.shuffle(b)
        batches.append(torch.from_numpy(b))

    def go():
        g = torch.Generator(device=dev).manual_seed(9)
        m = BPR(U, I, D, max_batch=B).to(dev)
        with torch.no_grad():
            m.embed_user.weight.normal_(0.0, 0.1, generator=g)
            m.embed_item.weight.normal_(0.0, 0.1, generator=g)
        opt = BPRSGD(m, lr=0.01, weight_decay=WD)
        loss = torch.zeros(K, dtype=torch.float64, device=dev)
        ts = [t.to(dev) for t in batches]
        torch.cuda.synchronize()
        for k, t in enumerate(ts):
            opt.step(t, loss_out=loss[k:k + 1], ready=True)
        torch.cuda.synchronize()
        m.check()
        c = m.decay_scale
        P, Q = m._tables()
        out = (P.detach().clone(), Q.detach().clone(), c, loss.tolist())
        del m, opt, ts
        torch.cuda.empty_cache()
        return out

    a, b = both(monkeypatch, go)
    assert a[2] == b[2] and a[3] == b[3]
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
