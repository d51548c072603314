"""GPU tests of the BPR step the way bench.py times it: steps issued back to back with no host synchronisation, so the
bookkeeping of steps n+1 and n+2 runs on the library's side stream while the table kernels of step n are still
running (three rotating bookkeeping sets, captured bookkeeping graphs; DESIGN.md section 4 "Pipelining").

Every overlapped issue mode must give the bits of the synchronous one (the loss read after every step), and the
synchronous run must match the float64 closed-form oracle.  The modes:

  sync      opt.step(t) and opt.loss_sum() after every step (test_bpr_gpu.run_steps)
  ready     batches uploaded and synchronised first, then opt.step(t, ready=True, loss_out=slot k): bench.py's loop
  produced  ready=False; every batch is copied into ONE reused device buffer on the caller's stream right before its
            step (the bookkeeping must wait for the copy, and the next copy for the bookkeeping)
  host      a pinned host tensor per step (daisy_bpr_step_host: the H2D copy heads the bookkeeping chain)
  epoch     one BPRSGD.epoch call over all batches (daisy_bpr_epoch)

Environment switches are read when a handle is created, so every mode builds a fresh model.
"""
import functools

import numpy as np
import pytest

from conftest import rel_err
from test_bpr_gpu import make_model, oracle_run, rand_problem, run_steps, tables, torch_reference_step

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

# switches this file sets; the cached default runs are made without them
SWITCHES = ("DAISY_PIPELINE", "DAISY_MERGED_SORT")
# ~50 ms of the caller's stream at B200 clocks: long enough that unordered bookkeeping would read a stale buffer
SLEEP_CYCLES = 100_000_000


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (there is no CPU fallback to test)"
    return torch.device("cuda:0")


def run(mode, P0, Q0, batches, lr, wd, dev, max_batch=None):
    """Steps over `batches` in one issue mode; returns (P, Q, decay scale before materialising, per-step losses).
    The epoch mode returns one loss, the sum the device accumulated over the call."""
    from recommend_lib_b200.bpr import BPRSGD
    max_batch = max_batch or max(1, max(len(b) for b in batches))
    m = make_model(P0, Q0, dev, max_batch=max_batch)
    mk = lambda b: torch.from_numpy(np.ascontiguousarray(b, dtype=np.int32))
    if mode == "sync":
        losses = run_steps(m, batches, lr, wd)
    else:
        opt = BPRSGD(m, lr=lr, weight_decay=wd)
        loss_dev = torch.zeros(len(batches), dtype=torch.float64, device=dev)
        if mode == "ready":
            ts = [mk(b).to(dev) for b in batches]
            torch.cuda.synchronize()
            for k, t in enumerate(ts):
                opt.step(t, loss_out=loss_dev[k:k + 1], ready=True)
        elif mode == "produced":
            ts = [mk(b).to(dev) for b in batches]
            buf = torch.zeros((max_batch, 3), dtype=torch.int32, device=dev)
            torch.cuda.synchronize()
            for k, t in enumerate(ts):
                view = buf[:t.shape[0]]
                view.copy_(t)
                opt.step(view, loss_out=loss_dev[k:k + 1])
        elif mode == "host":
            ts = [mk(b).pin_memory() if len(b) else mk(b) for b in batches]
            for k, t in enumerate(ts):
                opt.step(t, loss_out=loss_dev[k:k + 1])
        elif mode == "epoch":
            assert all(len(b) == len(batches[0]) for b in batches)
            opt.epoch(mk(np.concatenate(batches)).to(dev), len(batches[0]), loss_out=loss_dev[:1])
            loss_dev = loss_dev[:1]
        else:
            raise ValueError(mode)
        torch.cuda.synchronize()
        m.check()
        losses = loss_dev.tolist()
    c = m.decay_scale
    P, Q = tables(m)
    return P, Q, c, losses


def assert_bit_identical(got, want, what):
    (P, Q, c, losses), (Pw, Qw, cw, lw) = got, want
    assert np.array_equal(P, Pw) and np.array_equal(Q, Qw), (what, rel_err(P, Pw), rel_err(Q, Qw))
    assert c == cw, (what, c, cw)
    assert losses == lw, (what, losses, lw)


def assert_oracle(got, ref, what):
    (P, Q, _, losses), (Pr, Qr, lr_) = got, ref
    assert rel_err(P, Pr) <= 1e-5 and rel_err(Q, Qr) <= 1e-5, (what, rel_err(P, Pr), rel_err(Q, Qr))
    assert np.allclose(losses, lr_, rtol=1e-5, atol=1e-9), what


# ------------------------------------------------------------------------------------------------
# every bookkeeping path, every issue mode
# ------------------------------------------------------------------------------------------------
# name: (U, I, D, B); K = 7 batches reuse each of the three bookkeeping sets twice
SHAPES = {
    "small": (5000, 3000, 32, 4096),            # k_small_book (B <= 8 192)
    "mid": (5000, 3000, 64, 40000),             # k_mid_book (B <= 65 536)
    "graphed": (5000, 3000, 128, 100000),       # general chain replayed from a captured graph (B <= 262 144)
    "direct": (5000, 3000, 100, 300000),        # general chain launched kernel by kernel
}
K = 7
WD = 0.001


def lr_for(B):
    """A learning rate that keeps the hot rows of rand_problem (a third of the batch on one item, an eighth on one
    user) from running away at large B: the float64 run then stays well conditioned, and the tables still move by
    tens of percent in 7 steps."""
    return min(0.01, 40.0 / B)


@functools.lru_cache(maxsize=None)
def baseline(name):
    """(problem, sync run with default switches, float64 oracle) of a SHAPES entry, computed once per session."""
    U, I, D, B = SHAPES[name]
    P0, Q0, batches = rand_problem(U, I, D, B, K, seed=B)
    with pytest.MonkeyPatch.context() as mp:
        for k in SWITCHES:
            mp.delenv(k, raising=False)
        sync = run("sync", P0, Q0, batches, lr_for(B), WD, torch.device("cuda:0"))
    return (P0, Q0, batches), sync, oracle_run(P0, Q0, batches, lr_for(B), WD)


@pytest.mark.parametrize("name", list(SHAPES))
def test_back_to_back_issue_equals_synchronous_issue(dev, name):
    """ready / produced / host / epoch give the bits of sync; sync matches the oracle.  The epoch's one loss is the
    step losses added in step order, which is what the device does into its one accumulator."""
    (P0, Q0, batches), sync, ref = baseline(name)
    lr = lr_for(len(batches[0]))
    assert_oracle(sync, ref, name)
    for mode in ("ready", "produced", "host"):
        assert_bit_identical(run(mode, P0, Q0, batches, lr, WD, dev), sync, (name, mode))
    P, Q, c, sync_losses = sync
    assert_bit_identical(run("epoch", P0, Q0, batches, lr, WD, dev), (P, Q, c, [sum(sync_losses)]), (name, "epoch"))


def test_config4_back_to_back_equals_synchronous(dev):
    """The benchmark's configuration (10 M x 2 M, D 128, B 1 M, lr 0.01, wd 0.001, Zipf(1.0) positives, N(0, 0.01^2)
    tables): 7 steps issued as bench.py issues them give the bits of the same steps read one by one; those match the
    float64 torch restatement of the step."""
    from recommend_lib_b200.bpr import BPR, BPRSGD
    from recommend_lib_b200.sampler import synthetic_triples
    U, I, D, B, lr, wd = 10_000_000, 2_000_000, 128, 1_000_000, 0.01, 0.001
    torch.manual_seed(2019)
    P0 = torch.empty((U, D), device=dev).normal_(0, 0.01)
    Q0 = torch.empty((I, D), device=dev).normal_(0, 0.01)
    tri = [torch.from_numpy(synthetic_triples(B, U, I, seed=11 + k, zipf=1.0)).to(dev) for k in range(K)]

    def model():
        m = BPR(1, 1, D, max_batch=B)          # tiny CPU init, the real tables are device copies of P0 / Q0
        m.user_num, m.item_num = U, I
        m.embed_user.weight = torch.nn.Parameter(P0.clone(), requires_grad=False)
        m.embed_item.weight = torch.nn.Parameter(Q0.clone(), requires_grad=False)
        return m, BPRSGD(m, lr=lr, weight_decay=wd)

    m, opt = model()
    loss_dev = torch.zeros(K, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    for k in range(K):
        opt.step(tri[k], loss_out=loss_dev[k:k + 1], ready=True)
    torch.cuda.synchronize()
    m.check()
    ready_losses, ready_c = loss_dev.tolist(), m.decay_scale
    m.materialize()
    ready_P, ready_Q = m._tables()

    m, opt = model()
    Pr, Qr, sync_losses = P0, Q0, []
    for k in range(K):
        opt.step(tri[k])
        sync_losses.append(opt.loss_sum())
        m.check()
        Pr, Qr, loss_r = torch_reference_step(Pr, Qr, tri[k], lr, wd)
        assert abs(sync_losses[k] - loss_r) / loss_r < 1e-5, (k, sync_losses[k], loss_r)
    assert m.decay_scale == ready_c and sync_losses == ready_losses
    m.materialize()
    P1, Q1 = m._tables()
    assert float((P1 - Pr).abs().max() / Pr.abs().max()) <= 1e-5
    assert float((Q1 - Qr).abs().max() / Qr.abs().max()) <= 1e-5
    del Pr, Qr
    assert torch.equal(P1, ready_P) and torch.equal(Q1, ready_Q)


def test_mixed_sizes_share_the_sets_while_earlier_steps_run(dev):
    """One handle (max_batch 300 000), every path in one sequence issued without synchronising: the small, mid,
    graphed and direct bookkeeping take turns on the three sets, an empty batch only decays, a one-triple batch, and
    more (set, batch size) graphs are captured than the handle keeps (9), so graphs are captured and older ones evicted
    while earlier steps are still queued.  Bit-identical to sync, which matches the oracle."""
    sizes = [300000, 4096, 100000, 0, 40000, 1, 100000, 300000, 8192, 70000, 90000, 110000, 130000, 150000, 170000,
             190000, 210000, 230000, 250000, 100000, 70000, 0, 4096]
    # the library's bookkeeping sets rotate once per non-empty step; batches of 65 537 .. 262 144 triples are graphed
    graphed, s = set(), 0
    for B in sizes:
        if B:
            if 65536 < B <= 262144:
                graphed.add((s, B))
            s = (s + 1) % 3
    assert len(graphed) > 9
    U, I, D = 3000, 2000, 32
    P0, Q0, _ = rand_problem(U, I, D, 1, 1, seed=40)
    batches = [rand_problem(U, I, D, B, 1, seed=41 + n)[2][0] for n, B in enumerate(sizes)]
    lr = lr_for(300000)
    sync = run("sync", P0, Q0, batches, lr, WD, dev, max_batch=300000)
    assert_oracle(sync, oracle_run(P0, Q0, batches, lr, WD), "sync")
    for mode in ("ready", "produced", "host"):
        assert_bit_identical(run(mode, P0, Q0, batches, lr, WD, dev, max_batch=300000), sync, mode)


# ------------------------------------------------------------------------------------------------
# runtime switches
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(SHAPES))
def test_pipeline_off_is_bit_identical(dev, monkeypatch, name):
    """DAISY_PIPELINE=0: bookkeeping and table kernels all on the caller's stream, same kernels, same bits."""
    (P0, Q0, batches), sync, ref = baseline(name)
    monkeypatch.setenv("DAISY_PIPELINE", "0")
    got = run("ready", P0, Q0, batches, lr_for(len(batches[0])), WD, dev)
    assert_oracle(got, ref, name)
    assert_bit_identical(got, sync, name)


def hot_edges(b, U, I):
    """The highest ids as hot rows: the merged sort's user keys are I + 1 + u, the largest key is I + U."""
    b = b.copy()
    n = len(b)
    b[: n // 5, 0] = U - 1
    b[n // 4: n // 4 + n // 6, 1] = I - 1
    b[-n // 7:, 2] = I - 1
    np.random.default_rng(n).shuffle(b)
    return b


@pytest.mark.parametrize("U,I,D,B", [(300, 200, 64, 100000),           # auto: two sorts
                                     (70000, 70000, 32, 300000),       # auto: merged sort
                                     (70000, 61072, 32, 100000)])      # U + I = 2^17: key width 18 bits
def test_merged_sort_forced_either_way_is_bit_identical(dev, monkeypatch, U, I, D, B):
    """DAISY_MERGED_SORT=0 / 1: one stable sort of all 3B refs or two sorts give the same products (DESIGN.md section
    4), at shapes where the automatic choice goes either way and where I + U is a power of two."""
    P0, Q0, batches = rand_problem(U, I, D, B, 3, seed=U + I)
    batches = [hot_edges(b, U, I) for b in batches]
    lr = lr_for(B) / 10                                      # the hot edges come on top of rand_problem's hot rows
    outs = {}
    for forced in ("auto", "0", "1"):
        if forced == "auto":
            monkeypatch.delenv("DAISY_MERGED_SORT", raising=False)
        else:
            monkeypatch.setenv("DAISY_MERGED_SORT", forced)
        outs[forced] = run("ready", P0, Q0, batches, lr, WD, dev)
    assert_oracle(outs["auto"], oracle_run(P0, Q0, batches, lr, WD), "auto")
    assert_bit_identical(outs["0"], outs["auto"], "two sorts")
    assert_bit_identical(outs["1"], outs["auto"], "merged sort")


# ------------------------------------------------------------------------------------------------
# the lazy-decay fold between queued steps
# ------------------------------------------------------------------------------------------------
def test_decay_fold_inside_a_pipelined_run(dev):
    """lr 0.05, wd 5: every step shrinks c by 0.75, so c drops below 1e-4 after 33 steps and sgd_step folds it into
    the tables (daisy_materialize) between two queued steps.  Bit-identical to sync, which matches the oracle."""
    lr, wd = 0.05, 5.0
    P0, Q0, batches = rand_problem(300, 200, 32, 2000, 40, seed=50)
    sync = run("sync", P0, Q0, batches, lr, wd, dev)
    assert 1e-4 <= sync[2] < 1.0 and 0.75 ** 40 < 1e-4      # c went below 1e-4 once and was folded
    assert_oracle(sync, oracle_run(P0, Q0, batches, lr, wd), "sync")
    for mode in ("ready", "produced"):
        assert_bit_identical(run(mode, P0, Q0, batches, lr, wd, dev), sync, mode)


# ------------------------------------------------------------------------------------------------
# the inputs-ready flag stays on the handle: calls that do not take it must still wait for their producer
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [300000, 100000])
def test_epoch_after_ready_steps_waits_for_its_producer(dev, B):
    """step(ready=True) twice leaves the handle's inputs-ready flag set.  An epoch over device triples that the
    caller's stream writes after a delay must still see them (daisy_bpr_epoch orders its bookkeeping behind the
    caller's stream): the same bits as with a synchronise before the epoch.  B = 100 000 also covers the copy into
    the set's landing zone that a graphed bookkeeping chain starts with."""
    from recommend_lib_b200.bpr import BPRSGD
    P0, Q0, batches = rand_problem(3000, 2000, 64, B, 4, seed=60 + B)
    outs = []
    for synchronise in (True, False):
        m = make_model(P0, Q0, dev, max_batch=B)
        opt = BPRSGD(m, lr=lr_for(B), weight_decay=WD)
        first = [torch.from_numpy(b).to(dev) for b in batches[:2]]
        buf = torch.cat(first)                              # valid triples, overwritten below
        nxt = torch.from_numpy(np.concatenate(batches[2:])).to(dev)
        torch.cuda.synchronize()
        for t in first:
            opt.step(t, ready=True)
        torch.cuda._sleep(SLEEP_CYCLES)
        buf.copy_(nxt)
        if synchronise:
            torch.cuda.synchronize()
        opt.epoch(buf, B)
        loss = opt.loss_sum()
        m.check()
        c = m.decay_scale
        outs.append((*tables(m), c, [loss]))
    Pr, Qr, lr_ = oracle_run(P0, Q0, batches, lr_for(B), WD)
    assert_oracle(outs[0], (Pr, Qr, [sum(lr_)]), "synchronised")
    assert_bit_identical(outs[1], outs[0], "unsynchronised")


@pytest.mark.parametrize("B", [300000, 100000])
def test_adam_step_after_ready_step_waits_for_its_producer(dev, B):
    """BPRAdam.step on a model whose handle carries the inputs-ready flag of an earlier BPRSGD.step(ready=True): its
    bookkeeping must wait for the caller's stream to write the batch.  The oracle checks the loss only: a first Adam
    step moves every element by about +-lr whatever |g| is, so an element whose gradient sums to nearly zero may
    round to either sign, and the table comparison is the bit-identity of the two runs."""
    from oracle import bpr_oracle
    from recommend_lib_b200.bpr import BPRAdam, BPRSGD
    P0, Q0, batches = rand_problem(3000, 2000, 64, B, 3, seed=70 + B)
    outs = []
    for synchronise in (True, False):
        m = make_model(P0, Q0, dev, max_batch=B)
        t0, buf = (torch.from_numpy(b).to(dev) for b in batches[:2])   # buf: valid triples, overwritten below
        nxt = torch.from_numpy(batches[2]).to(dev)
        torch.cuda.synchronize()
        BPRSGD(m, lr=lr_for(B), weight_decay=WD).step(t0, ready=True)
        adam = BPRAdam(m, lr=0.01)
        torch.cuda._sleep(SLEEP_CYCLES)
        buf.copy_(nxt)
        if synchronise:
            torch.cuda.synchronize()
        adam.step(buf)
        loss = adam.loss_sum()
        m.check()
        outs.append((*tables(m), m.decay_scale, [loss]))
    P1, Q1, _ = oracle_run(P0, Q0, batches[:1], lr_for(B), WD)
    moments = [np.zeros_like(a) for a in (P1, P1, Q1, Q1)]
    *_, loss_r = bpr_oracle.bpr_adam_step_closed_form(P1, Q1, *moments, batches[2], 1, 0.01)
    assert abs(outs[0][3][0] - loss_r) / loss_r < 1e-5
    assert_bit_identical(outs[1], outs[0], "unsynchronised")


def test_gmf_epoch_with_inputs_ready_waits_for_its_producer(dev):
    """daisy_gmf_epoch on a handle with the inputs-ready flag set, over device samples the caller's stream writes
    after a delay: the same bits as with a synchronise before the epoch, and the oracle's Adam run."""
    from oracle import gmf_oracle
    from recommend_lib_b200.ncf import GMFAdam, NCF
    rng = np.random.default_rng(80)
    U, I, D, B, steps = 300, 200, 32, 4096, 3
    P0 = (rng.standard_normal((U, D)) * 0.3).astype(np.float32)
    Q0 = (rng.standard_normal((I, D)) * 0.3).astype(np.float32)
    w0, b0 = (rng.standard_normal(D) * 0.5).astype(np.float32), np.array([0.1], np.float32)
    mk = lambda n: np.stack([rng.integers(0, U, n), rng.integers(0, I, n), rng.integers(0, 2, n)], 1).astype(np.int32)
    old, new = mk(B * steps), mk(B * steps)
    new[: B // 3, 0] = 2                                     # a hot user and a hot item
    new[B // 2: B // 2 + B // 8, 1] = 1
    outs = []
    for synchronise in (True, False):
        m = NCF(U, I, D, 3, 0.0, "GMF", max_batch=B)
        with torch.no_grad():
            m.embed_user_GMF.weight.copy_(torch.from_numpy(P0))
            m.embed_item_GMF.weight.copy_(torch.from_numpy(Q0))
            m.predict_layer.weight.copy_(torch.from_numpy(w0.reshape(1, -1)))
            m.predict_layer.bias.copy_(torch.from_numpy(b0))
        m = m.to(dev)
        m.handle(B).set_inputs_ready(True)
        opt = GMFAdam(m, lr=0.002)
        buf = torch.from_numpy(old).to(dev)                 # valid samples, overwritten below
        nxt = torch.from_numpy(new).to(dev)
        torch.cuda.synchronize()
        torch.cuda._sleep(SLEEP_CYCLES)
        buf.copy_(nxt)
        if synchronise:
            torch.cuda.synchronize()
        opt.epoch(buf, B)
        loss = opt.last_loss()
        m.check()
        outs.append(([t.detach().cpu().numpy().reshape(t.shape[0], -1) for t in m._tensors()], loss))
    (got, loss), (got2, loss2) = outs
    assert all(np.array_equal(a, b) for a, b in zip(got, got2)) and loss == loss2
    st = gmf_oracle.GMFAdam(P0, Q0, w0, b0, lr=0.002)
    loss_r = 0.0
    for s in range(0, len(new), B):
        loss_r += st.step(new[s:s + B, 0], new[s:s + B, 1], new[s:s + B, 2].astype(np.float32))
    assert rel_err(got[0], st.P) <= 1e-5 and rel_err(got[1], st.Q) <= 1e-5
    assert rel_err(got[2].reshape(-1), st.w) <= 1e-5
    assert abs(loss - loss_r) <= 1e-5 * abs(loss_r)
