"""CPU execution of the batch-norm BPR-FM fold (csrc/fmbn.cu: daisy_fmbn_rank_tables) under the host emulation of
tests/emu: the folded tables and C0 against numpy (F not a multiple of 4, padding columns exactly 0), then those tables
ranked by the unchanged ranking units (csrc/bpr_eval.cu: daisy_topk_candidates; csrc/topk_full.cu: daisy_topk_full on
its exact path and on its CUDA-core filter) against the float64 oracle.  The same checks at real sizes run on the B200
in tests/test_bprfm_rank_gpu.py."""
import ctypes
import os
import sys

import numpy as np
import pytest

from bprfm_rank_testing import BN_EPS, check_ranking, oracle_scores, random_state
from conftest import ROOT

sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
import build_emu  # noqa: E402

from recommend_lib_b200 import _lib  # noqa: E402  (only the ctypes structure definitions are used here)

c_vp, c_i64, c_i32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int


def _p(a):
    return c_vp(a.ctypes.data) if a is not None else None


def _lib_emu(unit, U, I, W):
    L = ctypes.CDLL(build_emu.build(unit))
    L.emu_handle_dims.restype = c_vp
    L.emu_handle_dims.argtypes = [ctypes.c_longlong, ctypes.c_longlong, c_i32]
    L.emu_err_flag.argtypes = [c_vp]
    L.emu_last_error.restype = ctypes.c_char_p
    for name in ("daisy_fmbn_rank_tables", "daisy_topk_candidates", "daisy_topk_full", "daisy_topk_full_path"):
        if hasattr(L, name):
            getattr(L, name).argtypes = _lib.SIGNATURES[name]
    return L, c_vp(L.emu_handle_dims(U, I, W))


def fold(st, U, W):
    """(P, Q, c0, library, handle) of daisy_fmbn_rank_tables over the emulated unit."""
    L, h = _lib_emu("fmbn", U, st["E"].shape[0] - U, W)
    F = st["E"].shape[1]
    T = {k: np.ascontiguousarray(st[k]) for k in ("E", "b", "gamma", "beta", "rm", "rv")}
    prm = _lib.FMBNParams(_p(T["E"]), _p(T["b"]), None, None, _p(T["gamma"]), _p(T["beta"]), None, None, _p(T["rm"]),
                          _p(T["rv"]), 0.0, 1e-10, BN_EPS, 0.1, U, st["E"].shape[0], F)
    P = np.full((U, W), np.nan, np.float32)
    Q = np.full((st["E"].shape[0] - U, W), np.nan, np.float32)
    c0 = np.full(1, np.nan, np.float32)
    rc = L.daisy_fmbn_rank_tables(h, ctypes.byref(prm), W, _p(P), _p(Q), _p(c0), None)
    assert rc == 0, L.emu_last_error()
    return P, Q, c0, L, h, prm


@pytest.mark.parametrize("U,I,F", [(9, 150, 5), (7, 40, 1), (5, 33, 8), (4, 60, 255)])
def test_fmbn_rank_tables_emulated(U, I, F):
    rng = np.random.default_rng(U * 1000 + F)
    st = random_state(rng, U, I, F, bn=True)
    W = (F + 4) // 4 * 4
    P, Q, c0, L, h, prm = fold(st, U, W)
    Pn, Qn = numpy_fold(st, U, W)                   # a_f in fp32 as k_fm_forward forms it; padding columns exactly 0
    assert np.array_equal(P.view(np.int32), Pn.view(np.int32)) and np.array_equal(Q.view(np.int32), Qn.view(np.int32))
    a64 = st["gamma"].astype(np.float64) / np.sqrt(st["rv"].astype(np.float64) + BN_EPS)
    want = float((st["beta"] - a64 * st["rm"]).sum())
    assert abs(float(c0[0]) - want) <= 1e-6 * (np.abs(st["beta"]).sum() + np.abs(a64 * st["rm"]).sum()) + 1e-7
    P2, Q2, c02 = fold(st, U, W)[:3]                                                        # the same bits again
    assert np.array_equal(P.view(np.int32), P2.view(np.int32)) and np.array_equal(Q.view(np.int32), Q2.view(np.int32))
    assert c0.view(np.int32)[0] == c02.view(np.int32)[0]
    # argument checks: W below F + 1 or not a multiple of 4, null outputs
    for bad_w in (W - 4, W + 2):
        if bad_w >= 1:
            assert L.daisy_fmbn_rank_tables(h, ctypes.byref(prm), bad_w, _p(P), _p(Q), _p(c0), None) != 0
    assert L.daisy_fmbn_rank_tables(h, ctypes.byref(prm), W, None, _p(Q), _p(c0), None) != 0
    assert L.emu_err_flag(h) == 0


def _offsets(st, U, users, c0):
    return (st["b"][users] + st["bias_"]) + c0[0]


def test_fmbn_folded_tables_rank_emulated_against_the_oracle():
    """The folded tables through daisy_topk_candidates and daisy_topk_full (exact path, with exclusions), plus the
    per-user term added afterwards, as metrics.topk_candidates / topk_full do."""
    rng = np.random.default_rng(11)
    U, I, F, N, C, K = 13, 300, 7, 5, 120, 10
    st = random_state(rng, U, I, F, bn=True)
    W = 8
    P, Q, c0 = fold(st, U, W)[:3]
    users = rng.integers(0, U, N).astype(np.int32)
    users[1] = users[0]
    cands = np.stack([rng.permutation(I)[:C] for _ in range(N)]).astype(np.int32)
    L, h = _lib_emu("bpr_eval", U, I, W)
    pos, item, score = np.zeros((N, K), np.int32), np.zeros((N, K), np.int32), np.zeros((N, K), np.float32)
    rc = L.daisy_topk_candidates(h, _p(P), _p(Q), _p(users), _p(cands), N, C, K, _p(pos), _p(item), _p(score), None)
    assert rc == 0 and L.emu_err_flag(h) == 0, L.emu_last_error()
    assert np.array_equal(item, np.take_along_axis(cands, pos, 1))
    check_ranking(pos, score + _offsets(st, U, users, c0)[:, None], *oracle_scores(st, U, users, cands))
    L, h = _lib_emu("topk_full", U, I, W)
    excl = [np.sort(rng.choice(I, 6, replace=False)).astype(np.int32) for _ in range(N)]
    ptr = np.zeros(N + 1, np.int64)
    ptr[1:] = np.cumsum([len(e) for e in excl])
    idx = np.concatenate(excl)
    fi, fs = np.zeros((N, K), np.int32), np.zeros((N, K), np.float32)
    rc = L.daisy_topk_full(h, _p(P), _p(Q), _p(users), N, K, _p(ptr), _p(idx), _p(fi), _p(fs), None)
    assert rc == 0 and L.emu_err_flag(h) == 0, L.emu_last_error()
    ora, eps = oracle_scores(st, U, users, np.tile(np.arange(I), (N, 1)))
    for n in range(N):
        ora[n, excl[n]] = -np.inf
    check_ranking(fi, fs + _offsets(st, U, users, c0)[:, None], ora, eps)


def numpy_fold(st, U, W):
    """The fold in numpy fp32, formed as k_fm_rank_rows forms it: (P, Q)."""
    F = st["E"].shape[1]
    a = st["gamma"] * (np.float32(1) / np.sqrt(st["rv"] + np.float32(BN_EPS)))
    P = np.zeros((U, W), np.float32)
    Q = np.zeros((st["E"].shape[0] - U, W), np.float32)
    P[:, :F], P[:, F] = a * st["E"][:U], 1
    Q[:, :F], Q[:, F] = st["E"][U:], st["b"][U:]
    return P, Q


def test_fmbn_folded_tables_full_catalogue_filter_emulated(monkeypatch):
    """At I = 131 072 (the smallest catalogue the filter serves) daisy_topk_full's CUDA-core filter returns the exact
    path's items and scores bit for bit on the folded tables, and both match the oracle.  Folding 131 072 rows takes
    minutes on host threads (every CUDA thread is an OS thread), so by default the emulated fold covers the users and the
    first 2 048 items and must equal the numpy fp32 fold there bit for bit; the rest of Q is that numpy fold.
    DAISY_EMU_FULL=1 folds every row under the emulation."""
    rng = np.random.default_rng(12)
    U, I, F, N, K = 20, 131072, 3, 3, 10
    st = random_state(rng, U, I, F, bn=True)
    W = 4
    full = os.environ.get("DAISY_EMU_FULL") == "1"
    part = st if full else dict(st, E=st["E"][:U + 2048], b=st["b"][:U + 2048])
    P, Qe, c0 = fold(part, U, W)[:3]
    Pn, Q = numpy_fold(st, U, W)
    assert np.array_equal(P.view(np.int32), Pn.view(np.int32))
    assert np.array_equal(Qe.view(np.int32), Q[:len(Qe)].view(np.int32))
    users = rng.integers(0, U, N).astype(np.int32)
    served = c_i32(), c_i64(), c_i64()
    out = {}
    for path in ("exact", "filter"):
        monkeypatch.setenv("DAISY_TOPK_PATH", path)
        L, h = _lib_emu("topk_full", U, I, W)
        fi, fs = np.zeros((N, K), np.int32), np.zeros((N, K), np.float32)
        rc = L.daisy_topk_full(h, _p(P), _p(Q), _p(users), N, K, None, None, _p(fi), _p(fs), None)
        assert rc == 0 and L.emu_err_flag(h) == 0, L.emu_last_error()
        assert L.daisy_topk_full_path(h, *map(ctypes.byref, served)) == 0
        assert served[0].value == (1 if path == "filter" else 0), path                  # DAISY_TOPK_PATH_SIMT / _EXACT
        out[path] = fi, fs
    assert np.array_equal(out["exact"][0], out["filter"][0])
    assert np.array_equal(out["exact"][1].view(np.int32), out["filter"][1].view(np.int32))
    ora, eps = oracle_scores(st, U, users, np.tile(np.arange(I), (N, 1)))
    check_ranking(out["exact"][0], out["exact"][1] + _offsets(st, U, users, c0)[:, None], ora, eps)
