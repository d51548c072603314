"""CPU execution of the NeuMF ranking unit (csrc/neumf_rank.cu: daisy_neumf_topk_candidates / daisy_neumf_topk_full) under
the host emulation of tests/emu, against the float64 NeuMF oracle: small shapes of both models and both modes, the
padded layer-0 path (MLP width not a multiple of 4), the mode and batching invariants, and the bad-id flags.  The same
checks at real sizes run on the B200 in tests/test_neumf_rank_gpu.py."""
import ctypes
import os
import sys

import numpy as np
import pytest

from conftest import ROOT
from neumf_rank_testing import check_ranking, oracle_scores, random_tower

sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
import build_emu  # noqa: E402

from recommend_lib_b200 import _lib  # noqa: E402  (only the ctypes structure definitions are used here)

c_vp, c_i64, c_i32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int


class RankEmu:
    def __init__(self, init, model, L, U, I):
        self.L = ctypes.CDLL(build_emu.build("neumf_rank"))
        PP = ctypes.POINTER(_lib.NeuMFParams)
        self.L.daisy_neumf_topk_candidates.argtypes = [c_vp, PP, c_vp, c_vp, c_i64, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp]
        self.L.daisy_neumf_topk_full.argtypes = [c_vp, PP, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp]
        self.L.emu_handle_dims.restype = c_vp
        self.L.emu_handle_dims.argtypes = [ctypes.c_longlong, ctypes.c_longlong, c_i32]
        self.L.emu_err_flag.argtypes = [c_vp]
        self.L.emu_last_error.restype = ctypes.c_char_p
        self.h = c_vp(self.L.emu_handle_dims(U, I, 4))
        self.T = {k: np.ascontiguousarray(v, dtype=np.float32).copy() for k, v in init.items()}
        p = lambda a: c_vp(a.ctypes.data)
        arr = lambda xs: (c_vp * 6)(*[x.ctypes.data for x in xs], *([None] * (6 - L)))
        T = self.T
        self.prm = _lib.NeuMFParams(int(model != "MLP"), L, T["Pg"].shape[1], U, I, p(T["Pg"]), p(T["Qg"]), p(T["Pm"]),
                                    p(T["Qm"]), arr([T[f"W{l}"] for l in range(L)]), arr([T[f"b{l}"] for l in range(L)]),
                                    p(T["wp"]), p(T["bp"]))   # moment pointers left NULL: only the forward fields are read

    def cand(self, users, cands, K):
        users, cands = np.ascontiguousarray(users, np.int32), np.ascontiguousarray(cands, np.int32)
        N, C = cands.shape
        pos, item, score = np.zeros((N, K), np.int32), np.zeros((N, K), np.int32), np.zeros((N, K), np.float32)
        rc = self.L.daisy_neumf_topk_candidates(self.h, ctypes.byref(self.prm), c_vp(users.ctypes.data),
                                                c_vp(cands.ctypes.data), N, C, K, c_vp(pos.ctypes.data),
                                                c_vp(item.ctypes.data), c_vp(score.ctypes.data), None)
        assert rc == 0, self.L.emu_last_error()
        return pos, item, score

    def full(self, users, K, excl=None):
        users = np.ascontiguousarray(users, np.int32)
        N = len(users)
        item, score = np.zeros((N, K), np.int32), np.zeros((N, K), np.float32)
        ptr = idx = None
        if excl is not None:
            ptr = np.zeros(N + 1, np.int64)
            ptr[1:] = np.cumsum([len(e) for e in excl])
            idx = np.concatenate([np.asarray(e, np.int32) for e in excl]).astype(np.int32)
        rc = self.L.daisy_neumf_topk_full(self.h, ctypes.byref(self.prm), c_vp(users.ctypes.data), N, K,
                                          c_vp(ptr.ctypes.data) if ptr is not None else None,
                                          c_vp(idx.ctypes.data) if idx is not None else None,
                                          c_vp(item.ctypes.data), c_vp(score.ctypes.data), None)
        assert rc == 0, self.L.emu_last_error()
        return item, score

    def err(self):
        return self.L.emu_err_flag(self.h)


# (model, U, I, F, L): two hidden layers with a partial weight chunk; the GMF branch; L = 1 with an MLP width of 3
# (padded layer-0 operands); a width above 256 (the 64-item tile)
@pytest.mark.parametrize("model,U,I,F,L", [("NeuMF-end", 9, 150, 8, 3), ("MLP", 7, 70, 3, 1), ("NeuMF-end", 5, 40, 5, 2),
                                           ("MLP", 4, 70, 160, 2)])
def test_neumf_rank_emulated_matches_the_oracle(model, U, I, F, L):
    rng = np.random.default_rng(U * 100 + F)
    init = random_tower(rng, U, I, F, L, model)
    m = RankEmu(init, model, L, U, I)
    N, C, K = 3, min(I, 131), 7
    users = rng.integers(0, U, N).astype(np.int32)
    users[1] = users[0]                                                  # a repeated user
    cands = np.stack([rng.permutation(I)[:C] for _ in range(N)]).astype(np.int32)
    pos, item, score = m.cand(users, cands, K)
    assert np.array_equal(item, np.take_along_axis(cands, pos, 1))
    check_ranking(pos, score, oracle_scores(init, model, L, users, cands))
    # full catalogue with exclusions; then the invariants: C = I candidates in item order equals full mode, a user
    # ranked alone equals the same user in a batch
    excl = [rng.choice(I, 5, replace=False) for _ in range(N)]
    fi, fs = m.full(users, K, excl)
    ora = oracle_scores(init, model, L, users, np.tile(np.arange(I), (N, 1)))
    for n in range(N):
        ora[n, excl[n]] = -np.inf
    check_ranking(fi, fs, ora)
    fi, fs = m.full(users, K)
    p2, i2, s2 = m.cand(users, np.tile(np.arange(I, dtype=np.int32), (N, 1)), K)
    assert np.array_equal(fi, i2) and np.array_equal(fs.view(np.int32), s2.view(np.int32))
    ai, as_ = m.full(users[2:3], K)
    assert np.array_equal(ai[0], fi[2]) and np.array_equal(as_[0].view(np.int32), fs[2].view(np.int32))
    assert m.err() == 0


@pytest.mark.parametrize("what", ["user", "candidate", "exclusion"])
def test_neumf_rank_emulated_flags_bad_ids(what):
    rng = np.random.default_rng(4)
    U, I, F, L = 6, 50, 4, 2
    init = random_tower(rng, U, I, F, L, "NeuMF-end")
    m = RankEmu(init, "NeuMF-end", L, U, I)
    users = np.array([1, 2, 3], np.int32)
    cands = np.stack([rng.permutation(I)[:20] for _ in range(3)]).astype(np.int32)
    if what == "user":
        users[1] = U
        m.cand(users, cands, 5)
    elif what == "candidate":
        cands[2, 7] = I
        m.cand(users, cands, 5)
    else:
        m.full(users, 5, [[1], [I + 3], []])
    assert m.err() == 1
