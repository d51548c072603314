"""CPU execution of kernels that have NOT run on a GPU yet (csrc/fmbn.cu, csrc/sgns.cu, csrc/neumf.cu, csrc/svdpp.cu;
SURVEY.md section 8f rows N3 / N4).

tests/emu compiles the product's own translation units for the host against a functional emulation of the CUDA
execution model (OS threads, block / warp barriers, shuffle exchange buffers) and this file drives the SAME extern "C"
entry points the GPU path exports, against the golden runs of the unmodified reference and the oracle.  It checks
indexing, reductions and arithmetic; it is not a product path (nothing in recommend_lib_b200 can reach it), not a
performance statement, and not a substitute for tests/test_bprfm_bn_gpu.py / test_sgns_gpu.py / test_neumf_gpu.py on the B200.

Memcheck (compute-sanitizer is closed on the GPU pool): the same tests pass with the units built under AddressSanitizer +
UBSan --
    DAISY_EMU_SANITIZE=1 LD_PRELOAD="$(gcc -print-file-name=libasan.so) $(gcc -print-file-name=libubsan.so)" \
        ASAN_OPTIONS=detect_leaks=0 python -m pytest tests/test_kernel_emulation.py
(12 passed, no report, with all three units, at the state of the commit that added csrc/neumf.cu).
Race check: every emulated CUDA thread is an OS thread, so ThreadSanitizer sees a missing __syncthreads or two threads
writing one location (validated on a kernel with its barrier removed: one report; with it: none) --
    DAISY_EMU_SANITIZE=thread LD_PRELOAD="$(gcc -print-file-name=libtsan.so)" TSAN_OPTIONS=report_signal_unsafe=0 \
        python -m pytest tests/test_kernel_emulation.py
(12 passed, no data-race report; the SVD++ unit added later: its four kernel tests clean under both as well, and the
whole file -- 26 tests, the emulated GPU-test runs included -- passes under AddressSanitizer + UBSan without a report).

The gated GPU test FILES of the experimental units also run here, over the emulated kernels (last section): a small
parameter set by default, the rest with DAISY_EMU_FULL=1 (about a quarter of an hour on 8 host cores)."""
import ctypes
import os
import sys

import numpy as np
import pytest

from conftest import ROOT, rel_err

sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
import build_emu  # noqa: E402

from recommend_lib_b200 import _lib  # noqa: E402  (only the ctypes structure definitions are used here)

c_vp, c_i64, c_i32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int


def _load(unit):
    L = ctypes.CDLL(build_emu.build(unit))
    L.emu_handle.restype = c_vp
    L.emu_last_error.restype = ctypes.c_char_p
    L.emu_err_flag.argtypes = [c_vp]
    L.emu_err_pos.argtypes = [c_vp]
    return L


def _p(a):
    return c_vp(a.ctypes.data) if a is not None else None


def _scratch(nbytes):
    raw = np.zeros(nbytes + 256, dtype=np.uint8)
    off = (-raw.ctypes.data) % 256
    return raw, c_vp(raw.ctypes.data + off)


# ------------------------------------------------------------------------------------------------ BPR-FM, batch norm
class FmEmu:
    def __init__(self, E0, b0, U, lr, acc0):
        self.L = _load("fmbn")
        self.L.daisy_fmbn_scratch_bytes.argtypes = [c_i64, c_i32, ctypes.POINTER(c_i64)]
        self.L.daisy_fmbn_step.argtypes = [c_vp, ctypes.POINTER(_lib.FMBNParams), c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp]
        self.L.daisy_fmbn_forward.argtypes = [c_vp, ctypes.POINTER(_lib.FMBNParams), c_vp, c_i64, c_vp, c_vp, c_vp]
        self.h = c_vp(self.L.emu_handle())
        f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32).copy()
        self.E, self.b = f32(E0), f32(b0)
        N, F = self.E.shape
        self.accE, self.accb = np.full_like(self.E, acc0), np.full_like(self.b, acc0)
        self.gamma, self.beta = np.ones(F, np.float32), np.zeros(F, np.float32)
        self.accg, self.accbt = np.full(F, acc0, np.float32), np.full(F, acc0, np.float32)
        self.rm, self.rv = np.zeros(F, np.float32), np.ones(F, np.float32)
        self.prm = _lib.FMBNParams(_p(self.E), _p(self.b), _p(self.accE), _p(self.accb), _p(self.gamma), _p(self.beta),
                                   _p(self.accg), _p(self.accbt), _p(self.rm), _p(self.rv), lr, 1e-10, 1e-5, 0.1, U, N, F)
        self.loss = np.zeros(1, np.float64)

    def step(self, tri, mi, mj):
        tri = np.ascontiguousarray(tri, dtype=np.int32)
        mi = None if mi is None else np.ascontiguousarray(mi, dtype=np.float32)
        mj = None if mj is None else np.ascontiguousarray(mj, dtype=np.float32)
        need = c_i64()
        assert self.L.daisy_fmbn_scratch_bytes(len(tri), self.E.shape[1], ctypes.byref(need)) == 0
        raw, sp = _scratch(need.value)
        self.loss[0] = 0
        rc = self.L.daisy_fmbn_step(self.h, ctypes.byref(self.prm), _p(tri), len(tri), _p(mi), _p(mj), sp, need.value,
                                    _p(self.loss), None)
        assert rc == 0, self.L.emu_last_error()
        return float(self.loss[0])

    def forward(self, tri):
        tri = np.ascontiguousarray(tri, dtype=np.int32)
        pi, pj = np.zeros(len(tri), np.float32), np.zeros(len(tri), np.float32)
        assert self.L.daisy_fmbn_forward(self.h, ctypes.byref(self.prm), _p(tri), len(tri), _p(pi), _p(pj), None) == 0
        return pi, pj


@pytest.mark.parametrize("branch,tol_E,tol_b", [("cond", 1e-5, 1e-5), ("script", 1e-4, 2e-4)])
def test_fmbn_kernels_emulated_match_the_reference_golden_run(golden, branch, tol_E, tol_b):
    g = golden("bprfm_bn_small.npz")
    k = lambda name: g[f"{branch}_{name}"]
    U = int(k("user_num"))
    m = FmEmu(k("E0"), k("b0"), U, float(k("lr")), float(k("acc0")))
    for s in range(2):                                           # two of the four recorded steps keep the test short
        tri = np.stack([k("fi")[s][:, 0], k("fi")[s][:, 1] - U, k("fj")[s][:, 1] - U], 1)
        loss = m.step(tri, k("mi")[s], k("mj")[s])
        assert abs(loss - k("loss")[s]) <= 1e-5 * k("loss")[s], s
        assert rel_err(m.E, k("E")[s]) <= tol_E, (s, rel_err(m.E, k("E")[s]))
        assert rel_err(m.b, k("b")[s]) <= tol_b, (s, rel_err(m.b, k("b")[s]))
        assert rel_err(m.gamma, k("gamma")[s]) <= 1e-5 and rel_err(m.beta, k("beta")[s]) <= 2e-5, s
        assert rel_err(m.rm, k("rm")[s]) <= 1e-5 and rel_err(m.rv, k("rv")[s]) <= 1e-5, s


def test_fmbn_kernels_emulated_match_the_oracle_and_flag_bad_ids():
    from oracle import bprfm_oracle
    rng = np.random.default_rng(4)
    U, I, F, B, p = 30, 25, 40, 70, 0.5                          # F > 32: two lane-strided passes; ragged last block
    E0 = (rng.standard_normal((U + I, F)) * 0.4).astype(np.float32)
    b0 = (rng.standard_normal(U + I) * 0.05).astype(np.float32)
    tri = np.stack([rng.integers(0, U, B), rng.integers(0, I, B), rng.integers(0, I, B)], 1).astype(np.int32)
    tri[:20, 0] = 3
    tri[30:45, 1] = 5
    tri[-9:, 2] = 5
    tri[0, 2] = tri[0, 1]                                        # i == j
    keep = lambda: ((rng.random((B, F)) >= p) / (1 - p)).astype(np.float32)
    m = FmEmu(E0, b0, U, 0.05, 0.1)
    ora = bprfm_oracle.BPRFMFull(E0, b0, 0.0, True, lr=0.05, initial_accumulator_value=0.1)
    fi, fj = np.stack([tri[:, 0], U + tri[:, 1]], 1), np.stack([tri[:, 0], U + tri[:, 2]], 1)
    ones = np.ones((B, 2))
    for s, masks in enumerate([(keep(), keep()), (None, None)]):
        loss = m.step(tri, *masks)
        lo = ora.step(fi, ones, fj, ones, *masks)
        assert abs(loss - lo) <= 1e-5 * lo, s
        assert rel_err(m.E, ora.E) <= 1e-5 and rel_err(m.b, ora.bias) <= 1e-5, (s, rel_err(m.E, ora.E), rel_err(m.b, ora.bias))
        assert rel_err(m.gamma, ora.gamma) <= 1e-5 and rel_err(m.beta, ora.beta) <= 2e-5, s
        assert rel_err(m.rm, ora.running_mean) <= 1e-5 and rel_err(m.rv, ora.running_var) <= 1e-5, s
    pi, pj = m.forward(tri)
    oi, oj = ora.forward(fi, ones, fj, ones)
    ub = ora.bias[tri[:, 0]]                                     # the library leaves the user bias + bias_ to the caller
    assert np.allclose(pi + ub, oi, rtol=1e-4, atol=1e-5) and np.allclose(pj + ub, oj, rtol=1e-4, atol=1e-5)
    assert m.L.emu_err_flag(m.h) == 0
    bad = tri.copy()
    bad[17, 2] = I
    m.step(bad, None, None)
    assert m.L.emu_err_flag(m.h) == 1 and m.L.emu_err_pos(m.h) == 17


# ------------------------------------------------------------------------------------------------ Item2Vec / SGNS
class SgEmu:
    def __init__(self, iv0, ov0):
        self.L = _load("sgns")
        self.L.daisy_sgns_scratch_bytes.argtypes = [c_i64, c_i32, c_i32, c_i64, c_i32, ctypes.POINTER(c_i64)]
        self.L.daisy_sgns_step.argtypes = [c_vp, ctypes.POINTER(_lib.SGNSParams), c_vp, c_vp, c_vp, c_i64, c_i32, c_i32, c_i64,
                                           c_vp, c_i64, c_vp, c_vp]
        self.h = c_vp(self.L.emu_handle())
        f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32).copy()
        self.iv, self.ov = f32(iv0), f32(ov0)
        self.mom = [np.zeros_like(self.iv) for _ in range(4)]
        V, D = self.iv.shape
        self.prm = _lib.SGNSParams(_p(self.iv), _p(self.ov), _p(self.mom[0]), _p(self.mom[1]), _p(self.mom[2]), _p(self.mom[3]),
                                   1e-3, 0.9, 0.999, 1e-8, V, D, 0)
        self.t = 0
        self.loss = np.zeros(1, np.float64)

    def step(self, iw, ow, nw):
        i32 = lambda a: np.ascontiguousarray(a, dtype=np.int32)
        iw, ow, nw = i32(iw), i32(ow), i32(nw)
        B, C = ow.shape
        N = nw.shape[1] // C
        V, D = self.iv.shape
        need = c_i64()
        assert self.L.daisy_sgns_scratch_bytes(B, C, N, V, D, ctypes.byref(need)) == 0
        raw, sp = _scratch(need.value)
        self.t += 1
        self.loss[0] = 0
        rc = self.L.daisy_sgns_step(self.h, ctypes.byref(self.prm), _p(iw), _p(ow), _p(nw) if N else None, B, C, N, self.t, sp,
                                    need.value, _p(self.loss), None)
        assert rc == 0, self.L.emu_last_error()
        return float(self.loss[0])


@pytest.mark.parametrize("branch", ["w", "u"])
def test_sgns_kernels_emulated_match_the_reference_golden_run(golden, branch):
    g = golden("sgns_small.npz")
    k = lambda name: g[f"{branch}_{name}"]
    m = SgEmu(k("iv0"), k("ov0"))
    for s in range(2):
        loss = m.step(k("iword")[s], k("owords")[s], k("nwords")[s])
        assert abs(loss - k("losses")[s]) <= 1e-5 * k("losses")[s], s
        assert rel_err(m.iv, k("iv")[s]) <= 1e-5 and rel_err(m.ov, k("ov")[s]) <= 1e-5, (s, rel_err(m.iv, k("iv")[s]))
        assert np.abs(m.iv[0]).max() == 0 and np.abs(m.ov[0]).max() == 0


@pytest.mark.parametrize("V,D,B,C,N", [(23, 44, 19, 3, 2),       # D > 32, ragged block, rows without any ref
                                        (17, 8, 9, 5, 8),         # 45 refs per example: two groups of coalesced id loads
                                        (9, 300, 5, 2, 1),        # the script's e_dim: the 10-values-per-lane kernels
                                        (9, 420, 4, 1, 2)])       # ... and the 16-values-per-lane ones
def test_sgns_kernels_emulated_match_the_oracle_and_flag_bad_ids(V, D, B, C, N):
    from oracle import sgns_oracle
    rng = np.random.default_rng(8)
    iv0 = (rng.standard_normal((V, D)) * 0.3).astype(np.float32)
    ov0 = (rng.standard_normal((V, D)) * 0.3).astype(np.float32)
    iv0[0] = 0
    ov0[0] = 0
    m, ora = SgEmu(iv0, ov0), sgns_oracle.SGNSAdam(iv0, ov0)
    for s in range(2):
        iw, ow, nw = rng.integers(1, V - 3, B), rng.integers(0, V - 3, (B, C)), rng.integers(0, V - 3, (B, C * N))
        iw[:6] = 3
        nw[:, 0] = 5                                             # a hot output row: several slices in k_sgns_rows
        loss = m.step(iw, ow, nw)
        lo = ora.step(iw, ow, nw)
        assert abs(loss - lo) <= 1e-5 * lo, s
        assert rel_err(m.iv, ora.iv) <= 1e-5 and rel_err(m.ov, ora.ov) <= 1e-5, (s, rel_err(m.iv, ora.iv), rel_err(m.ov, ora.ov))
    assert m.L.emu_err_flag(m.h) == 0
    nw[B - 2, -1] = V
    m.step(iw, ow, nw)
    assert m.L.emu_err_flag(m.h) == 1 and m.L.emu_err_pos(m.h) == B - 2


# ------------------------------------------------------------------------------------------------ NCF: MLP / NeuMF-end
class NmEmu:
    def __init__(self, name, Pg, Qg, Pm, Qm, Ws, bs, wp, bp, lr):
        self.L = _load("neumf")
        PP = ctypes.POINTER(_lib.NeuMFParams)
        self.L.daisy_neumf_scratch_bytes.argtypes = [PP, c_i64, ctypes.POINTER(c_i64)]
        self.L.daisy_neumf_forward.argtypes = [c_vp, PP, c_vp, c_i64, c_vp, c_vp]
        self.L.daisy_neumf_step.argtypes = [c_vp, PP, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp]
        self.h = c_vp(self.L.emu_handle())
        f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32).copy()
        self.T = dict(Pg=f32(Pg), Qg=f32(Qg), Pm=f32(Pm), Qm=f32(Qm), wp=f32(wp).reshape(-1), bp=f32(bp).reshape(-1))
        self.W, self.b = [f32(W) for W in Ws], [f32(b) for b in bs]
        z = np.zeros_like
        self.M = {k: (z(v), z(v)) for k, v in self.T.items()}
        self.MW = [(z(W), z(W)) for W in self.W]
        self.Mb = [(z(b), z(b)) for b in self.b]
        nl = len(Ws)
        arr = lambda xs: (c_vp * 6)(*[x.ctypes.data for x in xs], *([None] * (6 - nl)))
        T, M = self.T, self.M
        self.prm = _lib.NeuMFParams(
            int(name != "MLP"), nl, T["Pg"].shape[1], T["Pm"].shape[0], T["Qm"].shape[0],
            _p(T["Pg"]), _p(T["Qg"]), _p(T["Pm"]), _p(T["Qm"]), arr(self.W), arr(self.b), _p(T["wp"]), _p(T["bp"]),
            _p(M["Pg"][0]), _p(M["Pg"][1]), _p(M["Qg"][0]), _p(M["Qg"][1]), _p(M["Pm"][0]), _p(M["Pm"][1]),
            _p(M["Qm"][0]), _p(M["Qm"][1]), arr([m for m, _ in self.MW]), arr([v for _, v in self.MW]),
            arr([m for m, _ in self.Mb]), arr([v for _, v in self.Mb]), _p(M["wp"][0]), _p(M["wp"][1]),
            _p(M["bp"][0]), _p(M["bp"][1]), lr, 0.9, 0.999, 1e-8)
        self.t = 0
        self.loss = np.zeros(1, np.float64)

    def step(self, users, items, labels):
        smp = np.ascontiguousarray(np.stack([users, items, np.asarray(labels).astype(np.int64)], 1), dtype=np.int32)
        need = c_i64()
        assert self.L.daisy_neumf_scratch_bytes(ctypes.byref(self.prm), len(smp), ctypes.byref(need)) == 0
        raw, sp = _scratch(need.value)
        self.t += 1
        self.loss[0] = 0
        rc = self.L.daisy_neumf_step(self.h, ctypes.byref(self.prm), _p(smp), len(smp), self.t, sp, need.value, _p(self.loss), None)
        assert rc == 0, self.L.emu_last_error()
        return float(self.loss[0])

    def forward(self, users, items):
        smp = np.ascontiguousarray(np.stack([users, items, np.zeros_like(users)], 1), dtype=np.int32)
        out = np.zeros(len(smp), np.float32)
        assert self.L.daisy_neumf_forward(self.h, ctypes.byref(self.prm), _p(smp), len(smp), _p(out), None) == 0
        return out


@pytest.mark.parametrize("tag,name", [("mlp", "MLP"), ("neumf", "NeuMF-end")])
def test_neumf_kernels_emulated_match_the_reference_golden_run(golden, tag, name):
    g = golden("neumf_small.npz")
    k = lambda n: g[f"{tag}_{n}"]
    L = int(k("num_layers"))
    m = NmEmu(name, k("Pg_0"), k("Qg_0"), k("Pm_0"), k("Qm_0"), [k(f"W{l}_0") for l in range(L)],
              [k(f"b{l}_0") for l in range(L)], k("wp_0"), k("bp_0"), float(k("lr")))
    for s in range(2):                                           # two of the four recorded steps keep the test short
        loss = m.step(k("users")[s], k("items")[s], k("labels")[s])
        assert abs(loss - k("loss")[s]) <= 1e-5 * k("loss")[s], s
        for key in ("Pg", "Qg", "Pm", "Qm", "wp"):
            assert rel_err(m.T[key], k(key)[s]) <= 1e-5, (s, key, rel_err(m.T[key], k(key)[s]))
        assert abs(m.T["bp"][0] - k("bp")[s][0]) <= 1e-6
        for l in range(L):
            assert rel_err(m.W[l], k(f"W{l}")[s]) <= 1e-5 and rel_err(m.b[l], k(f"b{l}")[s]) <= 2e-5, (s, l)
    if tag == "mlp":
        assert np.array_equal(m.T["Pg"], k("Pg_0")) and np.array_equal(m.T["Qg"], k("Qg_0"))


def test_neumf_kernels_emulated_match_the_oracle_and_flag_bad_ids():
    from oracle import neumf_oracle
    rng = np.random.default_rng(12)
    U, I, F, L, B = 21, 33, 12, 2, 37                           # F not a multiple of 32, ragged, items > users
    Dm = F << (L - 1)
    init = lambda *sh: (rng.standard_normal(sh) * 0.3).astype(np.float32)
    Pg, Qg, Pm, Qm = init(U, F), init(I, F), init(U, Dm), init(I, Dm)
    Ws, bs, n_in = [], [], 2 * Dm
    for l in range(L):
        Ws.append(init(n_in // 2, n_in))
        bs.append(init(n_in // 2) * 0.1)
        n_in //= 2
    wp, bp = init(2 * F), init(1)
    m = NmEmu("NeuMF-end", Pg, Qg, Pm, Qm, Ws, bs, wp, bp, 1e-3)
    ora = neumf_oracle.NeuMFAdam("NeuMF-end", Pg, Qg, Pm, Qm, Ws, bs, wp, bp, lr=1e-3)
    for s in range(2):
        u, i, y = rng.integers(0, U, B), rng.integers(0, I, B), (rng.random(B) < 0.3).astype(np.int64)
        u[:9] = 3
        i[10:18] = 5
        loss, lo = m.step(u, i, y), ora.step(u, i, y)
        assert abs(loss - lo) <= 1e-5 * lo, s
        for key, ref in (("Pg", ora.Pg), ("Qg", ora.Qg), ("Pm", ora.Pm), ("Qm", ora.Qm), ("wp", ora.wp), ("bp", ora.bp)):
            assert rel_err(m.T[key], ref) <= 1e-5, (s, key, rel_err(m.T[key], ref))
        for l in range(L):
            assert rel_err(m.W[l], ora.Ws[l]) <= 1e-5 and rel_err(m.b[l], ora.bs[l]) <= 1e-5, (s, l)
    assert np.allclose(m.forward(u, i), ora.forward(u, i), rtol=1e-4, atol=1e-5)
    assert m.L.emu_err_flag(m.h) == 0
    u[4] = U
    m.step(u, i, y)
    assert m.L.emu_err_flag(m.h) == 1 and m.L.emu_err_pos(m.h) == 4


# ------------------------------------------------------------------------------------------------ SVD++
class SvdppEmu:
    """daisy_svdpp_fit / daisy_svdpp_user_factors of csrc/svdpp.cu on host threads, fed by the product's own host logic
    (recommend_lib_b200.svdpp.user_histories)."""

    def __init__(self, U, I, D):
        self.L = _load("svdpp")
        self.L.daisy_svdpp_fit.argtypes = [c_vp] * 9 + [c_i64, c_i32, c_vp, c_vp, c_vp, ctypes.POINTER(_lib.SVDppParams), c_vp, c_vp]
        self.L.daisy_svdpp_user_factors.argtypes = [c_vp] * 7
        self.h = _dims_handle(self.L, U, I, D)
        self.U, self.I, self.D = U, I, D

    def fit(self, users, items, ratings, pu, qi, yj, epochs, lr=.007, reg=.02, mu=None):
        from recommend_lib_b200.svdpp import user_histories
        users = np.ascontiguousarray(users, dtype=np.int32)
        items = np.ascontiguousarray(items, dtype=np.int32)
        ratings = np.ascontiguousarray(ratings, dtype=np.float64)
        ptr, idx, mult = user_histories(np.clip(users, 0, self.U - 1), items, self.U)
        self.ptr, self.idx, self.mult = ptr, idx, mult
        o = dict(pu=np.array(pu, dtype=np.float64), qi=np.array(qi, dtype=np.float64), yj=np.array(yj, dtype=np.float64),
                 bu=np.zeros(self.U), bi=np.zeros(self.I), sse=np.zeros(max(epochs, 1)))
        prm = _lib.SVDppParams(lr, lr, lr, lr, lr, reg, reg, reg, reg, reg, float(ratings.mean() if mu is None else mu))
        rc = self.L.daisy_svdpp_fit(self.h, _p(o["pu"]), _p(o["qi"]), _p(o["yj"]), _p(o["bu"]), _p(o["bi"]), _p(users), _p(items),
                                    _p(ratings), len(ratings), epochs, _p(ptr), _p(idx), _p(mult), ctypes.byref(prm),
                                    _p(o["sse"]), None)
        assert rc == 0, self.L.emu_last_error()
        return o

    def user_factors(self, pu, yj):
        z = np.zeros_like(pu)
        assert self.L.daisy_svdpp_user_factors(self.h, _p(pu), _p(yj), _p(self.ptr), _p(self.idx), _p(z), None) == 0
        return z


def test_svdpp_kernels_emulated_match_the_reference_golden_run(golden, monkeypatch):
    """tests/golden/svdpp_small.npz: 3 epochs of the reference's own compiled SVDpp (repeated (user, item) ratings
    included).  float64, sums re-associated over warps / lanes -> 1e-9 like the funk-SVD tests."""
    monkeypatch.setenv("DAISY_SVDPP_THREADS", "64")                 # 2 warps: histories longer than the warp count
    g = golden("svdpp_small.npz")
    U, I, D, E = int(g["U"]), int(g["I"]), int(g["D"]), int(g["E"])
    e = SvdppEmu(U, I, D)
    o = e.fit(g["users"], g["items"], g["ratings"], g["pu0"], g["qi0"], g["yj0"], E)
    assert e.mult is not None and e.mult.max() >= 2                 # the fixture does repeat a (user, item) pair
    for k in ("pu", "qi", "yj", "bu", "bi"):
        assert np.allclose(o[k], g[k], rtol=1e-9, atol=1e-12), k
    z = e.user_factors(o["pu"], o["yj"])
    pred = float(g["mu"]) + o["bu"][g["users"][:15]] + o["bi"][g["items"][:15]] + \
        np.einsum("nd,nd->n", o["qi"][g["items"][:15]], z[g["users"][:15]])
    assert np.allclose(pred, g["pred"], rtol=1e-9, atol=1e-12)
    assert e.L.emu_err_flag(e.h) == 0


@pytest.mark.parametrize("U,I,D,n,E,threads", [(17, 23, 44, 260, 2, 64),     # D > 32, ragged
                                              (9, 12, 130, 90, 1, 160),     # D > 128, 5 warps
                                              (1, 40, 8, 2100, 1, 64)])     # a history longer than the shared-memory list
def test_svdpp_kernels_emulated_match_the_oracle_and_flag_bad_ids(monkeypatch, U, I, D, n, E, threads):
    from oracle import mf_oracle
    monkeypatch.setenv("DAISY_SVDPP_THREADS", str(threads))
    rng = np.random.default_rng(U * 1000 + D)
    users = rng.integers(0, max(U - 2, 1), n)                       # the last users have no rating at all
    items = (rng.zipf(1.3, n) - 1) % I                              # skewed: items repeat across and within histories
    users[5], items[5] = users[4], items[4]                         # a repeated (user, item) pair for sure
    ratings = rng.integers(1, 6, n).astype(np.float64)
    pu0, qi0, yj0 = (rng.normal(0, .1, s) for s in ((U, D), (I, D), (I, D)))
    ref = mf_oracle.svdpp_fit(users, items, ratings, pu0, qi0, yj0, n_epochs=E)
    e = SvdppEmu(U, I, D)
    o = e.fit(users, items, ratings, pu0, qi0, yj0, E)
    rptr, ridx = mf_oracle.user_item_lists(users, items, U)
    assert np.array_equal(e.ptr, rptr) and np.array_equal(e.idx, ridx)
    for k in ("pu", "qi", "yj", "bu", "bi"):
        assert np.allclose(o[k], ref[k], rtol=1e-9, atol=1e-12), k
    assert np.isclose(o["sse"][E - 1], ref["sse"], rtol=1e-9)
    z = e.user_factors(o["pu"], o["yj"])
    for u in (0, U - 1):
        Iu = ridx[rptr[u]:rptr[u + 1]]
        want = o["pu"][u] + (o["yj"][Iu].sum(0) / np.sqrt(len(Iu)) if len(Iu) else 0)
        assert np.allclose(z[u], want, rtol=1e-12, atol=1e-14)
    assert e.L.emu_err_flag(e.h) == 0
    # an out-of-range item: flagged, nothing written
    bad = items.copy()
    bad[n // 2] = I
    e2 = SvdppEmu(U, I, D)
    o2 = e2.fit(users, np.minimum(bad, I - 1), ratings, pu0, qi0, yj0, 0)      # lists built from valid ids
    prm = _lib.SVDppParams(.007, .007, .007, .007, .007, .02, .02, .02, .02, .02, float(ratings.mean()))
    bad32, u32 = bad.astype(np.int32), users.astype(np.int32)
    assert e2.L.daisy_svdpp_fit(e2.h, _p(o2["pu"]), _p(o2["qi"]), _p(o2["yj"]), _p(o2["bu"]), _p(o2["bi"]), _p(u32), _p(bad32),
                                _p(ratings), n, 1, _p(e2.ptr), _p(e2.idx), _p(e2.mult), ctypes.byref(prm), None, None) == 0
    assert e2.L.emu_err_flag(e2.h) & 2 and e2.L.emu_err_pos(e2.h) == n // 2
    assert np.array_equal(o2["pu"], pu0) and np.array_equal(o2["yj"], yj0) and not o2["bu"].any()


def test_svdpp_drop_in_class_host_logic_over_the_emulated_kernels(golden, monkeypatch):
    """recommend_lib_b200.svdpp.SVDpp end to end (frame -> histories -> daisy_svdpp_fit -> attributes, predict, ur,
    user_factors) with the library handle swapped for the host build of csrc/svdpp.cu: the Python around the C ABI is
    exercised before it ever costs GPU time.  Only test scaffolding is patched; the product has no such switch."""
    import torch
    pd = pytest.importorskip("pandas")
    from recommend_lib_b200 import svdpp as mod
    L = _load("svdpp")
    L.emu_check.argtypes = [c_vp, c_vp]

    class EmuHandle:
        def __init__(self, device_index, user_num, item_num, dim, max_batch, flags=0):
            self.L = L
            self.ptr = _dims_handle(L, user_num, item_num, dim)
            L.daisy_check = L.emu_check

        def close(self):
            pass

    monkeypatch.setenv("DAISY_SVDPP_THREADS", "64")
    monkeypatch.setattr(mod._lib, "Handle", EmuHandle)
    monkeypatch.setattr(mod._lib, "require_cuda", lambda: torch)
    monkeypatch.setattr(mod._lib, "stream_ptr", lambda t, d: None)
    for name in ("daisy_svdpp_fit", "daisy_svdpp_user_factors"):      # what _lib.load() does for the real library
        getattr(L, name).argtypes = _lib.SIGNATURES[name]
    g = golden("svdpp_small.npz")
    U, I, D, E = int(g["U"]), int(g["I"]), int(g["D"]), int(g["E"])
    a = mod.SVDpp(U, I, n_factors=D, n_epochs=E, verbose=False, device="cpu:0")
    frame = pd.DataFrame({"user": g["users"], "item": g["items"], "rating": g["ratings"]})
    state = np.random.get_state()
    np.random.seed(3)
    a.fit(frame)                                                   # draws pu, qi, yj from numpy's global RNG like the reference
    np.random.seed(3)
    pu0, qi0, yj0 = (np.random.normal(0, .1, size=s) for s in ((U, D), (I, D), (I, D)))
    np.random.set_state(state)
    from oracle import mf_oracle
    ref = mf_oracle.svdpp_fit(g["users"], g["items"], g["ratings"], pu0, qi0, yj0, n_epochs=E)
    for k in ("pu", "qi", "yj", "bu", "bi"):
        assert np.allclose(getattr(a, k), ref[k], rtol=1e-9, atol=1e-12), k
    assert np.isclose(a.global_mean, ref["global_mean"]) and np.isclose(a.sse_[E - 1], ref["sse"], rtol=1e-9)
    for u, i in zip(g["users"][:10], g["items"][:10]):
        assert np.isclose(a.predict(int(u), int(i)), mf_oracle.svdpp_predict(int(u), int(i), ref), rtol=1e-9)
    u0 = int(g["users"][0])
    sel = g["users"] == u0
    assert a.ur[u0] == list(zip(g["items"][sel].tolist(), g["ratings"][sel].tolist()))      # the reference's self.ur
    z = a.user_factors()
    Iu = [j for j, _ in a.ur[u0]]
    assert np.allclose(z[u0], a.pu[u0] + a.yj[Iu].sum(0) / np.sqrt(len(Iu)), rtol=1e-12)
    with pytest.raises(ValueError, match="Invalid user code"):
        a.predict(U, 0)
    with pytest.raises(ValueError, match="Invalid item code"):
        a.fit(pd.DataFrame({"user": [0, 1], "item": [0, I], "rating": [3.0, 4.0]}))
    with pytest.raises(ValueError, match="Invalid user code"):
        a.fit(pd.DataFrame({"user": [0, U], "item": [0, 1], "rating": [3.0, 4.0]}))


# ------------------------------------------------------------------------------------------------ units that DO run on the GPU
# csrc/bpr_eval.cu (SURVEY 8a rows A2 / A8) and csrc/sampler.cu (8f row N1) are GPU-verified product code
# (tests/test_bpr_gpu.py, tests/test_sampler_gpu.py).  They are plain CUDA, so the same emulation gives them what the
# closed compute-sanitizer cannot on this pool: a memcheck / racecheck run (DAISY_EMU_SANITIZE=1 / thread, see above).
def _dims_handle(L, U, I, D):
    L.emu_handle_dims.restype = c_vp
    L.emu_handle_dims.argtypes = [ctypes.c_longlong, ctypes.c_longlong, c_i32]
    return c_vp(L.emu_handle_dims(U, I, D))


def test_eval_kernels_emulated_forward_and_candidate_topk():
    from oracle import bpr_oracle
    L = _load("bpr_eval")
    rng = np.random.default_rng(21)
    U, I, D, B, N, C, K = 37, 131, 24, 45, 11, 100, 10             # D / 4 = 6 lanes active; ragged B; C > 3 x 32
    P = (rng.standard_normal((U, D)) * 0.3).astype(np.float32)
    Q = (rng.standard_normal((I, D)) * 0.3).astype(np.float32)
    h = _dims_handle(L, U, I, D)
    tri = np.stack([rng.integers(0, U, B), rng.integers(0, I, B), rng.integers(0, I, B)], 1).astype(np.int32)
    pi, pj = np.zeros(B, np.float32), np.zeros(B, np.float32)
    L.daisy_bpr_forward.argtypes = [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp]
    assert L.daisy_bpr_forward(h, _p(P), _p(Q), _p(tri), B, _p(pi), _p(pj), None) == 0, L.emu_last_error()
    ri, rj = bpr_oracle.bpr_scores(P, Q, tri[:, 0], tri[:, 1], tri[:, 2])
    assert np.allclose(pi, ri, rtol=1e-5, atol=1e-6) and np.allclose(pj, rj, rtol=1e-5, atol=1e-6)
    users = rng.integers(0, U, N).astype(np.int32)
    cands = np.stack([rng.permutation(I)[:C - 1] for _ in range(N)]).astype(np.int32)
    cands = np.concatenate([cands, cands[:, :1]], 1)               # a duplicated candidate: an exact score tie
    cands = np.ascontiguousarray(cands[:, :C])
    assert cands.shape == (N, C)
    pos, item, score = np.zeros((N, K), np.int32), np.zeros((N, K), np.int32), np.zeros((N, K), np.float32)
    L.daisy_topk_candidates.argtypes = [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp]
    assert L.daisy_topk_candidates(h, _p(P), _p(Q), _p(users), _p(cands), N, C, K, _p(pos), _p(item), _p(score), None) == 0
    for g in range(N):
        sc = bpr_oracle.candidate_scores(P, Q, users[g], cands[g])
        assert np.array_equal(item[g], cands[g][pos[g]])
        assert np.allclose(score[g], sc[pos[g]], rtol=1e-5, atol=1e-6)
        assert np.all(np.diff(score[g]) <= 0)                                       # descending
        kth = np.sort(sc)[::-1][K - 1]
        assert score[g][-1] >= kth - 1e-5                                           # nothing better was left out
        ties = [a for a in range(K - 1) if score[g][a] == score[g][a + 1]]
        assert all(pos[g][a] < pos[g][a + 1] for a in ties)                         # ties: position ascending
    assert L.emu_err_flag(h) == 0


@pytest.mark.parametrize("shuffle", [0, 1])
def test_sampler_kernels_emulated_match_the_oracle_bit_for_bit(shuffle):
    from oracle import sampler_oracle
    L = _load("sampler")
    rng = np.random.default_rng(31)
    U, I, n_pairs, num_ng = 40, 23, 150, 3                        # dense positives: many rejected draws
    pairs = np.unique(np.stack([rng.integers(0, U, n_pairs), rng.integers(0, I, n_pairs)], 1), axis=0).astype(np.int32)
    keys = np.unique(pairs[:, 0].astype(np.int64) * I + pairs[:, 1]).astype(np.int64)
    h = _dims_handle(L, U, I, 4)
    out = np.zeros((len(pairs) * num_ng, 3), np.int32)
    L.daisy_sample_triples.argtypes = [c_vp, c_vp, c_i64, c_i32, c_vp, c_i64, ctypes.c_uint64, ctypes.c_uint32, c_i32, c_vp, c_vp]
    rc = L.daisy_sample_triples(h, _p(pairs), len(pairs), num_ng, _p(keys), len(keys), 2019, 5, shuffle, _p(out), None)
    assert rc == 0, L.emu_last_error()
    want = sampler_oracle.sample_epoch(pairs, I, num_ng, 2019, 5, bool(shuffle))
    assert np.array_equal(out, want)
    assert L.emu_err_flag(h) == 0


@pytest.mark.parametrize("world,n,batch", [(2, 1000, 256), (3, 777, 100), (4, 37, 8), (2, 5, 100)])
def test_route_triples_emulated_is_the_rank_share_of_every_global_batch(world, n, batch):
    """daisy_route_triples (csrc/sampler.cu; the e2e region of the N > 1 bench and PeerShardedBPR.fit route with it):
    every rank's share of a global epoch -- users in [u0, u1), order kept, user column made local, per-batch offsets --
    against the numpy routing of tests/sharded_testing.py."""
    from recommend_lib_b200.sharded import ShardLayout
    from sharded_testing import route
    L = _load("sampler")
    U, I = 203, 77
    rng = np.random.default_rng(n)
    tri = np.stack([rng.integers(0, U, n), rng.integers(0, I, n), rng.integers(0, I, n)], 1).astype(np.int32)
    layout = ShardLayout(U, I, world)
    h = _dims_handle(L, U, I, 4)
    L.daisy_route_triples.argtypes = [c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp]
    nb = (n + batch - 1) // batch
    total = 0
    for rank in range(world):
        u0, u1 = layout.user_range(rank)
        out = np.full((n, 3), -1, np.int32)
        off = np.full(nb + 1, -1, np.int64)
        rc = L.daisy_route_triples(h, _p(tri), n, batch, u0, u1, _p(out), _p(off), None)
        assert rc == 0, L.emu_last_error()
        assert off[0] == 0 and np.all(np.diff(off) >= 0)
        for k in range(nb):
            want = route(tri[k * batch:(k + 1) * batch], layout, rank)
            assert np.array_equal(out[off[k]:off[k + 1]], want), (rank, k)
        total += int(off[-1])
    assert total == n
    assert L.emu_err_flag(h) == 0


@pytest.mark.parametrize("I,D,N,K,paths", [(300, 16, 5, 10, ("exact",)), (131072, 8, 3, 10, ("exact", "filter"))])
def test_full_catalogue_topk_emulated(monkeypatch, I, D, N, K, paths):
    """csrc/topk_full.cu (row A9, GPU-verified): both selection strategies under the emulation; the filtered path must
    return exactly what the materialise-and-select path returns.  The filter case needs I >= 131 072: below that the
    sample threshold's rank passes 128 and the call takes the exact path whatever it is asked for.  Under the emulation
    the filter is the CUDA-core one (the tensor-core kernel is outside its reach)."""
    L = _load("topk_full")
    L.daisy_topk_full.argtypes = [c_vp, c_vp, c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp]
    L.daisy_topk_full_path.argtypes = [c_vp, ctypes.POINTER(c_i32), ctypes.POINTER(c_i64), ctypes.POINTER(c_i64)]
    served = c_i32(), c_i64(), c_i64()
    rng = np.random.default_rng(I + N)
    U = 20
    P = rng.standard_normal((U, D)).astype(np.float32)
    Q = rng.standard_normal((I, D)).astype(np.float32)
    Q[rng.integers(0, I, I // 20)] = Q[rng.integers(0, I, I // 20)]                # exactly tied scores
    users = rng.integers(0, U, N).astype(np.int32)
    excl = [np.sort(rng.choice(I, size=rng.integers(0, 30), replace=False)) for _ in range(N)]
    ptr = np.zeros(N + 1, np.int64)
    ptr[1:] = np.cumsum([len(e) for e in excl])
    idx = (np.concatenate(excl) if ptr[-1] else np.zeros(0)).astype(np.int32)
    ref = P[users].astype(np.float64) @ Q.astype(np.float64).T
    out = {}
    for path in paths:
        monkeypatch.setenv("DAISY_TOPK_PATH", path)
        h = _dims_handle(L, U, I, D)
        items, scores = np.zeros((N, K), np.int32), np.zeros((N, K), np.float32)
        rc = L.daisy_topk_full(h, _p(P), _p(Q), _p(users), N, K, _p(ptr), _p(idx) if len(idx) else None, _p(items), _p(scores), None)
        assert rc == 0, L.emu_last_error()
        assert L.emu_err_flag(h) == 0
        assert L.daisy_topk_full_path(h, *map(ctypes.byref, served)) == 0
        want = (1, N, 0) if path == "filter" else (0, 0, 0)                          # DAISY_TOPK_PATH_SIMT / _EXACT
        assert tuple(v.value for v in served) == want, path
        out[path] = (items, scores)
        for n in range(N):
            r = ref[n].copy()
            r[excl[n]] = -np.inf
            got = items[n]
            assert len(set(got.tolist())) == K and not (set(got.tolist()) & set(excl[n].tolist()))
            assert np.allclose(scores[n], r[got], rtol=1e-4, atol=1e-4)
            assert (np.diff(scores[n]) <= 0).all()
            tie = np.diff(scores[n]) == 0
            assert (np.diff(got)[tie] > 0).all()
            kth = np.sort(r)[-K]
            assert set(np.nonzero(r > kth + 1e-3)[0].tolist()) <= set(got.tolist()) and r[got].min() >= kth - 1e-3
    if len(paths) == 2:
        assert np.array_equal(out["exact"][0], out["filter"][0]) and np.array_equal(out["exact"][1], out["filter"][1])
        # an exclusion id outside the catalogue raises the error flag on the filtered path too, not only in k_mask
        bad = idx.copy() if len(idx) else np.zeros(1, np.int32)
        bad[-1] = I
        ptr_bad = ptr.copy()
        ptr_bad[-1] = len(bad)
        h = _dims_handle(L, U, I, D)
        rc = L.daisy_topk_full(h, _p(P), _p(Q), _p(users), N, K, _p(ptr_bad), _p(bad), _p(items), _p(scores), None)
        assert rc == 0 and L.emu_err_flag(h) != 0 and L.emu_err_pos(h) == N - 1
        assert L.daisy_topk_full_path(h, *map(ctypes.byref, served)) == 0 and served[0].value == 1


# ------------------------------------------------------------------------------------------------ the gated GPU tests themselves
# The functions of tests/test_*_gpu.py of the four experimental units are called here directly (their skip marks only act
# under collection) with the product's library handle swapped for the host build of the unit and `dev` = the CPU: the
# Python around the C ABI -- module structure, argument marshalling, scratch sizing, error mapping -- and the GPU tests'
# own assertions run before they cost GPU time.  Only small parameter sets (every CUDA thread is an OS thread).
class _EmuProduct:
    """Swap recommend_lib_b200._lib's device plumbing for the host build of one unit (test scaffolding only)."""

    def __init__(self, monkeypatch, unit):
        import torch
        from recommend_lib_b200 import _lib as plib
        L = _load(unit)
        L.emu_check.argtypes = [c_vp, c_vp]
        L.daisy_check = L.emu_check
        L.daisy_launch_count = lambda *a: 0
        for name, argtypes in plib.SIGNATURES.items():      # what _lib.load() does for the real library
            if name != "daisy_check" and hasattr(L, name):
                getattr(L, name).argtypes = argtypes
                getattr(L, name).restype = ctypes.c_int

        class EmuHandle:
            def __init__(self, device_index, user_num, item_num, dim, max_batch, flags=0):
                self.L, self.device_index = L, device_index
                self.ptr = _dims_handle(L, user_num, item_num, dim)

            def close(self):
                pass

        real_empty = torch.empty

        def aligned_empty(*size, **kw):         # scratch buffers must be 256-byte aligned (CUDA allocations are)
            if kw.get("dtype") is torch.uint8 and len(size) == 1 and isinstance(size[0], int):
                raw = real_empty(size[0] + 256, **kw)
                off = (-raw.data_ptr()) % 256
                out = raw[off:off + size[0]]
                out._keepalive = raw
                return out
            return real_empty(*size, **kw)

        monkeypatch.setattr(plib, "Handle", EmuHandle)
        monkeypatch.setattr(plib, "require_cuda", lambda: torch)
        monkeypatch.setattr(plib, "stream_ptr", lambda t, d: None)
        monkeypatch.setattr(torch, "empty", aligned_empty)
        monkeypatch.setattr(torch.cuda, "current_device", lambda: 0)
        self.L = L


def test_sgns_gpu_tests_pass_over_the_emulated_kernels(golden, monkeypatch):
    import torch
    import test_sgns_gpu as G
    from recommend_lib_b200 import item2vec
    _EmuProduct(monkeypatch, "sgns")
    monkeypatch.setattr(item2vec.SGNSAdam, "_device", lambda self: self.sgns.embedding.ivectors.weight.device)
    cpu = torch.device("cpu")
    G.test_sgns_against_oracle(cpu, 64, 36, 7, 1, 0)
    G.test_sgns_reports_bad_ids(cpu)
    if os.environ.get("DAISY_EMU_FULL") == "1":                  # minutes on host threads
        G.test_sgns_golden_five_steps(golden, cpu, "u")
        G.test_sgns_golden_five_steps(golden, cpu, "w")
        G.test_sgns_against_oracle(cpu, 50, 16, 33, 3, 2)
        G.test_sgns_is_bit_reproducible_and_draws_its_own_negatives(cpu)


def test_fmbn_gpu_tests_pass_over_the_emulated_kernels(golden, monkeypatch):
    import torch
    import test_bprfm_bn_gpu as G
    from recommend_lib_b200 import bprfm_bn
    _EmuProduct(monkeypatch, "fmbn")
    monkeypatch.setattr(bprfm_bn.BPRFMBN, "_device", lambda self: self.embeddings.weight.device)
    cpu = torch.device("cpu")
    G.test_fmbn_golden_four_steps(golden, cpu, "cond", 1e-5, 1e-5)
    G.test_fmbn_against_oracle(cpu, 50, 40, 8, 96, 0.5)
    G.test_fmbn_reports_bad_ids_and_refuses_training_mode_forward(cpu)
    if os.environ.get("DAISY_EMU_FULL") == "1":
        G.test_fmbn_golden_four_steps(golden, cpu, "script", 1e-4, 2e-4)
        G.test_fmbn_is_bit_reproducible_and_draws_its_own_masks(cpu)


def test_neumf_gpu_tests_pass_over_the_emulated_kernels(golden, monkeypatch):
    import torch
    import test_neumf_gpu as G
    from recommend_lib_b200 import ncf_mlp
    _EmuProduct(monkeypatch, "neumf")
    monkeypatch.setattr(ncf_mlp.NeuMF, "_device", lambda self: self.embed_user_MLP.weight.device)
    cpu = torch.device("cpu")
    G.test_neumf_against_oracle(cpu, "MLP", 50, 70, 8, 1, 33)
    if os.environ.get("DAISY_EMU_FULL") == "1":
        G.test_neumf_golden_four_steps(golden, cpu, "mlp", "MLP")
        G.test_neumf_golden_four_steps(golden, cpu, "neumf", "NeuMF-end")
        G.test_neumf_is_bit_reproducible_and_reports_bad_ids(cpu)


def test_svdpp_gpu_tests_pass_over_the_emulated_kernels(golden, monkeypatch):
    import torch
    import test_svdpp_gpu as G
    from recommend_lib_b200 import svdpp as mod
    _EmuProduct(monkeypatch, "svdpp")
    d = list(mod.SVDpp.__init__.__defaults__)
    assert d[-1] == "cuda"
    monkeypatch.setattr(mod.SVDpp.__init__, "__defaults__", tuple(d[:-1] + ["cpu:0"]))

    def predict_many(user_num, item_num, n_factors, A, Bm, ba, bb, users, items, with_bias, mu, device):
        u, i = np.asarray(users), np.asarray(items)          # daisy_mf_predict lives in csrc/mf.cu (GPU-verified, not emulable)
        return mu + ba[u] + bb[i] + np.einsum("nd,nd->n", Bm[i], A[u])

    monkeypatch.setattr(mod, "_predict_many", predict_many)
    G.test_svdpp_golden(golden, monkeypatch, "64")
    G.test_svdpp_fit_seeds_like_the_reference(golden)
    monkeypatch.setenv("DAISY_SVDPP_THREADS", "64")
    G.test_svdpp_against_c_oracle(5, 30, 20, 200, 1)
    G.test_svdpp_bad_item_raises_and_leaves_no_partial_state()
