"""CPU execution of csrc/ref_sort.cuh: the stable compaction + LSD radix sort whose element count stays on the device,
which the general BPR bookkeeping uses to sort the refs of repeated rows.

tests/emu/ref_sort_unit.cu includes the header and is compiled for the host against tests/emu/emu.h (the launch syntax
rewritten by build_emu.rewrite); the results must equal numpy's stable argsort of the kept elements.  Blocks run one
after the other in the emulation, so the decoupled look-back always finds its predecessor's prefix; the GPU tests
(tests/test_bpr_dup_sort_gpu.py) run the kernels concurrently.

Memcheck and race check, as for tests/test_kernel_emulation.py:
    DAISY_EMU_SANITIZE=1 LD_PRELOAD="$(gcc -print-file-name=libasan.so) $(gcc -print-file-name=libubsan.so)" \\
        ASAN_OPTIONS=detect_leaks=0 python -m pytest tests/test_ref_sort_emulation.py
    DAISY_EMU_SANITIZE=thread LD_PRELOAD="$(gcc -print-file-name=libtsan.so)" TSAN_OPTIONS=report_signal_unsafe=0 \\
        python -m pytest tests/test_ref_sort_emulation.py
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
import build_emu  # noqa: E402

TILE = 2048


def _build():
    src = os.path.join(build_emu.HERE, "ref_sort_unit.cu")
    mode = os.environ.get("DAISY_EMU_SANITIZE", "")
    os.makedirs(build_emu.OUT, exist_ok=True)
    so = os.path.join(build_emu.OUT, f"libref_sort_emu{'_' + mode if mode else ''}.so")
    deps = [src, os.path.join(build_emu.CSRC, "ref_sort.cuh"), os.path.join(build_emu.HERE, "emu.h"), build_emu.__file__, __file__]
    if os.path.exists(so) and all(os.path.getmtime(so) >= os.path.getmtime(d) for d in deps):
        return so
    cpp = os.path.join(build_emu.OUT, "ref_sort_emu.cpp")
    with open(cpp, "w") as f:
        f.write(open(src).read())
    with open(os.path.join(build_emu.CSRC, "ref_sort.cuh")) as f:   # the launches are in the header (dsort_launch)
        hdr = build_emu.rewrite(f.read())
    inc = os.path.join(build_emu.OUT, "ref_sort_inc")
    os.makedirs(inc, exist_ok=True)
    with open(os.path.join(inc, "ref_sort.cuh"), "w") as f:
        f.write(hdr)
    san = {"": [], "1": ["-fsanitize=address,undefined", "-fno-omit-frame-pointer", "-g"],
           "thread": ["-fsanitize=thread", "-fno-omit-frame-pointer", "-g"]}[mode]
    subprocess.check_call(["g++", "-std=c++20", "-O1", "-pthread", "-shared", "-fPIC", "-w", *san,
                           "-I", inc, "-I", build_emu.HERE, "-o", so, cpp])
    return so


@pytest.fixture(scope="module")
def lib():
    L = ctypes.CDLL(_build())
    p = ctypes.c_void_p
    L.rs_sort.argtypes = [p, p, ctypes.c_int, ctypes.c_uint32, ctypes.c_int, ctypes.c_int, p, p, p]
    return L


def _run(L, key, keep, split, bits, pass_blocks=0):
    key = np.ascontiguousarray(key, dtype=np.uint32)
    keep = np.ascontiguousarray(keep, dtype=np.uint8)
    n = len(key)
    ok = np.zeros(max(n, 1), np.uint32)
    ov = np.zeros(max(n, 1), np.uint32)
    cnt = np.zeros(2, np.uint32)
    launches = L.rs_sort(key.ctypes.data, keep.ctypes.data, n, split, bits, pass_blocks, ok.ctypes.data, ov.ctypes.data,
                         cnt.ctypes.data)
    idx = np.nonzero(keep)[0]
    order = idx[np.argsort(key[idx], kind="stable")]
    assert cnt[0] == len(idx)
    assert cnt[1] == int(np.count_nonzero(key[idx] < split))
    np.testing.assert_array_equal(ov[:len(idx)], order.astype(np.uint32))
    np.testing.assert_array_equal(ok[:len(idx)], key[order])
    return launches


def test_empty_input_launches_nothing(lib):
    assert _run(lib, np.zeros(0, np.uint32), np.zeros(0, np.uint8), 5, 24) == 0


def test_single_element(lib):
    assert _run(lib, [0xFFFFFF], [1], 1 << 23, 24) == 1 + 3
    _run(lib, [7], [0], 8, 24)   # dropped: nothing to sort


def test_partial_tiles_and_dropped_elements(lib):
    rng = np.random.default_rng(1)
    n = 2 * TILE + 777
    key = rng.integers(0, 1 << 24, n, dtype=np.uint32)
    key[::5] = key[0]   # repeated keys: their order must be kept
    keep = rng.random(n) < 0.6
    _run(lib, key, keep, 1 << 23, 24)


def test_all_keys_equal(lib):
    n = TILE + 300
    _run(lib, np.full(n, 0xABCDEF, np.uint32), np.ones(n, np.uint8), 0xABCDEF, 24)


def test_all_keys_distinct_descending_with_the_largest_24_bit_key(lib):
    n = 3 * TILE - 1
    key = (0xFFFFFF - np.arange(n) * 2731).astype(np.uint32)
    assert key.max() == 0xFFFFFF
    _run(lib, key, np.ones(n, np.uint8), 1 << 23, 24)


def test_fewer_blocks_than_tiles_and_other_pass_counts(lib):
    rng = np.random.default_rng(2)
    n = 3 * TILE + 5
    for bits in (5, 16, 32):
        key = rng.integers(0, 1 << bits, n, dtype=np.uint64).astype(np.uint32)
        keep = rng.random(n) < 0.9
        _run(lib, key, keep, 1 << (bits - 1), bits, pass_blocks=2)


def test_bpr_ref_layout(lib):
    """Keys as the BPR bookkeeping builds them: negatives, run heads (I = not a head, dropped), users at I + 1 + u;
    kept = the rows referenced at least twice in their table."""
    rng = np.random.default_rng(3)
    B, U, I = 1500, 900, 400
    u = rng.integers(0, U, B)
    i = np.sort(rng.integers(0, I, B))
    j = rng.integers(0, I, B)
    head = np.r_[True, i[1:] != i[:-1]]
    key = np.r_[j, np.where(head, i, I), I + 1 + u].astype(np.uint32)
    items = np.r_[j, i[head]]
    icnt = np.bincount(items, minlength=I)
    ucnt = np.bincount(u, minlength=U)
    keep = np.r_[icnt[j] > 1, head & (icnt[i] > 1), ucnt[u] > 1]
    _run(lib, key, keep, I, int(I + U).bit_length())
