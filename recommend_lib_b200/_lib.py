"""ctypes binding of libdaisy_b200.so (include/daisy_b200.h).  No fallback: a missing library raises."""
from __future__ import annotations

import ctypes
import os

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# DAISY_LIB_VARIANT=<name> loads libdaisy_b200_<name>.so, an experimental build made by build.py with DAISY_NVCC_EXTRA
_VARIANT = os.environ.get("DAISY_LIB_VARIANT", "")
LIB_PATH = os.path.join(_HERE, "libdaisy_b200" + ("_" + _VARIANT if _VARIANT else "") + ".so")

OK, EINVAL, ECUDA, EINDEX, EUNSUPPORTED, ENOMEM = 0, -1, -2, -3, -4, -5
FLAG_EAGER_DECAY = 1
TOPK_PATHS = ("exact", "filter-simt", "filter-tc")   # DAISY_TOPK_PATH_EXACT, _SIMT, _TC
NUM_PHASES = 11
PHASES = ("prep", "sort_i", "refs", "sort_u", "sort_q", "slots", "main", "seg_u", "seg_q", "heavy", "loss")

c_i32, c_i64, c_f32, c_f64, c_vp = ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_double, ctypes.c_void_p


class MFParams(ctypes.Structure):
    """daisy_mf_params"""
    _fields_ = [("variant", c_i32), ("biased", c_i32),
                ("lr_bu", c_f64), ("lr_bi", c_f64), ("lr_pu", c_f64), ("lr_qi", c_f64),
                ("reg_bu", c_f64), ("reg_bi", c_f64), ("reg_pu", c_f64), ("reg_qi", c_f64),
                ("reg2", c_f64), ("global_mean", c_f64)]


class SVDppParams(ctypes.Structure):
    """daisy_svdpp_params"""
    _fields_ = [("lr_bu", c_f64), ("lr_bi", c_f64), ("lr_pu", c_f64), ("lr_qi", c_f64), ("lr_yj", c_f64),
                ("reg_bu", c_f64), ("reg_bi", c_f64), ("reg_pu", c_f64), ("reg_qi", c_f64), ("reg_yj", c_f64),
                ("global_mean", c_f64)]


class FMBNParams(ctypes.Structure):
    """daisy_fmbn_params"""
    _fields_ = [("E", c_vp), ("bias", c_vp), ("accE", c_vp), ("accb", c_vp), ("gamma", c_vp), ("beta", c_vp),
                ("acc_gamma", c_vp), ("acc_beta", c_vp), ("running_mean", c_vp), ("running_var", c_vp),
                ("lr", c_f32), ("eps", c_f32), ("bn_eps", c_f32), ("momentum", c_f32),
                ("user_num", c_i64), ("num_features", c_i64), ("F", c_i32)]


class SGNSParams(ctypes.Structure):
    """daisy_sgns_params"""
    _fields_ = [("iv", c_vp), ("ov", c_vp), ("m_iv", c_vp), ("v_iv", c_vp), ("m_ov", c_vp), ("v_ov", c_vp),
                ("lr", c_f32), ("beta1", c_f32), ("beta2", c_f32), ("eps", c_f32),
                ("vocab", c_i64), ("D", c_i32), ("padding_idx", c_i32)]


NEUMF_MAX_LAYERS = 6
_vp6 = c_vp * NEUMF_MAX_LAYERS


class NeuMFParams(ctypes.Structure):
    """daisy_neumf_params"""
    _fields_ = [("neumf", c_i32), ("num_layers", c_i32), ("factor", c_i32), ("user_num", c_i64), ("item_num", c_i64),
                ("Pg", c_vp), ("Qg", c_vp), ("Pm", c_vp), ("Qm", c_vp), ("W", _vp6), ("b", _vp6), ("wp", c_vp), ("bp", c_vp),
                ("m_Pg", c_vp), ("v_Pg", c_vp), ("m_Qg", c_vp), ("v_Qg", c_vp), ("m_Pm", c_vp), ("v_Pm", c_vp),
                ("m_Qm", c_vp), ("v_Qm", c_vp), ("m_W", _vp6), ("v_W", _vp6), ("m_b", _vp6), ("v_b", _vp6),
                ("m_wp", c_vp), ("v_wp", c_vp), ("m_bp", c_vp), ("v_bp", c_vp),
                ("lr", c_f32), ("beta1", c_f32), ("beta2", c_f32), ("eps", c_f32)]


# name -> argtypes; every entry returns int except daisy_last_error.  Kept in one table so that the CPU test
# can check it against the prototypes of include/daisy_b200.h.
SIGNATURES = {
    "daisy_abi_version": [],
    "daisy_create": [ctypes.POINTER(c_vp), c_i32, c_i64, c_i64, c_i32, c_i64, ctypes.c_uint],
    "daisy_destroy": [c_vp],
    "daisy_check": [c_vp, c_vp],
    "daisy_get_scale": [c_vp, ctypes.POINTER(c_f64)],
    "daisy_set_scale": [c_vp, c_f64],
    "daisy_materialize": [c_vp, c_vp, c_vp, c_vp],
    "daisy_bpr_forward": [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp],
    "daisy_set_inputs_ready": [c_vp, c_i32],
    "daisy_bpr_step": [c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_f32, c_vp, c_vp],
    "daisy_bpr_step_host": [c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_f32, c_vp, c_vp],
    "daisy_bpr_epoch": [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i32, c_f32, c_f32, c_vp, c_vp],
    "daisy_bprfm_adagrad_step": [c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_f32, c_vp, c_vp],
    "daisy_gmf_forward": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp],
    "daisy_gmf_epoch": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i32, c_f32, c_f32,
                        c_f32, c_f32, c_i64, c_vp, c_vp],
    "daisy_gmf_step": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_f32, c_f32,
                       c_f32, c_i64, c_vp, c_vp],
    "daisy_bpr_shard_step": [c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_f32, c_f32, c_vp, c_vp, c_vp],
    "daisy_owner_apply": [c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_f32, c_vp],
    "daisy_shard_arena_size": [c_i32, c_i64, c_i32, c_i64, ctypes.POINTER(c_i64)],
    "daisy_shard_init": [c_vp, c_i32, c_i32, c_i64, c_vp],
    "daisy_shard_arena": [c_vp, ctypes.POINTER(c_vp), ctypes.POINTER(c_vp), ctypes.POINTER(c_i64)],
    "daisy_shard_ipc_handle": [c_vp, c_vp],
    "daisy_shard_attach": [c_vp, c_vp, c_vp, c_i32],
    "daisy_shard_step": [c_vp, c_vp, c_vp, c_i64, c_f32, c_f32, c_vp, c_vp],
    "daisy_shard_step_host": [c_vp, c_vp, c_vp, c_i64, c_f32, c_f32, c_vp, c_vp],
    "daisy_shard_compute": [c_vp, c_vp, c_vp, c_i64, c_f32, c_f32, c_vp, c_vp],
    "daisy_shard_prepare": [c_vp, c_vp, c_vp, c_i64, c_vp],
    "daisy_shard_classify": [c_vp, c_vp],
    "daisy_shard_barrier": [c_vp, c_vp],
    "daisy_shard_apply": [c_vp, c_f32, c_f32, c_vp],
    "daisy_shard_materialize": [c_vp, c_vp, c_vp],
    "daisy_shard_schedule": [c_i32, c_i32, c_i32, ctypes.POINTER(c_i32)],
    "daisy_shard_last_counts": [c_vp, c_vp, c_vp],
    "daisy_shard_peer_q": [c_vp, c_i32, ctypes.POINTER(c_vp)],
    "daisy_gather_rows": [c_vp, c_vp, c_vp, c_i64, c_vp, c_vp],
    "daisy_shard_phase_ms": [c_vp, ctypes.POINTER(c_f64), ctypes.POINTER(c_i64)],
    "daisy_bpr_adam_step": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_f64, c_f64, c_f32,
                            c_i64, c_vp, c_vp],
    "daisy_topk_candidates": [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp],
    "daisy_topk_full": [c_vp, c_vp, c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp],
    "daisy_topk_full_path": [c_vp, ctypes.POINTER(c_i32), ctypes.POINTER(c_i64), ctypes.POINTER(c_i64)],
    "daisy_sample_triples": [c_vp, c_vp, c_i64, c_i32, c_vp, c_i64, ctypes.c_uint64, ctypes.c_uint32, c_i32, c_vp, c_vp],
    "daisy_route_triples": [c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp],
    "daisy_mf_fit": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i32, ctypes.POINTER(MFParams),
                     c_vp, c_vp],
    "daisy_mf_predict": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i32, c_f64, c_vp, c_vp],
    "daisy_svdpp_fit": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp,
                        ctypes.POINTER(SVDppParams), c_vp, c_vp],
    "daisy_svdpp_user_factors": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp],
    "daisy_fmbn_scratch_bytes": [c_i64, c_i32, ctypes.POINTER(c_i64)],
    "daisy_fmbn_step": [c_vp, ctypes.POINTER(FMBNParams), c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp],
    "daisy_fmbn_forward": [c_vp, ctypes.POINTER(FMBNParams), c_vp, c_i64, c_vp, c_vp, c_vp],
    "daisy_fmbn_rank_tables": [c_vp, ctypes.POINTER(FMBNParams), c_i32, c_vp, c_vp, c_vp, c_vp],
    "daisy_sgns_scratch_bytes": [c_i64, c_i32, c_i32, c_i64, c_i32, ctypes.POINTER(c_i64)],
    "daisy_sgns_step": [c_vp, ctypes.POINTER(SGNSParams), c_vp, c_vp, c_vp, c_i64, c_i32, c_i32, c_i64, c_vp, c_i64, c_vp,
                        c_vp],
    "daisy_neumf_scratch_bytes": [ctypes.POINTER(NeuMFParams), c_i64, ctypes.POINTER(c_i64)],
    "daisy_neumf_forward": [c_vp, ctypes.POINTER(NeuMFParams), c_vp, c_i64, c_vp, c_vp],
    "daisy_neumf_step": [c_vp, ctypes.POINTER(NeuMFParams), c_vp, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp],
    "daisy_neumf_topk_candidates": [c_vp, ctypes.POINTER(NeuMFParams), c_vp, c_vp, c_i64, c_i32, c_i32, c_vp, c_vp, c_vp,
                                    c_vp],
    "daisy_neumf_topk_full": [c_vp, ctypes.POINTER(NeuMFParams), c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp],
    "daisy_launch_count": [c_vp, ctypes.POINTER(c_i64)],
    "daisy_set_timing": [c_vp, c_i32],
    "daisy_last_step_timing": [c_vp, ctypes.POINTER(c_f32), ctypes.POINTER(c_f32)],
    "daisy_main_kernel_ms": [c_vp, ctypes.POINTER(c_f64), ctypes.POINTER(c_i64)],
    "daisy_topk_tc_ms": [c_vp, ctypes.POINTER(c_f64), ctypes.POINTER(c_f64), ctypes.POINTER(c_i64)],
    "daisy_phase_ms": [c_vp, ctypes.POINTER(c_f64), c_i32, ctypes.POINTER(c_i64)],
    "daisy_set_l2_window": [c_vp, c_vp, c_i64, c_f32, c_vp],
    "daisy_trace": [c_vp, c_i32, ctypes.POINTER(c_f64), c_i32, ctypes.POINTER(c_i32)],
}

_lib = None


class DaisyError(RuntimeError):
    pass


def dlopen():
    """dlopen libdaisy_b200.so.  It links the shared CUDA runtime (libcudart.so.12): importing torch first makes
    the dynamic loader bind it to the runtime torch already mapped; otherwise the usual locations are tried."""
    if not os.path.exists(LIB_PATH):
        raise DaisyError(
            f"{LIB_PATH} is missing: build it with `python -m recommend_lib_b200.build` "
            "(or __graft_entry__.build()).  There is no CPU fallback.")
    try:
        import torch  # noqa: F401  (maps libcudart.so.12 from the nvidia-cuda-runtime wheel)
    except Exception:
        pass
    try:
        return ctypes.CDLL(LIB_PATH)
    except OSError:
        import glob
        import site
        cands = []
        for sp in site.getsitepackages():
            cands += glob.glob(os.path.join(sp, "nvidia", "cuda_runtime", "lib", "libcudart.so.12*"))
        cands += glob.glob("/usr/local/cuda/lib64/libcudart.so.12*")
        for c in cands:
            try:
                ctypes.CDLL(c, mode=ctypes.RTLD_GLOBAL)
                return ctypes.CDLL(LIB_PATH)
            except OSError:
                continue
        raise


def load():
    """Load the shared library (once).  Raises if it has not been built -- there is no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    L = dlopen()
    for name, argtypes in SIGNATURES.items():
        fn = getattr(L, name)          # AttributeError if the library does not export a declared symbol
        fn.argtypes = argtypes
        fn.restype = c_i32
    L.daisy_last_error.argtypes = []
    L.daisy_last_error.restype = ctypes.c_char_p
    if L.daisy_abi_version() != 1:
        raise DaisyError("libdaisy_b200.so ABI version mismatch")
    _lib = L
    return L


def last_error():
    return load().daisy_last_error().decode("utf-8", "replace")


def check(rc):
    """Map a DAISY_E* return code to the exception the reference surface would raise."""
    if rc == OK:
        return
    msg = last_error()
    if rc == EINDEX:
        raise IndexError(msg)
    if rc in (EINVAL, EUNSUPPORTED):
        raise ValueError(msg)
    if rc == ENOMEM:
        raise MemoryError(msg)
    raise DaisyError(msg)


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise DaisyError("recommend_lib_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch


def stream_ptr(torch, device):
    return c_vp(torch.cuda.current_stream(device).cuda_stream)


class Handle:
    """RAII wrapper of daisy_handle_t bound to (device, user_num, item_num, dim, max_batch)."""

    def __init__(self, device_index, user_num, item_num, dim, max_batch, flags=0):
        self.L = load()
        self.ptr = c_vp()
        check(self.L.daisy_create(ctypes.byref(self.ptr), int(device_index), int(user_num), int(item_num), int(dim),
                                  int(max_batch), int(flags)))
        self.device_index = int(device_index)
        self.user_num, self.item_num, self.dim, self.max_batch = int(user_num), int(item_num), int(dim), int(max_batch)

    def close(self):
        if getattr(self, "ptr", None) is not None and self.ptr.value:
            self.L.daisy_destroy(self.ptr)
            self.ptr = c_vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- small conveniences ------------------------------------------------------------------
    @property
    def scale(self):
        c = c_f64()
        check(self.L.daisy_get_scale(self.ptr, ctypes.byref(c)))
        return c.value

    @scale.setter
    def scale(self, v):
        check(self.L.daisy_set_scale(self.ptr, float(v)))

    @property
    def launches(self):
        n = c_i64()
        check(self.L.daisy_launch_count(self.ptr, ctypes.byref(n)))
        return n.value

    def set_inputs_ready(self, on):
        check(self.L.daisy_set_inputs_ready(self.ptr, int(bool(on))))

    def trace_start(self):
        check(self.L.daisy_trace(self.ptr, 1, None, 0, None))

    def trace_dump(self):
        """[(book_begin, book_end, kernels_begin, kernels_end)] in ms for the traced steps; stops tracing."""
        arr = (c_f64 * (4 * 48))()
        n = c_i32()
        check(self.L.daisy_trace(self.ptr, 0, arr, 4 * 48, ctypes.byref(n)))
        return [tuple(arr[4 * i:4 * i + 4]) for i in range(n.value)]

    def set_timing(self, mode):
        check(self.L.daisy_set_timing(self.ptr, int(mode)))

    def main_kernel_ms(self):
        avg, cnt = c_f64(), c_i64()
        check(self.L.daisy_main_kernel_ms(self.ptr, ctypes.byref(avg), ctypes.byref(cnt)))
        return avg.value, cnt.value

    def topk_tc_ms(self):
        """(filter kernel ms, rescore kernel ms, launches measured) of daisy_topk_full's tensor-core filter since the last call."""
        f, r, cnt = c_f64(), c_f64(), c_i64()
        check(self.L.daisy_topk_tc_ms(self.ptr, ctypes.byref(f), ctypes.byref(r), ctypes.byref(cnt)))
        return f.value, r.value, cnt.value

    def topk_full_path(self):
        """(path, filtered, redone) of the last daisy_topk_full call: path is one of TOPK_PATHS, filtered the users
        whose top K came from a candidate list, redone the users the exact path redid."""
        path, filtered, redone = c_i32(), c_i64(), c_i64()
        check(self.L.daisy_topk_full_path(self.ptr, ctypes.byref(path), ctypes.byref(filtered), ctypes.byref(redone)))
        return TOPK_PATHS[path.value], filtered.value, redone.value

    def phase_ms(self):
        arr = (c_f64 * NUM_PHASES)()
        steps = c_i64()
        check(self.L.daisy_phase_ms(self.ptr, arr, NUM_PHASES, ctypes.byref(steps)))
        return dict(zip(PHASES, list(arr))), steps.value


class HandleOwner:
    """A model (or optimiser) that owns one ``Handle``: the device check, the handle's lifecycle and, for the models that
    rank, the ranking calls of ``metrics.topk_candidates`` / ``topk_full``.

    A subclass names the weight it runs on (``_weight``, and ``_cpu_error`` for that weight on the CPU) and the handle's
    dims (``_handle_dims``).  With ``_batch_grows`` the handle holds a step workspace of ``_max_batch`` rows and is
    re-created for a larger batch; otherwise it is light (max_batch 0: device, error flag and launch counter).  Adds no
    parameter, buffer or submodule to an ``nn.Module``."""

    _handle = None
    _max_batch = 0
    _batch_grows = False
    _handle_flags = 0
    # metric_eval(algo='bpr') ranks as the reference's _bpr_topk, which scores with model(user, item_i, item_j)
    bpr_topk = True

    def _device(self):
        W = self._weight()
        if not W.is_cuda:
            require_cuda()
            raise DaisyError(self._cpu_error)
        return W.device

    def handle(self, batch=None):
        """The library handle for the weights' current device; re-created when the device changes or, for a handle with a
        step workspace, when a larger batch arrives."""
        dev = self._device()
        idx = dev.index if dev.index is not None else torch.cuda.current_device()
        need = max(self._max_batch, int(batch or 0)) if self._batch_grows else 0
        h = self._handle
        if h is None or h.device_index != idx or (need and h.max_batch < need):   # a light handle never grows
            self._close_handle()
            self._max_batch = need
            self._handle = h = Handle(idx, *self._handle_dims(), need, self._handle_flags)
        return h

    def _close_handle(self):
        if self._handle is not None:
            self._handle.close()
            self._handle = None

    def check(self):
        """Synchronise and raise IndexError if any id seen since the last check was out of range."""
        h = self._handle
        if h is not None:
            check(h.L.daisy_check(h.ptr, stream_ptr(torch, self._device())))

    def __getstate__(self):             # a handle does not pickle: the copy makes its own on first use
        d = self.__dict__.copy()
        d["_handle"] = None
        return d

    def _apply(self, fn, *a, **k):      # .cuda() / .cpu() / .to(): the weights move, the handle is rebuilt lazily
        self._close_handle()
        return super()._apply(fn, *a, **k)

    # -- ranking: a dot-product model's score is <P[u], Q[i]> (+ a term that is the same for every item of a user) ------
    def user_term(self, users, c0):
        """[N] the score's term that is the same for every item of a user, or None when the score is the dot product."""
        return None

    def rank_candidates(self, users, cands, top_k):
        """users [N], cands [N, C] int32 device tensors -> (pos, items, scores) [N, top_k]."""
        h = self.handle()
        P, Q, c0 = self.rank_tables()
        pos, items, scores = call_topk_candidates(h, P.data_ptr(), Q.data_ptr(), users, cands, top_k,
                                                  stream_ptr(torch, users.device))
        self.check()                    # before the term's gather: an out-of-range user id raises here
        off = self.user_term(users, c0)
        if off is not None:
            scores += off[:, None]
        return pos, items, scores

    def rank_full(self, users, k, excl):
        """users [N] int32 device tensor, excl the ``exclusion_csr`` pair -> (items, scores) [N, k]."""
        h = self.handle()
        P, Q, c0 = self.rank_tables()
        items, scores = call_topk_full(h, P.data_ptr(), Q.data_ptr(), users, k, excl, stream_ptr(torch, users.device))
        self.check()
        off = self.user_term(users, c0)
        if off is not None:
            scores += off[:, None]
        return items, scores


def call_topk_candidates(h, P, Q, users, cands, top_k, stream):
    """``daisy_topk_candidates`` over the tables at device addresses P, Q: users [N], cands [N, C] int32 device tensors
    -> (pos, items, scores) [N, top_k] on the users' device."""
    N, C = cands.shape
    pos = torch.empty((N, top_k), dtype=torch.int32, device=users.device)
    items = torch.empty((N, top_k), dtype=torch.int32, device=users.device)
    scores = torch.empty((N, top_k), dtype=torch.float32, device=users.device)
    check(h.L.daisy_topk_candidates(h.ptr, c_vp(P), c_vp(Q), c_vp(users.data_ptr()), c_vp(cands.data_ptr()), N, C,
                                    int(top_k), c_vp(pos.data_ptr()), c_vp(items.data_ptr()), c_vp(scores.data_ptr()),
                                    stream))
    return pos, items, scores


def call_topk_full(h, P, Q, users, k, excl, stream):
    """``daisy_topk_full`` over the tables at device addresses P, Q: users [N] int32 device tensor, excl the
    ``exclusion_csr`` pair -> (items, scores) [N, k] on the users' device."""
    N = users.shape[0]
    ptr, idx = excl
    items = torch.empty((N, k), dtype=torch.int32, device=users.device)
    scores = torch.empty((N, k), dtype=torch.float32, device=users.device)
    check(h.L.daisy_topk_full(h.ptr, c_vp(P), c_vp(Q), c_vp(users.data_ptr()), N, int(k),
                              c_vp(ptr.data_ptr()) if ptr is not None else None,
                              c_vp(idx.data_ptr()) if idx is not None and idx.numel() else None,
                              c_vp(items.data_ptr()), c_vp(scores.data_ptr()), stream))
    return items, scores


def exclusion_csr(exclude, n, device, window=None):
    """(ptr [n + 1] int64, idx int32) on ``device``: the n per-user lists of item ids ``exclude`` as CSR, or (None, None)
    without lists.  ``window=(i0, i1)`` keeps the ids in [i0, i1), made relative to i0 (one shard of the item table)."""
    if exclude is None:
        return None, None
    if window is None:
        ex = [np.asarray(e, dtype=np.int32) for e in exclude]
    else:
        i0, i1 = window
        ex = [np.asarray(e, dtype=np.int64) for e in exclude]
        ex = [(e[(e >= i0) & (e < i1)] - i0).astype(np.int32) for e in ex]
    ptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.fromiter((len(e) for e in ex), dtype=np.int64, count=n), out=ptr[1:])
    idx = np.concatenate(ex) if ptr[-1] else np.zeros(0, np.int32)
    return torch.from_numpy(ptr).to(device), torch.from_numpy(idx).to(device)
