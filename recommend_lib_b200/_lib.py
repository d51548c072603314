"""ctypes binding of libdaisy_b200.so (include/daisy_b200.h).  No fallback: a missing library raises."""
from __future__ import annotations

import ctypes
import os

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
