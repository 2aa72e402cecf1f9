"""ctypes binding of libctdd_b200.so (include/ctdd.h). There is no CPU or PyTorch fallback: if the library
is missing or a call fails, a RuntimeError is raised."""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int32, c_int64, c_longlong, c_uint64, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libctdd_b200.so")

# enums of include/ctdd.h
BRANCH_TAULDR, BRANCH_SDDM_DIRECT, BRANCH_SDDM_REVERSE_PROB, BRANCH_SDDM_REVERSE_LOGSCALE = 0, 1, 2, 3
MODE_TAU_LEAP, MODE_TAU_LEAP_CORR, MODE_MIDPOINT_DRIFT, MODE_MIDPOINT_JUMP, MODE_EULER, MODE_EULER_CORR, MODE_RATES_ONLY, MODE_EXACT = range(8)
IMPL_AUTO, IMPL_SIMT, IMPL_TC = 0, 1, 2
HEAD_LOGITS, HEAD_LOGISTIC, HEAD_LOGISTIC_FIX = 0, 1, 2
DTYPE_F32, DTYPE_BF16 = 0, 1
STAT_CHANGED_BASE, STAT_NONZERO_JUMP, STAT_CHANGED_EVAL, STAT_ROWS_JUMPED, STAT_ROWS_MULTI = 0, 1, 2, 3, 4
STAT_COUNT = 8
LOSS_CTELBO, LOSS_CRM, LOSS_SDDM = 0, 1, 2

TAULDR_LOSSES = ("CTElbo", "NLL", "CTElboLambda")
_LOGIT_BRANCH = {"direct": BRANCH_SDDM_DIRECT, "reverse_prob": BRANCH_SDDM_REVERSE_PROB,
                 "reverse_logscale": BRANCH_SDDM_REVERSE_LOGSCALE}


def branch_for(loss_name: str, logit_type) -> int:
    """lib/sampling/sampling.py:32,61 — tauLDR math for CTElbo/NLL/CTElboLambda, SDDM math for everything else."""
    if loss_name in TAULDR_LOSSES:
        return BRANCH_TAULDR
    if logit_type not in _LOGIT_BRANCH:
        raise ValueError("Unknown logit_type: %s" % logit_type)
    return _LOGIT_BRANCH[logit_type]


class StepParams(ctypes.Structure):
    _fields_ = [
        ("mode", c_int32), ("branch", c_int32), ("impl", c_int32),
        ("N", c_int32), ("D", c_int32), ("S", c_int32),
        ("row_offset", c_int64),
        ("logits", c_void_p), ("ld_logits", c_int64), ("batch_stride_logits", c_int64),
        ("x_eval", c_void_p), ("x_base", c_void_p),
        ("Q", c_void_p), ("QT", c_void_p), ("Rb", c_void_p), ("RbT", c_void_p),
        ("tc_tables", c_void_p), ("tc_static", c_void_p),
        ("beta", c_float), ("h", c_float), ("eps", c_float),
        ("reject_multi", c_int32),
        ("seed", c_uint64), ("offset", c_uint64),
        ("x_out", c_void_p), ("rr_out", c_void_p), ("ratio_out", c_void_p),
        ("stats_out", c_void_p), ("workspace", c_void_p),
        ("head", c_int32), ("head_mu", c_void_p), ("head_log_scale", c_void_p), ("head_batch_stride", c_int64),
        ("logits_dtype", c_int32), ("head_dtype", c_int32),
    ]


def logits_dtype_of(t) -> int:
    """ctdd_step_params.logits_dtype / ctdd_loss_params.logits_dtype of a logits tensor the kernels read as they are
    (fp32, bf16)."""
    return DTYPE_BF16 if t.dtype == torch.bfloat16 else DTYPE_F32


class LossParams(ctypes.Structure):
    _fields_ = [
        ("kind", c_int32), ("logit_type", c_int32), ("crm_type", c_int32),
        ("B", c_int32), ("D", c_int32), ("S", c_int32),
        ("logits", c_void_p), ("Q", c_void_p), ("QT", c_void_p), ("Rb", c_void_p), ("beta", c_void_p),
        ("x0", c_void_p), ("xt", c_void_p), ("x_tilde", c_void_p),
        ("eps", c_float),
        ("out_a", c_void_p), ("out_b", c_void_p), ("out_c", c_void_p), ("out_d", c_void_p), ("out_nll", c_void_p),
        ("ga", c_void_p), ("gb", c_void_p), ("gd", c_void_p), ("gn", c_void_p),
        ("grad_logits", c_void_p), ("workspace", c_void_p), ("tc_scratch", c_void_p),
        ("logits_dtype", c_int32),
    ]


_lib = None


def lib() -> ctypes.CDLL:
    """Load libctdd_b200.so; fail loudly when it has not been built (python __graft_entry__.py build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA extension is not built. Run `python -c 'import __graft_entry__ as g; "
            "g.build()'` (needs nvcc). There is no CPU fallback for the ctdd_b200 hot path.")
    L = ctypes.CDLL(LIB_PATH)
    L.ctdd_version.restype = c_int
    L.ctdd_last_error.restype = c_char_p
    L.ctdd_launch_count.restype = c_longlong
    L.ctdd_build_qt0.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p]
    L.ctdd_build_rate.argtypes = [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]
    L.ctdd_step_workspace_bytes.argtypes = [c_int64, c_int, c_int]
    L.ctdd_step_workspace_bytes.restype = c_int64
    L.ctdd_reverse_step.argtypes = [ctypes.POINTER(StepParams), c_void_p]
    L.ctdd_tc_tables_bytes.argtypes = [c_int]
    L.ctdd_tc_tables_bytes.restype = c_int64
    L.ctdd_tc_static_bytes.argtypes = [c_int]
    L.ctdd_tc_static_bytes.restype = c_int64
    L.ctdd_tc_static_align.argtypes = []
    L.ctdd_tc_static_align.restype = c_int64
    L.ctdd_prep_tc_static.argtypes = [c_void_p, c_int, c_void_p, c_void_p]
    L.ctdd_prep_tc_static.restype = c_int
    L.ctdd_prep_tc_tables.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_int, c_void_p, c_void_p]
    L.ctdd_sample_categorical_shared.argtypes = [c_void_p, c_int, c_int64, c_int64, c_uint64, c_uint64, c_void_p, c_void_p]
    L.ctdd_noise_xt.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_uint64, c_uint64, c_void_p, c_void_p, c_void_p]
    L.ctdd_logistic_logits.argtypes = [c_void_p, c_void_p, c_int, c_int, c_int64, c_int, c_int, c_void_p, c_void_p]
    L.ctdd_logistic_logits.restype = c_int
    L.ctdd_logistic_logits_backward.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_int, c_int, c_void_p,
                                                c_void_p, c_void_p]
    L.ctdd_logistic_logits_backward.restype = c_int
    L.ctdd_logistic_logits_ex.argtypes = [c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_int, c_int, c_void_p, c_int,
                                          c_void_p]
    L.ctdd_logistic_logits_ex.restype = c_int
    L.ctdd_logistic_logits_backward_ex.argtypes = [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int64, c_int,
                                                   c_int, c_void_p, c_void_p, c_void_p]
    L.ctdd_logistic_logits_backward_ex.restype = c_int
    L.ctdd_pair_partials.argtypes = [c_int, c_int]
    L.ctdd_pair_partials.restype = c_int64
    L.ctdd_pair_similarity.argtypes = [c_void_p, c_int, c_void_p, c_int, c_int, c_float, c_int, c_void_p, c_void_p]
    L.ctdd_pair_similarity.restype = c_int
    L.ctdd_pair_similarity_sum.argtypes = [c_void_p, c_int, c_void_p, c_int, c_int, c_float, c_int, c_int, c_void_p, c_void_p, c_void_p]
    L.ctdd_pair_similarity_sum.restype = c_int
    L.ctdd_state_histogram.argtypes = [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p]
    L.ctdd_state_histogram.restype = c_int
    L.ctdd_ema_chunk_elems.restype = c_int64
    L.ctdd_ema_update.argtypes = [c_void_p, c_int, c_float, c_void_p]
    L.ctdd_ema_update.restype = c_int
    L.ctdd_loss_workspace_bytes.argtypes = [c_int, c_int, c_int]
    L.ctdd_loss_workspace_bytes.restype = c_int64
    L.ctdd_loss_forward.argtypes = [ctypes.POINTER(LossParams), c_void_p]
    L.ctdd_loss_backward.argtypes = [ctypes.POINTER(LossParams), c_void_p]
    L.ctdd_loss_tc_scratch_bytes.argtypes = [c_int, c_int, c_int]
    L.ctdd_loss_tc_scratch_bytes.restype = c_int64
    L.ctdd_bgemm256_tc.argtypes = [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]
    L.ctdd_bgemm256_tc.restype = c_int
    for name in ("ctdd_build_qt0", "ctdd_build_rate", "ctdd_reverse_step", "ctdd_prep_tc_tables",
                 "ctdd_sample_categorical_shared", "ctdd_noise_xt", "ctdd_loss_forward", "ctdd_loss_backward"):
        getattr(L, name).restype = c_int
    if L.ctdd_version() != 1:
        raise RuntimeError(f"libctdd_b200.so ABI version {L.ctdd_version()} != 1; rebuild")
    _lib = L
    return L


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise RuntimeError(f"libctdd_b200 {what} failed (rc={rc}): {lib().ctdd_last_error().decode()}")


def ptr(t) -> int:
    """Device pointer of a CUDA tensor (None -> NULL). Refuses host tensors: no CPU path exists."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("ctdd_b200 kernels need CUDA tensors; got a host tensor (there is no CPU fallback)")
    if not t.is_contiguous():
        raise RuntimeError("ctdd_b200 kernels need contiguous tensors")
    if t.device.index != torch.cuda.current_device():
        raise RuntimeError(f"ctdd_b200: tensor on {t.device} but the current CUDA device is cuda:{torch.cuda.current_device()}; "
                           "the kernels launch on the current device's stream (wrap the call in torch.cuda.device(...))")
    return t.data_ptr()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _first_cuda_tensor(objs):
    for o in objs:
        if isinstance(o, torch.Tensor):
            if o.is_cuda:
                return o
        elif isinstance(o, (list, tuple)):
            t = _first_cuda_tensor(o)
            if t is not None:
                return t
        elif hasattr(o, "mu") and isinstance(getattr(o, "mu"), torch.Tensor) and o.mu.is_cuda:   # ops.LogisticHead
            return o.mu
    return None


def on_tensor_device(fn):
    """Run `fn` with the CUDA device of its first CUDA tensor argument current: the library launches on the current
    device's stream and keeps per-device state (cudaGetDevice), so a tensor on cuda:1 while cuda:0 is current would
    otherwise be an illegal access.  ptr() refuses such a mismatch outright."""
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kw):
        t = _first_cuda_tensor(args)
        if t is None:
            t = _first_cuda_tensor(tuple(kw.values()))
        if t is None or t.device.index == torch.cuda.current_device():
            return fn(*args, **kw)
        with torch.cuda.device(t.device):
            return fn(*args, **kw)
    return wrapper


def on_device(device):
    """Context manager: make `device` (a torch.device / str / model.device) current if it is a CUDA device."""
    import contextlib
    dev = torch.device(device) if device is not None else None
    if dev is None or dev.type != "cuda":
        return contextlib.nullcontext()
    return torch.cuda.device(dev)


def launch_count() -> int:
    return int(lib().ctdd_launch_count())
