"""ctypes binding of ``libmms_b200.so`` (C ABI declared in ``include/mms_b200.h``).

There is no CPU fallback anywhere in this package: if the shared library is
missing, or the device is not a B200 (sm_100), every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import torch

_PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("MMS_B200_LIB", _PKG / "libmms_b200.so"))

c_f32p = C.c_void_p      # device pointers travel as integers
c_i64 = C.c_int64
c_i32 = C.c_int32
c_u64 = C.c_uint64
c_f32 = C.c_float

MAX_SEGMENTS = 64
MAX_ADAM_RANGES = 96
GRAD_CLIP_SCRATCH_BYTES = 1040


class MmsError(RuntimeError):
    pass


class CnnGruDesc(C.Structure):
    _fields_ = [
        ("batch", c_i32), ("in_channels", c_i32), ("seq_len", c_i32), ("num_classes", c_i32),
        ("cnn_out", c_i32), ("hidden", c_i32), ("layers", c_i32), ("training", c_i32),
        ("attention", c_i32), ("need_grad", c_i32), ("dropout_p", c_f32),
        ("rng_seed", c_u64), ("rng_offset", c_u64), ("rng_offset_dev", C.c_void_p),
        ("global_batch", c_i32), ("class_weight", C.c_void_p),
        ("frozen_segments", c_u64), ("adam_ranges_host", C.c_void_p), ("adam_steps", C.c_void_p), ("adam_nranges", c_i32),
        ("clip_max_norm", C.c_void_p), ("clip_record", C.c_void_p), ("clip_scratch", C.c_void_p),
    ]


class GruDirFwd(C.Structure):
    _fields_ = [
        ("gi", C.c_void_p), ("gi_bs", c_i64), ("gi_ts", c_i64),
        ("w_hh", C.c_void_p), ("b_hh", C.c_void_p),
        ("hs", C.c_void_p), ("hs_bs", c_i64), ("hs_ts", c_i64),
        ("hs_drop", C.c_void_p), ("drop_base", c_i64),
        ("stash", C.c_void_p), ("st_bs", c_i64), ("st_ts", c_i64),
        ("t0", c_i32), ("dt", c_i32), ("nsteps", c_i32),
    ]


class GruDirBwd(C.Structure):
    _fields_ = [
        ("w_hh", C.c_void_p),
        ("stash", C.c_void_p), ("st_bs", c_i64), ("st_ts", c_i64),
        ("hs", C.c_void_p), ("hs_bs", c_i64), ("hs_ts", c_i64),
        ("dout", C.c_void_p), ("do_bs", c_i64), ("do_ts", c_i64), ("drop_base", c_i64), ("drop_mask", c_i32),
        ("dout_last", C.c_void_p), ("dl_ld", c_i64), ("dl_at_first", c_i32),
        ("dh_head", C.c_void_p), ("w0", C.c_void_p), ("w0_ld", c_i64), ("w0_col", c_i32),
        ("D", C.c_void_p), ("d_bs", c_i64), ("d_ts", c_i64),
        ("t0", c_i32), ("dt", c_i32), ("nsteps", c_i32),
    ]


class TnCall(C.Structure):
    """mms_tn_call (include/mms_b200.h): one weight-gradient product of the batched tensor-core kernel."""
    _fields_ = [
        ("A", C.c_void_p), ("lda", c_i64), ("a_split", c_i32), ("a_skip", c_i32),
        ("Bm", C.c_void_p), ("ldb", c_i64), ("shift", c_i32), ("seq", c_i32),
        ("C", C.c_void_p), ("ldc", c_i64), ("bias_grad", C.c_void_p),
        ("M", c_i32), ("N1", c_i32), ("N2", c_i32),
    ]


P = C.c_void_p
_SIGNATURES = {
    "mms_version": (c_i32, []),
    "mms_last_error": (C.c_char_p, []),
    "mms_init": (c_i32, [c_i32]),
    "mms_launch_count": (c_i64, []),
    "mms_profile_enable": (c_i32, [c_i32]),
    "mms_profile_report": (c_i32, [C.c_char_p, c_i64]),
    "mms_timeline_enable": (c_i32, [c_i32]),
    "mms_timeline_report": (c_i32, [C.c_char_p, c_i64]),
    "mms_set_side_streams": (c_i32, [c_i32]),
    "mms_set_option": (c_i32, [C.c_char_p, c_i32]),
    "mms_get_option": (c_i32, [C.c_char_p, c_i32]),
    "mms_clear_option": (c_i32, [C.c_char_p]),
    "mms_cnngru_param_layout": (c_i32, [C.POINTER(CnnGruDesc), C.POINTER(c_i64), C.POINTER(c_i64), c_i32, C.POINTER(c_i64)]),
    "mms_cnngru_workspace_bytes": (c_i64, [C.POINTER(CnnGruDesc)]),
    "mms_cnngru_forward": (c_i32, [C.POINTER(CnnGruDesc), P, P, P, P, P, P, P]),
    "mms_cnngru_backward": (c_i32, [C.POINTER(CnnGruDesc), P, P, P, P, P, P, P, P]),
    "mms_cnngru_input_gradient": (c_i32, [C.POINTER(CnnGruDesc), P, P, P, P, P, P, P]),
    "mms_cnngru_mc_workspace_bytes": (c_i64, [C.POINTER(CnnGruDesc), c_i32]),
    "mms_cnngru_mc_forward": (c_i32, [C.POINTER(CnnGruDesc), P, P, P, P, c_i32, c_i64, P, P]),
    "mms_mc_accumulate": (c_i32, [P, c_i32, c_i32, c_i32, c_i64, c_i32, P, P, P, P, P, P]),
    "mms_ig_interpolate": (c_i32, [P, P, c_i32, P, c_i32, c_i32, c_i32, c_i32, c_i32, c_i64, c_i32, P, P, P]),
    "mms_ig_accumulate": (c_i32, [P, P, c_i32, P, c_i32, c_i32, c_i32, c_i32, c_i64, c_i32, P, P, P]),
    "mms_cross_entropy": (c_i32, [P, P, c_i32, c_i32, P, P, P, P]),
    "mms_cross_entropy_partial": (c_i32, [P, P, c_i32, c_i32, c_i32, P, P, P, P]),
    "mms_cross_entropy_weighted": (c_i32, [P, P, c_i32, c_i32, P, P, P, P, P, P]),
    "mms_class_weight_sum": (c_i32, [P, c_i32, c_i32, P, P, P]),
    "mms_cnngru_forward_phase": (c_i32, [C.POINTER(CnnGruDesc), c_i32, P, P, P, P, P, P, P]),
    "mms_cnngru_backward_phase": (c_i32, [C.POINTER(CnnGruDesc), c_i32, P, P, P, P, P, P, P]),
    "mms_cnngru_sync_offsets": (c_i32, [C.POINTER(CnnGruDesc), C.POINTER(c_i64), C.POINTER(c_i64)]),
    "mms_peer_allreduce_f64": (c_i32, [P, P, c_i32, c_i32, c_i32, c_i32, P, P]),
    "mms_peer_status": (c_i32, [P]),
    "mms_peer_allreduce_adam": (c_i32, [P, P, P, c_i32, c_i32, c_i32, P, P, c_i64, P, c_f32, c_f32, c_f32, c_f32, P, P, P, P]),
    "mms_peer_allreduce_adam_ranges": (c_i32, [P, P, P, c_i32, c_i32, c_i32, P, P, P, c_i32, P, P, c_f32, c_f32, c_f32, c_f32, P, P,
                                               P, P]),
    "mms_adam_flat_step": (c_i32, [P, P, P, P, c_i64, P, c_f32, c_f32, c_f32, c_f32, P, P, P]),
    "mms_adam_ranges_step": (c_i32, [P, P, P, P, P, c_i32, P, P, c_f32, c_f32, c_f32, c_f32, P, P, P]),
    "mms_grad_norm": (c_i32, [P, c_i64, P, c_i32, P, P, P, P]),
    "mms_adam_flat_clip_step": (c_i32, [P, P, P, P, c_i64, P, c_f32, c_f32, c_f32, c_f32, P, P, P, P]),
    "mms_adam_ranges_clip_step": (c_i32, [P, P, P, P, P, c_i32, P, P, c_f32, c_f32, c_f32, c_f32, P, P, P, P]),
    "mms_peer_grad_norm": (c_i32, [P, P, c_i32, c_i32, c_i32, c_i64, P, c_i32, P, P, P, P, P]),
    "mms_peer_allreduce_adam_clip": (c_i32, [P, P, P, c_i32, c_i32, c_i32, P, P, c_i64, P, c_f32, c_f32, c_f32, c_f32, P, P, P, P, P]),
    "mms_peer_allreduce_adam_ranges_clip": (c_i32, [P, P, P, c_i32, c_i32, c_i32, P, P, P, c_i32, P, P, c_f32, c_f32, c_f32, c_f32,
                                                    P, P, P, P, P]),
    "mms_cnngru_train_step": (c_i32, [C.POINTER(CnnGruDesc), P, P, P, P, P, P, P, P, P, P, P, P, P,
                                      c_f32, c_f32, c_f32, c_f32, P, P, P]),
    "mms_batch_gather": (c_i32, [P, P, P, P, c_i64, c_i64, c_i32, P, P, c_i32, P, P]),
    "mms_eval_accumulate": (c_i32, [P, P, c_i32, c_i32, P, P, P, P]),
    "mms_eval_accumulate_weighted": (c_i32, [P, P, c_i32, c_i32, P, c_i32, P, P, P, P]),
    "mms_chan_attn_fwd": (c_i32, [P, P, P, c_i32, c_i32, c_i32, P, P, P, P]),
    "mms_chan_attn_bwd": (c_i32, [P, P, P, P, P, P, c_i32, c_i32, c_i32, P, P, P, P, P]),
    "mms_conv1d_fwd": (c_i32, [c_i32, P, P, P, c_i32, c_i32, c_i32, c_i32, P, P, P]),
    "mms_conv1d_fwd_tc": (c_i32, [c_i32, P, P, P, c_i32, c_i32, c_i32, c_i32, P, P, P]),
    "mms_conv1d_dgrad": (c_i32, [c_i32, P, P, c_i32, c_i32, c_i32, c_i32, P, P, P, P]),
    "mms_conv1d_wgrad": (c_i32, [c_i32, P, P, P, c_i32, c_i32, c_i32, c_i32, P, P]),
    "mms_bn_relu_pool_fwd": (c_i32, [P, P, P, P, P, P, P, c_i32, c_i32, c_i32, c_i32, c_i32, P, P]),
    "mms_bn_relu_pool_bwd": (c_i32, [P, P, P, P, P, P, P, c_i32, c_i32, c_i32, c_i32, c_i32, P, P, P, P, P]),
    "mms_tc_gemm_nt": (c_i32, [P, c_i64, P, c_i64, P, P, c_i64, c_i32, c_i32, c_i32, c_i32, P]),
    "mms_tc_gemm_tn_batch": (c_i32, [C.POINTER(TnCall), c_i32, P]),
    "mms_tc_gemm_tn": (c_i32, [P, c_i64, c_i32, c_i32, P, c_i64, c_i32, c_i32, P, c_i64, P, c_i32, c_i32, c_i32, P]),
    "mms_gemm_nt_bias": (c_i32, [P, c_i64, P, c_i64, P, P, c_i64, c_i32, c_i32, c_i32, P]),
    "mms_gemm_skinny": (c_i32, [P, c_i64, P, c_i64, c_i32, P, P, c_i64, c_i32, c_i32, c_i32, c_i32, c_i64, c_i64, c_f32, c_u64, c_u64, P, P]),
    "mms_gemm_nn": (c_i32, [P, c_i64, P, c_i64, P, c_i64, c_i32, c_i32, c_i32, c_i32, P]),
    "mms_gemm_tn_acc": (c_i32, [P, c_i64, c_i32, c_i32, P, c_i64, c_i32, c_i32, P, c_i64, P, c_i32, c_i32, c_i32, P]),
    "mms_dropout_apply": (c_i32, [P, P, c_i64, c_i64, c_f32, c_u64, c_u64, P, P]),
    "mms_gru_recur_fwd": (c_i32, [C.POINTER(GruDirFwd), c_i32, c_i32, c_i32, c_f32, c_u64, c_u64, P, P]),
    "mms_gru_recur_bwd": (c_i32, [C.POINTER(GruDirBwd), c_i32, c_i32, c_i32, c_f32, c_u64, c_u64, P, P]),
    "mms_head_fwd": (c_i32, [P, P, P, P, P, c_i32, c_i32, c_i32, c_f32, c_u64, c_u64, P, P, P, P]),
    "mms_head_bwd": (c_i32, [P, P, P, P, c_i32, c_i32, c_i32, c_f32, c_u64, c_u64, P, P, P, P, P, P, P]),
    "mms_resample_workspace_bytes": (c_i64, [c_i64, c_i64, c_i32]),
    "mms_resample_f64": (c_i32, [P, c_i64, c_i64, c_i32, P, P, c_i64, P]),
    "mms_window_gather": (c_i32, [P, c_i32, c_i64, P, c_i32, c_i32, c_i32, P, P, P, P, P]),
    "mms_window_stats": (c_i32, [P, c_i32, c_i64, P, c_i32, c_i32, P, P, P]),
}

# every symbol include/mms_b200.h declares (checked by tests/test_abi.py)
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None
_initialised_devices = set()


def load_library() -> C.CDLL:
    """dlopen the shared library (no CUDA call is made) and type every symbol."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise MmsError(
            f"{LIB_PATH} is missing: build it with `python -m multimodalsignal_b200.build` "
            "(nvcc, sm_100a). This package has no CPU or PyTorch fallback.")
    lib = C.CDLL(str(LIB_PATH))
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def lib() -> C.CDLL:
    """The library, initialised for the current CUDA device (raises without a B200)."""
    l = load_library()
    if not torch.cuda.is_available():
        raise MmsError("multimodalsignal_b200 needs a CUDA device (B200, sm_100); there is no CPU fallback")
    dev = torch.cuda.current_device()
    if dev not in _initialised_devices:
        torch.cuda.init()
        check(l.mms_init(dev))
        _initialised_devices.add(dev)
    return l


def check(rc: int) -> int:
    if rc < 0:
        msg = load_library().mms_last_error()
        raise MmsError(f"libmms_b200 error {rc}: {msg.decode() if msg else '?'}")
    return rc


def ptr(t) -> int | None:
    """Device pointer of a tensor (None -> NULL).  The tensor must be contiguous."""
    if t is None:
        return None
    if not t.is_cuda:
        raise MmsError("expected a CUDA tensor (no CPU fallback)")
    if not t.is_contiguous():
        raise MmsError("expected a contiguous tensor")
    return t.data_ptr()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream
