"""ctypes binding of the C-ABI shared library (include/wekws_b200.h).

The library is built in-tree (``python -c 'import __graft_entry__ as g; g.build()'`` or
``make -C wekws_b200/csrc``).  There is NO fallback: if the library is missing or a call
fails, a RuntimeError carrying ``wekws_last_error()`` is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# WEKWS_B200_LIB: development override (A/B of two builds of the same ABI); the product default is the in-tree library
LIB_PATH = os.environ.get("WEKWS_B200_LIB") or os.path.join(_HERE, "libwekws_b200.so")

# enums (include/wekws_b200.h)
BACKBONE_MDTC, BACKBONE_TCN, BACKBONE_DSTCN, BACKBONE_GRU, BACKBONE_FSMN = 0, 1, 2, 3, 4
ACT_IDENTITY, ACT_SIGMOID = 0, 1
PCM_S16, PCM_F32 = 0, 1
FWD_SOFTMAX = 1
ABI_VERSION = 6
KWS_RESULT_FIELDS = 6


class FbankConfig(C.Structure):
    _fields_ = [("sample_rate", C.c_int32), ("frame_length", C.c_int32), ("frame_shift", C.c_int32),
                ("n_fft", C.c_int32), ("num_mel_bins", C.c_int32), ("preemphasis", C.c_float),
                ("remove_dc", C.c_int32), ("log_floor", C.c_float)]


class ModelConfig(C.Structure):
    _fields_ = [("backbone", C.c_int32), ("idim", C.c_int32), ("hdim", C.c_int32), ("odim", C.c_int32),
                ("num_layers", C.c_int32), ("num_stack", C.c_int32), ("stack_size", C.c_int32),
                ("kernel_size", C.c_int32), ("activation", C.c_int32), ("norm_var", C.c_int32),
                ("fsmn_input_affine_dim", C.c_int32), ("fsmn_linear_dim", C.c_int32), ("fsmn_proj_dim", C.c_int32),
                ("fsmn_left_order", C.c_int32), ("fsmn_right_order", C.c_int32),
                ("fsmn_output_affine_dim", C.c_int32)]


class KwsConfig(C.Structure):
    _fields_ = [("threshold", C.c_double), ("min_frames", C.c_int32), ("max_frames", C.c_int32),
                ("interval_frames", C.c_int32), ("score_beam", C.c_int32), ("path_beam", C.c_int32),
                ("frame_skip", C.c_int32)]


class CtcScoreConfig(C.Structure):
    _fields_ = [("threshold", C.c_double), ("min_frames", C.c_int32), ("max_frames", C.c_int32),
                ("score_beam", C.c_int32), ("path_beam", C.c_int32), ("frame_skip", C.c_int32),
                ("max_detections", C.c_int32)]


# name -> (restype, argtypes); every symbol include/wekws_b200.h declares
SIGNATURES = {
    "wekws_last_error": (C.c_char_p, []),
    "wekws_abi_version": (C.c_int, []),
    "wekws_launch_count": (C.c_uint64, []),
    "wekws_fbank_create": (C.c_int, [C.POINTER(FbankConfig), C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "wekws_fbank_destroy": (None, [C.c_void_p]),
    "wekws_fbank_num_frames": (C.c_int64, [C.c_void_p, C.c_int64]),
    "wekws_fbank_num_mel_bins": (C.c_int, [C.c_void_p]),
    "wekws_fbank_feature_dim": (C.c_int, [C.c_void_p]),
    "wekws_fbank_set_mfcc": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "wekws_fbank_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int64,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "wekws_model_create": (C.c_int, [C.POINTER(ModelConfig), C.POINTER(C.c_void_p)]),
    "wekws_model_destroy": (None, [C.c_void_p]),
    "wekws_model_padding": (C.c_int, [C.c_void_p]),
    "wekws_model_set_tensor": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64]),
    "wekws_model_pack": (C.c_int, [C.c_void_p]),
    "wekws_model_finalize": (C.c_int, [C.c_void_p]),
    "wekws_model_set_precision": (C.c_int, [C.c_void_p, C.c_int]),
    "wekws_model_uses_tensor_cores": (C.c_int, [C.c_void_p, C.c_int64]),
    "wekws_model_uses_tensor_cores_bt": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64]),
    "wekws_model_packed_floats": (C.c_int64, [C.c_void_p, C.c_int]),
    "wekws_model_packed_copy": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64]),
    "wekws_model_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_int64, C.c_int64, C.c_uint32, C.c_void_p]),
    "wekws_det_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                  C.c_void_p, C.c_void_p, C.c_void_p]),
    "wekws_ctc_state_bytes": (C.c_int64, []),
    "wekws_ctc_prefix_beam_search": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_int,
                                               C.c_int, C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                               C.c_void_p]),
    "wekws_ctc_keyword_hit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                                        C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p]),
    "wekws_context_expand_frames": (C.c_int64, [C.c_int64, C.c_int, C.c_int]),
    "wekws_context_expand": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_void_p, C.c_int64, C.c_void_p]),
    "wekws_kws_state_bytes": (C.c_int64, []),
    "wekws_kws_reset": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "wekws_kws_detect": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int,
                                   C.c_void_p, C.c_void_p, C.c_int, C.POINTER(KwsConfig), C.c_void_p, C.c_void_p,
                                   C.c_void_p]),
    "wekws_kws_splice": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]),
    "wekws_kws_context": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_int64, C.c_void_p, C.c_void_p]),
    "wekws_ctc_stream_score": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_int,
                                         C.c_void_p, C.c_void_p, C.c_int, C.POINTER(CtcScoreConfig), C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "wekws_ctc_det_sweep": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p,
                                      C.c_void_p, C.c_void_p]),
    "wekws_pipeline_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64,
                                         C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_uint32, C.c_void_p]),
}

_lib = None


def lib() -> C.CDLL:
    """Loads libwekws_b200.so once; raises if it is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"wekws_b200: native library {LIB_PATH} is not built. Run "
                "`python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc). "
                "There is no CPU or PyTorch fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)      # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        got = l.wekws_abi_version()
        if got != ABI_VERSION:
            raise RuntimeError(f"wekws_b200: ABI version mismatch (library {got}, binding {ABI_VERSION})")
        _lib = l
    return _lib


def last_error() -> str:
    return lib().wekws_last_error().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"wekws_b200: {what} failed (status {rc}): {last_error()}")


def launch_count() -> int:
    return int(lib().wekws_launch_count())
