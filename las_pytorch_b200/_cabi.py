"""ctypes binding of include/las_b200.h (the C-ABI shared library `liblas_b200.so`).

This is the whole "custom-op layer": Python hands raw device pointers (`tensor.data_ptr()`), sizes and the
current CUDA stream handle to `extern "C"` functions.  There is no CPU fallback: if the library is missing or the
device is not sm_100 the call raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblas_b200.so")

ABI_VERSION = 7
MODE_FP32 = 0
MODE_BF16 = 1
MODE_F16 = 2
DECODE_RAW = 0
DECODE_GREEDY = 1
DECODE_SAMPLE = 2
CELL_LSTM, CELL_GRU, CELL_RNN = 0, 1, 2
CELLS = {"LSTM": CELL_LSTM, "GRU": CELL_GRU, "RNN": CELL_RNN}


class ListenerDims(C.Structure):
    _fields_ = [("B", C.c_int32), ("T", C.c_int32), ("F", C.c_int32), ("H", C.c_int32), ("L", C.c_int32), ("cell", C.c_int32)]


class LstmWeights(C.Structure):
    _fields_ = [("w_ih", C.c_void_p), ("w_hh", C.c_void_p), ("b_ih", C.c_void_p), ("b_hh", C.c_void_p)]


class SpellerDims(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("U", C.c_int32), ("E", C.c_int32), ("Hs", C.c_int32),
        ("sl", C.c_int32), ("V", C.c_int32), ("D", C.c_int32), ("heads", C.c_int32), ("no_mlp", C.c_int32), ("cell", C.c_int32),
    ]


class SpellerWeights(C.Structure):
    _fields_ = [
        ("rnn_host", C.POINTER(LstmWeights)),
        ("w_phi", C.c_void_p), ("b_phi", C.c_void_p),
        ("w_psi", C.c_void_p), ("b_psi", C.c_void_p),
        ("w_cd", C.c_void_p), ("b_cd", C.c_void_p),
        ("w_dr", C.c_void_p), ("b_dr", C.c_void_p),
    ]


class DecodeIO(C.Structure):
    _fields_ = [
        ("enc", C.c_void_p), ("psi", C.c_void_p),
        ("gt_dense", C.c_void_p), ("gt_index", C.c_void_p), ("gt_steps", C.c_int32),
        ("enc_lengths", C.c_void_p), ("sample_seed", C.c_uint64),
        ("h_state", C.c_void_p), ("c_state", C.c_void_p), ("word", C.c_void_p), ("context", C.c_void_p),
        ("logp", C.c_void_p), ("attn", C.c_void_p), ("tokens", C.c_void_p),
        ("nll_labels", C.c_void_p), ("nll_steps", C.c_int32), ("nll_terms", C.c_void_p),
        ("segment_steps", C.c_int32), ("early_exit", C.c_int32), ("eos_token", C.c_int32), ("steps_done", C.c_void_p),
    ]


class BeamIO(C.Structure):
    _fields_ = [
        ("enc", C.c_void_p), ("enc_lengths", C.c_void_p),
        ("beam", C.c_int32), ("nbest", C.c_int32), ("eos_token", C.c_int32), ("length_penalty", C.c_float),
        ("tokens", C.c_void_p), ("token_logp", C.c_void_p), ("lengths", C.c_void_p), ("scores", C.c_void_p),
        ("attn", C.c_void_p), ("attn_work", C.c_void_p),
        ("early_exit", C.c_int32), ("segment_steps", C.c_int32), ("steps_done", C.c_void_p),
    ]


class PipelineArgs(C.Structure):
    _fields_ = [
        ("dec_io", C.POINTER(DecodeIO)), ("speller_packed", C.c_void_p), ("speller_dims", C.POINTER(SpellerDims)),
        ("steps", C.c_int32), ("decode_mode", C.c_int32), ("relu", C.c_int32), ("speller_ws", C.c_void_p), ("speller_ws_bytes", C.c_size_t),
        ("x", C.c_void_p), ("x_lengths", C.c_void_p), ("listener_packed", C.c_void_p), ("listener_dims", C.POINTER(ListenerDims)),
        ("enc", C.c_void_p), ("enc_lengths", C.c_void_p), ("listener_ws", C.c_void_p), ("listener_ws_bytes", C.c_size_t),
    ]


# name -> (restype, argtypes); every name here must be declared in include/las_b200.h (tests check both ways)
PROTOTYPES = {
    "las_abi_version": (C.c_int, []),
    "las_last_error": (C.c_char_p, []),
    "las_device_check": (C.c_int, []),
    "las_mode_available": (C.c_int, [C.c_int]),
    "las_launch_count": (C.c_int64, [C.c_int]),
    "las_prof_enable": (C.c_int, [C.c_int]),
    "las_prof_report": (C.c_int, [C.c_char_p, C.c_size_t]),
    "las_listener_packed_bytes": (C.c_size_t, [C.POINTER(ListenerDims), C.c_int]),
    "las_listener_pack": (C.c_int, [C.POINTER(LstmWeights), C.POINTER(ListenerDims), C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "las_listener_workspace_bytes": (C.c_size_t, [C.POINTER(ListenerDims), C.c_int]),
    "las_listener_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(ListenerDims), C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "las_listener_forward_masked": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(ListenerDims), C.c_int, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_size_t, C.c_void_p]),
    "las_speller_packed_bytes": (C.c_size_t, [C.POINTER(SpellerDims), C.c_int]),
    "las_speller_pack": (C.c_int, [C.POINTER(SpellerWeights), C.POINTER(SpellerDims), C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "las_psi_precompute": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "las_attention_forward": (C.c_int, [C.c_void_p] * 5 + [C.c_int] * 7 + [C.c_void_p] * 6),
    "las_speller_workspace_bytes": (C.c_size_t, [C.POINTER(SpellerDims), C.c_int, C.c_int]),
    "las_speller_decode": (C.c_int, [C.POINTER(DecodeIO), C.c_void_p, C.POINTER(SpellerDims), C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "las_speller_beam_packed_bytes": (C.c_size_t, [C.POINTER(SpellerDims), C.c_int]),
    "las_speller_beam_pack": (C.c_int, [C.POINTER(SpellerWeights), C.POINTER(SpellerDims), C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "las_speller_beam_workspace_bytes": (C.c_size_t, [C.POINTER(SpellerDims), C.c_int, C.c_int, C.c_int]),
    "las_speller_beam_search": (C.c_int, [C.POINTER(BeamIO), C.c_void_p, C.POINTER(SpellerDims), C.c_int, C.c_int, C.c_int, C.c_void_p,
                                          C.c_size_t, C.c_void_p]),
    "las_pipeline_step": (C.c_int, [C.POINTER(PipelineArgs), C.c_int, C.c_void_p]),
    "las_pipeline_overlaps": (C.c_int, [C.POINTER(ListenerDims), C.POINTER(SpellerDims), C.c_int, C.c_int]),
    "las_debug_gemm_bf16": (C.c_int, [C.c_void_p] * 4 + [C.c_int] * 3 + [C.c_void_p]),
    "las_debug_umma_probe": (C.c_int, [C.c_void_p] * 3 + [C.c_int] * 5 + [C.c_void_p]),
    "las_debug_set_trace": (C.c_int, [C.c_void_p]),
    "las_debug_set_option": (C.c_int, [C.c_int, C.c_int]),
    "las_nll_sums": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "las_label_smoothing_terms": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p]),
}

_lib = None


class LasB200Error(RuntimeError):
    pass


def load_library(path: str | None = None):
    """dlopen liblas_b200.so and attach prototypes.  Raises if the library has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise LasB200Error(
            f"{p} not found: the CUDA extension has not been built (run `python -m las_pytorch_b200.build` or "
            "`__graft_entry__.build()`).  There is no CPU fallback."
        )
    lib = C.CDLL(p)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.las_abi_version() != ABI_VERSION:
        raise LasB200Error(f"ABI version mismatch: library reports {lib.las_abi_version()}, binding expects {ABI_VERSION}")
    # Shared devices: the listener's input-projection GEMM normally runs CONCURRENTLY with its layer's recurrence, which spin-waits
    # on the GEMM's tile flags -- that needs both kernels co-resident, which CUDA only gives when the SMs the recurrence leaves free
    # are really free.  LAS_B200_NO_OVERLAP=1 runs the GEMM in front of the recurrence instead (same results, ~10 % slower listener).
    if os.environ.get("LAS_B200_NO_OVERLAP", "") not in ("", "0"):
        lib.las_debug_set_option(6, 0)
    if path is None:
        _lib = lib
    return lib


def check(status: int):
    """Translate a negative status into a RuntimeError carrying the library's thread-local message."""
    if status != 0:
        msg = load_library().las_last_error()
        raise LasB200Error(f"las_b200 error {status}: {msg.decode() if msg else '?'}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def current_stream_ptr(device=None):
    import torch

    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
