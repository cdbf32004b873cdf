"""ctypes binding of libppasr_b200.so (the C-ABI declared in include/ppasr_b200.h).

The library is the product: there is no Python/CPU fallback. If the shared object is missing the
import raises with build instructions (`python -m ppasr_b200.build`).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libppasr_b200.so")

c_void_p = ctypes.c_void_p
c_int = ctypes.c_int
c_int64 = ctypes.c_int64
c_float = ctypes.c_float
c_char_p = ctypes.c_char_p

_lib = None


class PPASRB200Error(Exception):
    """Raised when a C-ABI call returns a non-zero status (message from ppasr_b200_last_error)."""


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PPASRB200Error(
            f"{LIB_PATH} not found: build it with `python -m ppasr_b200.build` "
            "(there is no CPU fallback for the hot path)")
    lib = ctypes.CDLL(LIB_PATH)
    lib.ppasr_b200_last_error.restype = c_char_p
    lib.ppasr_b200_last_error.argtypes = []
    lib.ppasr_b200_abi_version.restype = c_int
    _declare(lib)
    _lib = lib
    return lib


def check(status):
    if status != 0:
        msg = load().ppasr_b200_last_error()
        raise PPASRB200Error(f"ppasr_b200 status {status}: {msg.decode('utf-8', 'replace') if msg else ''}")


# name -> (restype, argtypes); kept in one table so tests can verify every symbol of the header
c_int32 = ctypes.c_int32
P = c_void_p
I = c_int32
PROTOTYPES = {
    "ppasr_b200_launch_count": (c_int64, []),
    "ppasr_b200_set_pdl": (c_int, [I]),
    "ppasr_b200_set_ffn_split": (c_int, [I]),
    "ppasr_b200_get_ffn_split": (c_int, []),
    "ppasr_b200_create": (c_int, [P, ctypes.POINTER(P)]),
    "ppasr_b200_destroy": (c_int, [P]),
    "ppasr_b200_load_tensor": (c_int, [P, c_char_p, P, I, P]),
    "ppasr_b200_finalize": (c_int, [P]),
    "ppasr_b200_encode": (c_int, [P, P, I, P, I, I, P]),
    "ppasr_b200_out_frames": (c_int, [P, I]),
    "ppasr_b200_ctc_probs": (c_int, [P, P, I, P]),
    "ppasr_b200_ctc_logits": (c_int, [P, P, I, P]),
    "ppasr_b200_ctc_greedy": (c_int, [P, P, P, P, P, P, I, I, I, P]),
    "ppasr_b200_stream_reset": (c_int, [P, I]),
    "ppasr_b200_encode_chunk": (c_int, [P, P, I, I, I, I, P]),
    "ppasr_b200_stream_info": (c_int, [P, P, P]),
    "ppasr_b200_sessions_init": (c_int, [P, I]),
    "ppasr_b200_sessions_reset": (c_int, [P, I]),
    "ppasr_b200_sessions_step": (c_int, [P, P, I, P, I, I, I, P]),
    "ppasr_b200_fbank_frames": (c_int, [I]),
    "ppasr_b200_fbank": (c_int, [P, I, c_int64, I, P, I, I, I, c_float, P, P, I, P]),
    "ppasr_b200_ds2_states": (c_int, [P, P, P, I, P]),
    "ppasr_b200_stream_export": (c_int, [P, P, P, I, P]),
    "ppasr_b200_beam_state_bytes": (c_int64, [I, I, I]),
    "ppasr_b200_beam_workspace_bytes": (c_int64, [I, I]),
    "ppasr_b200_beam_reset": (c_int, [P, I, I, I, P]),
    "ppasr_b200_beam_advance": (c_int, [P, I, I, I, P, I, c_float, I, I, P, I, P, P]),
    "ppasr_b200_beam_advance_lm": (c_int, [P, I, I, I, P, I, c_float, I, I, P, I, P, P, P, P, P, c_int64, I, c_float, c_float, P]),
    "ppasr_b200_beam_result": (c_int, [P, I, I, I, P, I, P, P, P]),
    "ppasr_b200_beam_result_nbest": (c_int, [P, I, I, I, I, P, I, P, P, P]),
    "ppasr_b200_op_ctc_prune": (c_int, [P, I, I, c_float, I, P, P]),
    "ppasr_b200_greedy_decode": (c_int, [P, I, I, I, P, I, P, I, P, P, P, P, P]),
    "ppasr_b200_op_linear": (c_int, [P, c_int64, P, c_int64, P, P, c_int64, I, I, I, I, I, c_float, I, P, I, I, P]),
    "ppasr_b200_op_layernorm": (c_int, [P, P, P, P, P, P, P, I, I, I, c_float, P]),
    "ppasr_b200_op_dwconv": (c_int, [P, P, P, P, P, P, I, P, I, I, I, I, I, I, c_float, P]),
    "ppasr_b200_op_softmax": (c_int, [P, I, P, I, I, P]),
    "ppasr_b200_op_fused_ffn": (c_int, [P, P, P, P, P, P, P, P, P, P, P, I, I, c_float, P]),
    "ppasr_b200_op_attention": (c_int, [P, P, P, I, P, I, I, I, I, P, I, I, I, I, P, P]),
    "ppasr_b200_op_qkv_attention": (c_int, [P, P, P, P, P, P, I, I, I, I, P, I, I, P, I, P]),
    "ppasr_b200_op_grouped_attention": (c_int, [P, P, I, P, I, P, P, I, I, I, I, P, P]),
    "ppasr_b200_debug_copy_x": (c_int, [P, P, P]),
    "ppasr_b200_debug_copy_phase": (c_int, [P, P, P, P]),
    "ppasr_b200_set_option": (c_int, [P, c_char_p, I]),
    "ppasr_b200_graph_begin": (c_int, [P, P]),
    "ppasr_b200_graph_end": (c_int, [P, P]),
    "ppasr_b200_graph_launch": (c_int, [P, P]),
    "ppasr_b200_graph_kernels": (c_int, [P]),
    "ppasr_b200_profile_enable": (c_int, [P, I]),
    "ppasr_b200_profile_num_classes": (c_int, []),
    "ppasr_b200_profile_class_name": (c_char_p, [I]),
    "ppasr_b200_profile_read": (c_int, [P, P, P]),
}


def _declare(lib):
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args


def ptr(t):
    """Device/host pointer of a torch tensor (or None)."""
    if t is None:
        return None
    return c_void_p(t.data_ptr())


def stream_ptr(stream=None):
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return c_void_p(s.cuda_stream)
