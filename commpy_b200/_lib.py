"""ctypes binding of libcommpy_b200.so (the C-ABI declared in include/commpy_b200.h).

There is NO CPU fallback: if the shared library is missing or the GPU is absent, every decode
entry point raises.  Importing this module does not touch CUDA."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcommpy_b200.so")

CPB_OK, CPB_EINVAL, CPB_EUNSUPPORTED, CPB_ECUDA, CPB_ENOMEM, CPB_ETRELLIS = range(6)
CPB_U8, CPB_F32 = 0, 1
VITERBI_MODES = {"hard": 0, "soft": 1, "unquantized": 2}
LDPC_FP32, LDPC_FP64 = 0, 1
OPT_VITERBI_FORCE_GENERIC, OPT_LDPC_NO_BULK, OPT_BCJR_WINDOW, OPT_BCJR_PER_STEP_SCALING, OPT_TURBO_FRAME_MAJOR, OPT_TX_FORCE_GENERIC = 0, 1, 2, 3, 4, 5

# every symbol include/commpy_b200.h declares (tests/test_abi.py checks the header against this list)
SYMBOLS = [
    "cpb_strerror", "cpb_last_cuda_error", "cpb_version", "cpb_device_info", "cpb_release_scratch", "cpb_set_option", "cpb_get_option",
    "cpb_trellis_create", "cpb_trellis_destroy", "cpb_trellis_fast_path",
    "cpb_viterbi_sizes", "cpb_viterbi_workspace_bytes", "cpb_viterbi_decode", "cpb_viterbi_decode_host", "cpb_viterbi_decode_packed", "cpb_viterbi_decode_host_packed",
    "cpb_viterbi_punctured_workspace_bytes", "cpb_viterbi_decode_punctured",
    "cpb_map_workspace_bytes", "cpb_map_decode", "cpb_turbo_workspace_bytes", "cpb_turbo_decode",
    "cpb_map_decode_host", "cpb_turbo_decode_host", "cpb_ldpc_decode_host", "cpb_demod_soft_host",
    "cpb_ldpc_create", "cpb_ldpc_destroy", "cpb_ldpc_workspace_bytes", "cpb_ldpc_minsum", "cpb_ldpc_sumproduct",
    "cpb_modem_create", "cpb_modem_destroy", "cpb_modem_is_separable", "cpb_demod_soft", "cpb_demod_hard",
    "cpb_count_errors", "cpb_conv_link_tx", "cpb_conv_link_tx_punctured", "cpb_turbo_link_tx",
]

_lib = None


class CommpyB200Error(RuntimeError):
    pass


def load():
    """Load the library (no CUDA call is made)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CommpyB200Error(
                "libcommpy_b200.so is not built (%s). Run `python -m commpy_b200.build`; "
                "there is no CPU fallback." % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        lib.cpb_strerror.restype = C.c_char_p
        lib.cpb_strerror.argtypes = [C.c_int]
        lib.cpb_last_cuda_error.restype = C.c_char_p
        for name in SYMBOLS:
            fn = getattr(lib, name, None)
            if fn is not None and name not in ("cpb_strerror", "cpb_last_cuda_error"):
                fn.restype = C.c_int
        _lib = lib
    return _lib


def check(status, what=""):
    """Map a cpb status to the exception type the reference raises for the same mistake."""
    if status == CPB_OK:
        return
    lib = load()
    msg = "%s: %s" % (what, lib.cpb_strerror(status).decode())
    if status in (CPB_EINVAL, CPB_ETRELLIS):
        raise ValueError(msg)
    if status == CPB_EUNSUPPORTED:
        raise NotImplementedError(msg)
    raise CommpyB200Error(msg + " | " + lib.cpb_last_cuda_error().decode())


def set_option(option_id, value):
    """cpb_set_option: explicit test / cross-check switches (the library never reads the environment)."""
    check(load().cpb_set_option(int(option_id), int(value)), "set_option")


def release_scratch():
    """cpb_release_scratch: hand the unused part of the library's device scratch pool back to the driver."""
    check(load().cpb_release_scratch(), "release_scratch")


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise CommpyB200Error("commpy_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback.")
    return torch


def ptr(t):
    """device/host pointer of a torch tensor or numpy array as c_void_p"""
    if t is None:
        return C.c_void_p(0)
    if hasattr(t, "data_ptr"):
        return C.c_void_p(t.data_ptr())
    return C.c_void_p(t.ctypes.data)


def stream_ptr(torch):
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
