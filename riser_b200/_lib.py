"""ctypes binding of libriser_b200.so (include/riser_b200.h).

There is no CPU fallback: if the library is missing, or a launch function is
called without an sm_100 device, this raises."""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RISER_B200_LIB", os.path.join(HERE, "libriser_b200.so"))

c_int, c_i64, c_void_p, c_size_t, c_float = (ctypes.c_int, ctypes.c_int64, ctypes.c_void_p,
                                             ctypes.c_size_t, ctypes.c_float)
P = ctypes.POINTER

# name -> (restype, argtypes); must list every symbol include/riser_b200.h declares
SIGNATURES = {
    "riser_version": (c_int, []),
    "riser_last_error": (ctypes.c_char_p, []),
    "riser_device_info": (c_int, [c_int, P(c_int), P(c_int), P(c_int)]),
    "riser_normalise_max_len": (c_int, []),
    "riser_normalise": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_i64,
                                c_void_p, c_void_p]),
    "riser_normalise_f32_max_len": (c_int, []),
    "riser_normalise_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_void_p, c_i64, c_void_p]),
    "riser_normalise_f32_live": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_i64, c_void_p, c_void_p]),
    "riser_normalise_long_workspace_bytes": (c_size_t, [c_int, c_int]),
    "riser_normalise_long": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_i64,
                                     c_void_p, c_void_p, c_size_t, c_void_p]),
    "riser_normalise_f32_long": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_int, c_void_p, c_i64,
                                         c_void_p, c_void_p, c_size_t, c_void_p]),
    "riser_polya_end": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int,
                                c_void_p]),
    "riser_polya_end_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int,
                                    c_void_p]),
    "riser_select_window": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                    c_void_p]),
    "riser_model_create": (c_int, [P(c_void_p), c_int, P(c_int), P(c_void_p), P(c_void_p), c_void_p,
                                   c_void_p, c_int, c_int]),
    "riser_model_destroy": (c_int, [c_void_p]),
    "riser_workspace_bytes": (c_size_t, [c_void_p, c_int, c_int]),
    "riser_plan_create": (c_int, [P(c_void_p), c_void_p, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "riser_plan_destroy": (c_int, [c_void_p]),
    "riser_forward": (c_int, [c_void_p, c_void_p, c_i64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "riser_forward_stage": (c_int, [c_void_p, c_int, c_void_p, c_i64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "riser_forward_launches": (c_int, [c_void_p]),
    "riser_plan_fused_layer0": (c_int, [c_void_p]),
    "riser_plan_layer_info": (c_int, [c_void_p, c_int, P(c_i64), P(c_int), P(c_int), P(c_int), P(c_int)]),
    "riser_plan_layer_eo": (c_int, [c_void_p, c_int]),
    "riser_plan_layer_format": (c_int, [c_void_p, c_int]),
    "riser_plan_layer_kernel": (c_int, [c_void_p, c_int]),
    "riser_conv1d_cl": (c_int, [c_void_p] * 7 + [c_int] * 9 + [c_void_p]),
    "riser_stem_pool_cl": (c_int, [c_void_p, c_i64] + [c_void_p] * 6 + [c_int] * 6 + [c_void_p]),
    "riser_res_tc_smem": (c_size_t, [c_int] * 8),
    "riser_res_tc": (c_int, [c_void_p] * 10 + [c_float, c_float] + [c_int] * 11 + [c_void_p]),
    "riser_res_tc_smem_ex": (c_size_t, [c_int] * 9),
    "riser_res_tc_ex": (c_int, [c_void_p] * 10 + [c_float, c_float] + [c_int] * 11 + [c_void_p, c_int]),
    "riser_len_chain": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p]),
    "riser_maxpool1d_cl": (c_int, [c_void_p] * 4 + [c_int] * 4 + [c_void_p]),
    "riser_maxpool1d_pad_cl": (c_int, [c_void_p] * 4 + [c_int] * 5 + [c_void_p]),
    "riser_gap_linear_softmax": (c_int, [c_void_p] * 5 + [c_int] * 4 + [c_void_p]),
    "riser_decide": (c_int, [c_void_p, c_void_p, c_int, c_int, c_float, c_int, c_int, c_void_p, c_void_p]),
}

_lib = None


class RiserError(RuntimeError):
    pass


def lib():
    """The loaded library (loads on first use; raises if it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RiserError(f"{LIB_PATH} not found: build it with `python -m riser_b200.build` "
                             "(there is no CPU fallback)")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)      # AttributeError if the symbol is missing
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(status, what):
    if status != 0:
        msg = lib().riser_last_error().decode(errors="replace")
        raise RiserError(f"{what} failed (status {status}): {msg}")


def require_device():
    """Raise unless torch sees an sm_100 CUDA device (no CPU fallback)."""
    import torch
    if not torch.cuda.is_available():
        raise RiserError("riser_b200 needs a CUDA sm_100 (B200) device; none is visible and there is "
                         "no CPU fallback")
    major, _ = torch.cuda.get_device_capability()
    if major != 10:
        raise RiserError(f"riser_b200 kernels are built for sm_100a only; found sm_{major}x")
    return torch.device("cuda", torch.cuda.current_device())


def stream_ptr():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device (or host) pointer of a torch tensor / None as c_void_p."""
    if t is None:
        return ctypes.c_void_p(0)
    return ctypes.c_void_p(t.data_ptr())
