"""ctypes binding of libspconv.so (include/spconv.h).  No fallback: if the library is missing or
a call fails, we raise -- the product never computes on the CPU or through torch.nn.Conv2d."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libspconv.so")

SPC_F32, SPC_BF16 = 0, 1
SPC_POOL_MAX, SPC_POOL_AVG = 0, 1
SPC_ALGO_AUTO, SPC_ALGO_DIRECT, SPC_ALGO_TCGEN05, SPC_ALGO_TF32 = 0, 1, 2, 3
IPC_HANDLE_BYTES = 64


class ConvDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                ("N", "C", "H", "W", "K", "R", "S", "stride_h", "stride_w", "pad_h", "pad_w", "dtype", "algo")]


class PoolDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("N", "C", "H", "W", "k", "stride", "pad", "mode", "dtype")]


class Halo(C.Structure):
    _fields_ = [("strip", C.c_void_p * 9)]


# every symbol include/spconv.h declares: (name, restype, argtypes)
_P = C.c_void_p
SYMBOLS = [
    ("spc_version", C.c_int, []),
    ("spc_last_error", C.c_char_p, []),
    ("spc_device_info", C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    ("spc_launch_count", C.c_longlong, [C.c_int]),
    ("spc_reload_env", None, []),
    ("spc_conv2d_fwd", C.c_int, [C.POINTER(ConvDesc), _P, C.POINTER(Halo), _P, _P, _P, _P, C.c_size_t, _P]),
    ("spc_conv2d_fwd_interior", C.c_int, [C.POINTER(ConvDesc), _P, _P, _P, _P, _P, C.c_size_t, _P]),
    ("spc_conv2d_fwd_boundary", C.c_int, [C.POINTER(ConvDesc), _P, C.POINTER(Halo), _P, _P, _P, _P]),
    ("spc_conv2d_dgrad", C.c_int, [C.POINTER(ConvDesc), _P, _P, _P, _P, C.c_size_t, _P]),
    ("spc_conv2d_wgrad", C.c_int, [C.POINTER(ConvDesc), _P, C.POINTER(Halo), _P, _P, _P, C.c_int, _P, C.c_size_t, _P]),
    ("spc_conv_workspace_bytes", C.c_size_t, [C.POINTER(ConvDesc), C.c_int]),
    ("spc_conv_uses_tcgen05", C.c_int, [C.POINTER(ConvDesc), C.c_int]),
    ("spc_conv_out_shape", None, [C.POINTER(ConvDesc), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    ("spc_pool2d_fwd", C.c_int, [C.POINTER(PoolDesc), _P, C.POINTER(Halo), _P, _P]),
    ("spc_pool2d_bwd", C.c_int, [C.POINTER(PoolDesc), _P, C.POINTER(Halo), _P, _P, _P]),
    ("spc_bn_stats", C.c_int, [C.c_int, C.c_int, C.c_longlong, C.c_int, _P, _P, _P, _P]),
    ("spc_bn_apply", C.c_int, [C.c_int, C.c_int, C.c_longlong, C.c_int, _P, _P, _P, _P, _P, C.c_int, _P, _P]),
    ("spc_bn_bwd_reduce", C.c_int, [C.c_int, C.c_int, C.c_longlong, C.c_int, _P, _P, _P, _P, _P, _P, C.c_int, _P, _P, _P]),
    ("spc_bn_bwd_apply", C.c_int, [C.c_int, C.c_int, C.c_longlong, C.c_int, _P, _P, _P, _P, _P, _P, C.c_int, _P, _P, _P, _P]),
    ("spc_halo_pack", C.c_int, [C.c_int] * 7 + [_P, C.POINTER(_P * 9), _P]),
    ("spc_halo_pad", C.c_int, [C.c_int] * 7 + [_P, C.POINTER(Halo), _P, _P]),
    ("spc_halo_crop", C.c_int, [C.c_int] * 7 + [_P, _P, _P]),
    ("spc_mailbox_create", C.c_int, [C.POINTER(_P), C.c_size_t, C.c_int]),
    ("spc_mailbox_destroy", None, [_P]),
    ("spc_mailbox_data", _P, [_P]),
    ("spc_mailbox_export", C.c_int, [_P, C.c_char_p]),
    ("spc_mailbox_open", C.c_int, [C.POINTER(_P), C.c_char_p, C.c_size_t, C.c_int]),
    ("spc_halo_post", C.c_int, [C.c_int] * 7 + [_P, C.POINTER(_P * 9), _P, C.POINTER(_P * 9), C.POINTER(C.c_int * 9),
                                C.c_uint32, C.POINTER(C.c_int * 9), C.c_uint32, _P]),
    ("spc_halo_collect", C.c_int, [C.POINTER(_P * 9), C.POINTER(_P * 9), C.POINTER(C.c_size_t * 9), _P, C.POINTER(_P * 9),
                                   C.POINTER(C.c_int * 9), C.c_uint32, C.POINTER(C.c_int * 9), _P]),
    ("spc_halo_post_auto", C.c_int, [C.c_int] * 7 + [_P, C.POINTER(_P * 9), C.c_size_t, _P, C.POINTER(_P * 9),
                                     C.POINTER(C.c_int * 9), C.POINTER(C.c_int * 9), C.c_int, C.c_int, _P]),
    ("spc_halo_collect_auto", C.c_int, [C.POINTER(_P * 9), C.POINTER(_P * 9), C.POINTER(C.c_size_t * 9), C.c_size_t, _P,
                                        C.POINTER(_P * 9), C.POINTER(C.c_int * 9), C.POINTER(C.c_int * 9), C.c_int, C.c_int,
                                        _P]),
    ("spc_mailbox_signal", C.c_int, [_P, C.c_int, C.c_uint32, _P]),
    ("spc_mailbox_wait", C.c_int, [_P, C.c_int, C.c_uint32, _P]),
]

_lib = None


class SpconvError(RuntimeError):
    pass


def lib():
    """Load libspconv.so (once).  Raises if it has not been built (python -m mpi4dl_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SpconvError(
                "libspconv.so not found at %s -- build it with `python mpi4dl_b200/build.py` "
                "(there is no CPU / PyTorch fallback for the spatial conv path)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(L, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc, what):
    if rc != 0:
        raise SpconvError("%s failed (%d): %s" % (what, rc, lib().spc_last_error().decode()))


def dtype_code(torch_dtype):
    import torch

    if torch_dtype == torch.float32:
        return SPC_F32
    if torch_dtype == torch.bfloat16:
        return SPC_BF16
    raise SpconvError("libspconv supports float32 and bfloat16 tensors, got %s" % torch_dtype)


def make_halo(strips):
    """strips: list of 9 (tensor or None) -> Halo struct (keeps no references!)."""
    h = Halo()
    for i in range(9):
        t = strips[i] if strips is not None else None
        h.strip[i] = t.data_ptr() if (t is not None and i != 4) else None
    return h
