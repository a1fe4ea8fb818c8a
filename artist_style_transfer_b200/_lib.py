"""ctypes binding of libast_b200.so (the C ABI declared in include/ast.h).

There is no CPU or PyTorch fallback: if the library is missing or a call fails, this raises.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# AST_B200_LIB points at another build of the same library (kernel A/B experiments); default: the in-tree build
LIB_PATH = os.environ.get("AST_B200_LIB") or os.path.join(_HERE, "libast_b200.so")

AST_F32, AST_BF16, AST_TF32, AST_U8, AST_F16 = 0, 1, 2, 3, 4
AST_MAX_TAPS = 81
CONV_RELU, CONV_REFLECT, CONV_TENSOR = 1, 2, 4
CONV_POOL_ONLY = 16
CONV_ROUND_TF32 = 8
GRAM_COUNTERS_PER_IMAGE = 16

_DTYPES = {torch.float32: AST_F32, torch.bfloat16: AST_BF16, torch.uint8: AST_U8, torch.float16: AST_F16}


class Image(ctypes.Structure):
    _fields_ = [("ptr", ctypes.c_void_p), ("dtype", ctypes.c_int32),
                ("n", ctypes.c_int32), ("h", ctypes.c_int32), ("w", ctypes.c_int32), ("c", ctypes.c_int32),
                ("sn", ctypes.c_int64), ("sh", ctypes.c_int64), ("sw", ctypes.c_int64), ("sc", ctypes.c_int64)]


class GatherGeom(ctypes.Structure):
    _fields_ = [("mi", ctypes.c_int32), ("mj", ctypes.c_int32), ("si", ctypes.c_int32), ("so", ctypes.c_int32),
                ("oy0", ctypes.c_int32), ("ox0", ctypes.c_int32), ("ntaps", ctypes.c_int32),
                ("flags", ctypes.c_int32),
                ("dy", ctypes.c_int16 * AST_MAX_TAPS), ("dx", ctypes.c_int16 * AST_MAX_TAPS),
                ("w_img_stride", ctypes.c_int64), ("stats", ctypes.c_void_p), ("pooled", ctypes.POINTER(Image)),
                ("pool_codes", ctypes.POINTER(Image))]


AST_MAX_VTAPS = 32


class StackedGeom(ctypes.Structure):
    _fields_ = [("nblk", ctypes.c_int32), ("mi", ctypes.c_int32), ("mj", ctypes.c_int32), ("sy", ctypes.c_int32),
                ("soy", ctypes.c_int32), ("sox", ctypes.c_int32), ("oy", ctypes.c_int32 * 4), ("ox", ctypes.c_int32 * 4),
                ("nvt", ctypes.c_int32), ("ntaps", ctypes.c_int32), ("flags", ctypes.c_int32),
                ("dy", ctypes.c_int16 * AST_MAX_VTAPS), ("dx", ctypes.c_int16 * AST_MAX_VTAPS),
                ("stats", ctypes.c_void_p)]


class PackMap(ctypes.Structure):
    _fields_ = [("off", ctypes.c_int64), ("stride", ctypes.c_int64 * 2), ("tap", ctypes.c_int32), ("dtype", ctypes.c_int32),
                ("rep_stride", ctypes.c_int64), ("rep", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class ParamDesc(ctypes.Structure):
    _fields_ = [("p_off", ctypes.c_int64), ("s_off", ctypes.c_int64), ("numel", ctypes.c_int64),
                ("dim", ctypes.c_int32 * 4), ("g_off", ctypes.c_int64), ("g_stride", ctypes.c_int64 * 2),
                ("g_tap", ctypes.c_int32), ("n_pack", ctypes.c_int32), ("pack", PackMap * 2)]


class AdamState(ctypes.Structure):
    _fields_ = [(n, ctypes.c_float) for n in ("lr", "beta1", "beta2", "eps", "weight_decay", "grad_scale", "step",
                                              "bias_c1", "bias_c2")]


class ReduceDesc(ctypes.Structure):
    _fields_ = [("src_off", ctypes.c_int64), ("dst_off", ctypes.c_int64), ("row_stride", ctypes.c_int64),
                ("rows", ctypes.c_int32), ("cols", ctypes.c_int32)]


_lib = None
_P = ctypes.POINTER
_vp = ctypes.c_void_p

_SIGNATURES = {
    "ast_conv_gather": [_P(Image), _vp, _vp, _vp, _P(Image), _P(Image), _P(Image), _P(GatherGeom), _vp],
    "ast_conv_stacked": [_P(Image), _vp, _vp, _P(Image), _P(Image), _P(Image), _P(StackedGeom), _vp],
    "ast_wgrad_gather": [_P(Image), _P(Image), _vp, _vp, ctypes.c_int64, ctypes.c_int64, _P(GatherGeom), _vp],
    "ast_pack_weights": [_vp, _vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int64, ctypes.c_int64,
                         _vp, ctypes.c_int32, _vp],
    "ast_pack_weights_ex": [_vp, _vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                            ctypes.c_int32, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, _vp, ctypes.c_int32, _vp],
    "ast_row_im2col": [_P(Image), _P(Image), _vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                       ctypes.c_int32, ctypes.c_int32, _vp],
    "ast_fold_rows": [_P(Image), _P(Image), _vp, ctypes.c_int32, ctypes.c_int32, _vp],
    "ast_instnorm_stats": [_P(Image), _vp, _vp, ctypes.c_float, _vp, _vp],
    "ast_instnorm_finalize": [_vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_float, _vp, _vp, _vp],
    "ast_instnorm_apply": [_P(Image), _vp, _vp, _vp, _vp, _P(Image), _P(Image), ctypes.c_int32, ctypes.c_int32, _vp],
    "ast_instnorm_bwd": [_P(Image), _vp, _vp, _vp, _vp, _P(Image), ctypes.c_int32, _P(Image), ctypes.c_int32,
                         _vp, _vp, _vp, _P(Image), _P(Image), _vp],
    "ast_maxpool2_fwd": [_P(Image), _P(Image), _P(Image), _vp],
    "ast_maxpool2_bwd": [_P(Image), _P(Image), _P(Image), _P(Image), _P(Image), _vp],
    "ast_gram": [_P(Image), _vp, ctypes.c_float, ctypes.c_int32, _vp],
    "ast_gram_mse": [_P(Image), _vp, ctypes.c_float, _vp, ctypes.c_int64, _vp, ctypes.c_float, _vp, ctypes.c_float, _vp,
                     ctypes.c_int32, _vp],
    "ast_adam_step": [_vp, ctypes.c_int32, _vp, ctypes.c_int32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, ctypes.c_int32, _vp],
    "ast_batch_reduce": [_vp, _vp, _vp, ctypes.c_int32, ctypes.c_int32, _vp],
    "ast_channel_sum": [_P(Image), _vp, _vp],
    "ast_mse": [_P(Image), _P(Image), _vp, ctypes.c_float, _P(Image), ctypes.c_float, _vp],
    "ast_copy_image": [_P(Image), _P(Image), _vp, ctypes.c_int32, _vp],
    "ast_reflect_fold": [_P(Image), _P(Image), _P(Image), ctypes.c_int32, _vp],
    "ast_accumulate": [_P(Image), _P(Image), _vp],
    "ast_mask_add": [_P(Image), _P(Image), _P(Image), _P(Image), _vp],
}
EXPORTS = sorted(list(_SIGNATURES) + ["ast_instnorm_workspace_bytes", "ast_last_error", "ast_abi_version",
                                      "ast_launch_count", "ast_capabilities", "ast_adam_work_item", "ast_family_count",
                                      "ast_family_name", "ast_family_stats", "ast_family_reset"])


def load():
    """Load the shared library (no CUDA call is made here, so this also works on a CPU-only box)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C artist_style_transfer_b200/csrc`). There is no CPU/PyTorch fallback for this path.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = ctypes.c_int
    lib.ast_instnorm_workspace_bytes.argtypes = [ctypes.c_int32, ctypes.c_int32]
    lib.ast_instnorm_workspace_bytes.restype = ctypes.c_int64
    lib.ast_last_error.restype = ctypes.c_char_p
    lib.ast_abi_version.restype = ctypes.c_int
    lib.ast_launch_count.restype = ctypes.c_int64
    lib.ast_capabilities.restype = ctypes.c_int
    lib.ast_adam_work_item.restype = ctypes.c_int32
    lib.ast_family_count.restype = ctypes.c_int
    lib.ast_family_name.argtypes = [ctypes.c_int]
    lib.ast_family_name.restype = ctypes.c_char_p
    lib.ast_family_stats.argtypes = [ctypes.c_int, _P(ctypes.c_int64), _P(ctypes.c_double), _P(ctypes.c_double)]
    lib.ast_family_stats.restype = ctypes.c_int
    lib.ast_family_reset.restype = None
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().ast_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (rc={rc}): {msg}")


def stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _check_device(t):
    """The library launches on the CURRENT device / current stream (one process per GPU): a tensor that lives on another
    GPU would be handed to a kernel running on the wrong device, so refuse it loudly."""
    if not t.is_cuda:
        raise RuntimeError("artist_style_transfer_b200 kernels need CUDA tensors (no CPU fallback)")
    if t.device.index != torch.cuda.current_device():
        raise RuntimeError(f"tensor on cuda:{t.device.index} but the current device is cuda:{torch.cuda.current_device()}; "
                           "call torch.cuda.set_device(...) (one process per GPU) or wrap the call in torch.cuda.device(...)")


def image(t):
    """ast_image of a 4-D tensor given in logical (N, H, W, C) order with arbitrary strides."""
    if t is None:
        return None
    _check_device(t)
    n, h, w, c = t.shape
    sn, sh, sw, sc = t.stride()
    return Image(t.data_ptr(), _DTYPES[t.dtype], n, h, w, c, sn, sh, sw, sc)


def ref(img):
    return None if img is None else ctypes.byref(img)


def has_tc_conv():
    """tcgen05 conv kernel built in (AST_DISABLE_TC=1 is a debugging knob that routes fast mode to the SIMT kernels)."""
    return bool(load().ast_capabilities() & 1) and os.environ.get("AST_DISABLE_TC") != "1"


def has_tc_gram():
    return bool(load().ast_capabilities() & 2) and os.environ.get("AST_DISABLE_TC") != "1"


def launch_count():
    return int(load().ast_launch_count())


def family_stats():
    """{family: (launches, algorithmic flops, algorithmic bytes)} of everything launched by this process so far."""
    lib = load()
    out = {}
    for f in range(lib.ast_family_count()):
        n, fl, by = ctypes.c_int64(), ctypes.c_double(), ctypes.c_double()
        lib.ast_family_stats(f, ctypes.byref(n), ctypes.byref(fl), ctypes.byref(by))
        out[lib.ast_family_name(f).decode()] = (n.value, fl.value, by.value)
    return out


def family_delta(before, after=None):
    after = family_stats() if after is None else after
    return {k: tuple(a - b for a, b in zip(after[k], before[k])) for k in after}


def device_bytes(ctypes_obj, device):
    """Upload a ctypes struct / array to a uint8 device tensor (descriptor tables of the table-driven kernels)."""
    buf = bytes(ctypes_obj)
    return torch.frombuffer(bytearray(buf), dtype=torch.uint8).to(device)
