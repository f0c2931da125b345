"""ctypes binding of libbin_b200.so (include/bin_b200.h).  Fails loudly when the CUDA
library is missing -- there is no CPU or PyTorch fallback on the product path."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libbin_b200.so")

BIN_MAX_CALLS = 6
BIN_MAX_FRAMES = 5
BIN_BACKBONE_NCONV = 66
EPI_P8, EPI_PIXSHUF, EPI_FINAL = 0, 1, 2
ABI_VERSION = 2
BIN_MAX_METRIC_PAIRS = 64
SSIM_BOX7, SSIM_GAUSS11 = 0, 1
BIN_TRAIN_FRAMES = 17
BIN_MAX_TRAIN_SAMPLES = 64


class Act(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("B", C.c_int), ("planes", C.c_int), ("H", C.c_int), ("W", C.c_int)]


class Frames(C.Structure):
    _fields_ = [("frame", (C.c_void_p * BIN_MAX_FRAMES) * BIN_MAX_CALLS),
                ("out", C.c_void_p * BIN_MAX_CALLS),
                ("ncalls", C.c_int), ("nframes", C.c_int), ("Bc", C.c_int)]


class ConvArgs(C.Structure):
    _fields_ = [("in0", Act), ("in0_plane0", C.c_int), ("in0_planes", C.c_int),
                ("in1", Act), ("in1_plane0", C.c_int), ("in1_planes", C.c_int),
                ("w_packed", C.c_void_p), ("bias", C.c_void_p),
                ("ksize", C.c_int), ("cout_pad", C.c_int), ("relu", C.c_int), ("epilogue", C.c_int), ("variant", C.c_int),
                ("b_begin", C.c_int), ("b_count", C.c_int), ("y_begin", C.c_int), ("y_count", C.c_int), ("store_planes", C.c_int), ("x3", C.c_int),
                ("out", Act), ("out_plane0", C.c_int),
                ("res", Act), ("res_plane0", C.c_int),
                ("fr", Frames)]


class Net(C.Structure):
    _fields_ = [("blob", C.c_void_p * 4), ("lstm_w", C.c_void_p * 6), ("lstm_b", C.c_void_p * 6)]


class TrainSample(C.Structure):
    _fields_ = [("src", C.c_void_p * BIN_TRAIN_FRAMES), ("y0", C.c_int), ("x0", C.c_int), ("flip", C.c_int)]


class BinB200Error(RuntimeError):
    pass


_SIGS = {
    "bin_abi_version": (C.c_int, []),
    "bin_last_error": (C.c_char_p, []),
    "bin_check_device": (C.c_int, []),
    "bin_nchw_to_p8": (C.c_int, [C.c_void_p, C.c_int, Act, C.c_int, C.c_void_p]),
    "bin_p8_to_nchw": (C.c_int, [Act, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "bin_pack_frames": (C.c_int, [C.POINTER(Frames), C.c_int, C.c_int, Act, C.c_void_p]),
    "bin_packed_weight_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "bin_pack_conv_weight": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "bin_conv_fwd": (C.c_int, [C.POINTER(ConvArgs), C.c_void_p]),
    "bin_pack_conv_weight_t": (C.c_int, [C.c_void_p] + [C.c_int] * 7 + [C.c_void_p, C.c_void_p]),
    "bin_conv_wgrad_workspace_bytes": (C.c_size_t, []),
    "bin_conv_wgrad": (C.c_int, [Act, C.c_int, C.c_int, Act, C.c_int, C.c_int, Act, C.c_int, C.c_int, C.c_int, C.c_int,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bin_convlstm_fwd": (C.c_int, [C.c_void_p] * 7 + [C.c_int] * 3 + [C.c_void_p]),
    "bin_convlstm_bwd": (C.c_int, [C.c_void_p] * 13 + [C.c_int] * 3 + [C.c_void_p]),
    "bin_backbone_packed_bytes": (C.c_size_t, [C.c_int]),
    "bin_backbone_pack": (C.c_int, [C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p]),
    "bin_backbone_workspace_bytes": (C.c_size_t, [C.c_int] * 4),
    "bin_backbone_fwd": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(Frames), C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "bin_backbone_packed_t_bytes": (C.c_size_t, [C.c_int]),
    "bin_backbone_pack_t": (C.c_int, [C.c_int, C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p]),
    "bin_backbone_train_workspace_bytes": (C.c_size_t, [C.c_int] * 4),
    "bin_backbone_fwd_train": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(Frames), C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "bin_backbone_grad_workspace_bytes": (C.c_size_t, [C.c_int] * 4),
    "bin_backbone_grad_param_floats": (C.c_size_t, [C.c_int]),
    "bin_backbone_bwd": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(Frames), C.POINTER(Frames), C.c_int, C.c_int, C.c_void_p,
                                   C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bin_grad_scale": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_size_t, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bin_rdb_fwd": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                              C.c_void_p, C.c_size_t, C.c_void_p]),
    "bin_window_workspace_bytes": (C.c_size_t, [C.c_int] * 3),
    "bin_window_fwd": (C.c_int, [C.POINTER(Net), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int, C.c_int,
                                 C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "bin_backbone_packed_bytes_p": (C.c_size_t, [C.c_int, C.c_int]),
    "bin_backbone_pack_p": (C.c_int, [C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_void_p, C.c_int, C.c_void_p]),
    "bin_backbone_workspace_bytes_p": (C.c_size_t, [C.c_int] * 5),
    "bin_backbone_fwd_p": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(Frames), C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "bin_window_workspace_bytes_p": (C.c_size_t, [C.c_int] * 4),
    "bin_window_fwd_p": (C.c_int, [C.POINTER(Net), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int, C.c_int,
                                   C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "bin_pyramid3_fwd": (C.c_int, [C.POINTER(Net), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int, C.c_int,
                                   C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "bin_pixel_loss_fwd": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int, C.c_size_t, C.c_int, C.c_float, C.c_void_p, C.c_void_p]),
    "bin_pixel_loss_bwd": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int,
                                    C.c_size_t, C.c_int, C.c_float, C.c_void_p, C.c_void_p]),
    "bin_tensor2img_u8": (C.c_int, [C.c_void_p] + [C.c_int] * 6 + [C.c_void_p, C.c_void_p]),
    "bin_u8_to_frame": (C.c_int, [C.c_void_p] + [C.c_int] * 6 + [C.c_void_p, C.c_void_p]),
    "bin_rdb_tail_fwd": (C.c_int, [C.POINTER(Act), C.c_int, C.POINTER(Act), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.POINTER(Act), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "bin_adam_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int] + [C.c_float] * 8 + [C.c_void_p]),
    "bin_blur_average_u8": (C.c_int, [C.c_void_p, C.c_int, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "bin_image_metrics_workspace_bytes": (C.c_size_t, [C.c_int] * 5),
    "bin_image_metrics_u8": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)] + [C.c_int] * 5 +
                             [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "bin_train_batch_u8": (C.c_int, [C.POINTER(TrainSample)] + [C.c_int] * 5 + [C.c_void_p] * 4),
}
# measurement tooling (libbin_b200_tools.so, csrc/tools_abi.h) -- bound only when BIN_B200_LIB points at that library
_TOOLS_SIGS = {
    "bin_tools_microbench_mma": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    "bin_tools_debug_timeline": (C.c_int, [C.POINTER(C.c_longlong), C.c_int]),
}

_lib = None


def lib() -> C.CDLL:
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        path = os.environ.get("BIN_B200_LIB") or LIB_PATH          # tools point this at libbin_b200_tools.so
        tools = os.path.basename(path) == "libbin_b200_tools.so"
        # A fresh checkout carries sources only, and an in-tree library may be older than the sources: (re)build when the
        # source digest differs from the stamp next to the .so (a no-op otherwise; ~1 min with nvcc).  If that is not
        # possible and no library exists the package is unusable -- there is deliberately no CPU / PyTorch fallback.
        try:
            from . import build as _build
            if path in (LIB_PATH, _build.TOOLS_LIB):
                _build.build(tools=tools)
        except Exception as e:  # noqa: BLE001
            if not os.path.exists(path) or "failed" in str(e):       # a compile/link error is never papered over
                raise BinB200Error(
                    f"{path} not found and building it failed ({e}). Build with `python -m bin_b200.build` "
                    "(nvcc, sm_100a). bin_b200 has no CPU/PyTorch fallback.") from e
            import warnings
            warnings.warn(f"bin_b200: could not verify/rebuild {path} against the sources ({e}); using it as is")
        L = C.CDLL(path)
        sigs = dict(_SIGS)
        if tools:
            sigs.update(_TOOLS_SIGS)
        for name, (res, args) in sigs.items():
            fn = getattr(L, name)          # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        if L.bin_abi_version() != ABI_VERSION:
            raise BinB200Error(f"{os.path.basename(path)} ABI version mismatch")
        _lib = L
    return _lib


def check(code: int) -> None:
    if code != 0:
        raise BinB200Error(f"bin_b200 error {code}: {lib().bin_last_error().decode()}")


def exported_symbols():
    return list(_SIGS.keys())
