"""ctypes binding of libxvec_b200.so (C ABI in include/xvec_b200.h).

The library is the product's only compute path.  If it cannot be loaded (or built) every entry point
raises — there is deliberately no PyTorch/CPU fallback.
"""
from __future__ import annotations

import ctypes
import os
import threading
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("XVEC_LIB") or os.path.join(HERE, "libxvec_b200.so")  # XVEC_LIB: developer A/B builds

F32, BF16, F16 = 0, 1, 2
E_ARG, E_CUDA, E_DEVICE = -1, -2, -3
TILE_N, POOL_BLOCK, POOL_CHUNK, MAX_TAPS = 256, 128, 128, 8
ABI_VERSION = 8
MAX_STACK = 6
STACK_MAX_TAP_OFFSET = 8  # XVEC_STACK_MAX_TAP_OFFSET

class LayerDesc(ctypes.Structure):
    """XvecLayerDesc of include/xvec_b200.h."""
    _fields_ = [("w_packed_dev", c_void_p), ("bias_dev", c_void_p), ("n", c_int32), ("cin", c_int32), ("taps", c_int32),
                ("dtype", c_int32), ("tap_offsets", c_int32 * MAX_TAPS), ("w_plain_dev", c_void_p)]


_SIGNATURES = {
    "xvec_abi_version": (c_int, []),
    "xvec_last_error": (c_char_p, []),
    "xvec_device_check": (c_int, []),
    "xvec_watchdog_code": (c_int, []),
    "xvec_watchdog_reset": (None, []),
    "xvec_debug_trace": (c_int, [c_void_p, c_int]),
    "xvec_packed_k": (c_int64, [c_int, c_int, c_int]),
    "xvec_packed_n": (c_int64, [c_int]),
    "xvec_pack_weight": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "xvec_tdnn_layer": (c_int, [c_void_p, c_int, c_int64, c_int, c_int64, c_void_p, c_int, POINTER(c_int32), c_int,
                                c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int64, c_int64, c_void_p, c_int64, c_void_p]),
    "xvec_splitk_workspace_bytes": (c_int64, [c_int64, c_int, c_int, c_int, c_int]),
    "xvec_tdnn_pool_fused": (c_int, [c_void_p, c_int, c_int64, c_int, c_int64, c_void_p, c_int, POINTER(c_int32), c_int,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "xvec_build_layout": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int64, c_void_p, c_void_p, c_void_p]),
    "xvec_stats_pool_partial": (c_int, [c_void_p, c_int, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                        c_void_p, c_void_p, c_void_p]),
    "xvec_pool_finalize": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_int, c_int64, c_void_p]),
    "xvec_extract_forward": (c_int, [POINTER(LayerDesc), c_int, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, POINTER(LayerDesc), c_int,
                                     c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p]),
    "xvec_stack_ctrl_bytes": (c_int64, [c_int64, c_int]),
    "xvec_stack_plan": (c_int64, [c_int64, c_int, POINTER(c_int32), c_int, c_void_p, c_int64]),
    "xvec_linear_small": (c_int, [c_void_p, c_int, c_int64, c_int, c_int64, c_void_p, c_int, c_int64, c_void_p, c_int, c_void_p, c_int, c_int64,
                                  c_void_p]),
    "xvec_tdnn_stack": (c_int, [POINTER(LayerDesc), c_int, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                                c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    "xvec_mfcc_num_frames": (c_int64, [c_int64]),
    "xvec_mfcc": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "xvec_wav_minmax": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "xvec_cast": (c_int, [c_void_p, c_int64, c_void_p, c_int, c_int64, c_int64, c_int, c_void_p]),
    "xvec_cosine_trials": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "xvec_split_tf32": (c_int, [c_void_p, c_int64, c_int64, c_int, c_void_p, c_int64, c_void_p]),
    "xvec_plda_rowterm": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "xvec_plda_trials": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_float, c_float,
                                 c_void_p, c_void_p]),
}
EXPORTS = tuple(_SIGNATURES)

_lock = threading.Lock()
_lib = None


class XvecError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libxvec_b200 error {code}: {msg}")
        self.code = code


def load(build_if_missing: bool = True) -> ctypes.CDLL:
    """Load (building in-tree with nvcc if the .so is absent) and type the library."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            if not build_if_missing:
                raise ImportError(f"{LIB_PATH} is missing; run speaker-recognition-x-vectors_b200/build.py")
            from . import build as _build
            _build.build()
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        if lib.xvec_abi_version() != ABI_VERSION:
            raise ImportError(f"{LIB_PATH}: ABI {lib.xvec_abi_version()} != expected {ABI_VERSION}; rebuild")
        _lib = lib
        return lib


def check(rc: int) -> None:
    if rc != 0:
        raise XvecError(rc, load().xvec_last_error().decode("utf-8", "replace"))


def ptr(t) -> int | None:
    """Device pointer of a torch tensor (None passes NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr(device_index: int | None = None) -> int:
    """cudaStream_t of torch's current stream on the given (default: current) device — the raw C query: torch.cuda.current_stream()
    builds a Python Stream object and costs ~15 us, which matters at ten thousand calls per second and rank."""
    import torch
    return torch._C._cuda_getCurrentRawStream(torch.cuda.current_device() if device_index is None else device_index)


class on_device:
    """`with on_device(dev):` = torch.cuda.device(dev), skipping the device switch (and ~15 us of Python) when `dev` is current."""
    __slots__ = ("ctx",)

    def __init__(self, device):
        import torch
        idx = device.index if device.index is not None else torch.cuda.current_device()
        self.ctx = None if idx == torch.cuda.current_device() else torch.cuda.device(idx)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *a):
        if self.ctx is not None:
            return self.ctx.__exit__(*a)


def dtype_code(torch_dtype) -> int:
    import torch
    if torch_dtype == torch.float32:
        return F32
    if torch_dtype == torch.bfloat16:
        return BF16
    if torch_dtype == torch.float16:
        return F16
    raise ValueError(f"unsupported dtype {torch_dtype}; the kernels take float32 (TF32 math), bfloat16 or float16")


def taps_array(offsets):
    arr = (c_int32 * len(offsets))(*[int(o) for o in offsets])
    return arr
