"""ctypes binding of the C ABI declared in include/ievm.h, plus the in-tree nvcc build.

The shared library is the product: there is no Python/CPU fallback.  ``load()`` raises if the
library is missing instead of degrading.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
LIB_PATH = os.environ.get("IEVM_LIB_PATH") or os.path.join(PKG_DIR, "libievm_b200.so")   # override: A/B builds
CSRC = os.path.join(PKG_DIR, "csrc")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-ffp-contract=off", "-shared",
]

EXPORTS = [
    "ievm_create", "ievm_destroy", "ievm_forward_i8", "ievm_forward_f16", "ievm_forward_i8_host",
    "ievm_forward_f16_host", "ievm_set_option", "ievm_num_tensors", "ievm_tensor_shape",
    "ievm_launches_per_forward", "ievm_layer_launch", "ievm_debug_read_tensor", "ievm_debug_conv_acc", "ievm_kd_loss",
    "ievm_last_error", "ievm_build_info", "ievm_probe_im2col", "ievm_profile_read", "ievm_probe_patch",
    "ievm_debug_frontend", "ievm_set_input_lut", "ievm_forward_u8", "ievm_forward_u8_host",
    "ievm_count_correct", "ievm_set_resize", "ievm_forward_u8_resize", "ievm_forward_u8_resize_host", "ievm_debug_resize",
    "ievm_observer_points", "ievm_observe", "ievm_observer_read", "ievm_observer_capacity", "ievm_observer_set_groups",
    "ievm_observer_read_hist", "ievm_observer_clear",
    "ievm_submit_i8_host", "ievm_submit_f16_host", "ievm_submit_u8_host", "ievm_submit_u8_resize_host", "ievm_wait",
    "ievm_probe_mma_peak", "ievm_set_wait_limit_ms",
]


class LayerDesc(C.Structure):
    _fields_ = [
        ("op", C.c_int32), ("in_tensor", C.c_int32), ("res_tensor", C.c_int32), ("out_tensor", C.c_int32),
        ("cin", C.c_int32), ("cout", C.c_int32), ("ksize", C.c_int32), ("stride", C.c_int32), ("pad", C.c_int32),
        ("relu", C.c_int32),
        ("weight", C.c_void_p), ("bias", C.c_void_p), ("w_scale", C.c_void_p),
        ("in_scale", C.c_float), ("in_zp", C.c_int32),
        ("out_scale", C.c_float), ("out_zp", C.c_int32),
        ("res_scale", C.c_float), ("res_zp", C.c_int32),
        ("add_scale", C.c_float), ("add_zp", C.c_int32),
    ]


class NetDesc(C.Structure):
    _fields_ = [
        ("dtype", C.c_int32), ("num_layers", C.c_int32),
        ("in_c", C.c_int32), ("in_h", C.c_int32), ("in_w", C.c_int32), ("num_classes", C.c_int32),
        ("in_scale", C.c_float), ("in_zp", C.c_int32),
        ("layers", C.POINTER(LayerDesc)),
    ]


def sources():
    return [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh"))] + \
        [os.path.join(ROOT, "include", "ievm.h")]


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(s) > t for s in sources())


def build(force: bool = False, verbose: bool = False, defines=(), out: str = None) -> str:
    """Compile csrc/ievm.cu for sm_100a into libievm_b200.so (in-tree, so it travels to the GPU box).
    ``defines`` / ``out`` build an experimental variant (-DNAME=VALUE ...) to another path."""
    out = out or LIB_PATH
    if not force and not defines and not needs_build():
        return out
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + [f"-D{d}" for d in defines] + \
        ["-o", out, os.path.join(CSRC, "ievm.cu")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return out


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "This engine has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    H = C.c_void_p
    lib.ievm_create.argtypes = [C.POINTER(NetDesc), C.c_int, C.c_int, C.POINTER(H)]
    lib.ievm_create.restype = C.c_int
    lib.ievm_destroy.argtypes = [H]
    lib.ievm_destroy.restype = None
    lib.ievm_forward_i8.argtypes = [H, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.ievm_forward_f16.argtypes = [H, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.ievm_forward_i8_host.argtypes = [H, C.c_void_p, C.c_int, C.c_void_p]
    lib.ievm_forward_f16_host.argtypes = [H, C.c_void_p, C.c_int, C.c_void_p]
    lib.ievm_set_option.argtypes = [H, C.c_char_p, C.c_int]
    lib.ievm_num_tensors.argtypes = [H]
    lib.ievm_tensor_shape.argtypes = [H, C.c_int, C.POINTER(C.c_int32 * 6)]
    lib.ievm_launches_per_forward.argtypes = [H]
    lib.ievm_layer_launch.argtypes = [H, C.c_int]
    lib.ievm_layer_launch.restype = C.c_int
    lib.ievm_debug_read_tensor.argtypes = [H, C.c_int, C.c_void_p, C.c_uint64]
    lib.ievm_debug_conv_acc.argtypes = [H, C.c_int, C.c_int, C.c_void_p, C.c_uint64]
    lib.ievm_kd_loss.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p,
                                 C.c_void_p]
    lib.ievm_probe_im2col.argtypes = [C.c_void_p] + [C.c_int] * 12 + [C.c_void_p]
    lib.ievm_probe_im2col.restype = C.c_int
    lib.ievm_probe_patch.argtypes = [C.c_void_p] + [C.c_int] * 10 + [C.c_void_p]
    lib.ievm_probe_patch.restype = C.c_int
    lib.ievm_set_input_lut.argtypes = [H, C.c_void_p]
    lib.ievm_set_input_lut.restype = C.c_int
    lib.ievm_forward_u8.argtypes = [H, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.ievm_forward_u8.restype = C.c_int
    lib.ievm_forward_u8_host.argtypes = [H, C.c_void_p, C.c_int, C.c_void_p]
    lib.ievm_forward_u8_host.restype = C.c_int
    lib.ievm_set_resize.argtypes = [H, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    lib.ievm_set_resize.restype = C.c_int
    lib.ievm_forward_u8_resize.argtypes = [H, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.ievm_forward_u8_resize.restype = C.c_int
    lib.ievm_forward_u8_resize_host.argtypes = [H, C.c_void_p, C.c_int, C.c_void_p]
    lib.ievm_forward_u8_resize_host.restype = C.c_int
    lib.ievm_debug_resize.argtypes = [H, C.c_void_p, C.c_int, C.c_void_p, C.c_uint64]
    lib.ievm_debug_resize.restype = C.c_int
    lib.ievm_count_correct.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.ievm_count_correct.restype = C.c_int
    lib.ievm_debug_frontend.argtypes = [H, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64]
    lib.ievm_debug_frontend.restype = C.c_int
    lib.ievm_profile_read.argtypes = [H, C.c_int, C.c_void_p, C.c_void_p]
    lib.ievm_profile_read.restype = C.c_int
    lib.ievm_observer_points.argtypes = [H]
    lib.ievm_observer_points.restype = C.c_int
    lib.ievm_observe.argtypes = [H, C.c_void_p, C.c_void_p]
    lib.ievm_observe.restype = C.c_int
    lib.ievm_observer_read.argtypes = [H, C.c_void_p, C.c_int]
    lib.ievm_observer_read.restype = C.c_int
    lib.ievm_observer_capacity.argtypes = [H]
    lib.ievm_observer_capacity.restype = C.c_int
    lib.ievm_observer_set_groups.argtypes = [H, C.c_void_p, C.c_int]
    lib.ievm_observer_set_groups.restype = C.c_int
    lib.ievm_observer_read_hist.argtypes = [H, C.c_void_p, C.c_void_p, C.c_int]
    lib.ievm_observer_read_hist.restype = C.c_int
    lib.ievm_observer_clear.argtypes = [H]
    lib.ievm_observer_clear.restype = C.c_int
    for name in ("ievm_submit_i8_host", "ievm_submit_f16_host", "ievm_submit_u8_host", "ievm_submit_u8_resize_host"):
        getattr(lib, name).argtypes = [H, C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_int64)]
        getattr(lib, name).restype = C.c_int
    lib.ievm_wait.argtypes = [H, C.c_int64]
    lib.ievm_wait.restype = C.c_int
    lib.ievm_probe_mma_peak.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double)]
    lib.ievm_probe_mma_peak.restype = C.c_int
    lib.ievm_set_wait_limit_ms.argtypes = [C.c_int, C.c_int64]
    lib.ievm_set_wait_limit_ms.restype = C.c_int
    for name in ("ievm_forward_i8", "ievm_forward_f16", "ievm_forward_i8_host", "ievm_forward_f16_host",
                 "ievm_set_option", "ievm_num_tensors", "ievm_tensor_shape", "ievm_launches_per_forward",
                 "ievm_debug_read_tensor", "ievm_debug_conv_acc", "ievm_kd_loss"):
        getattr(lib, name).restype = C.c_int
    lib.ievm_last_error.restype = C.c_char_p
    lib.ievm_build_info.restype = C.c_char_p
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().ievm_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (status {rc}): {msg}")
