"""ctypes binding of libnexar_clip_b200.so (include/nexar_clip_transform.h).

There is no CPU fallback: if the CUDA library cannot be loaded (and cannot be
built because nvcc is absent) importing the product path raises.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

import numpy as np

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT_DIR = os.path.dirname(PKG_DIR)
LIB_PATH = os.environ.get("NEXAR_LIB") or os.path.join(PKG_DIR, "libnexar_clip_b200.so")  # NEXAR_LIB: experiment builds
SOURCES = [os.path.join(PKG_DIR, "csrc", "clip_transform.cu")]
HEADERS = [os.path.join(ROOT_DIR, "include", "nexar_clip_transform.h")]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-shared", "-Xcompiler", "-fPIC", "-diag-suppress", "550"]

NEXAR_ABI_VERSION = 1
OK, ERR_INVALID, ERR_CUDA, ERR_WORKSPACE, ERR_UNSUPPORTED = 0, -1, -2, -3, -4
SRC_U8, SRC_F32, SRC_NV12 = 0, 1, 2
YUV_NV12, YUV_I420 = 0, 1
YUV_BT601, YUV_BT709 = 0, 1
YUV_LIMITED, YUV_FULL = 0, 1
DST_F32, DST_BF16, DST_F16 = 0, 1, 2
FLIP, AUG, AFFINE, GRAYSCALE, NOISE, BLUR, POSTERIZE, SOLARIZE, INVERT, CUTOUT, RANGE_255 = (1 << i for i in range(11))
MAX_CUTOUT = 8
MAX_BLUR_TAPS = 33

CLIP_PARAMS_DTYPE = np.dtype([
    ("flags", "<u4"), ("crop_dy", "<i4"), ("crop_dx", "<i4"),
    ("brightness", "<f4"), ("contrast", "<f4"), ("contrast_q", "<f4"),
    ("saturation", "<f4"), ("saturation_q", "<f4"), ("hue", "<f4"),
    ("grid", "<f4", (6,)), ("solarize_threshold", "<f4"), ("posterize_bits", "<i4"),
    ("noise_level", "<f4"), ("noise_seed", "<u4", (2,)), ("blur_ksize", "<i4"),
    ("blur_taps", "<f4", (MAX_BLUR_TAPS,)), ("n_cutout", "<i4"), ("cutout", "<i4", (MAX_CUTOUT, 4)),
])


class Geometry(C.Structure):
    _fields_ = [("src_h", C.c_int32), ("src_w", C.c_int32), ("canvas", C.c_int32),
                ("resize_h", C.c_int32), ("resize_w", C.c_int32), ("off_y", C.c_int32), ("off_x", C.c_int32)]

    def as_tuple(self):
        return (self.src_h, self.src_w, self.canvas, self.resize_h, self.resize_w, self.off_y, self.off_x)


class TransformArgs(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("n_clips", C.c_int32), ("frames_per_clip", C.c_int32),
                ("src", C.c_void_p), ("frame_offsets", C.c_void_p), ("src_row_stride", C.c_int64),
                ("params", C.c_void_p), ("any_flags", C.c_uint32), ("dst", C.c_void_p),
                ("dst_dtype", C.c_int32), ("normalize", C.c_int32), ("dst_stride", C.c_int64 * 5),
                ("mean", C.c_float * 3), ("std", C.c_float * 3),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t), ("stream", C.c_void_p)]


class YuvFormat(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("layout", C.c_int32), ("matrix", C.c_int32), ("range", C.c_int32),
                ("luma_rows", C.c_int32)]


class NexarError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libnexar_clip_b200 error {code}: {msg}")
        self.code = code


def needs_build() -> bool:
    if not os.path.isfile(LIB_PATH):
        return True
    if os.environ.get("NEXAR_LIB"):      # an experiment build is used as it is, never rebuilt from the current sources
        return False
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(s) > t for s in SOURCES + HEADERS if os.path.isfile(s))


def build_library(force: bool = False, verbose: bool = False) -> str:
    """nvcc -> libnexar_clip_b200.so, in tree (cross-compiles without a GPU)."""
    if not force and not needs_build():
        return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.isfile(nvcc):
        raise RuntimeError("libnexar_clip_b200.so is missing/stale and nvcc was not found; there is no CPU fallback")
    cmd = [nvcc] + NVCC_FLAGS + ["-I", os.path.join(ROOT_DIR, "include"), "-o", LIB_PATH] + SOURCES
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return LIB_PATH


_lib = None


def lib():
    """Load (building first if the sources are newer and nvcc exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if needs_build():
        build_library()
    L = C.CDLL(LIB_PATH)
    L.nexar_abi_version.restype = C.c_int
    L.nexar_sizeof_clip_params.restype = C.c_size_t
    L.nexar_sizeof_transform_args.restype = C.c_size_t
    L.nexar_last_error.restype = C.c_char_p
    L.nexar_letterbox_geometry.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.POINTER(Geometry)]
    L.nexar_resize_crop_geometry.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(Geometry)]
    L.nexar_aa_taps.argtypes = [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                C.POINTER(C.c_int32)]
    L.nexar_plan_create.argtypes = [C.POINTER(Geometry), C.c_int32, C.POINTER(C.c_void_p)]
    L.nexar_plan_destroy.argtypes = [C.c_void_p]
    L.nexar_plan_destroy.restype = None
    L.nexar_plan_geometry.argtypes = [C.c_void_p, C.POINTER(Geometry)]
    L.nexar_workspace_bytes.argtypes = [C.c_void_p, C.c_int32, C.c_int32]
    L.nexar_workspace_bytes.restype = C.c_size_t
    L.nexar_workspace_bytes_for.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_uint32]
    L.nexar_workspace_bytes_for.restype = C.c_size_t
    L.nexar_clip_transform.argtypes = [C.c_void_p, C.POINTER(TransformArgs)]
    L.nexar_last_launch_count.restype = C.c_int
    L.nexar_gather_windows.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p]
    L.nexar_set_resize_kernel.argtypes = [C.c_int32]
    L.nexar_set_fast_bands.argtypes = [C.c_int32]
    L.nexar_set_geometry_kernel.argtypes = [C.c_int32]
    L.nexar_set_chunk_clips.argtypes = [C.c_int32]
    L.nexar_profile_begin.argtypes = [C.c_int32]
    L.nexar_profile_end.argtypes = [C.c_void_p, C.c_int32]
    if L.nexar_abi_version() != NEXAR_ABI_VERSION:
        raise RuntimeError("libnexar_clip_b200.so ABI version mismatch")
    if L.nexar_sizeof_clip_params() != CLIP_PARAMS_DTYPE.itemsize:
        raise RuntimeError("NexarClipParams layout mismatch between the header and the Python binding")
    if L.nexar_sizeof_transform_args() != C.sizeof(TransformArgs):
        raise RuntimeError("NexarTransformArgs layout mismatch between the header and the Python binding")
    _lib = L
    return L


_yuv_bound = False


def yuv_lib():
    """``lib()`` with the YUV 4:2:0 entry points bound.  They are bound on first use only, so that a library built
    before they existed (selected with NEXAR_LIB) still loads and serves every other call."""
    global _yuv_bound
    L = lib()
    if not _yuv_bound:
        L.nexar_plan_create_yuv.argtypes = [C.POINTER(Geometry), C.POINTER(YuvFormat), C.POINTER(C.c_void_p)]
        L.nexar_yuv_coefficients.argtypes = [C.c_int32, C.c_int32, C.c_void_p]
        L.nexar_sizeof_yuv_format.restype = C.c_size_t
        if L.nexar_sizeof_yuv_format() != C.sizeof(YuvFormat):
            raise RuntimeError("NexarYuvFormat layout mismatch between the header and the Python binding")
        _yuv_bound = True
    return L


_yuv16_bound = False


def yuv16_lib():
    """``yuv_lib()`` with ``nexar_plan_create_yuv16`` bound (16-bit P010 / I010 surfaces), on first use only: a library
    built before it existed serves every 8-bit format and refuses the 16-bit ones with this error."""
    global _yuv16_bound
    L = yuv_lib()
    if not _yuv16_bound:
        try:
            fn = L.nexar_plan_create_yuv16
        except AttributeError:
            raise RuntimeError(f"{LIB_PATH} predates 16-bit YUV surfaces (no nexar_plan_create_yuv16); rebuild it to "
                               "convert p010 / i010 frames") from None
        fn.argtypes = [C.POINTER(Geometry), C.POINTER(YuvFormat), C.c_int32, C.POINTER(C.c_void_p)]
        _yuv16_bound = True
    return L


_ring_bound = False


def ring_lib():
    """``lib()`` with ``nexar_gather_windows_ring`` bound, on first use only: a library built before it existed serves
    every other call and refuses window streams with this error."""
    global _ring_bound
    L = lib()
    if not _ring_bound:
        try:
            fn = L.nexar_gather_windows_ring
        except AttributeError:
            raise RuntimeError(f"{LIB_PATH} predates window streams (no nexar_gather_windows_ring); rebuild it to "
                               "stream sliding windows") from None
        fn.argtypes = [C.c_void_p, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_int64,
                       C.c_void_p, C.c_void_p]
        _ring_bound = True
    return L


_table_bound = False


def table_lib():
    """``lib()`` with ``nexar_gather_windows_table`` bound, on first use only: a library built before it existed serves
    every other call and refuses multi-stream windows with this error."""
    global _table_bound
    L = lib()
    if not _table_bound:
        try:
            fn = L.nexar_gather_windows_table
        except AttributeError:
            raise RuntimeError(f"{LIB_PATH} predates multi-stream windows (no nexar_gather_windows_table); rebuild it to "
                               "serve many streams") from None
        fn.argtypes = [C.c_void_p, C.c_int32, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                       C.c_void_p]
        _table_bound = True
    return L


_probe_bound = False


def last_resize_kernel():
    """-> (fast, KX, NT, RS, AL4) of the resize kernel the last transform call on this thread launched (all 0 for the
    general kernel).  Bound on first use only: a library built before it existed serves every other call."""
    global _probe_bound
    L = lib()
    if not _probe_bound:
        try:
            fn = L.nexar_last_resize_kernel
        except AttributeError:
            raise RuntimeError(f"{LIB_PATH} predates the resize instance probe (no nexar_last_resize_kernel); "
                               "rebuild it") from None
        fn.argtypes = [C.c_void_p]
        _probe_bound = True
    out = (C.c_int32 * 5)()
    check(L.nexar_last_resize_kernel(out))
    return tuple(int(v) for v in out)


def yuv_coefficients(matrix: int, range_: int):
    """-> (Yo, Ys, Rv, Gu, Gv, Bu), the integer conversion coefficients the library uses."""
    out = (C.c_int32 * 6)()
    check(yuv_lib().nexar_yuv_coefficients(matrix, range_, out))
    return tuple(int(v) for v in out)


def check(code: int):
    if code != OK:
        raise NexarError(code, lib().nexar_last_error().decode())


def letterbox_geometry(h: int, w: int, cs: int) -> Geometry:
    g = Geometry()
    check(lib().nexar_letterbox_geometry(h, w, cs, C.byref(g)))
    return g


def resize_crop_geometry(h: int, w: int, size: int, cs: int) -> Geometry:
    g = Geometry()
    check(lib().nexar_resize_crop_geometry(h, w, size, cs, C.byref(g)))
    return g


def aa_taps(in_size: int, out_size: int, cap: int = 64):
    start = np.zeros(out_size, np.int32)
    count = np.zeros(out_size, np.int32)
    wts = np.zeros((out_size, cap), np.float32)
    k = C.c_int32(0)
    check(lib().nexar_aa_taps(in_size, out_size, start.ctypes.data, count.ctypes.data, wts.ctypes.data, cap, C.byref(k)))
    return start, count, wts[:, :k.value].copy()


def profile_end(cap: int = 1 << 16):
    """-> list of per-call durations (ms) of the resize kernel since nexar_profile_begin."""
    buf = np.zeros(cap, np.float32)
    n = lib().nexar_profile_end(buf.ctypes.data, cap)
    return [float(x) for x in buf[:n]]
