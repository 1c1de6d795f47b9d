"""The source formats of the clip transform, and the only module that knows their rules: which frame tensors a format
takes (``SourceFormat``) and how the library reads such a frame (``FrameSource``, ``PlanKey``)."""
from __future__ import annotations

import functools
from typing import NamedTuple, Optional, Tuple

import numpy as np
import torch

from . import _lib

# name -> (NexarYuvFormat layout, sample shift: the left shift that puts a 16-bit sample at the top of its word, P010 /
# P016 being MSB-aligned already and yuv420p10le keeping its 10 bits in the low bits; None for 8-bit samples)
_YUV = {"nv12": (_lib.YUV_NV12, None), "i420": (_lib.YUV_I420, None),
        "p010": (_lib.YUV_NV12, 0), "i010": (_lib.YUV_I420, 6)}
_MATRIX = {"bt601": _lib.YUV_BT601, "bt709": _lib.YUV_BT709}
_RANGE = {"limited": _lib.YUV_LIMITED, "full": _lib.YUV_FULL}
PIXEL_FORMATS = ("rgb",) + tuple(_YUV)


class PlanKey(NamedTuple):
    """The plan's library call: ``nexar_plan_create(geom, src)`` if ``yuv`` (the ``NexarYuvFormat``) is None, else
    ``nexar_plan_create_yuv(geom, yuv)`` or ``nexar_plan_create_yuv16(geom, yuv, sample_shift)``."""
    src: int
    pixel_bytes: int        # of a pixel in a row of the RGB frame or of the Y plane
    yuv: Optional[Tuple[int, int, int, int]] = None
    sample_shift: Optional[int] = None


RGB_U8 = PlanKey(_lib.SRC_U8, 3)
RGB_F32 = PlanKey(_lib.SRC_F32, 12)
_RGB_KEYS = {torch.uint8: RGB_U8, torch.float32: RGB_F32}
# nexar_plan_create serves NV12 BT.601 limited range without padded luma rows also in libraries without the YUV calls
_NV12_KEY = PlanKey(_lib.SRC_NV12, 1)


class FrameSource(NamedTuple):
    """A frame as the kernels read it; sources are equal when their format, shape, dtype and ``frame_size`` are."""
    format: SourceFormat
    shape: Tuple[int, ...]
    dtype: torch.dtype
    frame_size: Optional[Tuple[int, int]]
    h: int                  # the visible picture
    w: int
    frame_bytes: int
    row_stride: int
    plan_key: PlanKey


class SourceFormat(NamedTuple):
    """The validated source-format keywords of ``forward_batch`` (``SourceFormat.of``); ``_asdict()`` returns them."""
    pixel_format: str
    color_matrix: str
    color_range: str

    @staticmethod
    @functools.lru_cache(maxsize=None)
    def of(pixel_format: str = "rgb", color_matrix: str = "bt601", color_range: str = "limited") -> SourceFormat:
        if pixel_format not in PIXEL_FORMATS:
            raise ValueError(f"unknown pixel_format {pixel_format!r}; expected one of {PIXEL_FORMATS}")
        if color_matrix not in _MATRIX:
            raise ValueError(f"unknown color_matrix {color_matrix!r}; expected one of {tuple(_MATRIX)}")
        if color_range not in _RANGE:
            raise ValueError(f"unknown color_range {color_range!r}; expected one of {tuple(_RANGE)}")
        return SourceFormat(pixel_format, color_matrix, color_range)

    @property
    def yuv(self) -> bool:
        return self.pixel_format != "rgb"

    @property
    def dtype(self) -> torch.dtype:
        """The element type of decoded frames."""
        return torch.uint16 if self.yuv and _YUV[self.pixel_format][1] is not None else torch.uint8

    def frame_shape(self, h: int, w: int) -> Tuple[int, ...]:
        """The shape of an unpadded frame of an ``h x w`` picture."""
        return (h * 3 // 2, w) if self.yuv else (h, w, 3)

    def blank_frame(self, shape) -> np.ndarray:
        """A frame that converts to RGB zeros: zero bytes for RGB; for a YUV surface Y = 16 (limited range) or 0 (full
        range) and U = V = 128 (zero bytes there would be a strongly coloured picture), in the format's sample scale."""
        if not self.yuv:
            return np.zeros(shape, np.uint8)
        shift = _YUV[self.pixel_format][1]
        scale = 1 if shift is None else 1 << (8 - shift)
        f = np.full(shape, 128 * scale, np.uint8 if shift is None else np.uint16)
        f[: shape[0] * 2 // 3] = 16 * scale if self.color_range == "limited" else 0
        return f

    def describe(self, frame_shape, dtype: torch.dtype, frame_size=None, *, decoded: bool = False) -> FrameSource:
        """Checks a frame ``[H,W,3]`` (RGB: uint8 or float32) or ``[R,P]`` (YUV) and the ``frame_size`` of a surface ->
        its ``FrameSource``.  ``decoded``: frames as a decoder delivers them, no float32 RGB, floats are a TypeError."""
        frame_size = None if frame_size is None else (int(frame_size[0]), int(frame_size[1]))
        return _describe(self, frame_shape, dtype, frame_size, decoded)


@functools.lru_cache(maxsize=1024)      # a stream describes every chunk: the same few sources over and over
def _describe(fmt: SourceFormat, frame_shape, dtype: torch.dtype, frame_size, decoded: bool) -> FrameSource:
    if decoded and dtype.is_floating_point:
        raise TypeError(f"decoded {fmt.pixel_format} frames are {fmt.dtype}, got {dtype}")
    if not fmt.yuv:
        if len(frame_shape) != 3 or frame_shape[2] != 3:
            raise ValueError(f"rgb frames are [H,W,3], got frames of shape {tuple(frame_shape)}")
        if frame_size is not None:
            raise ValueError(f"frame_size is the visible picture of YUV surfaces; rgb frames have no padding, got "
                             f"frame_size {frame_size}")
        key = _RGB_KEYS.get(dtype)
        if key is None:             # uint16 is a ValueError: 16-bit YUV surfaces without their pixel_format
            error = ValueError if decoded or dtype == torch.uint16 else TypeError
            raise error(f"rgb frames are torch.uint8{'' if decoded else ' or torch.float32'}, got {dtype}")
        h, w = frame_shape[0], frame_shape[1]
    else:
        if len(frame_shape) != 2 or dtype != fmt.dtype or frame_shape[0] % 3 or frame_shape[1] % 2:
            raise ValueError(f"{fmt.pixel_format} frames are {fmt.dtype} [H*3/2,W] surfaces with even H and W, got "
                             f"{dtype} frames of shape {tuple(frame_shape)}")
        luma_rows, pitch = frame_shape[0] * 2 // 3, frame_shape[1]
        h, w = frame_size or (luma_rows, pitch)
        if h <= 0 or w <= 0 or h % 2 or w % 2 or h > luma_rows or w > pitch:
            raise ValueError(f"frame_size {(h, w)} of {fmt.pixel_format} surfaces must be even and fit the {luma_rows} "
                             f"luma rows x {pitch} pitch surface")
        layout, shift = _YUV[fmt.pixel_format]
        if fmt == ("nv12", "bt601", "limited") and h == luma_rows:
            key = _NV12_KEY
        else:
            key = PlanKey(_lib.SRC_NV12, 1 if shift is None else 2,
                          (layout, _MATRIX[fmt.color_matrix], _RANGE[fmt.color_range], luma_rows), shift)
    row = frame_shape[1] * key.pixel_bytes
    return FrameSource(fmt, tuple(frame_shape), dtype, frame_size, h, w, frame_shape[0] * row, row, key)
