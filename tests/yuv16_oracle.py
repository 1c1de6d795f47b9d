"""TEST INFRASTRUCTURE ONLY: the numpy statement of the 16-bit-sample YUV 4:2:0 -> RGB conversion
(include/nexar_clip_transform.h, nexar_plan_create_yuv16): P010 / P016 (semi-planar, MSB-aligned) and yuv420p10le
(planar, LSB-aligned 10-bit), every matrix and range, padded surfaces.  Every sample is read as the word
w = (sample << shift) & 0xFFFF and, with the integer coefficients of oracle/yuv420_oracle.py unchanged,

    C = w_Y - (Yo << 8), D = w_U - 32768, E = w_V - 32768
    R = clip((Ys C + Rv E + 32768) >> 16), G = clip((Ys C - Gu D - Gv E + 32768) >> 16), B = clip((Ys C + Bu D + 32768) >> 16)

so words x << 8 give exactly ``yuv420_to_rgb`` of the 8-bit codes x.
"""
import numpy as np

from oracle.yuv420_oracle import yuv_int_coefficients

SAMPLE_SHIFT = {"p010": 0, "i010": 6}


def yuv420_16_to_rgb(buf: np.ndarray, layout: str = "nv12", matrix: str = "bt601", range_: str = "limited",
                     frame_size=None, shift: int = 0) -> np.ndarray:
    """uint16 [..., L*3/2, P] surfaces -> uint8 [..., h, w, 3], addressed as ``yuv420_to_rgb`` with P the pitch in
    samples (layout "nv12": interleaved U V words after the Y plane; "i420": U plane then V plane, [L/2][P/2] each).
    ``frame_size=(h, w)`` is the visible picture (default (L, P)); nothing outside it and its chroma is read."""
    rows, pitch = buf.shape[-2], buf.shape[-1]
    lr = rows * 2 // 3
    h, w = frame_size if frame_size is not None else (lr, pitch)
    lead = buf.shape[:-2]
    words = (buf.astype(np.int64) << shift) & 0xFFFF
    y = words[..., :h, :w]
    chroma = words[..., lr:, :]
    if layout == "nv12":
        uv = chroma[..., : h // 2, :w].reshape(lead + (h // 2, w // 2, 2))
        u, v = uv[..., 0], uv[..., 1]
    elif layout == "i420":
        planes = chroma.reshape(lead + (lr, pitch // 2))        # L/2 rows of P samples = L rows of P/2: U then V
        u = planes[..., : h // 2, : w // 2]
        v = planes[..., lr // 2: lr // 2 + h // 2, : w // 2]
    else:
        raise ValueError(f"unknown layout {layout!r}")
    u = np.repeat(np.repeat(u, 2, axis=-2), 2, axis=-1)
    v = np.repeat(np.repeat(v, 2, axis=-2), 2, axis=-1)
    yo, ys, rv, gu, gv, bu = yuv_int_coefficients(matrix, range_)
    c, d, e = y - (yo << 8), u - 32768, v - 32768
    r = (ys * c + rv * e + 32768) >> 16
    g = (ys * c - gu * d - gv * e + 32768) >> 16
    b = (ys * c + bu * d + 32768) >> 16
    return np.stack([r, g, b], axis=-1).clip(0, 255).astype(np.uint8)
