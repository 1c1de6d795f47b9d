"""TEST INFRASTRUCTURE ONLY (never imported by the product path).

YUV 4:2:0 -> RGB oracle for every supported decoder-surface variant (include/nexar_clip_transform.h, NexarYuvFormat):
NV12 and I420 layouts, BT.601 and BT.709 matrices, limited and full range, padded surfaces.  As for nv12_oracle.py the
conversion is a STATED formula, the classic 8-bit integer form with nearest-neighbour chroma,

    C = Y - Yo, D = U - 128, E = V - 128
    R = clip((Ys C + Rv E + 128) >> 8), G = clip((Ys C - Gu D - Gv E + 128) >> 8), B = clip((Ys C + Bu D + 128) >> 8)

where every integer coefficient is round(256 * c) of the float coefficient derived from the standard's Kr / Kb.  The
BT.601 limited-range instance is nv12_to_rgb's formula.
"""
import numpy as np

KR_KB = {"bt601": (0.299, 0.114), "bt709": (0.2126, 0.0722)}


def yuv_float_coefficients(matrix: str, range_: str):
    """-> (Yo, luma scale, Rv, Gu, Gv, Bu) as floats: R = s (Y - Yo) + Rv E, G = s (Y - Yo) - Gu D - Gv E, B = s (Y - Yo) + Bu D."""
    kr, kb = KR_KB[matrix]
    kg = 1.0 - kr - kb
    if range_ == "limited":
        yo, ys, cs = 16, 255.0 / 219.0, 255.0 / 224.0
    elif range_ == "full":
        yo, ys, cs = 0, 1.0, 1.0
    else:
        raise ValueError(f"unknown range {range_!r}")
    return (yo, ys, 2 * (1 - kr) * cs, 2 * kb * (1 - kb) / kg * cs, 2 * kr * (1 - kr) / kg * cs, 2 * (1 - kb) * cs)


def yuv_int_coefficients(matrix: str, range_: str):
    """-> (Yo, Ys, Rv, Gu, Gv, Bu): every float coefficient as round(256 * c)."""
    yo, *rest = yuv_float_coefficients(matrix, range_)
    return (yo,) + tuple(int(np.floor(256 * c + 0.5)) for c in rest)


def yuv420_to_rgb(buf: np.ndarray, layout: str = "nv12", matrix: str = "bt601", range_: str = "limited",
                  frame_size=None) -> np.ndarray:
    """uint8 [..., L*3/2, P] surfaces -> uint8 [..., h, w, 3].  L = luma rows, P = pitch; ``frame_size=(h, w)`` is the
    visible picture in the top-left corner (default (L, P)).  NV12: UV plane [L/2][P] after the Y plane; I420: U plane
    then V plane, [L/2][P/2] each.  Nothing outside the visible picture and its chroma samples is read."""
    rows, pitch = buf.shape[-2], buf.shape[-1]
    lr = rows * 2 // 3
    h, w = frame_size if frame_size is not None else (lr, pitch)
    lead = buf.shape[:-2]
    y = buf[..., :h, :w].astype(np.int32)
    chroma = buf[..., lr:, :]
    if layout == "nv12":
        uv = chroma[..., : h // 2, :w].reshape(lead + (h // 2, w // 2, 2))
        u, v = uv[..., 0], uv[..., 1]
    elif layout == "i420":
        planes = chroma.reshape(lead + (lr, pitch // 2))        # L/2 rows of P bytes = L rows of P/2 bytes: U then V
        u = planes[..., : h // 2, : w // 2]
        v = planes[..., lr // 2: lr // 2 + h // 2, : w // 2]
    else:
        raise ValueError(f"unknown layout {layout!r}")
    u = np.repeat(np.repeat(u.astype(np.int32), 2, axis=-2), 2, axis=-1)
    v = np.repeat(np.repeat(v.astype(np.int32), 2, axis=-2), 2, axis=-1)
    yo, ys, rv, gu, gv, bu = yuv_int_coefficients(matrix, range_)
    c, d, e = y - yo, u - 128, v - 128
    r = (ys * c + rv * e + 128) >> 8
    g = (ys * c - gu * d - gv * e + 128) >> 8
    b = (ys * c + bu * d + 128) >> 8
    return np.stack([r, g, b], axis=-1).clip(0, 255).astype(np.uint8)
