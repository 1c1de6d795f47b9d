"""Deterministic synthetic dashcam clips (integer arithmetic only, so numpy on
the host and torch on the device produce identical bytes).

Two distributions (SURVEY.md section 8d): ``noise`` — i.i.d. uniform bytes, the
worst case for antialiased-resize parity; ``dashcam`` — sky-to-road vertical
gradient, lane/horizon block structure drifting with time, and +-16 noise.
"""
from __future__ import annotations

import numpy as np

_M32 = 0xFFFFFFFF


def _hash32(idx, seed: int):
    """32-bit integer hash evaluated in 64-bit integers (works for numpy int64
    arrays and torch int64 tensors alike; only the low 32 bits are kept)."""
    x = (idx * 2654435761 + (seed * 40503 + 0x9E3779B9)) & _M32
    x = x ^ (x >> 15)
    x = (x * 2246822519) & _M32
    x = x ^ (x >> 13)
    x = (x * 3266489917) & _M32
    x = x ^ (x >> 16)
    return x


def _pattern(t, y, x, c, h: int, seed: int, kind: str, lin):
    noise = _hash32(lin, seed)
    if kind == "noise":
        return noise & 0xFF
    if kind != "dashcam":
        raise ValueError(f"unknown synthetic kind {kind!r}")
    sky = 215 - (y * 150) // max(h, 1)
    blocks = (((x + 3 * t) // 32 + y // 24) % 2) * 28
    lane = ((x + y // 2 + 5 * t) % 160 < 6) * 40
    tint = c * 9
    v = sky + blocks + lane - tint + (noise & 31) - 16
    return v.clip(0, 255) if hasattr(v, "clip") else v.clamp(0, 255)


def make_clip_np(t: int, h: int, w: int, seed: int = 0, kind: str = "noise") -> np.ndarray:
    """uint8 [T,H,W,3] on the host."""
    tt, yy, xx, cc = np.meshgrid(np.arange(t, dtype=np.int64), np.arange(h, dtype=np.int64),
                                 np.arange(w, dtype=np.int64), np.arange(3, dtype=np.int64), indexing="ij")
    lin = ((tt * h + yy) * w + xx) * 3 + cc
    return _pattern(tt, yy, xx, cc, h, seed, kind, lin).astype(np.uint8)


def make_clip_torch(t: int, h: int, w: int, seed: int = 0, kind: str = "noise", device="cuda"):
    """uint8 [T,H,W,3] generated on ``device`` (same bytes as make_clip_np)."""
    import torch

    ar = lambda n: torch.arange(n, dtype=torch.int64, device=device)
    tt = ar(t).view(t, 1, 1, 1)
    yy = ar(h).view(1, h, 1, 1)
    xx = ar(w).view(1, 1, w, 1)
    cc = ar(3).view(1, 1, 1, 3)
    lin = ((tt * h + yy) * w + xx) * 3 + cc
    return _pattern(tt, yy, xx, cc, h, seed, kind, lin).to(torch.uint8)


def rgb_to_nv12(clip):
    """Synthetic decoder surfaces from RGB frames: uint8 ``[...,H,W,3]`` -> uint8 ``[...,H*3/2,W]`` (Y plane, then the
    interleaved UV plane of the 2 x 2 block means), BT.601 limited range in the usual 8-bit integer form
    (Y = ((66R + 129G + 25B + 128) >> 8) + 16, U = ((-38R - 74G + 112B + 128) >> 8) + 128, V = ((112R - 94G - 18B + 128) >> 8) + 128).
    Works on numpy arrays and torch tensors (integer arithmetic only, identical bytes)."""
    is_np = isinstance(clip, np.ndarray)
    x = clip.astype(np.int32) if is_np else clip.int()
    r, g, b = x[..., 0], x[..., 1], x[..., 2]
    y = ((66 * r + 129 * g + 25 * b + 128) >> 8) + 16
    h, w = y.shape[-2], y.shape[-1]
    if h % 2 or w % 2:
        raise ValueError("nv12 needs an even height and width")

    def blocks(v):  # mean of each 2 x 2 block, rounded
        v = v.reshape(v.shape[:-2] + (h // 2, 2, w // 2, 2))
        return (v.sum(axis=-1).sum(axis=-2) + 2) >> 2 if is_np else (v.sum(dim=-1).sum(dim=-2) + 2) >> 2

    rm, gm, bm = blocks(r), blocks(g), blocks(b)
    u = ((-38 * rm - 74 * gm + 112 * bm + 128) >> 8) + 128
    v = ((112 * rm - 94 * gm - 18 * bm + 128) >> 8) + 128
    if is_np:
        uv = np.stack([u, v], axis=-1).reshape(u.shape[:-1] + (w,))
        return np.concatenate([y, uv], axis=-2).clip(0, 255).astype(np.uint8)
    import torch
    uv = torch.stack([u, v], dim=-1).reshape(u.shape[:-1] + (w,))
    return torch.cat([y, uv], dim=-2).clamp(0, 255).to(torch.uint8)


def rgb_to_yuv420(clip: np.ndarray, layout: str = "nv12", matrix: str = "bt601", range_: str = "limited",
                  luma_rows: int = None, pitch: int = None) -> np.ndarray:
    """Synthetic decoder surfaces of any supported 4:2:0 variant: uint8 ``[...,H,W,3]`` -> uint8 ``[...,L*3/2,P]``
    (``L = luma_rows`` >= H, ``P = pitch`` >= W, both default to the picture size; NV12: Y plane then the interleaved
    UV plane, I420: Y, U and V planes; include/nexar_clip_transform.h).  The encode is the float64 one of the
    standard with 2 x 2 chroma means, rounded to bytes; every padding byte is 255, so a reader that strays into the
    padding shows."""
    kr, kb = {"bt601": (0.299, 0.114), "bt709": (0.2126, 0.0722)}[matrix]
    if range_ not in ("limited", "full") or layout not in ("nv12", "i420"):
        raise ValueError(f"unknown range or layout: {range_!r}, {layout!r}")
    x = clip.astype(np.float64)
    h, w = x.shape[-3], x.shape[-2]
    lr = h if luma_rows is None else luma_rows
    p = w if pitch is None else pitch
    if h % 2 or w % 2 or lr % 2 or lr < h or p < w or (layout == "i420" and p % 2):
        raise ValueError(f"bad surface: picture {h}x{w}, luma rows {lr}, pitch {p}")
    yv = kr * x[..., 0] + (1 - kr - kb) * x[..., 1] + kb * x[..., 2]
    blk = x.reshape(x.shape[:-3] + (h // 2, 2, w // 2, 2, 3)).mean(axis=(-4, -2))
    ym = kr * blk[..., 0] + (1 - kr - kb) * blk[..., 1] + kb * blk[..., 2]
    pb = (blk[..., 2] - ym) / (2 * (1 - kb))
    pr = (blk[..., 0] - ym) / (2 * (1 - kr))
    if range_ == "limited":
        y, u, v = 16 + yv * 219 / 255, 128 + pb * 224 / 255, 128 + pr * 224 / 255
    else:
        y, u, v = yv, 128 + pb, 128 + pr
    q = lambda a: np.clip(np.floor(a + 0.5), 0, 255).astype(np.uint8)
    lead = x.shape[:-3]
    out = np.full(lead + (lr * 3 // 2, p), 255, np.uint8)
    out[..., :h, :w] = q(y)
    if layout == "nv12":
        out[..., lr: lr + h // 2, :w] = np.stack([q(u), q(v)], axis=-1).reshape(lead + (h // 2, w))
    else:
        planes = np.full(lead + (lr, p // 2), 255, np.uint8)    # U plane rows, then V plane rows, P/2 bytes each
        planes[..., : h // 2, : w // 2] = q(u)
        planes[..., lr // 2: lr // 2 + h // 2, : w // 2] = q(v)
        out[..., lr:, :] = planes.reshape(lead + (lr // 2, p))
    return out


def rgb_to_yuv420_16(clip: np.ndarray, layout: str = "p010", matrix: str = "bt601", range_: str = "limited",
                     luma_rows: int = None, pitch: int = None) -> np.ndarray:
    """Synthetic 10-bit decoder surfaces: uint8 ``[...,H,W,3]`` -> uint16 ``[...,L*3/2,P]`` (``P`` the pitch in samples),
    ``layout`` "p010" (semi-planar, the 10 bits in the high bits of each word) or "i010" (planar, the 10 bits in the low
    bits: yuv420p10le).  The encode is the float64 one of ``rgb_to_yuv420`` at 10-bit precision, a 10-bit code being
    4 x the 8-bit one (limited range: Y in [64, 940]); every padding sample is 0xFFFF."""
    if layout not in ("p010", "i010") or range_ not in ("limited", "full"):
        raise ValueError(f"unknown range or layout: {range_!r}, {layout!r}")
    kr, kb = {"bt601": (0.299, 0.114), "bt709": (0.2126, 0.0722)}[matrix]
    x = clip.astype(np.float64)
    h, w = x.shape[-3], x.shape[-2]
    lr = h if luma_rows is None else luma_rows
    p = w if pitch is None else pitch
    if h % 2 or w % 2 or lr % 2 or lr < h or p < w or p % 2:
        raise ValueError(f"bad surface: picture {h}x{w}, luma rows {lr}, pitch {p}")
    yv = kr * x[..., 0] + (1 - kr - kb) * x[..., 1] + kb * x[..., 2]
    blk = x.reshape(x.shape[:-3] + (h // 2, 2, w // 2, 2, 3)).mean(axis=(-4, -2))
    ym = kr * blk[..., 0] + (1 - kr - kb) * blk[..., 1] + kb * blk[..., 2]
    pb = (blk[..., 2] - ym) / (2 * (1 - kb))
    pr = (blk[..., 0] - ym) / (2 * (1 - kr))
    if range_ == "limited":
        y, u, v = 16 + yv * 219 / 255, 128 + pb * 224 / 255, 128 + pr * 224 / 255
    else:
        y, u, v = yv, 128 + pb, 128 + pr
    shift = 6 if layout == "p010" else 0
    q = lambda a: (np.clip(np.floor(4 * a + 0.5), 0, 1023).astype(np.uint16) << shift).astype(np.uint16)
    lead = x.shape[:-3]
    out = np.full(lead + (lr * 3 // 2, p), 0xFFFF, np.uint16)
    out[..., :h, :w] = q(y)
    if layout == "p010":
        out[..., lr: lr + h // 2, :w] = np.stack([q(u), q(v)], axis=-1).reshape(lead + (h // 2, w))
    else:
        planes = np.full(lead + (lr, p // 2), 0xFFFF, np.uint16)   # U plane rows, then V plane rows, P/2 samples each
        planes[..., : h // 2, : w // 2] = q(u)
        planes[..., lr // 2: lr // 2 + h // 2, : w // 2] = q(v)
        out[..., lr:, :] = planes.reshape(lead + (lr // 2, p))
    return out
