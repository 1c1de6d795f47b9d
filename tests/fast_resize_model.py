"""The fast resize kernel (resize_fast_kernel in csrc/clip_transform.cu) restated in numpy: which instance launch_all
selects for a letterbox, and the exact bits that instance writes.

Selection: every refusal of build_fast_tables, the source checks of launch_all (uint8 frames, 16-byte aligned base and
row stride), the thread count, the padded tap count ``kx_al``, the 8-byte window rule (AL4) and the compile-time row
strides.  ``select(h, w, cs, stride, base)`` names the cell ``(KX, NT, RS, AL4)``, or why the general kernel runs.

Arithmetic, from the float tap tables ``_lib.aa_taps`` (pinned to ATen elsewhere):
  * taps: ``floor(w * 2^15)`` per output row / column, plus one on the largest remainders up to a sum of 2^15;
  * vertical: ``acc = 128 + sum(q * x)`` over source rows, staged as ``(acc >> 8) & 0xFFFF`` (the value * 128);
  * horizontal: ``S = sum(q' * staged)``, ``r = f32(S) * (f32(scale) * 2^-22)``, scale 1/255 or 1;
  * normalisation ``fmaf(r, nscale, nbias)`` with the nexar_clip_transform constants, emulated exactly;
  * placement: letterbox offsets, the mirror ``x -> cs - 1 - x`` of flipped clips, pads at the normalised zero.
The sums are evaluated in int64, exactly.
"""
from __future__ import annotations

import functools
from typing import NamedTuple, Optional

import numpy as np

from oracle import np_oracle as O

SHIFT = 15
ONE = 1 << SHIFT
MAX_PAIRS = 1024
RS_SPEC = {(14, 256): 3840, (10, 320): 3840, (20, 384): 5760}   # launch_all's NEXAR_FAST_SPEC row strides
F32, F64 = np.float32, np.float64


class Cell(NamedTuple):
    kx: int
    nt: int
    rs: int
    al4: bool

    def probe(self):
        """What nexar_last_resize_kernel reports for this instance."""
        return (1, self.kx, self.nt, self.rs, int(self.al4))


# every instance launch_all can launch (per output type)
INSTANCES = frozenset(
    [Cell(10, nt, 0, al) for nt in (256, 320, 384) for al in (False, True)]
    + [Cell(10, 320, 3840, al) for al in (False, True)]
    + [Cell(kx, nt, 0, False) for kx in (14, 20) for nt in (256, 320, 384)]
    + [Cell(14, 256, 3840, False), Cell(20, 384, 5760, False)])


def quantise(w) -> np.ndarray:
    """quantise_taps: the 15-bit taps of one row, floor(w * 2^15) plus one for the taps with the largest remainders
    (the first of equal ones) until the row sums to 2^15."""
    x = np.ldexp(np.asarray(w, F32).astype(F64), SHIFT)
    q = np.floor(x).astype(np.int64)
    order = np.argsort(-(x - q), kind="stable")
    q[order[:ONE - int(q.sum())]] += 1
    return q


class Axis(NamedTuple):
    start: np.ndarray     # [n_out] first tap
    count: np.ndarray     # [n_out]
    w: np.ndarray         # [n_out, kmax] float32 taps
    q: np.ndarray         # [n_out, kmax] int64 quantised taps (0 past count)
    kmax: int

    def apply(self, x: np.ndarray) -> np.ndarray:
        """sum_k q[i, k] * x[start[i] + k] along the first axis of an int64 array, exactly: one gather per tap
        (elementwise integer arithmetic, no BLAS and so no BLAS thread pool in the test process)."""
        n_in = x.shape[0]
        out = np.zeros((len(self.start),) + x.shape[1:], np.int64)
        shape = (-1,) + (1,) * (x.ndim - 1)
        for k in range(self.kmax):
            out += self.q[:, k].reshape(shape) * x[np.minimum(self.start + k, n_in - 1)]   # q is 0 past count
        return out


@functools.lru_cache(maxsize=None)
def axis(n_in: int, n_out: int) -> Axis:
    from vision_collision_detection_b200 import _lib
    start, count, w = _lib.aa_taps(n_in, n_out)
    q = np.zeros(w.shape, np.int64)
    for i, c in enumerate(count):
        q[i, :c] = quantise(w[i, :c])
    return Axis(start.astype(np.int64), count.astype(np.int64), w, q, w.shape[1])


def geometry(h: int, w: int, cs: int):
    """-> (rh, rw, off_y, off_x) of the letterbox."""
    return O.letterbox_geometry(h, w, cs)


def _vertical_table_refusal(ax: Axis, h: int, rh: int) -> Optional[str]:
    """The per-row refusals of build_fast_tables' pair table (two accumulator slots, rows consumed in pairs)."""
    n_pairs = (h + 1) // 2
    if n_pairs > MAX_PAIRS:
        return "more than 1024 row pairs"
    X = np.zeros(n_pairs + 1, np.int64)
    Y = np.zeros(n_pairs + 1, np.int64)
    Z = np.zeros(n_pairs + 1, np.int64)
    W = np.zeros(n_pairs + 1, np.int64)
    ys, yc = ax.start, ax.count
    for i in range(rh):
        s, c = int(ys[i]), int(yc[i])
        if c <= 0:
            return "empty row"
        if i + 2 < rh and ys[i + 2] < s + c:
            return "three rows alive"
        if i + 1 < rh and ys[i + 1] + yc[i + 1] <= s + c:
            return "rows finish out of order"
        q = ax.q[i, :c]
        if q.min() < 0 or q.max() > 65535:
            return "vertical tap out of range"
        slot = i % 2
        prev_last = int(ys[i - 2] + yc[i - 2] - 1) if i >= 2 else -1
        begun = False
        for k in range(c):
            y = s + k
            p = y // 2
            if prev_last >= 0 and prev_last // 2 == p:
                if not (y & 1) or W[p]:
                    return "post tap"
                W[p] = int(q[k]) << 16
                begun = begun or bool(q[k])
            else:
                ws = Y if slot else X
                if not begun and q[k]:
                    if ws[p]:
                        return "slot restarted twice"
                    Z[p] |= 8 if slot else 4
                    begun = True
                ws[p] |= int(q[k]) << (16 * (y & 1))
        e = (s + c - 1) // 2
        if Z[e] & 1:
            return "two flushes in one pair"
        if i >= 4096:
            return "more than 4096 rows"
        Z[e] |= 1 | (slot << 1) | (i << 4)
    if np.any((W != 0) & ((Z & 1) == 0)):
        return "post tap without a flush"
    return None


class Selection(NamedTuple):
    cell: Optional[Cell]
    reason: str            # why the general kernel runs ("" when the fast one does)


@functools.lru_cache(maxsize=None)
def _fast_tables(h: int, w: int, cs: int):
    """build_fast_tables -> (refusal or None, kx_al, x_align4)."""
    rh, rw, _, _ = geometry(h, w, cs)
    if (w * 3) % 16 or w * 3 // 16 > 384 or h & 1:
        return "row width or odd height", 0, False
    if h < 2 * rh or w < rw:
        return "scale below 2 (rows) or 1 (columns)", 0, False
    if min(rw, cs) > 384:
        return "more than 384 output columns", 0, False
    ay, axx = axis(h, rh), axis(w, rw)
    kx_al = next((k for k in (10, 14, 20) if axx.kmax + 1 <= k), 0)
    if not kx_al:
        return "more than 19 horizontal taps", 0, False
    al4 = kx_al == 10 and bool(np.all(axx.count + (axx.start & 3) <= kx_al))
    wmax = float(ay.w.max())
    if not wmax > 0 or np.ldexp(wmax, SHIFT) > 65535:
        return "vertical tap out of range", 0, False
    why = _vertical_table_refusal(ay, h, rh)
    if why:
        return why, 0, False
    if axx.q.min() < 0 or axx.q.max() > 65535:
        return "horizontal tap out of range", 0, False
    return None, kx_al, al4


def select(h: int, w: int, cs: int, stride: Optional[int] = None, base: int = 0) -> Selection:
    """The resize kernel launch_all runs for an h x w uint8 letterbox to cs with row stride ``stride`` (default packed)
    and the source base address ``base`` (mod 16)."""
    stride = w * 3 if stride is None else stride
    why, kx_al, al4 = _fast_tables(h, w, cs)
    if why:
        return Selection(None, why)
    if stride % 16 or base % 16:
        return Selection(None, "source not 16-byte aligned")
    rh, rw, _, _ = geometry(h, w, cs)
    need = max(w * 3 // 16, min(rw, cs))
    nt = 256 if need <= 256 else 320 if need <= 320 else 384
    rs = stride if RS_SPEC.get((kx_al, nt)) == stride else 0
    return Selection(Cell(kx_al, nt, rs, al4), "")


# ---------------------------------------------------------------------------------------------------------------------
# arithmetic
# ---------------------------------------------------------------------------------------------------------------------
def norm_constants(mean, std):
    """nexar_clip_transform: nscale = f32(1 / (double)std), nbias = f32(-(double)mean / (double)std)."""
    m = np.asarray(mean, F32).astype(F64)
    inv = 1.0 / np.asarray(std, F32).astype(F64)
    return inv.astype(F32), (-m * inv).astype(F32)


def fmaf(a, b, c) -> np.ndarray:
    """float32 fused multiply-add, correctly rounded: the float64 product of two floats is exact; the float64 sum is
    rounded once, and the one case where rounding it again to float32 can go wrong, a float64 sum exactly halfway
    between two floats with a non-zero rounding error, is resolved with the exact error (TwoSum)."""
    p = np.asarray(a, F32).astype(F64) * np.asarray(b, F32).astype(F64)
    c = np.broadcast_to(np.asarray(c, F32).astype(F64), p.shape)
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)
    r = s.astype(F32)
    d = s - r.astype(F64)
    other = np.nextafter(r, np.where(d > 0, np.inf, -np.inf).astype(F32))
    mid = (d != 0) & ((r.astype(F64) + other.astype(F64)) * 0.5 == s)
    fix = mid & (err != 0)
    return np.where(fix, np.where(err > 0, np.maximum(r, other), np.minimum(r, other)), r).astype(F32)


def resample(frames: np.ndarray, h: int, w: int, cs: int, scale_255: bool = True) -> np.ndarray:
    """[T,H,W,3] uint8 -> [3,T,rh,rw] float32: the kernel's value before normalisation."""
    rh, rw, _, _ = geometry(h, w, cs)
    t = frames.shape[0]
    ay, ax = axis(h, rh), axis(w, rw)
    scale = F32(1.0) / F32(255.0) if scale_255 else F32(1.0)
    post = F32(scale * F32(2.0 ** -22))
    out = np.empty((3, t, rh, rw), F32)
    for f in range(t):                                                      # a frame at a time: bounded memory
        x = np.ascontiguousarray(frames[f], np.uint8).reshape(h, w * 3).astype(np.int64)
        staged = ((ay.apply(x) + 128) >> 8) & 0xFFFF                        # [rh, W*3]
        s = ax.apply(staged.reshape(rh, w, 3).transpose(1, 0, 2))          # [rw, rh, 3], < 2^31
        out[:, f] = s.transpose(2, 1, 0).astype(F32) * post
    return out


def fast_resize(frames: np.ndarray, cs: int, *, normalize: bool = True, mean=(0.45,) * 3, std=(0.225,) * 3,
                flip: bool = False, scale_255: bool = True) -> np.ndarray:
    """The fp32 output of the fast kernel for one clip without augmentation: [3, T, cs, cs]."""
    t, h, w, _ = frames.shape
    rh, rw, oy, ox = geometry(h, w, cs)
    r = resample(frames, h, w, cs, scale_255)
    ns, nb = norm_constants(mean, std)
    out = np.zeros((3, t, cs, cs), F32)
    for c in range(3):
        if normalize:
            out[c] = nb[c]
            out[c, :, oy:oy + rh, ox:ox + rw] = fmaf(r[c], ns[c], nb[c])
        else:
            out[c, :, oy:oy + rh, ox:ox + rw] = r[c]
    return np.ascontiguousarray(out[..., ::-1]) if flip else out


def worst_case(h: int, w: int, cs: int) -> float:
    """Upper bound, in 0..255 levels, of |kernel - exact resample with the float taps| over every uint8 content:
    the tap rounding of either pass at its worst sign pattern, the staging rounding (half a step of 1/128) and the
    float conversion and scaling (two roundings of 2^-24 relative)."""
    rh, rw, _, _ = geometry(h, w, cs)

    def taps(ax):
        d = ax.q.astype(F64) / ONE - ax.w.astype(F64)
        return float(max(np.clip(d, 0, None).sum(1).max(), np.clip(-d, 0, None).sum(1).max()))

    return 255.0 * (taps(axis(h, rh)) + taps(axis(w, rw))) + 0.5 / 128 + 255.0 * 2.0 ** -23


# ---------------------------------------------------------------------------------------------------------------------
# content
# ---------------------------------------------------------------------------------------------------------------------
def _rounding_aligned_mask(n_in: int, n_out: int) -> np.ndarray:
    """Source lines (rows or columns) whose quantised tap exceeds the exact one for the output they weigh most."""
    ax = axis(n_in, n_out)
    best = np.full(n_in, -1.0)
    up = np.zeros(n_in, bool)
    for i, (s, c) in enumerate(zip(ax.start, ax.count)):
        for k in range(c):
            wv = float(ax.w[i, k])
            if wv > best[s + k]:
                best[s + k] = wv
                up[s + k] = ax.q[i, k] > wv * ONE
    return up


def adversarial(h: int, w: int, cs: int) -> dict:
    """uint8 [H,W,3] frames that drive the fixed-point rounding: 0/255 stripes of period 1 and 2 on both axes, all-255
    and the 'rounding-aligned' lines (rows, columns and their intersection)."""
    rh, rw, _, _ = geometry(h, w, cs)
    yy, xx = np.arange(h)[:, None], np.arange(w)[None, :]
    ry = _rounding_aligned_mask(h, rh)[:, None]
    rx = _rounding_aligned_mask(w, rw)[None, :]
    pats = {
        "rows_p1": (yy & 1) == 1, "rows_p2": (yy >> 1 & 1) == 1, "cols_p1": (xx & 1) == 1, "cols_p2": (xx >> 1 & 1) == 1,
        "all255": np.ones((h, w), bool), "aligned_rows": ry & (xx >= 0), "aligned_cols": rx & (yy >= 0),
        "aligned_both": ry & rx,
    }
    return {k: np.repeat((np.broadcast_to(v, (h, w)) * np.uint8(255)).astype(np.uint8)[..., None], 3, axis=2)
            for k, v in pats.items()}


def noise(h: int, w: int, seed: int) -> np.ndarray:
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)
