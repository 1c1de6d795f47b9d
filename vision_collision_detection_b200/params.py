"""Host-side random decisions of the clip transform.

The reference draws every augmentation decision from Python's global ``random``
(Mersenne Twister) in a fixed order (SURVEY.md section 8a row R0):
``nexar_video_aug.py:748`` flip, then ``:112-180`` the VideoAugmentation block.
Keeping the draws on the host, from the same generator and in the same order,
makes flip decisions, crop offsets and every jitter factor bit-exact by
construction; the GPU only ever sees the resulting numbers, packed one
``NexarClipParams`` (include/nexar_clip_transform.h) per clip.
"""
from __future__ import annotations

import math
import random as _random
from typing import Any, Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib

F32 = np.float32


class VideoAugmentation:
    """Parameter sampler with the constructor signature and draw order of the
    reference's ``VideoAugmentation`` (nexar_video_aug.py:18-182).  The pixel
    work itself happens in the CUDA kernels."""

    def __init__(self, brightness_range=(1.0, 1.0), contrast_range=(1.0, 1.0), saturation_range=(1.0, 1.0),
                 hue_range=(0.0, 0.0), rotation_range=(0.0, 0.0), scale_range=(1.0, 1.0), shear_range=(0.0, 0.0),
                 translate_range=(0.0, 0.0), grayscale_prob=0.0, noise_level=0.0, blur_sigma=0.0,
                 cutout_prob=0.0, cutout_count_range=(1, 3), cutout_size_range=(0.1, 0.2),
                 color_inversion_prob=0.0, solarization_prob=0.0, solarization_threshold=0.5,
                 posterization_prob=0.0, posterization_bits_range=(3, 6), aug_probability=1.0, debug=False):
        self.brightness_range = brightness_range
        self.contrast_range = contrast_range
        self.saturation_range = saturation_range
        self.hue_range = hue_range
        self.rotation_range = rotation_range
        self.scale_range = scale_range
        self.shear_range = shear_range
        self.translate_range = translate_range
        self.grayscale_prob = grayscale_prob
        self.noise_level = noise_level
        self.blur_sigma = blur_sigma
        self.cutout_prob = cutout_prob
        self.cutout_count_range = cutout_count_range
        self.cutout_size_range = cutout_size_range
        self.color_inversion_prob = color_inversion_prob
        self.solarization_prob = solarization_prob
        self.solarization_threshold = solarization_threshold
        self.posterization_prob = posterization_prob
        self.posterization_bits_range = posterization_bits_range
        self.aug_probability = aug_probability
        self.debug = debug

    def _sample_augmentation_parameters(self, shape, rng=_random) -> Dict[str, Any]:
        """Same keys, same draw order as nexar_video_aug.py:97-182."""
        _, _, h, w = shape
        if rng.random() > self.aug_probability:
            return {"skip_augmentation": True}
        u = rng.uniform
        p: Dict[str, Any] = {
            "brightness": u(self.brightness_range[0], self.brightness_range[1]),
            "contrast": u(self.contrast_range[0], self.contrast_range[1]),
            "saturation": u(self.saturation_range[0], self.saturation_range[1]),
            "hue": u(self.hue_range[0], self.hue_range[1]),
            "rotation": u(self.rotation_range[0], self.rotation_range[1]),
            "scale": u(self.scale_range[0], self.scale_range[1]),
            "shear": u(self.shear_range[0], self.shear_range[1]),
        }
        p["translate_x"] = u(-self.translate_range[1], self.translate_range[1]) * w
        p["translate_y"] = u(-self.translate_range[1], self.translate_range[1]) * h
        p["apply_affine"] = bool(p["rotation"] != 0 or p["scale"] != 1 or p["shear"] != 0
                                 or p["translate_x"] != 0 or p["translate_y"] != 0)
        p["apply_grayscale"] = rng.random() < self.grayscale_prob
        p["apply_noise"] = self.noise_level > 0
        p["apply_blur"] = self.blur_sigma > 0
        p["apply_cutout"] = rng.random() < self.cutout_prob
        if p["apply_cutout"]:
            p["cutout_count"] = rng.randint(self.cutout_count_range[0], self.cutout_count_range[1])
            boxes = []
            for _ in range(p["cutout_count"]):
                frac = u(self.cutout_size_range[0], self.cutout_size_range[1])
                cut_h, cut_w = int(h * frac), int(w * frac)
                max_top, max_left = max(0, h - cut_h - 1), max(0, w - cut_w - 1)
                if max_top > 0 and max_left > 0:
                    top = rng.randint(0, max_top)
                    boxes.append((top, rng.randint(0, max_left), cut_h, cut_w))
            p["cutout_boxes"] = boxes
        p["apply_color_inversion"] = rng.random() < self.color_inversion_prob
        p["apply_solarization"] = rng.random() < self.solarization_prob
        p["apply_posterization"] = rng.random() < self.posterization_prob
        if p["apply_posterization"]:
            p["posterization_bits"] = rng.randint(self.posterization_bits_range[0], self.posterization_bits_range[1])
        if self.debug:
            print("Video Augmentation Parameters:")
            for k, v in p.items():
                if k != "cutout_boxes":
                    print(f"  {k}: {v}")
        return p


def inverse_affine_matrix(angle: float, translate: Sequence[float], scale: float, shear: Sequence[float]) -> List[float]:
    """tv:functional.py:1006-1064, centre (0,0), inverted; float64 like torchvision."""
    if scale <= 0.0:
        raise ValueError("Argument scale should be positive")
    rot, sx, sy = math.radians(angle), math.radians(shear[0]), math.radians(shear[1])
    tx, ty = translate
    a = math.cos(rot - sy) / math.cos(sy)
    b = -math.cos(rot - sy) * math.tan(sx) / math.cos(sy) - math.sin(rot)
    c = math.sin(rot - sy) / math.cos(sy)
    d = -math.sin(rot - sy) * math.tan(sx) / math.cos(sy) + math.cos(rot)
    m = [v / scale for v in (d, -b, 0.0, -c, a, 0.0)]
    m[2] += m[0] * (-tx) + m[1] * (-ty)
    m[5] += m[3] * (-tx) + m[4] * (-ty)
    return m


def draw_noise_seed() -> Tuple[int, int]:
    """Two 32-bit words from torch's GLOBAL generator - the stream the reference's ``torch.randn_like`` consumes
    (nexar_video_aug.py:245) - so ``torch.manual_seed`` controls the noise here as it does there, and Python's
    ``random`` draw order (SURVEY.md R0) is untouched."""
    import torch
    a, b = torch.randint(0, 2 ** 32, (2,), dtype=torch.int64).tolist()
    return int(a), int(b)


def gaussian_taps(sigma: float) -> np.ndarray:
    """nexar_video_aug.py:253 kernel size + tv _get_gaussian_kernel1d, float32."""
    ksize = int(sigma * 4) * 2 + 1
    half = (ksize - 1) * 0.5
    x = np.linspace(-half, half, ksize).astype(F32)
    pdf = np.exp(F32(-0.5) * (x / F32(sigma)) ** 2).astype(F32)
    return (pdf / pdf.sum(dtype=F32)).astype(F32)


_F = {name: (_lib.CLIP_PARAMS_DTYPE.fields[name][1] // 4) for name in _lib.CLIP_PARAMS_DTYPE.names}   # word offset of each field
_WORDS = _lib.CLIP_PARAMS_DTYPE.itemsize // 4


def pack_clip_params(records: Sequence[Dict[str, Any]], canvas: int,
                     aug_cfg: Optional[VideoAugmentation] = None) -> Tuple[np.ndarray, int]:
    """records[i] = {'flip': bool, 'aug': dict|None, 'crop': (dy, dx)|None, optional 'range_255': bool} ->
    (structured array of NexarClipParams, OR of all flags).  Raises the errors
    torchvision would raise for out-of-range factors.  Scalars are gathered into
    per-field columns and written with a few vectorised assignments (this runs once
    per batch on the host, in front of every kernel launch)."""
    n = len(records)
    words = np.zeros((n, _WORDS), np.uint32)
    fview = words.view(F32)
    iview = words.view(np.int32)
    flags_col = [0] * n
    # neutral values so that an un-augmented clip is well defined: brightness, contrast, saturation = 1
    colour = [[1.0, 1.0, 0.0, 1.0, 0.0, 0.0] for _ in range(n)]   # brightness, contrast, contrast_q, saturation, saturation_q, hue
    grids: List[Tuple[int, List[float]]] = []
    half = float(F32(0.5 * canvas))
    any_flags = 0
    for i, rec in enumerate(records):
        flags = _lib.FLIP if rec.get("flip") else 0
        if rec.get("range_255"):      # bytes 0..255: divided by 255 whatever the clip's maximum (WindowStream's chunks)
            flags |= _lib.RANGE_255
        crop = rec.get("crop")
        if crop is not None:
            iview[i, _F["crop_dy"]] = int(crop[0])
            iview[i, _F["crop_dx"]] = int(crop[1])
        p = rec.get("aug")
        if p is not None and not p.get("skip_augmentation", False):
            if aug_cfg is None:
                raise ValueError("augmentation parameters given without the VideoAugmentation config")
            flags |= _lib.AUG
            br, co, sa, hu = p["brightness"], p["contrast"], p["saturation"], p["hue"]
            if br < 0 or co < 0 or sa < 0:      # tv:_functional_tensor.py:172,182,225
                name, val = next((k, v) for k, v in (("brightness", br), ("contrast", co), ("saturation", sa)) if v < 0)
                raise ValueError(f"{name}_factor ({val}) is not non-negative.")
            if not (-0.5 <= hu <= 0.5):          # tv:_functional_tensor.py:199
                raise ValueError(f"hue_factor ({hu}) is not in [-0.5, 0.5].")
            colour[i] = [br, co, 1.0 - co, sa, 1.0 - sa, hu]
            if p["apply_affine"]:
                flags |= _lib.AFFINE
                grids.append((i, inverse_affine_matrix(p["rotation"], [p["translate_x"], p["translate_y"]],
                                                       p["scale"], [p["shear"], 0.0])))
            if p["apply_grayscale"]:
                flags |= _lib.GRAYSCALE
            if p["apply_noise"]:
                flags |= _lib.NOISE
                fview[i, _F["noise_level"]] = aug_cfg.noise_level
                # per-clip seed of the counter-based generator: the record's (drawn by sample_params, so a record
                # reproduces its noise), else a fresh draw - never a constant (the reference draws fresh
                # torch.randn_like noise for every frame of every call, nexar_video_aug.py:245)
                words[i, _F["noise_seed"]:_F["noise_seed"] + 2] = rec.get("noise_seed") or draw_noise_seed()
            if p["apply_blur"]:
                taps = gaussian_taps(aug_cfg.blur_sigma)
                if len(taps) > _lib.MAX_BLUR_TAPS:
                    raise ValueError(f"blur kernel of {len(taps)} taps exceeds NEXAR_MAX_BLUR_TAPS")
                if len(taps) // 2 >= canvas:
                    raise ValueError("blur kernel larger than the frame (reflect padding would fail)")
                if len(taps) > 1:
                    flags |= _lib.BLUR
                    iview[i, _F["blur_ksize"]] = len(taps)
                    fview[i, _F["blur_taps"]:_F["blur_taps"] + len(taps)] = taps
            if p["apply_posterization"]:
                flags |= _lib.POSTERIZE
                iview[i, _F["posterize_bits"]] = int(p["posterization_bits"])
            if p["apply_solarization"]:
                flags |= _lib.SOLARIZE
                fview[i, _F["solarize_threshold"]] = aug_cfg.solarization_threshold
            if p["apply_color_inversion"]:
                flags |= _lib.INVERT
            if p["apply_cutout"] and p.get("cutout_boxes"):
                boxes = p["cutout_boxes"]
                if len(boxes) > _lib.MAX_CUTOUT:
                    raise ValueError(f"{len(boxes)} cutout boxes exceed NEXAR_MAX_CUTOUT")
                flags |= _lib.CUTOUT
                iview[i, _F["n_cutout"]] = len(boxes)
                iview[i, _F["cutout"]:_F["cutout"] + 4 * len(boxes)] = np.asarray(boxes, np.int32).reshape(-1)
        flags_col[i] = flags
        any_flags |= flags
    words[:, _F["flags"]] = flags_col
    fview[:, _F["brightness"]:_F["brightness"] + 6] = np.asarray(colour, np.float64).astype(F32)   # float32(python double)
    if grids:
        idx = [g[0] for g in grids]
        theta = np.asarray([g[1] for g in grids], np.float64).astype(F32)     # torch.tensor(matrix, dtype=float32)
        fview[idx, _F["grid"]:_F["grid"] + 6] = theta / F32(half)             # tv _gen_affine_grid: theta^T / [0.5w, 0.5h]
    return words.view(_lib.CLIP_PARAMS_DTYPE).reshape(n), any_flags
