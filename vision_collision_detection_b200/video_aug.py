"""Drop-in mirror of the reference's transform factories for the GPU path.

``create_video_transforms(**kwargs)`` has the signature of
``nexar_video_aug.create_video_transforms`` (nexar_video_aug.py:636-696) and
returns an ``nn.Module`` with the same call contract
(``module(video[C,T,H,W] uint8|float) -> [C,T,cs,cs] float32``,
nexar_videos.py:444-445) and a ``.transforms`` list, but the pixel work runs in
the fused CUDA kernels of libnexar_clip_b200.so.  As in the reference, the
kwargs ``aug_probability, cutout_count, cutout_size_range,
posterization_bits_range, solarization_threshold, perspective_distortion,
jpeg_quality, min_size, max_size, num_samples, video_key, convert_to_float`` are
accepted and have no effect (they are never forwarded, :762-788).

``create_video_transform`` mirrors the reference's second, never-called factory
(:318-565): short-side antialiased resize followed by letterbox (what its
``forward`` actually does, because ``crop_tensor`` defaults to
``use_letterbox=True``) or, with ``use_letterbox=False``, the centre / random
crop north_star names.

Extra, GPU-only entry points: ``forward_batch`` (device-resident
``[B,T,H,W,3]`` clips or YUV 4:2:0 decoder surfaces in, ``[B,3,T,cs,cs]`` out,
fp32 or bf16, optional frame gather) — the call the loaders and bench use.
"""
from __future__ import annotations

import random
from typing import Any, Dict, List, Optional, Tuple

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from .engine import _alloc_out, get_engine
from .params import VideoAugmentation, draw_noise_seed, pack_clip_params
from .source_format import RGB_F32, FrameSource, PlanKey, SourceFormat


class _Stage:
    """Named entry of ``.transforms`` (the reference keeps closures there)."""

    def __init__(self, name: str, **info):
        self.__name__ = name
        self.info = info

    def __repr__(self):
        return f"<gpu stage {self.__name__} {self.info}>"


class GpuVideoTransform(nn.Module):
    def __init__(self, *, mode: str, crop_size: int, normalize: bool, video_mean, video_std,
                 horizontal_flip_prob: float, video_aug: Optional[VideoAugmentation],
                 resize_short_side: Optional[int] = None, use_letterbox: bool = True, center_crop: bool = False,
                 out_dtype: torch.dtype = torch.float32, device=None, output_device: str = "input",
                 deferred: bool = False):
        super().__init__()
        self.deferred = bool(deferred)
        if self.deferred:
            if resize_short_side is not None:
                raise ValueError("deferred=True supports the letterbox factory (create_video_transforms) only")
            from .deferred import install_collate_hooks
            install_collate_hooks()
        self.mode = mode
        self.crop_size = int(crop_size)
        self.normalize = bool(normalize)
        self.video_mean = tuple(float(v) for v in video_mean)
        self.video_std = tuple(float(v) for v in video_std)
        self.horizontal_flip_prob = horizontal_flip_prob
        self.video_aug = video_aug
        self.resize_short_side = resize_short_side
        self.use_letterbox = use_letterbox
        self.center_crop = center_crop
        self.out_dtype = out_dtype
        self.device = device
        self.output_device = output_device
        self.last_params: Optional[List[Dict[str, Any]]] = None
        self.transforms: List[Any] = []
        if resize_short_side is not None:
            self.transforms.append(_Stage("resize_tensor", size=resize_short_side))
            self.transforms.append(_Stage("crop_tensor", crop_size=crop_size, use_letterbox=use_letterbox))
        else:
            self.transforms.append(_Stage("letterbox_resize", crop_size=crop_size))
        if self._flips:
            self.transforms.append(_Stage("horizontal_flip", prob=horizontal_flip_prob))
        if video_aug is not None:
            self.transforms.append(video_aug)
        if normalize:
            self.transforms.append(_Stage("normalize_tensor", mean=self.video_mean, std=self.video_std))

    @property
    def _flips(self) -> bool:
        return self.mode == "train" and self.horizontal_flip_prob > 0

    # -- picklable description (deferred clips carry it from the DataLoader worker to the process that owns the GPU) ----
    _AUG_FIELDS = ("brightness_range", "contrast_range", "saturation_range", "hue_range", "rotation_range", "scale_range",
                   "shear_range", "translate_range", "grayscale_prob", "noise_level", "blur_sigma", "cutout_prob",
                   "cutout_count_range", "cutout_size_range", "color_inversion_prob", "solarization_prob",
                   "solarization_threshold", "posterization_prob", "posterization_bits_range", "aug_probability")

    def spec(self) -> Tuple:
        """Hashable constructor arguments: ``GpuVideoTransform.from_spec(tf.spec())`` transforms like ``tf``."""
        aug = None
        if self.video_aug is not None:
            aug = tuple((k, tuple(v) if isinstance(v, (list, tuple)) else v)
                        for k in self._AUG_FIELDS for v in [getattr(self.video_aug, k)])
        return (("mode", self.mode), ("crop_size", self.crop_size), ("normalize", self.normalize),
                ("video_mean", self.video_mean), ("video_std", self.video_std),
                ("horizontal_flip_prob", self.horizontal_flip_prob), ("video_aug", aug),
                ("resize_short_side", self.resize_short_side), ("use_letterbox", self.use_letterbox),
                ("center_crop", self.center_crop))

    _spec_cache: Dict[Tuple, "GpuVideoTransform"] = {}

    @classmethod
    def from_spec(cls, spec: Tuple) -> "GpuVideoTransform":
        tf = cls._spec_cache.get(spec)
        if tf is None:
            kw = dict(spec)
            if kw["video_aug"] is not None:
                kw["video_aug"] = VideoAugmentation(**dict(kw["video_aug"]))
            tf = cls._spec_cache[spec] = cls(**kw)
        return tf

    # -- random decisions, reference order -------------------------------------------
    def _resized_hw(self, h: int, w: int) -> Tuple[int, int]:
        s = self.resize_short_side
        return (s * h // w, s) if h > w else (s, s * w // h)

    def sample_params(self, n_clips: int, h: int, w: int, rng=random) -> List[Dict[str, Any]]:
        recs = []
        cs = self.crop_size
        for _ in range(n_clips):
            rec: Dict[str, Any] = {"flip": False, "aug": None, "crop": None}
            if self.resize_short_side is not None and not self.use_letterbox:
                rh, rw = self._resized_hw(h, w)
                ctop, cleft = (rh - cs) // 2, (rw - cs) // 2
                if self.center_crop or self.mode != "train":
                    top, left = ctop, cleft
                else:                                   # nexar_video_aug.py:472-473
                    top = rng.randint(0, rh - cs) if rh > cs else 0
                    left = rng.randint(0, rw - cs) if rw > cs else 0
                rec["crop"] = (ctop - top, cleft - left)   # relative to the plan's centre-crop offset
                rec["crop_top_left"] = (top, left)
            if self._flips:
                rec["flip"] = rng.random() < self.horizontal_flip_prob      # :748
            if self.video_aug is not None:
                rec["aug"] = self.video_aug._sample_augmentation_parameters((3, 0, cs, cs), rng)  # :290
                if rec["aug"].get("apply_noise"):      # fresh noise per clip and call (torch's generator, as :245)
                    rec["noise_seed"] = draw_noise_seed()
            recs.append(rec)
        return recs

    # -- plans -----------------------------------------------------------------------
    def _plan(self, eng, h: int, w: int, key):
        if not isinstance(key, PlanKey):    # a pixel format name or an RGB dtype: unpadded h x w frames
            fmt = SourceFormat.of(key if isinstance(key, str) else "rgb")
            key = fmt.describe(fmt.frame_shape(h, w), fmt.dtype if fmt.yuv else key).plan_key
        cs = self.crop_size
        if self.resize_short_side is None:
            return eng.letterbox_plan(h, w, cs, key)
        if self.use_letterbox:
            raise RuntimeError("two-pass variant: handled by _forward_two_pass")
        return eng.resize_crop_plan(h, w, self.resize_short_side, cs, key)

    def _forward_two_pass(self, eng, frames, source, offsets, n_clips, t_out, packed, any_flags, out, strides):
        """The never-called factory's default forward (nexar_video_aug.py:407-463): an antialiased short-side
        resize followed by a SECOND antialiased resize inside crop_tensor(use_letterbox=True).  Pass 1 writes
        the [0,1] float frames of size (rh, rw) on a square scratch canvas; pass 2 letterboxes those float
        frames (strided rows) and applies flip / augmentation / normalisation.  A record's byte-range flag describes the
        source frames, so it goes to pass 1 only: pass 2 reads values that are already in [0,1]."""
        rh, rw = self._resized_hw(source.h, source.w)
        cm = max(rh, rw)
        plan1 = eng.plan(_lib.Geometry(source.h, source.w, cm, rh, rw, 0, 0), source.plan_key)
        mid, mid_strides = _alloc_out("BTHWC", n_clips, t_out, cm, torch.float32, frames.device)
        range_255 = packed["flags"] & _lib.RANGE_255
        neutral, _ = pack_clip_params([{"flip": False, "aug": None, "range_255": bool(r)} for r in range_255], cm, None)
        packed["flags"] &= ~range_255
        eng.run(plan1, frames, offsets, n_clips, t_out, eng.upload_params(neutral), 0, mid, mid_strides,
                False, self.video_mean, self.video_std)
        plan2 = eng.plan(_lib.letterbox_geometry(rh, rw, self.crop_size), RGB_F32)
        offsets2 = eng.contiguous_offsets(n_clips * t_out, cm * cm * 3 * 4)
        eng.run(plan2, mid, offsets2, n_clips, t_out, eng.upload_params(packed), any_flags, out, strides,
                self.normalize, self.video_mean, self.video_std, src_row_stride=cm * 3 * 4)
        return out

    # -- batch entry point -------------------------------------------------------------
    @torch.no_grad()
    def forward_batch(self, frames: torch.Tensor, params: Optional[List[Dict[str, Any]]] = None,
                      frame_index: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
                      layout: str = "BCTHW", out_dtype: Optional[torch.dtype] = None, rng=random,
                      engine=None, pixel_format: str = "rgb", color_matrix: str = "bt601",
                      color_range: str = "limited", frame_size: Optional[Tuple[int, int]] = None) -> torch.Tensor:
        """frames: CUDA ``[B,T,H,W,3]`` (uint8 or float32, contiguous) — or, with ``frame_index``
        (int64 ``[B,T']`` indices into the flattened ``B*T`` frame axis), a frame pool from which each
        output clip gathers its frames (temporal sampling without a copy).  Returns ``[B,3,T',cs,cs]``.

        ``pixel_format="nv12"``: frames are decoder surfaces, uint8 ``[B,T,H*3/2,W]`` (Y plane, then the
        interleaved UV plane), 1.5 bytes per pixel; they are converted on the device (BT.601 limited range,
        include/nexar_clip_transform.h) to the RGB bytes the reference's decoder would have delivered
        (nexar_videos.py:360,422) and take the uint8 path from there.

        ``pixel_format="i420"``: planar surfaces, the Y plane then the U and V planes of half the pitch each (what
        libavcodec's ``yuv420p`` delivers).  ``color_matrix`` ("bt601" | "bt709") and ``color_range`` ("limited" |
        "full") select the conversion of either YUV layout.  YUV frames are ``[B,T,R,P]`` surfaces with
        ``L = R*2/3`` luma rows and pitch ``P``; ``frame_size=(h, w)`` is the visible picture in their top-left corner
        (default ``(L, P)``), e.g. ``(1080, 1920)`` in the 1088-row surfaces of a hardware decoder.  The random
        decisions are drawn for the visible ``h x w``, as for an RGB clip of that size.

        ``pixel_format="p010"`` / ``"i010"``: the same two layouts with 16-bit little-endian samples, frames
        ``torch.uint16 [B,T,R,P]`` with ``P`` the pitch in samples (a byte buffer can be passed as ``.view(torch.uint16)``).
        ``"p010"`` is semi-planar with the sample in the high bits of its word (P010, and P012 / P016 alike: what a
        hardware decoder delivers for 10-bit HEVC); ``"i010"`` is planar 10-bit in the low bits (libavcodec's
        ``yuv420p10le``).  They are converted to the same RGB bytes, rounded once from the full sample precision
        (include/nexar_clip_transform.h)."""
        fmt = SourceFormat.of(pixel_format, color_matrix, color_range)
        if frames.dim() != (4 if fmt.yuv else 5):
            raise ValueError(f"{pixel_format} frames are [B,T,{'R,P' if fmt.yuv else 'H,W,3'}], got {tuple(frames.shape)}")
        source = fmt.describe(frames.shape[2:], frames.dtype, frame_size)
        b, t = frames.shape[:2]
        if not frames.is_cuda:
            raise ValueError("forward_batch needs device-resident frames (use forward() for host tensors)")
        if not frames.is_contiguous():
            frames = frames.contiguous()
        eng = engine if engine is not None else get_engine(frames.device)
        if frame_index is not None:
            if frame_index.dim() != 2:
                raise ValueError("frame_index must be [n_clips, frames_per_clip]")
            n_clips, t_out = frame_index.shape
            if frame_index.numel() == 0:
                raise ValueError("frame_index is empty")
            # the kernels turn these into raw byte offsets: refuse anything outside the frame pool (a host tensor is
            # checked here; a device tensor is checked on the device without a sync, the failure surfaces at the next one)
            if frame_index.is_cuda:
                torch._assert_async(((frame_index >= 0) & (frame_index < b * t)).all())
            elif int(frame_index.min()) < 0 or int(frame_index.max()) >= b * t:
                raise ValueError(f"frame_index must lie in [0, {b * t}); got [{int(frame_index.min())}, {int(frame_index.max())}]")
            offsets = (frame_index.to(device=frames.device, dtype=torch.int64) * source.frame_bytes).reshape(-1).contiguous()
        else:
            n_clips, t_out = b, t
            offsets = eng.contiguous_offsets(b * t, source.frame_bytes)
        if params is None:
            params = self.sample_params(n_clips, source.h, source.w, rng)
        if len(params) != n_clips:
            raise ValueError("one parameter record per clip is required")
        self.last_params = params
        packed, any_flags = pack_clip_params(params, self.crop_size, self.video_aug)
        return self._transform_packed(eng, frames, offsets, n_clips, t_out, packed, any_flags, source, out, layout,
                                      out_dtype or self.out_dtype)

    def _transform_packed(self, eng, frames: torch.Tensor, offsets: torch.Tensor, n_clips: int, t_out: int,
                          packed: np.ndarray, any_flags: int, source: FrameSource, out: Optional[torch.Tensor],
                          layout: str, out_dtype: torch.dtype) -> torch.Tensor:
        """The library call behind ``forward_batch``: ``n_clips`` clips of ``t_out`` frames read at the byte
        ``offsets`` (int64, on the device) from ``frames.data_ptr()``, with the packed parameter records ``packed`` (one
        per clip, ``pack_clip_params``).  ``frames`` only gives the base address, device and element type, so the
        frames may lie anywhere above it (``MultiWindowStream`` gathers frames of many tensors in one call)."""
        two_pass = self.resize_short_side is not None and self.use_letterbox
        if source.format.yuv and two_pass:
            raise ValueError(f"{source.format.pixel_format} frames are not supported by the two-pass (short-side resize + letterbox) variant")
        plan = None if two_pass else self._plan(eng, source.h, source.w, source.plan_key)
        if out is None:
            out, strides = _alloc_out(layout, n_clips, t_out, self.crop_size, out_dtype, frames.device)
        else:
            probe, strides = _alloc_out(layout, n_clips, t_out, self.crop_size, out.dtype, "meta")
            if tuple(out.shape) != tuple(probe.shape) or not out.is_contiguous():
                raise ValueError(f"out must be a contiguous {tuple(probe.shape)} tensor for layout {layout}")
        if two_pass:
            return self._forward_two_pass(eng, frames, source, offsets, n_clips, t_out, packed, any_flags, out, strides)
        pdev = eng.upload_params(packed)
        eng.run(plan, frames, offsets, n_clips, t_out, pdev, any_flags, out, strides,
                self.normalize, self.video_mean, self.video_std, src_row_stride=source.row_stride)
        return out

    @torch.no_grad()
    def forward_model_input(self, frames: torch.Tensor, params: Optional[List[Dict[str, Any]]] = None,
                            out_dtype: Optional[torch.dtype] = None, rng=random) -> torch.Tensor:
        """Opt-in fast path for the consumer (SURVEY.md section 8f F2).  ``nexar_arch.EnhancedFrameCNN.forward``
        keeps every other frame when T > 10 and immediately reshapes to ``[B*T',3,H,W]`` (nexar_arch.py:411-419);
        this transforms only the frames the model keeps and writes them frame-major: returns ``[B,T',3,cs,cs]``
        (``.flatten(0,1)`` is the backbone input; ``.permute(0,2,1,3,4)`` is the ``[B,3,T',H,W]`` the model's public
        signature takes).  Same random decisions per clip as ``forward_batch``; parity mode still produces all T."""
        b, t = frames.shape[0], frames.shape[1]
        keep = list(range(0, t, 2)) if t > 10 else list(range(t))
        index = (torch.arange(b, dtype=torch.int64).view(b, 1) * t + torch.tensor(keep, dtype=torch.int64).view(1, -1))
        return self.forward_batch(frames, params=params, frame_index=index, layout="BTCHW", out_dtype=out_dtype, rng=rng)

    # -- reference-compatible call -----------------------------------------------------
    @torch.no_grad()
    def forward(self, video: torch.Tensor) -> torch.Tensor:
        """``video``: ``[C,T,H,W]`` uint8 or float (typically the ``permute(3,0,1,2)`` view of decoded
        THWC frames, nexar_videos.py:441).  Returns ``[C,T,cs,cs]`` (float32 unless ``out_dtype`` was
        changed), on the input's device unless ``output_device='cuda'``."""
        if video.dim() != 4 or video.shape[0] != 3:
            raise ValueError(f"expected [3,T,H,W], got {tuple(video.shape)}")
        if video.dtype not in (torch.uint8, torch.float32):
            video = video.float()                       # nexar_video_aug.py:811-812
        if self.deferred and not video.is_cuda:
            # host part only (this runs inside a DataLoader worker): the random decisions, in the reference's order, and
            # the decoded frames; the pixel work happens at ``batch['frames']....to(device)`` (deferred.py)
            from .deferred import DeferredClip
            thwc = video.permute(1, 2, 3, 0).contiguous()        # a no-copy view when the memory is THWC
            params = self.sample_params(1, thwc.shape[1], thwc.shape[2])[0]
            self.last_params = [params]
            return DeferredClip(thwc, params, self.spec(), self.crop_size)
        src_device = video.device
        thwc = video.permute(1, 2, 3, 0)                 # a no-copy view when the memory is THWC
        dev = torch.device(self.device) if self.device is not None else (
            src_device if src_device.type == "cuda" else torch.device("cuda", torch.cuda.current_device()))
        thwc = thwc.to(dev, non_blocking=True).contiguous()
        out = self.forward_batch(thwc.unsqueeze(0))[0]
        if self.output_device == "input" and src_device.type != "cuda":
            out = out.to(src_device)
        return out


def create_video_transforms(
        mode='train', video_key=None, num_samples=75, convert_to_float=True, crop_size=224,
        normalize=True, video_mean=(0.45, 0.45, 0.45), video_std=(0.225, 0.225, 0.225),
        min_size=224, max_size=320, horizontal_flip_prob=0.5,
        enable_custom_augmentation=False, aug_probability=1.0,
        brightness_range=(0.9, 1.1), contrast_range=(0.9, 1.1), saturation_range=(0.9, 1.1),
        hue_range=(-0.05, 0.05), rotation_range=(-5, 5), scale_range=(0.95, 1.05), shear_range=(-2, 2),
        translate_range=(0.0, 0.05), perspective_distortion=0.0, noise_level=0.0, blur_sigma=0.0,
        jpeg_quality=0, grayscale_prob=0.0, cutout_prob=0.0, cutout_count=(1, 3),
        cutout_size_range=(0.1, 0.2), color_inversion_prob=0.0, solarization_prob=0.0,
        posterization_prob=0.0, posterization_bits_range=(3, 6), solarization_threshold=0.5, debug=False,
        *, out_dtype=torch.float32, device=None, output_device="input", deferred=False):
    """Same positional/keyword surface as nexar_video_aug.py:636-696; the keyword-only arguments after ``debug``
    are GPU additions (``deferred=True``: the zero-line DataLoader drop-in of deferred.py)."""
    aug = None
    if mode == 'train' and enable_custom_augmentation:
        aug = VideoAugmentation(                      # exactly the kwargs forwarded at :762-788
            brightness_range=brightness_range, contrast_range=contrast_range,
            saturation_range=saturation_range, hue_range=hue_range, rotation_range=rotation_range,
            scale_range=scale_range, shear_range=shear_range, translate_range=translate_range,
            grayscale_prob=grayscale_prob, noise_level=noise_level, blur_sigma=blur_sigma,
            cutout_prob=cutout_prob, color_inversion_prob=color_inversion_prob,
            solarization_prob=solarization_prob, posterization_prob=posterization_prob, debug=debug)
    return GpuVideoTransform(mode=mode, crop_size=crop_size, normalize=normalize, video_mean=video_mean,
                             video_std=video_std, horizontal_flip_prob=horizontal_flip_prob, video_aug=aug,
                             out_dtype=out_dtype, device=device, output_device=output_device, deferred=deferred)


def create_video_transform(
        mode='train', normalize=True, video_mean=(0.45, 0.45, 0.45), video_std=(0.225, 0.225, 0.225),
        min_size=224, max_size=None, crop_size=224, center_crop=False, horizontal_flip_prob=0.5,
        enable_advanced_augmentation=False,
        brightness_range=(0.8, 1.2), contrast_range=(0.8, 1.2), saturation_range=(0.8, 1.2),
        hue_range=(-0.1, 0.1), rotation_range=(-10, 10), scale_range=(0.9, 1.1), shear_range=(-5, 5),
        translate_range=(0.0, 0.1), grayscale_prob=0.02, noise_level=0.02, blur_sigma=0.0, cutout_prob=0.0,
        color_inversion_prob=0.0, solarization_prob=0.0, posterization_prob=0.0, debug=False,
        *, use_letterbox=True, out_dtype=torch.float32, device=None, output_device="input"):
    """Mirror of the never-called factory (nexar_video_aug.py:318-565).  The resize size is drawn
    once, here, like the reference does (:399-404).  ``use_letterbox=False`` selects the crop branch
    (:464-482) that the reference only reaches through ``tf.transforms[1](video, use_letterbox=False)``."""
    if mode == 'train' and max_size is not None and max_size > min_size:
        size = random.randint(min_size, max_size)
    else:
        size = min_size
    aug = None
    if mode == 'train' and enable_advanced_augmentation:
        aug = VideoAugmentation(
            brightness_range=brightness_range, contrast_range=contrast_range,
            saturation_range=saturation_range, hue_range=hue_range, rotation_range=rotation_range,
            scale_range=scale_range, shear_range=shear_range, translate_range=translate_range,
            grayscale_prob=grayscale_prob, noise_level=noise_level, blur_sigma=blur_sigma,
            cutout_prob=cutout_prob, color_inversion_prob=color_inversion_prob,
            solarization_prob=solarization_prob, posterization_prob=posterization_prob, debug=debug)
    return GpuVideoTransform(mode=mode, crop_size=crop_size, normalize=normalize, video_mean=video_mean,
                             video_std=video_std, horizontal_flip_prob=horizontal_flip_prob, video_aug=aug,
                             resize_short_side=size, use_letterbox=use_letterbox, center_crop=center_crop,
                             out_dtype=out_dtype, device=device, output_device=output_device)
