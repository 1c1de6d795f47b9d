"""Inference-time windowing on the device.

``nexar_inference.py:211-231`` feeds the model one centred ``fps*duration`` window
per video through the Dataset with ``create_video_transforms(mode='val')``;
``center_window`` reproduces that.  The reference has no sliding-window code
(SURVEY.md headline 7); ``SlidingWindowTransform`` is the extension BASELINE
config 4 asks for: the val chain is per-frame and window-independent, so every
frame of the video is transformed exactly once and the windows are strided views
(or one gather when a materialised ``[K,3,T,cs,cs]`` batch is wanted).
Window rule: starts ``k*stride`` for ``k = 0..floor((N-window)/stride)``; a video
shorter than the window is padded by repeating its last frame (nexar_videos.py:429-433).
Every entry point also takes a video of YUV 4:2:0 decoder surfaces ``[N,R,P]`` with the
``pixel_format`` / ``color_matrix`` / ``color_range`` / ``frame_size`` keywords of
``GpuVideoTransform.forward_batch``.
"""
from __future__ import annotations

from typing import Any, Callable, Dict, List, Optional

import numpy as np
import torch

from . import _lib
from .video_aug import GpuVideoTransform, check_pixel_format, create_video_transforms
from .videos import select_start_frame, window_indices


def sliding_window_starts(num_frames: int, window: int, stride: int) -> List[int]:
    if num_frames <= window:
        return [0]
    return [k * stride for k in range((num_frames - window) // stride + 1)]


@torch.no_grad()
def center_window(video_u8: torch.Tensor, transform: Optional[GpuVideoTransform] = None, fps: int = 10,
                  duration: int = 5, **source_format) -> torch.Tensor:
    """[N,H,W,3] uint8 (device) -> [1,3,fps*duration,cs,cs]: sample_strategy='center' + val transform.  A video of YUV
    surfaces [N,R,P] takes the source-format keywords of forward_batch (``pixel_format="i420"``, ...)."""
    tf = transform or create_video_transforms(mode="val")
    n = video_u8.shape[0]
    need = fps * duration
    idx = window_indices(n, need, select_start_frame(n, need, "center"))
    return tf.forward_batch(video_u8.unsqueeze(0), frame_index=torch.tensor([idx], dtype=torch.int64), **source_format)


class SlidingWindowTransform:
    def __init__(self, window: int = 16, stride: int = 8, transform: Optional[GpuVideoTransform] = None,
                 out_dtype: torch.dtype = torch.bfloat16):
        self.window, self.stride = window, stride
        self.tf = transform or create_video_transforms(mode="val", out_dtype=out_dtype)
        self.out_dtype = out_dtype

    @torch.no_grad()
    def frames(self, video_u8: torch.Tensor, pixel_format: str = "rgb", color_matrix: str = "bt601",
               color_range: str = "limited", frame_size=None) -> torch.Tensor:
        """[N,H,W,3] uint8 on the device -> [N,3,cs,cs]: every frame transformed once.  YUV surfaces [N,R,P] with
        ``pixel_format="nv12"`` / ``"i420"`` (uint16 with ``"p010"`` / ``"i010"``) and the other source-format keywords
        of forward_batch."""
        if check_pixel_format(pixel_format, color_matrix, color_range):
            if video_u8.dim() != 3:
                raise ValueError(f"expected [N,R,P] {pixel_format} surfaces, got {tuple(video_u8.shape)}")
        elif video_u8.dim() != 4 or video_u8.shape[-1] != 3:
            raise ValueError(f"expected [N,H,W,3], got {tuple(video_u8.shape)}")
        n = video_u8.shape[0]
        out = self.tf.forward_batch(video_u8.unsqueeze(0), layout="BTCHW", out_dtype=self.out_dtype, pixel_format=pixel_format,
                                    color_matrix=color_matrix, color_range=color_range, frame_size=frame_size)  # [1,N,3,cs,cs]
        if n < self.window:       # pad by repeating the last frame
            out = torch.cat([out, out[:, -1:].expand(1, self.window - n, *out.shape[2:])], dim=1)
        return out[0]

    def windows(self, video_u8: torch.Tensor, materialize: bool = False, **source_format) -> torch.Tensor:
        """-> [K,3,window,cs,cs].  A zero-copy strided view of the per-frame result unless ``materialize``."""
        fr = self.frames(video_u8, **source_format)                  # [N',3,cs,cs]
        starts = sliding_window_starts(fr.shape[0], self.window, self.stride)
        k = len(starts)
        s = fr.stride()
        if materialize:            # whole-plane gather through the library (one launch, streaming stores)
            out = torch.empty((k, 3, self.window, fr.shape[2], fr.shape[3]), dtype=fr.dtype, device=fr.device)
            with torch.cuda.device(fr.device):
                _lib.check(_lib.lib().nexar_gather_windows(fr.data_ptr(), fr.shape[0], fr.shape[2] * fr.shape[3] * fr.element_size(),
                                                           self.window, self.stride, k, out.data_ptr(),
                                                           torch.cuda.current_stream(fr.device).cuda_stream))
            return out
        return fr.as_strided((k, 3, self.window, fr.shape[2], fr.shape[3]),
                             (self.stride * s[0], s[1], s[0], s[2], s[3]))


CLASS_MAP = {0: "Normal", 1: "Near Collision", 2: "Collision"}      # nexar_inference.py:239


def classify_outputs(outputs: torch.Tensor, num_classes: int = 3):
    """Logits -> (probabilities [K,C] numpy, predicted classes [K] numpy), the post-processing of
    nexar_inference.py:250-266 (sigmoid + 0.5 threshold for two classes, softmax + argmax otherwise)."""
    if num_classes == 2:
        probs = torch.sigmoid(outputs.float()).cpu().numpy()
        if probs.ndim == 1:
            probs = np.column_stack((1 - probs, probs))
        pred = (probs > 0.5).astype(int)
        if pred.ndim == 1:
            pred = pred[:, 1]
        elif pred.ndim == 2:
            pred = pred[:, -1]
        return probs, pred
    probs = torch.softmax(outputs.float(), dim=1).cpu().numpy()
    pred = torch.argmax(outputs, dim=1).cpu().numpy()
    return probs, pred


class WindowPredictor:
    """Sliding-window inference service shaped like ``InferenceEngine.predict`` (nexar_inference.py:103-340), for one
    decoded video already on the device: every frame goes through the val transform once, the model sees batches of
    ``[b,3,window,cs,cs]`` windows (strided views of the per-frame result, made contiguous per batch only), and one
    result dictionary per window comes back with the reference's keys plus the window position.

    ``model``: any callable taking ``[b,3,T,cs,cs]`` and returning logits ``[b,num_classes]`` (the reference passes
    ``frames.permute(0,4,1,2,3).float().to(device)``, :248; here the tensor is born on the device in that layout)."""

    def __init__(self, model: Callable[[torch.Tensor], torch.Tensor], window: int = 16, stride: int = 8, batch_size: int = 8,
                 num_classes: int = 3, transform: Optional[GpuVideoTransform] = None, out_dtype: torch.dtype = torch.float32):
        self.model = model
        self.batch_size = int(batch_size)
        self.num_classes = int(num_classes)
        self.swt = SlidingWindowTransform(window=window, stride=stride, transform=transform, out_dtype=out_dtype)

    @torch.no_grad()
    def predict(self, video_u8: torch.Tensor, video_path: str = "", fps: float = 30.0,
                **source_format) -> List[Dict[str, Any]]:
        """``source_format``: the forward_batch keywords of a video of YUV surfaces (``pixel_format="i420"``, ...)."""
        view = self.swt.windows(video_u8, **source_format)             # [K,3,T,cs,cs] strided view
        starts = sliding_window_starts(max(video_u8.shape[0], self.swt.window), self.swt.window, self.swt.stride)
        results: List[Dict[str, Any]] = []
        for lo in range(0, view.shape[0], self.batch_size):
            batch = view[lo:lo + self.batch_size].contiguous()
            probs, pred = classify_outputs(self.model(batch), self.num_classes)
            for i in range(batch.shape[0]):
                cls = int(pred[i])
                results.append({
                    "predicted_class": cls,
                    "predicted_class_name": CLASS_MAP.get(cls, f"Class {cls}"),
                    "probabilities": {CLASS_MAP.get(k, f"Class {k}"): float(probs[i, k]) for k in range(probs.shape[1])},
                    "video_path": video_path,
                    "window_start": starts[lo + i],
                    "window_start_sec": starts[lo + i] / float(fps),
                    "center_frame": starts[lo + i] + self.swt.window // 2,
                })
        return results
