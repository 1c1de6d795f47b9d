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
``WindowStream`` / ``WindowPredictor.predict_stream`` take the same video chunk by chunk, as a decoder delivers it, and
keep only the last ``window - 1`` transformed frames plus one chunk on the device: any length, bounded memory.
"""
from __future__ import annotations

import itertools
from typing import Any, Callable, Dict, Iterable, Iterator, List, Optional, Tuple

import numpy as np
import torch

from . import _lib
from .video_aug import GpuVideoTransform, check_pixel_format, create_video_transforms, source_dtype
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


def windows_complete(num_frames: int, window: int, stride: int) -> int:
    """How many windows of ``sliding_window_starts`` lie wholly inside the first ``num_frames`` frames of a video."""
    return 0 if num_frames < window else (num_frames - window) // stride + 1


def ring_schedule(seen: int, n: int, window: int, stride: int, max_chunk: int) -> List[Tuple[int, int, list, int, int]]:
    """The work of pushing video frames ``seen .. seen+n-1`` into a ``WindowStream`` ring of ``window - 1 + max_chunk``
    slots (video frame f in slot f % ring size).  One group ``(lo, hi, writes, k0, k1)`` per ``max_chunk`` frames of the
    chunk: chunk frames ``lo .. hi-1`` are transformed into the ring by ``writes``, a list of ``(slot, offset, count)``
    (chunk frames ``offset .. offset+count-1`` into slots ``slot ..``; two writes when the group wraps the ring), and
    then windows ``k0 .. k1-1`` are complete.  Their frames are all still in the ring: before a group every window that
    ends before it is out, so the next one starts at or after frame ``seen + lo - window + 1``, and the group's at most
    ``max_chunk`` frames overwrite only older slots."""
    ring = window - 1 + max_chunk
    groups = []
    k0 = windows_complete(seen, window, stride)
    for lo in range(0, n, max_chunk):
        hi = min(n, lo + max_chunk)
        writes, pos = [], lo
        while pos < hi:
            slot = (seen + pos) % ring
            count = min(hi - pos, ring - slot)
            writes.append((slot, pos, count))
            pos += count
        k1 = windows_complete(seen + hi, window, stride)
        groups.append((lo, hi, writes, k0, k1))
        k0 = k1
    return groups


class WindowStream:
    """Sliding windows over a video that arrives in chunks of consecutive frames, in bounded device memory.

    ``push(chunk)`` transforms the chunk's frames into a ring of ``window - 1 + max_chunk`` per-frame results and returns
    ``(starts, windows)``: the start frames and a contiguous ``[k,3,window,cs,cs]`` tensor of every window the chunk
    completes (``k`` may be 0).  ``finish()`` returns the one padded window of a video shorter than ``window`` (its last
    frame repeated, nexar_videos.py:429-433) and nothing otherwise.  Concatenated, the results are
    ``SlidingWindowTransform(window, stride, transform, out_dtype).windows(video, materialize=True)`` bit for bit, with
    ``sliding_window_starts(N, window, stride)`` as starts, for any chunking, provided that

    - the video has a pixel above 1 (every chunk is scaled by 1/255, ``NEXAR_RANGE_255``; the offline call leaves a
      video whose values are all 0 or 1 unscaled, nexar_video_aug.py:809-821), and
    - the transform draws no gaussian noise (noise is seeded per call).

    The parameter record is drawn once, on the first push, with ``transform.sample_params(1, h, w)`` as ``frames()``
    draws it for a whole video, and every chunk uses it.  Chunks are uint8 ``[n,H,W,3]`` or YUV surfaces ``[n,R,P]``
    with the source-format keywords of ``forward_batch``, on the device or on the host: a host chunk is copied into a
    device staging buffer with a non-blocking copy, which overlaps when the host memory is pinned (do not overwrite a
    pinned chunk before the work of its push has run).  Device memory depends on ``window``, ``max_chunk``, the frame
    size and ``cs``, never on the length of the video.  Everything is enqueued on the current CUDA stream."""

    def __init__(self, window: int = 16, stride: int = 8, transform: Optional[GpuVideoTransform] = None,
                 out_dtype: torch.dtype = torch.bfloat16, max_chunk: int = 64):
        if window < 1 or stride < 1 or max_chunk < 1:
            raise ValueError(f"window, stride and max_chunk must be >= 1, got {window}, {stride}, {max_chunk}")
        self.window, self.stride, self.max_chunk = int(window), int(stride), int(max_chunk)
        self.ring_frames = self.window - 1 + self.max_chunk
        self.tf = transform or create_video_transforms(mode="val", out_dtype=out_dtype)
        self.out_dtype = out_dtype
        self.frames_seen = 0
        self._finished = False
        self._source = None       # (frame shape, dtype, source format) of the first chunk: every chunk must match it
        self._format: Dict[str, Any] = {}
        self._params = None
        self._ring: Optional[torch.Tensor] = None
        self._staging: Optional[torch.Tensor] = None

    def _start(self, frames: torch.Tensor, yuv: bool):
        if frames.dtype != source_dtype(self._format["pixel_format"]):
            raise ValueError(f"{self._format['pixel_format']} frames are {source_dtype(self._format['pixel_format'])}, "
                             f"got {frames.dtype}")
        if yuv:
            size = self._format["frame_size"]
            h, w = (frames.shape[1] * 2 // 3, frames.shape[2]) if size is None else size
        else:
            h, w = frames.shape[1], frames.shape[2]
        rec = dict(self.tf.sample_params(1, h, w)[0])
        rec["range_255"] = True
        self._params = [rec]
        dev = frames.device if frames.is_cuda else torch.device("cuda", torch.cuda.current_device())
        _lib.ring_lib()           # a library without the ring gather fails here, before any work
        cs = self.tf.crop_size
        self._ring = torch.empty((self.ring_frames, 3, cs, cs), dtype=self.out_dtype, device=dev)

    def _windows_out(self, k: int) -> torch.Tensor:
        cs = self.tf.crop_size
        return torch.empty((k, 3, self.window, cs, cs), dtype=self.out_dtype, device=self._ring.device)

    def _gather(self, out: torch.Tensor, first_frame: int, last_frame: int):
        ring = self._ring
        with torch.cuda.device(ring.device):
            _lib.check(_lib.ring_lib().nexar_gather_windows_ring(
                ring.data_ptr(), self.ring_frames, ring[0, 0].numel() * ring.element_size(), self.window, self.stride,
                first_frame, last_frame, out.shape[0], out.data_ptr(), torch.cuda.current_stream(ring.device).cuda_stream))

    @torch.no_grad()
    def push(self, frames: torch.Tensor, pixel_format: str = "rgb", color_matrix: str = "bt601",
             color_range: str = "limited", frame_size=None) -> Tuple[List[int], torch.Tensor]:
        """A chunk of ``n >= 1`` consecutive frames -> (start frames, ``[k,3,window,cs,cs]``) of the windows it completes."""
        if self._finished:
            raise ValueError("push() after finish(): start a new WindowStream for the next video")
        yuv = check_pixel_format(pixel_format, color_matrix, color_range)
        if frames.dtype.is_floating_point:
            raise TypeError(f"WindowStream takes decoded uint8 frames or YUV surfaces, got {frames.dtype}")
        if yuv and frames.dim() != 3:
            raise ValueError(f"expected a chunk of [n,R,P] {pixel_format} surfaces, got {tuple(frames.shape)}")
        if not yuv and (frames.dim() != 4 or frames.shape[-1] != 3):
            raise ValueError(f"expected a chunk of [n,H,W,3] frames, got {tuple(frames.shape)}")
        if frames.shape[0] < 1:
            raise ValueError("empty chunk")
        fmt = dict(pixel_format=pixel_format, color_matrix=color_matrix, color_range=color_range,
                   frame_size=None if frame_size is None else (int(frame_size[0]), int(frame_size[1])))
        source = (tuple(frames.shape[1:]), frames.dtype, tuple(fmt.values()))
        if self._source is None:
            self._format = fmt
            self._start(frames, yuv)
            self._source = source
        elif source != self._source:
            raise ValueError(f"the stream's frames are {self._source}; a chunk of {source} cannot join it")
        dev = self._ring.device
        if frames.is_cuda and frames.device != dev:
            raise ValueError(f"the stream lives on {dev}, the chunk on {frames.device}")
        n = frames.shape[0]
        k_first = windows_complete(self.frames_seen, self.window, self.stride)
        out = self._windows_out(windows_complete(self.frames_seen + n, self.window, self.stride) - k_first)
        for lo, hi, writes, k0, k1 in ring_schedule(self.frames_seen, n, self.window, self.stride, self.max_chunk):
            group = frames[lo:hi]
            if not frames.is_cuda:
                if self._staging is None:
                    self._staging = torch.empty((self.max_chunk,) + tuple(frames.shape[1:]), dtype=frames.dtype, device=dev)
                self._staging[:hi - lo].copy_(group, non_blocking=True)
                group = self._staging[:hi - lo]
            for slot, offset, count in writes:
                src = group[offset - lo:offset - lo + count]
                self.tf.forward_batch(src.unsqueeze(0), params=self._params, layout="BTCHW",
                                      out=self._ring[slot:slot + count].unsqueeze(0), **self._format)
            if k1 > k0:
                self._gather(out[k0 - k_first:k1 - k_first], k0 * self.stride, self.frames_seen + hi - 1)
        self.frames_seen += n
        return [k * self.stride for k in range(k_first, k_first + out.shape[0])], out

    @torch.no_grad()
    def finish(self) -> Tuple[List[int], torch.Tensor]:
        """Ends the video: the padded window of a video shorter than ``window``, else no window."""
        if self._finished:
            raise ValueError("finish() was called already")
        if self.frames_seen == 0:
            raise ValueError("the stream saw no frames: a video has at least one")
        self._finished = True
        if self.frames_seen >= self.window:
            return [], self._windows_out(0)
        out = self._windows_out(1)
        self._gather(out, 0, self.frames_seen - 1)
        return [0], out


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
            results.extend(self._classify(view[lo:lo + self.batch_size].contiguous(), starts[lo:lo + self.batch_size],
                                          video_path, fps))
        return results

    @torch.no_grad()
    def predict_stream(self, chunks: Iterable[torch.Tensor], video_path: str = "", fps: float = 30.0,
                       **source_format) -> Iterator[Dict[str, Any]]:
        """``predict`` over a video that arrives in chunks of consecutive frames (``WindowStream``): yields the same
        dictionaries in the same order, each batch of ``batch_size`` windows as soon as its last window is complete, the
        remainder at the end.  Device memory stays bounded whatever the length of the video.  ``source_format``: the
        forward_batch keywords of YUV surfaces (``pixel_format="nv12"``, ...), the same for every chunk."""
        stream = WindowStream(self.swt.window, self.swt.stride, transform=self.swt.tf, out_dtype=self.swt.out_dtype)
        parts: List[torch.Tensor] = []        # windows waiting for a full batch, and their starts
        part_starts: List[int] = []
        for chunk in itertools.chain(chunks, [None]):
            starts, win = stream.finish() if chunk is None else stream.push(chunk, **source_format)
            i = 0
            while i < len(starts):
                take = min(self.batch_size - len(part_starts), len(starts) - i)
                parts.append(win[i:i + take])
                part_starts.extend(starts[i:i + take])
                i += take
                if len(part_starts) == self.batch_size:
                    yield from self._classify(parts[0] if len(parts) == 1 else torch.cat(parts), part_starts, video_path, fps)
                    parts, part_starts = [], []
        if part_starts:
            yield from self._classify(parts[0] if len(parts) == 1 else torch.cat(parts), part_starts, video_path, fps)

    def _classify(self, batch: torch.Tensor, starts: List[int], video_path: str, fps: float) -> List[Dict[str, Any]]:
        """One model call on a contiguous ``[b,3,T,cs,cs]`` batch -> one result dictionary per window."""
        probs, pred = classify_outputs(self.model(batch), self.num_classes)
        results: List[Dict[str, Any]] = []
        for i in range(batch.shape[0]):
            cls = int(pred[i])
            results.append({
                "predicted_class": cls,
                "predicted_class_name": CLASS_MAP.get(cls, f"Class {cls}"),
                "probabilities": {CLASS_MAP.get(k, f"Class {k}"): float(probs[i, k]) for k in range(probs.shape[1])},
                "video_path": video_path,
                "window_start": starts[i],
                "window_start_sec": starts[i] / float(fps),
                "center_frame": starts[i] + self.swt.window // 2,
            })
        return results
