"""Device-side engine: owns plans, workspaces and parameter staging, and calls
``nexar_clip_transform`` (include/nexar_clip_transform.h) on torch's current
CUDA stream.  PyTorch is used for device memory and streams only.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from .source_format import RGB_U8, PlanKey

_DST = {torch.float32: _lib.DST_F32, torch.bfloat16: _lib.DST_BF16, torch.float16: _lib.DST_F16}

# output layouts: name -> (shape builder, element strides for (clip, channel, frame, y, x))
LAYOUTS = ("BCTHW", "BTCHW", "BTHWC")


def _alloc_out(layout: str, b: int, t: int, cs: int, dtype, device):
    if layout == "BCTHW":
        out = torch.empty((b, 3, t, cs, cs), dtype=dtype, device=device)
        s = out.stride()
        return out, (s[0], s[1], s[2], s[3], s[4])
    if layout == "BTCHW":
        out = torch.empty((b, t, 3, cs, cs), dtype=dtype, device=device)
        s = out.stride()
        return out, (s[0], s[2], s[1], s[3], s[4])
    if layout == "BTHWC":
        out = torch.empty((b, t, cs, cs, 3), dtype=dtype, device=device)
        s = out.stride()
        return out, (s[0], s[4], s[1], s[2], s[3])
    raise ValueError(f"unknown layout {layout!r}; expected one of {LAYOUTS}")


class Plan:
    """RAII wrapper of NexarPlan."""

    def __init__(self, geom: _lib.Geometry, key: PlanKey):
        self.geom = geom
        self.key = key
        h = C.c_void_p()
        f = None if key.yuv is None else _lib.YuvFormat(C.sizeof(_lib.YuvFormat), *key.yuv)
        if f is None:
            _lib.check(_lib.lib().nexar_plan_create(C.byref(geom), key.src, C.byref(h)))
        elif key.sample_shift is None:
            _lib.check(_lib.yuv_lib().nexar_plan_create_yuv(C.byref(geom), C.byref(f), C.byref(h)))
        else:
            _lib.check(_lib.yuv16_lib().nexar_plan_create_yuv16(C.byref(geom), C.byref(f), key.sample_shift, C.byref(h)))
        self.handle = h

    def workspace_bytes(self, n_clips: int, t: int, any_flags: int = 0xFFFFFFFF) -> int:
        return int(_lib.lib().nexar_workspace_bytes_for(self.handle, n_clips, t, any_flags & 0xFFFFFFFF))

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                _lib.lib().nexar_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class ClipTransformEngine:
    """One per (process, device).  Not thread-safe; one per stream if you need concurrency."""

    def __init__(self, device: Optional[torch.device] = None):
        if not torch.cuda.is_available():
            raise RuntimeError("ClipTransformEngine needs a CUDA device; there is no CPU fallback")
        _lib.lib()  # fail loudly if the CUDA library is missing
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self._plans: Dict[Tuple, Plan] = {}
        self._workspace: Optional[torch.Tensor] = None
        self._ring = [[None, None] for _ in range(8)]
        self._ring_pos = 0
        self._offsets: Dict[Tuple, torch.Tensor] = {}
        self.last_launches = 0

    # -- plans ---------------------------------------------------------------------
    def plan(self, geom: _lib.Geometry, key: PlanKey) -> Plan:
        cache_key = geom.as_tuple() + (key,)
        p = self._plans.get(cache_key)
        if p is None:
            with torch.cuda.device(self.device):
                p = Plan(geom, key)
            self._plans[cache_key] = p
        return p

    def letterbox_plan(self, h: int, w: int, cs: int, key: PlanKey = RGB_U8) -> Plan:
        return self.plan(_lib.letterbox_geometry(h, w, cs), key)

    def resize_crop_plan(self, h: int, w: int, size: int, cs: int, key: PlanKey = RGB_U8) -> Plan:
        return self.plan(_lib.resize_crop_geometry(h, w, size, cs), key)

    # -- buffers -------------------------------------------------------------------
    def _get_workspace(self, nbytes: int) -> torch.Tensor:
        if self._workspace is None or self._workspace.numel() < nbytes:
            self._workspace = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        return self._workspace

    def contiguous_offsets(self, n_frames: int, frame_bytes: int) -> torch.Tensor:
        key = (n_frames, frame_bytes)
        t = self._offsets.get(key)
        if t is None:
            t = torch.arange(n_frames, dtype=torch.int64, device=self.device) * frame_bytes
            if len(self._offsets) > 64:
                self._offsets.clear()
            self._offsets[key] = t
        return t

    def upload_params(self, params: np.ndarray) -> torch.Tensor:
        """structured NexarClipParams array -> device bytes, through a small ring of pinned
        staging buffers (an event per slot says when its last async copy was consumed)."""
        raw = np.ascontiguousarray(params).view(np.uint8).reshape(-1)
        n = raw.size
        slot = self._ring[self._ring_pos]
        self._ring_pos = (self._ring_pos + 1) % len(self._ring)
        if slot[0] is None or slot[0].numel() < n:
            slot[0] = torch.empty(max(n, 1 << 15), dtype=torch.uint8).pin_memory()
            slot[1] = torch.cuda.Event()
        else:
            slot[1].synchronize()
        slot[0][:n].numpy()[:] = raw
        dev = slot[0][:n].to(self.device, non_blocking=True)
        slot[1].record(torch.cuda.current_stream(self.device))
        return dev

    # -- the call ------------------------------------------------------------------
    def run(self, plan: Plan, src: torch.Tensor, frame_offsets: torch.Tensor, n_clips: int, frames_per_clip: int,
            params_dev: torch.Tensor, any_flags: int, out: torch.Tensor, dst_stride: Sequence[int],
            normalize: bool, mean: Sequence[float], std: Sequence[float], src_row_stride: Optional[int] = None):
        """Enqueue the transform on the current stream.  ``src`` is any CUDA tensor whose storage holds the
        decoded frames; ``frame_offsets`` are byte offsets from ``src.data_ptr()``."""
        if src.device != self.device or out.device != self.device or params_dev.device != self.device:
            raise ValueError("src/out/params must live on the engine's device")
        if frame_offsets.dtype != torch.int64 or frame_offsets.numel() != n_clips * frames_per_clip:
            raise ValueError("frame_offsets must be int64 [n_clips*frames_per_clip]")
        if out.dtype not in _DST:
            raise TypeError(f"unsupported output dtype {out.dtype}")
        a = _lib.TransformArgs()
        a.struct_size = C.sizeof(_lib.TransformArgs)
        a.n_clips, a.frames_per_clip = n_clips, frames_per_clip
        a.src = src.data_ptr()
        a.frame_offsets = frame_offsets.data_ptr()
        a.src_row_stride = src_row_stride if src_row_stride is not None else plan.geom.src_w * plan.key.pixel_bytes
        a.params = params_dev.data_ptr()
        a.any_flags = any_flags
        a.dst = out.data_ptr()
        a.dst_dtype = _DST[out.dtype]
        a.normalize = 1 if normalize else 0
        for i in range(5):
            a.dst_stride[i] = int(dst_stride[i])
        for i in range(3):
            a.mean[i], a.std[i] = float(mean[i]), float(std[i])
        ws = self._get_workspace(plan.workspace_bytes(n_clips, frames_per_clip, any_flags))
        a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
        a.stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().nexar_clip_transform(plan.handle, C.byref(a)))
        self.last_launches = int(_lib.lib().nexar_last_launch_count())
        return out


_engines: Dict[int, ClipTransformEngine] = {}


def get_engine(device=None) -> ClipTransformEngine:
    dev = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    e = _engines.get(idx)
    if e is None:
        e = _engines[idx] = ClipTransformEngine(torch.device("cuda", idx))
    return e
