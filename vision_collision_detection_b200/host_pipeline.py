"""Host-buffer entry point: pinned uint8 clips in host memory -> H2D -> fused transform -> D2H.

This is the path a DataLoader-side caller exercises (decoded frames live in host memory,
nexar_videos.py:422-438) and what bench.py reports as ``e2e``.  The batch is cut into chunks
that round-robin over a few CUDA streams so that the H2D copy of one chunk overlaps the
kernels and the D2H copy of its neighbours (PCIe is full duplex).
"""
from __future__ import annotations

from typing import Any, Dict, List, Optional

import torch

from .engine import ClipTransformEngine
from .video_aug import GpuVideoTransform, check_pixel_format, source_dtype


def bind_to_gpu_numa_node(device_index: int) -> Optional[List[int]]:
    """Pin the calling process to the CPUs NVML reports as local to the GPU, so that pinned buffers allocated afterwards
    (first touch) and the copy-submitting thread sit on the GPU's own NUMA node.  With several ranks per host this is
    what keeps every GPU's H2D stream off the inter-socket link.  Returns the CPU list, or None when NVML or the
    affinity call is unavailable (nothing is changed then)."""
    try:
        import os

        import pynvml
        pynvml.nvmlInit()
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = device_index
        if visible:
            ids = [v.strip() for v in visible.split(",") if v.strip()]
            if device_index < len(ids) and ids[device_index].isdigit():
                phys = int(ids[device_index])
        handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(handle, (n_cpu + 63) // 64)
        cpus = [64 * i + b for i, wd in enumerate(words) for b in range(64) if (int(wd) >> b) & 1]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return allowed
    except Exception:  # noqa: BLE001 - an optimisation only
        return None


class HostClipPipeline:
    def __init__(self, transform: GpuVideoTransform, n_clips: int, frames: int, height: int, width: int,
                 device=None, clips_per_chunk: int = 4, n_streams: int = 3, out_dtype: Optional[torch.dtype] = None,
                 pixel_format: str = "rgb", color_matrix: str = "bt601", color_range: str = "limited"):
        """``pixel_format="nv12"`` / ``"i420"``: the host clips are YUV 4:2:0 decoder surfaces, uint8 ``[B,T,H*3/2,W]``
        — half the bytes of RGB over PCIe (the link is what bounds this path), converted to RGB on the device with
        ``color_matrix`` / ``color_range`` (see ``GpuVideoTransform.forward_batch``).  ``"p010"`` / ``"i010"``: 16-bit
        surfaces, uint16 ``[B,T,H*3/2,W]`` — as many bytes as RGB over PCIe."""
        self.tf = transform
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        yuv = check_pixel_format(pixel_format, color_matrix, color_range)
        self.pixel_format = pixel_format
        self.yuv_kw = dict(pixel_format=pixel_format, color_matrix=color_matrix, color_range=color_range)
        self.shape = (n_clips, frames, height * 3 // 2, width) if yuv else (n_clips, frames, height, width, 3)
        self.dtype = source_dtype(pixel_format)
        self.chunk = max(1, min(clips_per_chunk, n_clips))
        self.out_dtype = out_dtype or transform.out_dtype
        cs = transform.crop_size
        self.streams = [torch.cuda.Stream(self.device) for _ in range(n_streams)]
        self.engines = [ClipTransformEngine(self.device) for _ in range(n_streams)]
        self.dev_in = [torch.empty((self.chunk,) + self.shape[1:], dtype=self.dtype, device=self.device)
                       for _ in range(n_streams)]
        self.dev_out = [torch.empty((self.chunk, 3, frames, cs, cs), dtype=self.out_dtype, device=self.device)
                        for _ in range(n_streams)]
        # two result buffers so that submit() of batch i+1 can overlap the D2H tail of batch i (PCIe is full duplex)
        self.host_outs = [torch.empty((n_clips, 3, frames, cs, cs), dtype=self.out_dtype).pin_memory() for _ in range(2)]
        self.host_out = self.host_outs[0]
        self._done = [[torch.cuda.Event() for _ in range(n_streams)] for _ in range(2)]
        self._slot = 0

    def pinned_input(self) -> torch.Tensor:
        return torch.empty(self.shape, dtype=self.dtype).pin_memory()

    @torch.no_grad()
    def submit(self, host_clips: torch.Tensor, params: Optional[List[Dict[str, Any]]] = None) -> int:
        """Enqueue one batch (pinned uint8 [B,T,H,W,3], or the surfaces of ``pixel_format``); returns a ticket for ``wait``.  At most two batches may be
        in flight; the input buffer must stay untouched until its ticket has been waited for."""
        if tuple(host_clips.shape) != self.shape or host_clips.dtype != self.dtype:
            raise ValueError(f"expected {self.dtype} {self.shape}")
        n = self.shape[0]
        if params is None:
            h = self.shape[2] * 2 // 3 if self.pixel_format != "rgb" else self.shape[2]
            params = self.tf.sample_params(n, h, self.shape[3])
        slot = self._slot
        self._slot ^= 1
        host_out = self.host_outs[slot]
        # inputs and outputs are host buffers: nothing to order against the caller's stream, and consecutive
        # batches may overlap freely (each side stream is in-order, so its staging buffers are reused safely)
        for k, lo in enumerate(range(0, n, self.chunk)):
            hi = min(n, lo + self.chunk)
            i = k % len(self.streams)
            with torch.cuda.stream(self.streams[i]):
                din = self.dev_in[i][: hi - lo]
                din.copy_(host_clips[lo:hi], non_blocking=True)
                dout = self.dev_out[i][: hi - lo]
                self.tf.forward_batch(din, params=params[lo:hi], out=dout, engine=self.engines[i], **self.yuv_kw)
                host_out[lo:hi].copy_(dout, non_blocking=True)
        for i, s in enumerate(self.streams):
            self._done[slot][i].record(s)
        return slot

    def wait(self, ticket: int) -> torch.Tensor:
        """Block until the batch behind ``ticket`` is complete; returns its pinned [B,3,T,cs,cs] result."""
        for ev in self._done[ticket]:
            ev.synchronize()
        return self.host_outs[ticket]

    @torch.no_grad()
    def run(self, host_clips: torch.Tensor, params: Optional[List[Dict[str, Any]]] = None) -> torch.Tensor:
        """host_clips: pinned uint8 [B,T,H,W,3] (or [B,T,H*3/2,W] for nv12 / i420, uint16 for p010 / i010).  Returns the pinned [B,3,T,cs,cs] result (valid on return)."""
        return self.wait(self.submit(host_clips, params))
