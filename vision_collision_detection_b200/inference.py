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
``MultiWindowStream`` / ``WindowPredictor.predict_step`` do that for many videos at once (one per camera), with a few
library calls per step whatever the number of videos.
"""
from __future__ import annotations

import itertools
from typing import Any, Callable, Dict, Iterable, Iterator, List, NamedTuple, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from .engine import get_engine
from .params import pack_clip_params
from .source_format import FrameSource, SourceFormat
from .video_aug import GpuVideoTransform, create_video_transforms
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
        out = self.tf.forward_batch(video_u8.unsqueeze(0), layout="BTCHW", out_dtype=self.out_dtype, pixel_format=pixel_format,
                                    color_matrix=color_matrix, color_range=color_range, frame_size=frame_size)  # [1,N,3,cs,cs]
        n = out.shape[1]
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


def check_chunk(frames: torch.Tensor, pixel_format: str = "rgb", color_matrix: str = "bt601", color_range: str = "limited",
                frame_size=None) -> FrameSource:
    """Validates a chunk ``[n,*frame]`` of ``n >= 1`` decoded frames and its source-format keywords -> the source that
    every later chunk of the same video must equal."""
    source = SourceFormat.of(pixel_format, color_matrix, color_range).describe(frames.shape[1:], frames.dtype, frame_size,
                                                                              decoded=True)
    if frames.shape[0] < 1:
        raise ValueError("empty chunk")
    return source


def _mismatch(have, source) -> str:
    return f"the stream's frames are {have}; a chunk of {source} cannot join it"


def _draw_record(tf: GpuVideoTransform, source: FrameSource) -> Dict[str, Any]:
    """The parameter record of a video of frames ``source``, drawn for its visible ``h x w`` as ``frames()`` draws it
    for a whole video, with the byte-range flag (every chunk is scaled by 1/255, ``NEXAR_RANGE_255``)."""
    return dict(tf.sample_params(1, source.h, source.w)[0], range_255=True)


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
        self._source: Optional[FrameSource] = None      # the first chunk's: every chunk must equal it
        self._format: Dict[str, Any] = {}                # its forward_batch keywords
        self._params = None
        self._ring: Optional[torch.Tensor] = None
        self._staging: Optional[torch.Tensor] = None

    def _start(self, frames: torch.Tensor, source: FrameSource):
        self._params = [_draw_record(self.tf, source)]
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
        source = check_chunk(frames, pixel_format, color_matrix, color_range, frame_size)
        if self._source is None:
            self._start(frames, source)
            self._format = dict(source.format._asdict(), frame_size=source.frame_size)
            self._source = source
        elif source != self._source:
            raise ValueError(_mismatch(self._source, source))
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


class StepRound(NamedTuple):
    """One round of a ``MultiWindowStream`` step (``multi_stream_schedule``).

    - ``pieces``: ``(q, lo, hi, slot)``: frames ``lo .. hi-1`` of queue entry ``q`` are transformed into step slots
      ``slot ..``; ordered by source group (in order of first appearance), then push order, so each group's frames
      fill a contiguous run of step slots.
    - ``groups``: ``(group, p0, p1)``: pieces ``p0 .. p1-1`` belong to ``group``.
    - ``windows``: ``(v, start)`` of every window the round completes, by video then start.
    - ``gather``: int32 ``[len(windows) * window]``: the pool slot of each window frame (the table of
      ``nexar_gather_windows_table``).
    - ``copy_src`` / ``copy_dst``: int32 step slots and tail slots: each video's last ``min(window - 1, new frames)``
      frames are copied into its tail, after the gather.
    - ``done``: videos that end in this round (closed, every frame seen): their tail slots are free after it."""
    pieces: List[Tuple[int, int, int, int]]
    groups: List[Tuple[Any, int, int]]
    windows: List[Tuple[int, int]]
    gather: np.ndarray
    copy_src: np.ndarray
    copy_dst: np.ndarray
    done: List[int]


def multi_stream_schedule(videos: Sequence[Tuple[int, int, bool]], queue: Sequence[Tuple[int, int, Any]], window: int,
                          stride: int, step_frames: int) -> List[StepRound]:
    """The work of one ``MultiWindowStream`` step, on the host.  ``videos[v] = (seen, tail, closed)``: frames already
    transformed, the first of the video's ``window - 1`` tail slots, and whether the video has been closed.
    ``queue[q] = (v, n, group)``: the chunks pushed since the last step, in push order (``group``: the source group).

    Pool slots ``0 .. step_frames-1`` are the step region.  Video frame ``f`` of an earlier round or step lives in tail
    slot ``tail + f % (window - 1)``; only its last ``window - 1`` frames are kept, and a window that completes in a round
    starts at or after ``seen - window + 1``, so each of its frames is either there or new in the round.  The frames are
    taken in push order, at most ``step_frames`` per round.  A closed video ends in the round that takes its last frame
    (round 0 when it has none queued); one that saw fewer than ``window`` frames then gets its padded window (its last
    frame repeated, nexar_videos.py:429-433)."""
    tail_len = window - 1
    nv = len(videos)
    seen = np.array([v[0] for v in videos], np.int64)
    tail = np.array([v[1] for v in videos], np.int64)
    left = np.zeros(nv, np.int64)                  # frames still queued per video
    for v, n, _ in queue:
        left[v] += n
    ended = np.zeros(nv, bool)
    rounds: List[StepRound] = []
    qi, qoff = 0, 0
    while True:
        taken, budget = [], step_frames
        while qi < len(queue) and budget > 0:
            v, n, g = queue[qi]
            take = min(n - qoff, budget)
            taken.append((qi, qoff, qoff + take))
            budget -= take
            qoff += take
            if qoff == n:
                qi, qoff = qi + 1, 0
        order: Dict[Any, int] = {}
        for q, _, _ in taken:
            order.setdefault(queue[q][2], len(order))
        taken.sort(key=lambda p: order[queue[p[0]][2]])          # stable: push order within a group
        pieces, groups, new_slots = [], [], {}
        slot = 0
        for i, (q, lo, hi) in enumerate(taken):
            g = queue[q][2]
            if not groups or groups[-1][0] != g:
                groups.append([g, i, i])
            groups[-1][2] = i + 1
            pieces.append((q, lo, hi, slot))
            new_slots.setdefault(queue[q][0], []).extend(range(slot, slot + hi - lo))
            slot += hi - lo
        n_new = np.zeros(nv, np.int64)
        for v, sl in new_slots.items():
            n_new[v] = len(sl)
            left[v] -= len(sl)
        done = [v for v in range(nv) if videos[v][2] and not ended[v] and left[v] == 0]
        ended[done] = True
        # windows, by video then start
        win_v, win_s = [], []
        for v in sorted(set(new_slots) | set(done)):
            k0 = windows_complete(int(seen[v]), window, stride)
            k1 = windows_complete(int(seen[v] + n_new[v]), window, stride)
            win_v += [v] * (k1 - k0)
            win_s += [k * stride for k in range(k0, k1)]
            if v in done and seen[v] + n_new[v] < window:
                win_v.append(v)
                win_s.append(0)
        gather = np.zeros(0, np.int32)
        if win_v:
            wv, ws = np.array(win_v, np.int64), np.array(win_s, np.int64)
            vids = sorted(new_slots)
            flat = np.array([s for v in vids for s in new_slots[v]] or [0], np.int64)
            off = np.zeros(nv, np.int64)
            pos = 0
            for v in vids:
                off[v] = pos
                pos += len(new_slots[v])
            f = np.minimum(ws[:, None] + np.arange(window)[None, :], (seen[wv] + n_new[wv] - 1)[:, None])
            s0 = seen[wv][:, None]
            is_new = f >= s0
            from_step = flat[np.clip(off[wv][:, None] + f - s0, 0, flat.size - 1)]
            from_tail = tail[wv][:, None] + f % max(tail_len, 1)
            gather = np.where(is_new, from_step, from_tail).astype(np.int32).reshape(-1)
        copy_src, copy_dst = [], []
        if tail_len > 0:
            for v, sl in new_slots.items():
                if ended[v]:
                    continue                                     # nothing reads the tail of a video that has ended
                keep = min(tail_len, len(sl))
                first = int(seen[v]) + len(sl) - keep
                copy_src += sl[len(sl) - keep:]
                copy_dst += [int(tail[v]) + (first + i) % tail_len for i in range(keep)]
        seen += n_new
        rounds.append(StepRound(pieces, [tuple(g) for g in groups], list(zip(win_v, win_s)), gather,
                                np.array(copy_src, np.int32), np.array(copy_dst, np.int32), done))
        if qi == len(queue):
            return rounds


def group_frames(parts: Sequence[torch.Tensor], frame_bytes: int, device: torch.device,
                 staging_for: Callable[[int], torch.Tensor]) -> Tuple[torch.Tensor, np.ndarray]:
    """The frames of one transform call from several chunks -> (base tensor, int64 byte offset of every frame from its
    ``data_ptr()``), the frames in the order of ``parts``.  A part on ``device`` whose address is a multiple of 16 is
    read in place; every other part (host frames, or a device view at any other address) is copied, with one
    non-blocking copy, into the buffer ``staging_for(n)`` returns for the ``n`` frames staged.  The library reads the
    frames with 16-byte loads at base + offset whenever the base and the row stride are multiples of 16, and a frame
    at any other address would be a misaligned-address fault; the parts taken in place and the staging buffer both
    start on 16 bytes, so with frames of a multiple of 16 bytes every offset is one."""
    in_place = [p.device == device and p.data_ptr() % 16 == 0 for p in parts]
    n_staged = sum(p.shape[0] for p, keep in zip(parts, in_place) if not keep)
    staging = staging_for(n_staged) if n_staged else None
    srcs, addr, at = [], [], 0
    for part, keep in zip(parts, in_place):
        if not keep:
            dst = staging[at:at + part.shape[0]]
            dst.copy_(part, non_blocking=True)
            at += part.shape[0]
            part = dst
        srcs.append(part)
        addr.append(part.data_ptr() + frame_bytes * np.arange(part.shape[0], dtype=np.int64))
    base = min(srcs, key=lambda t: t.data_ptr())       # offsets from the lowest frame address: all >= 0
    return base, np.concatenate(addr) - base.data_ptr()


class _Video:
    """A video of a ``MultiWindowStream``: its key, record / tail slot, frame counts and source."""
    __slots__ = ("key", "slot", "seen", "closed", "source")

    def __init__(self, key, slot: int, source: FrameSource):
        self.key, self.slot, self.source = key, slot, source
        self.seen, self.closed = 0, False


class MultiWindowStream:
    """Sliding windows over many videos at once, each arriving in chunks of consecutive frames (one per camera, say),
    in bounded device memory: every ``step()`` transforms the frames pushed since the last one with one transform call per
    source group (frames of equal shape, dtype and source format), then builds every window they complete with one
    gather and updates each video's last frames with one copy, whatever the number of videos.

    ``push(key, chunk, **source_format)`` queues a chunk of video ``key`` (any hashable; the first push opens the video,
    and draws its parameter record as ``WindowStream`` does); ``close(key)`` ends it.  ``step()`` returns ``(keys, starts,
    windows)``: ``windows`` is a contiguous ``[K,3,window,cs,cs]`` tensor of every window completed, grouped by video in the
    order the videos were opened and by start within a video, with each window's key and start frame.  For every video,
    the windows it gets across all steps equal ``WindowStream(window, stride, transform, out_dtype)`` fed the same chunks,
    bit for bit, under that class's conditions (a pixel above 1 in the video, no gaussian noise), for any interleaving of
    pushes, steps and closes.  A video shorter than ``window`` gets its padded window at the step after its ``close``; a
    push after ``close`` opens a new video under the same key.

    Chunks are what ``WindowStream.push`` takes, on the device (read in place when it starts on a 16-byte boundary, as
    every tensor torch allocates does; copied otherwise) or the host (copied with a non-blocking copy; do not overwrite
    a pinned chunk before the step's work has run).  Videos may differ in resolution and format.
    Device memory is one pool of ``max_frames_per_step`` step slots plus ``window - 1`` slots per open video, and a
    host-staging buffer of at most ``max_frames_per_step`` frames per source group; a step with more queued frames than
    ``max_frames_per_step`` runs in rounds, in push order.  It never depends on how long a video runs, and it is released
    when every video has been closed and stepped.  All videos live on one device (the first chunk's, or the current one
    for a host chunk); everything is enqueued on its current CUDA stream."""

    def __init__(self, window: int = 16, stride: int = 8, transform: Optional[GpuVideoTransform] = None,
                 out_dtype: torch.dtype = torch.bfloat16, max_frames_per_step: int = 1024):
        if window < 1 or stride < 1 or max_frames_per_step < 1:
            raise ValueError(f"window, stride and max_frames_per_step must be >= 1, got {window}, {stride}, "
                             f"{max_frames_per_step}")
        self.window, self.stride, self.max_frames_per_step = int(window), int(stride), int(max_frames_per_step)
        self.tf = transform or create_video_transforms(mode="val", out_dtype=out_dtype)
        self.out_dtype = out_dtype
        self.device: Optional[torch.device] = None
        self._videos: Dict[int, _Video] = {}      # every video not yet ended, in the order they were opened
        self._open: Dict[Any, _Video] = {}        # key -> the video that takes its pushes
        self._queue: List[Tuple[_Video, torch.Tensor]] = []
        self._next_id = 0
        self._free: List[int] = []                # record / tail slots of ended videos
        self._n_slots = 0
        self._records: Optional[np.ndarray] = None      # packed NexarClipParams, one per record slot
        self._pool: Optional[torch.Tensor] = None       # [max_frames_per_step + n_slots * (window - 1), 3, cs, cs]
        self._staging: Dict[FrameSource, torch.Tensor] = {}

    def _tail(self, slot: int) -> int:
        return self.max_frames_per_step + slot * (self.window - 1)

    def _take_slot(self, dev: torch.device) -> int:
        if not self._free:                  # grow the pool and the records by doubling; the tails move with the copy
            n = max(4, 2 * self._n_slots)
            cs = self.tf.crop_size
            pool = torch.empty((self._tail(n), 3, cs, cs), dtype=self.out_dtype, device=dev)
            records = np.zeros(n, _lib.CLIP_PARAMS_DTYPE)
            if self._pool is not None:
                pool[:self._pool.shape[0]].copy_(self._pool)
                records[:self._n_slots] = self._records
            self._pool, self._records = pool, records
            self._free = list(range(n - 1, self._n_slots - 1, -1))
            self._n_slots = n
        return self._free.pop()

    @torch.no_grad()
    def push(self, key, frames: torch.Tensor, pixel_format: str = "rgb", color_matrix: str = "bt601",
             color_range: str = "limited", frame_size=None) -> None:
        """Queues a chunk of ``n >= 1`` consecutive frames of video ``key`` for the next ``step()``."""
        source = check_chunk(frames, pixel_format, color_matrix, color_range, frame_size)
        video = self._open.get(key)
        if video is not None and source != video.source:
            raise ValueError(_mismatch(video.source, source))
        dev = self.device if self.device is not None else (
            frames.device if frames.is_cuda else torch.device("cuda", torch.cuda.current_device()))
        if frames.is_cuda and frames.device != dev:
            raise ValueError(f"the streams live on {dev}, the chunk on {frames.device}")
        if video is None:
            rec = _draw_record(self.tf, source)
            packed, _ = pack_clip_params([rec], self.tf.crop_size, self.tf.video_aug)
            _lib.table_lib()          # a library without the table gather fails here, before any work
            self.device = dev
            video = _Video(key, self._take_slot(dev), source)
            self._records[video.slot] = packed[0]
            self._videos[self._next_id] = self._open[key] = video
            self._next_id += 1
        self._queue.append((video, frames.contiguous() if frames.is_cuda else frames))

    def close(self, key) -> None:
        """Ends video ``key``: its last windows (the padded one of a video shorter than ``window``) come out of the next
        ``step()``, and its slots are freed there."""
        video = self._open.pop(key, None)
        if video is None:
            raise ValueError(f"no open video under key {key!r}")
        video.closed = True

    def _windows_out(self, k: int) -> torch.Tensor:
        cs = self.tf.crop_size
        dev = self.device if self.device is not None else torch.device("cuda", torch.cuda.current_device())
        return torch.empty((k, 3, self.window, cs, cs), dtype=self.out_dtype, device=dev)

    def _staging_for(self, source: FrameSource, n: int) -> torch.Tensor:
        buf = self._staging.get(source)
        if buf is None or buf.shape[0] < n:
            rows = min(self.max_frames_per_step, max(n, 2 * buf.shape[0] if buf is not None else n))
            buf = self._staging[source] = torch.empty((rows,) + source.shape, dtype=source.dtype, device=self.device)
        return buf

    def _gather(self, table: torch.Tensor, n: int, dst: Optional[torch.Tensor], dst_slots: Optional[torch.Tensor]):
        pool = self._pool
        _lib.check(_lib.table_lib().nexar_gather_windows_table(
            pool.data_ptr(), pool.shape[0], pool[0, 0].numel() * pool.element_size(), 1 if dst is None else self.window,
            table.data_ptr(), n, None if dst is None else dst.data_ptr(), None if dst_slots is None else dst_slots.data_ptr(),
            torch.cuda.current_stream(pool.device).cuda_stream))

    def _round(self, eng, rnd: StepRound, videos: List[_Video]) -> Optional[torch.Tensor]:
        """Enqueues one round: a transform call per source group into the step slots, the window gather, the tail copy."""
        calls, offsets = [], []
        for _, p0, p1 in rnd.groups:
            pieces = rnd.pieces[p0:p1]
            fs, n = self._queue[pieces[0][0]][0].source, sum(hi - lo for _, lo, hi, _ in pieces)
            base, offs = group_frames([self._queue[q][1][lo:hi] for q, lo, hi, _ in pieces], fs.frame_bytes, self.device,
                                      lambda k: self._staging_for(fs, k))
            offsets.append(offs)
            rec = [np.full(hi - lo, self._queue[q][0].slot, np.int64) for q, lo, hi, _ in pieces]
            params = self._records[np.concatenate(rec)]          # one vectorised index into the packed records
            calls.append((base, fs, pieces[0][3], n, params))
        # frame offsets and both slot tables: one upload through the engine's pinned staging
        parts = offsets + [rnd.gather, rnd.copy_src, rnd.copy_dst]
        raw = eng.upload_params(np.concatenate([np.ascontiguousarray(x).view(np.uint8) for x in parts])) \
            if any(x.size for x in parts) else None
        views, at = [], 0
        for x in parts:
            views.append(raw[at:at + x.nbytes].view(torch.int64 if x.dtype == np.int64 else torch.int32) if x.size else None)
            at += x.nbytes
        for (base, fs, slot, n, params), offs in zip(calls, views):
            any_flags = int(np.bitwise_or.reduce(params["flags"]))
            self.tf._transform_packed(eng, base, offs, n, 1, params, any_flags, fs, self._pool[slot:slot + n].unsqueeze(1),
                                      "BTCHW", self.out_dtype)
        gather, copy_src, copy_dst = views[len(calls):]
        out = None
        if rnd.windows:
            out = self._windows_out(len(rnd.windows))
            self._gather(gather, len(rnd.windows), out, None)
        if copy_src is not None:             # after the gather, which may read the tail slots this overwrites
            self._gather(copy_src, rnd.copy_src.size, None, copy_dst)
        return out

    @torch.no_grad()
    def step(self) -> Tuple[List[Any], List[int], torch.Tensor]:
        """Transforms every queued frame -> (keys, starts, ``[K,3,window,cs,cs]``) of the windows completed, grouped by
        video in the order the videos were opened, by start within a video.  A step with nothing queued and no video
        closed launches nothing."""
        if not self._queue and not any(v.closed for v in self._videos.values()):
            return [], [], self._windows_out(0)
        ids = list(self._videos)
        videos = [self._videos[i] for i in ids]
        pos = {id(v): i for i, v in enumerate(videos)}
        rounds = multi_stream_schedule([(v.seen, self._tail(v.slot), v.closed) for v in videos],
                                       [(pos[id(v)], c.shape[0], v.source) for v, c in self._queue],
                                       self.window, self.stride, self.max_frames_per_step)
        eng = get_engine(self.device)
        outs, order = [], []
        with torch.cuda.device(self.device):
            for rnd in rounds:
                out = self._round(eng, rnd, videos)
                if out is not None:
                    outs.append(out)
                    order += rnd.windows
                for q, lo, hi, _ in rnd.pieces:
                    self._queue[q][0].seen += hi - lo
                for v in rnd.done:
                    self._free.append(videos[v].slot)
                    del self._videos[ids[v]]
        self._queue = []
        if not self._videos:                 # every video has ended: give the pool and the staging buffers back
            self._pool, self._records, self._free, self._n_slots, self._staging = None, None, [], 0, {}
        if not outs:
            return [], [], self._windows_out(0)
        windows = outs[0]
        if len(outs) > 1:                    # rounds: put each video's windows together again
            perm = sorted(range(len(order)), key=lambda i: order[i])
            windows = torch.cat(outs)[torch.tensor(perm, dtype=torch.int64)]
            order = [order[i] for i in perm]
        return [videos[v].key for v, _ in order], [s for _, s in order], windows


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

    @torch.no_grad()
    def predict_step(self, keys: Sequence[Any], starts: Sequence[int], windows: torch.Tensor,
                     fps: float = 30.0) -> List[Dict[str, Any]]:
        """Classifies the windows of one ``MultiWindowStream.step()`` (made with this predictor's window) in batches of
        ``batch_size``: one dictionary per window, in the step's order, as ``predict`` returns them with the window's
        stream key as ``video_path``."""
        results: List[Dict[str, Any]] = []
        for lo in range(0, len(keys), self.batch_size):
            batch = self._classify(windows[lo:lo + self.batch_size], list(starts[lo:lo + self.batch_size]), "", fps)
            for r, key in zip(batch, keys[lo:lo + self.batch_size]):
                r["video_path"] = key
            results.extend(batch)
        return results

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
