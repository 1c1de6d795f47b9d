"""Clip sampler, Dataset mirror and GPU augmentation loader.

Mirrors the tensor-shaping half of the reference Datasets
(``NvidiaDashcamDataset`` nexar_videos.py:39-496, ``VideoDataset``
nexar_complete_with_validation.py:57-234, the notebook's uniform sampler
inference.ipynb cell 0) around the fused GPU transform:

* ``select_start_frame`` / ``window_indices`` / ``uniform_indices`` — the integer
  window rules, drawing from ``random`` exactly where the reference does.
* ``GpuDashcamDataset`` — same constructor signature and ``__getitem__`` contract
  (``{'frames': [T,cs,cs,3] f32, 'sensor': [T,4], 'target', 'id'}``, zeros on any
  error).  Video decode is a pluggable callable (decord is the default when it is
  installed; decode itself is outside this path).  With ``defer=True`` it returns
  the raw uint8 window and the clip's random decisions instead, so that forked
  DataLoader workers never touch CUDA.
* ``GpuAugLoader`` — wraps a DataLoader over deferred items, copies each uint8
  batch to the device and runs the fused kernel once per batch; yields batches
  whose ``'frames'`` is a ``[B,T,cs,cs,3]`` view of the ``[B,3,T,cs,cs]`` result, so
  the trainers' ``batch['frames'].permute(0,4,1,2,3).float().to(device)``
  (distributed_video_classifier.py:708) is a no-op view chain.
"""
from __future__ import annotations

import random
from typing import Any, Callable, Dict, Iterable, List, Optional, Sequence

import numpy as np
import torch
from torch.utils.data import Dataset, default_collate

from .sensors import find_sensor_path, load_and_sync_sensor, window_sensor
from .source_format import SourceFormat
from .video_aug import GpuVideoTransform


# ---------------------------------------------------------------------------------
# R1: temporal window selection
# ---------------------------------------------------------------------------------
def select_start_frame(num_frames: int, frames_needed: int, strategy: str = "random", rng=random,
                       timestamp_sec: Optional[float] = None, video_fps: float = 0.0) -> int:
    """nexar_videos.py:364-415 (strategies 'random', 'center', 'metadata_time') and
    nexar_complete_with_validation.py:126-155 ('metadata_center')."""
    if strategy in ("metadata_time", "metadata_center"):
        if timestamp_sec is not None and video_fps > 0:
            start = max(0, int(timestamp_sec * video_fps) - frames_needed // 2)
            if start + frames_needed > num_frames:
                start = max(0, num_frames - frames_needed)
        elif strategy == "metadata_time":
            start = rng.randint(0, max(0, num_frames - frames_needed))
        else:
            start = rng.randint(0, num_frames - frames_needed) if num_frames > frames_needed else 0
    elif strategy == "center":
        start = 0
        if num_frames > frames_needed:
            start = max(0, num_frames // 2 - frames_needed // 2)
            if start + frames_needed > num_frames:
                start = max(0, num_frames - frames_needed)
    else:   # 'random'; unknown strategies fall back to it (nexar_videos.py:57-58)
        start = rng.randint(0, num_frames - frames_needed) if num_frames > frames_needed else 0
    return max(0, min(start, num_frames - 1))


def window_indices(num_frames: int, frames_needed: int, start: int) -> List[int]:
    """nexar_videos.py:416-435: consecutive frames, the last one repeated when the video is short."""
    idx = list(range(start, min(start + frames_needed, num_frames)))
    if idx and len(idx) < frames_needed:
        idx += [idx[-1]] * (frames_needed - len(idx))
    return idx[:frames_needed]


def uniform_indices(total_frames: int, num_frames: int) -> List[int]:
    """inference.ipynb cell 0: wrap-pad short videos, else truncating linspace."""
    if total_frames < num_frames:
        idx = np.pad(np.arange(total_frames), (0, num_frames - total_frames), mode="wrap")
    else:
        idx = np.linspace(0, total_frames - 1, num_frames, dtype=int)
    return [int(i) for i in idx]


def model_frame_subsample(num_frames: int) -> List[int]:
    """nexar_arch.py:411-415: the model keeps every other frame when T > 10."""
    return list(range(0, num_frames, 2)) if num_frames > 10 else list(range(num_frames))


# ---------------------------------------------------------------------------------
# Dataset mirror
# ---------------------------------------------------------------------------------
def find_video_path(video_id, base_dirs: Sequence[str]) -> Optional[str]:
    """``_find_video_and_sensor_paths`` (nexar_videos.py:17-36): the FIRST entry of ``os.listdir(<base>/<id>)`` that ends
    in ``.mp4`` or ``.mov`` (e.g. the ``anonymized_<id>.mp4`` files of some source directories), in the first base
    directory that has one; None when there is none."""
    import os
    for base in base_dirs:
        if base is None:
            continue
        video_dir = os.path.join(base, str(video_id))
        if not os.path.exists(video_dir):
            continue
        for name in os.listdir(video_dir):
            if name.endswith(".mp4") or name.endswith(".mov"):
                return os.path.join(video_dir, name)
    return None


def _in_dataloader_worker() -> bool:
    import torch.utils.data as tud
    return tud.get_worker_info() is not None


def _decord_reader(path: str):
    import decord  # not installed in every image; only needed when no decoder is injected
    return decord.VideoReader(path, ctx=decord.cpu(0))


def _to_uint8_array(frames) -> np.ndarray:
    if hasattr(frames, "asnumpy"):
        frames = frames.asnumpy()
    elif isinstance(frames, torch.Tensor):
        frames = frames.cpu().numpy()
    return np.asarray(frames)


def _source_format(defer: bool, pixel_format: str, color_matrix: str, color_range: str) -> SourceFormat:
    """The source format of a dataset's decoded frames: YUV 4:2:0 surfaces are converted on the device by GpuAugLoader."""
    fmt = SourceFormat.of(pixel_format, color_matrix, color_range)
    if fmt.yuv and not defer:
        raise ValueError(f"pixel_format={pixel_format!r} needs defer=True: the surfaces are converted on the device by "
                         "GpuAugLoader")
    return fmt


def _blank_frame(shape, fmt: Optional[Dict[str, str]]) -> np.ndarray:
    return SourceFormat.of(**(fmt or {})).blank_frame(shape)        # fmt: forward_batch keywords, None for RGB


def _deferred_item(frames: torch.Tensor, fmt: SourceFormat, transform: Optional[GpuVideoTransform], **item):
    """A ``defer=True`` item: the window, its record drawn for the visible ``h x w`` and the keywords of YUV surfaces.  A
    decoder that delivers frames the transform cannot take is a set-up error, not a failed item."""
    source = fmt.describe(frames.shape[1:], frames.dtype)
    params = transform.sample_params(1, source.h, source.w)[0] if transform is not None else None
    item = dict(frames_u8=frames, params=params, **item)
    if fmt.yuv:
        item["format"] = fmt._asdict()
    return item


class GpuDashcamDataset(Dataset):
    """``NvidiaDashcamDataset(metadata_df, base_dirs, fps, duration, is_train, skip_missing, transform,
    sample_strategy, sensor_subdir, time_column)`` work-alike for the frames path.  ``metadata_df`` may be a
    pandas DataFrame or a list of dicts with 'id', 'video_type' and, optionally, 'path' / the time column.
    'sensor' is the accelerometer CSV interpolated at the frame times and cut to the clip's window
    (``sensors.py``; nexar_videos.py:301-346, 453-477), zeros when there is no CSV beside the video - pass
    ``sensor_resolver`` to find it somewhere else.

    ``pixel_format="nv12"`` / ``"i420"`` (``defer=True`` only): the decoder's ``get_batch`` returns packed YUV 4:2:0
    surfaces ``[n,H*3/2,W]``; they are what crosses to the main process (half the bytes of RGB) and ``GpuAugLoader``
    converts them on the device with ``color_matrix`` / ``color_range``.  ``"p010"`` / ``"i010"``: uint16 surfaces of
    10-bit video (see ``GpuVideoTransform.forward_batch``), as many bytes as RGB."""

    def __init__(self, metadata_df, base_dirs=None, fps=10, duration=5, is_train=True, skip_missing=True,
                 transform: Optional[GpuVideoTransform] = None, sample_strategy="random", sensor_subdir="signals",
                 time_column=None, *, decoder: Optional[Callable[[str], Any]] = None,
                 path_resolver: Optional[Callable[[str], Optional[str]]] = None, defer: bool = False,
                 video_fps_lookup: Optional[Callable[[str], float]] = None,
                 sensor_resolver: Optional[Callable[[str], Optional[str]]] = None, pixel_format: str = "rgb",
                 color_matrix: str = "bt601", color_range: str = "limited"):
        self.source_format = _source_format(defer, pixel_format, color_matrix, color_range)
        rows = metadata_df.to_dict("records") if hasattr(metadata_df, "to_dict") else list(metadata_df)
        self.fps, self.duration, self.is_train = fps, duration, is_train
        self.transform = transform
        self.sample_strategy = sample_strategy if sample_strategy in ("random", "metadata_time", "center") else "random"
        if self.sample_strategy == "metadata_time" and (time_column is None or not rows or time_column not in rows[0]):
            self.sample_strategy = "random"
        self.time_column = time_column
        self.base_dirs = base_dirs if isinstance(base_dirs, (list, tuple)) else [base_dirs]
        self.decoder = decoder or _decord_reader
        self.defer = defer
        self.video_fps_lookup = video_fps_lookup
        import os
        self.sensor_subdir = sensor_subdir
        self.rows, self.video_paths, self.sensor_paths = [], [], []
        for row in rows:
            path = row.get("path")
            if path is None and path_resolver is not None:
                path = path_resolver(row["id"])
            if path is None and self.base_dirs[0] is not None:
                path = find_video_path(row["id"], self.base_dirs)
                if path is None and not skip_missing:      # nexar_videos.py:80-85: kept, decodes to the zero clip
                    path = os.path.join(self.base_dirs[0], str(row["id"]), f"{row['id']}.mp4")
            if path is None and skip_missing:
                continue
            self.rows.append(row)
            self.video_paths.append(path)
            self.sensor_paths.append(sensor_resolver(path) if sensor_resolver is not None
                                     else find_sensor_path(path, sensor_subdir))

    def __len__(self):
        return len(self.video_paths)

    def _video_fps(self, reader, idx) -> float:
        if self.video_fps_lookup:
            return float(self.video_fps_lookup(self.video_paths[idx]))
        get = getattr(reader, "get_avg_fps", None)
        return float(get()) if get is not None else 30.0

    def _window(self, reader, row, idx):
        """-> (frame indices asked of the decoder, start, end) of nexar_videos.py:364-419; a short window is padded
        afterwards by repeating the last decoded frame (:428-433)."""
        n = len(reader)
        need = self.fps * self.duration
        ts, vfps = None, 0.0
        if self.sample_strategy == "metadata_time":
            ts = row.get(self.time_column)
            vfps = self._video_fps(reader, idx)
        start = select_start_frame(n, need, self.sample_strategy, random, ts, vfps)
        end = min(start + need, n)
        return list(range(start, end)), start, end      # nexar_videos.py:416-419: the decoder is asked for these only

    def _sensor(self, reader, idx, start, end) -> torch.Tensor:
        """nexar_videos.py:453-477 (frame count / fps come from the decoder instead of a second cv2 open)."""
        need = self.fps * self.duration
        n = len(reader)
        table = load_and_sync_sensor(self.sensor_paths[idx], n, self._video_fps(reader, idx), need) \
            if self.sensor_paths[idx] else np.zeros((need, 4), np.float32)
        return torch.from_numpy(window_sensor(table, n, start, end, need)).float()

    def __getitem__(self, idx):
        row = self.rows[idx]
        need = self.fps * self.duration
        target, vid = row.get("video_type"), row.get("id")
        if not self.defer and self.transform is not None and _in_dataloader_worker():
            raise RuntimeError("GpuDashcamDataset(defer=False) runs the CUDA transform inside __getitem__, which cannot "
                               "work in a DataLoader worker process; use defer=True with deferred_collate + GpuAugLoader "
                               "(INTEGRATION.md) or num_workers=0")
        # nexar_videos.py:479-489 swallows EVERY failure and returns an all-zeros clip.  That contract is kept for what
        # can legitimately fail per item - opening / decoding the video, the window arithmetic (e.g. a NaN timestamp),
        # the sensor file - but NOT for the GPU transform: a CUDA, library or out-of-memory error there is a bug or a
        # broken set-up, and training silently on black clips would hide it.
        try:
            reader = self.decoder(self.video_paths[idx])
            indices, start, end = self._window(reader, row, idx)
            frames = _to_uint8_array(reader.get_batch(indices))
            if len(frames) < need:          # nexar_videos.py:429-433
                fmt = self.source_format
                last = frames[-1] if len(frames) else fmt.blank_frame(frames.shape[1:] or fmt.frame_shape(720, 1280))
                frames = np.concatenate([frames, np.repeat(last[None], need - len(frames), axis=0)], axis=0)
            frames = torch.from_numpy(np.ascontiguousarray(frames[:need]))
            sensor = self._sensor(reader, idx, start, end)
        except Exception:
            size = (224, 224) if self.transform else (720, 1280)
            if self.defer:
                return {"frames_u8": None, "params": None, "sensor": torch.zeros(need, 4), "target": target, "id": vid,
                        "need": need}
            return {"frames": torch.zeros(need, size[0], size[1], 3), "sensor": torch.zeros(need, 4), "target": target,
                    "id": vid}
        if self.defer:
            return _deferred_item(frames, self.source_format, self.transform, sensor=sensor, target=target, id=vid,
                                  need=need)
        video = frames.permute(3, 0, 1, 2)                      # nexar_videos.py:441
        video = self.transform(video) if self.transform else video.float() / 255.0
        return {"frames": video.permute(1, 2, 3, 0), "sensor": sensor, "target": target, "id": vid}   # :451


class GpuVideoDataset(Dataset):
    """``VideoDataset(video_paths, labels, video_ids, fps, duration, is_train, transform, sample_strategy,
    center_time_column, metadata_df)`` work-alike (nexar_complete_with_validation.py:57-234): explicit path / label
    lists, strategies 'random', 'center' and 'metadata_center' (window centred on ``metadata_df[center_time_column]``
    seconds, random window when the value is missing), items ``{'frames', 'target', 'id'}`` - no sensor stream.
    ``defer=True`` returns the uint8 window plus the clip's parameter record for ``GpuAugLoader``; ``pixel_format``,
    ``color_matrix`` and ``color_range`` as for ``GpuDashcamDataset``."""

    def __init__(self, video_paths, labels, video_ids=None, fps=10, duration=5, is_train=True,
                 transform: Optional[GpuVideoTransform] = None, sample_strategy="metadata_center",
                 center_time_column=None, metadata_df=None, *, decoder: Optional[Callable[[str], Any]] = None,
                 defer: bool = False, video_fps_lookup: Optional[Callable[[str], float]] = None,
                 pixel_format: str = "rgb", color_matrix: str = "bt601", color_range: str = "limited"):
        self.source_format = _source_format(defer, pixel_format, color_matrix, color_range)
        assert len(video_paths) == len(labels), "video_paths and labels must have same length"      # ncwv:94
        assert sample_strategy in ("random", "center", "metadata_center"), \
            "sample_strategy must be 'random', 'center', or 'metadata_center'"                       # ncwv:95-96
        self.video_paths, self.labels = list(video_paths), list(labels)
        self.video_ids = list(video_ids) if video_ids is not None else list(range(len(self.video_paths)))
        self.fps, self.duration, self.is_train = fps, duration, is_train
        self.transform, self.sample_strategy = transform, sample_strategy
        self.center_time_column = center_time_column
        self.decoder = decoder or _decord_reader
        self.defer = defer
        self.video_fps_lookup = video_fps_lookup
        self._center_time: Dict[Any, Any] = {}
        if sample_strategy == "metadata_center":
            assert metadata_df is not None, "metadata_df required for 'metadata_center' strategy"  # ncwv:99
            assert center_time_column is not None, "center_time_column required for 'metadata_center' strategy"
            rows = metadata_df.to_dict("records") if hasattr(metadata_df, "to_dict") else list(metadata_df)
            assert not rows or center_time_column in rows[0], f"Column '{center_time_column}' not found in metadata"
            for row in rows:                                     # first row per id wins (ncwv:207 .iloc[0])
                self._center_time.setdefault(row.get("id"), row.get(center_time_column))

    def __len__(self):
        return len(self.video_paths)

    def _center(self, idx):
        """ncwv:198-211: None when the id is unknown or the value is NaN / missing."""
        v = self._center_time.get(self.video_ids[idx])
        try:
            return None if v is None or v != v else float(v)
        except (TypeError, ValueError):
            return None

    def __getitem__(self, idx):
        label, vid = self.labels[idx], self.video_ids[idx]
        need = self.fps * self.duration
        if not self.defer and self.transform is not None and _in_dataloader_worker():
            raise RuntimeError("GpuVideoDataset(defer=False) runs the CUDA transform inside __getitem__, which cannot work "
                               "in a DataLoader worker process; use defer=True with deferred_collate + GpuAugLoader or "
                               "num_workers=0")
        try:   # decode / window failures become the zero clip (ncwv:183-190); transform errors propagate
            reader = self.decoder(self.video_paths[idx])
            n = len(reader)
            ts, vfps = None, 0.0
            if self.sample_strategy == "metadata_center":
                ts = self._center(idx)
                if self.video_fps_lookup:
                    vfps = float(self.video_fps_lookup(self.video_paths[idx]))
                else:                                            # ncwv:107-116: 30.0 when the container does not say
                    get = getattr(reader, "get_avg_fps", None)
                    vfps = float(get()) if get is not None else 30.0
                    vfps = vfps if vfps > 0 else 30.0
            start = select_start_frame(n, need, self.sample_strategy, random, ts, vfps)
            indices = list(range(start, min(start + need, n)))
            frames = _to_uint8_array(reader.get_batch(indices))
            if len(frames) < need:                               # ncwv:213-227
                if len(frames) > 0:
                    frames = np.concatenate([frames, np.repeat(frames[-1][None], need - len(frames), axis=0)], axis=0)
                else:
                    blank = self.source_format.blank_frame(self.source_format.frame_shape(720, 1280))
                    frames = np.repeat(blank[None], need, axis=0)
            frames = torch.from_numpy(np.ascontiguousarray(frames[:need]))
        except Exception:
            if self.defer:
                return {"frames_u8": None, "params": None, "target": label, "id": vid, "need": need}
            size = (224, 224) if self.transform else (720, 1280)   # ncwv:183-190
            return {"frames": torch.zeros(need, size[0], size[1], 3), "target": label, "id": vid}
        if self.defer:
            return _deferred_item(frames, self.source_format, self.transform, target=label, id=vid, need=need)
        video = frames.permute(3, 0, 1, 2)                      # ncwv:172
        video = self.transform(video) if self.transform else video.float() / 255.0
        return {"frames": video.permute(1, 2, 3, 0), "target": label, "id": vid}   # ncwv:181


def deferred_collate(items: Sequence[Dict[str, Any]]) -> Dict[str, Any]:
    """collate_fn for ``defer=True`` datasets.  The uint8 windows are stacked PER SOURCE RESOLUTION (a batch may mix
    720p, 1080p and portrait videos: the reference transforms every clip to cs x cs before collation, so it never
    sees the difference): ``groups`` is a list of ``{'frames_u8': [n,T,H,W,3], 'index': positions in the batch,
    'params': [...]}``, plus the source ``'format'`` (forward_batch keywords) for YUV surfaces.  Failed items
    (``frames_u8 is None``) are in no group and become the zero clip.  'sensor' is present for the NvidiaDashcamDataset
    protocol only."""
    by_shape: Dict[Any, Dict[str, Any]] = {}
    for pos, it in enumerate(items):
        f = it["frames_u8"]
        if f is None:
            continue
        fmt = it.get("format")
        g = by_shape.setdefault((tuple(f.shape), tuple(sorted(fmt.items())) if fmt else None),
                                {"frames": [], "index": [], "params": [], "format": fmt})
        g["frames"].append(f)
        g["index"].append(pos)
        g["params"].append(it["params"])
    batch = {   # default_collate: inside a DataLoader worker the stacks go straight into shared memory (deferred.py)
        "groups": [dict({"frames_u8": default_collate(g["frames"]), "index": g["index"], "params": g["params"]},
                        **({"format": g["format"]} if g["format"] else {}))
                   for g in by_shape.values()],
        "valid": [it["frames_u8"] is not None for it in items],
        "target": [it["target"] for it in items],
        "id": [it["id"] for it in items],
        "need": items[0].get("need") if items else None,
    }
    if items and all("sensor" in it for it in items):
        batch["sensor"] = default_collate([it["sensor"] for it in items])
    return batch


class GpuAugLoader:
    """Iterates a DataLoader of deferred batches and runs the fused transform on the device: once per batch, or once
    per source resolution when a batch mixes several."""

    def __init__(self, loader: Iterable, transform: GpuVideoTransform, device=None, out_dtype: Optional[torch.dtype] = None):
        self.loader, self.transform = loader, transform
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.out_dtype = out_dtype

    def __len__(self):
        return len(self.loader)

    def __iter__(self):
        tf = self.transform
        cs = tf.crop_size
        for batch in self.loader:
            n = len(batch["valid"])
            groups = batch["groups"]
            out = None
            if len(groups) == 1 and len(groups[0]["index"]) == n:      # the common case: one resolution, nothing failed
                g = groups[0]
                params = g["params"] if all(p is not None for p in g["params"]) else None
                out = tf.forward_batch(g["frames_u8"].to(self.device, non_blocking=True), params=params,
                                       out_dtype=self.out_dtype, **g.get("format", {}))         # [n,3,T,cs,cs]
            else:
                for g in groups:
                    params = g["params"] if all(p is not None for p in g["params"]) else None
                    res = tf.forward_batch(g["frames_u8"].to(self.device, non_blocking=True), params=params,
                                           out_dtype=self.out_dtype, **g.get("format", {}))
                    if out is None:   # failed items stay the reference's all-zeros clip (nexar_videos.py:479-489)
                        out = torch.zeros((n,) + tuple(res.shape[1:]), dtype=res.dtype, device=self.device)
                    out[torch.tensor(g["index"], device=self.device)] = res
                if out is None:
                    t = batch["need"] if batch.get("need") else batch["sensor"].shape[1]
                    out = torch.zeros((n, 3, t, cs, cs), dtype=self.out_dtype or tf.out_dtype, device=self.device)
            res_batch = {"frames": out.permute(0, 2, 3, 4, 1), "target": batch["target"], "id": batch["id"]}
            if "sensor" in batch:
                res_batch["sensor"] = batch["sensor"]
            yield res_batch


def shard_clips(n_clips: int, rank: int, world: int) -> range:
    """Contiguous split of a batch over ranks (SURVEY.md section 8e): clips are independent, no collective."""
    per = (n_clips + world - 1) // world
    return range(min(n_clips, rank * per), min(n_clips, (rank + 1) * per))
