"""Zero-line drop-in for the reference's Dataset and trainers (SURVEY.md section 8b, option ii).

The reference transforms every clip on the CPU inside ``Dataset.__getitem__`` (forked DataLoader workers,
nexar_videos.py:444-451), collates the float results with ``default_collate``, pins them, and the trainer
runs ``batch['frames'].permute(0, 4, 1, 2, 3).float().to(device)`` (nexar_train.py:1139, dvc:708,
nexar_inference.py:248).  CUDA cannot run in those workers.  A transform built with ``deferred=True``
therefore does only the host part of its job inside ``__getitem__`` — it draws the clip's random decisions from
``random`` in the reference's order and keeps the decoded uint8 frames — and returns a :class:`DeferredClip`.
That object follows the reference's own lines unchanged:

    frames = self.transform(frames)           # -> DeferredClip                      nexar_videos.py:445
    frames = frames.permute(1, 2, 3, 0)       # recorded                             :451
    default_collate([...])                    # -> DeferredBatch (uint8 stacked per source resolution)
    pin_memory thread                         # pins the uint8 frames
    batch['frames'].permute(0, 4, 1, 2, 3).float().to(device)   # H2D of the uint8 frames + ONE fused launch set

and only the last call touches the GPU.  Nothing in the Dataset, the DataLoader construction or the trainer changes;
the only swap is the factory (``shims.install(replace_video_aug=True)`` or an import of this package's
``create_video_transforms`` with ``deferred=True``).  What crosses PCIe is the uint8 source (44 MB per 16 x 720p clip)
instead of the float result (9.6 MB): 4.6x more bytes, which is why the NV12 source format exists.

Items whose decode failed arrive as the reference's plain all-zeros tensors (nexar_videos.py:479-489) and stay zeros.
"""
from __future__ import annotations

from typing import Any, Dict, List, Optional, Sequence, Tuple

import torch
from torch.utils.data import default_collate

_CANON_CLIP = ("C", "T", "H", "W")


def _check_perm(dims: Sequence[int], n: int) -> Tuple[int, ...]:
    if len(dims) == 1 and isinstance(dims[0], (tuple, list)):
        dims = tuple(dims[0])
    dims = tuple(int(d) % n for d in dims)
    if sorted(dims) != list(range(n)):
        raise ValueError(f"invalid permutation {dims} for a {n}-d deferred tensor")
    return dims


class _Lazy:
    """Shape bookkeeping shared by DeferredClip / DeferredBatch: a canonical shape plus the axis order requested so far."""

    _canon_shape: Tuple[int, ...]
    _order: Tuple[int, ...]

    @property
    def shape(self) -> torch.Size:
        return torch.Size(self._canon_shape[a] for a in self._order)

    def size(self, dim: Optional[int] = None):
        return self.shape if dim is None else self.shape[dim]

    def dim(self) -> int:
        return len(self._order)

    ndim = property(dim)

    def __len__(self) -> int:
        return self.shape[0]

    @property
    def dtype(self):
        return torch.float32

    @property
    def device(self):
        return torch.device("cpu")

    def numel(self) -> int:
        n = 1
        for s in self._canon_shape:
            n *= s
        return n


def _spec_transform(spec):
    from .video_aug import GpuVideoTransform
    return GpuVideoTransform.from_spec(spec)


class DeferredClip(_Lazy):
    """One clip whose pixel work has not run yet: the decoded frames ``[T,H,W,3]`` (uint8 or float32, host), the
    clip's random decisions, and the transform's picklable spec.  Behaves like the ``[3,T,cs,cs]`` float32 tensor the
    reference's transform returns as far as the Dataset code goes (``permute``, ``shape``, ``float``)."""

    def __init__(self, frames_thwc: torch.Tensor, params: Dict[str, Any], spec: Tuple, crop_size: int):
        self.frames = frames_thwc
        self.params = params
        self.spec = spec
        self._canon_shape = (3, int(frames_thwc.shape[0]), int(crop_size), int(crop_size))
        self._order = (0, 1, 2, 3)

    def permute(self, *dims) -> "DeferredClip":
        dims = _check_perm(dims, 4)
        out = DeferredClip.__new__(DeferredClip)
        out.__dict__.update(self.__dict__)
        out._order = tuple(self._order[d] for d in dims)
        return out

    def float(self) -> "DeferredClip":
        return self

    def contiguous(self) -> "DeferredClip":
        return self

    def materialize(self, device=None) -> torch.Tensor:
        """Run the transform for this clip alone (GPU) and return the tensor in the requested axis order, on the host
        unless ``device`` is given.  For code that needs the pixels inside the Dataset; the batch path never calls it."""
        tf = _spec_transform(self.spec)
        dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        out = tf.forward_batch(self.frames.unsqueeze(0).to(dev), params=[self.params], out_dtype=torch.float32)[0]
        out = out.permute(*self._order)
        return out if device is not None else out.cpu()

    def cpu(self) -> torch.Tensor:
        return self.materialize()

    def numpy(self):
        return self.materialize().numpy()

    def __repr__(self):
        return f"DeferredClip(shape={tuple(self.shape)}, source={tuple(self.frames.shape)} {self.frames.dtype})"


class DeferredBatch(_Lazy):
    """What ``default_collate`` makes of a list of DeferredClip (see :func:`install_collate_hooks`): the uint8 windows
    stacked per source resolution plus every clip's parameters.  ``.permute(...)``, ``.float()`` and ``.pin_memory()``
    are bookkeeping; ``.to(cuda_device)`` / ``.cuda()`` copies the uint8 frames and runs the fused transform, returning
    the real float32 tensor in the axis order asked for."""

    def __init__(self, groups: List[Dict[str, Any]], n: int, frames_per_clip: int, crop_size: int, spec: Tuple,
                 clip_order: Tuple[int, ...]):
        self.groups = groups            # [{'frames': [m,T,H,W,3], 'index': [...], 'params': [...]}]
        self.n = n
        self.spec = spec
        self._canon_shape = (n, 3, int(frames_per_clip), int(crop_size), int(crop_size))
        self._order = (0,) + tuple(1 + a for a in clip_order)

    def _clone(self) -> "DeferredBatch":
        out = DeferredBatch.__new__(DeferredBatch)
        out.__dict__.update(self.__dict__)
        return out

    def permute(self, *dims) -> "DeferredBatch":
        dims = _check_perm(dims, 5)
        out = self._clone()
        out._order = tuple(self._order[d] for d in dims)
        return out

    def float(self) -> "DeferredBatch":
        return self

    def contiguous(self) -> "DeferredBatch":
        return self

    def pin_memory(self, device=None) -> "DeferredBatch":
        out = self._clone()
        out.groups = [dict(g, frames=g["frames"].pin_memory()) for g in self.groups]
        return out

    def is_pinned(self) -> bool:
        return all(g["frames"].is_pinned() for g in self.groups)

    def _run(self, device: torch.device) -> torch.Tensor:
        tf = _spec_transform(self.spec)
        n, _, t, cs, _ = self._canon_shape
        out = None
        for g in self.groups:
            res = tf.forward_batch(g["frames"].to(device, non_blocking=True), params=g["params"], out_dtype=torch.float32)
            if len(self.groups) == 1 and len(g["index"]) == n:
                out = res
            else:
                if out is None:   # items that are in no group (failed decode) stay the reference's all-zeros clip
                    out = torch.zeros((n, 3, t, cs, cs), dtype=torch.float32, device=device)
                out[torch.tensor(g["index"], device=device)] = res
        if out is None:
            out = torch.zeros((n, 3, t, cs, cs), dtype=torch.float32, device=device)
        return out.permute(*self._order)

    def to(self, *args, **kwargs):
        device = kwargs.get("device")
        for a in args:
            if isinstance(a, (torch.device, str, int)) and not isinstance(a, bool):
                device = a
        if device is None:                       # .to(torch.float32) and friends: still deferred
            return self
        device = torch.device(device) if not isinstance(device, int) else torch.device("cuda", device)
        if device.type != "cuda":
            return self._run(torch.device("cuda", torch.cuda.current_device())).to(device)
        return self._run(device)

    def cuda(self, device=None, non_blocking: bool = False):
        return self.to(torch.device("cuda", torch.cuda.current_device() if device is None else
                                    (device if isinstance(device, int) else torch.device(device).index or 0)))

    def cpu(self) -> torch.Tensor:
        return self.to("cpu")

    def __repr__(self):
        return f"DeferredBatch(shape={tuple(self.shape)}, groups={[tuple(g['frames'].shape) for g in self.groups]})"


def collate_deferred(batch: Sequence[Any], *, collate_fn_map=None) -> DeferredBatch:
    """``default_collate`` hook: a list of DeferredClip (possibly mixed with the reference's all-zeros tensors of failed
    items) -> DeferredBatch.  Clips are stacked per source resolution; every clip of a batch must come from the same
    transform and have been permuted the same way (it is the same Dataset line for all of them)."""
    clips = [b for b in batch if isinstance(b, DeferredClip)]
    first = clips[0]
    by_shape: Dict[Any, Dict[str, Any]] = {}
    for pos, b in enumerate(batch):
        if not isinstance(b, DeferredClip):
            if isinstance(b, torch.Tensor) and not bool(b.any()):
                continue                          # failed item: stays zeros
            raise TypeError("a deferred batch may only mix DeferredClip with all-zeros fallback tensors")
        if b.spec != first.spec or b._order != first._order or b._canon_shape != first._canon_shape:
            raise ValueError("clips of one batch must come from the same deferred transform and Dataset code path")
        g = by_shape.setdefault((tuple(b.frames.shape), b.frames.dtype), {"frames": [], "index": [], "params": []})
        g["frames"].append(b.frames)
        g["index"].append(pos)
        g["params"].append(b.params)
    # default_collate stacks tensors the way it does for the reference's own items: inside a DataLoader worker straight
    # into shared memory, so the batch crosses to the main process as a file descriptor and the result queue's feeder
    # thread has no storage to move (an error there is only printed, and the batch is lost)
    groups = [{"frames": default_collate(g["frames"]), "index": g["index"], "params": g["params"]}
              for g in by_shape.values()]
    return DeferredBatch(groups, len(batch), first._canon_shape[1], first._canon_shape[2], first.spec, first._order)


_hooks_installed = False


def install_collate_hooks() -> None:
    """Teach ``torch.utils.data.default_collate`` about DeferredClip (idempotent; forked workers inherit it).  Plain
    tensors keep their collate function unless a DeferredClip sits in the same list (a failed item first in the batch)."""
    global _hooks_installed
    if _hooks_installed:
        return
    from torch.utils.data._utils import collate as C
    tensor_fn = C.default_collate_fn_map[torch.Tensor]

    def tensor_or_deferred(batch, *, collate_fn_map=None):
        if any(isinstance(b, DeferredClip) for b in batch):
            return collate_deferred(batch, collate_fn_map=collate_fn_map)
        return tensor_fn(batch, collate_fn_map=collate_fn_map)

    C.default_collate_fn_map[DeferredClip] = collate_deferred
    C.default_collate_fn_map[torch.Tensor] = tensor_or_deferred
    _hooks_installed = True
