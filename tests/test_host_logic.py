"""CPU-only tests of the host side: C-ABI library exports, geometry / tap tables against the oracle,
parameter sampling and packing, clip sampler, Dataset mirror plumbing.  No kernel is launched."""
import ctypes
import os
import random
import re

import numpy as np
import pytest
import torch

from oracle import clip_sampler_oracle as S
from oracle import np_oracle as O
from vision_collision_detection_b200 import _lib, create_video_transforms
from vision_collision_detection_b200 import params as PR
from vision_collision_detection_b200 import videos as V
from vision_collision_detection_b200.inference import sliding_window_starts

from golden_util import META, case_names, load_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "nexar_clip_transform.h")).read()
    names = set(re.findall(r"\b(nexar_[a-z0-9_]+)\s*\(", hdr))
    assert {"nexar_clip_transform", "nexar_plan_create", "nexar_workspace_bytes", "nexar_aa_taps"} <= names
    L = _lib.lib()
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for n in sorted(names):
        assert hasattr(raw, n), f"{n} declared in the header but not exported"
    assert L.nexar_abi_version() == _lib.NEXAR_ABI_VERSION
    assert L.nexar_sizeof_clip_params() == _lib.CLIP_PARAMS_DTYPE.itemsize
    assert L.nexar_sizeof_transform_args() == ctypes.sizeof(_lib.TransformArgs)


def test_resize_kernel_knob_refuses_unknown_variants():
    """0 auto, 1 general, 2 serialised.  4, the removed fused cluster kernel, is refused as unsupported.  Anything else,
    such as the removed variant 3, used to be accepted and silently run the default path."""
    L = _lib.lib()
    try:
        for v in (0, 1, 2):
            assert L.nexar_set_resize_kernel(v) == _lib.OK, v
        assert L.nexar_set_resize_kernel(4) == _lib.ERR_UNSUPPORTED
        for v in (3, 5, -1, 1 << 20):
            assert L.nexar_set_resize_kernel(v) == _lib.ERR_INVALID, v
            assert b"variant" in L.nexar_last_error()
    finally:
        assert L.nexar_set_resize_kernel(0) == _lib.OK


def test_geometry_matches_reference_table():
    for key, (nh, nw, ph, pw) in META["geometry"].items():
        hw, cs = key.split("->")
        h, w = map(int, hw.split("x"))
        g = _lib.letterbox_geometry(h, w, int(cs))
        assert (g.resize_h, g.resize_w, g.off_y, g.off_x) == (nh, nw, ph, pw), key
    g = _lib.resize_crop_geometry(96, 160, 56, 56)
    assert (g.resize_h, g.resize_w, g.off_y, g.off_x) == (56, 93, 0, -18)
    with pytest.raises(_lib.NexarError):
        _lib.letterbox_geometry(0, 10, 8)


@pytest.mark.parametrize("sizes", [(720, 125), (1280, 224), (1080, 126), (1920, 224), (720, 180), (40, 37),
                                   (60, 56), (97, 47), (131, 64), (5, 5), (3, 9)])
def test_tap_tables_bit_exact_with_oracle(sizes):
    start, count, wts = _lib.aa_taps(*sizes)
    xs, xc, xw = O.aa_taps(*sizes)
    assert (start == xs).all() and (count == xc).all()
    assert wts.shape == xw.shape and (wts == xw).all()
    assert np.abs(wts.sum(axis=1) - 1.0).max() < 1e-6


@pytest.mark.parametrize("name", case_names("custom_small") + case_names("ncwv_small") + case_names("allfx_small")
                         + case_names("poster_small") + ["train_portrait_flip"])
def test_param_sampler_is_bit_exact_with_the_reference(name):
    """R0: flip decision and every augmentation factor drawn from ``random`` equal the reference's."""
    c = load_case(name)
    tf = create_video_transforms(**c["kwargs"])
    random.seed(c["random_seed"])
    rec = tf.sample_params(1, 96, 160)[0]
    assert rec["flip"] == c["params"]["flip"]
    want = c["params"]["aug"]
    if want is None:
        assert rec["aug"] is None
    else:
        got = dict(rec["aug"])
        if "cutout_boxes" in got:
            got["cutout_boxes"] = [tuple(b) for b in got["cutout_boxes"]]
        assert got == want


def test_pack_clip_params_layout_and_errors():
    aug = PR.VideoAugmentation(brightness_range=(0.9, 1.1), rotation_range=(-5, 5), cutout_prob=1.0,
                               posterization_prob=1.0, blur_sigma=0.5, solarization_prob=1.0)
    random.seed(3)
    p = aug._sample_augmentation_parameters((3, 0, 56, 56))
    packed, flags = PR.pack_clip_params([{"flip": True, "aug": p, "crop": (1, -2)}], 56, aug)
    r = packed[0]
    assert flags == int(r["flags"]) and flags & _lib.FLIP and flags & _lib.AUG and flags & _lib.AFFINE
    assert flags & _lib.BLUR and r["blur_ksize"] == 5 and abs(r["blur_taps"][:5].sum() - 1) < 1e-6
    assert (r["crop_dy"], r["crop_dx"]) == (1, -2)
    assert r["brightness"] == np.float32(p["brightness"]) and r["contrast_q"] == np.float32(1.0 - p["contrast"])
    m = O.inverse_affine_matrix(p["rotation"], [p["translate_x"], p["translate_y"]], p["scale"], [p["shear"], 0.0])
    assert np.allclose(r["grid"], (np.asarray(m, np.float32) / np.float32(28.0)), rtol=0, atol=0)
    assert r["n_cutout"] == len(p["cutout_boxes"]) and tuple(r["cutout"][0]) == tuple(p["cutout_boxes"][0])
    bad = dict(p, hue=0.7)
    with pytest.raises(ValueError):         # torchvision raises for |hue| > 0.5
        PR.pack_clip_params([{"flip": False, "aug": bad}], 56, aug)
    bad = dict(p, brightness=-0.1)
    with pytest.raises(ValueError):
        PR.pack_clip_params([{"flip": False, "aug": bad}], 56, aug)
    # an un-augmented clip has no aug flags
    packed, flags = PR.pack_clip_params([{"flip": False, "aug": None}], 56, None)
    assert flags == 0 and packed[0]["flags"] == 0


def test_factory_signature_matches_reference_kwargs():
    """create_video_transforms accepts the reference's full kwarg surface (nexar_video_aug.py:636-696)."""
    ref_kwargs = ["mode", "video_key", "num_samples", "convert_to_float", "crop_size", "normalize", "video_mean",
                  "video_std", "min_size", "max_size", "horizontal_flip_prob", "enable_custom_augmentation",
                  "aug_probability", "brightness_range", "contrast_range", "saturation_range", "hue_range",
                  "rotation_range", "scale_range", "shear_range", "translate_range", "perspective_distortion",
                  "noise_level", "blur_sigma", "jpeg_quality", "grayscale_prob", "cutout_prob", "cutout_count",
                  "cutout_size_range", "color_inversion_prob", "solarization_prob", "posterization_prob",
                  "posterization_bits_range", "solarization_threshold", "debug"]
    import inspect
    sig = list(inspect.signature(create_video_transforms).parameters)
    assert sig[:len(ref_kwargs)] == ref_kwargs
    tf = create_video_transforms(mode="train", enable_custom_augmentation=True, aug_probability=0.1)
    assert tf.video_aug.aug_probability == 1.0      # dropped by the reference factory too (:762-788)
    names = [getattr(t, "__name__", type(t).__name__) for t in tf.transforms]
    assert names == ["letterbox_resize", "horizontal_flip", "VideoAugmentation", "normalize_tensor"]
    assert [getattr(t, "__name__", "") for t in create_video_transforms(mode="val").transforms] == \
        ["letterbox_resize", "normalize_tensor"]


def test_clip_sampler_matches_oracle():
    for n in [1, 10, 49, 50, 51, 120, 300, 1200]:
        for st in ["random", "center", "metadata_time", "metadata_center", "uniform"]:
            for ts, fps in [(None, 0.0), (3.7, 30.0), (0.1, 29.97), (38.0, 30.0)]:
                random.seed(n * 7 + 3)
                a = V.select_start_frame(n, 50, st, random, ts, fps)
                random.seed(n * 7 + 3)
                b = S.start_frame(n, 50, st, random, ts, fps)
                assert a == b
                assert V.window_indices(n, 50, a) == S.window_indices(n, 50, b)
        assert V.uniform_indices(n, 16) == S.uniform_indices(n, 16)
        assert V.model_frame_subsample(n) == S.model_subsample(n)
    for s in (1, 8, 16):
        assert sliding_window_starts(1200, 16, s) == S.sliding_window_starts(1200, 16, s)
    assert sliding_window_starts(10, 16, 8) == [0]


class _FakeReader:
    def __init__(self, n, h=48, w=64):
        self.frames = (np.arange(n * h * w * 3, dtype=np.int64) % 251).astype(np.uint8).reshape(n, h, w, 3)

    def __len__(self):
        return len(self.frames)

    def get_batch(self, idx):
        return self.frames[list(idx)]


def test_deferred_dataset_and_collate_without_cuda():
    rows = [{"id": "a", "video_type": "Normal", "path": "a.mp4"}, {"id": "b", "video_type": "Collision", "path": "b.mp4"},
            {"id": "bad", "video_type": "Normal", "path": "missing.mp4"}]

    def decoder(path):
        if "missing" in path:
            raise IOError("no such video")
        return _FakeReader(30 if path.startswith("a") else 80)

    tf = create_video_transforms(mode="train", crop_size=32)
    ds = V.GpuDashcamDataset(rows, fps=10, duration=5, transform=tf, sample_strategy="center", decoder=decoder, defer=True)
    assert len(ds) == 3
    random.seed(0)
    a, b, bad = ds[0], ds[1], ds[2]
    assert tuple(a["frames_u8"].shape) == (50, 48, 64, 3) and a["frames_u8"].dtype == torch.uint8
    assert torch.equal(a["frames_u8"][29], a["frames_u8"][49])           # short video: last frame repeated
    assert torch.equal(b["frames_u8"][0], torch.from_numpy(_FakeReader(80).frames[15]))   # centre window start 40-25
    assert bad["frames_u8"] is None                                      # any failure is swallowed
    assert isinstance(a["params"]["flip"], bool)
    batch = V.deferred_collate([a, b, bad])
    assert len(batch["groups"]) == 1 and batch["valid"] == [True, True, False]
    g = batch["groups"][0]
    assert tuple(g["frames_u8"].shape) == (2, 50, 48, 64, 3) and g["index"] == [0, 1] and len(g["params"]) == 2
    assert batch["target"] == ["Normal", "Collision", "Normal"]
    # a batch that mixes source resolutions is stacked per resolution (the reference transforms before it collates)
    other = dict(a, frames_u8=torch.zeros(50, 36, 64, 3, dtype=torch.uint8))
    mixed = V.deferred_collate([a, other, b, bad])
    assert [tuple(g["frames_u8"].shape[2:4]) for g in mixed["groups"]] == [(48, 64), (36, 64)]
    assert [g["index"] for g in mixed["groups"]] == [[0, 2], [1]] and mixed["valid"] == [True, True, True, False]
    assert list(V.shard_clips(10, 1, 4)) == [3, 4, 5] and list(V.shard_clips(10, 3, 4)) == [9]


def test_sensor_sync_is_bit_exact_with_the_reference_pandas_expression():
    """SURVEY F4 (nexar_videos.py:318-341): numpy.interp on the valid samples == reindex/union/interpolate('index')."""
    from oracle.sensor_oracle import sync_sensor_pandas
    from vision_collision_detection_b200.sensors import sync_sensor_to_frames
    rng = np.random.default_rng(0)
    checked = 0
    for trial in range(24):
        n = int(rng.integers(2, 300))
        fps = float(rng.choice([30.0, 29.97, 25.0, 10.0, 59.94]))
        fc = int(rng.integers(1, 900))
        t = 1.7e9 + np.cumsum(rng.uniform(0.005, 0.02, n))
        a = rng.normal(size=(n, 4))
        if trial % 5 == 0:
            a[rng.integers(0, n, 3), rng.integers(0, 4, 3)] = np.nan      # holes are interpolated over
        if trial % 7 == 0:
            a[0, 1] = np.nan                                              # a leading hole stays NaN
        if trial % 3 == 0:                                                # samples exactly on frame times
            k = min(n - 1, 5)
            t[1:1 + k] = t[0] + np.arange(1, 1 + k) / fps
            t = np.sort(t)
            if (np.diff(t) == 0).any():
                continue
        if trial % 4 == 0:                                                # unsorted file order
            perm = rng.permutation(n)
            perm = np.concatenate([[0], perm[perm != 0]])                 # the first row defines time zero
            t, a = t[perm], a[perm]
        got = sync_sensor_to_frames(t, a, fc, fps)
        want = sync_sensor_pandas(t, a, fc, fps)
        assert got.dtype == np.float64 and np.array_equal(got, want, equal_nan=True), trial
        checked += 1
    assert checked >= 16
    with pytest.raises(ValueError):                                       # pandas: cannot reindex on duplicate labels
        sync_sensor_to_frames(np.array([5.0, 5.5, 5.5]), np.zeros((3, 4)), 10, 30.0)


def test_dataset_sensor_window_follows_the_reference(tmp_path):
    """nexar_videos.py:453-477: rows [start, end) of the synced table, last row repeated, zeros without a CSV."""
    from oracle.sensor_oracle import sync_sensor_pandas
    from vision_collision_detection_b200 import sensors as SN
    rng = np.random.default_rng(3)
    n_frames, vfps = 80, 20.0
    t = 100.0 + np.cumsum(rng.uniform(0.004, 0.012, 700))
    a = rng.normal(size=(700, 4))
    for vid in ("with_csv", "no_csv", "short"):
        os.makedirs(tmp_path / vid / "signals", exist_ok=True)
        (tmp_path / vid / f"{vid}.mp4").write_bytes(b"")
    with open(tmp_path / "with_csv" / "signals" / SN.SENSOR_FILE, "w") as f:
        f.write(",time_sec,accel_x_G,accel_y_G,accel_z_G,accel_total_G\n")
        for i in range(len(t)):
            f.write(",".join([str(i)] + [repr(float(v)) for v in (t[i], *a[i])]) + "\n")
    with open(tmp_path / "short" / "signals" / SN.SENSOR_FILE, "w") as f:
        f.write(",time_sec,accel_x_G,accel_y_G,accel_z_G,accel_total_G\n0,1.0,0.1,0.2,0.3,0.4\n1,1.5,0.2,0.3,0.4,0.5\n")

    class Reader(_FakeReader):
        def get_avg_fps(self):
            return vfps

    rows = [{"id": v, "video_type": "Normal"} for v in ("with_csv", "no_csv", "short")]
    ds = V.GpuDashcamDataset(rows, [str(tmp_path)], fps=10, duration=5, transform=None, sample_strategy="center",
                             decoder=lambda p: Reader(30 if "short" in p else n_frames), defer=True)
    assert ds.sensor_paths[0].endswith(SN.SENSOR_FILE) and ds.sensor_paths[1] is None
    full = sync_sensor_pandas(t, a, n_frames, vfps)
    start = S.start_frame(n_frames, 50, "center")
    want = full[start:start + 50].astype(np.float32)
    got = ds[0]["sensor"]
    assert got.dtype == torch.float32 and tuple(got.shape) == (50, 4)
    assert np.array_equal(got.numpy(), want)
    assert float(ds[1]["sensor"].abs().max()) == 0.0                      # no CSV beside the video
    s = ds[2]["sensor"].numpy()                                           # 30-frame video, window 0..30: last row repeated
    tab = sync_sensor_pandas(np.array([1.0, 1.5]), np.array([[0.1, 0.2, 0.3, 0.4], [0.2, 0.3, 0.4, 0.5]]), 30, vfps)
    assert np.array_equal(s[:30], tab.astype(np.float32)) and np.array_equal(s[30:], np.repeat(s[29:30], 20, axis=0))


def test_video_dataset_mirror_follows_complete_with_validation():
    """nexar_complete_with_validation.py:57-234: explicit lists, 'metadata_center' windows, no sensor stream."""
    paths, labels, ids = ["a.mp4", "b.mp4", "c.mp4", "missing.mp4"], [0, 2, 1, 0], ["a", "b", "c", "m"]
    meta = [{"id": "a", "t_event": 3.0}, {"id": "b", "t_event": float("nan")}, {"id": "c", "t_event": 100.0}]

    class Reader(_FakeReader):
        def get_avg_fps(self):
            return 20.0

    def decoder(path):
        if "missing" in path:
            raise IOError("no such video")
        return Reader(120)

    with pytest.raises(AssertionError):
        V.GpuVideoDataset(paths, labels[:2])
    with pytest.raises(AssertionError):
        V.GpuVideoDataset(paths, labels, sample_strategy="metadata_center")        # needs metadata_df + column
    ds = V.GpuVideoDataset(paths, labels, ids, fps=10, duration=5, transform=None, sample_strategy="metadata_center",
                           center_time_column="t_event", metadata_df=meta, decoder=decoder, defer=True)
    ref = Reader(120).frames
    a = ds[0]                                                    # centre frame int(3.0 * 20) = 60 -> start 35
    assert sorted(a) == ["frames_u8", "id", "need", "params", "target"] and a["target"] == 0 and a["id"] == "a"
    assert torch.equal(a["frames_u8"][0], torch.from_numpy(ref[S.start_frame(120, 50, "metadata_center", random, 3.0, 20.0)]))
    assert S.start_frame(120, 50, "metadata_center", random, 3.0, 20.0) == 35
    random.seed(11)
    want = S.start_frame(120, 50, "metadata_center", random, None, 20.0)          # NaN centre time: random window
    random.seed(11)
    assert torch.equal(ds[1]["frames_u8"][0], torch.from_numpy(ref[want]))
    assert torch.equal(ds[2]["frames_u8"][0], torch.from_numpy(ref[70]))           # past the end: last full window
    assert ds[3]["frames_u8"] is None
    batch = V.deferred_collate([ds[0], ds[2], ds[3]])
    assert "sensor" not in batch and batch["valid"] == [True, True, False] and batch["need"] == 50
    plain = V.GpuVideoDataset(paths, labels, ids, sample_strategy="center", decoder=decoder)
    item = plain[0]
    assert sorted(item) == ["frames", "id", "target"] and tuple(item["frames"].shape) == (50, 48, 64, 3)
    assert float(item["frames"].max()) <= 1.0                     # no transform: frames / 255 (ncwv:178)
    assert tuple(plain[3]["frames"].shape) == (50, 720, 1280, 3)  # failure without a transform (ncwv:189-190)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "vision_collision_detection_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


def test_reference_import_shims():
    """nexar_inference.py:203-204 imports ``nexar_data.NvidiaDashcamDataset`` (a module the reference does not ship)
    and ``nexar_video_aug.create_video_transforms``; the shims make both resolve to the GPU path, only on request."""
    import importlib
    import sys

    from vision_collision_detection_b200 import create_video_transforms, shims
    from vision_collision_detection_b200.videos import GpuDashcamDataset
    saved = {k: sys.modules.get(k) for k in ("nexar_data", "nexar_video_aug")}
    try:
        for k in saved:
            sys.modules.pop(k, None)
        mods = shims.install()
        assert set(mods) == {"nexar_data"} and "nexar_video_aug" not in sys.modules
        assert importlib.import_module("nexar_data").NvidiaDashcamDataset is GpuDashcamDataset
        shims.install(replace_video_aug=True)
        from nexar_data import NvidiaDashcamDataset          # the reference's own import lines
        from nexar_video_aug import create_video_transforms as ctf
        assert NvidiaDashcamDataset is GpuDashcamDataset and ctf is create_video_transforms
        ds = NvidiaDashcamDataset(metadata_df=[{"id": "video_0", "video_type": "Normal"}], base_dirs=["/nonexistent"], fps=10,
                                  duration=5, is_train=False, skip_missing=False, transform=None, sample_strategy="center")
        assert len(ds) == 1                                   # the constructor call of nexar_inference.py:212-221
        shims.uninstall()
        assert "nexar_data" not in sys.modules and "nexar_video_aug" not in sys.modules
    finally:
        for k, v in saved.items():
            if v is not None:
                sys.modules[k] = v
            else:
                sys.modules.pop(k, None)


def test_deferred_transform_bookkeeping_without_cuda():
    """The zero-line drop-in (deferred.py): inside the Dataset the transform returns a DeferredClip that follows the
    reference's own lines (permute -> default_collate -> pin -> permute / float), nothing touches the GPU before .to()."""
    import pickle
    import random

    from torch.utils.data import default_collate

    from vision_collision_detection_b200 import GpuVideoTransform, create_video_transforms
    from vision_collision_detection_b200.deferred import DeferredBatch, DeferredClip
    tf = create_video_transforms(mode="train", enable_custom_augmentation=True, rotation_range=(-5, 5), deferred=True)
    assert GpuVideoTransform.from_spec(tf.spec()).spec() == tf.spec() and hash(tf.spec()) is not None
    plain = create_video_transforms(mode="train", enable_custom_augmentation=True, rotation_range=(-5, 5))
    random.seed(3)
    want_params = plain.sample_params(3, 36, 64)                 # same generator, same order as three deferred calls
    random.seed(3)
    items = []
    for i in range(3):
        frames = torch.randint(0, 255, (4, 36, 64, 3), dtype=torch.uint8)
        clip = tf(frames.permute(3, 0, 1, 2))                    # nexar_videos.py:441-445
        assert isinstance(clip, DeferredClip) and tuple(clip.shape) == (3, 4, 224, 224) and clip.dtype == torch.float32
        assert clip.params == want_params[i] and torch.equal(clip.frames, frames)
        clip = clip.permute(1, 2, 3, 0)                          # :451
        assert tuple(clip.shape) == (4, 224, 224, 3) and len(clip) == 4
        items.append({"frames": clip, "sensor": torch.zeros(4, 4), "target": "Normal", "id": f"v{i}"})
    items.insert(0, {"frames": torch.zeros(4, 224, 224, 3), "sensor": torch.zeros(4, 4), "target": "Normal", "id": "bad"})
    batch = default_collate(items)                               # the failed item comes first: the tensor hook delegates
    fb = batch["frames"]
    assert isinstance(fb, DeferredBatch) and tuple(fb.shape) == (4, 4, 224, 224, 3) and batch["id"] == ["bad", "v0", "v1", "v2"]
    assert tuple(batch["sensor"].shape) == (4, 4, 4)             # ordinary tensors still collate as before
    assert len(fb.groups) == 1 and fb.groups[0]["index"] == [1, 2, 3] and tuple(fb.groups[0]["frames"].shape) == (3, 4, 36, 64, 3)
    x = fb.permute(0, 4, 1, 2, 3).float()                        # the consumer line, up to .to(device)
    assert tuple(x.shape) == (4, 3, 4, 224, 224) and x._order == (0, 1, 2, 3, 4)
    again = pickle.loads(pickle.dumps(fb))                       # worker -> main process
    assert tuple(again.shape) == tuple(fb.shape) and again.groups[0]["params"] == fb.groups[0]["params"]
    with pytest.raises(ValueError):
        fb.permute(0, 1, 2, 3, 3)
    with pytest.raises(TypeError):
        default_collate([items[1]["frames"], torch.ones(4, 224, 224, 3)])      # only all-zeros fallbacks may be mixed in
