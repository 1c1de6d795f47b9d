"""YUV 4:2:0 decoder surfaces with 16-bit samples: P010 / P016 (semi-planar, MSB-aligned) and yuv420p10le (planar,
LSB-aligned 10-bit), every matrix and range, padded surfaces.  The numpy oracle and its two defining properties (the
8-bit widening identity and one rounding from 10-bit precision), the argument checks, and - on the GPU - that every
variant is the RGB path bit for bit once the surfaces are converted, through forward_batch, HostClipPipeline, the
deferred training loader and the inference windows."""
import ctypes
import random

import numpy as np
import pytest
import torch

from oracle import yuv420_oracle as Y
from yuv16_oracle import SAMPLE_SHIFT, yuv420_16_to_rgb
from vision_collision_detection_b200 import _lib
from vision_collision_detection_b200.synth import make_clip_np, rgb_to_yuv420, rgb_to_yuv420_16

MATRICES = ("bt601", "bt709")
RANGES = ("limited", "full")
PAIRS = [(m, r) for m in MATRICES for r in RANGES]
LAYOUT_8 = {"p010": "nv12", "i010": "i420"}          # the 8-bit format with the same layout
SHIFT = SAMPLE_SHIFT


def widen(surf8, fmt):
    """8-bit surfaces -> the 16-bit surfaces whose words are the codes << 8 (p010) / the 10-bit codes 4 x (i010)."""
    return surf8.astype(np.uint16) << (8 if fmt == "p010" else 2)


def conv16(surf, fmt, m, r, frame_size=None):
    return yuv420_16_to_rgb(surf, LAYOUT_8[fmt], m, r, frame_size, SHIFT[fmt])


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("m,r", PAIRS)
@pytest.mark.parametrize("fmt", ["p010", "i010"])
def test_oracle_widening_identity(fmt, m, r):
    """Random bytes (every clipping branch included): the words x << 8 convert exactly as the 8-bit codes x."""
    surf8 = np.random.RandomState(7).randint(0, 256, (3, 96, 128)).astype(np.uint8)
    want = Y.yuv420_to_rgb(surf8, LAYOUT_8[fmt], m, r)
    assert np.array_equal(conv16(widen(surf8, fmt), fmt, m, r), want)
    assert 0 in want and 255 in want


@pytest.mark.parametrize("m,r", PAIRS)
@pytest.mark.parametrize("fmt", ["p010", "i010"])
def test_oracle_within_one_level_of_exact_10bit_conversion(fmt, m, r):
    """Random 10-bit codes, read as 4 x an 8-bit code: the integer formula stays within one level of float64."""
    rs = np.random.RandomState(11)
    h, w = 256, 512
    codes = rs.randint(0, 1024, (h * 3 // 2, w)).astype(np.uint16)
    surf = codes << 6 if fmt == "p010" else codes | (rs.randint(0, 64, codes.shape).astype(np.uint16) << 10)  # i010: high bits ignored
    got = conv16(surf, fmt, m, r).astype(np.float64)
    yo, ys, rv, gu, gv, bu = Y.yuv_float_coefficients(m, r)
    y = codes[:h].astype(np.float64) / 4
    if fmt == "p010":
        u, v = codes[h:, 0::2] / 4, codes[h:, 1::2] / 4
    else:
        planes = codes[h:].reshape(h, w // 2) / 4
        u, v = planes[: h // 2], planes[h // 2:]
    u = np.repeat(np.repeat(u, 2, 0), 2, 1) - 128
    v = np.repeat(np.repeat(v, 2, 0), 2, 1) - 128
    c = ys * (y - yo)
    exact = np.stack([c + rv * v, c - gu * u - gv * v, c + bu * u], -1).clip(0, 255)
    assert np.abs(got - exact).max() <= 1.0


def test_oracle_layouts_padding_and_round_trip():
    clip = make_clip_np(3, 48, 64, 5, "dashcam")
    for m, r in PAIRS:
        p010 = rgb_to_yuv420_16(clip, "p010", m, r)
        i010 = rgb_to_yuv420_16(clip, "i010", m, r)
        assert p010.dtype == np.uint16 and p010.shape == (3, 72, 64) and int(i010.max()) < 1024
        want = conv16(p010, "p010", m, r)
        assert np.array_equal(conv16(i010, "i010", m, r), want)
        for fmt in ("p010", "i010"):
            padded = rgb_to_yuv420_16(clip, fmt, m, r, luma_rows=56, pitch=80)
            assert padded.shape == (3, 84, 80) and padded[:, 48:56].min() == 0xFFFF and padded[:, :48, 64:].min() == 0xFFFF
            assert np.array_equal(conv16(padded, fmt, m, r, frame_size=(48, 64)), want)
    with pytest.raises(ValueError):
        rgb_to_yuv420_16(clip, "nv12")
    with pytest.raises(ValueError):
        rgb_to_yuv420_16(clip, "i010", pitch=65)


@pytest.mark.parametrize("m,r", PAIRS)
@pytest.mark.parametrize("fmt", ["p010", "i010"])
def test_float_encode_integer_decode_round_trip(fmt, m, r):
    """Uniform 2 x 2 blocks survive the 10-bit encode and the integer decode within two levels, and closer on average
    than through 8-bit surfaces (the encode rounds at four times the precision)."""
    g = np.arange(0, 256, 5)
    rgb = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 1, 1, 3)
    rgb = np.broadcast_to(rgb, (rgb.shape[0], 2, 2, 3)).astype(np.uint8)
    err = np.abs(conv16(rgb_to_yuv420_16(rgb, fmt, m, r), fmt, m, r).astype(int) - rgb)
    err8 = np.abs(Y.yuv420_to_rgb(rgb_to_yuv420(rgb, LAYOUT_8[fmt], m, r), LAYOUT_8[fmt], m, r).astype(int) - rgb)
    assert err.max() <= 2 and err.mean() < err8.mean()


@pytest.mark.parametrize("fmt", ["p010", "i010"])
def test_blank_16bit_frames_convert_to_zeros(fmt):
    from vision_collision_detection_b200.videos import _blank_frame
    for m, r in PAIRS:
        f = _blank_frame((72, 64), {"pixel_format": fmt, "color_matrix": m, "color_range": r})
        assert f.dtype == np.uint16
        assert int(f[0, 0]) == ((16 << 8 if fmt == "p010" else 64) if r == "limited" else 0)
        assert int(f[-1, -1]) == (32768 if fmt == "p010" else 512)
        assert conv16(f, fmt, m, r).max() == 0


def test_forward_batch_argument_checks():
    from vision_collision_detection_b200 import create_video_transforms
    tf = create_video_transforms(mode="val", crop_size=32)
    s16 = torch.zeros((1, 2, 72, 64), dtype=torch.uint16)          # 48 luma rows, pitch 64 (host: rejected before use)
    s8 = torch.zeros((1, 2, 72, 64), dtype=torch.uint8)
    for fmt in ("p010", "i010"):
        with pytest.raises(ValueError):
            tf.forward_batch(s8, pixel_format=fmt)                                              # uint8 surfaces
        with pytest.raises(ValueError):
            tf.forward_batch(torch.zeros((1, 2, 72, 63), dtype=torch.uint16), pixel_format=fmt)  # odd pitch
        with pytest.raises(ValueError):
            tf.forward_batch(torch.zeros((1, 2, 71, 64), dtype=torch.uint16), pixel_format=fmt)  # not L * 3 / 2 rows
        for size in ((50, 64), (48, 66), (47, 64), (48, 63)):
            with pytest.raises(ValueError):
                tf.forward_batch(s16, pixel_format=fmt, frame_size=size)
        with pytest.raises(ValueError):
            tf.forward_batch(s16, pixel_format=fmt, color_matrix="bt2020")
    for fmt in ("nv12", "i420"):
        with pytest.raises(ValueError):
            tf.forward_batch(s16, pixel_format=fmt)                                             # uint16 for 8-bit
    with pytest.raises(ValueError):
        tf.forward_batch(torch.zeros((1, 2, 48, 64, 3), dtype=torch.uint16))                     # uint16 RGB


def test_dataset_argument_checks():
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.videos import GpuDashcamDataset, GpuVideoDataset
    tf = create_video_transforms(mode="val", crop_size=32)
    with pytest.raises(ValueError):
        GpuDashcamDataset([], transform=tf, pixel_format="p010")                        # defer=False
    with pytest.raises(ValueError):
        GpuVideoDataset([], [], transform=tf, sample_strategy="center", pixel_format="i010")

    class Reader:
        def __init__(self, dtype):
            self.frames = np.zeros((8, 72, 64), dtype)

        def __len__(self):
            return len(self.frames)

        def get_batch(self, idx):
            return self.frames[list(idx)]

    rows = [{"id": "v0", "video_type": "Normal", "path": "x"}]
    for fmt, dtype in (("p010", np.uint8), ("i010", np.uint8), ("i010", np.int32)):
        ds = GpuDashcamDataset(rows, fps=2, duration=2, transform=tf, decoder=lambda p, d=dtype: Reader(d), defer=True,
                               pixel_format=fmt)
        with pytest.raises(ValueError):
            ds[0]
    ds = GpuDashcamDataset(rows, fps=2, duration=2, transform=tf, decoder=lambda p: Reader(np.uint16), defer=True,
                           pixel_format="i010", color_matrix="bt709")
    item = ds[0]
    assert item["frames_u8"].dtype == torch.uint16 and tuple(item["frames_u8"].shape) == (4, 72, 64)
    assert item["format"] == {"pixel_format": "i010", "color_matrix": "bt709", "color_range": "limited"}


def test_plan_checks_of_the_c_abi():
    """nexar_plan_create_yuv16 validates the shift and the descriptor before it touches the device; the 8-bit entry
    point keeps refusing layout 2."""
    L = _lib.yuv16_lib()
    assert ctypes.sizeof(_lib.YuvFormat) == 20
    g = _lib.Geometry(48, 64, 32, 24, 32, 4, 0)

    def create16(shift=0, struct_size=ctypes.sizeof(_lib.YuvFormat), layout=0, matrix=0, range_=0, luma_rows=0, geom=g):
        f = _lib.YuvFormat(struct_size, layout, matrix, range_, luma_rows)
        h = ctypes.c_void_p()
        return L.nexar_plan_create_yuv16(ctypes.byref(geom), ctypes.byref(f), shift, ctypes.byref(h))

    for shift in (1, 5, 8, -1, 16):
        assert create16(shift=shift) == _lib.ERR_INVALID, shift
    for shift in (0, 4, 6):
        for bad in (dict(struct_size=16), dict(layout=2), dict(matrix=2), dict(range_=-1), dict(luma_rows=46),
                    dict(luma_rows=51), dict(geom=_lib.Geometry(48, 63, 32, 24, 32, 4, 0))):
            assert create16(shift=shift, **bad) == _lib.ERR_INVALID, (shift, bad)
    f = _lib.YuvFormat(ctypes.sizeof(_lib.YuvFormat), 2, 0, 0, 0)
    assert L.nexar_plan_create_yuv(ctypes.byref(g), ctypes.byref(f), ctypes.byref(ctypes.c_void_p())) == _lib.ERR_INVALID


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
KW_CUSTOM = dict(mode="train", enable_custom_augmentation=True, brightness_range=(0.9, 1.1), contrast_range=(0.9, 1.1),
                 saturation_range=(0.9, 1.1), rotation_range=(-5, 5))


def _transform(kw, cs, **extra):
    from vision_collision_detection_b200 import create_video_transforms
    return create_video_transforms(**kw, crop_size=cs, **extra)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("h,w,cs", [(720, 1280, 224), (90, 150, 64)], ids=["720p_vec", "90x150_any"])
@pytest.mark.parametrize("kw", [dict(mode="val"), KW_CUSTOM], ids=["val", "custom"])
@pytest.mark.parametrize("m,r", PAIRS)
@pytest.mark.parametrize("fmt", ["p010", "i010"])
def test_every_16bit_format_equals_rgb_path_on_converted_frames(h, w, cs, kw, m, r, fmt):
    """720p takes the vector conversion kernel and the fast resize, 90 x 150 the byte-wise conversion and the general
    resize.  The small size uses arbitrary words (clipping branches, and bits an LSB-aligned read must ignore)."""
    if w % 16:
        surf = np.random.RandomState(3).randint(0, 65536, (2, 3, h * 3 // 2, w)).astype(np.uint16)
    else:
        surf = rgb_to_yuv420_16(np.stack([make_clip_np(3, h, w, 11 + i, "dashcam") for i in range(2)]), fmt, m, r)
    rgb = conv16(surf, fmt, m, r)
    tf = _transform(kw, cs)
    random.seed(5)
    params = tf.sample_params(2, h, w)
    got = tf.forward_batch(_dev(surf), params=params, pixel_format=fmt, color_matrix=m, color_range=r)
    n16 = _lib.lib().nexar_last_launch_count()
    want = tf.forward_batch(_dev(rgb), params=params)
    assert n16 == _lib.lib().nexar_last_launch_count() + 1
    assert got.shape == (2, 3, 3, cs, cs) and torch.equal(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["p010", "i010"])
def test_widening_identity_on_the_device(fmt):
    """P010 made from NV12 and I010 made from I420 give the 8-bit call's output bit for bit, on both kernels."""
    tf = _transform(KW_CUSTOM, 112)
    layout = LAYOUT_8[fmt]
    for m, r in PAIRS:
        for h, w, surf8 in ((180, 320, rgb_to_yuv420(np.stack([make_clip_np(3, 180, 320, 40 + i, "dashcam") for i in range(2)]),
                                                     layout, m, r)),
                            (90, 150, np.random.RandomState(4).randint(0, 256, (2, 3, 135, 150)).astype(np.uint8))):
            random.seed(8)
            params = tf.sample_params(2, h, w)
            kw = dict(params=params, color_matrix=m, color_range=r)
            want = tf.forward_batch(_dev(surf8), pixel_format=layout, **kw)
            got = tf.forward_batch(_dev(widen(surf8, fmt)), pixel_format=fmt, **kw)
            assert torch.equal(got, want), (m, r, h)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,m,r", [("p010", "bt709", "limited"), ("i010", "bt709", "full"), ("p010", "bt601", "full")])
def test_padded_1080p_16bit_surfaces(fmt, m, r):
    """1080p in the 1088-row, 2048-sample surfaces of a hardware decoder (every padding sample 0xFFFF), and pitches that
    force the byte-wise kernel: every one equals the packed surface and the RGB path."""
    clip = make_clip_np(2, 1080, 1920, 21, "dashcam")
    packed = _dev(rgb_to_yuv420_16(clip, fmt, m, r)).unsqueeze(0)
    tf = _transform(KW_CUSTOM, 224)
    random.seed(2)
    params = tf.sample_params(1, 1080, 1920)
    kw = dict(params=params, pixel_format=fmt, color_matrix=m, color_range=r)
    want = tf.forward_batch(packed, **kw)
    # 2048: vector kernel; 1924 (3848 bytes): byte-wise for both layouts; 1928 (3856 bytes): byte-wise for the planar one
    for pitch in (2048, 1924, 1928):
        padded_np = rgb_to_yuv420_16(clip, fmt, m, r, luma_rows=1088, pitch=pitch)
        assert padded_np.shape == (2, 1632, pitch) and padded_np[:, 1080:1088].min() == 0xFFFF
        got = tf.forward_batch(_dev(padded_np).unsqueeze(0), frame_size=(1080, 1920), **kw)
        assert torch.equal(got, want), pitch
    rgb = tf.forward_batch(_dev(conv16(padded_np, fmt, m, r, (1080, 1920))).unsqueeze(0), params=params)
    assert torch.equal(want, rgb)


@pytest.mark.gpu
def test_unaligned_base_takes_the_byte_wise_kernel():
    """A surface view that starts 2 bytes into its storage cannot take the 16-byte loads; the result is the same."""
    clip = make_clip_np(2, 64, 128, 31, "dashcam")
    p010 = rgb_to_yuv420_16(clip, "p010", "bt709", "limited")
    flat = torch.zeros(p010.size + 1, dtype=torch.uint16, device="cuda")
    flat[1:] = _dev(p010).reshape(-1)
    shifted = flat[1:].view(1, 2, 96, 128)
    assert shifted.data_ptr() % 16 == 2
    tf = _transform(dict(mode="val"), 64)
    kw = dict(pixel_format="p010", color_matrix="bt709")
    assert torch.equal(tf.forward_batch(shifted, **kw), tf.forward_batch(_dev(p010).unsqueeze(0), **kw))


@pytest.mark.gpu
def test_frame_index_and_clip_max_rule():
    """A full-range clip whose luma converts to 0/1 with neutral chroma is NOT divided by 255, as the RGB clip of those
    values; frame_index gathers from the 16-bit frame pool."""
    h, w, cs = 96, 160, 64
    i010 = rgb_to_yuv420_16(np.stack([make_clip_np(4, h, w, 70 + i, "dashcam") for i in range(2)]), "i010", "bt709", "full")
    i010[1, :, :h] = np.random.RandomState(1).randint(0, 6, (4, h, w))        # 10-bit codes 0..5: RGB 0 or 1
    i010[1, :, h:] = 512
    rgb = conv16(i010, "i010", "bt709", "full")
    assert rgb[1].max() == 1 and rgb[1].min() == 0
    tf = _transform(dict(mode="val"), cs)
    index = torch.tensor([[3, 1, 1], [4, 7, 5]])
    got = tf.forward_batch(_dev(i010), frame_index=index, pixel_format="i010", color_matrix="bt709", color_range="full")
    want = tf.forward_batch(_dev(rgb), frame_index=index)
    assert torch.equal(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["p010", "i010"])
def test_host_pipeline_16bit(fmt):
    from vision_collision_detection_b200.host_pipeline import HostClipPipeline
    h, w, cs = 180, 320, 112
    tf = _transform(KW_CUSTOM, cs, out_dtype=torch.bfloat16)
    surf = torch.from_numpy(rgb_to_yuv420_16(np.stack([make_clip_np(4, h, w, 90 + i, "dashcam") for i in range(5)]),
                                             fmt, "bt709", "limited"))
    pipe = HostClipPipeline(tf, n_clips=5, frames=4, height=h, width=w, clips_per_chunk=2, pixel_format=fmt,
                            color_matrix="bt709")
    host = pipe.pinned_input()
    assert tuple(host.shape) == (5, 4, h * 3 // 2, w) and host.dtype == torch.uint16 and host.is_pinned()
    host.copy_(surf)
    random.seed(9)
    params = tf.sample_params(5, h, w)
    out = pipe.run(host, params=params).float().numpy().copy()
    want = tf.forward_batch(surf.cuda(), params=params, pixel_format=fmt, color_matrix="bt709").float().cpu().numpy()
    assert np.array_equal(out, want)
    with pytest.raises(ValueError):
        pipe.submit(torch.zeros(pipe.shape, dtype=torch.uint8))


class _Reader:
    def __init__(self, n, seed, h, w, fmt):
        rgb = make_clip_np(n, h, w, seed, "dashcam") if n else np.zeros((0, h, w, 3), np.uint8)
        if fmt == "rgb":
            self.frames = conv16(rgb_to_yuv420_16(rgb, "i010", "bt709", "limited"), "i010", "bt709", "limited") if n else rgb
        else:
            self.frames = rgb_to_yuv420_16(rgb, "i010", "bt709", "limited") if n else np.zeros((0, h * 3 // 2, w), np.uint16)

    def __len__(self):
        return len(self.frames)

    def get_batch(self, idx):
        return self.frames[list(idx)]


def _decoder(fmt):
    def open_(path):
        n, seed = map(int, path.split("_"))
        if n < 0:
            raise IOError("broken video")
        h, w = ((96, 160), (72, 128), (160, 96))[seed % 3]        # three source resolutions in one dataset
        return _Reader(n, seed, h, w, fmt)
    return open_


def _run_loader(fmt):
    from torch.utils.data import DataLoader
    from vision_collision_detection_b200.videos import GpuAugLoader, GpuDashcamDataset, deferred_collate
    tf = _transform(KW_CUSTOM, 56)
    rows = [{"id": f"v{i}", "video_type": "Normal", "path": f"{n}_{i}"} for i, n in enumerate([40, 30, -1, 64, 0, 8])]
    kw = dict(pixel_format="i010", color_matrix="bt709") if fmt == "i010" else {}
    ds = GpuDashcamDataset(rows, fps=4, duration=3, transform=tf, sample_strategy="random", decoder=_decoder(fmt),
                           defer=True, **kw)
    dl = DataLoader(ds, batch_size=3, shuffle=False, num_workers=2, collate_fn=deferred_collate, pin_memory=True,
                    multiprocessing_context="fork", worker_init_fn=lambda i: random.seed(100 + i))
    seen = []

    class Tap:
        def __iter__(self):
            for b in dl:
                seen.append(b)
                yield b

        def __len__(self):
            return len(dl)

    out = [b["frames"].cpu() for b in GpuAugLoader(Tap(), tf)]
    recs = [[(g["index"], g["params"]) for g in b["groups"]] for b in seen]
    return out, recs, seen


@pytest.mark.gpu
def test_training_loader_with_i010_surfaces_equals_rgb_loader():
    """Forked DataLoader workers over a dataset whose decoder delivers 10-bit planar BT.709 surfaces, mixed resolutions,
    one broken and one empty video: the same clips and parameter records as the loader over the oracle's RGB."""
    out_y, recs_y, seen = _run_loader("i010")
    out_rgb, recs_rgb, _ = _run_loader("rgb")
    assert len(out_y) == 2 and all(tuple(o.shape) == (3, 12, 56, 56, 3) for o in out_y)
    assert recs_y == recs_rgb
    assert all(g["format"] == {"pixel_format": "i010", "color_matrix": "bt709", "color_range": "limited"}
               and g["frames_u8"].dtype == torch.uint16 for b in seen for g in b["groups"])
    for a, b in zip(out_y, out_rgb):
        assert torch.equal(a, b)
    assert torch.all(out_y[0][2] == 0)                              # the broken video: the all-zeros clip
    empty = [g for g in seen[1]["groups"] if 1 in g["index"]][0]    # the empty video: neutral surfaces -> RGB zeros
    k = empty["index"].index(1)
    assert conv16(empty["frames_u8"][k].numpy(), "i010", "bt709", "limited").max() == 0


@pytest.mark.gpu
def test_sliding_windows_of_an_i010_video():
    from vision_collision_detection_b200.inference import SlidingWindowTransform, WindowPredictor, center_window
    rgb = make_clip_np(20, 720, 1280, 17, "dashcam")
    i010 = rgb_to_yuv420_16(rgb, "i010", "bt709", "limited")
    conv = _dev(conv16(i010, "i010", "bt709", "limited"))
    dev = _dev(i010)
    sw = SlidingWindowTransform(window=8, stride=4, out_dtype=torch.float32)
    kw = dict(pixel_format="i010", color_matrix="bt709")
    got = sw.windows(dev, **kw)
    assert tuple(got.shape) == (4, 3, 8, 224, 224) and torch.equal(got, sw.windows(conv))
    assert torch.equal(sw.windows(dev, materialize=True, **kw), sw.windows(conv, materialize=True))
    assert torch.equal(center_window(dev, fps=2, duration=4, **kw), center_window(conv, fps=2, duration=4))
    model = lambda x: x.float().mean(dim=(2, 3, 4))
    wp = WindowPredictor(model, window=8, stride=4)
    assert wp.predict(dev, **kw) == wp.predict(conv)
