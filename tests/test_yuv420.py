"""YUV 4:2:0 decoder surfaces of every supported variant (NV12 / I420, BT.601 / BT.709, limited / full range, padded
surfaces): the integer coefficients, the numpy oracle, the argument checks, and - on the GPU - that every variant is the
RGB path bit for bit once the surfaces are converted, through forward_batch, HostClipPipeline, the deferred training
loader and the inference windows."""
import ctypes
import random

import numpy as np
import pytest
import torch

from oracle import nv12_oracle as N
from oracle import yuv420_oracle as Y
from vision_collision_detection_b200 import _lib
from vision_collision_detection_b200.synth import make_clip_np, rgb_to_nv12, rgb_to_yuv420

MATRICES = ("bt601", "bt709")
RANGES = ("limited", "full")
PAIRS = [(m, r) for m in MATRICES for r in RANGES]


def nv12_to_i420(nv):
    """The same samples re-laid out: [..., L*3/2, P] NV12 -> I420."""
    lr, p = nv.shape[-2] * 2 // 3, nv.shape[-1]
    uv = nv[..., lr:, :]
    planes = np.concatenate([uv[..., 0::2], uv[..., 1::2]], axis=-2)          # [..., L, P/2]: U rows then V rows
    return np.concatenate([nv[..., :lr, :], planes.reshape(nv.shape[:-2] + (lr // 2, p))], axis=-2)


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_coefficients_are_rounded_standard_values():
    derived = {}
    for m, (kr, kb) in {"bt601": (0.299, 0.114), "bt709": (0.2126, 0.0722)}.items():
        kg = 1 - kr - kb
        for r, (yo, ys, cs) in {"limited": (16, 255 / 219, 255 / 224), "full": (0, 1.0, 1.0)}.items():
            c = [ys, 2 * (1 - kr) * cs, 2 * kb * (1 - kb) / kg * cs, 2 * kr * (1 - kr) / kg * cs, 2 * (1 - kb) * cs]
            derived[m, r] = (yo,) + tuple(int(round(256 * v)) for v in c)
    assert derived["bt601", "limited"] == (16, 298, 409, 100, 208, 516)      # nv12_to_rgb's constants
    assert derived["bt601", "full"] == (0, 256, 359, 88, 183, 454)
    assert derived["bt709", "limited"] == (16, 298, 459, 55, 136, 541)
    assert derived["bt709", "full"] == (0, 256, 403, 48, 120, 475)
    codes = {"bt601": _lib.YUV_BT601, "bt709": _lib.YUV_BT709, "limited": _lib.YUV_LIMITED, "full": _lib.YUV_FULL}
    for (m, r), want in derived.items():
        assert Y.yuv_int_coefficients(m, r) == want
        assert _lib.yuv_coefficients(codes[m], codes[r]) == want                # what the kernels use
    with pytest.raises(_lib.NexarError):
        _lib.yuv_coefficients(2, 0)


def _px(y, u, v, m, r, layout="nv12"):
    nv = np.array([[y, y], [y, y], [u, v]], np.uint8)          # one 2 x 2 block
    buf = nv if layout == "nv12" else nv12_to_i420(nv)
    return tuple(int(c) for c in Y.yuv420_to_rgb(buf, layout, m, r)[0, 0])


@pytest.mark.parametrize("m", MATRICES)
def test_known_answers(m):
    assert _px(16, 128, 128, m, "limited") == (0, 0, 0) and _px(235, 128, 128, m, "limited") == (255, 255, 255)
    assert _px(0, 128, 128, m, "full") == (0, 0, 0) and _px(255, 128, 128, m, "full") == (255, 255, 255)
    for layout in ("nv12", "i420"):
        assert all(_px(g, 128, 128, m, "full", layout) == (g, g, g) for g in range(256))   # full-range gray is itself
    assert np.array_equal(Y.yuv420_to_rgb(np.arange(6).reshape(3, 2).astype(np.uint8) * 40),
                          N.nv12_to_rgb(np.arange(6).reshape(3, 2).astype(np.uint8) * 40))


@pytest.mark.parametrize("m,r", PAIRS)
@pytest.mark.parametrize("layout", ["nv12", "i420"])
def test_float_encode_integer_decode_round_trip(m, r, layout):
    g = np.arange(0, 256, 5)
    rgb = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 1, 1, 3)
    rgb = np.broadcast_to(rgb, (rgb.shape[0], 2, 2, 3)).astype(np.uint8)       # each sample fills one 2 x 2 block
    back = Y.yuv420_to_rgb(rgb_to_yuv420(rgb, layout, m, r), layout, m, r)
    assert np.abs(back.astype(int) - rgb.astype(int)).max() <= 2


def test_layouts_agree_and_padding_is_ignored():
    clip = make_clip_np(3, 48, 64, 5, "dashcam")
    for m, r in PAIRS:
        nv = rgb_to_yuv420(clip, "nv12", m, r)
        i4 = rgb_to_yuv420(clip, "i420", m, r)
        assert np.array_equal(nv12_to_i420(nv), i4)
        want = Y.yuv420_to_rgb(nv, "nv12", m, r)
        assert np.array_equal(Y.yuv420_to_rgb(i4, "i420", m, r), want)
        for layout in ("nv12", "i420"):
            padded = rgb_to_yuv420(clip, layout, m, r, luma_rows=56, pitch=80)
            assert padded.shape == (3, 84, 80) and padded[:, 48:56].min() == 255 and padded[:, :48, 64:].min() == 255
            assert np.array_equal(Y.yuv420_to_rgb(padded, layout, m, r, frame_size=(48, 64)), want)
    assert np.array_equal(rgb_to_yuv420(clip[:, :, :, :]), rgb_to_yuv420(clip, "nv12", "bt601", "limited"))
    with pytest.raises(ValueError):
        rgb_to_yuv420(clip, "i420", "bt709", "full", luma_rows=46)
    with pytest.raises(ValueError):
        rgb_to_yuv420(clip, "yuv444")


def test_forward_batch_argument_checks():
    from vision_collision_detection_b200 import create_video_transforms
    tf = create_video_transforms(mode="val", crop_size=32)
    surf = torch.zeros((1, 2, 72, 64), dtype=torch.uint8)           # 48 luma rows, pitch 64 (host: rejected before use)
    for kw in (dict(pixel_format="yuv444"), dict(pixel_format="i420", color_matrix="bt2020"),
               dict(pixel_format="nv12", color_range="studio"), dict(pixel_format="i420", frame_size=(50, 64)),
               dict(pixel_format="i420", frame_size=(47, 64)), dict(pixel_format="nv12", frame_size=(48, 63)),
               dict(pixel_format="nv12", frame_size=(48, 66))):
        with pytest.raises(ValueError):
            tf.forward_batch(surf, **kw)
    with pytest.raises(ValueError):
        tf.forward_batch(torch.zeros((1, 2, 72, 63), dtype=torch.uint8), pixel_format="i420")     # odd pitch
    with pytest.raises(ValueError):
        tf.forward_batch(torch.zeros((1, 2, 71, 64), dtype=torch.uint8), pixel_format="i420")     # not L * 3 / 2 rows
    with pytest.raises(ValueError):
        tf.forward_batch(torch.zeros((1, 2, 48, 64, 3), dtype=torch.uint8), frame_size=(48, 64))  # RGB has no padding
    with pytest.raises(ValueError):
        tf.forward_batch(torch.zeros((1, 2, 48, 64, 3), dtype=torch.uint8), color_matrix="bt2020")
    from vision_collision_detection_b200.videos import GpuDashcamDataset, GpuVideoDataset
    with pytest.raises(ValueError):
        GpuDashcamDataset([], transform=tf, pixel_format="i420")                       # defer=False
    with pytest.raises(ValueError):
        GpuVideoDataset([], [], transform=tf, sample_strategy="center", pixel_format="nv12")
    with pytest.raises(ValueError):
        GpuDashcamDataset([], transform=tf, defer=True, pixel_format="i420", color_range="tv")


def test_plan_checks_of_the_c_abi():
    """nexar_plan_create_yuv validates the descriptor before it touches the device."""
    L = _lib.yuv_lib()
    assert L.nexar_sizeof_yuv_format() == ctypes.sizeof(_lib.YuvFormat) == 20
    g = _lib.Geometry(48, 64, 32, 24, 32, 4, 0)

    def create(struct_size=ctypes.sizeof(_lib.YuvFormat), layout=0, matrix=0, range_=0, luma_rows=0, geom=g):
        f = _lib.YuvFormat(struct_size, layout, matrix, range_, luma_rows)
        h = ctypes.c_void_p()
        return L.nexar_plan_create_yuv(ctypes.byref(geom), ctypes.byref(f), ctypes.byref(h))

    for bad in (dict(struct_size=16), dict(layout=2), dict(matrix=-1), dict(range_=2), dict(luma_rows=46),
                dict(luma_rows=51), dict(geom=_lib.Geometry(47, 64, 32, 24, 32, 4, 0))):
        assert create(**bad) == _lib.ERR_INVALID, bad


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
KW_CUSTOM = dict(mode="train", enable_custom_augmentation=True, brightness_range=(0.9, 1.1), contrast_range=(0.9, 1.1),
                 saturation_range=(0.9, 1.1), rotation_range=(-5, 5))


def _transform(kw, cs, **extra):
    from vision_collision_detection_b200 import create_video_transforms
    return create_video_transforms(**kw, crop_size=cs, **extra)


@pytest.mark.gpu
@pytest.mark.parametrize("h,w,cs", [(720, 1280, 224), (90, 150, 64)], ids=["720p_vec", "90x150_any"])
@pytest.mark.parametrize("kw", [dict(mode="val"), KW_CUSTOM], ids=["val", "custom"])
@pytest.mark.parametrize("m,r", PAIRS)
@pytest.mark.parametrize("layout", ["nv12", "i420"])
def test_every_format_equals_rgb_path_on_converted_frames(h, w, cs, kw, m, r, layout):
    """720p takes the vector conversion kernel and the fast resize, 90 x 150 the byte-wise conversion and the general
    resize.  The small size uses arbitrary bytes to exercise the clipping branches."""
    if w % 16:
        surf = np.random.RandomState(3).randint(0, 256, (2, 3, h * 3 // 2, w)).astype(np.uint8)
    else:
        surf = rgb_to_yuv420(np.stack([make_clip_np(3, h, w, 11 + i, "dashcam") for i in range(2)]), layout, m, r)
    rgb = Y.yuv420_to_rgb(surf, layout, m, r)
    tf = _transform(kw, cs)
    random.seed(5)
    params = tf.sample_params(2, h, w)
    got = tf.forward_batch(torch.from_numpy(surf).cuda(), params=params, pixel_format=layout, color_matrix=m,
                           color_range=r).cpu().numpy()
    want = tf.forward_batch(torch.from_numpy(rgb).cuda(), params=params).cpu().numpy()
    assert got.shape == (2, 3, 3, cs, cs) and np.array_equal(got, want)


@pytest.mark.gpu
def test_explicit_default_format_and_layouts_agree():
    tf = _transform(KW_CUSTOM, 112)
    nv = rgb_to_nv12(np.stack([make_clip_np(3, 180, 320, 40 + i, "dashcam") for i in range(2)]))
    random.seed(8)
    params = tf.sample_params(2, 180, 320)
    dev = torch.from_numpy(nv).cuda()
    plain = tf.forward_batch(dev, params=params, pixel_format="nv12")
    explicit = tf.forward_batch(dev, params=params, pixel_format="nv12", color_matrix="bt601", color_range="limited",
                                frame_size=(180, 320))
    assert torch.equal(plain, explicit)
    for m, r in PAIRS:
        a = tf.forward_batch(dev, params=params, pixel_format="nv12", color_matrix=m, color_range=r)
        b = tf.forward_batch(torch.from_numpy(nv12_to_i420(nv)).cuda(), params=params, pixel_format="i420",
                             color_matrix=m, color_range=r)
        assert torch.equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("layout,m,r", [("nv12", "bt709", "limited"), ("i420", "bt709", "full"), ("nv12", "bt601", "limited")])
def test_padded_1080p_surfaces(layout, m, r):
    """1080p in the 1088-row, pitch-2048 surfaces of a hardware decoder; every padding byte is 255."""
    clip = make_clip_np(2, 1080, 1920, 21, "dashcam")
    packed = torch.from_numpy(rgb_to_yuv420(clip, layout, m, r)).cuda().unsqueeze(0)
    padded_np = rgb_to_yuv420(clip, layout, m, r, luma_rows=1088, pitch=2048)
    assert padded_np.shape == (2, 1632, 2048) and padded_np[:, 1080:1088].min() == 255
    padded = torch.from_numpy(padded_np).cuda().unsqueeze(0)
    tf = _transform(KW_CUSTOM, 224)
    random.seed(2)
    params = tf.sample_params(1, 1080, 1920)
    kw = dict(params=params, pixel_format=layout, color_matrix=m, color_range=r)
    want = tf.forward_batch(packed, **kw)
    got = tf.forward_batch(padded, frame_size=(1080, 1920), **kw)
    assert torch.equal(got, want)
    rgb = tf.forward_batch(torch.from_numpy(Y.yuv420_to_rgb(padded_np, layout, m, r, (1080, 1920))).cuda().unsqueeze(0),
                           params=params)
    assert torch.equal(got, rgb)


@pytest.mark.gpu
def test_frame_index_and_clip_max_rule():
    """A full-range clip whose luma is 0/1 with neutral chroma converts to RGB 0/1 values: the clip maximum is <= 1, so
    it is NOT divided by 255 - exactly as the RGB clip of those values."""
    h, w, cs = 96, 160, 64
    i4 = rgb_to_yuv420(np.stack([make_clip_np(4, h, w, 70 + i, "dashcam") for i in range(2)]), "i420", "bt709", "full")
    i4[1, :, :h] = np.random.RandomState(1).randint(0, 2, (4, h, w))
    i4[1, :, h:] = 128
    rgb = Y.yuv420_to_rgb(i4, "i420", "bt709", "full")
    assert rgb[1].max() == 1 and rgb[1].min() == 0
    tf = _transform(dict(mode="val"), cs)
    index = torch.tensor([[3, 1, 1], [4, 7, 5]])
    got = tf.forward_batch(torch.from_numpy(i4).cuda(), frame_index=index, pixel_format="i420", color_matrix="bt709",
                           color_range="full").cpu().numpy()
    want = tf.forward_batch(torch.from_numpy(rgb).cuda(), frame_index=index).cpu().numpy()
    assert np.array_equal(got, want)


@pytest.mark.gpu
def test_host_pipeline_i420_bt709():
    from vision_collision_detection_b200.host_pipeline import HostClipPipeline
    h, w, cs = 180, 320, 112
    tf = _transform(KW_CUSTOM, cs, out_dtype=torch.bfloat16)
    surf = torch.from_numpy(rgb_to_yuv420(np.stack([make_clip_np(4, h, w, 90 + i, "dashcam") for i in range(5)]),
                                          "i420", "bt709", "limited"))
    pipe = HostClipPipeline(tf, n_clips=5, frames=4, height=h, width=w, clips_per_chunk=2, pixel_format="i420",
                            color_matrix="bt709")
    host = pipe.pinned_input()
    assert tuple(host.shape) == (5, 4, h * 3 // 2, w)
    host.copy_(surf)
    random.seed(9)
    params = tf.sample_params(5, h, w)
    out = pipe.run(host, params=params).float().numpy().copy()
    want = tf.forward_batch(surf.cuda(), params=params, pixel_format="i420", color_matrix="bt709").float().cpu().numpy()
    assert np.array_equal(out, want)


class _Reader:
    def __init__(self, n, seed, h, w, fmt):
        rgb = make_clip_np(n, h, w, seed, "dashcam") if n else np.zeros((0, h, w, 3), np.uint8)
        if fmt == "rgb":
            self.frames = Y.yuv420_to_rgb(rgb_to_yuv420(rgb, "i420", "bt709", "limited"), "i420", "bt709") if n else rgb
        else:
            self.frames = rgb_to_yuv420(rgb, "i420", "bt709", "limited") if n else np.zeros((0, h * 3 // 2, w), np.uint8)

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
    kw = dict(pixel_format="i420", color_matrix="bt709") if fmt == "i420" else {}
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
def test_training_loader_with_i420_surfaces_equals_rgb_loader():
    """Forked DataLoader workers over a dataset whose decoder delivers I420 BT.709 surfaces, mixed resolutions, one
    broken and one empty video: the same clips and parameter records as the same loader over the RGB frames the oracle
    converts those surfaces to."""
    out_y, recs_y, seen = _run_loader("i420")
    out_rgb, recs_rgb, _ = _run_loader("rgb")
    assert len(out_y) == 2 and all(tuple(o.shape) == (3, 12, 56, 56, 3) for o in out_y)
    assert recs_y == recs_rgb
    assert all(g["format"] == {"pixel_format": "i420", "color_matrix": "bt709", "color_range": "limited"}
               for b in seen for g in b["groups"])
    for a, b in zip(out_y, out_rgb):
        assert torch.equal(a, b)
    assert torch.all(out_y[0][2] == 0)                              # the broken video: the all-zeros clip
    empty = [g for g in seen[1]["groups"] if 1 in g["index"]][0]    # the empty video: neutral surfaces -> RGB zeros
    k = empty["index"].index(1)
    assert Y.yuv420_to_rgb(empty["frames_u8"][k].numpy(), "i420", "bt709").max() == 0


@pytest.mark.gpu
def test_sliding_windows_of_an_i420_video():
    from vision_collision_detection_b200.inference import SlidingWindowTransform, WindowPredictor, center_window
    rgb = make_clip_np(20, 720, 1280, 17, "dashcam")
    i4 = rgb_to_yuv420(rgb, "i420", "bt709", "limited")
    conv = torch.from_numpy(Y.yuv420_to_rgb(i4, "i420", "bt709")).cuda()
    dev = torch.from_numpy(i4).cuda()
    sw = SlidingWindowTransform(window=8, stride=4, out_dtype=torch.float32)
    kw = dict(pixel_format="i420", color_matrix="bt709")
    got = sw.windows(dev, **kw)
    assert tuple(got.shape) == (4, 3, 8, 224, 224) and torch.equal(got, sw.windows(conv))
    assert torch.equal(sw.windows(dev, materialize=True, **kw), sw.windows(conv, materialize=True))
    assert torch.equal(center_window(dev, fps=2, duration=4, **kw), center_window(conv, fps=2, duration=4))
    model = lambda x: x.float().mean(dim=(2, 3, 4))
    wp = WindowPredictor(model, window=8, stride=4)
    assert wp.predict(dev, **kw) == wp.predict(conv)
