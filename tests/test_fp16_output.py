"""fp16 output (NEXAR_DST_F16): every element is the fp32 result of the same call rounded to nearest even, so the tensor
is bit for bit what fp16 autocast makes of the fp32 output (include/nexar_clip_transform.h).

Every launch sequence of test_launch_paths.py runs again, with its case builders, into all three layouts with the
specialised and the general geometry kernel; fp16 and fp32 outputs are pre-filled with NaN and compared as int16 bit
patterns.  Then the store branches an unaligned destination takes, the overlapped launches, values outside fp16's
range, the YUV sources, the oracle, every entry point that takes an output dtype, and fp16 autocast itself.
"""
import ctypes
import os
import random
import re

import numpy as np
import pytest
import torch

from oracle import np_oracle as O
from vision_collision_detection_b200 import _lib

import test_launch_paths as LP
from golden_util import oracle_config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F16, F32 = torch.float16, torch.float32


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_header_binding_and_engine_agree_on_f16():
    hdr = open(os.path.join(ROOT, "include", "nexar_clip_transform.h")).read()
    enum = re.search(r"enum\s*\{\s*(NEXAR_DST_F32[^}]*)\}", hdr).group(1)
    values = {k: int(v) for k, v in re.findall(r"(NEXAR_DST_\w+)\s*=\s*(-?\d+)", enum)}
    assert values == {"NEXAR_DST_F32": _lib.DST_F32, "NEXAR_DST_BF16": _lib.DST_BF16, "NEXAR_DST_F16": _lib.DST_F16}
    assert _lib.DST_F16 == 2
    from vision_collision_detection_b200.engine import _DST
    assert _DST[F16] == _lib.DST_F16
    assert set(_DST) == {F32, torch.bfloat16, F16}


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
def _bits_equal(f16, f32):
    """fp16 tensor == fp32 tensor rounded to nearest even (torch's conversion), compared as bit patterns."""
    return torch.equal(f16.contiguous().view(torch.int16), f32.to(F16).contiguous().view(torch.int16))


def _nan_out(layout, b, t, cs, dt, dev, shift=0):
    """A NaN-filled ``out=`` tensor for ``layout``; ``shift`` elements into its storage when asked (a contiguous view)."""
    from vision_collision_detection_b200.engine import _alloc_out
    probe, _ = _alloc_out(layout, b, t, cs, dt, "meta")
    flat = torch.full((probe.numel() + shift,), float("nan"), dtype=dt, device=dev)
    return flat[shift:].view(probe.shape)


def _f16_layouts(tf, frames, params, launches, **kw):
    """One batch in every layout, with the specialised (0) and the general (1) geometry kernel, in fp32 and fp16, each
    into a NaN-filled ``out=``: every fp16 result must be the fp32 result of the same call rounded, every element
    written, and both calls must launch ``launches`` kernels."""
    L = _lib.lib()
    eng = LP._engine()
    b, t, cs = len(params), frames.shape[1], tf.crop_size
    try:
        for layout in LP.LAYOUTS:
            for geo in (0, 1):
                _lib.check(L.nexar_set_geometry_kernel(geo))
                got = {}
                for dt in (F32, F16):
                    out = _nan_out(layout, b, t, cs, dt, frames.device)
                    eng.last_launches = -1
                    tf.forward_batch(frames, params=params, out=out, layout=layout, **kw)
                    torch.cuda.synchronize()
                    assert eng.last_launches == launches, (layout, geo, dt, eng.last_launches, launches)
                    assert not bool(torch.isnan(out).any()), ("unwritten output elements", layout, geo, dt)
                    got[dt] = out
                assert _bits_equal(got[F16], got[F32]), (layout, geo)
    finally:
        L.nexar_set_geometry_kernel(0)


def _tf(**kw):
    from vision_collision_detection_b200 import create_video_transforms
    return create_video_transforms(**kw)


# ---------------------------------------------------------------------------------------------------------------------
# Every launch path, bit for bit
# ---------------------------------------------------------------------------------------------------------------------
PATHS = [(0, "fast"), (2, "fast"), (1, "general")]
PATH_IDS = ["fast", "serialised", "general"]


@pytest.mark.gpu
@pytest.mark.parametrize("variant,path", PATHS, ids=PATH_IDS)
@pytest.mark.parametrize("cs", [224, 320])
def test_plain_letterbox_on_every_path(cs, variant, path):
    """No augmentation: the resize kernels write the pad rows themselves (fill_pads' 16-byte branch on the fast path)."""
    clips = torch.stack([LP._clip(3, 720, 1280, 11), LP._clip(3, 720, 1280, 12, "noise")])
    tf = _tf(mode="train", crop_size=cs)
    params = [{"flip": True, "aug": None, "crop": None}, {"flip": False, "aug": None, "crop": None}]
    try:
        LP._set_resize(variant)
        _f16_layouts(tf, clips, params, LP.LAUNCHES[path][LP.NONE])
    finally:
        LP._set_resize(0)


@pytest.mark.gpu
@pytest.mark.parametrize("variant,path", PATHS, ids=PATH_IDS)
@pytest.mark.parametrize("cs", [224, 320])
def test_fixup_clips_with_augmentation_on_every_path(cs, variant, path):
    """Clips whose maximum is <= 1 with augmentation: fixup_frame_kernel (fast paths) or resize_general_kernel's pass 1
    (general path), gray slot 1, blur."""
    clips, params = LP._fixup_batch()
    tf = _tf(crop_size=cs, **LP.FIXUP_CFG_KW)
    try:
        LP._set_resize(variant)
        _f16_layouts(tf, clips, params, LP.LAUNCHES[path][LP.BLUR])
    finally:
        LP._set_resize(0)


@pytest.mark.gpu
@pytest.mark.parametrize("cs", [224, 320])
def test_blur_call_site_at_production_size(cs):
    """nexar_complete_with_validation.py's kwargs (blur, grayscale, cutout) with a skipped clip in the batch."""
    b, t = 8, 4
    tf = _tf(**dict(LP.KW_NCWV, crop_size=cs))
    clips = torch.stack([LP._clip(t, 720, 1280, 900 + i) for i in range(b)])
    random.seed(1208 + cs)
    params = tf.sample_params(b, 720, 1280)
    params[5]["aug"] = {"skip_augmentation": True}
    assert any(p["aug"].get("apply_blur") for p in params)
    _f16_layouts(tf, clips, params, LP.LAUNCHES["fast"][LP.BLUR])


@pytest.mark.gpu
@pytest.mark.parametrize("h,w,cs,zoom,path", [(448, 448, 224, 1.0, "general"), (720, 1280, 224, 2.0, "fast")])
def test_widest_blur(h, w, cs, zoom, path):
    """33 taps (blur_sigma=4.2): blur_kernel's own stores."""
    tf = _tf(mode="train", crop_size=cs, enable_custom_augmentation=True, blur_sigma=4.2)
    clips = torch.stack([LP._clip(2, h, w, h + cs, "noise"), LP._clip(2, h, w, h + cs + 1, "noise")])
    params = [{"flip": False, "aug": LP._aug(brightness=0.95, contrast=1.1, scale=zoom, apply_blur=True), "crop": None},
              {"flip": True, "aug": LP._aug(saturation=0.8, scale=zoom, apply_blur=True, apply_solarization=True),
               "crop": None}]
    _f16_layouts(tf, clips, params, LP.LAUNCHES[path][LP.BLUR])


@pytest.mark.gpu
@pytest.mark.parametrize("center", [True, False], ids=["center", "random"])
def test_resize_crop_with_augmentation(center):
    from vision_collision_detection_b200 import create_video_transform
    tf = create_video_transform(mode="train", enable_advanced_augmentation=True, use_letterbox=False, min_size=256,
                                max_size=None, crop_size=224, center_crop=center, noise_level=0.0, blur_sigma=0.5,
                                grayscale_prob=0.3, cutout_prob=0.5, solarization_prob=0.3, color_inversion_prob=0.3)
    clips = torch.stack([LP._clip(2, 720, 1280, 40), LP._clip(2, 720, 1280, 41), LP._clip(2, 720, 1280, 42, "noise") & 1])
    random.seed(464 + center)
    params = tf.sample_params(3, 720, 1280)
    _f16_layouts(tf, clips, params, LP.LAUNCHES["crop"][LP.BLUR])


@pytest.mark.gpu
def test_float_sources_with_augmentation():
    """float32 frames in [0,1] and [0,255] in one batch (general resize kernel, float source instances)."""
    tf = _tf(**dict(LP.KW_CUSTOM, blur_sigma=0.5))
    clips = torch.stack([LP._clip(2, 720, 1280, 51).float() / 255.0, LP._clip(2, 720, 1280, 52).float()])
    random.seed(51)
    params = tf.sample_params(2, 720, 1280)
    params[0]["aug"].update(apply_blur=False, apply_color_inversion=True)
    _f16_layouts(tf, clips, params, LP.LAUNCHES["general"][LP.BLUR])


@pytest.mark.gpu
def test_two_pass_factory():
    """create_video_transform's default forward: pass 1 into an fp32 scratch, pass 2 (float source) into fp16."""
    from vision_collision_detection_b200 import create_video_transform
    tf = create_video_transform(mode="train", enable_advanced_augmentation=True, min_size=256, max_size=None,
                                crop_size=224, noise_level=0.0, blur_sigma=0.5, grayscale_prob=0.3)
    clips = torch.stack([LP._clip(2, 720, 1280, 61), LP._clip(2, 720, 1280, 62, "noise") & 1])
    random.seed(407)
    params = tf.sample_params(2, 720, 1280)
    _f16_layouts(tf, clips, params, LP.LAUNCHES["general"][LP.BLUR])


@pytest.mark.gpu
@pytest.mark.parametrize("aug", [False, True], ids=["plain", "aug"])
def test_portrait_pad_columns(aug):
    tf = _tf(**(dict(LP.KW_CUSTOM) if aug else dict(mode="train")))
    clips = torch.stack([LP._clip(2, 1280, 720, 71), LP._clip(2, 1280, 720, 72, "noise")])
    random.seed(71)
    params = tf.sample_params(2, 1280, 720)
    params[0]["flip"], params[1]["flip"] = True, False
    _f16_layouts(tf, clips, params, LP.LAUNCHES["fast"][LP.AUG if aug else LP.NONE])


# ---------------------------------------------------------------------------------------------------------------------
# Store paths, overlap, range
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(mode="train"), LP.KW_CUSTOM], ids=["plain", "custom"])
@pytest.mark.parametrize("layout", LP.LAYOUTS)
def test_destination_one_element_past_16_bytes(kw, layout):
    """``out`` one element into its storage: store_pair's vec2 test and fill_pads' vec_ok test fail, so the scalar
    stores run; the result equals the aligned fp16 result and the fp32 result rounded."""
    clips = torch.stack([LP._clip(2, 720, 1280, 21), LP._clip(2, 720, 1280, 22, "noise")])
    tf = _tf(**kw)
    random.seed(22)
    params = tf.sample_params(2, 720, 1280)
    shifted = _nan_out(layout, 2, 2, 224, F16, clips.device, shift=1)
    assert shifted.is_contiguous() and shifted.data_ptr() % 16 == 2
    tf.forward_batch(clips, params=params, out=shifted, layout=layout)
    aligned = tf.forward_batch(clips, params=params, layout=layout, out_dtype=F16)
    want = tf.forward_batch(clips, params=params, layout=layout, out_dtype=F32)
    assert not bool(torch.isnan(shifted).any())
    assert _bits_equal(shifted, want) and _bits_equal(aligned, want)


@pytest.mark.gpu
def test_overlapped_equals_serialised_at_cfg2_shape():
    """32 x 16 x 720p -> 224 with the live call site's kwargs: the programmatic-dependent launches give the serialised
    result bit for bit in fp16, and both are the fp32 result rounded."""
    b, t = 32, 16
    tf = _tf(**LP.KW_CUSTOM)
    clips = torch.stack([LP._clip(t, 720, 1280, 700 + i) for i in range(b)])
    clips[7] &= 1
    random.seed(2003)
    params = tf.sample_params(b, 720, 1280)
    outs = {}
    try:
        for variant in (0, 2):
            LP._set_resize(variant)
            outs[variant] = tf.forward_batch(clips, params=params, out_dtype=F16)
        LP._set_resize(0)
        out32 = tf.forward_batch(clips, params=params, out_dtype=F32)
    finally:
        LP._set_resize(0)
    assert torch.equal(outs[0].view(torch.int16), outs[2].view(torch.int16))
    assert _bits_equal(outs[0], out32)


@pytest.mark.gpu
def test_unnormalised_and_out_of_range_values():
    """normalize=False keeps [0,1]; a std that scales past 65504 gives the +-inf torch's conversion gives."""
    clips = torch.stack([LP._clip(2, 720, 1280, 31), LP._clip(2, 720, 1280, 32, "noise")])
    for kw in (dict(normalize=False), dict(video_mean=(0.0, 0.5, 1.0), video_std=(1e-5, 1e-5, 1e-5))):
        tf = _tf(**dict(LP.KW_CUSTOM, **kw))
        random.seed(32)
        params = tf.sample_params(2, 720, 1280)
        _f16_layouts(tf, clips, params, LP.LAUNCHES["fast"][LP.AUG])
        f16 = tf.forward_batch(clips, params=params, out_dtype=F16)
        if kw.get("normalize") is False:
            assert 0 <= float(f16.min()) and float(f16.max()) <= 1
        else:
            assert bool(torch.isposinf(f16).any()) and bool(torch.isneginf(f16).any())
            assert bool(torch.isfinite(f16).any())


# ---------------------------------------------------------------------------------------------------------------------
# Sources and the oracle
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fmt,m,r", [("nv12", "bt601", "limited"), ("i420", "bt709", "full"),
                                     ("p010", "bt601", "limited"), ("i010", "bt709", "limited")])
def test_yuv_sources(fmt, m, r):
    from vision_collision_detection_b200.synth import make_clip_np, rgb_to_yuv420, rgb_to_yuv420_16
    rgb = np.stack([make_clip_np(2, 720, 1280, 40 + i, "dashcam") for i in range(2)])
    enc = rgb_to_yuv420_16 if fmt in ("p010", "i010") else rgb_to_yuv420
    surf = torch.from_numpy(enc(rgb, fmt, m, r)).cuda()
    tf = _tf(**LP.KW_CUSTOM)
    random.seed(7)
    params = tf.sample_params(2, 720, 1280)
    kw = dict(params=params, pixel_format=fmt, color_matrix=m, color_range=r)
    f16 = tf.forward_batch(surf, out_dtype=F16, **kw)
    assert f16.dtype == F16 and _bits_equal(f16, tf.forward_batch(surf, out_dtype=F32, **kw))


def _half_ulp_f16(v):
    """Half an fp16 ulp at each value (the subnormal spacing below 2^-14)."""
    _, e = np.frexp(np.maximum(np.abs(v), 2.0 ** -14))
    return np.ldexp(np.float64(1), e.astype(np.int64) - 12)


@pytest.mark.gpu
@pytest.mark.parametrize("cs", [224, 320])
def test_against_the_oracle(cs):
    from vision_collision_detection_b200.synth import make_clip_np
    clip = make_clip_np(2, 720, 1280, 500 + cs, "dashcam")
    kw = dict(LP.KW_CUSTOM, crop_size=cs)
    tf = _tf(**kw)
    random.seed(cs)
    params = tf.sample_params(1, 720, 1280)
    got = tf.forward_batch(torch.from_numpy(clip).cuda().unsqueeze(0), params=params, out_dtype=F16)[0]
    want = O.apply_clip_transform(clip.transpose(3, 0, 1, 2), oracle_config(kw),
                                  {"flip": params[0]["flip"], "aug": params[0]["aug"]}).astype(np.float64)
    err = np.abs(got.cpu().numpy().astype(np.float64) - want)
    assert float((err - (LP.TOL_AFTER + _half_ulp_f16(want))).max()) <= 0, float(err.max())


# ---------------------------------------------------------------------------------------------------------------------
# Entry points
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_forward_model_input_and_forward():
    b, t = 3, 16
    tf = _tf(**LP.KW_CUSTOM)
    clips = torch.stack([LP._clip(t, 720, 1280, 60 + i) for i in range(b)])
    random.seed(60)
    params = tf.sample_params(b, 720, 1280)
    f16 = tf.forward_model_input(clips, params=params, out_dtype=F16)
    assert f16.dtype == F16 and tuple(f16.shape) == (b, t // 2, 3, 224, 224) and f16.is_contiguous()
    assert _bits_equal(f16, tf.forward_model_input(clips, params=params, out_dtype=F32))
    val16, val32 = _tf(mode="val", out_dtype=F16), _tf(mode="val")
    video = clips[0].permute(3, 0, 1, 2)                      # [3,T,H,W]
    out = val16(video)
    assert out.dtype == F16 and _bits_equal(out, val32(video))


@pytest.mark.gpu
def test_host_pipeline():
    from vision_collision_detection_b200.host_pipeline import HostClipPipeline
    n, t, h, w = 5, 4, 180, 320
    tf = _tf(**dict(LP.KW_CUSTOM, crop_size=112))
    src = torch.stack([LP._clip(t, h, w, 90 + i) for i in range(n)]).cpu()
    pipe = HostClipPipeline(tf, n_clips=n, frames=t, height=h, width=w, clips_per_chunk=2, out_dtype=F16)
    host = pipe.pinned_input()
    host.copy_(src)
    random.seed(9)
    params = tf.sample_params(n, h, w)
    out = pipe.run(host, params=params)
    assert out.dtype == F16 and out.is_pinned() and out.element_size() == 2
    dev = tf.forward_batch(src.cuda(), params=params, out_dtype=F16)
    assert torch.equal(out.view(torch.int16), dev.cpu().view(torch.int16))
    assert _bits_equal(out, tf.forward_batch(src.cuda(), params=params, out_dtype=F32).cpu())


def _loader_frames(out_dtype):
    from torch.utils.data import DataLoader
    from vision_collision_detection_b200.videos import GpuAugLoader, GpuDashcamDataset, deferred_collate
    from test_yuv420_16bit import _decoder
    tf = _tf(**dict(LP.KW_CUSTOM, crop_size=56))
    rows = [{"id": f"v{i}", "video_type": "Normal", "path": f"{n}_{i}"} for i, n in enumerate([40, 30, -1, 64, 0, 8])]
    ds = GpuDashcamDataset(rows, fps=4, duration=3, transform=tf, sample_strategy="random", decoder=_decoder("rgb"),
                           defer=True)
    dl = DataLoader(ds, batch_size=3, shuffle=False, num_workers=2, collate_fn=deferred_collate, pin_memory=True,
                    multiprocessing_context="fork", worker_init_fn=lambda i: random.seed(100 + i))
    return [b["frames"] for b in GpuAugLoader(dl, tf, out_dtype=out_dtype)]


@pytest.mark.gpu
def test_training_loader_with_a_failed_item():
    """Forked workers, mixed resolutions, one broken video (index 2): its clip is fp16 zeros."""
    f16, f32 = _loader_frames(F16), _loader_frames(F32)
    assert len(f16) == 2 and all(o.dtype == F16 and tuple(o.shape) == (3, 12, 56, 56, 3) for o in f16)
    for a, b in zip(f16, f32):
        assert _bits_equal(a, b)
    assert bool(torch.all(f16[0][2] == 0)) and bool(torch.all(f16[0][2].view(torch.int16) == 0))


@pytest.mark.gpu
def test_sliding_windows_and_predictor():
    from vision_collision_detection_b200.inference import SlidingWindowTransform, WindowPredictor, center_window
    video = LP._clip(20, 720, 1280, 17)
    s16 = SlidingWindowTransform(window=8, stride=4, out_dtype=F16)
    s32 = SlidingWindowTransform(window=8, stride=4, out_dtype=F32)
    view = s16.windows(video)
    mat = s16.windows(video, materialize=True)
    assert view.dtype == mat.dtype == F16 and tuple(mat.shape) == (4, 3, 8, 224, 224)
    assert torch.equal(mat.view(torch.int16), view.contiguous().view(torch.int16))
    assert _bits_equal(view, s32.windows(video))
    c16 = center_window(video, transform=_tf(mode="val", out_dtype=F16), fps=2, duration=4)
    assert c16.dtype == F16 and _bits_equal(c16, center_window(video, fps=2, duration=4))
    seen = []

    def model(x):
        seen.append(x.dtype)
        return x.float().mean(dim=(2, 3, 4))

    got = WindowPredictor(model, window=8, stride=4, out_dtype=F16).predict(video)
    want = WindowPredictor(lambda x: model(x.to(F16)), window=8, stride=4).predict(video)
    assert seen == [F16] * len(seen) and got == want


# ---------------------------------------------------------------------------------------------------------------------
# Autocast and the C ABI
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_fp16_autocast_sees_the_same_input():
    """convnext_tiny's stem under fp16 autocast: the fp16 output gives the fp32 output's result bit for bit; bf16 does
    not (it is not what autocast makes of the fp32 values)."""
    tf = _tf(**LP.KW_CUSTOM)
    clips = torch.stack([LP._clip(16, 720, 1280, 80 + i) for i in range(2)])
    random.seed(80)
    params = tf.sample_params(2, 720, 1280)
    x = {dt: tf.forward_model_input(clips, params=params, out_dtype=dt).flatten(0, 1) for dt in (F32, F16, torch.bfloat16)}
    det, bench = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    try:
        torch.manual_seed(0)
        stem = torch.nn.Conv2d(3, 96, 4, stride=4).cuda()
        with torch.no_grad(), torch.autocast("cuda", dtype=F16):
            y = {dt: stem(v) for dt, v in x.items()}
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = det, bench
    assert y[F16].dtype == F16
    assert torch.equal(y[F16], y[F32])
    assert not torch.equal(y[torch.bfloat16], y[F32])


@pytest.mark.gpu
def test_c_abi_refuses_other_destination_types():
    from vision_collision_detection_b200.params import pack_clip_params
    eng = LP._engine()
    plan = eng.letterbox_plan(72, 128, 32)
    src = torch.zeros((1, 72, 128, 3), dtype=torch.uint8, device="cuda")
    out = torch.zeros((1, 3, 1, 32, 32), dtype=F16, device="cuda")
    params = eng.upload_params(pack_clip_params([{"flip": False, "aug": None}], 32, None)[0])
    ws = torch.empty(plan.workspace_bytes(1, 1), dtype=torch.uint8, device="cuda")
    offsets = eng.contiguous_offsets(1, 72 * 128 * 3)
    a = _lib.TransformArgs()
    a.struct_size = ctypes.sizeof(_lib.TransformArgs)
    a.n_clips = a.frames_per_clip = 1
    a.src, a.frame_offsets, a.src_row_stride = src.data_ptr(), offsets.data_ptr(), 128 * 3
    a.params, a.dst, a.normalize = params.data_ptr(), out.data_ptr(), 1
    for i, s in enumerate(out.stride()):
        a.dst_stride[i] = s
    for c in range(3):
        a.mean[c], a.std[c] = 0.45, 0.225
    a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
    a.stream = torch.cuda.current_stream().cuda_stream
    L = _lib.lib()
    for bad in (3, -1):
        a.dst_dtype = bad
        assert L.nexar_clip_transform(plan.handle, ctypes.byref(a)) == _lib.ERR_INVALID, bad
        assert "dst_dtype" in L.nexar_last_error().decode()
    a.dst_dtype = _lib.DST_F16
    _lib.check(L.nexar_clip_transform(plan.handle, ctypes.byref(a)))
    torch.cuda.synchronize()
    assert bool(torch.isfinite(out).all())
    with pytest.raises(TypeError):
        eng.run(plan, src, offsets, 1, 1, params, 0, out.double(), out.stride(), True, (0.45,) * 3, (0.225,) * 3)
