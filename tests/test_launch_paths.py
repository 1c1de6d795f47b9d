"""Every kernel sequence launch_all (csrc/clip_transform.cu) dispatches, against the numpy oracle at production sizes.

test_gpu_parity.py pins the path bench.py times (720p -> 224 / 320, fast resize kernel, colour and geometry kernels).
The other launch sequences have their own instruction streams and store code: the fix-up of clips whose maximum is
<= 1 (fixup_frame_kernel, which finishes augmented clips with fixup_colour_geometry), the general fp32 resize with its
gray slot for those clips, the blur kernel behind the specialised geometry kernel, the resize-crop variant, float
sources and the two-pass singular factory.  Each case asserts the launch count of the path it claims, writes every
output layout in fp32 and bf16 into tensors pre-filled with NaN, and compares the fp32 result with the oracle.

Gates as in test_gpu_parity.py: 1e-3 after normalisation on fp32; bf16 equals the fp32 result of the same kernels
rounded to nearest even, bit for bit.  Noise and posterize are off (noise is checked statistically elsewhere,
posterize may flip a level).  The per-frame chain has no temporal dependence, so the oracle checks a subset of the
frames of long 720p clips; the /255 decision is still taken on the whole clip.
"""
import functools
import random

import numpy as np
import pytest
import torch

from oracle import np_oracle as O

from golden_util import META, decode, oracle_config

pytestmark = pytest.mark.gpu

TOL_AFTER = 1e-3
SPEC_VS_GENERAL = 2e-6          # specialised vs general geometry kernel: one fused multiply-add differs
LAYOUTS = ("BCTHW", "BTCHW", "BTHWC")
_TO_BCTHW = {"BCTHW": (0, 1, 2, 3, 4), "BTCHW": (0, 2, 1, 3, 4), "BTHWC": (0, 4, 1, 2, 3)}

# Kernel launches of one call (nexar_last_launch_count), from launch_all:
#   fast letterbox   K1 + fix-up                        | + K2 + K3 (K1 writes the frame stats) | + blur
#   general letterbox K1 pass 0 + pass 1                | + frame stats + K2 + K3                | + blur
#   resize-crop      clip max + K1 pass 2               | + frame stats + K2 + K3                | + blur
# YUV sources add their conversion kernel; the two-pass forward reports its second (float source) pass.
LAUNCHES = {"fast": (2, 4, 5), "general": (2, 5, 6), "crop": (2, 5, 6)}
NONE, AUG, BLUR = 0, 1, 2

# nexar_complete_with_validation.py:1208-1225, the call site that enables blur (same kwargs as the golden ncwv cases)
KW_NCWV = {k: (tuple(v) if isinstance(v, list) else v) for k, v in decode(META["cases"]["ncwv_small_s0"]["kwargs"]).items()}
# nexar_videos.py:2003-2010
KW_CUSTOM = dict(mode="train", enable_custom_augmentation=True, brightness_range=(0.9, 1.1), contrast_range=(0.9, 1.1),
                 saturation_range=(0.9, 1.1), rotation_range=(-5, 5))


def _lib():
    from vision_collision_detection_b200 import _lib as L
    return L


def _engine():
    from vision_collision_detection_b200.engine import get_engine
    return get_engine(torch.device("cuda", torch.cuda.current_device()))


@functools.lru_cache(maxsize=None)
def _clip(t, h, w, seed, kind="dashcam"):
    """uint8 [T,H,W,3] on the device (the bytes of synth.make_clip_np, generated on the GPU)."""
    from vision_collision_detection_b200.synth import make_clip_torch
    return make_clip_torch(t, h, w, seed, kind)


def _set_resize(variant):
    _lib().check(_lib().lib().nexar_set_resize_kernel(variant))


def _aug(**kw):
    """A hand-written augmentation record: identity colour and geometry, every effect off, then ``kw``."""
    p = dict(brightness=1.0, contrast=1.0, saturation=1.0, hue=0.0, rotation=0.0, scale=1.0, shear=0.0,
             translate_x=0.0, translate_y=0.0, apply_grayscale=False, apply_noise=False, apply_blur=False,
             apply_cutout=False, cutout_boxes=[], apply_color_inversion=False, apply_solarization=False,
             apply_posterization=False)
    p.update(kw)
    p["apply_affine"] = any(p[n] != d for n, d in (("rotation", 0), ("scale", 1), ("shear", 0), ("translate_x", 0),
                                                   ("translate_y", 0)))
    return p


def _want(clip, cfg, params, frames):
    """Oracle of the listed frames of one clip ([T,H,W,3] uint8 or float32, host or device), [3, len(frames), cs, cs].
    The /255 rule (nexar_video_aug.py:814) looks at the WHOLE clip, so it is applied here before taking the subset."""
    v = clip.cpu().numpy() if isinstance(clip, torch.Tensor) else np.asarray(clip)
    sub = v[list(frames)].astype(np.float32)
    if v.max() > 1:
        sub = sub / np.float32(255.0)
    return O.apply_clip_transform(sub.transpose(3, 0, 1, 2), cfg, params)


def _assert_close(got, want, what):
    err = float(np.abs(got - want).max())
    assert err <= TOL_AFTER, (what, err)


def _run_layouts(tf, frames, params, launches, **kw):
    """One batch into every output layout, fp32 and bf16, each into an ``out=`` tensor pre-filled with NaN (a fresh
    torch.empty may reuse a block that already holds a previous call's values, so only this shows an element no
    kernel wrote).  BCTHW also runs with the general geometry kernel forced: it is what the other layouts take, so
    they must equal it bit for bit, and the specialised kernel must agree with it to SPEC_VS_GENERAL.  Every call must
    launch ``launches`` kernels.  Returns the fp32 [B,3,T,cs,cs] results (default kernels, general geometry kernel)."""
    from vision_collision_detection_b200.engine import _alloc_out
    L = _lib().lib()
    eng = _engine()
    b, t, cs = len(params), frames.shape[1], tf.crop_size
    got = {}
    try:
        for dt in (torch.float32, torch.bfloat16):
            for layout in LAYOUTS:
                for geo in ((0, 1) if layout == "BCTHW" else (0,)):
                    _lib().check(L.nexar_set_geometry_kernel(geo))
                    probe, _ = _alloc_out(layout, b, t, cs, dt, "meta")
                    out = torch.full(tuple(probe.shape), float("nan"), dtype=dt, device=frames.device)
                    eng.last_launches = -1
                    tf.forward_batch(frames, params=params, out=out, layout=layout, **kw)
                    torch.cuda.synchronize()
                    assert eng.last_launches == launches, (layout, dt, geo, eng.last_launches, launches)
                    assert not bool(torch.isnan(out).any()), ("unwritten output elements", layout, dt, geo)
                    got[dt, layout, geo] = out.permute(_TO_BCTHW[layout])
    finally:
        L.nexar_set_geometry_kernel(0)
    spec, gen = got[torch.float32, "BCTHW", 0], got[torch.float32, "BCTHW", 1]
    for dt in (torch.float32, torch.bfloat16):
        assert torch.equal(got[dt, "BCTHW", 1], gen.to(dt)), dt
        for layout in LAYOUTS[1:]:
            assert torch.equal(got[dt, layout, 0], got[dt, "BCTHW", 1]), (layout, dt)
    assert torch.equal(got[torch.bfloat16, "BCTHW", 0], spec.to(torch.bfloat16))
    assert float((spec - gen).abs().max()) <= SPEC_VS_GENERAL
    return spec.cpu().numpy(), gen.cpu().numpy()


# ---------------------------------------------------------------------------------------------------------------------
# 1. Fix-up clips (maximum <= 1) with augmentation, on every letterbox path
# ---------------------------------------------------------------------------------------------------------------------
FIXUP_T = 3
FIXUP_CFG_KW = dict(mode="train", enable_custom_augmentation=True, blur_sigma=0.5)


def _fixup_batch():
    """A normal dashcam clip, a {0,1} clip (flipped, affine, hue, contrast), an all-zero clip (affine, inverted) and a
    {0,1} clip with grayscale, inversion, solarisation, cutout and blur: 720p, 3 frames each."""
    clips = torch.stack([_clip(FIXUP_T, 720, 1280, 81), _clip(FIXUP_T, 720, 1280, 82, "noise") & 1,
                         torch.zeros(FIXUP_T, 720, 1280, 3, dtype=torch.uint8, device="cuda"),
                         _clip(FIXUP_T, 720, 1280, 83) & 1])
    params = [
        {"flip": False, "aug": _aug(brightness=1.05, contrast=0.93, saturation=1.08, hue=0.03, rotation=4.0,
                                    scale=0.97, shear=1.5, translate_x=2.0, translate_y=-1.5)},
        {"flip": True, "aug": _aug(brightness=0.9, contrast=1.6, saturation=1.2, hue=0.21, rotation=-9.0, scale=1.07,
                                   shear=3.0, translate_x=-5.5, translate_y=4.0)},
        {"flip": False, "aug": _aug(brightness=1.1, contrast=0.8, rotation=13.0, scale=0.9, translate_x=7.0,
                                    apply_color_inversion=True)},
        {"flip": True, "aug": _aug(brightness=1.02, contrast=1.1, saturation=0.7, hue=-0.08, rotation=2.0,
                                   apply_grayscale=True, apply_color_inversion=True, apply_solarization=True,
                                   apply_blur=True, apply_cutout=True,
                                   cutout_boxes=[(30, 40, 25, 30), (150, 100, 22, 22)])},
    ]
    for p in params:
        p["crop"] = None
    return clips, params


@functools.lru_cache(maxsize=None)
def _fixup_oracle(cs):
    clips, params = _fixup_batch()
    cfg = O.TransformConfig(crop_size=cs, enable_custom_augmentation=True, aug=O.AugConfig(blur_sigma=0.5))
    return [_want(clips[i], cfg, params[i], range(FIXUP_T)) for i in range(len(params))]


@pytest.mark.parametrize("variant,path", [(0, "fast"), (2, "fast"), (1, "general")], ids=["fast", "serialised", "general"])
@pytest.mark.parametrize("cs", [224, 320])
def test_fixup_clips_with_augmentation_on_every_path(cs, variant, path):
    """Clips whose maximum is <= 1 (a failed decode, the neutral surface of an undecodable YUV window) are not divided
    by 255.  On the fast path fixup_frame_kernel redoes them (fp32 resample + fixup_colour_geometry, gray slot 1); on
    the general path pass 1 of resize_general_kernel does, and frame_stats_kernel must read slot 1 for them.  BCTHW
    takes the specialised geometry kernel (125x224 / 180x320 content), the other layouts the general one."""
    from vision_collision_detection_b200 import create_video_transforms
    clips, params = _fixup_batch()
    tf = create_video_transforms(crop_size=cs, **FIXUP_CFG_KW)
    try:
        _set_resize(variant)
        spec, gen = _run_layouts(tf, clips, params, LAUNCHES[path][BLUR])
    finally:
        _set_resize(0)
    for i, want in enumerate(_fixup_oracle(cs)):
        _assert_close(spec[i], want, ("specialised", i))
        _assert_close(gen[i], want, ("general", i))


# ---------------------------------------------------------------------------------------------------------------------
# 2. The call site that enables blur, at its real size
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cs", [224, 320])
def test_ncwv_call_site_at_production_size(cs):
    """nexar_complete_with_validation.py's kwargs (blur_sigma=0.5, grayscale, cutout) at crop 224 (its default) and
    320: the specialised geometry kernel with the tail writes the planar canvas, blur_kernel reflects at its edge and
    stores through the output strides.  The reference factory does not forward aug_probability, so its draws never
    skip; a skipped record (what VideoAugmentation(aug_probability < 1) produces) is put in by hand, as is a grayscale
    clip when the seed draws none, so augmented, skipped and tail-effect clips share the batch."""
    from vision_collision_detection_b200 import create_video_transforms
    b, t = 8, 4
    tf = create_video_transforms(**dict(KW_NCWV, crop_size=cs))
    clips = torch.stack([_clip(t, 720, 1280, 900 + i) for i in range(b)])
    random.seed(1208 + cs)
    params = tf.sample_params(b, 720, 1280)
    if not any(p["aug"].get("skip_augmentation") for p in params):
        params[5]["aug"] = {"skip_augmentation": True}
    if not any(p["aug"].get("apply_grayscale") or p["aug"].get("apply_cutout") for p in params):
        params[2]["aug"]["apply_grayscale"] = True
    live = [p["aug"] for p in params if not p["aug"].get("skip_augmentation")]
    assert any(a["apply_blur"] for a in live) and len(live) < b
    assert any(a["apply_grayscale"] or a["apply_cutout"] for a in live)
    spec, gen = _run_layouts(tf, clips, params, LAUNCHES["fast"][BLUR])
    cfg = oracle_config(dict(KW_NCWV, crop_size=cs))
    for i in range(b):
        want = _want(clips[i], cfg, params[i], (0, t - 1))
        _assert_close(spec[i][:, [0, t - 1]], want, ("specialised", i))
        _assert_close(gen[i][:, [0, t - 1]], want, ("general", i))


# ---------------------------------------------------------------------------------------------------------------------
# 3. Blur kernel limits
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("h,w,cs,zoom,path", [(80, 80, 40, 1.0, "general"), (128, 128, 64, 1.0, "general"),
                                              (448, 448, 224, 1.0, "general"), (720, 1280, 224, 2.0, "fast")])
def test_widest_blur_kernel_against_oracle(h, w, cs, zoom, path):
    """blur_sigma=4.2 gives 33 taps (NEXAR_MAX_BLUR_TAPS): 16 reflected rows and columns at every edge.  A wrong
    reflection only shows where the border is content, not a constant pad band: square noise sources have no pad
    (they take the general resize kernel), and a 2x affine zoom of a 720p letterbox fills the whole canvas (fast
    resize kernel, specialised geometry kernel writing the blur canvas)."""
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.params import gaussian_taps
    assert len(gaussian_taps(4.2)) == _lib().MAX_BLUR_TAPS
    tf = create_video_transforms(mode="train", crop_size=cs, enable_custom_augmentation=True, blur_sigma=4.2)
    clips = torch.stack([_clip(2, h, w, h + cs, "noise"), _clip(2, h, w, h + cs + 1, "noise")])
    params = [{"flip": False, "aug": _aug(brightness=0.95, contrast=1.1, scale=zoom, apply_blur=True), "crop": None},
              {"flip": True, "aug": _aug(saturation=0.8, scale=zoom, apply_blur=True, apply_solarization=True),
               "crop": None}]
    spec, _ = _run_layouts(tf, clips, params, LAUNCHES[path][BLUR])
    cfg = O.TransformConfig(crop_size=cs, enable_custom_augmentation=True, aug=O.AugConfig(blur_sigma=4.2))
    for i in range(2):
        _assert_close(spec[i], _want(clips[i], cfg, params[i], range(2)), i)


def test_blur_kernel_over_the_tap_limit_is_refused_before_launch():
    """blur_sigma=4.25 gives 35 taps: ValueError from the parameter packing, and no kernel is enqueued."""
    from vision_collision_detection_b200 import create_video_transforms
    tf = create_video_transforms(mode="train", crop_size=224, enable_custom_augmentation=True, blur_sigma=4.25)
    eng = _engine()
    eng.last_launches = -1
    with pytest.raises(ValueError, match="35 taps"):
        tf.forward_batch(_clip(1, 720, 1280, 5).unsqueeze(0), params=[{"flip": False, "aug": _aug(apply_blur=True), "crop": None}])
    assert eng.last_launches == -1


# ---------------------------------------------------------------------------------------------------------------------
# 4. Resize-crop with augmentation
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("center", [True, False], ids=["center", "random"])
def test_resize_crop_with_augmentation(center):
    """create_video_transform(use_letterbox=False): clip_max_kernel + resize_general_kernel pass 2 + frame stats +
    colour kernel without overlap + general geometry kernel (+ blur).  Oracle from the pinned primitives: short side
    -> 256, 224 crop at the recorded offset, flip, augment_frame per frame, normalise."""
    from vision_collision_detection_b200 import create_video_transform
    t, size, cs = 2, 256, 224
    tf = create_video_transform(mode="train", enable_advanced_augmentation=True, use_letterbox=False, min_size=size,
                                max_size=None, crop_size=cs, center_crop=center, noise_level=0.0, blur_sigma=0.5,
                                grayscale_prob=0.3, cutout_prob=0.5, solarization_prob=0.3, color_inversion_prob=0.3)
    clips = torch.stack([_clip(t, 720, 1280, 40), _clip(t, 720, 1280, 41), _clip(t, 720, 1280, 42, "noise") & 1])
    random.seed(464 + center)
    params = tf.sample_params(3, 720, 1280)
    params[1]["aug"].update(apply_blur=False, apply_solarization=True)        # tail effects stored by the geometry kernel
    spec, _ = _run_layouts(tf, clips, params, LAUNCHES["crop"][BLUR])
    acfg = O.AugConfig(blur_sigma=0.5)
    for i, p in enumerate(params):
        top, left = p["crop_top_left"]
        if center:
            assert (top, left) == ((size - cs) // 2, (size * 1280 // 720 - cs) // 2)
        v = O.resize_crop_transform(clips[i].cpu().numpy().transpose(3, 0, 1, 2), size, cs, top, left)
        if p["flip"]:
            v = v[..., ::-1].copy()
        v = np.stack([O.augment_frame(v[:, k], p["aug"], acfg) for k in range(t)], axis=1)
        want = O.normalize(v, tf.video_mean, tf.video_std)
        _assert_close(spec[i], want, i)


# ---------------------------------------------------------------------------------------------------------------------
# 5. Float sources with augmentation
# ---------------------------------------------------------------------------------------------------------------------
def test_float_sources_with_augmentation():
    """float32 frames take the general resize kernel: a [0,1] clip (no /255, pass 1, gray slot 1) and a [0,255] clip
    (pass 0, slot 0) in one batch, with the live call site's kwargs plus blur."""
    from vision_collision_detection_b200 import create_video_transforms
    t = 2
    kw = dict(KW_CUSTOM, blur_sigma=0.5)
    tf = create_video_transforms(**kw)
    clips = torch.stack([_clip(t, 720, 1280, 51).float() / 255.0, _clip(t, 720, 1280, 52).float()])
    random.seed(51)
    params = tf.sample_params(2, 720, 1280)
    params[0]["aug"].update(apply_blur=False, apply_color_inversion=True)
    spec, _ = _run_layouts(tf, clips, params, LAUNCHES["general"][BLUR])
    cfg = O.TransformConfig(crop_size=224, enable_custom_augmentation=True, aug=O.AugConfig(blur_sigma=0.5))
    for i in range(2):
        _assert_close(spec[i], _want(clips[i], cfg, params[i], range(t)), i)


def test_singular_factory_two_pass_with_augmentation():
    """create_video_transform's default forward: short side -> 256 (uint8 source, no augmentation), then a letterbox
    of those float frames with flip, augmentation and normalisation.  The second pass is a float32 source, so it
    takes the general resize kernel; its [0,1] values are never divided again."""
    from vision_collision_detection_b200 import create_video_transform
    t, size, cs = 2, 256, 224
    tf = create_video_transform(mode="train", enable_advanced_augmentation=True, min_size=size, max_size=None,
                                crop_size=cs, noise_level=0.0, blur_sigma=0.5, grayscale_prob=0.3)
    clips = torch.stack([_clip(t, 720, 1280, 61), _clip(t, 720, 1280, 62, "noise") & 1])
    random.seed(407)
    params = tf.sample_params(2, 720, 1280)
    spec, _ = _run_layouts(tf, clips, params, LAUNCHES["general"][BLUR])
    acfg = O.AugConfig(blur_sigma=0.5)
    for i, p in enumerate(params):
        v = O.letterbox_resize(O.resize_short_side(O.prologue(clips[i].cpu().numpy().transpose(3, 0, 1, 2)), size), cs)
        if p["flip"]:
            v = v[..., ::-1].copy()
        v = np.stack([O.augment_frame(v[:, k], p["aug"], acfg) for k in range(t)], axis=1)
        _assert_close(spec[i], O.normalize(v, tf.video_mean, tf.video_std), i)


# ---------------------------------------------------------------------------------------------------------------------
# 6. Overlapped launches equal the serialised run at the benched shape
# ---------------------------------------------------------------------------------------------------------------------
def test_overlapped_equals_serialised_at_cfg2_shape():
    """K2 is a programmatic dependent of K1 and waits per frame on publication flags; the fix-up is a programmatic
    dependent of K3.  nexar_set_resize_kernel(2) orders all of them by the stream instead: the result must be the
    same bit for bit, at 32 x 16 x 720p -> 224 bf16 with two fix-up clips ({0,1} and all-zero) in the batch."""
    from vision_collision_detection_b200 import create_video_transforms
    b, t = 32, 16
    tf = create_video_transforms(**dict(KW_NCWV, crop_size=224))
    clips = torch.stack([_clip(t, 720, 1280, 700 + i) for i in range(b)])
    clips[7] &= 1
    clips[20].zero_()
    random.seed(2003)
    params = tf.sample_params(b, 720, 1280)
    if params[7]["aug"].get("skip_augmentation"):
        params[7]["aug"] = next(p["aug"] for p in params if not p["aug"].get("skip_augmentation"))
    eng = _engine()
    outs = {}
    try:
        for variant in (0, 2):
            _set_resize(variant)
            outs[variant] = tf.forward_batch(clips, params=params, out_dtype=torch.bfloat16)
            torch.cuda.synchronize()
            assert eng.last_launches == LAUNCHES["fast"][BLUR], (variant, eng.last_launches)
        _set_resize(0)
        out32 = tf.forward_batch(clips, params=params)
    finally:
        _set_resize(0)
    assert torch.equal(outs[0], outs[2])
    assert torch.equal(outs[0], out32.to(torch.bfloat16))
    cfg = oracle_config(dict(KW_NCWV, crop_size=224))
    for i in (3, 7, 29):
        want = _want(clips[i], cfg, params[i], (0, t - 1))
        _assert_close(out32[i][:, [0, t - 1]].cpu().numpy(), want, i)


# ---------------------------------------------------------------------------------------------------------------------
# 7. Portrait sources: the pad is columns
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("aug", [False, True], ids=["plain", "aug"])
def test_portrait_pad_columns_are_written(aug):
    """A 1280-row x 720-column source letterboxes to 224 x 126 with 49 / 49 pad COLUMNS: without augmentation the fast
    resize kernel writes them (fill_pads' column loop), with augmentation the geometry kernel does."""
    from vision_collision_detection_b200 import create_video_transforms
    t = 2
    kw = dict(KW_CUSTOM) if aug else dict(mode="train")
    tf = create_video_transforms(**kw)
    clips = torch.stack([_clip(t, 1280, 720, 71), _clip(t, 1280, 720, 72, "noise")])
    random.seed(71)
    params = tf.sample_params(2, 1280, 720)
    params[0]["flip"], params[1]["flip"] = True, False
    spec, _ = _run_layouts(tf, clips, params, LAUNCHES["fast"][AUG if aug else NONE])
    cfg = O.TransformConfig(crop_size=224, enable_custom_augmentation=aug, aug=O.AugConfig(rotation_range=(-5, 5)))
    for i in range(2):
        _assert_close(spec[i], _want(clips[i], cfg, params[i], range(t)), i)
