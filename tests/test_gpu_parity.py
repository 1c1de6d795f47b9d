"""GPU parity: the CUDA path (through the C ABI) against the numpy oracle and the
reference's frozen outputs.  Tolerances are north_star's: 1/255 max-abs before
normalisation, 1e-3 after (asserted on the fp32 output); bf16 output is held to
one bf16 ulp of the rounded oracle."""
import random

import numpy as np
import pytest
import torch

from oracle import np_oracle as O

from golden_util import case_names, load_case, special

pytestmark = pytest.mark.gpu

TOL_BEFORE = 1.0 / 255.0
TOL_AFTER = 1e-3


def _tf(kwargs, **extra):
    from vision_collision_detection_b200 import create_video_transforms
    return create_video_transforms(**kwargs, **extra)


def _run(tf, clip_u8, params):
    frames = torch.from_numpy(clip_u8).cuda().unsqueeze(0)
    rec = dict(params)
    rec.setdefault("crop", None)
    out = tf.forward_batch(frames, params=[rec])
    torch.cuda.synchronize()
    return out[0].float().cpu().numpy()


def _poster_ok(out, gold, tol, frac=5e-3):
    return (np.abs(out - gold) > tol).mean() <= frac


@pytest.mark.parametrize("name", case_names())
def test_matches_reference_golden(name):
    c = load_case(name)
    out = _run(_tf(c["kwargs"]), c["clip"], c["params"])
    assert out.shape == c["out"].shape
    tol = TOL_AFTER if c["cfg"].normalize else TOL_BEFORE
    if name.startswith("poster"):
        assert _poster_ok(out, c["out"], tol)
    else:
        assert np.abs(out - c["out"]).max() <= tol


@pytest.mark.parametrize("name", ["val_small", "val_portrait", "val_upscale", "custom_small_s0", "ncwv_small_s2",
                                  "allfx_small_s3", "allfx_small_s6"])
def test_before_normalisation_within_one_255th(name):
    c = load_case(name)
    kw = dict(c["kwargs"], normalize=False)
    out = _run(_tf(kw), c["clip"], c["params"])
    want = O.apply_clip_transform(c["clip"].transpose(3, 0, 1, 2), c["cfg"], c["params"], stage="aug")
    assert np.abs(out - want).max() <= TOL_BEFORE
    assert np.abs(out - want).max() <= 1e-4          # in practice ~1e-6


def test_reference_call_signature_and_rng_stream():
    """transform(video[C,T,H,W] u8 view) -> [C,T,cs,cs] f32, drawing from ``random`` like the reference."""
    c = load_case("custom_small_s1")
    tf = _tf(c["kwargs"])
    video = torch.from_numpy(c["clip"]).permute(3, 0, 1, 2)       # CPU, non-contiguous view
    random.seed(c["random_seed"])
    out = tf(video)
    assert out.device.type == "cpu" and out.dtype == torch.float32 and tuple(out.shape) == c["out"].shape
    assert np.abs(out.numpy() - c["out"]).max() <= TOL_AFTER
    assert tf.last_params[0]["flip"] == c["params"]["flip"]
    assert tf.last_params[0]["aug"] == c["params"]["aug"]          # bit-exact decisions
    random.seed(c["random_seed"])
    out_cuda = tf(video.cuda())
    assert out_cuda.is_cuda and torch.equal(out_cuda.cpu(), out)


def test_special_inputs_max_rule_and_float():
    sp = special()
    from vision_collision_detection_b200.synth import make_clip_np
    tf = _tf(dict(mode="val", crop_size=56))
    b01 = (make_clip_np(2, 96, 160, 50, "noise") & 1).astype(np.uint8)
    out = tf(torch.from_numpy(b01).permute(3, 0, 1, 2)).numpy()
    assert np.abs(out - sp["max1_u8"]).max() <= TOL_AFTER and out.max() > 1.0
    z = torch.zeros(3, 2, 96, 160, dtype=torch.uint8)
    assert np.abs(tf(z).numpy() - sp["zeros_u8"]).max() <= TOL_AFTER
    f01 = torch.from_numpy(make_clip_np(2, 96, 160, 51, "dashcam").astype(np.float32) / 255.0).permute(3, 0, 1, 2)
    assert np.abs(tf(f01).numpy() - sp["float01"]).max() <= TOL_AFTER
    f255 = torch.from_numpy(make_clip_np(2, 96, 160, 52, "dashcam").astype(np.float32)).permute(3, 0, 1, 2)
    assert np.abs(tf(f255).numpy() - sp["float255"]).max() <= TOL_AFTER


def test_mixed_batch_max_rule_is_per_clip():
    """One all-{0,1} clip inside a normal batch: only that clip skips the /255."""
    from vision_collision_detection_b200.synth import make_clip_np
    a = make_clip_np(2, 96, 160, 60, "dashcam")
    b = (make_clip_np(2, 96, 160, 61, "noise") & 1).astype(np.uint8)
    tf = _tf(dict(mode="val", crop_size=56))
    out = tf.forward_batch(torch.from_numpy(np.stack([a, b, a])).cuda()).cpu().numpy()
    cfg = O.TransformConfig(mode="val", crop_size=56)
    nop = {"flip": False, "aug": None}
    for i, clip in enumerate([a, b, a]):
        want = O.apply_clip_transform(clip.transpose(3, 0, 1, 2), cfg, nop)
        assert np.abs(out[i] - want).max() <= TOL_AFTER


def test_resize_crop_variant():
    """R11: short side -> size, centre / random crop (bit-exact offsets from the same seed)."""
    from vision_collision_detection_b200 import create_video_transform
    from vision_collision_detection_b200.synth import make_clip_np
    from golden_util import META
    sp = special()
    clip = make_clip_np(2, 96, 160, 53, "dashcam")
    video = torch.from_numpy(clip).permute(3, 0, 1, 2)
    tfc = create_video_transform(mode="val", min_size=56, crop_size=56, normalize=False, use_letterbox=False)
    assert np.abs(tfc(video).numpy() - sp["r11_center"]).max() <= TOL_BEFORE
    tfr = create_video_transform(mode="train", min_size=56, max_size=None, crop_size=56, normalize=False,
                                 use_letterbox=False, horizontal_flip_prob=0.0)
    random.seed(11)
    out = tfr(video).numpy()
    assert tfr.last_params[0]["crop_top_left"] == (0, META["r11_random_left"])
    assert np.abs(out - sp["r11_random"]).max() <= TOL_BEFORE


def test_singular_factory_default_two_pass():
    """create_video_transform's default forward chains two antialiased resizes (nexar_video_aug.py:407-463)."""
    from vision_collision_detection_b200 import create_video_transform
    from vision_collision_detection_b200.synth import make_clip_np
    sp = special()
    video = torch.from_numpy(make_clip_np(2, 96, 160, 53, "dashcam")).permute(3, 0, 1, 2)
    tf = create_video_transform(mode="val", min_size=40, crop_size=56)
    assert np.abs(tf(video).numpy() - sp["singular_val_40_56"]).max() <= TOL_AFTER
    tf = create_video_transform(mode="train", min_size=40, max_size=None, crop_size=56, horizontal_flip_prob=1.0)
    random.seed(5)
    assert np.abs(tf(video).numpy() - sp["singular_train_flip_40_56"]).max() <= TOL_AFTER


def test_bf16_output_and_layouts():
    c = load_case("custom_small_s2")
    want = torch.from_numpy(c["out"])
    tf = _tf(c["kwargs"])
    frames = torch.from_numpy(c["clip"]).cuda().unsqueeze(0)
    rec = dict(c["params"], crop=None)
    ref32 = tf.forward_batch(frames, params=[rec])[0]
    o16 = tf.forward_batch(frames, params=[rec], out_dtype=torch.bfloat16)[0]
    assert o16.dtype == torch.bfloat16
    assert torch.equal(o16, ref32.to(torch.bfloat16))             # same fp32 value, RNE
    # within one bf16 ulp of the rounded oracle
    w16 = want.to(torch.bfloat16).float()
    ulp = torch.maximum(w16.abs(), torch.tensor(2.0 ** -6)) * 2.0 ** -7
    assert ((o16.float().cpu() - w16).abs() <= ulp + 1e-3).all()
    bt = tf.forward_batch(frames, params=[rec], layout="BTCHW")[0]        # [T,C,H,W]
    assert torch.equal(bt.permute(1, 0, 2, 3), ref32)
    bl = tf.forward_batch(frames, params=[rec], layout="BTHWC")[0]        # [T,H,W,C] (Dataset layout)
    assert torch.equal(bl.permute(3, 0, 1, 2), ref32)


def test_frame_gather_equals_copy():
    """Temporal sampling by index gather (repeat-last-frame padding included) == materialised clip."""
    from vision_collision_detection_b200.synth import make_clip_np
    pool = make_clip_np(7, 96, 160, 70, "dashcam")
    idx = [2, 3, 4, 5, 6, 6, 6, 6]
    tf = _tf(dict(mode="val", crop_size=56))
    a = tf.forward_batch(torch.from_numpy(pool[idx]).cuda().unsqueeze(0))
    b = tf.forward_batch(torch.from_numpy(pool).cuda().unsqueeze(0), frame_index=torch.tensor([idx]))
    assert torch.equal(a, b)


def test_model_input_fast_path_equals_subsampled_full_result():
    """F2: only the frames the model keeps (nexar_arch.py:411-415), written frame-major."""
    c = load_case("custom_small_s3")
    from vision_collision_detection_b200.synth import make_clip_np
    clip = make_clip_np(12, 96, 160, 77, "dashcam")
    tf = _tf(c["kwargs"])
    frames = torch.from_numpy(np.stack([clip, clip[::-1].copy()])).cuda()
    recs = [dict(c["params"], crop=None), dict(c["params"], crop=None, flip=not c["params"]["flip"])]
    full = tf.forward_batch(frames, params=recs)                          # [2,3,12,cs,cs]
    fast = tf.forward_model_input(frames, params=recs)                    # [2,6,3,cs,cs]
    assert tuple(fast.shape) == (2, 6, 3, 56, 56)
    same = bool(torch.equal(fast.permute(0, 2, 1, 3, 4), full[:, :, ::2]))
    assert same
    short = tf.forward_model_input(frames[:, :8], params=recs)            # T <= 10: nothing is dropped
    assert tuple(short.shape) == (2, 8, 3, 56, 56)


def test_full_size_properties():
    """BASELINE cfg2 frame size (720p -> 224): size-independent properties on the device."""
    from vision_collision_detection_b200.synth import make_clip_torch
    clips = torch.stack([make_clip_torch(4, 720, 1280, s, "dashcam") for s in range(3)])
    tf = _tf(dict(mode="train"))
    recs = [{"flip": f, "aug": None, "crop": None} for f in (False, True, False)]
    out = tf.forward_batch(clips, params=recs)
    assert tuple(out.shape) == (3, 3, 4, 224, 224)
    assert torch.all(out[:, :, :, :49] == -2.0) and torch.all(out[:, :, :, 174:] == -2.0)   # 49 / 50 pad rows
    assert out[:, :, :, 49:174].min() > -2.0
    # flip is an exact mirror of the un-flipped result
    noflip = tf.forward_batch(clips[1:2], params=[{"flip": False, "aug": None, "crop": None}])
    assert torch.equal(out[1:2], noflip.flip(-1))
    # constant frames stay constant through the antialiased resize (weights sum to one)
    const = torch.full((1, 2, 720, 1280, 3), 200, dtype=torch.uint8, device="cuda")
    oc = tf.forward_batch(const, params=[{"flip": False, "aug": None, "crop": None}])
    want = (200.0 / 255.0 - 0.45) / 0.225
    assert (oc[:, :, :, 49:174] - want).abs().max() <= 1e-5
    # idempotence / determinism
    assert torch.equal(out, tf.forward_batch(clips, params=recs))


@pytest.mark.parametrize("name", ["val_720p_noise", "train_720p_dashcam", "custom_720p_dashcam", "val_1080p_noise",
                                  "val_720p_320", "val_small", "val_portrait", "train_portrait_flip",
                                  "custom_small_s0", "allfx_small_s1"])
@pytest.mark.parametrize("bands", [0, 1, 3, 7])
def test_fast_and_general_resize_kernels_agree(name, bands):
    """The fixed-point input-stationary kernel and the general fp32 kernel both meet the gate, for any banding; the
    serialised launch sequence (variant 2: no programmatic overlap) gives the default's result bit for bit."""
    from vision_collision_detection_b200 import _lib
    c = load_case(name)
    tol = TOL_AFTER if c["cfg"].normalize else TOL_BEFORE
    L = _lib.lib()
    try:
        _lib.check(L.nexar_set_resize_kernel(1))
        general = _run(_tf(c["kwargs"]), c["clip"], c["params"])
        _lib.check(L.nexar_set_resize_kernel(0))
        L.nexar_set_fast_bands(bands)
        fast = _run(_tf(c["kwargs"]), c["clip"], c["params"])
        _lib.check(L.nexar_set_resize_kernel(2))
        serial = _run(_tf(c["kwargs"]), c["clip"], c["params"])
    finally:
        L.nexar_set_resize_kernel(0)
        L.nexar_set_fast_bands(0)
    assert np.abs(general - c["out"]).max() <= tol
    assert np.abs(fast - c["out"]).max() <= tol
    assert np.abs(fast - general).max() <= 2.5e-4      # fixed-point budget: < 3e-5 of full scale, /0.225
    assert np.array_equal(serial, fast)


@pytest.mark.parametrize("h,w,cs", [(720, 1280, 448), (480, 640, 224), (360, 640, 224), (1080, 1920, 320),
                                    (2160, 3840, 224), (720, 1280, 112), (224, 224, 224), (300, 500, 224),
                                    (1280, 720, 224), (64, 64, 320)])
def test_geometry_zoo_against_oracle(h, w, cs):
    """Realistic and awkward geometries (fast kernel, general kernel, up-scale, portrait, 4K), one noise frame each."""
    from vision_collision_detection_b200.synth import make_clip_np
    clip = make_clip_np(1, h, w, h + w + cs, "noise")
    kw = dict(mode="train", crop_size=cs, horizontal_flip_prob=1.0)
    out = _run(_tf(kw), clip, {"flip": True, "aug": None})
    cfg = O.TransformConfig(mode="train", crop_size=cs, horizontal_flip_prob=1.0)
    want = O.apply_clip_transform(clip.transpose(3, 0, 1, 2), cfg, {"flip": True, "aug": None})
    err = float(np.abs(out - want).max())
    assert err <= TOL_AFTER, err


def test_gaussian_noise_is_statistically_right():
    """nexar_video_aug.py:244-246: clamp(frame + randn * level, 0, 1).  torch's generator cannot be matched bit for
    bit on the device, so the check is statistical: zero mean, sigma == noise_level, per-frame independence."""
    from vision_collision_detection_b200.synth import make_clip_np
    clip = np.full((3, 96, 160, 3), 128, np.uint8)                     # mid-gray: the clamp never bites at sigma 0.05
    base = dict(mode="train", crop_size=64, normalize=False, horizontal_flip_prob=0.0, enable_custom_augmentation=True,
                brightness_range=(1, 1), contrast_range=(1, 1), saturation_range=(1, 1), hue_range=(0, 0),
                rotation_range=(0, 0), scale_range=(1, 1), shear_range=(0, 0), translate_range=(0, 0))
    random.seed(0)
    clean = _tf(base)(torch.from_numpy(clip).permute(3, 0, 1, 2)).numpy()
    random.seed(0)
    noisy = _tf(dict(base, noise_level=0.05))(torch.from_numpy(clip).permute(3, 0, 1, 2)).numpy()
    content = (slice(None), slice(None), slice(13, 51), slice(None))   # letterbox content rows of 96x160 -> 64 (38 rows, pad 13)
    d = (noisy - clean)[content]
    assert abs(float(d.mean())) < 2e-3
    assert abs(float(d.std()) - 0.05) < 2.5e-3
    assert abs(float(np.corrcoef(d[:, 0].ravel(), d[:, 1].ravel())[0, 1])) < 0.05     # frames get independent noise
    assert abs(float(np.corrcoef(d[0].ravel(), d[1].ravel())[0, 1])) < 0.05           # and so do channels
    pad = (noisy - clean)[:, :, :13]                                    # pad rows: clamp(0 + n, 0, 1) keeps the positive half
    assert float(pad.min()) >= 0.0 and 0.015 < float(pad.mean()) < 0.025


def test_extreme_parameters_against_oracle():
    """Hue at +-0.5, strong rotation / scale / shear / translation, brightness clamp, zero saturation."""
    from vision_collision_detection_b200.synth import make_clip_np
    clip = make_clip_np(2, 96, 160, 91, "dashcam")
    cfg = O.TransformConfig(mode="train", crop_size=64, enable_custom_augmentation=True, aug=O.AugConfig())
    kw = dict(mode="train", crop_size=64, enable_custom_augmentation=True)
    for k, aug in enumerate([
        dict(brightness=1.9, contrast=0.2, saturation=0.0, hue=0.5, rotation=170.0, scale=0.5, shear=25.0, translate_x=20.0, translate_y=-13.0),
        dict(brightness=0.1, contrast=2.5, saturation=3.0, hue=-0.5, rotation=-90.0, scale=2.0, shear=-40.0, translate_x=-31.5, translate_y=7.25),
        dict(brightness=1.0, contrast=1.0, saturation=1.0, hue=0.0, rotation=0.0, scale=1.0, shear=0.0, translate_x=0.0, translate_y=0.0),
    ]):
        p = dict(aug, apply_affine=any(aug[n] != d for n, d in (("rotation", 0), ("scale", 1), ("shear", 0), ("translate_x", 0), ("translate_y", 0))),
                 apply_grayscale=False, apply_noise=False, apply_blur=False, apply_cutout=False,
                 apply_color_inversion=bool(k == 1), apply_solarization=bool(k == 0), apply_posterization=False)
        params = {"flip": bool(k & 1), "aug": p}
        out = _run(_tf(kw), clip, params)
        want = O.apply_clip_transform(clip.transpose(3, 0, 1, 2), cfg, params)
        err = float(np.abs(out - want).max())
        assert err <= TOL_AFTER, (k, err)


@pytest.mark.parametrize("t", [1, 3, 5, 9])
def test_frames_of_a_clip_do_not_depend_on_how_they_are_grouped(t):
    """K3 computes a pixel's geometry once and reuses it for groups of frames of the clip: a T-frame clip must equal
    its frames transformed one by one with the same parameters, bit for bit, for every group remainder; clips with
    and without augmentation (and with tail effects) share one batch."""
    from vision_collision_detection_b200.synth import make_clip_np
    kw = dict(mode="train", crop_size=64, enable_custom_augmentation=True)
    tf = _tf(kw)
    base = dict(brightness=1.05, contrast=0.93, saturation=1.08, hue=0.03, rotation=4.0, scale=0.97, shear=1.5,
                translate_x=2.0, translate_y=-1.5, apply_affine=True, apply_grayscale=False, apply_noise=False,
                apply_blur=False, apply_cutout=False, apply_color_inversion=False, apply_solarization=False,
                apply_posterization=False)
    recs = [{"flip": False, "aug": dict(base), "crop": None},
            {"flip": True, "aug": None, "crop": None},
            {"flip": True, "aug": dict(base, rotation=-11.0, apply_grayscale=True, apply_color_inversion=True), "crop": None},
            {"flip": False, "aug": dict(base, rotation=0.0, scale=1.0, shear=0.0, translate_x=0.0, translate_y=0.0,
                                        apply_affine=False), "crop": None}]
    clips = np.stack([make_clip_np(t, 96, 160, 300 + i, "dashcam") for i in range(len(recs))])
    frames = torch.from_numpy(clips).cuda()
    whole = tf.forward_batch(frames, params=recs).float().cpu().numpy()          # [B, 3, T, cs, cs]
    singles = frames.reshape(len(recs) * t, 1, 96, 160, 3)
    one = tf.forward_batch(singles, params=[r for r in recs for _ in range(t)]).float().cpu().numpy()
    one = one.reshape(len(recs), t, 3, 64, 64).transpose(0, 2, 1, 3, 4)
    assert np.array_equal(whole, one)
    cfg = O.TransformConfig(mode="train", crop_size=64, enable_custom_augmentation=True, aug=O.AugConfig())
    for i, r in enumerate(recs):
        if r["aug"] is None:
            continue
        want = O.apply_clip_transform(clips[i].transpose(3, 0, 1, 2), cfg, {"flip": r["flip"], "aug": r["aug"]})
        err = float(np.abs(whole[i] - want).max())
        assert err <= TOL_AFTER, (i, err)


@pytest.mark.parametrize("h,w,cs,pad", [(720, 1280, 224, 64), (96, 160, 56, 16), (97, 131, 64, 7)])
def test_padded_source_rows_equal_packed_rows(h, w, cs, pad):
    """Decoders hand out frames whose rows are padded: the C ABI takes the row stride in bytes.  A padded 720p
    source takes the run-time-stride instantiation of the fast kernel (the packed one is specialised on 3840 bytes),
    odd strides take the general kernel; all must equal the packed result bit for bit."""
    from vision_collision_detection_b200.engine import get_engine, _alloc_out
    from vision_collision_detection_b200.params import pack_clip_params
    from vision_collision_detection_b200.synth import make_clip_np
    t = 3
    clip = make_clip_np(t, h, w, 77, "dashcam")
    tf = _tf(dict(mode="train", crop_size=cs, enable_custom_augmentation=True))
    random.seed(5)
    frames = torch.from_numpy(clip).cuda().unsqueeze(0)
    want = tf.forward_batch(frames).float().cpu().numpy()
    params = tf.last_params
    eng = get_engine(frames.device)
    plan = tf._plan(eng, h, w, torch.uint8)
    stride = w * 3 + pad
    buf = torch.full((t, h, stride), 255, dtype=torch.uint8, device="cuda")       # the padding must never be read
    buf[:, :, :w * 3] = frames[0].reshape(t, h, w * 3)
    offsets = torch.arange(t, dtype=torch.int64, device="cuda") * (h * stride)
    packed, any_flags = pack_clip_params(params, cs, tf.video_aug)
    out, strides = _alloc_out("BCTHW", 1, t, cs, torch.float32, frames.device)
    eng.run(plan, buf, offsets, 1, t, eng.upload_params(packed), any_flags, out, strides,
            tf.normalize, tf.video_mean, tf.video_std, src_row_stride=stride)
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    if (w * 3) % 16 == 0 and stride % 16 == 0:
        assert np.array_equal(got, want)            # same kernel arithmetic, different addressing
    else:
        assert np.abs(got - want).max() <= 2.5e-4    # general kernel (fp32) against the fast kernel or itself


@pytest.mark.parametrize("name", ["custom_720p_dashcam", "custom_small_s0", "ncwv_small_s2"])
def test_result_does_not_depend_on_the_band_count(name):
    """The resize kernel splits a frame into bands of rows (the count follows the batch size); the frame's gray mean
    (contrast blend) is summed in fixed point, so augmented results are bit-identical for any banding - a clip's
    output does not depend on the batch it travels in."""
    from vision_collision_detection_b200 import _lib
    c = load_case(name)
    L = _lib.lib()
    outs = []
    try:
        for bands in (1, 2, 5, 8):
            L.nexar_set_fast_bands(bands)
            outs.append(_run(_tf(c["kwargs"]), c["clip"], c["params"]))
    finally:
        L.nexar_set_fast_bands(0)
    for o in outs[1:]:
        assert np.array_equal(o, outs[0])


@pytest.mark.parametrize("h,w,cs", [(720, 1280, 320), (720, 1280, 448), (360, 640, 288)])
def test_wide_outputs_with_augmentation_against_oracle(h, w, cs):
    """Outputs wider than the 256-thread block of the resize kernel (two pixels per thread in the horizontal pass;
    BASELINE config 3 is 720p -> 320) with the live call site's augmentation, two frames, against the oracle."""
    from vision_collision_detection_b200.synth import make_clip_np
    clip = make_clip_np(2, h, w, 500 + cs, "dashcam")
    kw = dict(mode="train", crop_size=cs, enable_custom_augmentation=True, brightness_range=(0.9, 1.1),
              contrast_range=(0.9, 1.1), saturation_range=(0.9, 1.1), rotation_range=(-5, 5))
    tf = _tf(kw)
    random.seed(cs)
    params = tf.sample_params(1, h, w)[0]
    out = _run(tf, clip, params)
    cfg = O.TransformConfig(mode="train", crop_size=cs, enable_custom_augmentation=True, aug=O.AugConfig(
        brightness_range=(0.9, 1.1), contrast_range=(0.9, 1.1), saturation_range=(0.9, 1.1), rotation_range=(-5, 5)))
    want = O.apply_clip_transform(clip.transpose(3, 0, 1, 2), cfg, {"flip": params["flip"], "aug": params["aug"]})
    err = float(np.abs(out - want).max())
    assert err <= TOL_AFTER, err


@pytest.mark.parametrize("mode", ["val", "train", "custom"])
def test_cfg1_sixteen_frame_720p_clip_against_the_reference(mode):
    """BASELINE.json configs[0] on the device: one 16-frame 1280x720 clip through the reference-compatible call
    (``tf(video[C,T,H,W])``), same ``random`` seed, against the output the UNMODIFIED reference produced
    (tests/golden/golden_cfg1_16f.npz: every 5th row / column of every frame + every frame's channel means)."""
    import os
    from golden_util import GOLDEN_DIR
    from vision_collision_detection_b200.synth import make_clip_np
    g = np.load(os.path.join(GOLDEN_DIR, "golden_cfg1_16f.npz"))
    kw = {"val": dict(mode="val"), "train": dict(mode="train"),
          "custom": dict(mode="train", enable_custom_augmentation=True, brightness_range=(0.9, 1.1),
                         contrast_range=(0.9, 1.1), saturation_range=(0.9, 1.1), rotation_range=(-5, 5))}[mode]
    video = torch.from_numpy(make_clip_np(16, 720, 1280, 101, "dashcam")).permute(3, 0, 1, 2)
    random.seed(2024)
    out = _tf(kw)(video.cuda()).float().cpu().numpy()
    assert out.shape == (3, 16, 224, 224)
    assert np.abs(out[:, :, ::5, ::5] - g[f"{mode}_sub"]).max() <= TOL_AFTER
    assert np.abs(out.astype(np.float64).mean(axis=(2, 3)) - g[f"{mode}_mean"]).max() <= 1e-4


def test_cfg2_batch_shape_against_the_cpu_port():
    """The benched shape itself (BASELINE.json configs[1]): 32 clips x 16 x 720p -> 224, 32 DIFFERENT parameter records,
    bf16 and fp32 outputs of the same launch sequence; three clips of the batch are checked against the CPU port of the
    reference (oracle/torch_port.py, itself pinned to the reference's outputs), the rest through batch independence:
    every clip must equal the same clip transformed alone, bit for bit."""
    from oracle import torch_port as P
    from vision_collision_detection_b200.synth import make_clip_torch
    kw = dict(mode="train", enable_custom_augmentation=True, brightness_range=(0.9, 1.1), contrast_range=(0.9, 1.1),
              saturation_range=(0.9, 1.1), rotation_range=(-5, 5))
    tf = _tf(kw)
    b, t, h, w = 32, 16, 720, 1280
    clips = torch.stack([make_clip_torch(t, h, w, seed=700 + i, kind="dashcam") for i in range(b)])
    random.seed(4321)
    recs = tf.sample_params(b, h, w)
    assert len({r["flip"] for r in recs}) == 2 and len({r["aug"]["rotation"] for r in recs}) == b
    out32 = tf.forward_batch(clips, params=recs)
    out16 = tf.forward_batch(clips, params=recs, out_dtype=torch.bfloat16)
    assert tuple(out32.shape) == (b, 3, t, 224, 224) and out16.dtype == torch.bfloat16
    assert torch.equal(out16, out32.to(torch.bfloat16))                      # bf16 = the fp32 result rounded to nearest even
    cfg = O.TransformConfig(mode="train", crop_size=224, enable_custom_augmentation=True, aug=O.AugConfig(rotation_range=(-5, 5)))
    for i in (0, 13, 31):
        want = P.apply_clip_transform(clips[i].cpu().permute(3, 0, 1, 2), cfg, {"flip": recs[i]["flip"], "aug": recs[i]["aug"]}).numpy()
        err = float(np.abs(out32[i].cpu().numpy() - want).max())
        assert err <= TOL_AFTER, (i, err)
    for i in (5, 22):
        alone = tf.forward_batch(clips[i:i + 1], params=[recs[i]])
        assert torch.equal(alone[0], out32[i]), i


def test_noise_is_fresh_per_call_and_reproducible_per_record():
    """ADVICE r1: the noise seed is drawn per clip and call from torch's global generator (the stream the reference's
    randn_like consumes), never a constant; a parameter record reproduces its own noise."""
    clip = np.full((2, 96, 160, 3), 128, np.uint8)
    kw = dict(mode="train", crop_size=64, normalize=False, horizontal_flip_prob=0.0, enable_custom_augmentation=True,
              brightness_range=(1, 1), contrast_range=(1, 1), saturation_range=(1, 1), hue_range=(0, 0),
              rotation_range=(0, 0), scale_range=(1, 1), shear_range=(0, 0), translate_range=(0, 0), noise_level=0.05)
    tf = _tf(kw)
    x = torch.from_numpy(clip).permute(3, 0, 1, 2)
    a = tf(x).numpy()
    rec_a = tf.last_params
    b = tf(x).numpy()
    content = (slice(None), slice(None), slice(13, 51), slice(None))
    da, db = (a - 128 / 255.0)[content], (b - 128 / 255.0)[content]
    assert abs(float(np.corrcoef(da.ravel(), db.ravel())[0, 1])) < 0.05      # two calls: uncorrelated noise
    assert rec_a[0]["noise_seed"] != tf.last_params[0]["noise_seed"]
    frames = torch.from_numpy(clip).cuda().unsqueeze(0)
    again = tf.forward_batch(frames, params=rec_a)[0].cpu().numpy()
    assert np.array_equal(again, a)                                          # the record reproduces its noise
    torch.manual_seed(77)
    c = tf(x).numpy()
    torch.manual_seed(77)
    assert np.array_equal(tf(x).numpy(), c)                                  # torch.manual_seed controls it, as in the reference


def test_frame_index_out_of_range_is_refused():
    tf = _tf(dict(mode="val", crop_size=32))
    frames = torch.zeros((1, 4, 48, 64, 3), dtype=torch.uint8, device="cuda")
    with pytest.raises(ValueError, match="frame_index"):
        tf.forward_batch(frames, frame_index=torch.tensor([[0, 1, 4]]))
    with pytest.raises(ValueError, match="frame_index"):
        tf.forward_batch(frames, frame_index=torch.tensor([[-1, 1, 2]]))
    assert tuple(tf.forward_batch(frames, frame_index=torch.tensor([[3, 3, 0]])).shape) == (1, 3, 3, 32, 32)


@pytest.mark.parametrize("cs,t", [(224, 3), (224, 9), (320, 2)])
def test_specialised_and_general_geometry_kernels_agree(cs, t):
    """720p -> 224 / 320 letterboxes writing a planar tensor take geometry_spec_kernel (compile-time frame sizes, one
    pointer per pixel, clamped 2 x 2 window, packed fp32 blend); everything else the general geometry_kernel.  Both
    must give the same pixels, for the live call site's parameters and for extreme ones (the whole canvas becomes
    boundary tiles), with and without the point effects, in fp32 and bf16, and both must match the oracle."""
    from vision_collision_detection_b200 import _lib
    from vision_collision_detection_b200.synth import make_clip_np
    clip = make_clip_np(t, 720, 1280, 700 + cs + t, "dashcam")
    kw = dict(mode="train", crop_size=cs, enable_custom_augmentation=True, brightness_range=(0.9, 1.1),
              contrast_range=(0.9, 1.1), saturation_range=(0.9, 1.1), rotation_range=(-5, 5))
    tf = _tf(kw)
    random.seed(31 * cs + t)
    live = tf.sample_params(1, 720, 1280)[0]
    wild = dict(brightness=1.4, contrast=0.6, saturation=1.7, hue=0.31, rotation=133.0, scale=0.6, shear=21.0,
                translate_x=37.0, translate_y=-55.5, apply_affine=True, apply_grayscale=False, apply_noise=False,
                apply_blur=False, apply_cutout=False, apply_color_inversion=True, apply_solarization=True,
                apply_posterization=False)
    zoom = dict(wild, rotation=-4.0, scale=2.2, shear=0.0, translate_x=-9.0, translate_y=3.0,
                apply_color_inversion=False, apply_solarization=False)
    ident = dict(wild, brightness=1.0, contrast=1.0, saturation=1.0, hue=0.0, rotation=0.0, scale=1.0, shear=0.0,
                 translate_x=0.0, translate_y=0.0, apply_affine=False, apply_color_inversion=False, apply_solarization=False)
    cfg = O.TransformConfig(mode="train", crop_size=cs, enable_custom_augmentation=True, aug=O.AugConfig(
        brightness_range=(0.9, 1.1), contrast_range=(0.9, 1.1), saturation_range=(0.9, 1.1), rotation_range=(-5, 5)))
    L = _lib.lib()
    for k, params in enumerate([live, {"flip": True, "aug": wild}, {"flip": False, "aug": zoom}, {"flip": True, "aug": ident}]):
        outs = {}
        try:
            for variant in (0, 1):
                L.nexar_set_geometry_kernel(variant)
                outs[variant] = _run(tf, clip, params)
                outs[variant, "bf16"] = _run(_tf(kw, out_dtype=torch.bfloat16), clip, params)
        finally:
            L.nexar_set_geometry_kernel(0)
        assert np.abs(outs[0] - outs[1]).max() <= 2e-6, k        # same formulas; one fused multiply-add differs
        assert np.abs(outs[0, "bf16"] - outs[1, "bf16"]).max() <= 2.0 ** -6, k   # at most one bf16 ulp at |v| < 4
        want = O.apply_clip_transform(clip.transpose(3, 0, 1, 2), cfg, {"flip": params["flip"], "aug": params["aug"]})
        err = float(np.abs(outs[0] - want).max())
        assert err <= TOL_AFTER, (k, err)


def test_result_does_not_depend_on_the_chunking():
    """nexar_set_chunk_clips processes a batch in groups of whole clips with separate workspace slices: bit-identical."""
    from vision_collision_detection_b200 import _lib
    from vision_collision_detection_b200.synth import make_clip_np
    kw = dict(mode="train", crop_size=224, enable_custom_augmentation=True, brightness_range=(0.9, 1.1),
              contrast_range=(0.9, 1.1), saturation_range=(0.9, 1.1), rotation_range=(-5, 5))
    tf = _tf(kw, out_dtype=torch.bfloat16)
    frames = torch.from_numpy(np.stack([make_clip_np(3, 720, 1280, 40 + i, "dashcam") for i in range(5)])).cuda()
    frames[3] = frames[3] & 1                       # one clip whose maximum is 1: the fix-up path inside a chunk
    random.seed(77)
    params = tf.sample_params(5, 720, 1280)
    L = _lib.lib()
    outs = []
    try:
        for chunk in (0, 1, 2, 4):
            L.nexar_set_chunk_clips(chunk)
            outs.append(tf.forward_batch(frames, params=params).float().cpu().numpy())
    finally:
        L.nexar_set_chunk_clips(0)
    for o in outs[1:]:
        assert np.array_equal(o, outs[0])
