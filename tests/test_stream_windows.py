"""Streaming sliding windows (inference.WindowStream, WindowPredictor.predict_stream, nexar_gather_windows_ring and the
NEXAR_RANGE_255 clip flag).  The contract: for any chunking, everything push() and finish() return, concatenated, is
SlidingWindowTransform.windows(video, materialize=True) bit for bit, with sliding_window_starts as starts."""
import ctypes as C
import random

import numpy as np
import pytest
import torch

from vision_collision_detection_b200.inference import ring_schedule, sliding_window_starts, windows_complete

gpu = pytest.mark.gpu
_INT = {torch.float32: torch.int32, torch.bfloat16: torch.int16, torch.float16: torch.int16}


def _sizes(kind, n, seed=0):
    """Chunk sizes covering n frames: an int is a fixed size, "random" seeded sizes from 1 to 150."""
    if kind == "random":
        rng = random.Random(seed)
        out = []
        while sum(out) < n:
            out.append(rng.randint(1, 150))
    else:
        out = [kind] * (n // kind + 1)
    sizes, left = [], n
    for s in out:
        if left <= 0:
            break
        sizes.append(min(s, left))
        left -= sizes[-1]
    return sizes


# ---- the window bookkeeping, on the host -------------------------------------------------------------------------------
@pytest.mark.parametrize("window,stride,max_chunk", [(16, 8, 64), (16, 16, 4), (4, 7, 3), (8, 1, 1), (1, 1, 5), (16, 3, 16)])
def test_ring_schedule_reads_only_frames_still_in_the_ring(window, stride, max_chunk):
    """Simulates the ring with frame numbers: every slot a gather reads holds the frame the window wants, the windows
    come out in order, and they are the offline ones (the padded window of a short video included)."""
    ring_frames = window - 1 + max_chunk
    for n_frames in (1, window - 1, window, window + 1, 3 * ring_frames + 5, 257):
        if n_frames < 1:
            continue
        for kind in (1, 7, stride, window, max_chunk + 3, "random"):
            ring = np.full(ring_frames, -1, np.int64)
            seen, got = 0, []
            for n in _sizes(kind, n_frames, seed=n_frames):
                for lo, hi, writes, k0, k1 in ring_schedule(seen, n, window, stride, max_chunk):
                    assert hi - lo <= max_chunk and sum(w[2] for w in writes) == hi - lo and len(writes) <= 2
                    for slot, offset, count in writes:
                        assert slot + count <= ring_frames
                        ring[slot:slot + count] = np.arange(seen + offset, seen + offset + count)
                    assert k0 == windows_complete(seen + lo, window, stride) and k0 == len(got)
                    last = seen + hi - 1
                    for k in range(k0, k1):                 # the formula of nexar_gather_windows_ring
                        f = np.minimum(k * stride + np.arange(window), last)
                        assert np.array_equal(ring[f % ring_frames], f)
                        got.append(k * stride)
                seen += n
            if seen < window:                               # finish(): one padded window of the first `seen` frames
                assert not got and np.array_equal(ring[np.minimum(np.arange(window), seen - 1) % ring_frames],
                                                  np.minimum(np.arange(window), seen - 1))
                got = [0]
            assert got == sliding_window_starts(n_frames, window, stride), (n_frames, kind)


def test_gather_windows_ring_refuses_bad_arguments():
    from vision_collision_detection_b200 import _lib
    L = _lib.ring_lib()
    buf = C.c_void_p(16)           # never dereferenced: every call below fails its argument checks on the host

    def call(ring=buf, ring_frames=8, plane_bytes=64, window=4, stride=2, first=0, last=7, n=1, dst=buf):
        return L.nexar_gather_windows_ring(ring, ring_frames, plane_bytes, window, stride, first, last, n, dst, None)

    for kw in (dict(ring=None), dict(dst=None), dict(ring_frames=0), dict(plane_bytes=0), dict(window=0), dict(stride=0),
               dict(n=0), dict(first=-1), dict(first=5, last=4), dict(window=9, last=20),      # 9 frames in 8 slots
               dict(n=4, stride=2, window=4, first=3, last=100)):                                 # frames 3..12
        assert call(**kw) == _lib.ERR_INVALID, kw
    assert "gather_windows_ring" in L.nexar_last_error().decode()
    assert _lib.lib().nexar_gather_windows(buf, 0, 64, 4, 2, 1, buf, None) == _lib.ERR_INVALID


def test_stream_argument_errors_on_the_host():
    from vision_collision_detection_b200.inference import WindowStream
    with pytest.raises(ValueError):
        WindowStream(window=0)
    with pytest.raises(ValueError):
        WindowStream(max_chunk=0)
    ws = WindowStream(window=4, stride=2)
    with pytest.raises(TypeError):                          # decoders deliver uint8 or YUV surfaces
        ws.push(torch.zeros((3, 8, 8, 3), dtype=torch.float32))
    with pytest.raises(ValueError):
        ws.push(torch.zeros((3, 8, 8), dtype=torch.uint8))                       # RGB needs [n,H,W,3]
    with pytest.raises(ValueError):
        ws.push(torch.zeros((3, 12, 8, 3), dtype=torch.uint8), pixel_format="nv12")   # YUV needs [n,R,P]
    with pytest.raises(ValueError):
        ws.push(torch.zeros((0, 8, 8, 3), dtype=torch.uint8))
    with pytest.raises(ValueError):                         # a stream with no frames has no windows
        ws.finish()


# ---- on the device ------------------------------------------------------------------------------------------------------
def _video(n, seed=5, h=48, w=80):
    from vision_collision_detection_b200.synth import make_clip_torch
    return make_clip_torch(n, h, w, seed, "dashcam")


def _run_stream(ws, video, sizes, **fmt):
    starts, wins, lo = [], [], 0
    for n in sizes:
        s, w = ws.push(video[lo:lo + n], **fmt)
        assert w.is_contiguous() and w.shape[0] == len(s)
        starts += s
        wins.append(w)
        lo += n
    assert lo == video.shape[0]
    s, w = ws.finish()
    return starts + s, torch.cat(wins + [w])


def _offline(tf, video, window=16, stride=8, out_dtype=torch.bfloat16, **fmt):
    from vision_collision_detection_b200.inference import SlidingWindowTransform
    return SlidingWindowTransform(window, stride, tf, out_dtype).windows(video, materialize=True, **fmt)


def _same_bits(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(a.view(_INT[a.dtype]), b.view(_INT[b.dtype]))


@gpu
@pytest.mark.parametrize("n_frames", [5, 15, 16, 17, 100, 1200])
@pytest.mark.parametrize("chunk", [1, 7, 8, 16, 100, "random"])
def test_stream_equals_offline_windows(n_frames, chunk):
    """Video lengths around the window, chunks of 1, 7, the stride, the window, more than max_chunk and random sizes."""
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.inference import WindowStream
    video = _video(n_frames)
    tf = create_video_transforms(mode="val", crop_size=56)
    want = _offline(tf, video)
    ws = WindowStream(16, 8, tf, max_chunk=64)
    starts, got = _run_stream(ws, video, _sizes(chunk, n_frames, seed=n_frames))
    assert starts == sliding_window_starts(n_frames, 16, 8)
    assert _same_bits(got, want)


@gpu
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_stream_wraps_the_ring_many_times(out_dtype):
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.inference import WindowStream
    video = _video(1200, seed=9)
    tf = create_video_transforms(mode="val", crop_size=56)
    ws = WindowStream(16, 4, tf, out_dtype=out_dtype, max_chunk=8)
    assert 1200 // ws.ring_frames >= 10
    starts, got = _run_stream(ws, video, _sizes("random", 1200, seed=3))
    assert starts == sliding_window_starts(1200, 16, 4)
    assert _same_bits(got, _offline(tf, video, 16, 4, out_dtype))


@gpu
@pytest.mark.parametrize("fmt", ["nv12", "i420_bt709", "p010"])
def test_stream_of_yuv_surfaces(fmt):
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.inference import WindowStream
    from vision_collision_detection_b200.synth import make_clip_np, rgb_to_yuv420, rgb_to_yuv420_16
    rgb = make_clip_np(90, 48, 80, 4, "dashcam")
    if fmt == "nv12":
        surf, kw = rgb_to_yuv420(rgb, "nv12"), dict(pixel_format="nv12")
    elif fmt == "i420_bt709":
        surf, kw = rgb_to_yuv420(rgb, "i420", "bt709"), dict(pixel_format="i420", color_matrix="bt709")
    else:
        surf, kw = rgb_to_yuv420_16(rgb, "p010"), dict(pixel_format="p010")
    video = torch.from_numpy(surf).cuda()
    tf = create_video_transforms(mode="val", crop_size=56)
    want = _offline(tf, video, **kw)
    starts, got = _run_stream(WindowStream(16, 8, tf, max_chunk=32), video, _sizes(13, 90), **kw)
    assert starts == sliding_window_starts(90, 16, 8) and _same_bits(got, want)


@gpu
@pytest.mark.parametrize("where", ["pageable", "pinned"])
def test_host_chunks_equal_device_chunks(where):
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.inference import WindowStream
    video = _video(150, seed=11)
    host = video.cpu()
    if where == "pinned":
        host = host.pin_memory()
    tf = create_video_transforms(mode="val", crop_size=56)
    dev_starts, dev_wins = _run_stream(WindowStream(16, 8, tf, max_chunk=32), video, _sizes("random", 150, seed=1))
    host_starts, host_wins = _run_stream(WindowStream(16, 8, tf, max_chunk=32), host, _sizes("random", 150, seed=2))
    assert host_starts == dev_starts and _same_bits(host_wins, dev_wins)
    assert _same_bits(host_wins, _offline(tf, video))


@gpu
def test_stream_with_custom_augmentation_and_two_pass_transforms():
    """The record is drawn once, on the first push, exactly as frames() draws it: same `random` seed, same windows.  The
    two-pass factory scales the bytes in its first pass only."""
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.inference import WindowStream
    from vision_collision_detection_b200.video_aug import create_video_transform
    video = _video(70, seed=13)
    aug = create_video_transforms(mode="train", crop_size=56, enable_custom_augmentation=True, brightness_range=(0.8, 1.2),
                                  contrast_range=(0.8, 1.2), saturation_range=(0.8, 1.2), hue_range=(-0.1, 0.1),
                                  rotation_range=(-10, 10), horizontal_flip_prob=0.5, cutout_prob=1.0, blur_sigma=0.8,
                                  grayscale_prob=0.3)
    two_pass = create_video_transform(mode="val", min_size=64, crop_size=56)
    for tf in (aug, two_pass):
        for seed in (1, 2, 3):
            random.seed(seed)
            want = _offline(tf, video, out_dtype=torch.float32)
            random.seed(seed)
            starts, got = _run_stream(WindowStream(16, 8, tf, out_dtype=torch.float32, max_chunk=16), video,
                                      _sizes("random", 70, seed=seed))
            assert starts == sliding_window_starts(70, 16, 8) and _same_bits(got, want), (tf.mode, seed)


def _bright_with_dark_run(n, lo, hi, h, w, seed):
    """A video whose frames lo..hi-1 hold only 0 and 1 (near-black frames): the rest is a synthetic dashcam video."""
    video = _video(n, seed, h, w)
    g = torch.Generator(device="cuda").manual_seed(seed)
    video[lo:hi] = torch.randint(0, 2, video[lo:hi].shape, generator=g, device="cuda", dtype=torch.uint8)
    return video


@gpu
def test_stream_scales_a_chunk_of_zeros_and_ones_like_the_whole_video():
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.inference import WindowStream
    video = _bright_with_dark_run(60, 20, 28, 48, 80, 3)
    tf = create_video_transforms(mode="val", crop_size=56)
    starts, got = _run_stream(WindowStream(16, 8, tf), video, [20, 8, 32])       # the dark run is a chunk of its own
    assert starts == sliding_window_starts(60, 16, 8) and _same_bits(got, _offline(tf, video))


@gpu
@pytest.mark.parametrize("path", ["fast", "general", "clip_max", "fast_aug"])
def test_range_255_flag_in_every_kernel_that_decides_the_scale(path):
    """A clip of 0 / 1 frames with NEXAR_RANGE_255 gives those frames' result inside a bright clip; without it the
    clip is left unscaled.  The fast resize kernel (720p letterbox), the general one, clip_max_kernel (crop geometry)
    and the augmented launch sequence behind the fast kernel."""
    from vision_collision_detection_b200 import _lib, create_video_transforms
    from vision_collision_detection_b200.video_aug import create_video_transform
    if path in ("fast", "fast_aug"):
        video, cs = _bright_with_dark_run(6, 2, 5, 720, 1280, 7), 224
    else:
        video, cs = _bright_with_dark_run(6, 2, 5, 48, 80, 7), 56
    if path == "clip_max":
        tf = create_video_transform(mode="val", min_size=64, crop_size=cs, use_letterbox=False)
    elif path == "fast_aug":
        tf = create_video_transforms(mode="train", crop_size=cs, enable_custom_augmentation=True,
                                     brightness_range=(0.9, 1.1), contrast_range=(0.9, 1.1), rotation_range=(-5, 5))
    else:
        tf = create_video_transforms(mode="val", crop_size=cs)
    random.seed(0)
    rec = tf.sample_params(1, video.shape[1], video.shape[2])[0]
    if path == "general":
        _lib.check(_lib.lib().nexar_set_resize_kernel(1))
    try:
        whole = tf.forward_batch(video[None], params=[rec])[0, :, 2:5]
        flagged = tf.forward_batch(video[None, 2:5], params=[dict(rec, range_255=True)])[0]
        plain = tf.forward_batch(video[None, 2:5], params=[rec])[0]
    finally:
        _lib.check(_lib.lib().nexar_set_resize_kernel(0))
    assert _same_bits(flagged, whole)
    assert not torch.equal(plain, whole)


@gpu
def test_seventy_thousand_frames_run_to_the_end():
    """Longer than one nexar_clip_transform call can take (65535 frames): windows along the way, across that mark
    included, equal the offline windows of their own frames."""
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.inference import SlidingWindowTransform, WindowStream
    n_frames, period = 70000, 997                          # frame f is base[f % period]: windows straddle the repeats
    base = _video(period, seed=21, h=24, w=32)
    tf = create_video_transforms(mode="val", crop_size=16)
    ws = WindowStream(16, 8, tf)
    n_windows = windows_complete(n_frames, 16, 8)
    check = {0, 1, 124, 125, n_windows // 2, 65535 // 8 - 1, 65535 // 8, n_windows - 1}
    kept, seen, count = {}, 0, 0
    while seen < n_frames:
        n = min(250, n_frames - seen)
        idx = torch.arange(seen, seen + n, device="cuda") % period
        starts, wins = ws.push(base[idx])
        for i, s in enumerate(starts):
            assert s == (count + i) * 8
            if count + i in check:
                kept[count + i] = wins[i].clone()
        count += len(starts)
        seen += n
    assert ws.finish()[0] == [] and count == n_windows and set(kept) == check
    one = SlidingWindowTransform(16, 16, tf)
    for k, got in kept.items():
        idx = torch.arange(k * 8, k * 8 + 16, device="cuda") % period
        assert _same_bits(got, one.windows(base[idx], materialize=True)[0]), k


@gpu
def test_device_memory_does_not_grow_with_the_video():
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.inference import WindowStream
    video = _video(2400, seed=2, h=96, w=160)
    tf = create_video_transforms(mode="val", crop_size=112)

    def peak(n):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        ws = WindowStream(16, 8, tf)
        for lo in range(0, n, 30):
            starts, wins = ws.push(video[lo:lo + 30])
        ws.finish()
        del ws, starts, wins
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base

    peak(2400)        # the engine's plans, workspace and frame-offset tables (one per chunk split): allocated once, kept
    short, long = peak(600), peak(2400)
    assert short == long and short > 0


@gpu
@pytest.mark.parametrize("n_frames", [10, 70, 203])
def test_predict_stream_equals_predict(n_frames):
    from vision_collision_detection_b200.inference import WindowPredictor
    video = _video(n_frames, seed=23, h=96, w=160)
    w_mat = torch.tensor([[1.0, -2.0, 0.5], [-0.3, 0.8, 1.1], [0.2, 0.1, -0.9]], device="cuda")
    calls = []

    def model(x):                                          # [b,3,T,cs,cs] -> logits [b,3]
        assert x.is_contiguous() and x.shape[1:3] == (3, 16)
        calls.append(x.shape[0])
        return x.float().mean(dim=(2, 3, 4)) @ w_mat

    wp = WindowPredictor(model, window=16, stride=8, batch_size=3)
    want = wp.predict(video, video_path="drive.mp4", fps=25.0)
    want_calls, calls[:] = list(calls), []
    chunks = (video[lo:lo + n] for lo, n in zip(np.cumsum([0] + _sizes("random", n_frames, seed=7)),
                                                 _sizes("random", n_frames, seed=7)))
    got = list(wp.predict_stream(chunks, video_path="drive.mp4", fps=25.0))
    assert calls == want_calls and got == want


@gpu
@pytest.mark.parametrize("plane_bytes", [4096, 3 * 224 * 224 * 2 // 3, 50, 7, 32768])
def test_gather_windows_ring_against_torch_indexing(plane_bytes):
    """Random bytes: planes that are and are not multiples of 16, a first frame just before the wrap, the last_frame
    clamp, and unaligned ring / destination pointers (the byte path)."""
    from vision_collision_detection_b200 import _lib
    L = _lib.ring_lib()
    ring_frames, window, stride = 23, 5, 3
    g = torch.Generator(device="cuda").manual_seed(plane_bytes)
    raw = torch.randint(0, 256, (ring_frames * 3 * plane_bytes + 16,), generator=g, device="cuda", dtype=torch.uint8)
    for shift in (0, 1):
        ring = raw[shift:shift + ring_frames * 3 * plane_bytes].view(ring_frames, 3, plane_bytes)
        for first, last, n in ((20, 20 + 2 * 3 + 4, 3), (44, 50, 4), (0, 22, 7), (5, 5, 2), (1000, 1013, 4)):
            k = torch.arange(n).view(n, 1)
            f = torch.clamp(first + k * stride + torch.arange(window).view(1, window), max=last) % ring_frames
            want = ring[f.cuda()].permute(0, 2, 1, 3)                     # [n,window,3,pb] -> [n,3,window,pb]
            dst = torch.full((n * 3 * window * plane_bytes + 16,), 7, dtype=torch.uint8, device="cuda")
            out = dst[shift:shift + n * 3 * window * plane_bytes]
            _lib.check(L.nexar_gather_windows_ring(ring.data_ptr(), ring_frames, plane_bytes, window, stride, first, last, n,
                                                   out.data_ptr(), torch.cuda.current_stream().cuda_stream))
            assert torch.equal(out.view(n, 3, window, plane_bytes), want), (shift, first, last, n)
            assert torch.all(dst[:shift] == 7) and torch.all(dst[shift + out.numel():] == 7)


@gpu
def test_stream_errors_on_the_device():
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.inference import WindowStream
    from vision_collision_detection_b200.synth import rgb_to_nv12
    video = _video(20)
    tf = create_video_transforms(mode="val", crop_size=56)
    ws = WindowStream(16, 8, tf)
    ws.push(video[:5])
    with pytest.raises(ValueError):
        ws.push(_video(5, h=64, w=80))                                     # frame geometry changes
    with pytest.raises(ValueError):
        ws.push(rgb_to_nv12(video[:4]), pixel_format="nv12")               # source format changes
    with pytest.raises(TypeError):
        ws.push(video[5:9].float())
    assert ws.push(video[5:20])[0] == [0]
    assert ws.finish()[0] == []
    with pytest.raises(ValueError):
        ws.push(video[:4])
    with pytest.raises(ValueError):
        ws.finish()
    short = WindowStream(16, 8, tf)
    short.push(video[:3])
    starts, win = short.finish()
    assert starts == [0] and _same_bits(win, _offline(tf, video[:3]))


@gpu
def test_stream_refused_first_chunk_leaves_it_unopened():
    """A first chunk the stream refuses (13 rows are no 4:2:0 surface) opens nothing: a correct video pushed next gets the
    offline windows."""
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.inference import WindowStream
    video = _video(40)
    tf = create_video_transforms(mode="val", crop_size=56)
    ws = WindowStream(16, 8, tf)
    with pytest.raises(ValueError):
        ws.push(torch.zeros((3, 13, 8), dtype=torch.uint8, device="cuda"), pixel_format="nv12")
    starts, got = _run_stream(ws, video, [7, 33])
    assert starts == sliding_window_starts(40, 16, 8)
    assert _same_bits(got, _offline(tf, video))
