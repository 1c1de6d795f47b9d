"""Many streams in one pool (inference.MultiWindowStream, WindowPredictor.predict_step, nexar_gather_windows_table).  The
contract: every stream's windows, across all steps, are WindowStream's on the same chunks, bit for bit."""
import ctypes as C
import random

import numpy as np
import pytest
import torch

from vision_collision_detection_b200.inference import multi_stream_schedule, sliding_window_starts

gpu = pytest.mark.gpu
_INT = {torch.float32: torch.int32, torch.bfloat16: torch.int16, torch.float16: torch.int16}


# ---- the bookkeeping, on the host ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("window,stride,step_frames", [(16, 8, 64), (16, 16, 7), (4, 7, 3), (8, 1, 200), (1, 1, 5),
                                                       (16, 3, 1024), (2, 5, 1)])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_schedule_reads_only_the_frames_each_window_wants(window, stride, step_frames, seed):
    """Random interleavings of open, push (1 to 200 frames), step, close and reopen over many streams, simulated with
    frame ids in the pool: every gather entry names a slot holding the frame its window wants (so no tail copy
    overwrote a slot a later window of the step reads), copies go from step slots to the video's own tail slots, every
    closed video ends exactly once (its slots come free), the pool stays in its bound, and each video's windows are
    the offline ones."""
    rng = random.Random(seed * 1000 + window * 10 + stride)
    tail_len = window - 1
    pool = {}                                  # slot -> (video uid, frame)
    videos = {}                                # uid -> dict(seen, tail, closed, pushed, starts)
    free, n_tails, max_open = [], 0, 0
    open_by_key, queue, uid = {}, [], 0
    finished = []

    def open_video():
        nonlocal uid, n_tails
        if not free:
            free.append(n_tails)
            n_tails += 1
        block = free.pop()
        videos[uid] = dict(seen=0, block=block, tail=step_frames + block * tail_len, closed=False, pushed=0, starts=[])
        uid += 1
        return uid - 1

    def step():
        order = list(videos)               # open order (dict insertion)
        pos = {u: i for i, u in enumerate(order)}
        rounds = multi_stream_schedule([(videos[u]["seen"], videos[u]["tail"], videos[u]["closed"]) for u in order],
                                       [(pos[u], n, videos[u]["tail"] % 3) for u, n in queue], window, stride, step_frames)
        q_first = {i: videos[u]["pushed_before"][i] for i, (u, n) in enumerate(queue)}
        for rnd in rounds:
            assert sum(hi - lo for _, lo, hi, _ in rnd.pieces) <= step_frames
            for g, p0, p1 in rnd.groups:       # a group's frames fill a contiguous run of step slots
                run = [s + i for _, lo, hi, s in rnd.pieces[p0:p1] for i in range(hi - lo)]
                assert run == list(range(run[0], run[0] + len(run))) if run else True
            for q, lo, hi, slot in rnd.pieces:
                u = queue[q][0]
                for i in range(hi - lo):
                    assert 0 <= slot + i < step_frames
                    pool[slot + i] = (u, q_first[q] + lo + i)
            for q, lo, hi, _ in rnd.pieces:
                videos[queue[q][0]]["seen_round"] = videos[queue[q][0]].get("seen_round", 0) + hi - lo
            table = rnd.gather.reshape(len(rnd.windows), window) if rnd.windows else np.zeros((0, window), int)
            for (v, start), row in zip(rnd.windows, table):
                u = order[v]
                last = videos[u]["seen"] + videos[u].get("seen_round", 0) - 1
                want = [(u, min(start + t, last)) for t in range(window)]
                assert [pool.get(int(s)) for s in row] == want, (u, start)
                videos[u]["starts"].append(start)
            assert sorted(rnd.windows) == list(rnd.windows)
            assert rnd.copy_src.size == rnd.copy_dst.size and len(set(rnd.copy_dst.tolist())) == rnd.copy_dst.size
            for s, d in zip(rnd.copy_src.tolist(), rnd.copy_dst.tolist()):
                u = pool[s][0]
                assert s < step_frames and videos[u]["tail"] <= d < videos[u]["tail"] + tail_len
            for s, d in zip(rnd.copy_src.tolist(), rnd.copy_dst.tolist()):
                pool[d] = pool[s]
            for u in order:
                if u in videos:
                    videos[u]["seen"] += videos[u].pop("seen_round", 0)
            for v in rnd.done:
                u = order[v]
                assert videos[u]["closed"] and videos[u]["seen"] == videos[u]["pushed"]
                finished.append((u, videos[u]))
                free.append(videos.pop(u)["block"])
        queue.clear()
        for u in list(videos):
            videos[u]["pushed_before"] = {}

    for i in range(400):
        op = rng.random()
        if op < 0.55:
            key = rng.randrange(12)
            u = open_by_key.get(key)
            if u is None:
                u = open_by_key[key] = open_video()
                videos[u]["pushed_before"] = {}
            n = rng.choice([1, 1, 2, rng.randint(1, 30), rng.randint(1, 200)])
            videos[u]["pushed_before"][len(queue)] = videos[u]["pushed"]
            queue.append((u, n))
            videos[u]["pushed"] += n
        elif op < 0.8:
            step()
        elif open_by_key:
            key = rng.choice(sorted(open_by_key))
            videos[open_by_key.pop(key)]["closed"] = True
        max_open = max(max_open, len(videos))
        assert all(s < step_frames + max_open * tail_len for s in pool)
    for key in list(open_by_key):
        videos[open_by_key.pop(key)]["closed"] = True
    step()
    assert not videos and sorted(free) == list(range(n_tails))        # every slot back on the free list
    assert finished
    for u, v in finished:
        assert v["starts"] == sliding_window_starts(v["pushed"], window, stride), u


def test_schedule_splits_a_step_into_rounds_in_push_order():
    rounds = multi_stream_schedule([(0, 10, False), (0, 25, False)], [(0, 5, "a"), (1, 4, "b"), (0, 3, "a")], 16, 8, 4)
    assert [[(q, lo, hi) for q, lo, hi, _ in r.pieces] for r in rounds] == \
        [[(0, 0, 4)], [(0, 4, 5), (1, 0, 3)], [(1, 3, 4), (2, 0, 3)]]   # groups in order of first appearance
    assert [r.pieces[0][3] for r in rounds] == [0, 0, 0]
    one = multi_stream_schedule([(0, 10, False), (0, 25, False)], [(0, 5, "a"), (1, 4, "b"), (0, 3, "a")], 16, 8, 64)
    assert len(one) == 1 and [g[0] for g in one[0].groups] == ["a", "b"]
    assert [(q, s) for q, _, _, s in one[0].pieces] == [(0, 0), (2, 5), (1, 8)]      # grouped: 'a' frames first


def test_empty_and_close_only_steps():
    assert [r.windows for r in multi_stream_schedule([], [], 16, 8, 64)] == [[]]
    (rnd,) = multi_stream_schedule([(3, 20, True), (40, 35, True)], [], 16, 8, 64)
    assert rnd.windows == [(0, 0)] and rnd.done == [0, 1] and rnd.copy_src.size == 0
    assert rnd.gather.tolist() == [20, 21, 22] + [22] * 13       # the padded window: frame 2 repeated, from the tail


def test_multi_stream_argument_errors_on_the_host():
    from vision_collision_detection_b200.inference import MultiWindowStream
    for kw in (dict(window=0), dict(stride=0), dict(max_frames_per_step=0)):
        with pytest.raises(ValueError):
            MultiWindowStream(**kw)
    ms = MultiWindowStream(window=4, stride=2)
    with pytest.raises(TypeError):
        ms.push("a", torch.zeros((3, 8, 8, 3), dtype=torch.float32))
    with pytest.raises(ValueError):
        ms.push("a", torch.zeros((3, 8, 8), dtype=torch.uint8))
    with pytest.raises(ValueError):
        ms.push("a", torch.zeros((0, 8, 8, 3), dtype=torch.uint8))
    with pytest.raises(ValueError):
        ms.push("a", torch.zeros((2, 8, 8, 3), dtype=torch.uint8), frame_size=(8, 8))      # RGB has no padding
    with pytest.raises(ValueError):
        ms.push("a", torch.zeros((2, 13, 8), dtype=torch.uint8), pixel_format="nv12")      # not a 4:2:0 surface
    with pytest.raises(ValueError):
        ms.close("never opened")


# ---- on the device ------------------------------------------------------------------------------------------------------
def _video(n, seed=5, h=48, w=80):
    from vision_collision_detection_b200.synth import make_clip_torch
    return make_clip_torch(n, h, w, seed, "dashcam")


def _same_bits(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(a.view(_INT[a.dtype]), b.view(_INT[b.dtype]))


def _collect(got, keys, starts, wins):
    for i, (k, s) in enumerate(zip(keys, starts)):
        got.setdefault(k, ([], []))
        got[k][0].append(s)
        got[k][1].append(wins[i:i + 1])


def _reference(tf, chunks, window=16, stride=8, out_dtype=torch.bfloat16, **fmt):
    """WindowStream fed the same chunks -> (starts, windows)."""
    from vision_collision_detection_b200.inference import WindowStream
    ws = WindowStream(window, stride, tf, out_dtype=out_dtype)
    starts, wins = [], []
    for c in chunks:
        s, w = ws.push(c, **fmt)
        starts += s
        wins.append(w)
    s, w = ws.finish()
    return starts + s, torch.cat(wins + [w])


def _check_against_window_stream(tf, got, log, window=16, stride=8, out_dtype=torch.bfloat16):
    """``log[key]`` = (chunks, source format) of each finished video under that key."""
    for key, (chunks, fmt) in log.items():
        want_s, want_w = _reference(tf, chunks, window, stride, out_dtype, **fmt)
        starts, wins = got.pop(key)
        assert starts == want_s, key
        assert _same_bits(torch.cat(wins), want_w), key
    assert not got


@gpu
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_many_streams_equal_window_stream(seed):
    """1 to 64 streams of 5 to 1200 frames, random chunk sizes, push order and step points; streams open and close mid-
    run and later ones reuse their slots."""
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.inference import MultiWindowStream
    rng = random.Random(seed)
    tf = create_video_transforms(mode="val", crop_size=32)
    n_videos = [1, 16, 64][seed]
    lengths = [rng.choice([5, 15, 16, 17, rng.randint(5, 300), 1200 if rng.random() < 0.1 else 60])
               for _ in range(n_videos + n_videos // 2)]
    bank = _video(1200, seed=seed, h=40, w=64)
    ms = MultiWindowStream(16, 8, tf, max_frames_per_step=rng.choice([64, 1024]))
    pending = list(range(len(lengths)))       # videos not yet started; at most n_videos run at a time
    running, log, got = {}, {}, {}
    while pending or running:
        while pending and len(running) < n_videos and rng.random() < 0.7:
            v = pending.pop()
            off = rng.randint(0, 1200 - lengths[v])
            running[f"cam{v}"] = [bank[off:off + lengths[v]], 0, []]
        for key in rng.sample(sorted(running), len(running)):
            video, at, chunks = running[key]
            if at < video.shape[0] and rng.random() < 0.8:
                n = min(video.shape[0] - at, rng.choice([1, 1, 3, rng.randint(1, 40)]))
                ms.push(key, video[at:at + n])
                chunks.append(video[at:at + n])
                running[key][1] = at + n
            elif at == video.shape[0]:
                ms.close(key)
                log[key] = (chunks, {})
                del running[key]
        if rng.random() < 0.6:
            _collect(got, *ms.step())
    _collect(got, *ms.step())
    assert ms._pool is None
    _check_against_window_stream(tf, got, log)


@gpu
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_one_step_of_mixed_sources(out_dtype):
    """RGB 720p and RGB of another size, NV12, I420 BT.709 full range, P010 in padded 1088-row surfaces and I010, on the
    device, in pageable and in pinned host memory, in the same steps."""
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.inference import MultiWindowStream
    from vision_collision_detection_b200.synth import make_clip_np, rgb_to_yuv420, rgb_to_yuv420_16
    tf = create_video_transforms(mode="val", crop_size=64)
    n = 20
    small = make_clip_np(n, 48, 80, 1, "dashcam")
    big = _video(n, seed=2, h=720, w=1280).cpu().numpy()
    hd = _video(n, seed=3, h=1080, w=1920).cpu().numpy()
    # 1088-row surfaces with 1080 visible rows, 10-bit words widened from the 8-bit samples (x << 8)
    p010 = rgb_to_yuv420(hd, "nv12", luma_rows=1088).astype(np.uint16) << 8
    sources = {
        "rgb720": (big, {}),
        "rgb_small": (small, {}),
        "nv12": (rgb_to_yuv420(small, "nv12"), dict(pixel_format="nv12")),
        "i420": (rgb_to_yuv420(small, "i420", "bt709", "full"),
                 dict(pixel_format="i420", color_matrix="bt709", color_range="full")),
        "p010": (p010, dict(pixel_format="p010", frame_size=(1080, 1920))),
        "i010": (rgb_to_yuv420_16(small, "i010"), dict(pixel_format="i010")),
    }
    ms = MultiWindowStream(16, 8, tf, out_dtype=out_dtype)
    log, got = {}, {}
    for i, (name, (arr, fmt)) in enumerate(sources.items()):
        for where in ("device", "pageable", "pinned"):
            t = torch.from_numpy(arr)
            t = t.cuda() if where == "device" else (t.pin_memory() if where == "pinned" else t)
            key = (name, where)
            log[key] = ([t[:7], t[7:8], t[8:20]], fmt)
    for part in range(3):
        for key, (chunks, fmt) in log.items():
            ms.push(key, chunks[part], **fmt)
        _collect(got, *ms.step())
    for key in log:
        ms.close(key)
    _collect(got, *ms.step())
    _check_against_window_stream(tf, got, log, out_dtype=out_dtype)


@gpu
def test_augmented_and_two_pass_transforms_draw_what_window_stream_draws():
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.inference import MultiWindowStream
    from vision_collision_detection_b200.video_aug import create_video_transform
    aug = create_video_transforms(mode="train", crop_size=56, enable_custom_augmentation=True, brightness_range=(0.8, 1.2),
                                  contrast_range=(0.8, 1.2), saturation_range=(0.8, 1.2), hue_range=(-0.1, 0.1),
                                  rotation_range=(-10, 10), horizontal_flip_prob=0.5, cutout_prob=1.0, blur_sigma=0.8,
                                  grayscale_prob=0.3)
    two_pass = create_video_transform(mode="val", min_size=64, crop_size=56)
    videos = {f"cam{i}": _video(30 + 11 * i, seed=40 + i) for i in range(4)}
    for tf in (aug, two_pass):
        random.seed(7)
        ms = MultiWindowStream(16, 8, tf, out_dtype=torch.float32)
        got, log = {}, {}
        for key, v in videos.items():                       # first pushes in this order: the records are drawn so
            ms.push(key, v[:5])
            log[key] = ([v[:5], v[5:]], {})
        for key, v in videos.items():
            ms.push(key, v[5:])
            ms.close(key)
        _collect(got, *ms.step())
        random.seed(7)                                      # ...and WindowStreams opened in the same order draw the same
        from vision_collision_detection_b200.inference import WindowStream
        streams = {key: WindowStream(16, 8, tf, out_dtype=torch.float32) for key in videos}
        for key, v in videos.items():
            streams[key].push(v[:5])
        for key, v in videos.items():
            s, w = streams[key].push(v[5:])
            s2, w2 = streams[key].finish()
            assert got[key][0] == s + s2 and _same_bits(torch.cat(got[key][1]), torch.cat([w, w2])), (tf.mode, key)


@gpu
@pytest.mark.parametrize("n_streams", [1, 16, 256])
def test_launches_per_step_do_not_depend_on_the_number_of_streams(n_streams, monkeypatch):
    from vision_collision_detection_b200 import _lib, create_video_transforms
    from vision_collision_detection_b200.engine import ClipTransformEngine
    from vision_collision_detection_b200.inference import MultiWindowStream
    from vision_collision_detection_b200.synth import rgb_to_nv12
    tf = create_video_transforms(mode="val", crop_size=32)
    runs, gathers = [], []
    real_run = ClipTransformEngine.run
    monkeypatch.setattr(ClipTransformEngine, "run", lambda self, *a, **k: (runs.append(1), real_run(self, *a, **k))[1])
    L = _lib.table_lib()
    real_gather = L.nexar_gather_windows_table

    class Counting:
        def __call__(self, *a):
            gathers.append(a[7] is None)                  # True: a window gather, False: a tail copy
            return real_gather(*a)
    monkeypatch.setattr(L, "nexar_gather_windows_table", Counting())
    rgb = _video(24, seed=3, h=32, w=48)
    nv = rgb_to_nv12(rgb)
    ms = MultiWindowStream(16, 8, tf)
    assert ms.step()[0] == [] and not runs and not gathers      # an empty step launches nothing
    for step in range(24):
        runs.clear(), gathers.clear()
        for s in range(n_streams):
            if s % 2:
                ms.push(s, nv[step:step + 1], pixel_format="nv12")
            else:
                ms.push(s, rgb[step:step + 1])
        keys, starts, wins = ms.step()
        groups = 2 if n_streams > 1 else 1
        assert len(runs) == groups
        complete = step + 1 >= 16 and (step + 1 - 16) % 8 == 0
        assert gathers == ([True] if complete else []) + [False]
        assert len(keys) == (n_streams if complete else 0)
    runs.clear(), gathers.clear()
    assert ms.step()[0] == [] and not runs and not gathers


@gpu
def test_memory_is_bounded_and_returned():
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.inference import MultiWindowStream, WindowStream
    tf = create_video_transforms(mode="val", crop_size=64)
    bank = _video(300, seed=8, h=96, w=160)

    def peak(n_frames, n_streams=8):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        ms = MultiWindowStream(16, 8, tf, max_frames_per_step=64)
        for lo in range(0, n_frames, 6):
            for s in range(n_streams):
                ms.push(s, bank[(lo + s) % 294:(lo + s) % 294 + 6])
            keys, starts, wins = ms.step()
        for s in range(n_streams):
            ms.close(s)
        ms.step()
        del keys, starts, wins
        torch.cuda.synchronize()
        after = torch.cuda.memory_allocated() - base
        return torch.cuda.max_memory_allocated() - base, after, ms

    peak(2400)
    (short, after_short, _), (long, after_long, ms) = peak(600), peak(2400)
    assert short == long and short > 0 and after_short == after_long == 0
    ms.push("again", bank[:40])                              # a reopened stream equals a fresh WindowStream
    ms.close("again")
    keys, starts, wins = ms.step()
    want_s, want_w = _reference(tf, [bank[:40]])
    assert keys == ["again"] * len(want_s) and starts == want_s and _same_bits(wins, want_w)


@gpu
def test_short_videos_and_rounds():
    """Videos shorter than the window get their padded window from close(); a max_frames_per_step smaller than what is
    queued gives what one big step gives."""
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.inference import MultiWindowStream
    tf = create_video_transforms(mode="val", crop_size=32)
    videos = {k: _video(n, seed=n) for k, n in (("a", 3), ("b", 15), ("c", 16), ("d", 90), ("e", 1), ("f", 41))}
    results = []
    for max_frames in (1024, 7, 1):
        ms = MultiWindowStream(16, 8, tf, max_frames_per_step=max_frames)
        for lo in range(0, 90, 30):
            for k, v in videos.items():
                if lo < v.shape[0]:
                    ms.push(k, v[lo:lo + 30])
        for k in videos:
            ms.close(k)
        results.append(ms.step())
    (k0, s0, w0) = results[0]
    for keys, starts, wins in results[1:]:
        assert keys == k0 and starts == s0 and _same_bits(wins, w0)
    got = {}
    _collect(got, k0, s0, w0)
    assert list(dict.fromkeys(k0)) == list(videos)           # grouped by stream, in opening order
    _check_against_window_stream(tf, got, {k: ([v[lo:lo + 30] for lo in range(0, v.shape[0], 30)], {})
                                           for k, v in videos.items()})


@gpu
def test_stream_errors_on_the_device():
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.inference import MultiWindowStream
    from vision_collision_detection_b200.synth import rgb_to_nv12
    tf = create_video_transforms(mode="val", crop_size=32)
    video = _video(20)
    ms = MultiWindowStream(16, 8, tf)
    ms.push("a", video[:5])
    with pytest.raises(ValueError):
        ms.push("a", _video(5, h=64, w=80))                              # frame geometry changes
    with pytest.raises(ValueError):
        ms.push("a", rgb_to_nv12(video[:4]), pixel_format="nv12")        # source format changes
    with pytest.raises(ValueError):
        ms.push("b", torch.empty((4, 48, 80, 3), dtype=torch.uint16, device="cuda"))   # RGB frames are uint8
    ms.push("b", rgb_to_nv12(video[:4]), pixel_format="nv12")          # another stream, another format
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            ms.push("c", video[:4].to("cuda:1"))
    ms.close("a")
    with pytest.raises(ValueError):
        ms.close("a")
    keys, starts, wins = ms.step()
    assert keys == ["a"] and starts == [0]


@gpu
@pytest.mark.parametrize("plane_bytes", [4096, 3 * 224 * 224 * 2 // 3, 50, 7, 32768])
def test_gather_windows_table_against_torch_indexing(plane_bytes):
    """Random tables with repeated and out-of-range slots (clamped), planes that are and are not multiples of 16,
    unaligned pointers (the byte path), a split plane (32768 bytes, few windows) and the dst_slots copy."""
    from vision_collision_detection_b200 import _lib
    L = _lib.table_lib()
    pool_frames, window = 23, 5
    g = torch.Generator(device="cuda").manual_seed(plane_bytes)
    stream = torch.cuda.current_stream().cuda_stream
    raw = torch.randint(0, 256, (pool_frames * 3 * plane_bytes + 16,), generator=g, device="cuda", dtype=torch.uint8)
    for shift in (0, 1):
        pool = raw[shift:shift + pool_frames * 3 * plane_bytes].view(pool_frames, 3, plane_bytes)
        for n in (1, 3, 40):
            slots = torch.randint(-3, pool_frames + 3, (n * window,), generator=g, device="cuda", dtype=torch.int32)
            want = pool[slots.clamp(0, pool_frames - 1).long()].view(n, window, 3, plane_bytes).permute(0, 2, 1, 3)
            dst = torch.full((n * 3 * window * plane_bytes + 16,), 7, dtype=torch.uint8, device="cuda")
            out = dst[shift:shift + n * 3 * window * plane_bytes]
            _lib.check(L.nexar_gather_windows_table(pool.data_ptr(), pool_frames, plane_bytes, window, slots.data_ptr(), n,
                                                    out.data_ptr(), None, stream))
            assert torch.equal(out.view(n, 3, window, plane_bytes), want), (shift, n)
            assert torch.all(dst[:shift] == 7) and torch.all(dst[shift + out.numel():] == 7)
        # the copy: slots 0..9 -> slots 13..22 (and one clamped destination), the rest untouched
        before = pool.clone()
        src = torch.arange(0, 10, dtype=torch.int32, device="cuda")
        dst_slots = torch.tensor([13, 14, 15, 16, 17, 18, 19, 20, 21, 99], dtype=torch.int32, device="cuda")
        _lib.check(L.nexar_gather_windows_table(pool.data_ptr(), pool_frames, plane_bytes, 1, src.data_ptr(), 10, None,
                                                dst_slots.data_ptr(), stream))
        want = before.clone()
        want[dst_slots.clamp(max=pool_frames - 1).long()] = before[src.long()]
        assert torch.equal(pool, want), shift


def test_gather_windows_table_refuses_bad_arguments():
    from vision_collision_detection_b200 import _lib
    L = _lib.table_lib()
    buf = C.c_void_p(16)           # never dereferenced: every call below fails its argument checks on the host

    def call(pool=buf, pool_frames=8, plane_bytes=64, window=4, slots=buf, n=1, dst=buf, dst_slots=None):
        return L.nexar_gather_windows_table(pool, pool_frames, plane_bytes, window, slots, n, dst, dst_slots, None)

    for kw in (dict(pool=None), dict(slots=None), dict(dst=None), dict(dst_slots=buf), dict(dst=None, dst_slots=buf),
               dict(pool_frames=0), dict(pool_frames=-1), dict(plane_bytes=0), dict(plane_bytes=-64), dict(window=0),
               dict(n=0), dict(n=-1), dict(n=2 ** 31 // 12 + 1), dict(window=2 ** 30, n=1)):
        assert call(**kw) == _lib.ERR_INVALID, kw
    assert "gather_windows_table" in L.nexar_last_error().decode()


@gpu
def test_predict_step_equals_predict_stream():
    from vision_collision_detection_b200.inference import MultiWindowStream, WindowPredictor
    w_mat = torch.tensor([[1.0, -2.0, 0.5], [-0.3, 0.8, 1.1], [0.2, 0.1, -0.9]], device="cuda")

    def model(x):
        return x.float().mean(dim=(2, 3, 4)) @ w_mat

    wp = WindowPredictor(model, window=16, stride=8, batch_size=3)
    videos = {f"cam{i}": _video(n, seed=30 + i, h=96, w=160) for i, n in enumerate((10, 70, 203))}
    ms = MultiWindowStream(16, 8, wp.swt.tf, out_dtype=wp.swt.out_dtype)
    got = {k: [] for k in videos}
    for lo in range(0, 203, 25):
        for k, v in videos.items():
            if lo < v.shape[0]:
                ms.push(k, v[lo:lo + 25])
            elif k in ms._open:
                ms.close(k)
        for r in wp.predict_step(*ms.step(), fps=25.0):
            got[r["video_path"]].append(r)
    for k in videos:
        if k in ms._open:
            ms.close(k)
    for r in wp.predict_step(*ms.step(), fps=25.0):
        got[r["video_path"]].append(r)
    for k, v in videos.items():
        want = list(wp.predict_stream((v[lo:lo + 25] for lo in range(0, v.shape[0], 25)), video_path="x", fps=25.0))
        assert len(got[k]) == len(want)
        for a, b in zip(got[k], want):
            assert a["video_path"] == k and b["video_path"] == "x"
            assert {x: y for x, y in a.items() if x not in ("video_path", "probabilities")} == \
                {x: y for x, y in b.items() if x not in ("video_path", "probabilities")}
            assert a["probabilities"] == pytest.approx(b["probabilities"], rel=1e-5, abs=1e-6)
