"""Source-format rules (source_format.py): every entry point that takes decoded frames refuses a malformed source the
same way, and the stream classes refuse it before any CUDA call and before they change any state."""
import pytest
import torch

U8, U16 = torch.uint8, torch.uint16


def _rgb(dtype=U8):
    return torch.zeros((2, 8, 8, 3), dtype=dtype)


def _surface(rows=12, pitch=8, dtype=U8):
    return torch.zeros((2, rows, pitch), dtype=dtype)


# (host chunk [n,*frame], keywords, exception of a WindowStream / MultiWindowStream push).  forward_batch and
# SlidingWindowTransform.frames refuse every row with ValueError on the host, where a source that passes the format
# checks is refused for not being on the device; only the int32 row differs, TypeError, on the device.
REFUSALS = [
    (_rgb(), dict(pixel_format="yuv444"), ValueError),
    (_rgb(), dict(color_matrix="bt2020"), ValueError),
    (_surface(), dict(pixel_format="nv12", color_range="tv"), ValueError),
    (_rgb(torch.float32), {}, TypeError),
    (_surface(dtype=torch.float32), dict(pixel_format="nv12"), TypeError),
    (_rgb(U16), {}, ValueError),
    (_surface(), dict(pixel_format="p010"), ValueError),
    (_surface(), dict(pixel_format="i010"), ValueError),
    (_surface(dtype=U16), dict(pixel_format="nv12"), ValueError),
    (_surface(dtype=U16), dict(pixel_format="i420"), ValueError),
    (_rgb(torch.int32), {}, ValueError),
    (_surface(rows=13), dict(pixel_format="nv12"), ValueError),
    (_surface(pitch=7), dict(pixel_format="i420"), ValueError),
    (_surface(rows=13, dtype=U16), dict(pixel_format="p010"), ValueError),
    (torch.zeros((2, 8, 8), dtype=U8), {}, ValueError),                         # RGB frames are [H,W,3]
    (_rgb(), dict(pixel_format="nv12"), ValueError),                           # YUV surfaces are [R,P]
    (_rgb(), dict(frame_size=(8, 8)), ValueError),                             # RGB frames have no padding
    (_surface(), dict(pixel_format="nv12", frame_size=(8, 7)), ValueError),    # odd
    (_surface(), dict(pixel_format="i420", frame_size=(10, 8)), ValueError),   # more rows than the 8 luma rows
    (_surface(dtype=U16), dict(pixel_format="i010", frame_size=(8, 10)), ValueError),   # wider than the pitch
]


def test_refusal_table_on_the_host():
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.inference import MultiWindowStream, SlidingWindowTransform, WindowStream
    tf = create_video_transforms(mode="val", crop_size=32)
    for chunk, kw, stream_error in REFUSALS:
        if chunk.dtype != torch.int32:
            with pytest.raises(ValueError):
                tf.forward_batch(chunk.unsqueeze(0), **kw)
            with pytest.raises(ValueError):
                SlidingWindowTransform(4, 2, tf).frames(chunk, **kw)
        ws = WindowStream(4, 2, tf)
        with pytest.raises(stream_error):
            ws.push(chunk, **kw)
        assert ws._source is None and ws._params is None and ws._ring is None, kw
        ms = MultiWindowStream(4, 2, tf)
        with pytest.raises(stream_error):
            ms.push("a", chunk, **kw)
        assert ms.device is None and not ms._open and ms._pool is None, kw
