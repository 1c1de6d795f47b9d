"""Property tests (CPU) of the host-side entry points of the C ABI against the numpy oracle, over random sizes:
letterbox geometry (nexar_video_aug.py:713-719), short-side resize + centre crop geometry (:411-415, :468-469), the ATen
antialias tap tables, and the bench's algorithmic-byte arithmetic (SURVEY.md section 8d)."""
import numpy as np
from hypothesis import assume, given, settings, strategies as st

from oracle import np_oracle as O
from vision_collision_detection_b200 import _lib


@settings(max_examples=300, deadline=None)
@given(st.integers(1, 2200), st.integers(1, 4000), st.integers(1, 512))
def test_letterbox_geometry_equals_the_python_formula(h, w, cs):
    scale = min(cs / h, cs / w)                       # nexar_video_aug.py:713
    nh, nw = int(h * scale), int(w * scale)           # :714-715 (float64 truncation)
    if nh <= 0 or nw <= 0:                            # torch's resize would raise; the C entry point returns an error
        try:
            _lib.letterbox_geometry(h, w, cs)
        except _lib.NexarError:
            return
        raise AssertionError("expected an error for an empty resize")
    g = _lib.letterbox_geometry(h, w, cs)
    assert (g.resize_h, g.resize_w, g.off_y, g.off_x) == (nh, nw, (cs - nh) // 2, (cs - nw) // 2)
    assert (nh, nw, (cs - nh) // 2, (cs - nw) // 2) == tuple(O.letterbox_geometry(h, w, cs))
    assert max(nh, nw) <= cs and g.off_y >= 0 and g.off_x >= 0


@settings(max_examples=200, deadline=None)
@given(st.integers(8, 1200), st.integers(8, 2000), st.integers(4, 400))
def test_resize_crop_geometry_equals_the_python_formula(h, w, size):
    cs = size                                         # the factories crop to the short side's size or smaller
    rh, rw = (size * h // w, size) if h > w else (size, size * w // h)      # nexar_video_aug.py:411-415
    if rh < cs or rw < cs:
        return
    g = _lib.resize_crop_geometry(h, w, size, cs)
    assert (g.resize_h, g.resize_w) == (rh, rw)
    assert (-g.off_y, -g.off_x) == ((rh - cs) // 2, (rw - cs) // 2)         # centre crop :468-469


@settings(max_examples=120, deadline=None)
@given(st.integers(1, 1400), st.integers(1, 500))
def test_tap_tables_equal_the_oracle_for_any_size(in_size, out_size):
    assume(int(np.ceil(max(in_size / out_size, 1.0))) * 2 + 1 <= 256)      # the table width the caller provides room for
    start, count, wts = _lib.aa_taps(in_size, out_size, cap=256)
    xs, xc, xw = O.aa_taps(in_size, out_size)
    assert np.array_equal(start, xs) and np.array_equal(count, xc)
    assert wts.shape == xw.shape and np.array_equal(wts, xw)
    assert (start >= 0).all() and (start + count <= in_size).all() and (count >= 1).all()
    assert np.abs(wts.sum(axis=1) - 1.0).max() < 2e-6


def test_algorithmic_bytes_match_the_survey():
    import bench
    assert bench.algorithmic_bytes_per_clip(16, 720, 1280, 224, 2) == 49_053_696       # cfg2, bf16 (SURVEY 8d)
    assert bench.algorithmic_bytes_per_clip(16, 720, 1280, 224, 4) == 53_870_592       # cfg2, fp32
    assert bench.algorithmic_bytes_per_clip(32, 720, 1280, 320, 2) == 108_134_400      # cfg3
    b, t, h, w, cs = bench.WORKLOADS["cfg3"]
    assert b == 256 and all(b % n == 0 for n in (1, 2, 4, 8))                          # one batch sharded over the GPUs
    assert bench.WORKLOADS["cfg2"] == (32, 16, 720, 1280, 224) and bench.WORKLOADS["cfg4"][1] == 1200


def test_dumped_outputs_are_whole_or_a_fixed_row_sample_within_64_mb():
    import torch

    import bench
    small = torch.arange(4 * 3 * 4 * 8 * 8, dtype=torch.float32).view(4, 3, 4, 8, 8).bfloat16()
    d = bench.sample_outputs({"out": small})
    assert list(d) == ["out"] and d["out"].dtype == np.float32 and np.array_equal(d["out"], small.float().numpy())
    # cfg2's output shape (bf16): too large to keep whole, so a seeded sample of whole rows with their indices
    big = torch.randn((32, 3, 16, 224, 224), generator=torch.Generator().manual_seed(3)).bfloat16()
    d = bench.sample_outputs({"out": big})
    rows, idx = d["out_rows"], d["out_rows_index"]
    assert rows.dtype == np.float32 and idx.dtype == np.float64 and rows.shape == (len(idx), 224) and idx.shape[1] == 4
    assert sum(a.nbytes + 128 for a in d.values()) <= 64 << 20 and len(idx) > 0.2 * 32 * 3 * 16 * 224
    assert np.array_equal(rows, big.float().numpy()[tuple(idx.astype(np.int64).T)])
    again = bench.sample_outputs({"out": big})
    assert all(np.array_equal(d[k], again[k]) for k in d)
