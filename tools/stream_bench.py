"""Streaming sliding-window inference (inference.WindowStream): tools/stream_bench.py OUT.jsonl [options]

Device leg: the BASELINE cfg4 video (1200 synthetic dashcam frames of 720p, device-resident, 3.3 GB) through the val
chain to 224 x 224 bf16, 16-frame windows at stride 8 (149 windows).  The offline call (SlidingWindowTransform.windows
with materialize=True: the whole video in one transform call, then one gather) alternates, round by round, with
WindowStream fed chunks of 1, 8, 30 and 120 frames (max_chunk 64).  Each timing is a host clock around one whole video
that ends in a device synchronise; each push is also bracketed by CUDA events, whose median is the time from a push
to its windows being ready.  The peak device memory of a video is torch.cuda.max_memory_allocated above what was
allocated before it (the source video excluded, the windows a push returns included until the next push).

Host legs: RGB and NV12 chunks of 30 frames pushed from pinned host memory (a 1200-frame pinned buffer), for the 40 s
video and for a 36000-frame "20 min drive" that cycles the same buffer.

--rounds rounds (default 5), the legs alternating in forward and reverse order; every line gives the per-round
values and their medians, with the GPU's name, power limit and maximum SM clock read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

N, H, W, CS, WINDOW, STRIDE = 1200, 720, 1280, 224, 16, 8


def gpu_provenance():
    q = "name,power.limit,clocks.max.sm"
    idx = torch.cuda.current_device()
    r = subprocess.run(["nvidia-smi", f"--id={idx}", f"--query-gpu={q}", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"query": q, "value": r.stdout.strip()} if r.returncode == 0 else {"query": q, "error": r.stderr.strip()}


def make_video(dev):
    """uint8 [1200,720,1280,3]: 12 distinct 100-frame synthetic dashcam clips, as bench.py builds cfg4."""
    from vision_collision_detection_b200.synth import make_clip_torch
    return torch.cat([make_clip_torch(100, H, W, seed=i, kind="dashcam", device=dev) for i in range(N // 100)])


def run_stream(tf, chunks, n_frames, fmt):
    """One video through a WindowStream -> (seconds, windows, [push ms], peak bytes above the start)."""
    from vision_collision_detection_b200.inference import WindowStream
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    events, count = [], 0
    t0 = time.perf_counter()
    ws = WindowStream(WINDOW, STRIDE, tf, out_dtype=torch.bfloat16, max_chunk=64)
    for chunk in chunks():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        starts, wins = ws.push(chunk, **fmt)
        e1.record()
        events.append((e0, e1))
        count += len(starts)
    starts, wins = ws.finish()
    count += len(starts)
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    peak = torch.cuda.max_memory_allocated() - base
    assert count == (n_frames - WINDOW) // STRIDE + 1
    del ws, wins
    return sec, count, [a.elapsed_time(b) for a, b in events], peak


def run_offline(tf, video):
    from vision_collision_detection_b200.inference import SlidingWindowTransform
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    out = SlidingWindowTransform(WINDOW, STRIDE, tf, torch.bfloat16).windows(video, materialize=True)
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    peak = torch.cuda.max_memory_allocated() - base
    k = out.shape[0]
    del out
    return sec, k, [], peak


def summarise(per_round):
    secs = [r[0] for r in per_round]
    k = per_round[0][1]
    pushes = [statistics.median(r[2]) for r in per_round if r[2]]
    med = statistics.median(secs)
    return {"ms_per_video": round(1e3 * med, 3), "windows": k, "windows_per_s": round(k / med, 1),
            "ms_per_video_rounds": [round(1e3 * s, 3) for s in secs],
            "spread_pct": round(100 * (max(secs) - min(secs)) / med, 1),
            "push_to_windows_ms_median": round(statistics.median(pushes), 4) if pushes else None,
            "peak_device_mb": round(max(r[3] for r in per_round) / 2 ** 20, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--drive-frames", type=int, default=36000)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "stream_bench measures on a CUDA device"
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.synth import rgb_to_nv12
    dev = torch.device("cuda", torch.cuda.current_device())
    prov = gpu_provenance()
    tf = create_video_transforms(mode="val", crop_size=CS)
    video = make_video(dev)
    pinned = {"rgb": video.cpu().pin_memory(),
              "nv12": torch.cat([rgb_to_nv12(video[lo:lo + 100]).cpu() for lo in range(0, N, 100)]).pin_memory()}

    def device_chunks(c):
        return lambda: (video[lo:lo + c] for lo in range(0, N, c))

    def host_chunks(src, n_frames):
        return lambda: (src[lo % N:lo % N + 30] for lo in range(0, n_frames, 30))

    device_legs = {"offline": (N, lambda: run_offline(tf, video))}
    for c in (1, 8, 30, 120):
        device_legs[f"device_chunk{c}"] = (N, lambda c=c: run_stream(tf, device_chunks(c), N, {}))
    host_legs = {}
    for fmt, src in pinned.items():
        kw = {"pixel_format": "nv12"} if fmt == "nv12" else {}
        for n_frames in (N, args.drive_frames):
            host_legs[f"pinned_{fmt}_chunk30_{n_frames}f"] = (
                n_frames, lambda src=src, n_frames=n_frames, kw=kw: run_stream(tf, host_chunks(src, n_frames), n_frames, kw))

    lines = []
    for legs, where in ((device_legs, "device-resident"), (host_legs, "pinned host memory")):
        if legs is host_legs:
            del video           # the host legs hold no video on the device
            torch.cuda.empty_cache()
        for _, fn in legs.values():      # warm-up: plans, workspace, staging, clocks
            fn()
        results = {name: [] for name in legs}
        for r in range(args.rounds):
            for name in (list(legs) if r % 2 == 0 else list(reversed(legs))):
                results[name].append(legs[name][1]())
        for name, per_round in results.items():
            line = {"leg": name, "source": where,
                    "video": f"{legs[name][0]} frames {H}x{W} synthetic dashcam",
                    "path": "SlidingWindowTransform.windows(materialize=True)" if name == "offline" else
                            "WindowStream(max_chunk=64).push",
                    "transform": f"val -> {CS}x{CS} bf16, windows of {WINDOW} at stride {STRIDE}",
                    "rounds": args.rounds, "gpu": prov, **summarise(per_round)}
            lines.append(line)
            print(json.dumps(line), flush=True)
    with open(args.out, "a") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
