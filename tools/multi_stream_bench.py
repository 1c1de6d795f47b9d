"""Many cameras on one GPU (inference.MultiWindowStream): tools/multi_stream_bench.py OUT.jsonl [options]

Workload: S cameras, each pushing one 720p frame per step, through the val chain to 224 x 224 bf16, windows of 16 at
stride 8 (a camera completes a window every 8 steps from step 16 on).  S in --cameras (default 1 16 64 256 1024), and
three sources: device-resident RGB, RGB in pinned host memory and NV12 in pinned host memory.  Camera s pushes frame
(s + step) % 64 of a bank of 64 synthetic dashcam frames, so the device bank (177 MB) stays small while every step
reads S distinct-enough frames; with S >= 64 a step reads more than the 126 MB of L2.

Two legs per (S, source), alternating round by round (forward, then reverse order):
- multi: one MultiWindowStream(max_frames_per_step=1024); each step pushes S one-frame chunks and calls step().
- separate: the status quo, S WindowStream(max_chunk=1) objects, each pushed its one frame per step.

Per step: wall time (host clock around the pushes and the step plus a device synchronise, averaged over --steps steps
after --warmup steps), host enqueue time (the same clock without the synchronise), frames/s, windows/s, cameras
sustained at 30 fps (frames/s / 30) and the peak device memory above what was allocated before the leg (the frame bank
excluded).  Every line gives the per-round values and their median, with the GPU's name, power limit and maximum SM
clock read in the same run.
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from stream_bench import gpu_provenance  # noqa: E402

H, W, CS, WINDOW, STRIDE, BANK = 720, 1280, 224, 16, 8, 64


def run_leg(kind, tf, bank, n_cams, steps, warmup, fmt):
    """-> (wall ms / step, enqueue ms / step, windows / step, peak bytes)."""
    from vision_collision_detection_b200.inference import MultiWindowStream, WindowStream
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    if kind == "multi":
        ms = MultiWindowStream(WINDOW, STRIDE, tf, out_dtype=torch.bfloat16, max_frames_per_step=1024)
    else:
        streams = [WindowStream(WINDOW, STRIDE, tf, out_dtype=torch.bfloat16, max_chunk=1) for _ in range(n_cams)]
    wall = enq = 0.0
    windows = 0
    for i in range(warmup + steps):
        if i == warmup:
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        if kind == "multi":
            for s in range(n_cams):
                f = (s + i) % BANK
                ms.push(s, bank[f:f + 1], **fmt)
            k = len(ms.step()[0])
        else:
            k = 0
            for s, ws in enumerate(streams):
                f = (s + i) % BANK
                k += len(ws.push(bank[f:f + 1], **fmt)[0])
        t1 = time.perf_counter()
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        if i >= warmup:
            enq += t1 - t0
            wall += t2 - t0
            windows += k
    peak = torch.cuda.max_memory_allocated() - base
    return 1e3 * wall / steps, 1e3 * enq / steps, windows / steps, peak


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--cameras", type=int, nargs="+", default=[1, 16, 64, 256, 1024])
    ap.add_argument("--sources", nargs="+", default=["device_rgb", "pinned_rgb", "pinned_nv12"])
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=16)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "multi_stream_bench measures on a CUDA device"
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.synth import make_clip_torch, rgb_to_nv12
    dev = torch.device("cuda", torch.cuda.current_device())
    prov = gpu_provenance()
    tf = create_video_transforms(mode="val", crop_size=CS)
    rgb = make_clip_torch(BANK, H, W, seed=0, kind="dashcam", device=dev)
    banks = {"device_rgb": (rgb, {}), "pinned_rgb": (rgb.cpu().pin_memory(), {}),
             "pinned_nv12": (rgb_to_nv12(rgb).cpu().pin_memory(), {"pixel_format": "nv12"})}
    lines = []
    for source in args.sources:
        bank, fmt = banks[source]
        for n_cams in args.cameras:
            legs = ["multi", "separate"]
            res = {k: [] for k in legs}
            for k in legs:                   # warm-up of both legs: plans, workspace, staging, clocks
                run_leg(k, tf, bank, n_cams, 4, WINDOW, fmt)
            for r in range(args.rounds):
                for k in (legs if r % 2 == 0 else legs[::-1]):
                    res[k].append(run_leg(k, tf, bank, n_cams, args.steps, args.warmup, fmt))
                    torch.cuda.empty_cache()
            for k, per_round in res.items():
                wall = statistics.median(x[0] for x in per_round)
                enq = statistics.median(x[1] for x in per_round)
                win = per_round[0][2]
                fps = n_cams / (wall / 1e3)
                line = {"leg": k, "source": source, "cameras": n_cams,
                        "path": "MultiWindowStream(max_frames_per_step=1024): S pushes + step()" if k == "multi" else
                                "S x WindowStream(max_chunk=1).push",
                        "workload": f"one {H}x{W} synthetic dashcam frame per camera per step, val -> {CS}x{CS} bf16, "
                                    f"windows of {WINDOW} at stride {STRIDE}",
                        "steps": args.steps, "warmup_steps": args.warmup, "rounds": args.rounds,
                        "wall_ms_per_step": round(wall, 4), "enqueue_ms_per_step": round(enq, 4),
                        "wall_ms_per_step_rounds": [round(x[0], 4) for x in per_round],
                        "spread_pct": round(100 * (max(x[0] for x in per_round) - min(x[0] for x in per_round)) / wall, 1),
                        "frames_per_s": round(fps, 1), "windows_per_s": round(win / (wall / 1e3), 1),
                        "cameras_at_30fps": round(fps / 30, 1),
                        "peak_device_mb": round(max(x[3] for x in per_round) / 2 ** 20, 1), "gpu": prov}
                lines.append(line)
                print(json.dumps(line), flush=True)
    with open(args.out, "a") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
