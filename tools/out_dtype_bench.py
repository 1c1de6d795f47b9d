"""Cost of each output type (fp32, bf16, fp16): tools/out_dtype_bench.py OUT.jsonl [--parent-lib LIB] [options]

Device-resident legs: cfg2 (32 clips x 16 frames, 720p -> 224) with the `custom` and `val` kwargs, and cfg3 (256 clips x
32 frames, 720p -> 320, `custom`), each written once per output type into a preallocated tensor.  The inputs are 1.4 GB
and 22.6 GB (more than the 126 MB L2), built from 4 distinct clips.  The output types alternate round by round in one
process (forward, then reverse order); each round times --steps steps (cfg3: --cfg3-steps) with CUDA events after a
warm-up of every type.  Each line carries the per-round times, their spread, and the difference to bf16 in the same round.

End-to-end legs: the cfg2 custom batch through HostClipPipeline from pinned host memory, once per output type, the types
alternating over --e2e-rounds rounds.

With --parent-lib, the f32 and bf16 cfg2 legs are then timed against that library (an older build selected through
NEXAR_LIB): child processes alternate between it and the current library, --ab-runs runs each, and every line records
the library it ran.  One JSON line per leg goes to stdout and is appended to OUT.jsonl, with the GPU's name, power
limit and maximum SM clock read in the same run.
"""
import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

KW = {
    "custom": dict(mode="train", enable_custom_augmentation=True, brightness_range=(0.9, 1.1),
                   contrast_range=(0.9, 1.1), saturation_range=(0.9, 1.1), rotation_range=(-5, 5)),
    "val": dict(mode="val"),
}
SHAPES = {"cfg2": (32, 16, 720, 1280, 224), "cfg3": (256, 32, 720, 1280, 320)}
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
LEGS = ("cfg2:custom", "cfg2:val", "cfg3:custom")


def gpu_provenance():
    q = "name,power.limit,clocks.max.sm"
    idx = torch.cuda.current_device()
    r = subprocess.run(["nvidia-smi", f"--id={idx}", f"--query-gpu={q}", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"query": q, "value": r.stdout.strip()} if r.returncode == 0 else {"query": q, "error": r.stderr.strip()}


def make_input(cfg, dev):
    """uint8 [B,T,H,W,3] on the device: 4 distinct synthetic dashcam clips repeated."""
    from vision_collision_detection_b200.synth import make_clip_torch
    b, t, h, w, _ = SHAPES[cfg]
    distinct = [make_clip_torch(t, h, w, seed=i, kind="dashcam", device=dev) for i in range(4)]
    x = torch.empty((b, t, h, w, 3), dtype=torch.uint8, device=dev)
    for i in range(b):
        x[i].copy_(distinct[i % 4])
    return x


def time_device_legs(legs, dtypes, steps, cfg3_steps, rounds, dev, emit, extra=None):
    from vision_collision_detection_b200 import create_video_transforms
    inputs = {}
    for leg in legs:
        cfg, mode = leg.split(":")
        b, t, h, w, cs = SHAPES[cfg]
        if cfg not in inputs:
            inputs = {cfg: make_input(cfg, dev)}          # one input resident at a time
        x = inputs[cfg]
        n = cfg3_steps if cfg == "cfg3" else steps
        tf = create_video_transforms(**KW[mode], crop_size=cs)
        outs = {d: torch.empty((b, 3, t, cs, cs), dtype=DTYPES[d], device=dev) for d in dtypes}
        random.seed(1234)
        params = [tf.sample_params(b, h, w) for _ in range(4)]

        def run(d, k):
            for i in range(k):
                tf.forward_batch(x, params=params[i % 4], out=outs[d])

        for d in dtypes:                                  # warm-up: plans, workspace, clocks
            run(d, max(4, n // 5))
        torch.cuda.synchronize()
        ms = {d: [] for d in dtypes}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for r in range(rounds):
            for d in (dtypes if r % 2 == 0 else dtypes[::-1]):
                e0.record()
                run(d, n)
                e1.record()
                torch.cuda.synchronize()
                ms[d].append(e0.elapsed_time(e1) / n)
        for d in dtypes:
            med = statistics.median(ms[d])
            out_bytes = outs[d].numel() * outs[d].element_size()
            rec = {"leg": "device", "workload": cfg, "mode": mode, "batch": [b, t, h, w], "crop": cs, "out": d,
                   "input_bytes": x.numel(), "output_bytes": out_bytes, "steps_per_round": n, "rounds": rounds,
                   "ms_step_median": round(med, 4), "ms_step_rounds": [round(v, 4) for v in ms[d]],
                   "spread_ms": round(max(ms[d]) - min(ms[d]), 4), "clips_per_s": round(b / (med * 1e-3), 1)}
            if "bf16" in ms and d != "bf16":
                diff = [a - c for a, c in zip(ms[d], ms["bf16"])]
                rec.update(minus_bf16_ms_median=round(statistics.median(diff), 4),
                           minus_bf16_ms_rounds=[round(v, 4) for v in diff])
            rec.update(extra or {})
            emit(rec)
        del outs
    del inputs
    torch.cuda.empty_cache()


def time_e2e(dtypes, steps, rounds, dev, emit):
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.host_pipeline import HostClipPipeline
    b, t, h, w, cs = SHAPES["cfg2"]
    tf = create_video_transforms(**KW["custom"], crop_size=cs)
    random.seed(1234)
    ps = [tf.sample_params(b, h, w) for _ in range(4)]
    x = make_input("cfg2", dev).cpu()
    pipes = {d: HostClipPipeline(tf, n_clips=b, frames=t, height=h, width=w, device=dev, out_dtype=DTYPES[d])
             for d in dtypes}
    ins = [pipes[dtypes[0]].pinned_input(), pipes[dtypes[0]].pinned_input()]     # shared by every pipeline
    for hbuf in ins:
        hbuf.copy_(x)
    for d in dtypes:
        for i in range(2):
            pipes[d].run(ins[i & 1], params=ps[i % 4])
    torch.cuda.synchronize()
    ms = {d: [] for d in dtypes}
    for r in range(rounds):
        for d in (dtypes if r % 2 == 0 else dtypes[::-1]):
            pipe = pipes[d]
            t0 = time.perf_counter()
            prev = None
            for i in range(steps):                       # batch i+1 is submitted before batch i is collected
                ticket = pipe.submit(ins[i & 1], params=ps[i % 4])
                if prev is not None:
                    pipe.wait(prev)
                prev = ticket
            pipe.wait(prev)
            torch.cuda.synchronize()
            ms[d].append((time.perf_counter() - t0) * 1e3 / steps)
    for d in dtypes:
        med = statistics.median(ms[d])
        d2h = b * 3 * t * cs * cs * DTYPES[d].itemsize
        emit({"leg": "e2e", "workload": "cfg2", "mode": "custom", "batch": [b, t, h, w], "crop": cs, "out": d,
              "h2d_bytes_per_step": x.numel(), "d2h_bytes_per_step": d2h, "steps_per_round": steps, "rounds": rounds,
              "ms_step_median": round(med, 3), "ms_step_rounds": [round(v, 3) for v in ms[d]],
              "spread_ms": round(max(ms[d]) - min(ms[d]), 3), "clips_per_s": round(b / (med * 1e-3), 1)})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--legs", default=",".join(LEGS))
    ap.add_argument("--dtypes", default="f32,bf16,f16")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--cfg3-steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--e2e-steps", type=int, default=12)
    ap.add_argument("--e2e-rounds", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--parent-lib", help="library of the parent commit: A/B its f32 and bf16 cfg2 legs against this one")
    ap.add_argument("--ab-runs", type=int, default=3)
    ap.add_argument("--ab-run", type=int, help=argparse.SUPPRESS)     # set in the A/B child processes
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("out_dtype_bench needs a GPU")
    from vision_collision_detection_b200 import _lib
    dtypes = args.dtypes.split(",")
    legs = args.legs.split(",")
    for v, known in ((dtypes, DTYPES), (legs, LEGS)):
        bad = [x for x in v if x not in known]
        if bad:
            raise SystemExit(f"unknown: {bad}")
    dev = torch.device("cuda", torch.cuda.current_device())
    prov = dict(gpu_provenance(), torch=torch.__version__, lib=os.path.basename(_lib.LIB_PATH))
    lines = []

    def emit(rec):
        rec["provenance"] = prov
        line = json.dumps(rec)
        print(line, flush=True)
        lines.append(line)

    extra = {"ab_run": args.ab_run} if args.ab_run is not None else None
    time_device_legs(legs, dtypes, args.steps, args.cfg3_steps, args.rounds, dev, emit, extra)
    if not args.no_e2e and args.ab_run is None:
        time_e2e(dtypes, args.e2e_steps, args.e2e_rounds, dev, emit)
    with open(args.out, "a") as f:
        f.write("\n".join(lines) + "\n")
    if args.parent_lib:
        current = os.path.abspath(_lib.LIB_PATH)
        parent = os.path.abspath(args.parent_lib)
        for run in range(2 * args.ab_runs):
            lib = (parent, current)[(run + run // 2) % 2]          # parent, current, current, parent, ...
            cmd = [sys.executable, os.path.abspath(__file__), args.out, "--legs", "cfg2:custom,cfg2:val",
                   "--dtypes", "f32,bf16", "--steps", str(args.steps), "--rounds", "3", "--ab-run", str(run + 1)]
            subprocess.run(cmd, env=dict(os.environ, NEXAR_LIB=lib), check=True)


if __name__ == "__main__":
    main()
