"""Cost of the YUV 4:2:0 source formats: tools/yuv_bench.py OUTDIR [--legs ...] [--modes ...] [--no-e2e]

Device-resident legs: the cfg2 batch of bench.py (32 clips x 16 frames, 720p -> 224, bf16) with the `val` and `custom`
kwargs, fed once per source format.  Every input is >= 0.7 GB (more than the 126 MB L2), built from 4 distinct clips.
The legs alternate round by round in one process; each round times >= 100 steps with CUDA events, and each leg's extra
time over the RGB leg is taken within the same round.  The 16-bit legs (p010, i010) carry 10-bit surfaces, uint16.
End-to-end legs: the same batch through HostClipPipeline from pinned host memory (rgb, nv12, i420, p010, i010).  One JSON line per leg goes to stdout and to OUTDIR/yuv_lines.jsonl, with the
GPU's name, power limit and maximum SM clock read in the same run.

With NEXAR_LIB pointing at an older build (which has only NV12 BT.601 limited range), run the `rgb` and `nv12_601l`
legs only, e.g. alternating two libraries:  for lib in A B A B; do NEXAR_LIB=$lib python tools/yuv_bench.py out
--legs rgb,nv12_601l --no-e2e; done
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

B, T, CS = 32, 16, 224
KW = {
    "custom": dict(mode="train", enable_custom_augmentation=True, brightness_range=(0.9, 1.1),
                   contrast_range=(0.9, 1.1), saturation_range=(0.9, 1.1), rotation_range=(-5, 5)),
    "val": dict(mode="val"),
}
# leg -> (picture h, w, forward_batch source keywords, surface luma rows, pitch); None keywords = RGB
LEGS = {
    "rgb": (720, 1280, None, None, None),
    "nv12_601l": (720, 1280, dict(pixel_format="nv12"), None, None),
    "nv12_709f": (720, 1280, dict(pixel_format="nv12", color_matrix="bt709", color_range="full"), None, None),
    "i420_709l": (720, 1280, dict(pixel_format="i420", color_matrix="bt709"), None, None),
    "rgb_1080p": (1080, 1920, None, None, None),
    "nv12_1080p_in_1088x2048": (1080, 1920, dict(pixel_format="nv12", color_matrix="bt709"), 1088, 2048),
    "p010_601l": (720, 1280, dict(pixel_format="p010"), None, None),
    "i010_709l": (720, 1280, dict(pixel_format="i010", color_matrix="bt709"), None, None),
    "p010_1080p_in_1088x2048": (1080, 1920, dict(pixel_format="p010", color_matrix="bt709"), 1088, 2048),
}
BASE = {"rgb": "rgb", "nv12_601l": "rgb", "nv12_709f": "rgb", "i420_709l": "rgb", "rgb_1080p": "rgb_1080p",
        "nv12_1080p_in_1088x2048": "rgb_1080p", "p010_601l": "rgb", "i010_709l": "rgb",
        "p010_1080p_in_1088x2048": "rgb_1080p"}


def gpu_provenance():
    q = "name,power.limit,clocks.max.sm"
    idx = torch.cuda.current_device()
    r = subprocess.run(["nvidia-smi", f"--id={idx}", f"--query-gpu={q}", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"query": q, "value": r.stdout.strip()} if r.returncode == 0 else {"query": q, "error": r.stderr.strip()}


_RGB = {}


def make_inputs(leg, dev):
    """Device tensor of B clips (4 distinct ones repeated) in the leg's source format, plus its picture size."""
    from vision_collision_detection_b200.synth import make_clip_torch, rgb_to_yuv420, rgb_to_yuv420_16
    h, w, kw, lr, pitch = LEGS[leg]
    distinct = []
    for i in range(4):
        if (h, w, i) not in _RGB:
            _RGB[h, w, i] = make_clip_torch(T, h, w, seed=i, kind="dashcam", device=dev).cpu().numpy()
        rgb = _RGB[h, w, i]
        if kw is None:
            distinct.append(torch.from_numpy(rgb))
        else:
            enc = rgb_to_yuv420_16 if kw["pixel_format"] in ("p010", "i010") else rgb_to_yuv420
            distinct.append(torch.from_numpy(enc(rgb, kw["pixel_format"], kw.get("color_matrix", "bt601"),
                                                 kw.get("color_range", "limited"), lr, pitch)))
    x = torch.empty((B,) + tuple(distinct[0].shape), dtype=distinct[0].dtype, device=dev)
    for i in range(B):
        x[i].copy_(distinct[i % 4])
    return x, h, w


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--legs", default=",".join(LEGS))
    ap.add_argument("--modes", default="val,custom")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--e2e-steps", type=int, default=12)
    ap.add_argument("--no-e2e", action="store_true")
    args = ap.parse_args()
    if args.steps < 100:
        raise SystemExit("--steps must be >= 100")
    if not torch.cuda.is_available():
        raise SystemExit("yuv_bench needs a GPU")
    os.makedirs(args.outdir, exist_ok=True)
    from vision_collision_detection_b200 import _lib, create_video_transforms
    legs = args.legs.split(",")
    for leg in legs:
        if leg not in LEGS:
            raise SystemExit(f"unknown leg {leg}")
        if BASE[leg] not in legs:
            legs.insert(0, BASE[leg])
    legs = list(dict.fromkeys(legs))
    dev = torch.device("cuda", torch.cuda.current_device())
    prov = dict(gpu_provenance(), torch=torch.__version__, lib=os.path.basename(_lib.LIB_PATH))
    out_lines = []

    def emit(rec):
        rec["provenance"] = prov
        line = json.dumps(rec)
        print(line, flush=True)
        out_lines.append(line)

    inputs = {leg: make_inputs(leg, dev) for leg in legs}
    for mode in args.modes.split(","):
        tf = create_video_transforms(**KW[mode], crop_size=CS, out_dtype=torch.bfloat16)
        out = torch.empty((B, 3, T, CS, CS), dtype=torch.bfloat16, device=dev)
        random.seed(1234)
        params = {hw: [tf.sample_params(B, *hw) for _ in range(4)] for hw in {(v[1], v[2]) for v in inputs.values()}}

        def step(leg, i):
            x, h, w = inputs[leg]
            kw = dict(LEGS[leg][2] or {})
            if LEGS[leg][3] is not None:
                kw["frame_size"] = (h, w)
            tf.forward_batch(x, params=params[h, w][i % 4], out=out, **kw)

        for leg in legs:                      # warm-up: plans, workspace, clocks
            for i in range(20):
                step(leg, i)
        torch.cuda.synchronize()
        ms = {leg: [] for leg in legs}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for r in range(args.rounds):
            for leg in (legs if r % 2 == 0 else legs[::-1]):
                e0.record()
                for i in range(args.steps):
                    step(leg, i)
                e1.record()
                torch.cuda.synchronize()
                ms[leg].append(e0.elapsed_time(e1) / args.steps)
        for leg in legs:
            med = statistics.median(ms[leg])
            extra = [a - b for a, b in zip(ms[leg], ms[BASE[leg]])]
            x, h, w = inputs[leg]
            emit({"leg": "device", "source": leg, "mode": mode, "batch": [B, T, h, w], "crop": CS, "out": "bf16",
                  "input_bytes": x.numel() * x.element_size(), "steps_per_round": args.steps, "rounds": args.rounds,
                  "ms_step_median": round(med, 4), "ms_step_rounds": [round(v, 4) for v in ms[leg]],
                  "spread_ms": round(max(ms[leg]) - min(ms[leg]), 4), "clips_per_s": round(B / (med * 1e-3), 1),
                  "extra_ms_over": BASE[leg], "extra_ms_median": round(statistics.median(extra), 4),
                  "extra_ms_rounds": [round(v, 4) for v in extra]})

    if not args.no_e2e:
        from vision_collision_detection_b200.host_pipeline import HostClipPipeline
        tf = create_video_transforms(**KW["custom"], crop_size=CS, out_dtype=torch.bfloat16)
        random.seed(1234)
        ps = [tf.sample_params(B, 720, 1280) for _ in range(4)]
        for src, leg in (("rgb", "rgb"), ("nv12", "nv12_601l"), ("i420", "i420_709l"), ("p010", "p010_601l"),
                         ("i010", "i010_709l")):
            x = inputs[leg][0] if leg in inputs else make_inputs(leg, dev)[0]
            nbytes = x.numel() * x.element_size()
            kw = LEGS[leg][2] or {}
            pipe = HostClipPipeline(tf, n_clips=B, frames=T, height=720, width=1280, device=dev, **kw)
            ins = [pipe.pinned_input(), pipe.pinned_input()]
            for hbuf in ins:
                hbuf.copy_(x.cpu())
            for i in range(2):
                pipe.run(ins[i & 1], params=ps[i % 4])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            prev = None
            for i in range(args.e2e_steps):       # batch i+1 is submitted before batch i is collected
                ticket = pipe.submit(ins[i & 1], params=ps[i % 4])
                if prev is not None:
                    pipe.wait(prev)
                prev = ticket
            pipe.wait(prev)
            torch.cuda.synchronize()
            ms_step = (time.perf_counter() - t0) * 1e3 / args.e2e_steps
            emit({"leg": "e2e", "source": src, "mode": "custom", "batch": [B, T, 720, 1280], "crop": CS, "out": "bf16",
                  "h2d_bytes_per_step": nbytes, "steps": args.e2e_steps, "ms_step": round(ms_step, 3),
                  "clips_per_s": round(B / (ms_step * 1e-3), 1),
                  "h2d_GBs": round(nbytes / (ms_step * 1e-3) / 1e9, 2)})
            del pipe, ins
    with open(os.path.join(args.outdir, "yuv_lines.jsonl"), "a") as f:
        f.write("\n".join(out_lines) + "\n")


if __name__ == "__main__":
    main()
