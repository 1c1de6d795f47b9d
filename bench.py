#!/usr/bin/env python
"""bench.py — clips/s of the clip-transform hot path on N B200s (one process per GPU).

A "step" is one pass of the fused transform over one batch of synthetic dashcam
clips.  Default workload = BASELINE.json configs[1]: train-time augmentation,
32 clips x 16 frames x 720x1280 uint8 -> [32,3,16,224,224] bf16 per GPU
(weak scaling: every rank transforms its own 32-clip shard, no collective on
the data path).  See DESIGN.md "Measurement".

  python bench.py [--gpus N] [--steps K] [--warmup W] [--mode custom|train|val] [--impl reference]
                  [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step returned as DIR/<name>.npy (at most 64 MB; a larger output as a
fixed, seeded sample of whole rows, see sample_outputs), so that two builds can be compared output for output: the
inputs and the random decisions are seeded, identical from run to run.
"""
import argparse
import json
import os
import random
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # name: (clips per GPU, T, H, W, crop_size)
    "cfg2": (32, 16, 720, 1280, 224),
    "cfg3": (256, 32, 720, 1280, 320),  # BASELINE configs[2]: ONE 256-clip batch, sharded over the GPUs (strong scaling)
    "tiny": (4, 4, 180, 320, 112),
    "cfg2s": (8, 16, 720, 1280, 224),   # a trainer-sized batch (cfg5 uses 8 clips per GPU): band-count tuning
    # BASELINE configs[3]: one 40 s x 30 fps 720p video, val chain, every frame transformed once,
    # 16-frame windows at stride 8 as strided views (149 windows); "clips" = windows
    "cfg4": (1, 1200, 720, 1280, 224),
}
# the live train call site nexar_videos.py:2003-2010
KW = {
    "custom": dict(mode="train", enable_custom_augmentation=True, brightness_range=(0.9, 1.1),
                   contrast_range=(0.9, 1.1), saturation_range=(0.9, 1.1), rotation_range=(-5, 5)),
    "train": dict(mode="train"),      # nexar_videos.py:936
    "val": dict(mode="val"),          # nexar_videos.py:947, nexar_inference.py:218
}
METRIC = "augmented clips/sec and achieved HBM GB/s (% of roofline) at 1/2/4/8 B200 vs host CPU"


def algorithmic_bytes_per_clip(t, h, w, cs, out_bytes):
    """SURVEY.md section 8(d): uint8 source read once + output written once."""
    return t * h * w * 3 + 3 * t * cs * cs * out_bytes


def ncu_traffic(workload, mode, out_dtype):
    """dram bytes per launch of the dominant kernel from the committed `ncu --set full` capture (profiles/)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(p) as f:
            return json.load(f).get(f"{workload}:{mode}:{out_dtype}")     # {"step": bytes, "kernels": {name: bytes}}
    except Exception:
        return None


DUMP_BYTES = 64 << 20          # --dump-outputs: at most this many bytes written in all
DUMP_SEED = 0


def sample_outputs(arrays):
    """{name: tensor} -> {file name: float32 / float64 ndarray} for --dump-outputs.  A tensor that fits its share of
    DUMP_BYTES is kept whole as ``<name>``; a larger one becomes a fixed, seeded sample of whole last-axis rows,
    ``<name>_rows`` [n, W] float32, with ``<name>_rows_index`` [n, ndim - 1] float64 holding each row's leading
    indices.  The sample depends only on the shape, so two runs with the same arguments pick the same rows."""
    share = DUMP_BYTES // len(arrays) - 4096        # room for the .npy headers
    res = {}
    for name, x in arrays.items():
        if x.numel() * 4 <= share:
            res[name] = x.float().cpu().numpy()
            continue
        lead, w = tuple(x.shape[:-1]), int(x.shape[-1])
        n_rows = x.numel() // w
        k = min(n_rows, share // (4 * w + 8 * len(lead)))
        pick = torch.randperm(n_rows, generator=torch.Generator().manual_seed(DUMP_SEED))[:k].sort().values
        idx = np.stack(np.unravel_index(pick.numpy(), lead), axis=1)
        rows = x[tuple(torch.from_numpy(idx[:, d]).to(x.device) for d in range(len(lead)))]    # [k, w], no full copy
        res[f"{name}_rows"] = rows.float().cpu().numpy()
        res[f"{name}_rows_index"] = idx.astype(np.float64)
    return res


def write_outputs(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def count(self, t0, t1):
        return sum(1 for ts, _ in list(self.rows) if t0 - 0.05 <= ts <= t1 + 0.15)

    def stop(self, t0, t1):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                clk, cmax = float(parts[0]), float(parts[1])
            except ValueError:
                continue
            mx = max(mx, cmax)
            if t0 - 0.05 <= ts <= t1 + 0.15:
                sm.append(clk)
                for n, v in zip(names, parts[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        if not sm:
            sm = [float(l.split(",")[0]) for _, l in self.rows[-3:] if l and l.split(",")[0].strip().replace(".", "").isdigit()]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def oracle_setup(mode, cs):
    from oracle import np_oracle as O
    kw = KW[mode]
    aug = O.AugConfig(rotation_range=(-5, 5)) if kw.get("enable_custom_augmentation") else O.AugConfig()
    return O.TransformConfig(mode=kw["mode"], crop_size=cs,
                             enable_custom_augmentation=bool(kw.get("enable_custom_augmentation")), aug=aug)


def cpu_port_clips_per_s(mode, t, h, w, cs, n_clips, threads):
    """Time the CPU port of the reference transform (oracle/torch_port.py) on ``n_clips`` clips, one process."""
    from oracle import torch_port as P
    from vision_collision_detection_b200.synth import make_clip_np
    torch.set_num_threads(threads)
    cfg = oracle_setup(mode, cs)
    clip = torch.from_numpy(make_clip_np(t, h, w, 0, "dashcam")).permute(3, 0, 1, 2)
    random.seed(1234)
    P.clip_transform(clip[:, :2], cfg, random)          # warm-up (thread pool, allocator)
    t0 = time.perf_counter()
    for _ in range(n_clips):
        P.clip_transform(clip, cfg, random)
    dt = time.perf_counter() - t0
    return n_clips / dt, dt


_WORKER_SRC = r"""
import os, sys, time, random
sys.path.insert(0, {root!r})
import torch
torch.set_num_threads({threads})
from oracle import torch_port as P, np_oracle as O
from vision_collision_detection_b200.synth import make_clip_np
mode, t, h, w, cs = {mode!r}, {t}, {h}, {w}, {cs}
aug = O.AugConfig(rotation_range=(-5, 5)) if mode == "custom" else O.AugConfig()
cfg = O.TransformConfig(mode="val" if mode == "val" else "train", crop_size=cs,
                        enable_custom_augmentation=(mode == "custom"), aug=aug)
clip = torch.from_numpy(make_clip_np(t, h, w, 0, "dashcam")).permute(3, 0, 1, 2)
random.seed(1234 + {wid})
P.clip_transform(clip[:, :2], cfg, random)
print("ready", flush=True)
for line in sys.stdin:                  # "go N": the start gun, every worker begins its N timed clips together
    parts = line.split()
    if not parts or parts[0] != "go":
        break
    t0 = time.time()
    for _ in range(int(parts[1])):
        P.clip_transform(clip, cfg, random)
    print("done %.6f %.6f" % (t0, time.time()), flush=True)
"""


class CpuWorkerPool:
    """The reference's deployment shape (nexar_complete_with_validation.py:49-51, nexar_train_distributed.py:97):
    ``n_workers`` DataLoader-style processes with OMP_NUM_THREADS=``threads`` each, every worker transforming its own clips."""

    def __init__(self, mode, t, h, w, cs, n_workers, threads):
        env = dict(os.environ, OMP_NUM_THREADS=str(threads), MKL_NUM_THREADS=str(threads))
        self.procs = []
        for wid in range(n_workers):
            src = _WORKER_SRC.format(root=ROOT, threads=threads, mode=mode, t=t, h=h, w=w, cs=cs, wid=wid)
            self.procs.append(subprocess.Popen([sys.executable, "-c", src], stdin=subprocess.PIPE, stdout=subprocess.PIPE,
                                               stderr=subprocess.DEVNULL, text=True, env=env))
        for p in self.procs:
            if not p.stdout.readline().startswith("ready"):
                self.close()
                raise RuntimeError("cpu worker failed to start")

    def run(self, clips_per_worker):
        """-> (aggregate clips/s, seconds) over the span from the common start to the last worker's finish."""
        for p in self.procs:
            p.stdin.write(f"go {clips_per_worker}\n")
            p.stdin.flush()
        t0s, t1s = [], []
        for p in self.procs:
            parts = p.stdout.readline().split()
            t0s.append(float(parts[1]))
            t1s.append(float(parts[2]))
        dt = max(t1s) - min(t0s)
        return len(self.procs) * clips_per_worker / dt, dt

    def close(self):
        for p in self.procs:
            try:
                p.stdin.close()
                p.wait(timeout=5)
            except Exception:  # noqa: BLE001
                p.kill()
        self.procs = []


def cpu_legs(mode, t, h, w, cs, budget_s=24.0):
    """BASELINE.md section 4's three CPU settings on this box, bounded to about ``budget_s`` seconds of wall time:
    (i) one process with every core as torch threads, (ii) P = cores/4 worker processes x 4 threads (the reference's
    real DataLoader deployment), (iii) one thread.  Returns (best value, legs dict)."""
    cores = os.cpu_count() or 1
    probe, dtp = cpu_port_clips_per_s(mode, t, h, w, cs, 1, cores)
    n_all = max(2, min(256, int(budget_s * 0.4 * probe)))
    all_cps, all_dt = cpu_port_clips_per_s(mode, t, h, w, cs, n_all, cores)
    legs = {"all_threads": {"value": all_cps, "procs": 1, "threads": cores, "clips": n_all, "seconds": round(all_dt, 2)}}
    nw = max(1, cores // 4)
    try:
        # a worker with 4 threads is roughly (4 / cores) of the all-thread rate or better; size for ~0.4 of the budget
        per_worker = max(1, int(budget_s * 0.4 * all_cps / nw * 1.5))
        pool = CpuWorkerPool(mode, t, h, w, cs, nw, 4)
        try:
            w_cps, w_dt = pool.run(per_worker)
        finally:
            pool.close()
        legs["workers"] = {"value": w_cps, "procs": nw, "threads": 4, "clips": nw * per_worker, "seconds": round(w_dt, 2),
                           "as": "nexar_complete_with_validation.py:49-51 (OMP_NUM_THREADS=4 per DataLoader worker)"}
    except Exception as e:  # noqa: BLE001
        legs["workers"] = {"value": None, "error": str(e)[:100]}
    n_one = max(1, min(16, int(budget_s * 0.15 * all_cps / max(1.0, cores / 3.0))))
    one_cps, one_dt = cpu_port_clips_per_s(mode, t, h, w, cs, n_one, 1)
    torch.set_num_threads(cores)
    legs["single_thread"] = {"value": one_cps, "procs": 1, "threads": 1, "clips": n_one, "seconds": round(one_dt, 2)}
    best = max((v for v in (legs["all_threads"]["value"], legs["workers"].get("value")) if v), default=all_cps)
    return best, legs


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path (the oracle port) on the host cores, rank 0 only.  Each step is a
    bounded sample of the workload; the faster of the two multi-core settings (all-thread process / cores/4 workers x 4
    threads, the reference's DataLoader shape) is the step's configuration, chosen in the warm-up."""
    if rank != 0:
        return
    b, t, h, w, cs = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    nw = max(1, cores // 4)
    probe, _ = cpu_port_clips_per_s(args.mode, t, h, w, cs, 1, cores)
    for _ in range(max(0, args.warmup - 1)):
        probe, _ = cpu_port_clips_per_s(args.mode, t, h, w, cs, 1, cores)
    pool = None
    try:
        pool = CpuWorkerPool(args.mode, t, h, w, cs, nw, 4)
        wprobe, _ = pool.run(1)
    except Exception:  # noqa: BLE001
        wprobe = 0.0
    use_workers = wprobe > probe
    rate = max(wprobe, probe)
    # bounded sample: the whole --steps run stays within about two minutes whatever K the driver passes
    per_step_s = min(20.0, 120.0 / max(1, args.steps))
    if use_workers:
        per_worker = max(1, int(per_step_s * rate / nw))
        sample_desc = f"{nw} worker processes x 4 threads, {per_worker} clip(s) of {t}x{h}x{w} each per step"
    else:
        sample = max(1, min(max(1, args.ref_clips), int(per_step_s * rate)))
        sample_desc = f"{sample} clip(s) of {t}x{h}x{w} per step, one process, torch threads={cores}"
    cps_runs = []
    t_all0 = time.perf_counter()
    for _ in range(args.steps):
        if use_workers:
            cps, _ = pool.run(per_worker)
        else:
            cps, _ = cpu_port_clips_per_s(args.mode, t, h, w, cs, sample, cores)
        cps_runs.append(cps)
    wall = time.perf_counter() - t_all0
    if pool is not None:
        pool.close()
    value = float(np.mean(cps_runs))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "clips/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload}:{args.mode} {t}x{h}x{w} u8 -> {cs}x{cs}", "out_dtype": "f32", "where": "host CPU",
                   "kwargs": "nexar_videos.py:2003-2010" if args.mode == "custom" else args.mode},
        "cpu_baseline": {"value": value, "unit": "clips/s", "cores": cores, "kind": "port", "sample": sample_desc,
                         "probe_all_threads": probe, "probe_workers": wprobe},
        "e2e": {"value": value, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_cfg4(args, rank, world, dev, out_dtype):
    """Inference windowing (BASELINE configs[3]): per-frame-once val transform of a 1200-frame 720p video; a "clip" is
    one 16-frame window.  The headline serves the windows as strided views of the per-frame result (stride 8, 149
    windows); the line also times the materialised [K,3,16,cs,cs] batches for stride 8 and stride 1 (SURVEY 8d)."""
    import torch.distributed as dist
    from vision_collision_detection_b200.engine import get_engine
    from vision_collision_detection_b200.inference import SlidingWindowTransform, sliding_window_starts
    from vision_collision_detection_b200.synth import make_clip_torch
    _, n, h, w, cs = WORKLOADS["cfg4"]
    video = torch.cat([make_clip_torch(100, h, w, seed=rank * 100 + i, kind="dashcam", device=dev) for i in range(n // 100)])
    steps = args.steps
    warm = max(3, args.warmup)

    def timed(fn):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            r = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / steps], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), r

    sw = SlidingWindowTransform(window=16, stride=8, out_dtype=out_dtype)
    ms, view = timed(lambda: sw.windows(video))
    dump = sample_outputs({"windows": view}) if args.dump_outputs and rank == 0 else None
    launches = get_engine(dev).last_launches
    ms_m8, m8 = timed(lambda: sw.windows(video, materialize=True))
    sw1 = SlidingWindowTransform(window=16, stride=1, out_dtype=out_dtype)
    ms_m1, m1 = timed(lambda: sw1.windows(video, materialize=True))
    esz0 = 2 if out_dtype == torch.bfloat16 else 4
    n_m8, bytes_m8, n_m1, bytes_m1 = int(m8.shape[0]), int(m8.numel() * esz0), int(m1.shape[0]), int(m1.numel() * esz0)
    del m8, m1
    # end to end: the decoded video sits in pinned HOST memory (what a CPU decoder leaves behind); its 75 consecutive
    # 16-frame chunks go through HostClipPipeline (H2D, val transform, D2H of the per-frame result), and the stride-8
    # windows are strided views of that host result
    e2e = None
    if not args.no_e2e:
        from vision_collision_detection_b200.host_pipeline import HostClipPipeline
        pipe = HostClipPipeline(sw.tf, n_clips=n // 16, frames=16, height=h, width=w, device=dev, out_dtype=out_dtype)
        host_video = pipe.pinned_input()
        host_video.copy_(video.view(n // 16, 16, h, w, 3).cpu())
        pipe.run(host_video)
        torch.cuda.synchronize()
        e_steps = 3
        t0 = time.perf_counter()
        for _ in range(e_steps):
            host_out = pipe.run(host_video)                       # [75,3,16,cs,cs] pinned
        ms_e = (time.perf_counter() - t0) * 1e3 / e_steps
        tms = torch.tensor([ms_e], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms_e = float(tms.item())
        e2e = {"value": world * len(sliding_window_starts(n, 16, 8)) / (ms_e * 1e-3), "unit": "clips/s", "source": "rgb",
               "ms_per_video": ms_e, "h2d_bytes_per_step": int(host_video.numel()),
               "d2h_bytes_per_step": int(host_out.numel() * host_out.element_size()), "steps": e_steps,
               "note": "PCIe-bound: 3.3 GB of uint8 frames per video"}
        del pipe, host_video
    if dump is not None:
        write_outputs(args.dump_outputs, dump)
    if rank == 0:
        peaks, kind = measured_peaks()
        k = len(sliding_window_starts(n, 16, 8))
        esz = 2 if out_dtype == torch.bfloat16 else 4
        bytes_alg = n * h * w * 3 + n * 3 * cs * cs * esz
        ach = bytes_alg / (ms * 1e-3) / 1e9
        print(json.dumps({
            "metric": METRIC, "value": world * k / (ms * 1e-3), "unit": "clips/s", "n_gpus": world, "steps": steps,
            "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": f"u8 -> i32 fixed-point (15-bit taps) / f32 -> {args.out_dtype}", "data": "synthetic",
            "config": {"workload": f"cfg4: {n} frames {h}x{w} u8 (40 s x 30 fps) -> val chain {cs}x{cs} {args.out_dtype}, every frame once, "
                                   f"{k} windows (= clips) of 16 at stride 8 as strided views", "windows_shape": list(view.shape),
                       "l2": f"input {n * h * w * 3 / 1e9:.1f} GB/step > 126 MB L2 (no flush needed)"},
            "ms_per_video": ms,
            "windows": {"views_stride8": {"ms": ms, "windows": k},
                        "materialised_stride8": {"ms": ms_m8, "windows": n_m8, "extra_bytes": bytes_m8,
                                                 "by": "nexar_gather_windows (whole-plane copies of the per-frame result)"},
                        "materialised_stride1": {"ms": ms_m1, "windows": n_m1, "extra_bytes": bytes_m1,
                                                 "by": "nexar_gather_windows (whole-plane copies of the per-frame result)"}},
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"],
                         "frac_of_8TBs_nominal": ach / 8000.0, "peak_kind": kind, "level": "step (every launch of the step)",
                         "algorithmic_bytes_per_step": bytes_alg, "traffic": None},
            "cpu_baseline": None, "e2e": e2e, "gpu_launches": launches * steps}), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--mode", default="custom", choices=sorted(KW))
    ap.add_argument("--out-dtype", default="bf16", choices=["bf16", "f32"])
    ap.add_argument("--ref-clips", type=int, default=8, help="clips per step for --impl reference (one-process setting)")
    ap.add_argument("--cpu-seconds", type=float, default=24.0, help="wall-time budget of the cpu_baseline legs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true", help="e2e legs: do not pin the rank to the GPU's NUMA-local CPUs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (float32, at most 64 MB in all: "
                         "a larger output is a fixed, seeded sample of whole rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup   # timing rules: W >= 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch.distributed as dist
    from vision_collision_detection_b200 import create_video_transforms
    from vision_collision_detection_b200.engine import get_engine
    from vision_collision_detection_b200.host_pipeline import HostClipPipeline
    from vision_collision_detection_b200.synth import make_clip_torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    b, t, h, w, cs = WORKLOADS[args.workload]
    scaling = "weak"
    if args.workload == "cfg3":
        # BASELINE configs[2] as written: ONE batch of 256 clips sharded over the GPUs (256 / 128 / 64 / 32 per GPU)
        if b % world:
            raise SystemExit(f"cfg3 shards {b} clips evenly: --gpus must divide {b}")
        b //= world
        scaling = "strong"
    out_dtype = torch.bfloat16 if args.out_dtype == "bf16" else torch.float32
    if args.workload == "cfg4":
        return run_cfg4(args, rank, world, dev, out_dtype)
    tf = create_video_transforms(**KW[args.mode], crop_size=cs, out_dtype=out_dtype)
    eng = get_engine(dev)
    if os.environ.get("NEXAR_FAST_BANDS"):
        from vision_collision_detection_b200 import _lib as _l
        _l.lib().nexar_set_fast_bands(int(os.environ["NEXAR_FAST_BANDS"]))
    if os.environ.get("NEXAR_CHUNK_CLIPS"):
        from vision_collision_detection_b200 import _lib as _l
        _l.lib().nexar_set_chunk_clips(int(os.environ["NEXAR_CHUNK_CLIPS"]))
    if os.environ.get("NEXAR_RESIZE_VARIANT"):      # experiments: 2 = the unfused K1 + K1.5 + K2 + K3 path
        from vision_collision_detection_b200 import _lib as _l
        _l.lib().nexar_set_resize_kernel(int(os.environ["NEXAR_RESIZE_VARIANT"]))

    # synthetic device-resident shard (1.4 GB for cfg2: larger than the 126 MB L2, so every step streams from HBM);
    # at most 32 distinct clips are synthesised, larger shards repeat them
    n_distinct = min(b, 32)
    clips = torch.empty((b, t, h, w, 3), dtype=torch.uint8, device=dev)
    for i in range(n_distinct):
        clips[i] = make_clip_torch(t, h, w, seed=rank * 1000 + i, kind="dashcam", device=dev)
    for i in range(n_distinct, b):
        clips[i] = clips[i % n_distinct]
    out = torch.empty((b, 3, t, cs, cs), dtype=out_dtype, device=dev)
    random.seed(1234 + rank)
    param_sets = [tf.sample_params(b, h, w) for _ in range(4)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(i):
        tf.forward_batch(clips, params=param_sets[i % len(param_sets)], out=out)

    # ---- device-resident timing ("value") ------------------------------------------------
    sampler = ClockSampler(local) if rank == 0 else None   # started early: nvidia-smi needs ~0.2 s to stream
    # Pre-heat (NOT steps of the transform): ~60 ms of plain torch copies so the SM clock has ramped before the W
    # warm-up steps the driver asked for; the warm-up itself is exactly --warmup steps (plan tables, workspace and the
    # pinned parameter ring are created in its first step).
    scratch = torch.empty_like(clips[: max(1, min(b, 8))])
    t_w = time.time()
    while time.time() - t_w < 0.06:
        scratch.copy_(clips[: scratch.shape[0]])
        torch.cuda.synchronize()
    del scratch
    for i in range(args.warmup):
        step(i)
    barrier()
    from vision_collision_detection_b200 import _lib
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    e0.record()
    for i in range(args.steps):
        step(i)
    t_enq = time.time()                  # the host has enqueued every step (the device is still working through them)
    e1.record()
    barrier()
    t_wall1 = time.time()
    last_out = out.clone() if args.dump_outputs and rank == 0 else None    # before the untimed steps below reuse out
    launches = eng.last_launches * args.steps
    ms_total = e0.elapsed_time(e1)
    if sampler is not None and sampler.proc is not None and sampler.count(t_wall0, t_wall1) < 3:
        # a short timed region (small --steps) can fall between two 100 ms samples: keep the SAME load running, untimed,
        # until the sampler has seen it (the clocks line then says how many samples came from the timed region itself)
        in_region = sampler.count(t_wall0, t_wall1)
        t_probe = time.time()
        while time.time() - t_probe < 0.8 and sampler.count(t_wall0, time.time()) < 3:
            for i in range(16):
                step(i)
            torch.cuda.synchronize()
        clocks = sampler.stop(t_wall0, time.time())
        if clocks is not None:
            clocks["samples_in_timed_region"] = in_region
    else:
        clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    tms = torch.tensor([ms_total], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_step = float(tms.item()) / args.steps
    # The resize kernel's own duration (sub-record of the roofline): an event pair recorded inside the library around
    # that launch, in a SEPARATE pass right after the timed region - the event between the kernels would switch off
    # the programmatic overlap of the colour kernel with the resize kernel's last wave in the timed steps themselves.
    k_steps = max(3, min(args.steps, 30))
    _lib.lib().nexar_profile_begin(64 * k_steps + 8)
    for i in range(k_steps):
        step(i)
    torch.cuda.synchronize()
    k1_ms = _lib.profile_end()
    value = world * b / (ms_step * 1e-3)

    # ---- end to end: pinned host clips -> H2D -> transform -> D2H (through the public host API) ----
    def run_e2e(pixel_format):
        """The same metric through HostClipPipeline with HOST buffers: every step copies its input clips from pinned
        host memory and reads the result back.  pixel_format "rgb": the uint8 RGB frames the reference's decoder
        delivers (44 MB per cfg2 clip); "nv12": decoder surfaces (22 MB per clip), converted on the device."""
        eb = min(b, 32)                            # host batch of the e2e leg (pinned memory: 22-88 MB per clip)
        pipe = HostClipPipeline(tf, n_clips=eb, frames=t, height=h, width=w, device=dev, pixel_format=pixel_format)
        host_in = pipe.pinned_input()
        if pixel_format == "nv12":
            from vision_collision_detection_b200.synth import rgb_to_nv12
            for i in range(eb):
                host_in[i].copy_(rgb_to_nv12(clips[i]).cpu())
        else:
            host_in.copy_(clips[:eb].cpu())
        e2e_steps = max(3, min(args.steps, 8))
        host_in2 = pipe.pinned_input()          # two input batches alternate: one is being copied while the next is "decoded"
        host_in2.copy_(host_in)
        ins = [host_in, host_in2]
        for i in range(2):
            pipe.run(ins[i & 1], params=param_sets[i % len(param_sets)][:eb])
        barrier()
        ts0 = time.perf_counter()
        e0.record()
        prev = None
        for i in range(e2e_steps):                # steady state: batch i+1 is submitted before batch i is collected
            ticket = pipe.submit(ins[i & 1], params=param_sets[i % len(param_sets)][:eb])
            if prev is not None:
                host_out = pipe.wait(prev)
            prev = ticket
        host_out = pipe.wait(prev)
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - ts0
        own_ms = max(e0.elapsed_time(e1), wall * 1e3) / e2e_steps
        barrier()
        ems = torch.tensor([own_ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ems, op=dist.ReduceOp.MAX)
        h2d_rank = torch.tensor([host_in.numel() / (own_ms * 1e-3) / 1e9], device=dev, dtype=torch.float64)
        h2d_all = [torch.zeros_like(h2d_rank) for _ in range(world)]
        if world > 1:
            dist.all_gather(h2d_all, h2d_rank)
        else:
            h2d_all = [h2d_rank]
        res = {"value": world * eb / (float(ems.item()) * 1e-3), "unit": "clips/s", "source": pixel_format,
               "h2d_bytes_per_step": int(host_in.numel()), "d2h_bytes_per_step": int(host_out.numel() * host_out.element_size()),
               "steps": e2e_steps, "clips_per_gpu_per_step": eb,
               "h2d_GBs_per_gpu": [round(float(x.item()), 2) for x in h2d_all],
               "h2d_GBs_aggregate": round(sum(float(x.item()) for x in h2d_all), 2)}
        del pipe, host_in, host_in2, ins
        return res

    e2e = e2e_nv12 = None
    if not args.no_e2e:
        from vision_collision_detection_b200.host_pipeline import bind_to_gpu_numa_node
        numa_cpus = None if args.no_numa_bind else bind_to_gpu_numa_node(local)   # before any pinned allocation of the leg
        e2e = run_e2e("rgb")
        e2e["numa_bound_cpus"] = len(numa_cpus) if numa_cpus else 0
        e2e["note"] = ("uint8 RGB over PCIe (the frames the reference's decoder delivers) bounds this leg; e2e_nv12 is the same "
                       "call fed with decoder surfaces (half the bytes), DESIGN.md F1")
        e2e_nv12 = run_e2e("nv12")
        if world > 1:
            e2e["note"] += ("; multi-GPU: h2d_GBs_per_gpu lists every rank's own rate - on a single-socket host the aggregate "
                            "saturates (about 190 GB/s on the 8 x B200 box of DESIGN.md section 6), which is what bounds this leg")

    if last_out is not None:
        write_outputs(args.dump_outputs, sample_outputs({"out": last_out}))
    if rank == 0:
        peaks, peak_kind = measured_peaks()
        per_clip = algorithmic_bytes_per_clip(t, h, w, cs, out.element_size())
        step_bytes = b * per_clip
        step_ach = step_bytes / (ms_step * 1e-3) / 1e9
        # dominant kernel: resize_fast_kernel (the only one that touches the source).  The sub-record divides the STEP's
        # algorithmic bytes (source read once + output written once) by that kernel's own duration, i.e. what the step
        # would reach if the colour / geometry kernels were free; the headline fraction below is the whole step.
        k_ms = (sum(k1_ms) / k_steps) if k1_ms else None   # per step: the sum over the chunks of a step
        kern = None
        if k_ms:
            k_ach = step_bytes / (k_ms * 1e-3) / 1e9
            kern = {"name": "resize_fast_kernel" + (" (then colour_kernel + geometry_spec_kernel)" if args.mode == "custom" else ""),
                    "ms": k_ms, "achieved": k_ach, "frac": k_ach / peaks["hbm_gbs"], "share_of_step": k_ms / ms_step,
                    "timed": f"CUDA event pair around the launch on its stream (nexar_profile_begin/end), {k_steps} extra steps right after the timed region"}
        # roofline.frac is STEP level (all launches of the step, device events): it is never better than the kernel's own
        traffic = ncu_traffic(args.workload, args.mode, args.out_dtype)
        if kern and traffic:
            kern["traffic"] = (traffic.get("kernels") or {}).get("resize_fast_kernel")
        roof = {"bound": "hbm", "achieved": step_ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": step_ach / peaks["hbm_gbs"],
                "frac_of_8TBs_nominal": step_ach / 8000.0, "peak_kind": peak_kind, "level": "step (every launch of the step)",
                "algorithmic_bytes_per_step": step_bytes, "kernel": kern,
                "traffic": (traffic or {}).get("step"), "traffic_by_kernel": (traffic or {}).get("kernels"),
                "traffic_source": "profiles/traffic.json (ncu dram bytes per launch of this command, committed)" if traffic else None}
        cpu = None
        if not args.no_cpu_baseline and world == 1:     # the CPU legs run on rank 0 of a single-GPU run only
            cores = os.cpu_count() or 1
            best, legs = cpu_legs(args.mode, t, h, w, cs, args.cpu_seconds)
            cpu = {"value": best, "unit": "clips/s", "cores": cores, "kind": "port",
                   "sample": f"oracle/torch_port.py on {t}x{h}x{w} clips; value = the faster multi-core setting; legs list clips and seconds",
                   "legs": legs}
        line = {
            "metric": METRIC, "value": value, "unit": "clips/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": f"u8 -> i32 fixed-point (15-bit taps) / f32 -> {args.out_dtype}", "data": "synthetic",
            "config": {"workload": f"{args.workload}:{args.mode} {t}x{h}x{w} u8 -> {cs}x{cs}", "out_dtype": args.out_dtype,
                       "clips_per_gpu_per_step": b, "where": "B200, inputs resident in HBM",
                       "kwargs": "nexar_videos.py:2003-2010" if args.mode == "custom" else args.mode,
                       "l2": f"input {b * t * h * w * 3 / 1e9:.1f} GB/step > 126 MB L2 (no flush needed)",
                       "sharding": f"{b} clips per GPU, no collective" + (" (one 256-clip batch split over the GPUs)" if scaling == "strong" else ""),
                       "preheat": "60 ms of torch copies before the warm-up (clock ramp; not transform steps)"},
            "output_GBs": world * b * 3 * t * cs * cs * out.element_size() / (ms_step * 1e-3) / 1e9,
            "host_enqueue_ms_per_step": 1e3 * (t_enq - t_wall0) / args.steps,
            "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "e2e_nv12": e2e_nv12, "gpu_launches": launches, "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
