#!/usr/bin/env python
"""BASELINE config 5: augmentation share of a DDP training step.

A minimal consumer with the reference model's input contract (nexar_arch.py:390-443: [B,3,T,H,W] in,
every other frame when T > 10, per-frame torchvision backbone, temporal GRU, 3-class head; random init)
is trained for a few steps under fp16 autocast on synthetic device-resident uint8 clips that go through
the fused GPU augmentation.  Reports t_aug / t_step from CUDA events (max over ranks).  The model is
library code (torchvision / cuDNN) and is NOT part of the product; this script only measures how much of
a real step the transform now costs.

  python tools/train_step_share.py [--batch 8] [--frames 16] [--steps 10] [--out-dtype f32|f16]
  python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/train_step_share.py
"""
import argparse
import json
import os
import random
import sys

import torch
import torch.distributed as dist
import torch.nn as nn

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vision_collision_detection_b200 import create_video_transforms  # noqa: E402
from vision_collision_detection_b200.synth import make_clip_torch  # noqa: E402


class FrameCnnGru(nn.Module):
    def __init__(self, num_classes=3):
        super().__init__()
        import torchvision
        self.backbone = torchvision.models.convnext_tiny(weights=None)
        dim = self.backbone.classifier[-1].in_features
        self.backbone.classifier[-1] = nn.Identity()
        self.gru = nn.GRU(dim, 256, batch_first=True, bidirectional=True)
        self.head = nn.Sequential(nn.Linear(512, 256), nn.ReLU(), nn.Dropout(0.5), nn.Linear(256, num_classes))

    def forward(self, x):                       # [B,3,T,H,W]
        b, c, t, h, w = x.shape
        if t > 10:
            x = x[:, :, ::2]
            t = x.shape[2]
        f = self.backbone(x.permute(0, 2, 1, 3, 4).reshape(b * t, c, h, w)).reshape(b, t, -1)
        out, _ = self.gru(f)
        return self.head(out.mean(dim=1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out-dtype", default="f32", choices=["f32", "f16"],
                    help="transform output: f16 is what autocast makes of the f32 output, at half the bytes")
    ap.add_argument("--sync-every-step", action="store_true", help="synchronize after every step (unoverlapped transform latency)")
    args = ap.parse_args()
    rank, world, local = (int(os.environ.get(k, d)) for k, d in (("RANK", 0), ("WORLD_SIZE", 1), ("LOCAL_RANK", 0)))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    model = FrameCnnGru().to(dev)
    if world > 1:
        model = nn.parallel.DistributedDataParallel(model, device_ids=[local])
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4)
    scaler = torch.amp.GradScaler("cuda")
    tf = create_video_transforms(mode="train", enable_custom_augmentation=True, brightness_range=(0.9, 1.1),
                                 contrast_range=(0.9, 1.1), saturation_range=(0.9, 1.1), rotation_range=(-5, 5))
    clips = torch.stack([make_clip_torch(args.frames, 720, 1280, rank * 100 + i, "dashcam", dev) for i in range(args.batch)])
    labels = torch.randint(0, 3, (args.batch,), device=dev)
    random.seed(1234 + rank)
    # One event triple per step and a single synchronize at the end: like a real training loop the host runs ahead of the
    # device, so ev[0] -> ev[1] is the time the DEVICE spends on the transform inside a step (the host-side parameter
    # packing of step i+1 overlaps the model's kernels of step i); --sync-every-step gives the unoverlapped latency instead.
    out_dtype = {"f32": torch.float32, "f16": torch.float16}[args.out_dtype]
    n_total = args.warmup + args.steps
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(n_total)]
    for i in range(n_total):
        ev = evs[i]
        ev[0].record()
        x = tf.forward_batch(clips, out_dtype=out_dtype)              # [B,3,T,224,224]
        ev[1].record()
        with torch.autocast("cuda", dtype=torch.float16):
            loss = nn.functional.cross_entropy(model(x), labels)
        opt.zero_grad(set_to_none=True)
        scaler.scale(loss).backward()
        scaler.step(opt)
        scaler.update()
        ev[2].record()
        if args.sync_every_step:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    t_aug = sum(ev[0].elapsed_time(ev[1]) for ev in evs[args.warmup:])
    t_step = evs[args.warmup][0].elapsed_time(evs[-1][2])            # wall time of the timed steps on the device
    t = torch.tensor([t_aug, t_step], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        a, s = (t / args.steps).tolist()
        print(json.dumps({"config": "cfg5: convnext_tiny+GRU (random init), fp16 autocast, AdamW, DDP" if world > 1 else
                          "cfg5 (1 GPU): convnext_tiny+GRU (random init), fp16 autocast, AdamW",
                          "model": "stand-in with the input contract and layer types of nexar_arch.EnhancedFrameCNN('convnext_tiny', "
                                   "temporal_mode='gru') (nexar_arch.py:390-443), built from torchvision; NOT the reference class",
                          "aug": "nexar_videos.py:2003-2010 kwargs, device-resident uint8 720p clips -> "
                                 f"{'fp32' if args.out_dtype == 'f32' else 'fp16'} [B,3,T,224,224]",
                          "n_gpus": world, "batch_per_gpu": args.batch, "frames": args.frames,
                          "ms_aug": a, "ms_step": s, "aug_share": a / s, "sync_every_step": bool(args.sync_every_step), "clips_per_s": world * args.batch / (s * 1e-3)}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
