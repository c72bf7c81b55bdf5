#!/usr/bin/env python
"""Kernel-time breakdown of the SigLIP image encoder with torch.profiler (CUDA activities): one chunk of --images images (default 256,
one chunk) encoded --steps times after a warm-up pass; prints device time per kernel per encode, its share, and the card's name and
power limit.  Run it apart from tools/bench_encoder.py: tracing slows the host.
  python tools/profile_encoder.py [--arch siglip-so400m|siglip-b16] [--images 256] [--steps 3]"""
import argparse, dataclasses, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
import torch
from torch.profiler import ProfilerActivity, profile
ap = argparse.ArgumentParser(); ap.add_argument("--arch", choices=("siglip-b16", "siglip-so400m"), default="siglip-so400m")
ap.add_argument("--images", type=int, default=256); ap.add_argument("--steps", type=int, default=3); args = ap.parse_args()
from novic_b200.encoder import SIGLIP_SO400M, SiglipDims, SiglipImageEncoder, synth_images, synth_siglip_state_dict
dev = torch.device("cuda", 0); torch.cuda.set_device(dev)
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, check=True)
d = SiglipDims() if args.arch == "siglip-b16" else SIGLIP_SO400M
enc = SiglipImageEncoder(d, images_per_chunk=args.images)
enc.load_state_dict(synth_siglip_state_dict(d, seed=7)); enc = enc.to(dev).eval()
img = synth_images(args.images, d).to(dev)
with torch.inference_mode():
    enc.encode_image(img, normalize=True); torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.steps): enc.encode_image(img, normalize=True)
        torch.cuda.synchronize()
rows = [(e.key, e.self_device_time_total / args.steps, e.count // args.steps) for e in prof.key_averages() if e.self_device_time_total > 0]
rows.sort(key=lambda r: -r[1])
total = sum(r[1] for r in rows)
print(f"{args.arch}: {args.images} images in one chunk, {q.stdout.strip()} (card, power limit); device time per encode {total / 1e3:.2f} ms")
print(f"{'us / encode':>12} {'share':>6} {'launches':>8}  kernel")
for name, us, n in rows:
    print(f"{us:12.1f} {100 * us / total:5.1f}% {n:8d}  {name[:150]}")
