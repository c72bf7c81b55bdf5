#!/usr/bin/env python
"""Image encoder + decoder throughput.
  --arch vit-h (default): BASELINE config #5 shape, random-init CLIP ViT-H/14-378 + default decoder on synthetic 378 x 378 images; one
      JSON line.  python tools/bench_encoder.py [--images 256] [--chunk 64] [--steps 2]
  --arch siglip-b16: the reference's default embedder, SigLIP ViT-B/16 on synthetic 224 x 224 images; one JSON line per measurement:
      the encoder alone at chunk sizes 64, 128 and 256 (or --chunk), then images -> labels with an F = 768 decoder, greedy and guided beam
      k = 10 (synthetic 43 000-target guide), at B = 256 and B = 1 (the two pipeline conditions of the paper's timing figures).  Every
      line carries the card's name and power limit, read in the same run.
  --arch siglip-so400m: the same lines for SigLIP SO400M/14 (the F = 1152 checkpoints' embedder) with an F = 1152 decoder."""
import argparse, dataclasses, json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
import torch
ap = argparse.ArgumentParser(); ap.add_argument("--images", type=int, default=None); ap.add_argument("--chunk", type=int, default=None)
ap.add_argument("--steps", type=int, default=None); ap.add_argument("--layers", type=int, default=None)
ap.add_argument("--arch", choices=("vit-h", "siglip-b16", "siglip-so400m"), default="vit-h"); args = ap.parse_args()
from novic_b200 import default_decoder, synth
from novic_b200.encoder import (SIGLIP_SO400M, EncoderDecoder, ImageEncoder, SiglipDims, SiglipImageEncoder, VitDims, synth_images,
                                synth_siglip_state_dict, synth_vit_state_dict)
dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0"))); torch.cuda.set_device(dev)
def timed(fn, n):
    fn(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n): out = fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / n, out
def tiled_images(n, d):
    img = synth_images(min(n, 64), d).to(dev)
    return img.repeat((n + img.shape[0] - 1) // img.shape[0], 1, 1, 1)[:n].contiguous()

if args.arch == "vit-h":
    args.images = args.images or 256; args.chunk = args.chunk or 64; args.steps = args.steps or 2
    d = VitDims(layers=args.layers or 32)
    enc = ImageEncoder(d, images_per_chunk=args.chunk)
    enc.load_state_dict(synth_vit_state_dict(d, seed=7)); enc = enc.to(dev).eval()
    dims = synth.DecoderDims()
    dec = default_decoder(dims, synth.synth_state_dict(dims, seed=1)).to(dev)
    both = EncoderDecoder(enc, dec)
    img = tiled_images(args.images, d)
    T, W, L, M = d.tokens, d.width, d.layers, d.mlp_dim
    flops_img = 2 * T * L * (4 * W * W + 2 * W * M) + 4 * T * T * W * L + 2 * (T - 1) * 588 * W
    with torch.inference_mode():
        enc_ms, e = timed(lambda: enc.encode_image(img, normalize=True), args.steps)
        all_ms, out = timed(lambda: both.generate(img), args.steps)
    print(json.dumps({"images": args.images, "chunk": args.chunk, "encoder_ms": enc_ms, "encoder_images_per_s": args.images / enc_ms * 1e3,
                      "encoder_tflops": flops_img * args.images / enc_ms / 1e9, "gflop_per_image": flops_img / 1e9,
                      "end_to_end_ms": all_ms, "end_to_end_images_per_s": args.images / all_ms * 1e3, "labels_shape": list(out[0].shape)}))
    sys.exit(0)

# ---- SigLIP ViT-B/16 and SO400M/14 ----
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(dev.index)], capture_output=True, text=True, check=True)
card, power = (s.strip() for s in q.stdout.strip().split(","))
preset = SiglipDims() if args.arch == "siglip-b16" else SIGLIP_SO400M
d = dataclasses.replace(preset, layers=args.layers or preset.layers)
n_img = args.images or 2048
steps = args.steps or 10
T, W, L, M, P = d.tokens, d.width, d.layers, d.mlp_dim, d.patch_size
# algorithmic work per image: trunk GEMMs (qkv, proj, fc1, fc2) 33.29 GFLOP, attention (QK^T and PV) 1.42, patch embedding 0.23,
# MAP head (kv over all tokens, then proj / fc1 / fc2 on one row) 0.47: 35.4 GFLOP at 224 x 224 for B/16; SO400M: 210.47 + 8.15 + 0.35
# + 1.38 = 220.3 GFLOP (the MLP counted at its 4304 channels, not the 4352 it runs padded to)
flops_trunk = 2 * T * L * (4 * W * W + 2 * W * M)
flops_attn = 4 * T * T * W * L
flops_patch = 2 * T * 3 * P * P * W
flops_head = 2 * T * W * 2 * W + 4 * T * W + 2 * W * W + 4 * W * M
flops_img = flops_trunk + flops_attn + flops_patch + flops_head
base = {"arch": args.arch, "card": card, "power_limit": power, "layers": L, "tokens": T, "gflop_per_image": flops_img / 1e9}
enc = SiglipImageEncoder(d)
enc.load_state_dict(synth_siglip_state_dict(d, seed=7)); enc = enc.to(dev).eval()
img = tiled_images(n_img, d)
with torch.inference_mode():
    for chunk in ([args.chunk] if args.chunk else [64, 128, 256]):
        enc.images_per_chunk = chunk
        ms, _ = timed(lambda: enc.encode_image(img, normalize=True), steps)
        print(json.dumps({**base, "what": "encoder", "images": n_img, "chunk": chunk, "steps": steps, "ms": ms,
                          "images_per_s": n_img / ms * 1e3, "tflops": flops_img * n_img / ms / 1e9}), flush=True)
    enc.images_per_chunk = args.chunk or 256
    dims = dataclasses.replace(synth.DecoderDims(), embed_dim=d.width)
    dec = default_decoder(dims, synth.synth_state_dict(dims, seed=1)).to(dev)
    both = EncoderDecoder(enc, dec)
    guide = synth.synth_guide_targets(43000, dims, seed=33).to(dev)
    for B in (256, 1):
        x = img[:B].contiguous()
        n = steps if B > 1 else 5 * steps
        for mode, fn in (("greedy", lambda: both.generate(x)),
                         ("guided_beam_k10", lambda: both.generate_beam(x, 10, 1.0, 0.0, None, False, 0.0, guide, False))):
            ms, _ = timed(fn, n)
            print(json.dumps({**base, "what": "images_to_labels", "mode": mode, "batch": B, "chunk": enc.images_per_chunk, "steps": n,
                              "ms": ms, "ms_per_image": ms / B, "images_per_s": B / ms * 1e3, "guide_targets": guide.shape[0] if "beam" in mode else 0}),
                  flush=True)
