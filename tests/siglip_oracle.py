"""CPU restatement of the SigLIP ViT-B/16 image encoder - PARITY UNPINNED.

The reference's default embedder (config/train.yaml:126) is open_clip `ViT-B-16-SigLIP`, called as `model.encode_image(images,
normalize=False)` followed by an fp32 normalise (embedders.py:759-764).  open_clip and timm are neither vendored nor installed, so
`encode_image_siglip` restates the architecture from memory (an assumption the repository cannot verify offline): `TimmModel` around
timm `vit_base_patch16_siglip_224` with timm_pool='map' and timm_proj='none':

    x = patch_embed.proj(image) + pos_embed        # 16 x 16 conv WITH bias; 14 x 14 = 196 tokens, no class token, no ln_pre
    for block in blocks:                           # pre-LN
        x = x + attn.proj(attn(norm1(x)))          # qkv [3 width, width] + bias, q; k; v head-major; 12 heads of 64, scale 1/8, no mask
        x = x + mlp.fc2(gelu(mlp.fc1(norm2(x))))   # exact erf GELU (timm's nn.GELU; big_vision's original uses the tanh form)
    x = norm(x)                                    # on ALL tokens
    # MAP head, timm AttentionPoolLatent
    q = attn_pool.q(attn_pool.latent)              # one query, the same for every image
    k, v = attn_pool.kv(x).chunk(2)                # [2 width, width] + bias, k first
    y = attn_pool.proj(softmax(q k^T / 8) v)       # per head
    return y + attn_pool.mlp.fc2(gelu(attn_pool.mlp.fc1(attn_pool.norm(y))))    # 768 wide, no projection after it

with width 768, 12 blocks, MLP 3072 (blocks and head), LayerNorm eps 1e-6, keys `visual.trunk.*`.
Written in the style of oracle/vit_oracle.py (the ViT-H restatement).  TEST INFRASTRUCTURE ONLY: nothing under novic_b200/ imports
this module.
"""
from __future__ import annotations

import dataclasses
import math

import torch
import torch.nn.functional as F


@dataclasses.dataclass(frozen=True)
class SiglipCfg:
    image_size: int = 224
    patch_size: int = 16
    width: int = 768
    layers: int = 12
    heads: int = 12
    mlp_dim: int = 3072
    ln_eps: float = 1e-6

    @property
    def tokens(self) -> int:
        return (self.image_size // self.patch_size) ** 2


def encode_image_siglip(cfg: SiglipCfg, sd: dict, images: torch.Tensor, normalize: bool = False, bf16_operands: bool = False) -> torch.Tensor:
    """images [B, 3, S, S] fp32 -> [B, width] fp32 (see the module docstring).
    bf16_operands: round where the CUDA path holds bf16 - the weights of every GEMM, LayerNorm outputs, the qkv and kv rows, the trunk's
    attention probabilities (un-normalised, as the flash kernel does) and outputs, the MLP hidden rows, and the pooled attention rows of
    the head.  The head's latent query and its softmax stay fp32, as in the kernels."""
    r = (lambda t: t.bfloat16().float()) if bf16_operands else (lambda t: t)
    B = images.shape[0]
    W, H = cfg.width, cfg.heads
    D = W // H
    t = "visual.trunk."

    def ln(x, name):
        return F.layer_norm(x, (W,), sd[name + ".weight"], sd[name + ".bias"], cfg.ln_eps)
    x = F.conv2d(r(images), r(sd[t + "patch_embed.proj.weight"]), sd[t + "patch_embed.proj.bias"], stride=cfg.patch_size)
    x = x.reshape(B, W, -1).permute(0, 2, 1) + sd[t + "pos_embed"]
    T = x.shape[1]
    for i in range(cfg.layers):
        p = f"{t}blocks.{i}."
        y = r(ln(x, p + "norm1"))
        qkv = r(F.linear(y, r(sd[p + "attn.qkv.weight"]), sd[p + "attn.qkv.bias"]))
        q, k, v = (u.reshape(B, T, H, D).transpose(1, 2) for u in qkv.chunk(3, dim=-1))
        sc = q @ k.transpose(-1, -2) / math.sqrt(D)
        if bf16_operands:
            e = torch.exp(sc - sc.amax(dim=-1, keepdim=True))
            att = (r(e) @ v) / e.sum(dim=-1, keepdim=True)
        else:
            att = torch.softmax(sc, dim=-1) @ v
        att = r(att.transpose(1, 2).reshape(B, T, W))
        x = x + F.linear(att, r(sd[p + "attn.proj.weight"]), sd[p + "attn.proj.bias"])
        y = r(ln(x, p + "norm2"))
        h = r(F.gelu(F.linear(y, r(sd[p + "mlp.fc1.weight"]), sd[p + "mlp.fc1.bias"])))
        x = x + F.linear(h, r(sd[p + "mlp.fc2.weight"]), sd[p + "mlp.fc2.bias"])
    y = r(ln(x, t + "norm"))
    a = t + "attn_pool."
    q = F.linear(sd[a + "latent"].reshape(1, W), sd[a + "q.weight"], sd[a + "q.bias"]).reshape(1, H, 1, D)
    kv = r(F.linear(y, r(sd[a + "kv.weight"]), sd[a + "kv.bias"]))
    k, v = (u.reshape(B, T, H, D).transpose(1, 2) for u in kv.chunk(2, dim=-1))
    o = torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(D), dim=-1) @ v                          # B x H x 1 x D
    o = r(o.transpose(1, 2).reshape(B, W))
    out = F.linear(o, r(sd[a + "proj.weight"]), sd[a + "proj.bias"])
    h = r(F.gelu(F.linear(r(ln(out, a + "norm")), r(sd[a + "mlp.fc1.weight"]), sd[a + "mlp.fc1.bias"])))
    out = out + F.linear(h, r(sd[a + "mlp.fc2.weight"]), sd[a + "mlp.fc2.bias"])
    return F.normalize(out, dim=-1) if normalize else out
