"""Image encoder in front of the decoder (SURVEY.md section 8 row f3; BASELINE config #5: CLIP ViT-H/14-378 + decoder end to end).

The reference gets its image embeddings from `open_clip`'s `model.encode_image(images, normalize=False)` and normalises them in fp32
(embedders.py:752-764).  `ImageEncoder` offers the same call on the same parameter names (`visual.*` of open_clip's
`VisionTransformer`), computed by libnovic_b200.so (novic_vit_encode: tcgen05 GEMMs with fused bias / QuickGELU / residual epilogues,
tensor-core flash attention, LayerNorm kernels); `EncoderDecoder` hands the embeddings to `PrefixedIterDecoder.generate` without leaving
the device.  open_clip_torch is an un-vendored dependency of the reference, so the architecture is an assumption spelt out in
DESIGN.md and parity is pinned only on the independent restatement oracle/vit_oracle.py ("parity unpinned").  No CPU path.

`SiglipImageEncoder` does the same for the reference's default embedder, open_clip `ViT-B-16-SigLIP` (config/train.yaml:126; timm
`vit_base_patch16_siglip_224` with its MAP attention-pool head, parameters `visual.trunk.*`; 768-dim embeddings for the F = 768
decoder), on the same kernels (novic_siglip_create / novic_siglip_set_weights + novic_vit_encode); its architecture is equally an
assumption (DESIGN.md §5d, tests/siglip_oracle.py:encode_image_siglip).  With `SIGLIP_SO400M` it is open_clip `ViT-SO400M-14-SigLIP`
(timm `vit_so400m_patch14_siglip_224`: heads of 72, MLP 4304; 1152-dim embeddings for the F = 1152 checkpoints), assumed to be the same
architecture at those dimensions.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import math

import numpy as np
import torch
import torch.nn as nn

from . import _abi


@dataclasses.dataclass(frozen=True)
class VitDims:
    """open_clip `ViT-H-14-378-quickgelu` (DFN5B-CLIP-ViT-H-14-378, config/train.yaml:104) as assumed in DESIGN.md."""
    image_size: int = 378
    patch_size: int = 14
    width: int = 1280
    layers: int = 32
    heads: int = 16
    mlp_dim: int = 5120
    out_dim: int = 1024
    ln_eps: float = 1e-5

    @property
    def tokens(self) -> int:
        return (self.image_size // self.patch_size) ** 2 + 1


@dataclasses.dataclass(frozen=True)
class SiglipDims:
    """open_clip `ViT-B-16-SigLIP` (config/train.yaml:126, the reference's default embedder) as assumed in DESIGN.md §5d."""
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

    @property
    def out_dim(self) -> int:
        return self.width

    @property
    def head_dim(self) -> int:
        return self.width // self.heads


# open_clip `ViT-SO400M-14-SigLIP` (timm `vit_so400m_patch14_siglip_224`), the image embedder of the F = 1152 checkpoints, as assumed in
# DESIGN.md §5d
SIGLIP_SO400M = SiglipDims(image_size=224, patch_size=14, width=1152, layers=27, heads=16, mlp_dim=4304)


# ---- parameter holders: they exist so that state_dict() has open_clip's key names; none has a forward() ----
class _Mlp(nn.Module):
    def __init__(self, width, mlp_dim):
        super().__init__()
        self.c_fc = nn.Linear(width, mlp_dim)
        self.c_proj = nn.Linear(mlp_dim, width)


class _Block(nn.Module):
    def __init__(self, width, heads, mlp_dim, eps):
        super().__init__()
        self.ln_1 = nn.LayerNorm(width, eps=eps)
        self.attn = nn.MultiheadAttention(width, heads)      # holder of in_proj_weight / in_proj_bias / out_proj.{weight,bias}
        self.ln_2 = nn.LayerNorm(width, eps=eps)
        self.mlp = _Mlp(width, mlp_dim)


class _Blocks(nn.Module):
    def __init__(self, d: VitDims):
        super().__init__()
        self.resblocks = nn.ModuleList([_Block(d.width, d.heads, d.mlp_dim, d.ln_eps) for _ in range(d.layers)])


class _Visual(nn.Module):
    def __init__(self, d: VitDims):
        super().__init__()
        self.conv1 = nn.Conv2d(3, d.width, kernel_size=d.patch_size, stride=d.patch_size, bias=False)
        self.class_embedding = nn.Parameter(torch.empty(d.width))
        self.positional_embedding = nn.Parameter(torch.empty(d.tokens, d.width))
        self.ln_pre = nn.LayerNorm(d.width, eps=d.ln_eps)
        self.transformer = _Blocks(d)
        self.ln_post = nn.LayerNorm(d.width, eps=d.ln_eps)
        self.proj = nn.Parameter(torch.empty(d.width, d.out_dim))


class _NativeEncoder(nn.Module):
    """The handle, weight upload and encode call that ImageEncoder and SiglipImageEncoder share (one libnovic_b200 handle per device;
    weights re-uploaded whenever a parameter tensor is replaced or modified in place)."""

    def _weight_tensors(self) -> list[torch.Tensor]:
        raise NotImplementedError

    def _create(self, lib) -> C.c_void_p:
        raise NotImplementedError

    def _set_weights(self, lib, st: dict, tensors: list[torch.Tensor], stream: int) -> None:
        raise NotImplementedError

    def _state(self, device: torch.device) -> dict:
        if device.type != "cuda":
            raise RuntimeError(f"novic_b200.{type(self).__name__} computes on CUDA (sm_100a) only; there is no CPU path. Got tensors on {device}.")
        lib = _abi.lib()
        idx = device.index if device.index is not None else torch.cuda.current_device()
        st = self._handles.get(idx)
        with torch.cuda.device(idx):
            if st is None:
                st = dict(handle=self._create(lib), wbuf=None, wkey=None, ws=None)
                self._handles[idx] = st
            tensors = self._weight_tensors()
            wkey = tuple((t.data_ptr(), 0 if t.is_inference() else t._version) for t in tensors)
            if st["wkey"] != wkey:
                for t in tensors:
                    if t.device.type != "cuda" or t.device.index != idx or t.dtype != torch.float32 or not t.is_contiguous():
                        raise RuntimeError(f"encoder parameters must be contiguous fp32 tensors on the input's CUDA device (found {t.dtype} on {t.device})")
                if st["wbuf"] is None:
                    st["wbuf"] = torch.empty(lib.novic_vit_weight_bytes(st["handle"]), dtype=torch.uint8, device=device)
                self._set_weights(lib, st, tensors, torch.cuda.current_stream(idx).cuda_stream)
                st["wkey"] = wkey
        return st

    def encode_image(self, images: torch.Tensor, normalize: bool = False) -> torch.Tensor:
        """images [B, 3, S, S] fp32 (preprocessed) on the CUDA device -> [B, out_dim] fp32 (open_clip's encode_image)."""
        d = self.dims
        assert images.ndim == 4 and images.shape[1] == 3 and images.shape[2] == images.shape[3] == d.image_size and images.dtype == torch.float32
        images = images.contiguous()
        dev = images.device
        st = self._state(dev)
        lib = _abi.lib()
        B = images.shape[0]
        chunk = max(1, min(self.images_per_chunk, B))
        need = lib.novic_vit_workspace_bytes(st["handle"], chunk)
        if st["ws"] is None or st["ws"].numel() < need:
            st["ws"] = None
            st["ws"] = torch.empty(need, dtype=torch.uint8, device=dev)
        out = torch.empty((B, d.out_dim), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _abi.check(lib.novic_vit_encode(st["handle"], images.data_ptr(), B, out.data_ptr(), int(bool(normalize)), chunk, st["ws"].data_ptr(),
                                            st["ws"].numel(), torch.cuda.current_stream(dev).cuda_stream))
        return out

    def forward(self, images: torch.Tensor, normalize: bool = False) -> torch.Tensor:
        return self.encode_image(images, normalize)

    def __del__(self):
        try:
            lib = _abi.lib()
            for st in getattr(self, "_handles", {}).values():
                lib.novic_vit_destroy(st["handle"])
        except Exception:
            pass


class ImageEncoder(_NativeEncoder):
    def __init__(self, dims: VitDims = VitDims(), images_per_chunk: int = 64):
        super().__init__()
        if dims.width != dims.heads * 80 or dims.width not in (640, 1280):
            raise ValueError("ImageEncoder (novic_b200) supports heads of 80 channels and width 640 or 1280")
        if dims.layers > _abi.NOVIC_VIT_MAX_LAYERS:
            raise ValueError(f"at most {_abi.NOVIC_VIT_MAX_LAYERS} blocks")
        self.dims = dims
        self.images_per_chunk = int(images_per_chunk)
        self.visual = _Visual(dims)
        self.reset_parameters()
        self._handles: dict[int, dict] = {}

    @torch.no_grad()
    def reset_parameters(self) -> None:
        """Random initialisation in the style of CLIP's (scale = width^-0.5 for embeddings and projection, attention / MLP weights
        scaled by width and depth); the benchmark only needs well-conditioned random weights of the right shapes."""
        d = self.dims
        scale = d.width ** -0.5
        v = self.visual
        nn.init.normal_(v.conv1.weight, std=(3 * d.patch_size ** 2) ** -0.5)
        nn.init.normal_(v.class_embedding, std=scale)
        nn.init.normal_(v.positional_embedding, std=scale)
        nn.init.normal_(v.proj, std=scale)
        proj_std = scale * (2 * d.layers) ** -0.5
        for b in v.transformer.resblocks:
            nn.init.normal_(b.attn.in_proj_weight, std=scale)
            nn.init.normal_(b.attn.out_proj.weight, std=proj_std)
            nn.init.normal_(b.mlp.c_fc.weight, std=(2 * d.width) ** -0.5)
            nn.init.normal_(b.mlp.c_proj.weight, std=proj_std)
            for t in (b.attn.in_proj_bias, b.attn.out_proj.bias, b.mlp.c_fc.bias, b.mlp.c_proj.bias):
                nn.init.zeros_(t)

    def _weight_tensors(self) -> list[torch.Tensor]:
        v = self.visual
        ts = [v.conv1.weight, v.class_embedding, v.positional_embedding, v.ln_pre.weight, v.ln_pre.bias, v.ln_post.weight, v.ln_post.bias, v.proj]
        for b in v.transformer.resblocks:
            ts += [b.ln_1.weight, b.ln_1.bias, b.attn.in_proj_weight, b.attn.in_proj_bias, b.attn.out_proj.weight, b.attn.out_proj.bias,
                   b.ln_2.weight, b.ln_2.bias, b.mlp.c_fc.weight, b.mlp.c_fc.bias, b.mlp.c_proj.weight, b.mlp.c_proj.bias]
        return ts

    def _create(self, lib) -> C.c_void_p:
        d = self.dims
        cfg = _abi.NovicVitCfg(d.image_size, d.patch_size, d.width, d.layers, d.heads, d.mlp_dim, d.out_dim, d.ln_eps)
        handle = C.c_void_p()
        _abi.check(lib.novic_vit_create(C.byref(cfg), C.byref(handle)))
        return handle

    def _set_weights(self, lib, st: dict, tensors: list[torch.Tensor], stream: int) -> None:
        w = _abi.NovicVitWeights()
        (w.conv1, w.class_embedding, w.positional_embedding, w.ln_pre_w, w.ln_pre_b, w.ln_post_w, w.ln_post_b, w.proj) = (t.data_ptr() for t in tensors[:8])
        names = ("ln1_w", "ln1_b", "in_proj_w", "in_proj_b", "out_proj_w", "out_proj_b", "ln2_w", "ln2_b", "fc_w", "fc_b", "cproj_w", "cproj_b")
        for i in range(self.dims.layers):
            for j, name in enumerate(names):
                getattr(w, name)[i] = tensors[8 + 12 * i + j].data_ptr()
        _abi.check(lib.novic_vit_set_weights(st["handle"], C.byref(w), st["wbuf"].data_ptr(), st["wbuf"].numel(), stream))


# ---- SigLIP parameter holders: timm VisionTransformer / AttentionPoolLatent key names under open_clip's `visual.trunk`; no forward() ----
class _SigMlp(nn.Module):
    def __init__(self, width, mlp_dim):
        super().__init__()
        self.fc1 = nn.Linear(width, mlp_dim)
        self.fc2 = nn.Linear(mlp_dim, width)


class _SigAttn(nn.Module):
    def __init__(self, width):
        super().__init__()
        self.qkv = nn.Linear(width, 3 * width)
        self.proj = nn.Linear(width, width)


class _SigBlock(nn.Module):
    def __init__(self, width, mlp_dim, eps):
        super().__init__()
        self.norm1 = nn.LayerNorm(width, eps=eps)
        self.attn = _SigAttn(width)
        self.norm2 = nn.LayerNorm(width, eps=eps)
        self.mlp = _SigMlp(width, mlp_dim)


class _SigPatchEmbed(nn.Module):
    def __init__(self, d: SiglipDims):
        super().__init__()
        self.proj = nn.Conv2d(3, d.width, kernel_size=d.patch_size, stride=d.patch_size, bias=True)


class _SigAttnPool(nn.Module):
    def __init__(self, d: SiglipDims):
        super().__init__()
        self.latent = nn.Parameter(torch.empty(1, 1, d.width))
        self.q = nn.Linear(d.width, d.width)
        self.kv = nn.Linear(d.width, 2 * d.width)
        self.proj = nn.Linear(d.width, d.width)
        self.norm = nn.LayerNorm(d.width, eps=d.ln_eps)
        self.mlp = _SigMlp(d.width, d.mlp_dim)


class _SigTrunk(nn.Module):
    def __init__(self, d: SiglipDims):
        super().__init__()
        self.patch_embed = _SigPatchEmbed(d)
        self.pos_embed = nn.Parameter(torch.empty(1, d.tokens, d.width))
        self.blocks = nn.ModuleList([_SigBlock(d.width, d.mlp_dim, d.ln_eps) for _ in range(d.layers)])
        self.norm = nn.LayerNorm(d.width, eps=d.ln_eps)
        self.attn_pool = _SigAttnPool(d)


class _SigVisual(nn.Module):
    def __init__(self, d: SiglipDims):
        super().__init__()
        self.trunk = _SigTrunk(d)


class SiglipImageEncoder(_NativeEncoder):
    """open_clip `ViT-B-16-SigLIP` image tower (`visual.trunk.*` parameters) on libnovic_b200: encode_image(images, normalize) on
    preprocessed 224 x 224 images (resize and mean / std 0.5 stay with the caller) -> [B, width] fp32.  `SiglipImageEncoder(SIGLIP_SO400M)`
    is the `ViT-SO400M-14-SigLIP` tower.  Supported: heads of 64 or 72 channels, width 640, 768, 1024, 1152 or 1280, an MLP width that
    is a multiple of 16."""

    def __init__(self, dims: SiglipDims = SiglipDims(), images_per_chunk: int = 64):
        super().__init__()
        if dims.heads < 1 or dims.width % dims.heads or dims.head_dim not in (64, 72):
            raise ValueError("SiglipImageEncoder (novic_b200) supports heads of 64 or 72 channels only (width = heads * 64 or heads * 72)")
        if dims.width not in (640, 768, 1024, 1152, 1280):
            raise ValueError(f"SiglipImageEncoder: width {dims.width} has no LayerNorm kernel (640, 768, 1024, 1152, 1280)")
        if not 1 <= dims.layers <= _abi.NOVIC_VIT_MAX_LAYERS:
            raise ValueError(f"SiglipImageEncoder: between 1 and {_abi.NOVIC_VIT_MAX_LAYERS} blocks")
        if dims.patch_size < 1 or dims.image_size % dims.patch_size:
            raise ValueError("SiglipImageEncoder: image_size must be a multiple of patch_size")
        if dims.mlp_dim < 16 or dims.mlp_dim % 16:
            raise ValueError("SiglipImageEncoder: mlp_dim must be a multiple of 16")
        self.dims = dims
        self.images_per_chunk = int(images_per_chunk)
        self.visual = _SigVisual(dims)
        self.reset_parameters()
        self._handles: dict[int, dict] = {}

    @torch.no_grad()
    def reset_parameters(self) -> None:
        """Random initialisation (normal weights scaled by fan-in, zero biases, unit LayerNorms); the benchmark only needs
        well-conditioned random weights of the right shapes."""
        d = self.dims
        t = self.visual.trunk
        nn.init.normal_(t.patch_embed.proj.weight, std=(3 * d.patch_size ** 2) ** -0.5)
        nn.init.zeros_(t.patch_embed.proj.bias)
        nn.init.normal_(t.pos_embed, std=d.width ** -0.5)
        nn.init.normal_(t.attn_pool.latent, std=d.width ** -0.5)
        for m in self.modules():
            if isinstance(m, nn.Linear):
                nn.init.normal_(m.weight, std=m.in_features ** -0.5)
                nn.init.zeros_(m.bias)

    def _weight_tensors(self) -> list[torch.Tensor]:
        t = self.visual.trunk
        ap = t.attn_pool
        ts = [t.patch_embed.proj.weight, t.patch_embed.proj.bias, t.pos_embed, t.norm.weight, t.norm.bias, ap.latent, ap.q.weight, ap.q.bias,
              ap.kv.weight, ap.kv.bias, ap.proj.weight, ap.proj.bias, ap.norm.weight, ap.norm.bias, ap.mlp.fc1.weight, ap.mlp.fc1.bias,
              ap.mlp.fc2.weight, ap.mlp.fc2.bias]
        for b in t.blocks:
            ts += [b.norm1.weight, b.norm1.bias, b.attn.qkv.weight, b.attn.qkv.bias, b.attn.proj.weight, b.attn.proj.bias,
                   b.norm2.weight, b.norm2.bias, b.mlp.fc1.weight, b.mlp.fc1.bias, b.mlp.fc2.weight, b.mlp.fc2.bias]
        return ts

    def _create(self, lib) -> C.c_void_p:
        d = self.dims
        cfg = _abi.NovicSiglipCfg(d.image_size, d.patch_size, d.width, d.layers, d.heads, d.mlp_dim, d.ln_eps)
        handle = C.c_void_p()
        _abi.check(lib.novic_siglip_create(C.byref(cfg), C.byref(handle)))
        return handle

    def _set_weights(self, lib, st: dict, tensors: list[torch.Tensor], stream: int) -> None:
        w = _abi.NovicSiglipWeights()
        heads = ("patch_w", "patch_b", "pos_embed", "norm_w", "norm_b", "pool_latent", "pool_q_w", "pool_q_b", "pool_kv_w", "pool_kv_b",
                 "pool_proj_w", "pool_proj_b", "pool_norm_w", "pool_norm_b", "pool_fc1_w", "pool_fc1_b", "pool_fc2_w", "pool_fc2_b")
        for name, t in zip(heads, tensors):
            setattr(w, name, t.data_ptr())
        names = ("norm1_w", "norm1_b", "qkv_w", "qkv_b", "proj_w", "proj_b", "norm2_w", "norm2_b", "fc1_w", "fc1_b", "fc2_w", "fc2_b")
        n0 = len(heads)
        for i in range(self.dims.layers):
            for j, name in enumerate(names):
                getattr(w, name)[i] = tensors[n0 + 12 * i + j].data_ptr()
        _abi.check(lib.novic_siglip_set_weights(st["handle"], C.byref(w), st["wbuf"].data_ptr(), st["wbuf"].numel(), stream))


class EncoderDecoder(nn.Module):
    """Images -> labels on the device: Embedder.inference_image (embedders.py:759-764: encode_image(normalize=False) + fp32 normalise)
    followed by GenerationTask.generate's greedy call (infer.py:567-576) or its beam search (`generate_beam`; the reference's default
    generation config is guided beam k = 10, infer.py:55).  The encoder is an ImageEncoder or a SiglipImageEncoder whose output width
    is the decoder's embed_dim."""

    def __init__(self, encoder: ImageEncoder | SiglipImageEncoder, decoder):
        super().__init__()
        if encoder.dims.out_dim != decoder.embed_dim:
            raise ValueError(f"the encoder's embeddings have {encoder.dims.out_dim} channels but the decoder's embed_dim is {decoder.embed_dim}")
        self.encoder, self.decoder = encoder, decoder

    def embed(self, images: torch.Tensor) -> torch.Tensor:
        return self.encoder.encode_image(images, normalize=True)

    def generate(self, images: torch.Tensor, temperature: float = 1.0, length_alpha: float = 0.0, guide_targets=None, guide_renorm: bool = False):
        target, padding, _, _, _, score = self.decoder.generate(self.embed(images), False, True, temperature, length_alpha, None, guide_targets, guide_renorm)
        return target.unsqueeze(1), padding.unsqueeze(1), score.unsqueeze(1)

    def generate_beam(self, images: torch.Tensor, topk: int, temperature: float = 1.0, length_alpha: float = 0.0, vocab_targets=None,
                      vocab_per_token: bool = False, vocab_scaler: float = 0.0, guide_targets=None, guide_renorm: bool = False):
        """Beam search on the images' normalised embeddings: PrefixedIterDecoder.generate_beam's (target, padding, score)."""
        return self.decoder.generate_beam(self.embed(images), topk, temperature, length_alpha, vocab_targets, vocab_per_token, vocab_scaler,
                                          guide_targets, guide_renorm)


def synth_vit_state_dict(dims: VitDims = VitDims(), seed: int = 7) -> dict:
    """Random `visual.*` state dict, reproducible from (seed, shape) alone (numpy PCG64): CLIP-style scales, LayerNorm gains jittered
    around 1 and small non-zero biases everywhere so that a kernel that forgot one of them is caught."""
    rng = np.random.default_rng(seed)
    W, L, M, O, T, P = dims.width, dims.layers, dims.mlp_dim, dims.out_dim, dims.tokens, dims.patch_size
    scale = W ** -0.5
    proj_std = scale * (2 * L) ** -0.5

    def n(shape, std):
        return torch.from_numpy((rng.standard_normal(shape) * std).astype(np.float32))

    def gain(k):
        return torch.from_numpy((1.0 + 0.2 * rng.standard_normal(k)).astype(np.float32))
    sd = {"visual.conv1.weight": n((W, 3, P, P), (3 * P * P) ** -0.5), "visual.class_embedding": n((W,), scale),
          "visual.positional_embedding": n((T, W), scale), "visual.ln_pre.weight": gain(W), "visual.ln_pre.bias": n((W,), 0.05),
          "visual.ln_post.weight": gain(W), "visual.ln_post.bias": n((W,), 0.05), "visual.proj": n((W, O), scale)}
    for i in range(L):
        p = f"visual.transformer.resblocks.{i}."
        sd[p + "ln_1.weight"] = gain(W); sd[p + "ln_1.bias"] = n((W,), 0.05)
        sd[p + "attn.in_proj_weight"] = n((3 * W, W), scale * 2.0); sd[p + "attn.in_proj_bias"] = n((3 * W,), 0.05)
        sd[p + "attn.out_proj.weight"] = n((W, W), proj_std * 4.0); sd[p + "attn.out_proj.bias"] = n((W,), 0.02)
        sd[p + "ln_2.weight"] = gain(W); sd[p + "ln_2.bias"] = n((W,), 0.05)
        sd[p + "mlp.c_fc.weight"] = n((M, W), (2 * W) ** -0.5 * 2.0); sd[p + "mlp.c_fc.bias"] = n((M,), 0.05)
        sd[p + "mlp.c_proj.weight"] = n((W, M), proj_std * 4.0); sd[p + "mlp.c_proj.bias"] = n((W,), 0.02)
    return sd


def synth_siglip_state_dict(dims: SiglipDims = SiglipDims(), seed: int = 7) -> dict:
    """Random `visual.trunk.*` state dict for SiglipImageEncoder, reproducible from (seed, shape) alone (numpy PCG64): fan-in scales,
    LayerNorm gains jittered around 1 and non-zero biases everywhere (the patch convolution's and the latent query's included) so that a
    kernel that forgot one of them is caught."""
    rng = np.random.default_rng(seed)
    W, L, M, T, P = dims.width, dims.layers, dims.mlp_dim, dims.tokens, dims.patch_size
    scale = W ** -0.5

    def n(shape, std):
        return torch.from_numpy((rng.standard_normal(shape) * std).astype(np.float32))

    def gain(k):
        return torch.from_numpy((1.0 + 0.2 * rng.standard_normal(k)).astype(np.float32))
    t = "visual.trunk."
    sd = {t + "patch_embed.proj.weight": n((W, 3, P, P), (3 * P * P) ** -0.5), t + "patch_embed.proj.bias": n((W,), 0.05),
          t + "pos_embed": n((1, T, W), scale)}
    for i in range(L):
        p = f"{t}blocks.{i}."
        sd[p + "norm1.weight"] = gain(W); sd[p + "norm1.bias"] = n((W,), 0.05)
        sd[p + "attn.qkv.weight"] = n((3 * W, W), scale * 2.0); sd[p + "attn.qkv.bias"] = n((3 * W,), 0.05)
        sd[p + "attn.proj.weight"] = n((W, W), scale * 0.5); sd[p + "attn.proj.bias"] = n((W,), 0.02)
        sd[p + "norm2.weight"] = gain(W); sd[p + "norm2.bias"] = n((W,), 0.05)
        sd[p + "mlp.fc1.weight"] = n((M, W), scale * 2.0); sd[p + "mlp.fc1.bias"] = n((M,), 0.05)
        sd[p + "mlp.fc2.weight"] = n((W, M), M ** -0.5 * 0.5); sd[p + "mlp.fc2.bias"] = n((W,), 0.02)
    sd[t + "norm.weight"] = gain(W); sd[t + "norm.bias"] = n((W,), 0.05)
    a = t + "attn_pool."
    sd[a + "latent"] = n((1, 1, W), 0.5)
    sd[a + "q.weight"] = n((W, W), scale * 2.0); sd[a + "q.bias"] = n((W,), 0.05)
    sd[a + "kv.weight"] = n((2 * W, W), scale * 2.0); sd[a + "kv.bias"] = n((2 * W,), 0.05)
    sd[a + "proj.weight"] = n((W, W), scale); sd[a + "proj.bias"] = n((W,), 0.05)
    sd[a + "norm.weight"] = gain(W); sd[a + "norm.bias"] = n((W,), 0.05)
    sd[a + "mlp.fc1.weight"] = n((M, W), scale * 2.0); sd[a + "mlp.fc1.bias"] = n((M,), 0.05)
    sd[a + "mlp.fc2.weight"] = n((W, M), M ** -0.5); sd[a + "mlp.fc2.bias"] = n((W,), 0.05)
    return sd


def synth_images(batch: int, dims: VitDims | SiglipDims = VitDims(), seed: int = 11) -> torch.Tensor:
    """Synthetic preprocessed images (zero mean, unit variance per channel, with some spatial structure)."""
    rng = np.random.default_rng(seed)
    S = dims.image_size
    base = rng.standard_normal((batch, 3, S // 7 + 1, S // 7 + 1)).astype(np.float32)
    img = np.repeat(np.repeat(base, 7, axis=2), 7, axis=3)[:, :, :S, :S]
    img = 0.7 * img + 0.7 * rng.standard_normal((batch, 3, S, S)).astype(np.float32)
    return torch.from_numpy(np.ascontiguousarray(img))
