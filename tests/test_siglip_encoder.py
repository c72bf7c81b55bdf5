"""SigLIP ViT-B/16 image encoder (the reference's default embedder, config/train.yaml:126) against the independent CPU restatement
tests/siglip_oracle.py:encode_image_siglip.

PARITY UNPINNED: open_clip_torch and timm are un-vendored dependencies of the reference, so the oracle restates the architecture from
memory (DESIGN.md §5d) and cannot be checked against the reference here.  What the GPU tests establish is that the CUDA path computes
that architecture: bf16 operands / fp32 accumulation and residual stream against fp32 on the CPU, with the tolerances of
tests/test_gpu_encoder.py - ||got - ref|| / ||ref|| <= 2 % after two blocks, <= 3 % after all twelve, no element off by more than six
times that, cosine >= 0.999, and <= 0.8 % against the restatement whose matrix-product operands are rounded to bf16.  The `b16_67_images`
tests run a production-sized chunk (every trunk GEMM on CTA pairs, tests/encoder_chunks.py): sampled images within the two-block bounds,
the same bits as chunks of two, under NOVIC_VIT_BN=256 / 128 and NOVIC_VIT_DIRECT=0, and on a workspace poisoned with 0xFF.
"""
import ctypes as C
import dataclasses
import os
import re

import pytest
import torch

from novic_b200 import _abi, default_decoder, synth
from novic_b200.encoder import EncoderDecoder, SiglipDims, SiglipImageEncoder, synth_images, synth_siglip_state_dict
from tests import siglip_oracle as vo
from tests.encoder_chunks import poisoned_workspace, production_chunk, same_under_switches

DEV = "cuda:0"
HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "novic_b200.h")
SMALL = SiglipDims(image_size=96, layers=2)        # 6 x 6 = 36 tokens


def expected_shapes(d: SiglipDims) -> dict:
    W, M, P, T = d.width, d.mlp_dim, d.patch_size, d.tokens
    t = "visual.trunk."
    s = {t + "patch_embed.proj.weight": (W, 3, P, P), t + "patch_embed.proj.bias": (W,), t + "pos_embed": (1, T, W),
         t + "norm.weight": (W,), t + "norm.bias": (W,)}
    for i in range(d.layers):
        p = f"{t}blocks.{i}."
        s.update({p + "norm1.weight": (W,), p + "norm1.bias": (W,), p + "attn.qkv.weight": (3 * W, W), p + "attn.qkv.bias": (3 * W,),
                  p + "attn.proj.weight": (W, W), p + "attn.proj.bias": (W,), p + "norm2.weight": (W,), p + "norm2.bias": (W,),
                  p + "mlp.fc1.weight": (M, W), p + "mlp.fc1.bias": (M,), p + "mlp.fc2.weight": (W, M), p + "mlp.fc2.bias": (W,)})
    a = t + "attn_pool."
    s.update({a + "latent": (1, 1, W), a + "q.weight": (W, W), a + "q.bias": (W,), a + "kv.weight": (2 * W, W), a + "kv.bias": (2 * W,),
              a + "proj.weight": (W, W), a + "proj.bias": (W,), a + "norm.weight": (W,), a + "norm.bias": (W,),
              a + "mlp.fc1.weight": (M, W), a + "mlp.fc1.bias": (M,), a + "mlp.fc2.weight": (W, M), a + "mlp.fc2.bias": (W,)})
    return s


@pytest.mark.parametrize("d", [SiglipDims(), SMALL], ids=["b16", "small"])
def test_state_dict_keys_and_shapes_follow_open_clip(d):
    want = expected_shapes(d)
    enc = SiglipImageEncoder(d)
    assert {k: tuple(v.shape) for k, v in enc.state_dict().items()} == want
    sd = synth_siglip_state_dict(d, seed=3)
    assert {k: tuple(v.shape) for k, v in sd.items()} == want
    enc.load_state_dict(sd, strict=True)
    assert torch.equal(enc.visual.trunk.attn_pool.latent, sd["visual.trunk.attn_pool.latent"])
    # every bias and the latent are non-zero, every LayerNorm gain differs from 1: a forgotten term shows in the GPU tests
    assert all(v.abs().min() > 0 for k, v in sd.items() if k.endswith(".bias") or k.endswith("latent"))
    assert all((v - 1).abs().max() > 0.1 for k, v in sd.items() if "norm" in k and k.endswith(".weight"))


@pytest.mark.parametrize("kw", [dict(heads=16), dict(width=512, heads=8), dict(layers=_abi.NOVIC_VIT_MAX_LAYERS + 1), dict(layers=0),
                                dict(image_size=100), dict(mlp_dim=3000)],
                         ids=["head_dim_48", "width_512", "too_many_layers", "no_layers", "ragged_patches", "mlp_3000"])
def test_unsupported_dims_are_rejected(kw):
    with pytest.raises(ValueError):
        SiglipImageEncoder(dataclasses.replace(SiglipDims(), **kw))


def test_cpu_tensors_have_no_cpu_path():
    with pytest.raises(RuntimeError, match="no CPU path"):
        SiglipImageEncoder(SMALL).encode_image(synth_images(1, SMALL))


def _header_struct(name: str) -> list[tuple[str, bool]]:
    """(field, is_array) in declaration order of `typedef struct name {...} name;` in include/novic_b200.h"""
    text = open(HEADER).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        decl = re.sub(r"^(const\s+)?(float|int32_t)\s*", "", decl)
        for part in decl.split(","):
            part = part.strip().lstrip("*").strip()
            arr = part.endswith("[NOVIC_VIT_MAX_LAYERS]")
            fields.append((part.replace("[NOVIC_VIT_MAX_LAYERS]", ""), arr))
    return fields


def test_ctypes_structs_match_the_header():
    for cls, name in ((_abi.NovicSiglipCfg, "NovicSiglipCfg"), (_abi.NovicSiglipWeights, "NovicSiglipWeights")):
        got = [(f, issubclass(t, C.Array)) for f, t in cls._fields_]
        assert got == _header_struct(name)
    assert C.sizeof(_abi.NovicSiglipCfg) == 7 * 4
    assert C.sizeof(_abi.NovicSiglipWeights) == 8 * (18 + 12 * _abi.NOVIC_VIT_MAX_LAYERS)


# ---------------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------------
def _cfg(d: SiglipDims) -> vo.SiglipCfg:
    return vo.SiglipCfg(**dataclasses.asdict(d))


def _compare(d: SiglipDims, batch: int, chunk: int, rel_tol: float, seed: int = 7, tight_tol: float = 0.0):
    sd = synth_siglip_state_dict(d, seed=seed)
    enc = SiglipImageEncoder(d, images_per_chunk=chunk)
    enc.load_state_dict(sd, strict=True)
    enc = enc.to(DEV).eval()
    img = synth_images(batch, d, seed=seed + 4)
    with torch.inference_mode():
        ref = vo.encode_image_siglip(_cfg(d), sd, img)
        ref16 = vo.encode_image_siglip(_cfg(d), sd, img, bf16_operands=True) if tight_tol else None
        got = enc.encode_image(img.to(DEV)).cpu()
        got_n = enc.encode_image(img.to(DEV), normalize=True).cpu()
    assert got.shape == ref.shape == (batch, d.width)
    rms = ref.pow(2).mean().sqrt().item()
    err = ((got - ref).norm() / ref.norm()).item()
    worst = (got - ref).abs().max().item() / rms
    cos = torch.nn.functional.cosine_similarity(got, ref, dim=1).min().item()
    print(f"SigLIP {d.width}x{d.layers} layers, {d.tokens} tokens, batch {batch}: ||d|| / ||ref|| = {err:.4f}, max |d| / rms = {worst:.4f}, min cosine = {cos:.6f}")
    assert err <= rel_tol and worst <= 6 * rel_tol and cos >= 0.999
    if ref16 is not None:
        err16 = ((got - ref16).norm() / ref16.norm()).item()
        print(f"    against the bf16-operand restatement: ||d|| / ||ref|| = {err16:.5f}")
        assert err16 <= tight_tol
    assert (got_n.norm(dim=1) - 1).abs().max().item() < 1e-5
    assert (got_n - torch.nn.functional.normalize(got, dim=1)).abs().max().item() < 1e-5
    return enc, img, got


@pytest.mark.gpu
def test_small_images_every_piece():
    """width 768, 2 blocks, 96 x 96 images: 36 tokens = one ragged query and key tile; batch 5 in chunks of 2 (ragged last chunk)."""
    _compare(SMALL, batch=5, chunk=2, rel_tol=0.02, tight_tol=0.008)


@pytest.mark.gpu
def test_224_two_blocks_196_tokens():
    """The real token count: 196 = 128 + 68 queries and keys per (image, head)."""
    _compare(SiglipDims(layers=2), batch=3, chunk=2, rel_tol=0.02, tight_tol=0.008)


def _f768_decoder():
    dims = dataclasses.replace(synth.DecoderDims(), embed_dim=768)
    sd = synth.make_eos_friendly(synth.synth_state_dict(dims, seed=2, token_scale=0.25, jitter_norms=True), dims, beta=0.1)
    return dims, default_decoder(dims, sd).to(DEV)


@pytest.mark.gpu
def test_full_depth_encoder_feeds_the_f768_decoder():
    """All 12 blocks on four images, then images -> labels on the device, greedy and guided beam k = 10 (the reference's default
    generation config): exactly what the decoder generates from the same normalised embeddings passed in by the caller."""
    enc, img, feats = _compare(SiglipDims(), batch=4, chunk=4, rel_tol=0.03, seed=9)
    dims, dec = _f768_decoder()
    both = EncoderDecoder(enc, dec)
    gt = synth.synth_guide_targets(500, dims, seed=33, first_pool=60).to(DEV)
    with torch.inference_mode():
        e = both.embed(img.to(DEV))
        assert (e.cpu() - torch.nn.functional.normalize(feats, dim=1)).abs().max().item() < 1e-5
        tok, pad, score = both.generate(img.to(DEV))
        t2, p2, _, _, _, s2 = dec.generate(e, False, True, 1.0, 0.0, None, None, False)
        bt, bp, bs = both.generate_beam(img.to(DEV), 10, 1.0, 0.0, None, False, 0.0, gt, False)
        bt2, bp2, bs2 = dec.generate_beam(e, 10, 1.0, 0.0, None, False, 0.0, gt, False)
    assert tok.shape[:2] == (4, 1)
    assert torch.equal(tok[:, 0], t2) and torch.equal(pad[:, 0], p2)
    assert (score[:, 0] - s2).abs().max().item() < 1e-3
    assert bt.shape[:2] == (4, 10)
    assert torch.equal(bt, bt2) and torch.equal(bp, bp2)
    assert (bs - bs2).abs().max().item() < 1e-3


B16_TWO = SiglipDims(layers=2)


@pytest.fixture(scope="module")
def b16_chunk():
    """67 images in one chunk after two blocks: 13 132 token rows = 103 row tiles (odd: the last pair's second CTA has no rows), so every
    trunk GEMM runs on CTA pairs (>= 2 x 148 tiles of 128 x 256).  The MAP head's GEMMs have one row per image and stay on 128 x 128 tiles
    (tests/test_gpu_vit_kernels.py covers their epilogue on pairs)."""
    sd = synth_siglip_state_dict(B16_TWO, seed=21)

    def make(n):
        enc = SiglipImageEncoder(B16_TWO, images_per_chunk=n)
        enc.load_state_dict(sd, strict=True)
        return enc.to(DEV).eval()
    restate = lambda x, bf16: vo.encode_image_siglip(_cfg(B16_TWO), sd, x, bf16_operands=bf16)
    return production_chunk(make, synth_images(67, B16_TWO, seed=25), restate, 0.02, 0.008, {"EpiVitBias", "EpiVitResid"}), make


@pytest.mark.gpu
def test_b16_67_images_in_one_chunk_run_on_cta_pairs(b16_chunk):
    """gemm2_kernel ran the bias and residual epilogues; the first, middle and last images are within the two-block bounds; every image
    equals its features from chunks of two, bit for bit."""
    run, _ = b16_chunk
    assert run.got.shape == (67, 768)


@pytest.mark.gpu
def test_b16_67_images_bit_identical_under_tile_and_store_switches(b16_chunk, monkeypatch):
    run, make = b16_chunk
    same_under_switches(run, make, monkeypatch)


@pytest.mark.gpu
def test_b16_67_images_poisoned_workspace(b16_chunk):
    """T = 196 < Tpad = 256: the V^T columns past T and the zero-filled key rows of the ragged tile are read on every item."""
    poisoned_workspace(b16_chunk[0])


def test_mismatched_embed_width_is_rejected():
    dims = synth.DecoderDims()            # embed_dim 1024: not SigLIP's 768
    dec = default_decoder(dims, synth.synth_state_dict(dims, seed=1))
    with pytest.raises(ValueError, match="embed_dim"):
        EncoderDecoder(SiglipImageEncoder(SMALL), dec)
