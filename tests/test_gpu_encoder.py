"""Image encoder (SURVEY.md section 8 row f3, BASELINE config #5) against the independent CPU restatement oracle/vit_oracle.py.

PARITY UNPINNED: open_clip_torch is an un-vendored dependency of the reference (requirements.txt:8), so the oracle restates the
published VisionTransformer from memory and cannot be checked against the reference here.  What these tests establish is that the
CUDA path computes that architecture: bf16 operands / fp32 accumulation and residual stream against fp32 on the CPU.
Tolerance (stated per test): ||got - ref|| / ||ref|| of the un-normalised features <= 2 % after two blocks, <= 3 % after all 32 (every
block rounds its GEMM and attention operands to bf16, ~0.4 % each), no element off by more than six times that, cosine >= 0.999; and
<= 0.8 % against the same restatement with its matrix-product operands rounded to bf16 (what separates a wrong kernel from rounding).
The `vith_11_images` tests run a production-sized chunk (every trunk GEMM on CTA pairs, tests/encoder_chunks.py): sampled images within
those bounds, the same bits as chunks of two and under NOVIC_VIT_BN=256 / 128 and NOVIC_VIT_DIRECT=0, and the mma.sync attention
(NOVIC_VIT_ATTN=mma) within the bounds.  Each kernel alone against fp64: tests/test_gpu_vit_kernels.py.
"""
import dataclasses

import pytest
import torch

from novic_b200 import default_decoder, synth
from novic_b200.encoder import EncoderDecoder, ImageEncoder, VitDims, synth_images, synth_vit_state_dict
from oracle import vit_oracle as vo
from tests.encoder_chunks import check_bounds, production_chunk, same_under_switches

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _cfg(d: VitDims) -> vo.VitCfg:
    return vo.VitCfg(**dataclasses.asdict(d))


def _compare(d: VitDims, batch: int, chunk: int, rel_tol: float, seed: int = 7, tight_tol: float = 0.0):
    sd = synth_vit_state_dict(d, seed=seed)
    enc = ImageEncoder(d, images_per_chunk=chunk)
    enc.load_state_dict(sd, strict=True)
    enc = enc.to(DEV).eval()
    img = synth_images(batch, d, seed=seed + 4)
    with torch.inference_mode():
        ref = vo.encode_image(_cfg(d), sd, img)
        ref16 = vo.encode_image(_cfg(d), sd, img, bf16_operands=True) if tight_tol else None
        got = enc.encode_image(img.to(DEV)).cpu()
        got_n = enc.encode_image(img.to(DEV), normalize=True).cpu()
    assert got.shape == ref.shape == (batch, d.out_dim)
    rms = ref.pow(2).mean().sqrt().item()
    err = ((got - ref).norm() / ref.norm()).item()
    worst = (got - ref).abs().max().item() / rms
    cos = torch.nn.functional.cosine_similarity(got, ref, dim=1).min().item()
    print(f"{d.width}x{d.layers} layers, {d.tokens} tokens, batch {batch}: ||d|| / ||ref|| = {err:.4f}, max |d| / rms = {worst:.4f}, min cosine = {cos:.6f}")
    assert err <= rel_tol and worst <= 6 * rel_tol and cos >= 0.999
    if ref16 is not None:   # against the restatement that sees the same bf16-rounded operands: only accumulation order and the exp2 path differ
        err16 = ((got - ref16).norm() / ref16.norm()).item()
        print(f"    against the bf16-operand restatement: ||d|| / ||ref|| = {err16:.5f}")
        assert err16 <= tight_tol
    assert (got_n.norm(dim=1) - 1).abs().max().item() < 1e-5
    assert (got_n - torch.nn.functional.normalize(got, dim=1)).abs().max().item() < 1e-5
    return enc, img, got


def test_small_encoder_every_piece():
    """width 640 (8 heads of 80), 2 blocks, 26 tokens (one ragged query / key tile), batch 5 in chunks of 2 (ragged last chunk)."""
    _compare(VitDims(image_size=70, width=640, heads=8, layers=2, mlp_dim=2560), batch=5, chunk=2, rel_tol=0.02, tight_tol=0.008)


def test_full_width_two_blocks_730_tokens():
    """The real token count: 730 = 5 x 128 + 90 queries per (image, head), 11 x 64 + 26 keys; width 1280, 16 heads, mlp 5120."""
    _compare(VitDims(layers=2), batch=3, chunk=2, rel_tol=0.02, tight_tol=0.008)


def test_full_depth_encoder_feeds_the_decoder():
    """All 32 blocks on two images (the CPU restatement costs about 2 TFLOP), then images -> labels on the device: the embeddings the
    encoder hands over make the decoder generate exactly what it generates from the same embeddings passed in by the caller."""
    enc, img, feats = _compare(VitDims(), batch=2, chunk=2, rel_tol=0.03, seed=9)
    dims = synth.DecoderDims()
    dec = default_decoder(dims, synth.make_eos_friendly(synth.synth_state_dict(dims, seed=2, token_scale=0.25, jitter_norms=True), dims, beta=0.1)).to(DEV)
    both = EncoderDecoder(enc, dec)
    with torch.inference_mode():
        tok, pad, score = both.generate(img.to(DEV))
        e = torch.nn.functional.normalize(feats, dim=1).to(DEV)
        t2, p2, _, _, _, s2 = dec.generate(e, False, True, 1.0, 0.0, None, None, False)
    assert tok.shape[0] == 2 and tok.shape[1] == 1
    assert torch.equal(tok[:, 0], t2) and torch.equal(pad[:, 0], p2)
    assert (score[:, 0] - s2).abs().max().item() < 1e-3


TWO = VitDims(layers=2)


@pytest.fixture(scope="module")
def vith_chunk():
    """11 images in one chunk after two blocks: 8 030 token rows and 8 019 patch rows, 63 row tiles each (odd: the last pair's second CTA
    has no rows), so every trunk GEMM runs on CTA pairs.  The final projection has one row per image and stays on 128 x 128 tiles."""
    sd = synth_vit_state_dict(TWO, seed=19)

    def make(n):
        enc = ImageEncoder(TWO, images_per_chunk=n)
        enc.load_state_dict(sd, strict=True)
        return enc.to(DEV).eval()
    restate = lambda x, bf16: vo.encode_image(_cfg(TWO), sd, x, bf16_operands=bf16)
    return production_chunk(make, synth_images(11, TWO, seed=29), restate, 0.02, 0.008, {"EpiVitBias", "EpiVitResid"}), make


def test_vith_11_images_in_one_chunk_run_on_cta_pairs(vith_chunk):
    """gemm2_kernel ran the bias and residual epilogues (patch mode included); sampled images within the two-block bounds; chunks of two
    give the same bits."""
    run, _ = vith_chunk
    assert run.got.shape == (11, 1024)


def test_vith_11_images_bit_identical_under_tile_and_store_switches(vith_chunk, monkeypatch):
    run, make = vith_chunk
    same_under_switches(run, make, monkeypatch)


def test_vith_11_images_mma_attention_within_bounds(vith_chunk, monkeypatch):
    """NOVIC_VIT_ATTN=mma: the mma.sync attention kernel accumulates in another order, so it is held to the restatement bounds."""
    run, make = vith_chunk
    monkeypatch.setenv("NOVIC_VIT_ATTN", "mma")
    with torch.inference_mode():
        got = make(11).encode_image(run.img.to(DEV)).cpu()
    check_bounds(got[run.sample], run.ref, run.ref16, 0.02, 0.008, "NOVIC_VIT_ATTN=mma, 11 images in one chunk")


def test_encoder_state_dict_keys_follow_open_clip():
    d = VitDims(image_size=70, width=640, heads=8, layers=2, mlp_dim=2560)
    keys = set(ImageEncoder(d).state_dict())
    assert {"visual.conv1.weight", "visual.class_embedding", "visual.positional_embedding", "visual.ln_pre.weight", "visual.ln_post.bias", "visual.proj",
            "visual.transformer.resblocks.1.attn.in_proj_weight", "visual.transformer.resblocks.1.attn.in_proj_bias",
            "visual.transformer.resblocks.0.attn.out_proj.weight", "visual.transformer.resblocks.0.mlp.c_fc.weight",
            "visual.transformer.resblocks.0.mlp.c_proj.bias", "visual.transformer.resblocks.0.ln_2.weight"} <= keys
    with pytest.raises(RuntimeError, match="no CPU path"):
        ImageEncoder(d).encode_image(synth_images(1, d))
