"""SigLIP SO400M/14 image encoder (the image embedder of the F = 1152 checkpoints: heads of 72, MLP 4304) against the independent CPU
restatement tests/siglip_oracle.py:encode_image_siglip.

PARITY UNPINNED, as for B/16 (tests/test_siglip_encoder.py): the architecture is restated from memory (DESIGN.md §5d).  The assumption
for SO400M: timm `vit_so400m_patch14_siglip_224` is B/16's architecture with 14 x 14 patches of 224 x 224 images (256 tokens), width 1152,
27 blocks of 16 heads of 72 (scale 1/sqrt(72)) and an MLP of 4304 in the blocks and the head.  encode_image_siglip derives the head
dimension as width / heads, so the same restatement serves at these dimensions (`SiglipCfg(**asdict(dims))`).  The GPU tests
establish that the CUDA path computes that architecture at these dimensions - attention at 72 stored / 80 computed channels per head,
the MAP head's 144-byte rows, the LayerNorm at width 1152 and the MLP padded from 4304 to 4352 hidden channels - with B/16's bounds
after two blocks (<= 2 % against fp32, <= 0.8 % against the bf16-operand restatement, cosine >= 0.999) and <= 4 % after all 27.  The
`so400m_31_images` tests run a production-sized chunk (every trunk GEMM on CTA pairs, with N = 1152 and 3456 ending inside a pair tile's
B half): sampled images within the two-block bounds, the same bits as chunks of two and under NOVIC_VIT_BN=256 / 128 and
NOVIC_VIT_DIRECT=0.
"""
import dataclasses

import pytest
import torch

from novic_b200 import SIGLIP_SO400M, _abi, default_decoder, synth
from novic_b200.encoder import EncoderDecoder, SiglipDims, SiglipImageEncoder, synth_images, synth_siglip_state_dict
from tests import siglip_oracle as vo
from tests.encoder_chunks import production_chunk, same_under_switches
from tests.test_siglip_encoder import _cfg, _compare, expected_shapes

DEV = "cuda:0"
TWO = dataclasses.replace(SIGLIP_SO400M, layers=2)


def test_preset_is_the_so400m_tower():
    d = SIGLIP_SO400M
    assert (d.image_size, d.patch_size, d.width, d.layers, d.heads, d.mlp_dim, d.ln_eps) == (224, 14, 1152, 27, 16, 4304, 1e-6)
    assert (d.tokens, d.head_dim, d.out_dim) == (256, 72, 1152)
    assert SiglipDims().head_dim == 64


def test_state_dict_keys_and_shapes_at_so400m_dims():
    want = expected_shapes(TWO)
    assert want["visual.trunk.blocks.1.mlp.fc1.weight"] == (4304, 1152)
    assert want["visual.trunk.attn_pool.mlp.fc2.weight"] == (1152, 4304)
    assert want["visual.trunk.patch_embed.proj.weight"] == (1152, 3, 14, 14)
    enc = SiglipImageEncoder(TWO)
    assert {k: tuple(v.shape) for k, v in enc.state_dict().items()} == want
    sd = synth_siglip_state_dict(TWO, seed=3)
    assert {k: tuple(v.shape) for k, v in sd.items()} == want
    enc.load_state_dict(sd, strict=True)
    assert all(v.abs().min() > 0 for k, v in sd.items() if k.endswith(".bias") or k.endswith("latent"))
    assert all((v - 1).abs().max() > 0.1 for k, v in sd.items() if "norm" in k and k.endswith(".weight"))


@pytest.mark.parametrize("kw", [dict(width=864, heads=12), dict(mlp_dim=4300), dict(heads=48)],
                         ids=["head_dim_72_at_width_864", "mlp_4300", "width_1152_head_dim_24"])
def test_unsupported_so400m_variants_are_rejected(kw):
    with pytest.raises(ValueError):
        SiglipImageEncoder(dataclasses.replace(TWO, **kw))


# ---------------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------------
def _a256(n: int) -> int:
    return (n + 255) // 256 * 256


@pytest.mark.gpu
def test_weight_and_workspace_bytes_hold_the_padded_mlp():
    """novic_vit_weight_bytes / novic_vit_workspace_bytes against hand arithmetic, with the MLPs at 4352 hidden channels."""
    d = TWO
    W, L, M, Mp, T, Kp = d.width, d.layers, d.mlp_dim, 4352, d.tokens, 640
    enc = SiglipImageEncoder(d).to(DEV)
    st = enc._state(torch.device(DEV))
    lib = _abi.lib()
    bf = [W * Kp] + [3 * W * W, W * W, Mp * W, W * Mp] * L + [2 * W * W, W * W, Mp * W, W * Mp]
    f32 = [W, T * W, W, W] + [W, W, W, W, 3 * W, W, Mp, W] * L + [2 * W, W, W, W, Mp, W] + [W]
    assert lib.novic_vit_weight_bytes(st["handle"]) == sum(_a256(2 * n) for n in bf) + sum(_a256(4 * n) for n in f32)
    for nc in (1, 2, 7):
        rows = nc * T
        parts = [2 * rows * Kp, 4 * rows * W, 2 * rows * W, 2 * rows * 3 * W, 2 * rows * W, 2 * rows * Mp, 2 * nc * W, 2 * nc * W * 256]
        assert lib.novic_vit_workspace_bytes(st["handle"], nc) == sum(_a256(p) for p in parts)
    assert M < Mp


@pytest.mark.gpu
def test_small_images_one_ragged_tile():
    """8 x 8 = 64 tokens: one ragged query and key tile; batch 5 in chunks of 2 (ragged last chunk)."""
    _compare(dataclasses.replace(TWO, image_size=112), batch=5, chunk=2, rel_tol=0.02, tight_tol=0.008)


@pytest.mark.gpu
def test_169_tokens_full_plus_ragged_tile():
    """13 x 13 = 169 = 128 + 41 queries and keys per (image, head)."""
    _compare(dataclasses.replace(TWO, image_size=182), batch=3, chunk=2, rel_tol=0.02, tight_tol=0.008)


@pytest.mark.gpu
def test_224_two_blocks_256_tokens():
    """The real token count: two full 128-token tiles."""
    _compare(TWO, batch=3, chunk=2, rel_tol=0.02, tight_tol=0.008)


@pytest.fixture(scope="module")
def full_depth():
    return _compare(SIGLIP_SO400M, batch=3, chunk=3, rel_tol=0.04, seed=9)


def _f1152_decoder():
    dims = dataclasses.replace(synth.DecoderDims(), embed_dim=1152)
    sd = synth.make_eos_friendly(synth.synth_state_dict(dims, seed=2, token_scale=0.25, jitter_norms=True), dims, beta=0.1)
    return dims, default_decoder(dims, sd).to(DEV)


@pytest.mark.gpu
def test_full_depth_encoder_feeds_the_f1152_decoder(full_depth):
    """All 27 blocks on three images, then images -> labels on the device, greedy and guided beam k = 10: exactly what the decoder
    generates from the same normalised embeddings passed in by the caller."""
    enc, img, feats = full_depth
    dims, dec = _f1152_decoder()
    both = EncoderDecoder(enc, dec)
    gt = synth.synth_guide_targets(500, dims, seed=33, first_pool=60).to(DEV)
    with torch.inference_mode():
        e = both.embed(img.to(DEV))
        assert (e.cpu() - torch.nn.functional.normalize(feats, dim=1)).abs().max().item() < 1e-5
        tok, pad, score = both.generate(img.to(DEV))
        t2, p2, _, _, _, s2 = dec.generate(e, False, True, 1.0, 0.0, None, None, False)
        bt, bp, bs = both.generate_beam(img.to(DEV), 10, 1.0, 0.0, None, False, 0.0, gt, False)
        bt2, bp2, bs2 = dec.generate_beam(e, 10, 1.0, 0.0, None, False, 0.0, gt, False)
    assert tok.shape[:2] == (3, 1)
    assert torch.equal(tok[:, 0], t2) and torch.equal(pad[:, 0], p2)
    assert (score[:, 0] - s2).abs().max().item() < 1e-3
    assert bt.shape[:2] == (3, 10)
    assert torch.equal(bt, bt2) and torch.equal(bp, bp2)
    assert (bs - bs2).abs().max().item() < 1e-3


@pytest.mark.gpu
def test_poisoned_workspace_gives_the_same_features(full_depth):
    """Every workspace byte an encode reads was written by the same encode: the padded hidden columns, the foreign Q / K / V^T channels
    of the 72-channel heads and the ragged tiles included.  A workspace filled with 0xFF (NaN in bf16 and fp32) changes nothing."""
    enc, img, _ = full_depth
    x = torch.cat([img, img[:1]]).to(DEV)          # four images in chunks of three: a ragged last chunk too
    with torch.inference_mode():
        a = enc.encode_image(x)
        ws = enc._handles[0]["ws"]
        ws.fill_(0xFF)
        b = enc.encode_image(x)
    assert torch.isfinite(a).all() and torch.isfinite(b).all()
    assert torch.equal(a, b)


@pytest.fixture(scope="module")
def so400m_chunk():
    """31 images in one chunk after two blocks: 7 936 token rows = 62 row tiles; N = 1152 (out-proj, fc2, patch embedding) ends in the B
    half of the last pair tile, N = 3456 (QKV) likewise."""
    sd = synth_siglip_state_dict(TWO, seed=23)

    def make(n):
        enc = SiglipImageEncoder(TWO, images_per_chunk=n)
        enc.load_state_dict(sd, strict=True)
        return enc.to(DEV).eval()
    restate = lambda x, bf16: vo.encode_image_siglip(_cfg(TWO), sd, x, bf16_operands=bf16)
    return production_chunk(make, synth_images(31, TWO, seed=27), restate, 0.02, 0.008, {"EpiVitBias", "EpiVitResid"}), make


@pytest.mark.gpu
def test_so400m_31_images_in_one_chunk_run_on_cta_pairs(so400m_chunk):
    """gemm2_kernel ran the bias and residual epilogues; sampled images within the two-block bounds; chunks of two give the same bits."""
    run, _ = so400m_chunk
    assert run.got.shape == (31, 1152)


@pytest.mark.gpu
def test_so400m_31_images_bit_identical_under_tile_and_store_switches(so400m_chunk, monkeypatch):
    run, make = so400m_chunk
    same_under_switches(run, make, monkeypatch)
