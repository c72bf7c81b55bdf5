"""Embedding-cache reader / device feeder (SURVEY.md section 8 row f4) against the unmodified reference reader.

tests/golden/cache_*.bin are cache files in the reference's format; tests/golden/cache_expected.npz holds what the reference's
EmbeddingCache.get_samples and EmbeddingCache.Dataset.__getitem__ return for them (oracle/make_cache_golden.py).  The CPU tests
run the reader with device='cpu' (it is I/O plumbing, not a compute path); the GPU tests check the device feeder and feed a
training step from it."""
import os
import struct

import numpy as np
import pytest
import torch

from novic_b200 import cache

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = {"multi": dict(N=37, F=16, C=6, M=3), "single": dict(N=21, F=8, C=7, M=1)}
SLICES = {"head": (0, 5), "mid": (5, 12), "tail": (-3, 4), "empty": (7, 7)}     # tail: (N - 3, N + 4)
MODES = {"eval": (False, 0), "train0": (True, 0), "train5": (True, 5), "trainwrap": (True, -3)}   # trainwrap: offset N - 3


@pytest.fixture(scope="module")
def expected():
    z = np.load(os.path.join(GOLDEN, "cache_expected.npz"))
    return lambda key: torch.from_numpy(z[key.replace("/", "__")]) if key.replace("/", "__") in z.files else None


def _same(got, want):
    if want is None:
        return got is None
    return got is not None and got.shape == want.shape and torch.equal(got.cpu(), want)


@pytest.mark.parametrize("name", sorted(CASES))
def test_header_and_layout(name):
    path = os.path.join(GOLDEN, f"cache_{name}.bin")
    with cache.EmbeddingCacheReader(path, device="cpu") as r:
        c = CASES[name]
        h = r.header
        assert (h.embed_num, h.embed_dim, h.target_dim, h.embed_targets_dim) == (c["N"], c["F"], c["C"], c["M"])
        assert h.use_targets and h.version == 1 and r.target_nouns[0] == "" and len(r.target_nouns) == h.target_nouns_num
        assert r.layout.total_size == os.path.getsize(path) and len(r) == c["N"]
        assert cache.CacheHeader.unpack(h.pack()) == h


@pytest.mark.parametrize("name", sorted(CASES))
@pytest.mark.parametrize("sl", sorted(SLICES))
def test_get_samples_vs_reference_reader(expected, name, sl):
    N = CASES[name]["N"]
    a, b = SLICES[sl]
    if sl == "tail":
        a, b = N + a, N + b
    with cache.EmbeddingCacheReader(os.path.join(GOLDEN, f"cache_{name}.bin"), device="cpu") as r:
        got = r.get_samples(a, b)
    for k, t in zip(("embed", "ids", "target", "mask", "weight"), got):
        assert _same(t, expected(f"{name}/samples/{sl}/{k}")), (name, sl, k)


@pytest.mark.parametrize("name", sorted(CASES))
@pytest.mark.parametrize("mode", sorted(MODES))
def test_batches_vs_reference_dataset(expected, name, mode):
    N = CASES[name]["N"]
    training, offset = MODES[mode]
    offset = N + offset if offset < 0 else offset
    with cache.EmbeddingCacheReader(os.path.join(GOLDEN, f"cache_{name}.bin"), device="cpu") as r:
        got = list(r.batches(8, training=training, epoch_index_offset=offset))
    assert len(got) == int(expected(f"{name}/batches/{mode}/count")[0])
    for i, b in enumerate(got):
        for k, t in zip(("embed", "target", "mask", "weight"), b):
            assert _same(t, expected(f"{name}/batches/{mode}/{i}/{k}")), (name, mode, i, k)


def test_rejects_damaged_files(tmp_path):
    src = open(os.path.join(GOLDEN, "cache_single.bin"), "rb").read()
    bad_magic = tmp_path / "magic.bin"
    bad_magic.write_bytes(b"\x00" * 32 + src[32:])                     # the writer stores the magic last: an unfinished file (embedding_cache.py:41)
    with pytest.raises(ValueError, match="magic"):
        cache.EmbeddingCacheReader(str(bad_magic), device="cpu")
    short = tmp_path / "short.bin"
    short.write_bytes(src[:-4])
    with pytest.raises(ValueError, match="size"):
        cache.EmbeddingCacheReader(str(short), device="cpu")
    future = tmp_path / "future.bin"
    future.write_bytes(src[:32] + struct.pack("<B", 9) + src[33:])
    with pytest.raises(ValueError, match="version"):
        cache.EmbeddingCacheReader(str(future), device="cpu")
    with pytest.raises(ValueError, match="dimension"):
        cache.EmbeddingCacheReader(os.path.join(GOLDEN, "cache_single.bin"), device="cpu", embed_dim=1024)


def test_cache_without_targets_round_trip(tmp_path):
    emb = torch.nn.functional.normalize(torch.randn(10, 32), dim=-1)
    path = str(tmp_path / "plain.bin")
    cache.write_cache(path, emb)
    with cache.EmbeddingCacheReader(path, device="cpu") as r:
        assert not r.use_targets
        e, ids, t, m, w = r.get_samples(2, 7)
        assert torch.equal(e, emb[2:7]) and ids is None and t is None and m is None and w is None
        assert [b[0].shape[0] for b in r.batches(4)] == [4, 4, 2]
        assert [b[0].shape[0] for b in r.batches(4, training=True)] == [4, 4]
        with pytest.raises(ValueError):
            cache.EmbeddingCacheReader(path, device="cpu", use_targets=True)


@pytest.mark.reference
def test_header_struct_and_offsets_match_the_reference(tmp_path):
    from oracle import refload
    refload.import_reference()
    import embedding_cache
    assert cache.HEADER_STRUCT.format == embedding_cache.Header.STRUCT_FORMAT and cache.MAGIC == embedding_cache.Header.MAGIC_BYTES
    for name in CASES:
        raw = open(os.path.join(GOLDEN, f"cache_{name}.bin"), "rb").read(128)
        rh = embedding_cache.Header(*embedding_cache.Header.STRUCT_FACTORY.unpack(raw))
        rm = embedding_cache.Meta.from_header(rh)
        lay = cache.CacheLayout.from_header(cache.CacheHeader.unpack(raw))
        assert (lay.target_nouns_offset, lay.target_offset, lay.target_mask_offset, lay.embed_targets_offset, lay.embed_target_weights_offset,
                lay.embed_offset, lay.embed_stride, lay.total_size) == (rm.target_nouns_offset, rm.target_offset, rm.target_mask_offset,
                                                                         rm.embed_targets_offset, rm.embed_target_weights_offset, rm.embed_offset,
                                                                         rm.embed_stride, rm.total_size)


def header_values() -> dict:
    """What test_header_struct_and_offsets_match_the_reference compares: the header struct format, the magic bytes and, per cache file,
    the eight section offsets / sizes of its layout."""
    out = {"struct_format": np.array(cache.HEADER_STRUCT.format), "magic": np.frombuffer(cache.MAGIC, dtype=np.uint8).copy()}
    for name in CASES:
        raw = open(os.path.join(GOLDEN, f"cache_{name}.bin"), "rb").read(128)
        lay = cache.CacheLayout.from_header(cache.CacheHeader.unpack(raw))
        out[f"{name}__layout"] = np.array([lay.target_nouns_offset, lay.target_offset, lay.target_mask_offset, lay.embed_targets_offset,
                                           lay.embed_target_weights_offset, lay.embed_offset, lay.embed_stride, lay.total_size], dtype=np.int64)
    return out


def test_header_struct_and_offsets_match_committed_reference_values():
    """test_header_struct_and_offsets_match_the_reference without the reference tree: against the stored values that test asserts
    equal to the reference's Header / Meta (tests/golden/live_twins.npz)."""
    from tests.golden_util import check_twin
    check_twin("cache", header_values())


# ------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_device_feeder_matches_reference_dataset(expected, name):
    with cache.EmbeddingCacheReader(os.path.join(GOLDEN, f"cache_{name}.bin"), device="cuda:0") as r:
        assert r.target_token_ids.is_cuda
        for mode, (training, offset) in MODES.items():
            offset = CASES[name]["N"] + offset if offset < 0 else offset
            got = list(r.batches(8, training=training, epoch_index_offset=offset))
            for i, b in enumerate(got):
                for k, t in zip(("embed", "target", "mask", "weight"), b):
                    assert t is None or t.is_cuda
                    assert _same(t, expected(f"{name}/batches/{mode}/{i}/{k}")), (name, mode, i, k)


@pytest.mark.gpu
def test_feeder_drives_a_training_step(tmp_path):
    """A synthetic cache of the default decoder's shapes (F = 1024, C = 16, multi-target M = 3 with weights) feeds
    PrefixedIterDecoder.forward in training mode: the batches have the reference's layout, so loss and backward run."""
    from novic_b200 import default_decoder, synth
    from novic_b200.factory import synthetic_data_config
    dims = synth.DecoderDims()
    N, R1, M = 256, 50, 3
    emb = synth.synth_embeddings(N, seed=3)
    noun_rows = synth.synth_guide_targets(R1, dims, seed=5)                       # R1 x C token rows ending in the end token 0
    mask = torch.zeros_like(noun_rows, dtype=torch.bool)
    mask[:, 1:] = (noun_rows[:, :-1] == 0)                                        # padding starts after the end token
    g = torch.Generator().manual_seed(7)
    et = torch.randint(1, R1 + 1, (N, M), dtype=torch.int32, generator=g)
    et[::4, 2] = 0
    w = torch.rand(N, M, generator=g).sort(dim=1, descending=True).values
    w[et == 0] = 0
    w = w / w.sum(dim=1, keepdim=True)
    path = str(tmp_path / "train.bin")
    cache.write_cache(path, emb, [f"n{i}" for i in range(R1)], noun_rows, mask, et, w)
    model = default_decoder(dims, synth.synth_state_dict(dims, seed=1), input_dropout=0.0, layer_dropout=0.0)
    model.data_config = synthetic_data_config(multi_target=True, use_weights=True)
    model = model.to("cuda:0").train()
    seen = 0
    with cache.EmbeddingCacheReader(path, device="cuda:0", embed_dim=dims.embed_dim) as r:
        for embed, target, tmask, weight in r.batches(64, training=True, fixed_token_length=True):
            assert embed.shape == (64, 1024) and target.shape == (64, 3, 16) and tmask.dtype == torch.bool and weight.shape == (64, 3)
            _, _, loss_sum, loss_basis, _ = model(embed, target, tmask, weight, True, True, False, None)
            (loss_sum / loss_basis).backward()
            assert torch.isfinite(loss_sum) and float(loss_basis) > 0
            seen += embed.shape[0]
    assert seen == 256 and model.logits_linear.weight.grad is not None
