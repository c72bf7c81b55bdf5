"""CPU-side checks: the C-ABI library loads and exports everything include/novic_b200.h declares, the host mirror
of the reference interface behaves (constructor contract, state-dict keys, error behaviour), and nothing in the
product imports the oracle or falls back to CPU compute."""
import ctypes as C
import os
import re

import pytest
import torch

import novic_b200
from novic_b200 import _abi, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_symbols_are_exported_and_bound(built_lib):
    header = open(os.path.join(ROOT, "include", "novic_b200.h")).read()
    declared = set(re.findall(r"\b(novic_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 15
    assert declared == set(_abi.SIGNATURES), declared ^ set(_abi.SIGNATURES)
    for name in declared:
        assert getattr(built_lib, name) is not None
    assert built_lib.novic_version() >= 1


def test_ctypes_structs_match_header_layout():
    assert C.sizeof(_abi.NovicCfg) == 12 * 4
    assert C.sizeof(_abi.NovicWeights) == 8 * (4 + 6 * _abi.NOVIC_MAX_LAYERS)
    assert C.sizeof(_abi.NovicNoiseCfg) == 7 * 4


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_gpu_fails_loudly(built_lib):
    cfg = _abi.NovicCfg(embed_dim=1024, hidden_dim=512, ffn_dim=128, num_layers=6, num_heads=8, prefix_len=4, vocab_size=6912,
                        token_length=16, strictly_causal=0, num_end_loss=1, ln_eps=1e-5, label_smoothing=0.0)
    h = C.c_void_p()
    assert built_lib.novic_create(C.byref(cfg), C.byref(h)) != 0
    assert b"no CPU fallback" in built_lib.novic_last_error()
    model = novic_b200.default_decoder()
    with pytest.raises(RuntimeError, match="CUDA"):
        model.generate(synth.synth_embeddings(2), False, True, 1.0, 0.0, None, None, False)
    with pytest.raises(RuntimeError, match="CUDA"):
        model.generate_beam(synth.synth_embeddings(2), 3, 1.0, 0.0, None, False, 0.0, None, False)
    with pytest.raises(RuntimeError, match="CUDA"):
        novic_b200.GaussElemNoise(1024, 3.25)(synth.synth_embeddings(2))


def test_bad_config_is_rejected_by_the_library(built_lib):
    bad = _abi.NovicCfg(embed_dim=1024, hidden_dim=256, ffn_dim=128, num_layers=6, num_heads=8, prefix_len=4, vocab_size=6912,
                        token_length=16, strictly_causal=0, num_end_loss=1, ln_eps=1e-5, label_smoothing=0.0)
    h = C.c_void_p()
    assert built_lib.novic_create(C.byref(bad), C.byref(h)) != 0
    assert b"hidden_dim" in built_lib.novic_last_error()


def test_product_never_imports_the_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU arm may touch oracle/: the package and the measurement tools must not."""
    for sub in ("novic_b200", "tools", "include"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, sub)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".inc", ".sh")):
                    text = open(os.path.join(dirpath, f)).read()
                    assert "import oracle" not in text and "from oracle" not in text and "novic_oracle" not in text, f
    # bench.py: the oracle is imported inside the CPU-baseline function only, never at module level
    src = open(os.path.join(ROOT, "bench.py")).read()
    top_level = [ln for ln in src.splitlines() if ln.startswith(("import ", "from "))]
    assert not any("oracle" in ln for ln in top_level)


def test_state_dict_contract_and_param_count():
    dims = synth.DecoderDims()
    model = novic_b200.default_decoder(dims)
    sd = model.state_dict()
    want = synth.synth_state_dict(dims, seed=3)
    assert list(sd.keys()).sort() == list(want.keys()).sort() and set(sd) == set(want)
    for k, v in want.items():
        assert sd[k].shape == v.shape and sd[k].dtype == v.dtype, k
    model.load_state_dict(want, strict=True)
    total, groups = model.get_num_params()
    assert total.total == total.used == 12730368                  # SURVEY.md section 8c
    assert groups["Input MLP"].used == 2097152 and groups["Token embed/logits"].used == 3538944
    assert groups["Positional embed"].used == 9728 and groups["Transformer"].used == 7084544
    assert "12730368 params" in total.to_str()
    assert torch.equal(model.causality_mask, want["causality_mask"])
    # init statistics of a freshly constructed model (SURVEY.md section 8c fact 2)
    torch.manual_seed(0)
    fresh = novic_b200.default_decoder(dims).state_dict()
    stds = synth.init_stds(dims)
    assert abs(fresh["embed_mlp.mlp.0.weight"].std().item() / stds["embed_mlp"] - 1) < 0.02
    assert abs(fresh["transformer.layers.3.self_attn.out_proj.weight"].std().item() / stds["out_proj"] - 1) < 0.02
    assert abs(fresh["transformer.layers.5.linear2.weight"].std().item() / stds["linear2"] - 1) < 0.02
    assert torch.allclose(fresh["transformer.norm.weight"], torch.full((512,), 512 ** -0.5))
    assert torch.allclose(fresh["transformer.layers.0.norm1.weight"], torch.ones(512))


def test_constructor_contract():
    kw = dict(novic_b200.DEFAULT_DECODER_KWARGS)
    from novic_b200.factory import synthetic_data_config, synthetic_embedder
    emb, dc = synthetic_embedder(), synthetic_data_config()
    with pytest.raises(TypeError):
        novic_b200.PrefixedIterDecoder(emb, dc, **kw)                # keyword-only like the reference
    for bad in (dict(hidden_dim=256), dict(feedfwd_scale='4'), dict(weight_tying=False), dict(layer_bias=True), dict(mlp_hidden_layer='min'),
                dict(layer_norm_first=False), dict(init_rezero_mode='perskip'), dict(num_heads=4), dict(feedfwd_scale='1/3')):
        with pytest.raises(ValueError):
            novic_b200.PrefixedIterDecoder(embedder=emb, data_config=dc, **{**kw, **bad})
    tk = novic_b200.PrefixedIterDecoder.get_target_config_kwargs(with_start_token=True, with_end_token=False, compact_ids=False, other=1)
    assert tk == dict(with_start_token=False, with_end_token=True, compact_ids=True, other=1)   # embedding_decoder.py:619-627
    assert novic_b200.PrefixedIterDecoder.get_data_config_kwargs(a=1) == dict(a=1)
    q = novic_b200.PrefixedIterDecoder(embedder=synthetic_embedder(synth.DecoderDims(vocab_size=6900)), data_config=dc, **{**kw, 'vocab_quant': True})
    assert q.vocab_size_quant == 6912 and q.logits_linear.weight.shape[0] == 6912 and (q.logits_linear.weight[6900:] == 0).all()
    assert q.get_num_params()[0].unused == 12 * 512


def test_unsupported_features_raise_not_fallback():
    model = novic_b200.default_decoder()
    e = synth.synth_embeddings(2)
    guide = torch.zeros(3, 16, dtype=torch.int64)
    with pytest.raises(NotImplementedError):   # a beam of one with a vocabulary prior is the one unsupported corner of generate_beam
        model.generate_beam(e, 1, 1.0, 0.0, guide, False, 0.5, None, False)
    with pytest.raises(ValueError):            # negative prior scaler: +inf scores outside the vocabulary in the reference
        model.generate_beam(e, 3, 1.0, 0.0, guide, False, -0.5, None, False)
    with pytest.raises(ValueError):
        model.generate(e, False, True, 0.0, 0.0, None, None, False)
    with pytest.raises(RuntimeError, match="no CPU path"):   # everything else computes on the GPU or raises
        model.generate_beam(e, 3, 1.0, 0.0, guide, False, 0.5, None, False)


@pytest.mark.reference
def test_drop_in_through_the_reference_loader():
    """infer.load_decoder_model (infer.py:713-778) must build OUR class after register(), with the checkpoint's
    state dict loading strictly - i.e. the seam the reference offers is honoured."""
    from oracle import refload
    ref = refload.import_reference()
    original = ref.embedding_decoder.PrefixedIterDecoder
    try:
        novic_b200.register(ref.embedding_decoder)
        sd = synth.synth_state_dict(seed=4)
        model = refload.build_reference_decoder(ref, sd)
        assert type(model) is novic_b200.PrefixedIterDecoder
        assert all(torch.equal(model.state_dict()[k], v) for k, v in sd.items())
        # the reference's own model accepts our state dict as well (same keys / shapes both ways)
        ref.embedding_decoder.PrefixedIterDecoder = original
        theirs = refload.build_reference_decoder(ref, novic_b200.default_decoder().state_dict())
        assert type(theirs) is original
        ours_count, theirs_count = model.get_num_params(), theirs.get_num_params()
        assert ours_count[0].used == theirs_count[0].used and set(ours_count[1]) == set(theirs_count[1])
        for k in ours_count[1]:
            assert ours_count[1][k].used == theirs_count[1][k].used
    finally:
        ref.embedding_decoder.PrefixedIterDecoder = original


def state_dict_values() -> dict:
    """What test_drop_in_through_the_reference_loader checks the reference model against: the default decoder's state-dict keys and
    shapes (each as ndim, shape), and the used parameter counts in all and per group."""
    import numpy as np
    model = novic_b200.default_decoder()
    sd = model.state_dict()
    total, groups = model.get_num_params()
    return {"keys": np.array(list(sd)), "shapes": np.array([n for v in sd.values() for n in (v.ndim, *v.shape)], dtype=np.int64),
            "groups": np.array(list(groups)), "params": np.array([total.used] + [c.used for c in groups.values()], dtype=np.int64)}


def test_state_dict_and_param_counts_match_committed_reference_values():
    """test_drop_in_through_the_reference_loader without the reference tree: the state-dict contract and parameter counts against the
    stored values that test asserts equal to the reference model's (tests/golden/live_twins.npz).  The loader seam itself
    (infer.load_decoder_model building this class after register()) needs the reference code and stays with the live test."""
    from tests.golden_util import check_twin
    check_twin("sd", state_dict_values())


@pytest.mark.reference
def test_oracle_matches_live_reference():
    from oracle import validate_vs_reference
    assert validate_vs_reference.run()


def test_wgrad_split_factor_properties(built_lib):
    """novic_debug_wgrad_splits (pure host arithmetic): no split may be empty, the work fits the round count it was chosen for,
    and the known shapes of the default decoder avoid a ragged extra round on 148 SMs."""
    lib = _abi.lib()
    ceil = lambda a, b: -(-a // b)
    for tiles in (1, 2, 4, 16, 48, 216, 300):
        for kblocks in (1, 2, 7, 8, 64, 240, 304, 1000):
            for sms in (1, 132, 148):
                sp = lib.novic_debug_wgrad_splits(tiles, kblocks, sms)
                assert 1 <= sp <= max(1, kblocks // 4)
                per = ceil(kblocks, sp)
                assert (sp - 1) * per < kblocks, (tiles, kblocks, sms, sp)          # last split not empty
    # linear1 / linear2 wgrad of the default decoder at 19 456 rows: 4 tiles x 304 k-blocks -> one round on 148 SMs
    sp = lib.novic_debug_wgrad_splits(4, 304, 148)
    assert 4 * sp <= 148 and sp >= 30
    # in_proj: 48 tiles; out_proj: 16 tiles -> whole rounds (at most 4 idle CTAs per round)
    for tiles in (16, 48):
        sp = lib.novic_debug_wgrad_splits(tiles, 304, 148)
        items = tiles * sp
        assert items % 148 == 0 or items % 148 >= 140, (tiles, sp)
    assert lib.novic_debug_wgrad_splits(0, 10, 148) == -1
