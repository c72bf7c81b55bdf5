"""Loader for tests/golden/reference_outputs.npz (outputs of the unmodified reference, see oracle/make_golden.py)."""
import os

import numpy as np
import torch

from novic_b200 import synth

import dataclasses

GOLDEN_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_outputs.npz")
VARIANTS_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_variants.npz")
TWINS_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "live_twins.npz")
B_GOLD = 32


class Golden:
    def __init__(self, path: str = GOLDEN_PATH):
        self._z = np.load(path)

    def __getitem__(self, key: str) -> torch.Tensor:
        return torch.from_numpy(self._z[key.replace("/", "__")])

    def has(self, key: str) -> bool:
        return key.replace("/", "__") in self._z.files


def check_twin(prefix: str, got: dict) -> None:
    """Compare values computed now with the `prefix__*` arrays of tests/golden/live_twins.npz (oracle/make_twin_golden.py): the same
    keys, shapes and dtypes; floating-point arrays within 1e-6, everything else exactly."""
    z = np.load(TWINS_PATH)
    want = {k[len(prefix) + 2:]: z[k] for k in z.files if k.startswith(prefix + "__")}
    assert want and set(got) == set(want), sorted(set(got) ^ set(want))[:10]
    for k, v in got.items():
        w = want[k]
        assert v.shape == w.shape and v.dtype == w.dtype, (k, v.shape, w.shape, v.dtype, w.dtype)
        assert np.allclose(v, w, rtol=0, atol=1e-6) if v.dtype.kind == "f" else np.array_equal(v, w), k


def weight_case(tag: str, dims: synth.DecoderDims = synth.DecoderDims()) -> dict:
    lively = synth.synth_state_dict(dims, seed=2, token_scale=0.25, jitter_norms=True)
    if tag == "lively":
        return lively
    if tag == "eos":
        return synth.make_eos_friendly(lively, dims, beta=0.1)
    if tag == "eosall":
        return synth.make_eos_ragged(lively)
    raise KeyError(tag)


def gold_embed() -> torch.Tensor:
    return synth.synth_embeddings(B_GOLD, seed=1234)


def guided_eval_case(dims: synth.DecoderDims = synth.DecoderDims()):
    """Guide set, targets drawn from it (one corrupted) and their padding - the inputs of the `tfg/*` fixtures (oracle/make_golden.py)."""
    gt = synth.synth_guide_targets(300, dims, seed=21, first_pool=24)
    idx = torch.randint(0, 300, (B_GOLD,), generator=torch.Generator().manual_seed(1))
    tgt = gt[idx].clone()
    tgt[5, 2] = 77
    pad = torch.zeros_like(tgt, dtype=torch.bool)
    pad[:, 1:] = (tgt[:, :-1] == 0).cummax(dim=1).values
    return gt, tgt, pad


# ----------------------------------------------------------------------------------------------------------------------
# Constructor variants (tests/golden/reference_variants.npz, written by oracle/make_golden_variants.py from the unmodified reference)
# ----------------------------------------------------------------------------------------------------------------------
BASE_DIMS = synth.DecoderDims()
# name -> (dims, constructor overrides)
VARIANTS = {
    "f768": (dataclasses.replace(BASE_DIMS, embed_dim=768), {}),
    "f1152": (dataclasses.replace(BASE_DIMS, embed_dim=1152), {}),
    "v6907": (dataclasses.replace(BASE_DIMS, vocab_size=6907), {}),
    "v6907q": (dataclasses.replace(BASE_DIMS, vocab_size=6907), dict(vocab_quant=True)),
    "ls01": (BASE_DIMS, dict(label_smoothing=0.1)),
    "nel2": (BASE_DIMS, dict(num_end_loss=2)),
    "causal": (BASE_DIMS, dict(strictly_causal=True)),
    "c12": (dataclasses.replace(BASE_DIMS, token_length=12), {}),
}
# name -> (dims, constructor overrides, multi-target count M or 0)
GRAD_CASES = {
    "grad_default": (BASE_DIMS, {}, 0),
    "grad_ls01": (BASE_DIMS, dict(label_smoothing=0.1), 0),
    "grad_v6907q": (dataclasses.replace(BASE_DIMS, vocab_size=6907), dict(vocab_quant=True), 0),
    "grad_nel2": (BASE_DIMS, dict(num_end_loss=2), 0),
    "grad_multi": (BASE_DIMS, {}, 3),
}
PROBE_SEED, NUM_PROBES = 99, 64
GRAD_PROBES, GRAD_PROJ = 256, 4


def variant_state_dict(dims: synth.DecoderDims, overrides: dict) -> dict:
    """The `eos` weight case at the variant's dimensions; with vocab_quant the tied matrix gets its quantisation rows
    (V .. ceil64(V)), which the reference requires to be zero when a checkpoint is loaded (verify_unused,
    embedding_decoder.py:437-441) and slices away from the logits (:726-727)."""
    lively = synth.synth_state_dict(dims, seed=2, token_scale=0.25, jitter_norms=True)
    sd = synth.make_eos_friendly(lively, dims, beta=0.1)
    if overrides.get("vocab_quant"):
        V = dims.vocab_size
        Vq = -(-V // 64) * 64
        sd["logits_linear.weight"] = torch.cat((sd["logits_linear.weight"], torch.zeros(Vq - V, dims.hidden_dim)), dim=0)
    if overrides.get("strictly_causal"):
        S = dims.max_seq_len
        sd["causality_mask"] = torch.triu(torch.full((S, S), float("-inf")), diagonal=1)
    return sd


def probe_columns(V: int) -> np.ndarray:
    return np.random.default_rng(PROBE_SEED).choice(V, size=NUM_PROBES, replace=False).astype(np.int64)


def grad_probe(index: int, numel: int):
    """Probed element indices and random projection vectors of the index-th parameter tensor (sorted by name)."""
    rng = np.random.default_rng(1000 + index)
    idx = rng.integers(0, numel, size=GRAD_PROBES)
    proj = rng.standard_normal((GRAD_PROJ, numel)).astype(np.float32)
    return idx, proj


def grad_case_inputs(dims: synth.DecoderDims, multi: int):
    """(embed, target, padding, weight) of a gradient fixture."""
    if multi:
        embed = synth.synth_embeddings(8, dims.embed_dim, seed=1234)
        tgt, pad = synth.synth_targets(8, dims, seed=6, multi=multi)
        w = torch.from_numpy(np.random.default_rng(8).random((8, multi)).astype(np.float32))
        w[1, 2] = 0.0
        return embed, tgt, pad, w
    embed = synth.synth_embeddings(B_GOLD, dims.embed_dim, seed=1234)
    tgt, pad = synth.synth_targets(B_GOLD, dims, seed=5)
    return embed, tgt, pad, None
