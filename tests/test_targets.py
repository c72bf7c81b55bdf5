"""Target id formats (SURVEY.md section 8 row f4): novic_b200.targets against the unmodified reference Embedder
(embedders.py:169-254 create_target_config, :331-385 tokenize_target, :387-406 detokenize_target) driven by a toy word-piece
tokenizer, over every combination of the format switches; plus reference-free round-trip properties."""
import itertools

import pytest
import torch

from novic_b200.targets import TokenizerIds, decode_targets, encode_targets, make_target_format
from oracle import refload

NOUNS = ("cat", "dog", "zebra", "ox", "armadillo", "bee", "yak", "a", "newt", "quokka")
BATCHES = (("cat", "armadillo", "ox"), ("a",), ("bee", "yak"), NOUNS)


def _raw(texts, start, end, pad, max_tokens=None):
    """Toy tokenizer: one id per letter (a = 5 ...), optional start token, end token, padded exactly to the longest text."""
    rows = [([start] if start is not None else []) + [5 + ord(c) - ord("a") for c in t] + [end] for t in texts]
    T = max(len(r) for r in rows)
    ids = torch.full((len(rows), T), pad, dtype=torch.int64)
    attn = torch.zeros((len(rows), T), dtype=torch.int64)
    for i, r in enumerate(rows):
        ids[i, : len(r)] = torch.tensor(r)
        attn[i, : len(r)] = 1
    return ids, attn


TOKENIZERS = {"clip_like": dict(start=40, end=41, pad=0), "no_start": dict(start=None, end=41, pad=0), "pad_is_end": dict(start=40, end=41, pad=41)}
SWITCHES = [dict(zip(("with_start_token", "with_end_token", "compact_ids", "fixed_token_length", "auto_fixed_token_length", "use_masks"), v))
            for v in itertools.product((False, True), repeat=6)]


def _tok(spec):
    return TokenizerIds(vocab_size=42, start_token_id=spec["start"], end_token_id=spec["end"], pad_token_id=spec["pad"], context_length=16)


@pytest.fixture(scope="module")
def ref():
    if not refload.available():
        pytest.skip("reference tree not present")
    return refload.import_reference()


def _toy_embedder(ref, spec):
    class Toy(ref.embedders.Embedder):
        def tokenize(self, text, max_tokens=None, output_dict=False):
            ids, attn = _raw((text,) if isinstance(text, str) else tuple(text), spec["start"], spec["end"], spec["pad"])
            return dict(input_ids=ids, attention_mask=attn) if output_dict else ids

        def detokenize(self, token_ids):
            return token_ids.clone()            # hand back what detokenize_target passes to the tokenizer

    return Toy(configuration={}, context_length=16, vocab_size=42, cased_tokens=False, start_token_id=spec["start"], end_token_id=spec["end"],
               pad_token_id=spec["pad"], token_dtype=torch.int64, embed_dtype=torch.float32, embed_dim=8, load_model=False, device="cpu")


@pytest.mark.parametrize("name", sorted(TOKENIZERS))
def test_formats_match_the_reference_embedder(ref, name):
    spec = TOKENIZERS[name]
    tok = _tok(spec)
    emb = _toy_embedder(ref, spec)
    all_ids, all_attn = _raw(NOUNS, spec["start"], spec["end"], spec["pad"])
    for sw in SWITCHES:
        cfg = emb.create_target_config(NOUNS, **sw)
        fmt = make_target_format(all_ids, all_attn, tok, **sw)
        for f in ("vocab_size", "token_dtype", "start_token_id", "end_token_id", "pad_token_id", "compact_ids", "fixed_token_length", "token_length", "use_masks"):
            assert getattr(fmt, f) == getattr(cfg, f), (sw, f)
        for f in ("compact_map", "compact_unmap"):
            a, b = getattr(fmt, f), getattr(cfg, f)
            assert (a is None) == (b is None) and (a is None or (a.dtype == b.dtype and torch.equal(a, b))), (sw, f)
        emb.configure_target(cfg, NOUNS)
        for batch in BATCHES:
            want_ids, want_mask = emb.tokenize_target(batch)
            ids, attn = _raw(batch, spec["start"], spec["end"], spec["pad"])
            got_ids, got_mask = encode_targets(ids, attn, tok, fmt)
            assert got_ids.dtype == want_ids.dtype and torch.equal(got_ids, want_ids), (sw, batch)
            assert (got_mask is None) == (want_mask is None) and (got_mask is None or torch.equal(got_mask, want_mask)), (sw, batch)
            assert torch.equal(decode_targets(got_ids, tok, fmt), emb.detokenize_target(want_ids)), (sw, batch)
            stacked = torch.stack((got_ids, got_ids.flip(0)), dim=1)                       # [B, K, S] like generate_beam's output
            want3 = torch.stack(emb.detokenize_target(stacked))
            assert torch.equal(decode_targets(stacked, tok, fmt), want3), (sw, batch)


@pytest.mark.parametrize("name", sorted(TOKENIZERS))
def test_round_trip_and_format_invariants(name):
    """Reference-free: compact ids are dense over exactly the used tokens, padding masks mark exactly the pad positions, and decoding
    gives back the tokenizer's content ids."""
    spec = TOKENIZERS[name]
    tok = _tok(spec)
    all_ids, all_attn = _raw(NOUNS, spec["start"], spec["end"], spec["pad"])
    letters = sorted({5 + ord(c) - ord("a") for t in NOUNS for c in t})
    for sw in SWITCHES:
        fmt = make_target_format(all_ids, all_attn, tok, **sw)
        longest = max(len(t) for t in NOUNS)
        have_start = sw["with_start_token"] and (sw["compact_ids"] or spec["start"] is not None)
        if not sw["fixed_token_length"] or sw["auto_fixed_token_length"]:
            assert fmt.token_length == longest + int(sw["with_start_token"]) + int(sw["with_end_token"])
        else:
            assert fmt.token_length == tok.context_length
        if sw["compact_ids"]:
            n_special = 1 + int(sw["with_start_token"])
            assert fmt.vocab_size == n_special + len(letters) and fmt.compact_unmap[n_special:].tolist() == letters
            assert fmt.compact_map[fmt.compact_unmap[n_special:]].tolist() == list(range(n_special, fmt.vocab_size))
            assert int((fmt.compact_map >= 0).sum()) >= len(letters)
        ids, attn = _raw(NOUNS, spec["start"], spec["end"], spec["pad"])
        out, mask = encode_targets(ids, attn, tok, fmt)
        assert int(out.min()) >= 0 and int(out.max()) < fmt.vocab_size
        if sw["fixed_token_length"]:
            assert out.shape[1] == fmt.token_length
        back = decode_targets(out, tok, fmt)
        for i, t in enumerate(NOUNS):
            content = [5 + ord(c) - ord("a") for c in t]
            row = back[i].tolist()
            off = 1 if (have_start and not (sw["compact_ids"] and spec["start"] is None)) else 0
            assert row[off: off + len(content)] == content, (sw, t)
            if mask is not None:
                n_kept = len(content) + int(have_start) + int(sw["with_end_token"])
                assert mask[i].tolist() == [False] * n_kept + [True] * (out.shape[1] - n_kept), (sw, t)


def test_bad_inputs_raise():
    tok = _tok(TOKENIZERS["clip_like"])
    ids, attn = _raw(NOUNS, 40, 41, 0)
    fmt = make_target_format(ids[:3], attn[:3], tok, with_start_token=False, with_end_token=True, compact_ids=True, fixed_token_length=True,
                             auto_fixed_token_length=True, use_masks=True)
    with pytest.raises(ValueError):
        encode_targets(ids, attn, tok, fmt)                       # 'armadillo' is longer than the fixed length derived from three short nouns
    with pytest.raises(ValueError):
        make_target_format(ids[0], attn[0], tok, with_start_token=False, with_end_token=True, compact_ids=True, fixed_token_length=False,
                           auto_fixed_token_length=False, use_masks=True)


@pytest.mark.parametrize("name", sorted(TOKENIZERS))
def test_formats_match_committed_reference_vectors(name):
    """The same comparison against tests/golden/targets_expected.npz (oracle/make_targets_golden.py: outputs of the unmodified
    reference) - runs where the reference tree is absent."""
    import os
    import numpy as np
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "targets_expected.npz"))
    spec = TOKENIZERS[name]
    tok = _tok(spec)
    all_ids, all_attn = _raw(NOUNS, spec["start"], spec["end"], spec["pad"])
    none = -(2 ** 31)
    for si, sw in enumerate(SWITCHES):
        fmt = make_target_format(all_ids, all_attn, tok, **sw)
        key = f"{name}__{si}"
        got = [fmt.vocab_size, none if fmt.start_token_id is None else fmt.start_token_id, none if fmt.end_token_id is None else fmt.end_token_id,
               fmt.pad_token_id, fmt.token_length]
        assert got == z[f"{key}__scalars"].tolist(), sw
        if fmt.compact_ids:
            assert np.array_equal(fmt.compact_map.numpy(), z[f"{key}__map"]) and np.array_equal(fmt.compact_unmap.numpy(), z[f"{key}__unmap"]), sw
        for bi, batch in enumerate(BATCHES):
            ids, attn = _raw(batch, spec["start"], spec["end"], spec["pad"])
            out, mask = encode_targets(ids, attn, tok, fmt)
            assert np.array_equal(out.numpy(), z[f"{key}__b{bi}__ids"]), (sw, batch)
            assert (mask is None) == (f"{key}__b{bi}__mask" not in z.files) and (mask is None or np.array_equal(mask.numpy(), z[f"{key}__b{bi}__mask"])), (sw, batch)
            assert np.array_equal(decode_targets(out, tok, fmt).numpy(), z[f"{key}__b{bi}__raw"]), (sw, batch)


def random_cases():
    """The cases of test_random_vocabularies_match_the_reference_embedder, drawn from the same seeded stream in the same order:
    (trial, case within the trial, tokenizer name, nouns, switch index, batch)."""
    import random
    rng = random.Random(1234)
    for trial in range(25):
        name = rng.choice(sorted(TOKENIZERS))
        alphabet = rng.sample("abcdefghijklmnopqrstuvwxyz", rng.randint(1, 26))
        nouns = tuple(dict.fromkeys("".join(rng.choice(alphabet) for _ in range(rng.randint(1, 12))) for _ in range(rng.randint(1, 30))))
        for k, sw in enumerate(rng.sample(SWITCHES, 6)):
            batch = tuple(rng.sample(nouns, rng.randint(1, len(nouns))))
            yield trial, k, name, nouns, SWITCHES.index(sw), batch


def random_vocabulary_values() -> dict:
    """Per trial of random_cases(): the format fields, compact maps, encoded ids / mask and decoded ids that the live test asserts
    equal to the reference Embedder's, packed into one int64 vector per trial (each case: switch index, vocab_size, start, end,
    pad, token_length with None as -2^31, then map, unmap, ids, mask, decoded ids, each as ndim, shape, values or as -1 when
    absent), and the trial's nouns and batches as words ("|" before each batch)."""
    import numpy as np
    none = -(2 ** 31)
    ints, words = {}, {}
    for trial, k, name, nouns, si, batch in random_cases():
        spec = TOKENIZERS[name]
        tok = _tok(spec)
        fmt = make_target_format(*_raw(nouns, spec["start"], spec["end"], spec["pad"]), tok, **SWITCHES[si])
        ids, mask = encode_targets(*_raw(batch, spec["start"], spec["end"], spec["pad"]), tok, fmt)
        parts = [[si, fmt.vocab_size, none if fmt.start_token_id is None else fmt.start_token_id,
                  none if fmt.end_token_id is None else fmt.end_token_id, fmt.pad_token_id, fmt.token_length]]
        for t in (fmt.compact_map if fmt.compact_ids else None, fmt.compact_unmap if fmt.compact_ids else None, ids, mask,
                  decode_targets(ids, tok, fmt)):
            parts += [[-1]] if t is None else [[t.ndim, *t.shape], t.flatten().tolist()]
        ints.setdefault(trial, []).extend(v for p in parts for v in p)
        words.setdefault(trial, list(nouns)).extend(("|",) + batch)
    out = {f"{t}__ints": np.array(v, dtype=np.int64) for t, v in ints.items()}
    out.update({f"{t}__words": np.array(v) for t, v in words.items()})
    return out


def test_random_vocabularies_match_committed_reference_values():
    """test_random_vocabularies_match_the_reference_embedder without the reference tree: the same seeded cases against the stored
    values that test asserts equal to the reference Embedder's (tests/golden/live_twins.npz)."""
    from tests.golden_util import check_twin
    check_twin("rand", random_vocabulary_values())


def test_random_vocabularies_match_the_reference_embedder(ref):
    """Seeded random noun lists (1-12 letters from random alphabets, duplicates of letters, single-noun lists) and random switch
    choices against the live reference."""
    import random
    rng = random.Random(1234)
    for trial in range(25):
        name = rng.choice(sorted(TOKENIZERS))
        spec = TOKENIZERS[name]
        tok = _tok(spec)
        alphabet = rng.sample("abcdefghijklmnopqrstuvwxyz", rng.randint(1, 26))
        nouns = tuple(dict.fromkeys("".join(rng.choice(alphabet) for _ in range(rng.randint(1, 12))) for _ in range(rng.randint(1, 30))))
        emb = _toy_embedder(ref, spec)
        all_ids, all_attn = _raw(nouns, spec["start"], spec["end"], spec["pad"])
        for sw in rng.sample(SWITCHES, 6):
            cfg = emb.create_target_config(nouns, **sw)
            fmt = make_target_format(all_ids, all_attn, tok, **sw)
            assert (fmt.vocab_size, fmt.start_token_id, fmt.end_token_id, fmt.pad_token_id, fmt.token_length) == \
                   (cfg.vocab_size, cfg.start_token_id, cfg.end_token_id, cfg.pad_token_id, cfg.token_length), (trial, sw)
            if cfg.compact_ids:
                assert torch.equal(fmt.compact_map, cfg.compact_map) and torch.equal(fmt.compact_unmap, cfg.compact_unmap), (trial, sw)
            emb.configure_target(cfg, nouns)
            batch = tuple(rng.sample(nouns, rng.randint(1, len(nouns))))
            want_ids, want_mask = emb.tokenize_target(batch)
            got_ids, got_mask = encode_targets(*_raw(batch, spec["start"], spec["end"], spec["pad"]), tok, fmt)
            assert torch.equal(got_ids, want_ids) and ((got_mask is None and want_mask is None) or torch.equal(got_mask, want_mask)), (trial, sw)
            assert torch.equal(decode_targets(got_ids, tok, fmt), emb.detokenize_target(want_ids)), (trial, sw)
