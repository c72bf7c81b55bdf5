"""novic_b200.stats.GenerationStats (SURVEY.md section 8 row f4): validity statistics on token ids against the reference's
GenerationTask.update (infer.py:613-644) run on strings.  The reference detokenises with the CLIP tokenizer (not available offline); the
test gives it an injective stand-in (the ids up to the end token, joined), for which string membership and id membership coincide."""
import types

import numpy as np
import pytest
import torch

from novic_b200 import stats, synth
from tests.golden_util import check_twin

DIMS = synth.DecoderDims()
G = DIMS.token_length - 1


def detok(rows: torch.Tensor):
    def one(r):
        out = []
        for t in r.tolist():
            if t == 0:
                break
            out.append(str(t))
        return " ".join(out)
    if rows.ndim == 3:
        return [[one(r) for r in b] for b in rows]
    return [one(r) for r in rows]


def make_case(seed=0, B=40, K=5):
    g = torch.Generator().manual_seed(seed)
    guide_t = synth.synth_guide_targets(120, DIMS, seed=41, first_pool=12)
    vocab_t = torch.cat((guide_t[:80], synth.synth_guide_targets(60, DIMS, seed=42, first_pool=12)))
    classes = [guide_t[torch.randint(0, 120, (3,), generator=g)] for _ in range(7)]
    # predictions: a mix of guide nouns, vocabulary-only nouns and random junk, with ragged padding
    pool = torch.cat((guide_t, vocab_t, synth.synth_guide_targets(60, DIMS, seed=43, first_pool=12)))
    target = pool[torch.randint(0, pool.shape[0], (B, K), generator=g)][:, :, :G].clone()
    padding = torch.zeros_like(target, dtype=torch.bool)
    padding[:, :, 1:] = (target[:, :, :-1] == 0).cummax(dim=2).values
    class_idx = torch.randint(0, 7, (B,), generator=g).tolist()
    return guide_t, vocab_t, classes, target, padding, class_idx


@pytest.mark.reference
@pytest.mark.parametrize("use_classes", (False, True))
def test_stats_match_reference_generation_task(use_classes):
    from oracle import refload
    ref = refload.import_reference()
    guide_t, vocab_t, classes, target, padding, class_idx = make_case()
    K = target.shape[1]
    fake_decoder = types.SimpleNamespace(embedder=types.SimpleNamespace(detokenize_target=detok, embed_dtype=torch.float32))
    gencfg = types.SimpleNamespace(topk=K, vocab_prior=False, guided=False, method="beam")
    task = ref.infer.GenerationTask(gencfg=gencfg, decoder=fake_decoder, vocab_targets_set=set(detok(vocab_t)), vocab_targets=None,
                                    guide_targets_set=set(detok(guide_t)), guide_targets=None,
                                    class_lists=[detok(c) for c in classes] if use_classes else None)
    mine = stats.GenerationStats(K, vocab_t, guide_t, G, DIMS.vocab_size, device="cpu", class_targets=classes if use_classes else None)
    score = torch.zeros(target.shape[:2])
    for lo, hi in ((0, 16), (16, 40)):           # two batches: the counters accumulate
        ci = class_idx[lo:hi] if use_classes else None
        task.update(target[lo:hi], padding[lo:hi], score[lo:hi], class_indices=ci)
        mine.update(target[lo:hi], padding[lo:hi], score[lo:hi], class_indices=ci)
        assert torch.equal(mine.valid_vocab, task.valid_vocab) and torch.equal(mine.valid_guide, task.valid_guide)
        assert torch.equal(mine.correct, task.correct) and torch.equal(mine.invalid, task.invalid) and torch.equal(mine.result, task.result)
        assert torch.equal(mine.topk_counts, task.topk_counts) and mine.num_samples == task.num_samples
        for name in ("topk", "topk_guide", "topk_vocab", "topk_invalid", "topk_valid"):
            assert torch.allclose(getattr(mine, name), getattr(task, name)), name
    assert mine.valid_guide.any() and mine.valid_vocab.any() and mine.invalid.any() and (not use_classes or mine.correct.any())


STATS_FIELDS = ("valid_vocab", "valid_guide", "correct", "invalid", "result", "topk_counts", "topk", "topk_guide", "topk_vocab", "topk_invalid",
                "topk_valid")


def stats_values(use_classes: bool) -> dict:
    """The counters test_stats_match_reference_generation_task compares, after each of its two batches: {"<batch>__<field>": array}."""
    guide_t, vocab_t, classes, target, padding, class_idx = make_case()
    K = target.shape[1]
    mine = stats.GenerationStats(K, vocab_t, guide_t, G, DIMS.vocab_size, device="cpu", class_targets=classes if use_classes else None)
    score = torch.zeros(target.shape[:2])
    out = {}
    for j, (lo, hi) in enumerate(((0, 16), (16, 40))):
        mine.update(target[lo:hi], padding[lo:hi], score[lo:hi], class_indices=class_idx[lo:hi] if use_classes else None)
        out.update({f"{j}__{f}": getattr(mine, f).numpy() for f in STATS_FIELDS})
        out[f"{j}__num_samples"] = np.array(mine.num_samples, dtype=np.int64)
    return out


@pytest.mark.parametrize("use_classes", (False, True))
def test_stats_match_committed_reference_values(use_classes):
    """test_stats_match_reference_generation_task without the reference tree: the same inputs against the stored values of the
    counters that test asserts equal to the reference's (tests/golden/live_twins.npz)."""
    check_twin(f"stats__{int(use_classes)}", stats_values(use_classes))


def test_membership_semantics_without_reference():
    guide_t, vocab_t, classes, target, padding, class_idx = make_case(seed=3)
    K = target.shape[1]
    mine = stats.GenerationStats(K, vocab_t, guide_t, G, DIMS.vocab_size, device="cpu", class_targets=classes)
    mine.update(target, padding, None, class_indices=class_idx)
    gset, vset = set(detok(guide_t)), set(detok(vocab_t))
    strs = detok(target)
    want_g = torch.tensor([[s in gset for s in row] for row in strs])
    want_v = torch.tensor([[s in vset for s in row] for row in strs])
    want_c = torch.tensor([[s in set(detok(classes[c])) for s in row] for c, row in zip(class_idx, strs)])
    assert torch.equal(mine.valid_guide, want_g) and torch.equal(mine.valid_vocab, want_v) and torch.equal(mine.correct, want_c)
    assert mine.topk_counts[-1, 0] == int(want_c.any(dim=1).sum())                 # top-K any-correct count
    assert (mine.topk[1:] >= mine.topk[:-1]).all() and (mine.topk_invalid[1:] >= mine.topk_invalid[:-1]).all()


@pytest.mark.gpu
def test_stats_on_device_after_guided_beam():
    """End of the real path: guided beam-5 on the GPU, statistics on the device - every beam must count as a valid guide noun."""
    from novic_b200 import default_decoder
    gt = synth.synth_guide_targets(500, DIMS, seed=33, first_pool=40)
    model = default_decoder(DIMS, synth.synth_state_dict(DIMS, seed=2, token_scale=0.25, jitter_norms=True)).to("cuda:0")
    embed = synth.synth_embeddings(64, seed=8).to("cuda:0")
    with torch.inference_mode():
        tok, pad, score = model.generate_beam(embed, 5, 1.0, 0.0, None, False, 0.0, gt.to("cuda:0"), False)
        st = stats.GenerationStats(5, gt[:300], gt, G, DIMS.vocab_size, device="cuda:0").update(tok, pad, score)
    assert st.valid_guide.all() and st.topk_guide[-1].item() == 1.0 and st.topk_invalid[-1].item() == 0.0
    assert 0.0 < st.valid_vocab.float().mean().item() < 1.0
