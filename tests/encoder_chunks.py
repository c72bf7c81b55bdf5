"""Shared by the encoder test modules: one encode at a production chunk size, where every trunk GEMM has enough tiles for the CTA-pair
kernel (at least 2 x 148 tiles of 128 x 256), checked against the CPU restatement on sampled images, against chunks of two, under the
tile and store switches and on a poisoned workspace.

Why the results must be bit-identical across chunk sizes and switches: every GEMM output element is one row of A against one row of W,
accumulated over the same k-blocks in the same order whatever the tile shape (128 x 128, 128 x 256, or a CTA pair's 256 x 256), and the
epilogues apply the same fp32 operations element by element; attention items (image, head, query tile) are independent of the grid and
of each other.  The mma.sync attention (NOVIC_VIT_ATTN=mma) accumulates in another order and is held to the restatement bounds instead.
"""
from __future__ import annotations

import dataclasses
from typing import Callable

import torch

DEV = "cuda:0"
SWITCHES = [("NOVIC_VIT_BN", "256"), ("NOVIC_VIT_BN", "128"), ("NOVIC_VIT_DIRECT", "0")]


@dataclasses.dataclass
class ChunkRun:
    enc: torch.nn.Module
    img: torch.Tensor                 # [n, 3, S, S] on the CPU
    got: torch.Tensor                 # features of all n images from one chunk, on the CPU
    sample: list                      # image indices checked against the restatement
    ref: torch.Tensor
    ref16: torch.Tensor


def pair_epilogues(fn: Callable[[], object]) -> set:
    """The epilogues that ran on gemm2_kernel (CTA pairs) while fn ran, from the torch.profiler kernel list."""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages() if "gemm2_kernel" in e.key]
    return {epi for epi in ("EpiVitBias", "EpiVitResid", "EpiVitStoreF32") if any(epi in n for n in names)}


def check_bounds(got: torch.Tensor, ref: torch.Tensor, ref16: torch.Tensor, rel_tol: float, tight_tol: float, what: str) -> None:
    """The encoder tests' bounds: ||d|| / ||ref|| <= rel_tol, max |d| <= 6 rel_tol * rms, cosine >= 0.999; <= tight_tol against the
    bf16-operand restatement."""
    rms = ref.pow(2).mean().sqrt().item()
    err = ((got - ref).norm() / ref.norm()).item()
    worst = (got - ref).abs().max().item() / rms
    cos = torch.nn.functional.cosine_similarity(got, ref, dim=1).min().item()
    err16 = ((got - ref16).norm() / ref16.norm()).item()
    print(f"{what}: ||d|| / ||ref|| = {err:.4f}, max |d| / rms = {worst:.4f}, min cosine = {cos:.6f}; against the bf16-operand restatement {err16:.5f}")
    assert err <= rel_tol and worst <= 6 * rel_tol and cos >= 0.999
    assert err16 <= tight_tol


def production_chunk(make_enc: Callable[[int], torch.nn.Module], images: torch.Tensor, restate: Callable, rel_tol: float, tight_tol: float,
                     pair_epis: set) -> ChunkRun:
    """All images in one chunk: the pair kernel ran for every epilogue in pair_epis; the first, middle and last images are within the
    restatement bounds; every image's features equal those from chunks of two, bit for bit."""
    n = images.shape[0]
    enc = make_enc(n)
    x = images.to(DEV)
    out = {}
    with torch.inference_mode():
        ran = pair_epilogues(lambda: out.setdefault("got", enc.encode_image(x)))
        got = out["got"].cpu()
        sample = [0, n // 2, n - 1]
        ref = restate(images[sample], False)
        ref16 = restate(images[sample], True)
        check_bounds(got[sample], ref, ref16, rel_tol, tight_tol, f"{n} images in one chunk, images {sample}")
        enc.images_per_chunk = 2
        got2 = enc.encode_image(x).cpu()
        enc.images_per_chunk = n
    assert pair_epis <= ran, f"gemm2_kernel ran for {sorted(ran)}, expected {sorted(pair_epis)}"
    assert torch.equal(got, got2), f"chunks of {n} and of 2 differ: max |d| = {(got - got2).abs().max().item():.3e}"
    return ChunkRun(enc, images, got, sample, ref, ref16)


def same_under_switches(run: ChunkRun, make_enc: Callable[[int], torch.nn.Module], monkeypatch) -> None:
    """NOVIC_VIT_BN=256 and 128 (single-CTA tiles) and NOVIC_VIT_DIRECT=0 (staged bf16 stores) give the same features bit for bit.
    The switches are read when a handle is created; a handle created after them without them is back on the defaults."""
    n = run.img.shape[0]
    x = run.img.to(DEV)
    for name, value in SWITCHES:
        with monkeypatch.context() as m:
            m.setenv(name, value)
            with torch.inference_mode():
                got = make_enc(n).encode_image(x).cpu()
        assert torch.equal(got, run.got), f"{name}={value} changes the features: max |d| = {(got - run.got).abs().max().item():.3e}"
    with torch.inference_mode():
        ran = pair_epilogues(lambda: make_enc(n).encode_image(x))
    assert "EpiVitBias" in ran, "a handle created without the switches is not back on CTA pairs"


def poisoned_workspace(run: ChunkRun) -> None:
    """A workspace filled with 0xFF (NaN in bf16 and fp32) gives the same features: every byte an encode reads, it wrote."""
    x = run.img.to(DEV)
    with torch.inference_mode():
        run.enc._handles[0]["ws"].fill_(0xFF)
        got = run.enc.encode_image(x).cpu()
    assert torch.isfinite(got).all()
    assert torch.equal(got, run.got)
