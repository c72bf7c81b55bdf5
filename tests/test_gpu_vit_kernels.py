"""The image encoders' kernels one at a time against float64 torch on the same bf16 operands, through the encoder's own launch helpers
(novic_debug_vit_gemm / _vit_attention / _siglip_map_attention / _vit_layernorm).

The end-to-end encoder tests see every kernel through LayerNorms and the residual stream, at a few images per chunk.  Here each kernel
runs alone, on the paths production chunk sizes take, with inputs chosen so that a subtle bug is large:

- GEMM: every ViT epilogue (EpiVitBias with no activation, QuickGELU and erf GELU, direct and staged stores; EpiVitResid in residual mode
  and in patch mode behind 0 or 1 class token; EpiVitStoreF32 with and without bias) on 128 x 128, 128 x 256 and CTA-pair 256 x 256 tiles,
  at ragged M (1, 127, 129, 257, 383: an odd number of 128-row tiles leaves the pair's second CTA without rows) and N (1152 and 3456 end
  inside the B half of the last pair tile), and on a grid divided by 8 and 37 so that few CTAs walk many tiles (both accumulator stages, the
  ring's phase wrap).  bf16 outputs are within one bf16 ulp of the rounded fp64 result (plus the fp32 accumulation allowance), fp32
  outputs within 1e-5 * sum|a * w|.
- tcgen05 attention (D = 64, 72, 80) and the mma.sync one (D = 80) at 1 to 730 tokens, on the encoder's grid and on 1 or 3 persistent
  CTAs, so that item boundaries fall at every phase of the three-stage K / V^T ring.  Inputs: every valid score about -30 (a padded key
  scores 0 and would take almost all the weight), one dominant key at 0, 127, 128 or T - 1, scores rising with the key index (the running
  maximum moves on every tile: the O rescale), and for D = 72 channels 0..7 of every next head (and K head 0, behind the last head's Q) at
  +-64, which any leak of the foreign channels 72..79 turns into a large error.  Bound: |got - ref| <= 4e-3 * max|v| + 2^-8 * |ref| (P is
  rounded to bf16, the output is bf16).
- The MAP head's attention at 1 to 3072 tokens, heads of 64 and 72, with the same inputs.
- LayerNorm at every instantiated width: rows of mean 1e3 and standard deviation 0.1 (a one-pass variance cancels catastrophically), the
  class-token seat, the chained second norm, in-place storage and a row stride of T * W.

Every output buffer starts as NaN with guard rows (and, where the layout has them, guard columns): each element a kernel owns is written,
and nothing else is.
"""
import math

import pytest
import torch

from novic_b200 import _abi

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F64 = torch.float64
WORST: dict = {}           # family -> worst |error| / bound seen in this session (printed by the last test of each family)


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _note(family: str, ratio: float) -> None:
    WORST[family] = max(WORST.get(family, 0.0), ratio)


def _bf16(shape, gen, std=1.0) -> torch.Tensor:
    return (torch.randn(shape, generator=gen, device=gen.device) * std).to(torch.bfloat16)


def _bf16_ulp(x: torch.Tensor) -> torch.Tensor:
    """bf16 spacing at |x| (8 significant bits)"""
    ax = x.abs().clamp_min(2.0 ** -126)
    return torch.exp2(torch.floor(torch.log2(ax)) - 7)


# ---------------------------------------------------------------------------------------------------------------------------------
# GEMM epilogues on every tile path
# ---------------------------------------------------------------------------------------------------------------------------------
SHAPES = [(1, 768, 640), (127, 1152, 768), (129, 2304, 1152), (257, 3456, 768), (383, 1152, 4352), (383, 4352, 640), (4096, 4352, 1152),
          (4096, 3456, 768)]
EPIS = [("bias_none_direct", 0, 0, 1), ("bias_none_staged", 0, 0, 0), ("bias_quickgelu_direct", 0, 1, 1), ("bias_quickgelu_staged", 0, 1, 0),
        ("bias_gelu_direct", 0, 2, 1), ("bias_gelu_staged", 0, 2, 0), ("resid", 1, 0, 0), ("patch_tok0", 1, 0, 0), ("patch_tok1", 1, 0, 0),
        ("f32_bias", 2, 0, 0), ("f32_nobias", 2, 0, 0)]
PRE = 256                  # guard elements in front of every output (keeps the 32-byte alignment of direct stores)


def _act(x: torch.Tensor, act: int) -> torch.Tensor:
    if act == 1:
        return x * torch.sigmoid(1.702 * x)
    if act == 2:
        return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))
    return x


def _run_gemm(name: str, epi: int, act: int, direct: int, M: int, N: int, K: int, path: int, grid_div: int, seed: int) -> float:
    gen = torch.Generator(device=DEV).manual_seed(seed)
    a = _bf16((M, K), gen)
    w = _bf16((N, K), gen, std=K ** -0.5)
    bias = None if name == "f32_nobias" else torch.randn(N, generator=gen, device=DEV) * 0.5
    acc = a.to(F64) @ w.to(F64).T
    absacc = a.to(F64).abs() @ w.to(F64).abs().T
    pre = acc + (bias.to(F64) if bias is not None else 0.0)
    lib = _abi.lib()
    table, patches, tok0 = None, 0, 0
    if epi == 2:
        ld, rows = N, M
    else:
        ld = N + 64                                        # guard columns
        rows = M
        if name.startswith("patch"):
            tok0 = 1 if name == "patch_tok1" else 0
            nimg = 16 if M == 4096 else 3 if M == 129 else 1
            patches = M // nimg
            rows = nimg * (patches + tok0)
            table = torch.randn(patches + tok0, ld, generator=gen, device=DEV)
    dtype = torch.bfloat16 if epi == 0 else torch.float32
    buf = torch.full((PRE + (rows + 3) * ld,), float("nan"), dtype=dtype, device=DEV)
    out = buf[PRE:PRE + rows * ld].view(rows, ld)
    x0 = None
    if name == "resid":
        x0 = torch.randn(rows, N, generator=gen, device=DEV)
        out[:, :N] = x0
    cls_rows = None
    if tok0:
        cls_rows = torch.arange(0, rows, patches + tok0, device=DEV)
        out[cls_rows] = torch.randn(len(cls_rows), ld, generator=gen, device=DEV)      # sentinels: must stay bit for bit
    before = buf.clone()
    rc = lib.novic_debug_vit_gemm(a.data_ptr(), w.data_ptr(), M, N, K, epi, act, direct, bias.data_ptr() if bias is not None else None,
                                  out.data_ptr(), ld, table.data_ptr() if table is not None else None, patches, tok0, path, grid_div, _stream())
    _abi.check(rc)
    torch.cuda.synchronize()
    # which elements the kernel owns, and what they must hold
    own = torch.zeros(rows, ld, dtype=torch.bool, device=DEV)
    ref = torch.zeros(rows, ld, dtype=F64, device=DEV)
    slack = torch.zeros(rows, ld, dtype=F64, device=DEV)
    if table is not None:
        img = torch.arange(M, device=DEV) // patches
        p = torch.arange(M, device=DEV) - img * patches
        dst = img * (patches + tok0) + tok0 + p
        own[dst, :N] = True
        ref[dst, :N] = pre + table[tok0 + p, :N].to(F64)
        slack[dst, :N] = absacc
    else:
        own[:M, :N] = True
        ref[:M, :N] = pre if x0 is None else pre + x0.to(F64)
        slack[:M, :N] = absacc
    got = out.to(F64)
    if epi == 0:
        y = _act(pre, act)
        ref[:M, :N] = y
        # one bf16 ulp of the rounded result; fp32 accumulation (x the activation's slope, <= 1.13); the fast erf / exp (<= 2e-7 |x|)
        bound = _bf16_ulp(torch.maximum(y.abs(), got[:M, :N].abs())) + 1.2e-5 * absacc + 1e-6 * (1 + pre.abs())
    else:
        bound = (1e-5 * slack + 2.0 ** -22 * (ref.abs() + (x0.to(F64).abs().max() if x0 is not None else 0)))[own].view(-1)
    err = (got - ref)
    if epi == 0:
        e = err[:M, :N].abs()
        assert not torch.isnan(got[:M, :N]).any(), f"{name}: owned elements left unwritten"
        ratio = (e / bound).max().item()
    else:
        e = err[own]
        assert not torch.isnan(e).any(), f"{name}: owned elements left unwritten"
        ratio = (e.abs() / bound).max().item()
    # nothing outside the owned elements changes: guard columns, guard rows, the prefix, class-token rows (bit for bit)
    owned_flat = torch.zeros_like(buf, dtype=torch.bool)
    owned_flat[PRE:PRE + rows * ld] = own.view(-1)
    untouched = ~owned_flat
    assert torch.equal(buf[untouched].view(torch.int16 if epi == 0 else torch.int32), before[untouched].view(torch.int16 if epi == 0 else torch.int32)), \
        f"{name}: elements outside the output were written"
    _note("gemm", ratio)
    return ratio


@pytest.mark.parametrize("path", [128, 256, 512])
@pytest.mark.parametrize("name,epi,act,direct", EPIS, ids=[e[0] for e in EPIS])
def test_vit_gemm_epilogue_on_every_path(name, epi, act, direct, path):
    worst = 0.0
    for i, (M, N, K) in enumerate(SHAPES):
        r = _run_gemm(name, epi, act, direct, M, N, K, path, 1, seed=1000 * i + path + 17 * epi + 5 * act + direct)
        assert r <= 1.0, f"{name} path {path} M={M} N={N} K={K}: error / bound = {r:.3f}"
        worst = max(worst, r)
    print(f"gemm {name} path {path}: worst error / bound {worst:.3f}")


@pytest.mark.parametrize("grid_div", [8, 37])
@pytest.mark.parametrize("path", [128, 256, 512])
@pytest.mark.parametrize("name", ["bias_gelu_direct", "bias_none_staged", "resid", "patch_tok1", "f32_bias"])
def test_vit_gemm_few_ctas_walk_many_tiles(name, path, grid_div):
    """148 / 37 = 4 CTAs (2 pairs) walk up to 1088 tiles: every accumulator stage and ring slot wraps many times."""
    _, epi, act, direct = next(e for e in EPIS if e[0] == name)
    for M, N, K in [(4096, 3456, 768), (383, 1152, 4352)]:
        r = _run_gemm(name, epi, act, direct, M, N, K, path, grid_div, seed=M + N + K + path + grid_div)
        assert r <= 1.0, f"{name} path {path} grid / {grid_div} M={M} N={N} K={K}: error / bound = {r:.3f}"
    print(f"gemm worst error / bound so far: {WORST['gemm']:.3f}")


def test_vit_gemm_rejects_bad_arguments():
    lib = _abi.lib()
    a = torch.zeros(128, 128, dtype=torch.bfloat16, device=DEV)
    o = torch.zeros(128, 128, dtype=torch.float32, device=DEV)
    for kw in (dict(K=100), dict(path=384), dict(epi=3), dict(grid_div=0), dict(epi=2, ld=160)):
        args = dict(M=128, N=128, K=128, epi=2, act=0, direct=0, ld=128, path=128, grid_div=1)
        args.update(kw)
        rc = lib.novic_debug_vit_gemm(a.data_ptr(), a.data_ptr(), args["M"], args["N"], args["K"], args["epi"], args["act"], args["direct"], None,
                                      o.data_ptr(), args["ld"], None, 0, 0, args["path"], args["grid_div"], _stream())
        assert rc != 0, kw


# ---------------------------------------------------------------------------------------------------------------------------------
# Attention
# ---------------------------------------------------------------------------------------------------------------------------------
HEADS = {64: 3, 72: 8, 80: 4}          # W = heads * D: a multiple of 64 (the V^T transpose works in 64-channel tiles)
TOKENS = [1, 2, 36, 64, 65, 127, 128, 129, 196, 256, 257, 730]
CASES = ["negative", "dominant", "rising", "foreign"]


def _attn_inputs(case: str, nimg: int, T: int, heads: int, D: int, seed: int, qdir=None):
    """q [nimg, heads, T, D], k, v as fp32 holding bf16 values; different data per image and head.  qdir [heads, D]: the query direction
    the dominant key is built for (default: the mean query of its image and head)."""
    g = torch.Generator().manual_seed(seed)
    shape = (nimg, heads, T, D)
    q = torch.randn(shape, generator=g) * 0.5
    k = torch.randn(shape, generator=g) * 0.5
    v = torch.randn(shape, generator=g) + torch.randn(nimg, heads, 1, D, generator=g)
    sd = math.sqrt(D)
    if case == "negative":          # every valid score ~ -30 (+- 0.5): a padded key's score of 0 would dominate
        q = 1.0 + 0.3 * torch.randn(shape, generator=g)
        k = -30.0 / sd + 0.5 * torch.randn(shape, generator=g)
    elif case == "dominant":        # one key per (image, head) ~8 above the rest, at 0, 127, 128 or T - 1
        q = torch.randn(nimg, heads, 1, D, generator=g) * 0.5 + 0.2 * torch.randn(shape, generator=g)
        pos = [p for p in (0, 127, 128, T - 1) if p < T]
        for i in range(nimg):
            for h in range(heads):
                j = pos[(i * heads + h) % len(pos)]
                qm = q[i, h].mean(0) if qdir is None else qdir[h]
                k[i, h, j] = qm * (8.0 * sd / qm.dot(qm).clamp_min(1e-3)) + 0.05 * torch.randn(D, generator=g)
                v[i, h, j] += 3.0
    elif case == "rising":          # score ~ -10 + 4 per 128 keys: the running maximum moves on every tile
        q = 1.0 + 0.1 * torch.randn(shape, generator=g)
        s = -10.0 + torch.arange(T, dtype=torch.float32) * (4.0 / 128) + 0.3 * torch.randn(nimg, heads, T, generator=g)
        k = (s * sd / q.sum(-1).mean(-1, keepdim=True)).unsqueeze(-1) + 0.05 * torch.randn(shape, generator=g)
    q, k, v = (t.to(torch.bfloat16).float() for t in (q, k, v))
    return q, k, v


def _pack_qkv(q, k, v, foreign: bool, gen) -> torch.Tensor:
    """[nimg * T, 3 W] rows q | k | v, head h at columns h * D"""
    nimg, heads, T, D = q.shape
    W = heads * D
    qkv = torch.cat([t.permute(0, 2, 1, 3).reshape(nimg, T, W) for t in (q, k, v)], dim=-1)
    if foreign:
        # channels 0..7 of every head but the first (q, k and v) and of K head 0 (what the last head's Q tile reads past its 72 channels)
        sign = lambda n: (torch.randint(0, 2, (nimg, T, n), generator=gen) * 2 - 1).float() * 64.0
        for part in range(3):
            for h in range(1, heads):
                c0 = part * W + h * D
                qkv[:, :, c0:c0 + 8] = sign(8)
        qkv[:, :, W:W + 8] = sign(8)
    return qkv.to(torch.bfloat16).reshape(nimg * T, 3 * W)


def _attn_ref(qkv: torch.Tensor, nimg: int, T: int, heads: int, D: int):
    W = heads * D
    x = qkv.to(F64).view(nimg, T, 3, heads, D).permute(2, 0, 3, 1, 4)            # [3, nimg, heads, T, D]
    s = x[0] @ x[1].transpose(-1, -2) / math.sqrt(D)
    o = torch.softmax(s, dim=-1) @ x[2]
    vmax = x[2].abs().amax(dim=(-1, -2), keepdim=True)                         # per (image, head)
    return o.permute(0, 2, 1, 3).reshape(nimg * T, W), vmax.expand(nimg, heads, T, D).permute(0, 2, 1, 3).reshape(nimg * T, W)


def _check_attn(got_buf, rows, W, ref, vmax, family, what, vtol):
    got = got_buf[PRE:PRE + rows * W].view(rows, W).to(F64)
    assert not torch.isnan(got).any(), f"{what}: owned elements left unwritten"
    assert torch.isnan(got_buf[:PRE].float()).all() and torch.isnan(got_buf[PRE + rows * W:].float()).all(), f"{what}: guard rows written"
    bound = vtol * vmax + 2.0 ** -8 * ref.abs()
    ratio = ((got - ref).abs() / bound).max().item()
    _note(family, ratio)
    assert ratio <= 1.0, f"{what}: error / bound = {ratio:.3f}"
    return ratio


ATTN_PARAMS = [(D, "tc", c) for D in (64, 72, 80) for c in (0, 1, 3)] + [(80, "mma", 0)]


@pytest.mark.parametrize("T", TOKENS)
@pytest.mark.parametrize("D,kernel,max_ctas", ATTN_PARAMS, ids=[f"d{D}_{k}_ctas{c}" for D, k, c in ATTN_PARAMS])
def test_vit_attention_against_fp64(D, kernel, max_ctas, T):
    heads, nimg = HEADS[D], 2
    W = heads * D
    rows = nimg * T
    lib = _abi.lib()
    worst = 0.0
    for ci, case in enumerate(CASES):
        if case == "foreign" and D != 72:
            continue
        gen = torch.Generator().manual_seed(31 * T + ci)
        q, k, v = _attn_inputs("dominant" if case == "foreign" else case, nimg, T, heads, D, seed=7 * T + 101 * ci + D)
        qkv = _pack_qkv(q, k, v, case == "foreign", gen).to(DEV)
        ref, vmax = _attn_ref(qkv, nimg, T, heads, D)
        buf = torch.full((PRE + (rows + 64) * W,), float("nan"), dtype=torch.bfloat16, device=DEV)
        _abi.check(lib.novic_debug_vit_attention(qkv.data_ptr(), nimg, T, W, heads, 0 if kernel == "tc" else 1, max_ctas, buf[PRE:].data_ptr(), _stream()))
        torch.cuda.synchronize()
        worst = max(worst, _check_attn(buf, rows, W, ref, vmax, f"attention_{kernel}", f"D={D} {kernel} ctas={max_ctas} T={T} {case}", 4e-3))
    print(f"attention D={D} {kernel} ctas={max_ctas} T={T}: worst error / bound {worst:.3f}")


def test_vit_attention_rejects_unsupported_heads():
    lib = _abi.lib()
    x = torch.zeros(3 * 128 * 2, dtype=torch.bfloat16, device=DEV)
    assert lib.novic_debug_vit_attention(x.data_ptr(), 1, 2, 128, 1, 0, 0, x.data_ptr(), _stream()) != 0        # D = 128
    assert lib.novic_debug_vit_attention(x.data_ptr(), 1, 2, 128, 2, 1, 0, x.data_ptr(), _stream()) != 0        # mma.sync at D = 64


MAP_TOKENS = [1, 36, 196, 256, 3072]


@pytest.mark.parametrize("T", MAP_TOKENS)
@pytest.mark.parametrize("D", [64, 72])
def test_siglip_map_attention_against_fp64(D, T):
    heads, nimg = (12 if D == 64 else 16), 3
    W = heads * D
    lib = _abi.lib()
    worst = 0.0
    for ci, case in enumerate(["negative", "dominant"]):
        qdir = (torch.randn(heads, D, generator=torch.Generator().manual_seed(T + D)) * 0.5).to(torch.bfloat16).float()
        q, k, v = _attn_inputs(case, nimg, T, heads, D, seed=13 * T + ci + D, qdir=qdir)
        qv = (qdir if case == "dominant" else q[0, :, 0, :]).reshape(W).to(DEV)  # the one latent query: fp32 [W]
        kv = torch.cat([t.permute(0, 2, 1, 3).reshape(nimg, T, W) for t in (k, v)], dim=-1).to(torch.bfloat16).reshape(nimg * T, 2 * W).to(DEV)
        x = kv.to(F64).view(nimg, T, 2, heads, D).permute(2, 0, 3, 1, 4)        # [2, nimg, heads, T, D]
        s = torch.einsum("hd,ihtd->iht", qv.to(F64).view(heads, D), x[0]) / math.sqrt(D)
        ref = torch.einsum("iht,ihtd->ihd", torch.softmax(s, dim=-1), x[1]).reshape(nimg, W)
        vmax = x[1].abs().amax(dim=(-1, -2)).repeat_interleave(D, dim=-1)
        buf = torch.full((PRE + (nimg + 4) * W,), float("nan"), dtype=torch.bfloat16, device=DEV)
        _abi.check(lib.novic_debug_siglip_map_attention(kv.data_ptr(), qv.data_ptr(), nimg, T, W, heads, buf[PRE:].data_ptr(), _stream()))
        torch.cuda.synchronize()
        worst = max(worst, _check_attn(buf, nimg, W, ref, vmax, "map_attention", f"MAP D={D} T={T} {case}", 1e-3))
    print(f"MAP attention D={D} T={T}: worst error / bound {worst:.3f}")


# ---------------------------------------------------------------------------------------------------------------------------------
# LayerNorm
# ---------------------------------------------------------------------------------------------------------------------------------
def _ln64(x, w, b, eps):
    m = x.mean(-1, keepdim=True)
    var = ((x - m) ** 2).mean(-1, keepdim=True)
    return (x - m) / torch.sqrt(var + eps) * w + b


@pytest.mark.parametrize("variant", ["plain", "ln_pre", "ln_post_stride"])
@pytest.mark.parametrize("W", [640, 768, 1024, 1152, 1280])
def test_vit_layernorm_against_fp64(W, variant):
    """plain: a block's norm -> bf16; ln_pre: class-token seat + in place + chained second norm (ViT-H's ln_pre + ln_1);
    ln_post_stride: every T-th row (in_stride = T * W) -> bf16, x untouched."""
    g = torch.Generator().manual_seed(W)
    T, nimg, eps = 37, 3, 1e-5
    n = nimg * T
    x0 = torch.randn(n, W, generator=g)
    x0[::2] = 1e3 + 0.1 * torch.randn(n - n // 2, W, generator=g)        # mean 1e3, std 0.1
    w1, b1, w2, b2 = (1 + 0.2 * torch.randn(W, generator=g)), 0.1 * torch.randn(W, generator=g), (1 + 0.2 * torch.randn(W, generator=g)), 0.1 * torch.randn(W, generator=g)
    cls = 1e3 + 0.1 * torch.randn(W, generator=g)
    pos0 = 0.05 * torch.randn(W, generator=g)
    w1, b1, w2, b2, cls, pos0 = (t.to(DEV) for t in (w1, b1, w2, b2, cls, pos0))
    xbuf = torch.full(((n + 4) * W,), float("nan"), device=DEV)
    xbuf[:n * W] = x0.to(DEV).view(-1)
    x = xbuf[:n * W].view(n, W)
    rows = nimg if variant == "ln_post_stride" else n
    obuf = torch.full((PRE + (rows + 4) * W,), float("nan"), dtype=torch.bfloat16, device=DEV)
    before = xbuf.clone()
    lib = _abi.lib()
    fp = lambda t: t.data_ptr()
    if variant == "plain":
        rc = lib.novic_debug_vit_layernorm(fp(x), W, fp(w1), fp(b1), None, None, 0, obuf[PRE:].data_ptr(), rows, W, eps, None, None, 0, _stream())
    elif variant == "ln_pre":
        rc = lib.novic_debug_vit_layernorm(fp(x), W, fp(w1), fp(b1), fp(w2), fp(b2), 1, obuf[PRE:].data_ptr(), rows, W, eps, fp(cls), fp(pos0), T, _stream())
    else:
        rc = lib.novic_debug_vit_layernorm(fp(x), T * W, fp(w1), fp(b1), None, None, 0, obuf[PRE:].data_ptr(), rows, W, eps, None, None, 0, _stream())
    _abi.check(rc)
    torch.cuda.synchronize()
    xin = x0.to(DEV).to(F64)
    if variant == "ln_pre":
        xin[::T] = (cls + pos0).to(F64)          # the kernel adds the two in fp32
    if variant == "ln_post_stride":
        xin = xin[::T]
    y = _ln64(xin, w1.to(F64), b1.to(F64), eps)
    out_ref = _ln64(y, w2.to(F64), b2.to(F64), eps) if variant == "ln_pre" else y
    # bf16 output: one rounding (2^-9 relative) after an fp32 pass whose mean carries ~1e-4 of error on the 1e3 rows (<= 2e-3 after / std)
    got = obuf[PRE:PRE + rows * W].view(rows, W).to(F64)
    assert not torch.isnan(got).any(), "owned elements left unwritten"
    assert torch.isnan(obuf[:PRE].float()).all() and torch.isnan(obuf[PRE + rows * W:].float()).all(), "guard rows of the output written"
    gain = (w2 if variant == "ln_pre" else w1).abs().to(F64)
    ratio = ((got - out_ref).abs() / (2.0 ** -8 * out_ref.abs() + 3e-3 * (gain + 0.1))).max().item()
    if variant == "ln_pre":                    # x <- y in place (fp32)
        xr = x.to(F64)
        ratio = max(ratio, ((xr - y).abs() / (1e-5 * y.abs() + 3e-3 * (w1.abs().to(F64) + 0.1))).max().item())
        assert torch.equal(xbuf[n * W:].view(torch.int32), before[n * W:].view(torch.int32)), "guard rows of x written"
    else:
        assert torch.equal(xbuf.view(torch.int32), before.view(torch.int32)), "x changed without store_x"
    _note("layernorm", ratio)
    print(f"layernorm W={W} {variant}: error / bound {ratio:.3f}")
    assert ratio <= 1.0


def test_worst_errors_per_family():
    """Runs last in this module: prints each family's worst error as a fraction of its bound."""
    for fam, r in sorted(WORST.items()):
        print(f"worst error / bound, {fam}: {r:.3f}")
