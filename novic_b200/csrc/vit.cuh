// CLIP ViT image encoder in front of the decoder (SURVEY.md section 8 row f3; call site embedders.py:759-764: encode_image(normalize=False)
// followed by an fp32 normalise).  BASELINE config #5 names DFN5B-CLIP-ViT-H-14-378; its definition lives in the un-vendored
// open_clip_torch (requirements.txt:8), so the architecture is an ASSUMPTION stated in DESIGN.md: open_clip's VisionTransformer,
// patch 14 on 378 x 378 (27 x 27 patches + class token = 730 tokens), width 1280, 32 pre-LN blocks of 16 heads x 80 with a 5120-wide
// QuickGELU MLP, biases on every linear, LayerNorm (weight + bias, eps 1e-5) before the blocks and on the class token after them,
// bias-free 1280 -> 1024 projection.  Parity is pinned only on an independent torch restatement (oracle/vit_oracle.py).
//
// The same kernels also run the reference's DEFAULT embedder, open_clip `ViT-B-16-SigLIP` (config/train.yaml:126), whose definition is
// equally un-vendored, so its architecture is an ASSUMPTION too (open_clip's TimmModel around timm `vit_base_patch16_siglip_224`,
// timm_pool 'map', timm_proj 'none', as remembered): a 16 x 16 patch convolution WITH bias on 224 x 224 images (14 x 14 = 196 tokens, no
// class token) plus a learned pos_embed, no ln_pre; 12 pre-LN blocks of width 768 (qkv [2304, 768] + bias laid out q; k; v, 12 heads of 64,
// scale 1/8, no mask; MLP 768 -> 3072 -> 768 with biases and the exact erf GELU of timm's nn.GELU - big_vision's original uses the tanh
// approximation); LayerNorm with weight + bias, eps 1e-6; the final `norm` on all tokens; then the MAP head (timm AttentionPoolLatent):
// q = q_proj(latent) (image independent), k, v = kv(x) ([1536, 768] + bias, k first), o = softmax(q k^T / 8) v per head (one query over
// the 196 keys), y = proj(o), y += fc2(GELU(fc1(norm(y)))); the output is y (768), no projection after it.  Parameter names follow
// open_clip (`visual.trunk.*`); parity is pinned only on tests/siglip_oracle.py:encode_image_siglip.
//
// open_clip `ViT-SO400M-14-SigLIP` (the image embedder of the F = 1152 checkpoints) is assumed to be the same architecture at other
// dimensions (TimmModel around timm `vit_so400m_patch14_siglip_224`, timm_pool 'map', timm_proj 'none', equally un-vendored): a 14 x 14
// patch convolution with bias on 224 x 224 images (16 x 16 = 256 tokens, no class token), 27 blocks of width 1152 with 16 heads of 72
// (scale 1/sqrt(72)), MLP 1152 -> 4304 -> 1152 with the exact erf GELU in the blocks and in the MAP head, LayerNorm eps 1e-6, the final
// norm on all tokens, the MAP head, output 1152 wide, the same `visual.trunk.*` names.  The GEMMs read K in 64-channel k-blocks, so the
// 4304-wide MLP runs padded to 4352 (zero fc1 rows and bias, zero fc2 columns: GELU(0) = 0 keeps the padded hidden columns exact zeros).
//
// The dense contractions (patch embedding, QKV, out-proj, both MLP layers: 99 % of the FLOPs outside attention) run on the persistent
// tcgen05 / TMEM / TMA GEMM of gemm.cuh through the epilogues below; attention (730 keys x 80 channels per head) runs on
// mma.sync.m16n8k16 tiles with an online softmax (flash-style: scores never leave the registers).
#pragma once

#include "gemm.cuh"
#include "train.cuh"   // ldsm_x4 / ldsm_x4_t / mma_bf16_16816

namespace novic {

constexpr int kVitHeadDim = 80;       // open_clip ViT-H/14 heads (the legacy mma.sync attention is built for this one)
constexpr int kSiglipHeadDim = 64;    // SigLIP ViT-B/16 heads
constexpr int kSo400mHeadDim = 72;    // SigLIP SO400M/14 heads

// activation of EpiVitBias
constexpr int kVitActNone = 0, kVitActQuickGelu = 1, kVitActGelu = 2;

// ---------------------------------------------------------------------------------------------------------
// GEMM epilogues (persistent gemm_kernel: 8 epilogue warps, thread = output row, 64 columns per thread)
// ---------------------------------------------------------------------------------------------------------

// out[row, n] = act(acc + bias[n]) as bf16 (QKV: no activation; MLP c_fc: QuickGELU x * sigmoid(1.702 x) for open_clip's ViT-H,
// the erf GELU for SigLIP)
struct EpiVitBias {
  struct Params {
    __nv_bfloat16* out;
    int ld;                 // elements per output row
    const float* bias;      // [N] or nullptr
    int n_valid;            // N (columns >= N of the last tile are not stored)
    int act;                // kVitActNone / kVitActQuickGelu / kVitActGelu
    int direct;             // != 0: rows stored straight from the registers with 256-bit stores (ld must be a multiple of 16 elements)
  };
  template <class Release>
  __device__ static __forceinline__ void run(const Params& p, const EpiCtx& c, Release release) {
    const int lane = lane_id();
    const int nhalf = c.ncols / kEpiCols;              // 1 (128-column tiles) or 2 (256-column tiles): 64 columns are staged at a time
#pragma unroll 1
    for (int hf = 0; hf < nhalf; ++hf) {
      const int n0 = c.n0 + hf * kEpiCols;
#pragma unroll
      for (int ch = 0; ch < kEpiCols / 32; ++ch) {
        float v[32];
        tmem_ld_32x32(c.tmem_row + hf * kEpiCols + ch * 32, v);
        if (hf == nhalf - 1 && ch == kEpiCols / 32 - 1) release();
        const int col0 = n0 + ch * 32;
        if (p.bias != nullptr && col0 < p.n_valid) {
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + col0) + q);   // N is a multiple of 32 for every ViT GEMM
            v[q * 4] += b.x; v[q * 4 + 1] += b.y; v[q * 4 + 2] += b.z; v[q * 4 + 3] += b.w;
          }
        }
        if (p.act == kVitActQuickGelu) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = v[j] * __fdividef(1.0f, 1.0f + __expf(-1.702f * v[j]));
        } else if (p.act == kVitActGelu) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = gelu_fast(v[j]);
        }
        if (p.direct) {
          // thread = row: 32 columns are 64 contiguous bytes of the row = two full 32-byte sectors (st.global.v8.b32); no staging tile
          if (c.row < c.M && col0 < p.n_valid) {
            __nv_bfloat16* dst = p.out + static_cast<size_t>(c.row) * p.ld + col0;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              uint32_t w[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) w[i] = pack_bf16x2(v[h * 16 + 2 * i], v[h * 16 + 2 * i + 1]);
              asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};\n" ::"l"(dst + h * 16), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]),
                           "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7])
                           : "memory");
            }
          }
        } else {
          stage_put32(c.stage, lane, ch * 32, v);
        }
      }
      if (p.direct) continue;
      if (n0 < p.n_valid)
        stage_copy_out(c.stage, lane, [&](int r) -> __nv_bfloat16* {
          const int row = c.warp_row0 + r;
          return row < c.M ? p.out + static_cast<size_t>(row) * p.ld + n0 : nullptr;
        });
      else __syncwarp();
    }
  }
};

// Residual / patch-embedding epilogue on the fp32 token stream x [images * T, W] (row-major):
//   residual mode (table == nullptr):  x[row, n] += acc + bias[n]                                  (attention out-proj, MLP c_proj)
//   patch mode    (table != nullptr):  x[img * T + tok0 + p, n] = acc + table[(tok0 + p) * W + n] + bias[n]
//                                      (conv1 as a GEMM over patches + positions; GEMM row = img * (T - tok0) + p; tok0 = 1 behind a
//                                      class token, 0 without one)
// The thread = row accumulator chunk goes through a warp-private XOR-swizzled fp32 tile so that every global access covers 4 rows x 128
// contiguous bytes.
struct EpiVitResid {
  struct Params {
    float* x;
    int ld;                 // W
    const float* bias;      // [W] or nullptr
    const float* table;     // patch mode: positional embedding [T, W]
    int patches;            // patch mode: T - tok0
    int n_valid;            // W (columns >= W of a ragged last tile are not touched)
    int tok0;               // patch mode: token index of the first patch (1 with a class token, 0 without)
  };
  template <class Release>
  __device__ static __forceinline__ void run(const Params& p, const EpiCtx& c, Release release) {
    const int lane = lane_id();
    float* st = reinterpret_cast<float*>(c.stage);            // 32 rows x 32 fp32 = 4096 B (kEpiStageBytes)
    const int sub = lane >> 3, chunk = lane & 7;
    const int nch = c.ncols / 32;
#pragma unroll 1
    for (int ch = 0; ch < nch; ++ch) {
      const bool live = c.n0 + ch * 32 < p.n_valid;           // warp-uniform
      const int col = c.n0 + ch * 32 + chunk * 4;
      // the residual (or position) values of this chunk do not depend on the accumulator: all eight 16-byte loads of the thread are
      // issued first, so that their latency overlaps the TMEM load and the staging (with the loads behind the staging the epilogue
      // of a tile took ~6 k cycles and bound the out-proj GEMM, whose main loop needs 2.6 k)
      float4 base[8];
      float* dst[8];
      if (live) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int r = i * 4 + sub;
          const int row = c.warp_row0 + r;
          dst[i] = nullptr;
          base[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (row < c.M) {
            if (p.table != nullptr) {
              const int img = row / p.patches, pp = row - img * p.patches;
              dst[i] = p.x + (static_cast<size_t>(img) * (p.patches + p.tok0) + p.tok0 + pp) * p.ld + col;
              base[i] = __ldg(reinterpret_cast<const float4*>(p.table + static_cast<size_t>(p.tok0 + pp) * p.ld + col));
            } else {
              dst[i] = p.x + static_cast<size_t>(row) * p.ld + col;
              base[i] = *reinterpret_cast<const float4*>(dst[i]);
            }
          }
        }
      }
      float v[32];
      tmem_ld_32x32(c.tmem_row + ch * 32, v);
      if (ch == nch - 1) release();
      if (!live) continue;
      __syncwarp();
#pragma unroll
      for (int q = 0; q < 8; ++q)
        *reinterpret_cast<float4*>(st + lane * 32 + ((q ^ (lane & 7)) << 2)) = make_float4(v[q * 4], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
      __syncwarp();
      float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
      if (p.bias != nullptr) b = __ldg(reinterpret_cast<const float4*>(p.bias + col));
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = i * 4 + sub;
        if (dst[i] == nullptr) continue;
        const float4 a = *reinterpret_cast<const float4*>(st + r * 32 + ((chunk ^ (r & 7)) << 2));
        *reinterpret_cast<float4*>(dst[i]) = make_float4(base[i].x + a.x + b.x, base[i].y + a.y + b.y, base[i].z + a.z + b.z, base[i].w + a.w + b.w);
      }
    }
  }
};

// out[row, n] = acc (+ bias[n]) (fp32, row-major): ViT-H's final 1280 -> 1024 projection of the class-token rows, SigLIP's MAP-head
// `proj` (B rows only)
struct EpiVitStoreF32 {
  struct Params {
    float* out;
    int ld;
    const float* bias;      // [ld] or nullptr
  };
  template <class Release>
  __device__ static __forceinline__ void run(const Params& p, const EpiCtx& c, Release release) {
    const int nch = c.ncols / 32;
#pragma unroll 1
    for (int ch = 0; ch < nch; ++ch) {
      float v[32];
      tmem_ld_32x32(c.tmem_row + ch * 32, v);
      if (ch == nch - 1) release();
      const int col0 = c.n0 + ch * 32;
      if (c.row < c.M && col0 < p.ld) {
        if (p.bias != nullptr) {
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + col0) + q);
            v[q * 4] += b.x; v[q * 4 + 1] += b.y; v[q * 4 + 2] += b.z; v[q * 4 + 3] += b.w;
          }
        }
        float4* d = reinterpret_cast<float4*>(p.out + static_cast<size_t>(c.row) * p.ld + col0);
#pragma unroll
        for (int q = 0; q < 8; ++q) d[q] = make_float4(v[q * 4], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
      }
    }
  }
};

// ---------------------------------------------------------------------------------------------------------
// Patches: images [B, 3, S, S] fp32 -> bf16 rows [B * np * np, Kp] with k = (c * 14 + py) * 14 + px (the order of conv1.weight flattened),
// zero-padded from 588 to Kp = 640 columns (a whole number of 64-wide k-blocks).  One warp per patch row.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) vit_patchify_kernel(const float* __restrict__ img, __nv_bfloat16* __restrict__ out, int B, int S, int P, int np, int Kp) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int total = B * np * np;
  if (warp >= total) return;
  const int b = warp / (np * np), pidx = warp - b * np * np, py0 = (pidx / np) * P, px0 = (pidx % np) * P;
  const int K = 3 * P * P;
  __nv_bfloat16* dst = out + static_cast<size_t>(warp) * Kp;
  for (int k = lane; k < Kp; k += 32) {
    float v = 0.f;
    if (k < K) {
      const int ch = k / (P * P), rem = k - ch * P * P, py = rem / P, px = rem - py * P;
      v = __ldg(img + ((static_cast<size_t>(b) * 3 + ch) * S + py0 + py) * S + px0 + px);
    }
    dst[k] = __float2bfloat16_rn(v);
  }
}

// ---------------------------------------------------------------------------------------------------------
// LayerNorm over rows of the fp32 token stream (weight + bias, biased variance).  One warp per row, the row in registers.
//   y = LN(x; w1, b1);  optional: x <- y (fp32, in place);  out_bf <- y (bf16), or out_bf <- LN(y; w2, b2) when w2 != nullptr
// (ln_pre followed by the first block's ln_1 is one pass), or out_f32 <- y for the class-token rows (ln_post: row stride `in_stride`).
// NV = W / 128 float4 per lane (W = 1280: 10).
// ---------------------------------------------------------------------------------------------------------
struct VitLnParams {
  float* x;                     // [rows * in_stride] fp32
  long long in_stride;          // elements between consecutive rows (W, or T * W to pick the class tokens)
  const float *w1, *b1, *w2, *b2;
  int store_x;                  // write y back to x
  __nv_bfloat16* out_bf;        // [rows, W] or nullptr
  int rows, W;
  float eps;
  const float* cls;             // optional: row r of x is first SET to cls + pos0 when (r % cls_period) == 0 (class token rows)
  const float* pos0;
  int cls_period;
};

template <int NV>
__global__ void __launch_bounds__(256) vit_layernorm_kernel(const VitLnParams p) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (row >= p.rows) return;
  float4 v[NV];
  float* xr = p.x + static_cast<size_t>(row) * p.in_stride;
  const bool is_cls = p.cls != nullptr && (row % p.cls_period) == 0;
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    const int c4 = lane + 32 * j;
    if (is_cls) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(p.cls) + c4), b = __ldg(reinterpret_cast<const float4*>(p.pos0) + c4);
      v[j] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
    } else {
      v[j] = *reinterpret_cast<const float4*>(xr + c4 * 4);
    }
  }
  auto normalise = [&](const float* w, const float* b) {
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j) s += v[j].x + v[j].y + v[j].z + v[j].w;
    s = warp_sum(s);
    const float mean = s / static_cast<float>(p.W);
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const float dx = v[j].x - mean, dy = v[j].y - mean, dz = v[j].z - mean, dw = v[j].w - mean;
      q += dx * dx + dy * dy + dz * dz + dw * dw;
    }
    q = warp_sum(q);
    const float rstd = rsqrtf(q / static_cast<float>(p.W) + p.eps);
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const int c4 = lane + 32 * j;
      const float4 g = __ldg(reinterpret_cast<const float4*>(w) + c4), bb = __ldg(reinterpret_cast<const float4*>(b) + c4);
      v[j] = make_float4((v[j].x - mean) * rstd * g.x + bb.x, (v[j].y - mean) * rstd * g.y + bb.y, (v[j].z - mean) * rstd * g.z + bb.z,
                         (v[j].w - mean) * rstd * g.w + bb.w);
    }
  };
  normalise(p.w1, p.b1);
  if (p.store_x) {
#pragma unroll
    for (int j = 0; j < NV; ++j) *reinterpret_cast<float4*>(xr + (lane + 32 * j) * 4) = v[j];
  }
  if (p.out_bf != nullptr) {
    if (p.w2 != nullptr) normalise(p.w2, p.b2);
    __nv_bfloat16* o = p.out_bf + static_cast<size_t>(row) * p.W;
#pragma unroll
    for (int j = 0; j < NV; ++j)
      *reinterpret_cast<uint2*>(o + (lane + 32 * j) * 4) = make_uint2(pack_bf16x2(v[j].x, v[j].y), pack_bf16x2(v[j].z, v[j].w));
  }
}

// ---------------------------------------------------------------------------------------------------------
// Attention of one ViT block: softmax(Q K^T / sqrt(80)) V over all T tokens of an image, no mask (flash-style).
// qkv: bf16 [images * T, 3 * W] row-major (q | k | v, head h at columns h * 80); out: bf16 [images * T, W].
// One CTA = 128 queries (8 warps x 16) of one (image, head); keys in tiles of 64 through a double-buffered cp.async ring;
// Q K^T and P V on mma.sync m16n8k16 from ldmatrix fragments, probabilities go from the score accumulators straight into the A fragments.
// ---------------------------------------------------------------------------------------------------------
constexpr int kVaQ = 128, kVaK = 64, kVaWarps = 8;
constexpr int kVaPitch = kVitHeadDim + 8;                         // 88 bf16 = 176 B rows: ldmatrix rows fall into distinct bank groups
constexpr int kVaStages = 3;                                      // K/V ring: one CTA barrier per key tile
constexpr int kVaSmemBytes = (kVaQ + 2 * kVaStages * kVaK) * kVaPitch * 2;    // Q + 3 x (K, V) = 90 112 B (two CTAs per SM)

struct VitAttnParams {
  const __nv_bfloat16* qkv;
  __nv_bfloat16* out;
  int T, W, heads;
  float scale_log2e;           // log2(e) / sqrt(80)
};

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, bool valid) {
  const uint32_t d = smem_u32(smem_dst);
  const int n = valid ? 16 : 0;       // src-size 0: the 16 bytes are zero-filled (rows past the end of the sequence)
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(gsrc), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// 2^x on the SFU (MUFU.EX2; exp2f without fast-math expands to a dozen instructions of range handling, which made the softmax - not the
// tensor pipe - the busiest part of the kernel); relative error 2^-22, inputs here are <= 0
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__global__ void __launch_bounds__(kVaWarps * 32, 2) vit_attention_kernel(const VitAttnParams p) {
  extern __shared__ __align__(16) uint8_t sm_va[];
  __nv_bfloat16* sq = reinterpret_cast<__nv_bfloat16*>(sm_va);
  __nv_bfloat16* skv = sq + kVaQ * kVaPitch;                       // [kVaStages][K | V][64][pitch]
  const int warp = threadIdx.x >> 5, lane = lane_id();
  const int lm = lane >> 3, lr = lane & 7, g = lane >> 2, t = lane & 3;
  const int qt = blockIdx.x, head = blockIdx.y, img = blockIdx.z;
  const int T = p.T, ld = 3 * p.W;
  const __nv_bfloat16* base = p.qkv + static_cast<size_t>(img) * T * ld + head * kVitHeadDim;
  const int q0 = qt * kVaQ;
  constexpr int kChunks = kVitHeadDim / 8;                         // 16-byte chunks per row: 10

  // Q tile (rows past T zero-filled), then K/V tile 0
  for (int i = threadIdx.x; i < kVaQ * kChunks; i += blockDim.x) {
    const int r = i / kChunks, c = i - r * kChunks;
    const bool ok = q0 + r < T;
    cp_async16(sq + r * kVaPitch + c * 8, base + static_cast<size_t>(ok ? q0 + r : 0) * ld + c * 8, ok);
  }
  auto load_kv = [&](int tile, int stage) {
    __nv_bfloat16* sk = skv + stage * 2 * kVaK * kVaPitch;
    __nv_bfloat16* sv = sk + kVaK * kVaPitch;
    const int k0 = tile * kVaK;
    for (int i = threadIdx.x; i < 2 * kVaK * kChunks; i += blockDim.x) {
      const int which = i / (kVaK * kChunks), j = i - which * kVaK * kChunks, r = j / kChunks, c = j - r * kChunks;
      const bool ok = k0 + r < T;
      cp_async16((which ? sv : sk) + r * kVaPitch + c * 8, base + static_cast<size_t>(ok ? k0 + r : 0) * ld + (1 + which) * p.W + c * 8, ok);
    }
  };
  const int ntiles = (T + kVaK - 1) / kVaK;
  load_kv(0, 0);
  cp_async_commit();
  if (ntiles > 1) load_kv(1, 1);
  cp_async_commit();

  float o[kVitHeadDim / 8][4];
#pragma unroll
  for (int ni = 0; ni < kVitHeadDim / 8; ++ni)
#pragma unroll
    for (int e = 0; e < 4; ++e) o[ni][e] = 0.f;
  float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};
  uint32_t aq[kVitHeadDim / 16][4];

  int stage = 0;
  for (int tile = 0; tile < ntiles; ++tile) {
    cp_async_wait<1>();                                            // everything but the newest group: this tile's (and Q's) bytes have landed
    __syncthreads();                                               // ... for every thread; and every warp is done with tile - 1, whose stage is refilled now
    {
      const int nxt = stage == 0 ? kVaStages - 1 : stage - 1;      // stage of tile - 1 = stage of tile + 2
      if (tile + 2 < ntiles) load_kv(tile + 2, nxt);
      cp_async_commit();
    }
    if (tile == 0) {
#pragma unroll
      for (int ki = 0; ki < kVitHeadDim / 16; ++ki) ldsm_x4(aq[ki], sq + (warp * 16 + (lm & 1) * 8 + lr) * kVaPitch + ki * 16 + (lm >> 1) * 8);
    }
    const __nv_bfloat16* sk = skv + stage * 2 * kVaK * kVaPitch;
    const __nv_bfloat16* sv = sk + kVaK * kVaPitch;
    float s[kVaK / 8][4];
#pragma unroll
    for (int ni = 0; ni < kVaK / 8; ++ni)
#pragma unroll
      for (int e = 0; e < 4; ++e) s[ni][e] = 0.f;
#pragma unroll
    for (int ki = 0; ki < kVitHeadDim / 16; ++ki) {
#pragma unroll
      for (int np = 0; np < kVaK / 16; ++np) {
        uint32_t bk[4];
        ldsm_x4(bk, sk + (np * 16 + (lm >> 1) * 8 + lr) * kVaPitch + ki * 16 + (lm & 1) * 8);
        mma_bf16_16816(s[np * 2], aq[ki], bk[0], bk[1]);
        mma_bf16_16816(s[np * 2 + 1], aq[ki], bk[2], bk[3]);
      }
    }
    // online softmax on this warp's 16 rows (thread: rows g and g + 8, columns ni * 8 + 2 t + {0, 1}); the 1 / sqrt(80) * log2(e) factor is
    // folded into the exponent: p = 2^(s * c - m * c) is one FFMA + one MUFU per score
    const int kbase = tile * kVaK;
    const bool ragged = kbase + kVaK > T;
    if (ragged) {
#pragma unroll
      for (int ni = 0; ni < kVaK / 8; ++ni)
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (kbase + ni * 8 + 2 * t + (e & 1) >= T) s[ni][e] = -INFINITY;
    }
    // both row halves at once, reductions as trees of independent partials (a 16-deep FMNMX / FADD chain per row costs more issue
    // latency than the tensor work of the tile hides at four warps per scheduler)
    float mx[2][4], sm[2][4];
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int q = 0; q < 4; ++q) mx[h][q] = fmaxf(fmaxf(s[2 * q][h * 2], s[2 * q][h * 2 + 1]), fmaxf(s[2 * q + 1][h * 2], s[2 * q + 1][h * 2 + 1]));
    float m_new[2], corr[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float m = fmaxf(fmaxf(mx[h][0], mx[h][1]), fmaxf(mx[h][2], mx[h][3]));
      m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 1));
      m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 2));
      m_new[h] = fmaxf(m_run[h], m * p.scale_log2e);               // finite: every tile holds at least one valid key (scale > 0)
      corr[h] = ex2_approx(m_run[h] - m_new[h]);
      m_run[h] = m_new[h];
    }
#pragma unroll
    for (int ni = 0; ni < kVaK / 8; ++ni)
#pragma unroll
      for (int e = 0; e < 4; ++e) s[ni][e] = ex2_approx(fmaf(s[ni][e], p.scale_log2e, -m_new[e >> 1]));
#pragma unroll
    for (int h = 0; h < 2; ++h) {
#pragma unroll
      for (int q = 0; q < 4; ++q) sm[h][q] = (s[2 * q][h * 2] + s[2 * q][h * 2 + 1]) + (s[2 * q + 1][h * 2] + s[2 * q + 1][h * 2 + 1]);
      float sum = (sm[h][0] + sm[h][1]) + (sm[h][2] + sm[h][3]);
      sum += __shfl_xor_sync(0xffffffffu, sum, 1);
      sum += __shfl_xor_sync(0xffffffffu, sum, 2);
      l_run[h] = l_run[h] * corr[h] + sum;
    }
#pragma unroll
    for (int ni = 0; ni < kVitHeadDim / 8; ++ni) { o[ni][0] *= corr[0]; o[ni][1] *= corr[0]; o[ni][2] *= corr[1]; o[ni][3] *= corr[1]; }
    // O += P V
#pragma unroll
    for (int ki = 0; ki < kVaK / 16; ++ki) {
      uint32_t ap[4];
      ap[0] = pack_bf16x2(s[2 * ki][0], s[2 * ki][1]);
      ap[1] = pack_bf16x2(s[2 * ki][2], s[2 * ki][3]);
      ap[2] = pack_bf16x2(s[2 * ki + 1][0], s[2 * ki + 1][1]);
      ap[3] = pack_bf16x2(s[2 * ki + 1][2], s[2 * ki + 1][3]);
#pragma unroll
      for (int np = 0; np < kVitHeadDim / 16; ++np) {
        uint32_t bv[4];
        ldsm_x4_t(bv, sv + (ki * 16 + (lm & 1) * 8 + lr) * kVaPitch + np * 16 + (lm >> 1) * 8);
        mma_bf16_16816(o[np * 2], ap, bv[0], bv[1]);
        mma_bf16_16816(o[np * 2 + 1], ap, bv[2], bv[3]);
      }
    }
    stage = stage + 1 == kVaStages ? 0 : stage + 1;
  }
  // normalise, stage through the Q tile (each warp reads and writes only its own 16 rows of it), store 16-byte chunks
  __nv_bfloat16* so = sq + warp * 16 * kVaPitch;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const float inv = 1.0f / l_run[h];
#pragma unroll
    for (int ni = 0; ni < kVitHeadDim / 8; ++ni)
      *reinterpret_cast<uint32_t*>(so + (h * 8 + g) * kVaPitch + ni * 8 + 2 * t) = pack_bf16x2(o[ni][h * 2] * inv, o[ni][h * 2 + 1] * inv);
  }
  __syncwarp();
  __nv_bfloat16* dst = p.out + static_cast<size_t>(img) * T * p.W + head * kVitHeadDim;
  for (int i = lane; i < 16 * kChunks; i += 32) {
    const int r = i / kChunks, c = i - r * kChunks;
    const int row = q0 + warp * 16 + r;
    if (row < T) *reinterpret_cast<uint4*>(dst + static_cast<size_t>(row) * p.W + c * 8) = *reinterpret_cast<const uint4*>(so + r * kVaPitch + c * 8);
  }
}

// ---------------------------------------------------------------------------------------------------------
// The same attention on the 5th-generation tensor cores (default; the mma.sync kernel above is NOVIC_VIT_ATTN=mma).
// One CTA = 128 queries of one (image, head), keys in tiles of 128:
//   S = Q K^T   tcgen05.mma M = 128, N = 128, five k-slices of 16 channels (the 80-wide head = one 64-channel k-block + the first slice of
//               the next; both operands K-major with the 128-byte swizzle straight from TMA boxes of the qkv rows) -> TMEM, two S buffers
//   softmax     eight warps, thread = query row x 64 keys: the scores leave TMEM once (two loads in flight), 2^(s c - m c) with the scale folded in, bf16
//               probabilities written as the K-major swizzled A operand of the second product, the O accumulator (TMEM) rescaled in
//               place when the running maximum moved
//   O += P V    tcgen05.mma M = 128, N = 80, eight k-slices over the tile's 128 keys; B = V^T rows [channel][key] (K-major), produced once
//               per block by vit_vt_kernel from the v columns of qkv
// Persistent CTAs (one per SM) walk the (image, head, query tile) items.  Warp 0 = TMA producer (three-stage K / V^T ring, running ahead
// into the next item), warp 1 = TMEM allocator + MMA issuer (Q K^T of tile t + 1 is issued before P V of tile t,
// so the tensor core computes the next scores while the softmax warps work), warps 2..9 = softmax / correction / epilogue (two warps per
// scheduler: with one, every dependent instruction of the exponential chain waits out its own latency - 473 us against ... for this kernel).
// ---------------------------------------------------------------------------------------------------------
//
// The kernel is a template on the head dimension D: D = 80 (ViT-H) as above; D = 64 (SigLIP B/16) takes Q and K as one 64-channel k-block
// each, S in four k-slices, Vᵀ tiles of 64 rows, O with N = 64, and the four 16-column O chunks split 2 / 2 between the two softmax halves.
// D = 72 (SigLIP SO400M) stores 72 channels per head but computes at the MMA width 80 (N = 72 is not a UMMA shape for M = 128): Q K^T
// reads one 64-channel k-block and one 16-channel slice whose channels 72..79 belong to the next head (or, for the last head's Q, to K) -
// they are zeroed in the Q tile once per item, so they add exact zeros; Vᵀ tiles have 80 rows (rows 72..79: the next head's channels or
// TMA zero-fill), and O columns 72..79 are computed but never stored.
__host__ __device__ constexpr int ta_mma_width(int d) { return (d + 15) / 16 * 16; }
constexpr int kTaQ = 128, kTaK = 128;
constexpr int kTaStages = 3;                              // K / V^T ring: a tile's load (~2 k cycles) overlaps two tiles of work
template <int D> constexpr int kTaQBytes = ((D + 63) / 64) * kABytes;   // Q: 128 rows x 128 B per 64-channel k-block (D = 80, 72: two)
template <int D> constexpr int kTaKBytes = kTaQBytes<D>;                // K tile: the same
template <int D> constexpr int kTaVBytes = 2 * ta_mma_width(D) * 128;   // V^T tile: two k-blocks (64 keys each) of MMA-width rows x 128 B
constexpr int kTaPBytes = 2 * kABytes;                    // P: 128 rows x 128 keys bf16
template <int D>
constexpr int kTaSmemBytes = kTaQBytes<D> + kTaStages * (kTaKBytes<D> + kTaVBytes<D>) + kTaPBytes + 1024 /*align*/ + 256 /*barriers*/ + 3 * 2 * 128 * 4 /*row exchange*/;   // D = 80: 224.3 KB
constexpr int kTaSoftWarps = 8;                            // two per TMEM lane quadrant: each thread owns one query row x 64 of the tile's 128 keys
constexpr int kTaThreads = 64 + 32 * kTaSoftWarps;

struct VitAttnTcParams {
  __nv_bfloat16* out;          // [images * T, W]
  int T, W, heads, nimg;
  float scale_log2e;
};

// V^T per image: vt[img][c][t] = qkv[img * T + t][2 W + c] (t < T; columns T .. Tpad - 1 stay zero).  64 x 64 tiles through shared memory.
__global__ void __launch_bounds__(256) vit_vt_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ vt, int T, int W, int Tpad) {
  __shared__ __nv_bfloat16 tile[64][64 + 2];
  const int t0 = blockIdx.x * 64, c0 = blockIdx.y * 64, img = blockIdx.z;
  const __nv_bfloat16* src = qkv + static_cast<size_t>(img) * T * 3 * W + 2 * W + c0;
  for (int i = threadIdx.x; i < 64 * 32; i += 256) {      // 64 tokens x 32 channel pairs
    const int r = i >> 5, cp = i & 31;
    __nv_bfloat162 v = __floats2bfloat162_rn(0.f, 0.f);
    if (t0 + r < T) v = *reinterpret_cast<const __nv_bfloat162*>(src + static_cast<size_t>(t0 + r) * 3 * W + cp * 2);
    tile[r][cp * 2] = v.x;
    tile[r][cp * 2 + 1] = v.y;
  }
  __syncthreads();
  __nv_bfloat16* dst = vt + (static_cast<size_t>(img) * W + c0) * Tpad + t0;
  for (int i = threadIdx.x; i < 64 * 32; i += 256) {      // 64 channels x 32 token pairs
    const int c = i >> 5, tp = i & 31;
    *reinterpret_cast<__nv_bfloat162*>(dst + static_cast<size_t>(c) * Tpad + tp * 2) = __halves2bfloat162(tile[tp * 2][c], tile[tp * 2 + 1][c]);
  }
}

template <int D>
__global__ void __launch_bounds__(kTaThreads, 1)
vit_attention_tc_kernel(const __grid_constant__ CUtensorMap tm_qkv, const __grid_constant__ CUtensorMap tm_vt, const VitAttnTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  constexpr int kQBytes = kTaQBytes<D>, kKBytes = kTaKBytes<D>, kVBytes = kTaVBytes<D>;
  constexpr int DM = ta_mma_width(D);                      // MMA width: D = 72 computes as 80
  uint8_t* sK = sQ + kQBytes;                              // [kTaStages]
  uint8_t* sV = sK + kTaStages * kKBytes;                  // [kTaStages]
  uint8_t* sP = sV + kTaStages * kVBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + kTaPBytes);
  uint64_t* q_full = bars;                                 // 1
  uint64_t* q_empty = bars + 1;                            // 1: every Q K^T of the item has been executed
  uint64_t* kv_full = bars + 2;                            // kTaStages
  uint64_t* kv_empty = bars + 2 + kTaStages;               // kTaStages
  uint64_t* s_full = bars + 2 + 2 * kTaStages;             // 2
  uint64_t* s_empty = s_full + 2;                          // 2
  uint64_t* p_full = s_full + 4;                           // 1
  uint64_t* p_empty = s_full + 5;                          // 1
  uint64_t* o_full = s_full + 6;                           // 1
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_full + 7);
  float* xch = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 256);   // [3][2 halves][128 rows]: row maxima (two tile parities), row sums

  const int warp = threadIdx.x >> 5, lane = static_cast<int>(lane_id());
  const int T = p.T, W = p.W;
  const int ntiles = (T + kTaK - 1) / kTaK;                // key tiles per item
  const int qtiles = (T + kTaQ - 1) / kTaQ;
  const int nitems = qtiles * p.heads * p.nimg;            // item = (image, head, query tile), query tile fastest: neighbours share K / V in L2

  if (warp == 0) {
    if (elect_one()) {
      tma_prefetch_desc(&tm_qkv);
      tma_prefetch_desc(&tm_vt);
      mbar_init(q_full, 1); mbar_init(q_empty, 1);
      for (int i = 0; i < kTaStages; ++i) { mbar_init(&kv_full[i], 1); mbar_init(&kv_empty[i], 1); }
      for (int i = 0; i < 2; ++i) { mbar_init(&s_full[i], 1); mbar_init(&s_empty[i], kTaSoftWarps); }
      mbar_init(p_full, kTaSoftWarps); mbar_init(p_empty, 1); mbar_init(o_full, 1);
      fence_mbar_init();
    }
  } else if (warp == 1) {
    tmem_alloc<512>(tmem_slot);
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  constexpr uint32_t kColS = 0, kColO = 256;

  // Persistent: CTA b walks items b, b + grid, ...; `it` counts this CTA's items, `g` its key tiles over all items (ring / buffer phases).
  if (warp == 0) {
    if (elect_one()) {
      int g = 0, it = 0;
      for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++it) {
        const int qt = item % qtiles, head = (item / qtiles) % p.heads, img = item / (qtiles * p.heads);
        // Q: channels [head * D, +64 per k-block) of the image's token rows (rows >= T are out of bounds: zero)
        mbar_wait(q_empty, (it & 1) ^ 1, 1);
        mbar_arrive_expect_tx(q_full, kQBytes);
        tma_load_3d_at(sQ, &tm_qkv, q_full, head * D, qt * kTaQ, img, kEvictNormal);
        if (D > 64) tma_load_3d_at(sQ + kABytes, &tm_qkv, q_full, head * D + 64, qt * kTaQ, img, kEvictNormal);
        for (int t = 0; t < ntiles; ++t, ++g) {
          const int st = g % kTaStages;
          mbar_wait(&kv_empty[st], ((g / kTaStages) & 1) ^ 1, 1);
          mbar_arrive_expect_tx(&kv_full[st], kKBytes + kVBytes);
          uint8_t* k = sK + st * kKBytes;
          uint8_t* v = sV + st * kVBytes;
          tma_load_3d_at(k, &tm_qkv, &kv_full[st], W + head * D, t * kTaK, img, kEvictLast);
          if (D > 64) tma_load_3d_at(k + kABytes, &tm_qkv, &kv_full[st], W + head * D + 64, t * kTaK, img, kEvictLast);
          tma_load_3d_at(v, &tm_vt, &kv_full[st], t * kTaK, head * D, img, kEvictLast);
          tma_load_3d_at(v + DM * 128, &tm_vt, &kv_full[st], t * kTaK + 64, head * D, img, kEvictLast);
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t kIdescS = umma_idesc_bf16_f32(kTaQ, kTaK);
      constexpr uint32_t kIdescO = umma_idesc_bf16_f32(kTaQ, DM);
      // Q K^T of global tile gq (scores buffer gq & 1)
      auto issue_qk = [&](int gq) {
        const int st = gq % kTaStages, sb = gq & 1;
        mbar_wait(&kv_full[st], (gq / kTaStages) & 1, 2);
        mbar_wait(&s_empty[sb], ((gq >> 1) & 1) ^ 1, 3);           // the softmax warps have read the previous scores of this buffer
        tc_fence_after_sync();
        const uint32_t a = smem_u32(sQ), b = smem_u32(sK + st * kKBytes);
        const uint32_t d = tmem_base + kColS + sb * kTaK;
#pragma unroll
        for (int k = 0; k < DM / kUmmaK; ++k) {                     // 4 slices of k-block 0 (D = 80, 72: and 1 of k-block 1)
          const uint32_t off = (k >> 2) * kABytes + (k & 3) * (kUmmaK * 2);
          umma_bf16_ss(d, umma_desc_sw128_kmajor(a + off), umma_desc_sw128_kmajor(b + off), kIdescS, k != 0 ? 1u : 0u);
        }
        umma_commit(&s_full[sb]);
      };
      int g = 0, it = 0;
      for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++it) {
        mbar_wait(q_full, it & 1, 4);
        if constexpr (DM != D) {
          // Q channels D..DM-1 (16-byte chunk 1 of k-block 1 in each 128-byte swizzled row) are another head's: zero them, so that
          // they multiply K's foreign channels (finite values of the qkv rows, or TMA zero-fill) into exact zeros
          static_assert(DM - D == 8 && D - 64 == 8, "one foreign 16-byte chunk per row");
          uint8_t* q1 = sQ + kABytes;
#pragma unroll 8
          for (int r = 0; r < kTaQ; ++r) *reinterpret_cast<uint4*>(q1 + r * 128 + ((1 ^ (r & 7)) << 4)) = make_uint4(0u, 0u, 0u, 0u);
          fence_proxy_async_smem();                                 // generic-proxy writes -> visible to the tensor core's reads
        }
        issue_qk(g);
        for (int t = 0; t < ntiles; ++t, ++g) {
          const int st = g % kTaStages;
          if (t + 1 < ntiles) issue_qk(g + 1);
          else umma_commit(q_empty);                                // the item's last Q K^T has been issued: Q may be replaced once they are done
          mbar_wait(p_full, g & 1, 5);                              // P(t) is in shared memory, O has been rescaled
          tc_fence_after_sync();
          const uint32_t a = smem_u32(sP), b = smem_u32(sV + st * kVBytes);
#pragma unroll
          for (int k = 0; k < kTaK / kUmmaK; ++k) {
            const uint32_t offa = (k >> 2) * kABytes + (k & 3) * (kUmmaK * 2);
            const uint32_t offb = (k >> 2) * (DM * 128) + (k & 3) * (kUmmaK * 2);
            umma_bf16_ss(tmem_base + kColO, umma_desc_sw128_kmajor(a + offa), umma_desc_sw128_kmajor(b + offb), kIdescO, (t | k) != 0 ? 1u : 0u);
          }
          umma_commit(&kv_empty[st]);
          umma_commit(p_empty);
          if (t + 1 == ntiles) umma_commit(o_full);
        }
      }
    }
  } else {
    const int quad = warp & 3;                                      // TMEM lane quadrant this warp may access
    const int half = (warp - 2) >> 2;                               // which 64 of the tile's 128 keys (and which part of O) this warp handles
    const int r = quad * 32 + lane;                                 // query row inside the tile
    const uint32_t tlane = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    const float c = p.scale_log2e;
    constexpr int kOSplit = (DM / 16 + 1) / 2;                      // D = 80, 72: chunks 0-2 | 3-4; D = 64: 0-1 | 2-3
    const int oc0 = half == 0 ? 0 : kOSplit, oc1 = half == 0 ? kOSplit : DM / 16;  // 16-column chunks of O this warp rescales / stages
    int g = 0, it = 0;
    for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++it) {
      const int qt = item % qtiles, head = (item / qtiles) % p.heads, img = item / (qtiles * p.heads);
      const int q0 = qt * kTaQ;
      float m_run = -INFINITY, l_run = 0.f;                          // l_run: this thread's 64 columns only; the halves are added at the end
      for (int t = 0; t < ntiles; ++t, ++g) {
        const int sb = g & 1;
        const int kbase = t * kTaK + half * 64;
        mbar_wait(&s_full[sb], (g >> 1) & 1, 6);
        tc_fence_after_sync();
        const uint32_t srow = tlane + kColS + sb * kTaK + half * 64;
        float v[2][32];
        tmem_ld_32x32_nowait(srow, v[0]);
        tmem_ld_32x32_nowait(srow + 32, v[1]);
        tmem_ld_wait();
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&s_empty[sb]);                   // the scores are in registers: the buffer may be overwritten
        if (kbase + 64 > T) {                                       // ragged last tile (warp-uniform): keys past the sequence get no weight
#pragma unroll
          for (int ch = 0; ch < 2; ++ch)
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (kbase + ch * 32 + j >= T) v[ch][j] = -INFINITY;
        }
        float m8[8];
#pragma unroll
        for (int i = 0; i < 8; ++i)
          m8[i] = fmaxf(fmaxf(fmaxf(v[0][i], v[0][i + 8]), fmaxf(v[0][i + 16], v[0][i + 24])), fmaxf(fmaxf(v[1][i], v[1][i + 8]), fmaxf(v[1][i + 16], v[1][i + 24])));
        float mx = fmaxf(fmaxf(fmaxf(m8[0], m8[1]), fmaxf(m8[2], m8[3])), fmaxf(fmaxf(m8[4], m8[5]), fmaxf(m8[6], m8[7])));
        // row maximum over both halves (the other half's thread of this row lives in warp +- 4)
        float* xm = xch + (g & 1) * 256;
        xm[half * 128 + r] = mx;
        asm volatile("bar.sync 2, 256;\n" ::: "memory");
        mx = fmaxf(mx, xm[(half ^ 1) * 128 + r]);
        const float m_new = fmaxf(m_run, mx * c);                   // finite: key 0 of every tile is valid
        const float corr = ex2_approx(m_run - m_new);
        m_run = m_new;
        float s8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int ch = 0; ch < 2; ++ch)
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            v[ch][j] = ex2_approx(fmaf(v[ch][j], c, -m_new));
            s8[j & 7] += v[ch][j];
          }
        // the previous P has been consumed (and, inside an item, O is complete) once the previous P V has been committed
        if (g > 0) mbar_wait(p_empty, (g - 1) & 1, 7);
        tc_fence_after_sync();
        if (t > 0 && __any_sync(0xffffffffu, corr != 1.0f)) {
#pragma unroll 1
          for (int ch = oc0; ch < oc1; ++ch) {
            float ov[16];
            tmem_ld_32x16(tlane + kColO + ch * 16, ov);
#pragma unroll
            for (int j = 0; j < 16; ++j) ov[j] *= corr;
            tmem_st_32x16(tlane + kColO + ch * 16, ov);
          }
          tmem_st_wait();
        }
        // bf16 -> K-major swizzled operand rows: this thread's 64 keys are exactly k-block `half` of its row
        uint8_t* prow = sP + half * kABytes + r * 128;
#pragma unroll
        for (int ch = 0; ch < 2; ++ch)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int chunk = ch * 4 + q;
            *reinterpret_cast<uint4*>(prow + ((chunk ^ (r & 7)) << 4)) =
                make_uint4(pack_bf16x2(v[ch][q * 8 + 0], v[ch][q * 8 + 1]), pack_bf16x2(v[ch][q * 8 + 2], v[ch][q * 8 + 3]),
                           pack_bf16x2(v[ch][q * 8 + 4], v[ch][q * 8 + 5]), pack_bf16x2(v[ch][q * 8 + 6], v[ch][q * 8 + 7]));
          }
        l_run = l_run * corr + (((s8[0] + s8[4]) + (s8[1] + s8[5])) + ((s8[2] + s8[6]) + (s8[3] + s8[7])));
        fence_proxy_async_smem();                                   // P rows -> visible to the tensor core's shared-memory reads
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_full);
      }
      // epilogue: O / l -> bf16 -> rows staged in the (consumed) P region -> 16-byte stores
      float* xl = xch + 512;
      xl[half * 128 + r] = l_run;
      mbar_wait(o_full, it & 1, 8);
      tc_fence_after_sync();
      asm volatile("bar.sync 2, 256;\n" ::: "memory");
      const float inv = 1.0f / (l_run + xl[(half ^ 1) * 128 + r]);
      __nv_bfloat16* so = reinterpret_cast<__nv_bfloat16*>(sP) + r * (DM + 8);
#pragma unroll 1
      for (int ch = oc0; ch < oc1; ++ch) {
        float ov[16];
        tmem_ld_32x16(tlane + kColO + ch * 16, ov);
        *reinterpret_cast<uint4*>(so + ch * 16) = make_uint4(pack_bf16x2(ov[0] * inv, ov[1] * inv), pack_bf16x2(ov[2] * inv, ov[3] * inv),
                                                             pack_bf16x2(ov[4] * inv, ov[5] * inv), pack_bf16x2(ov[6] * inv, ov[7] * inv));
        *reinterpret_cast<uint4*>(so + ch * 16 + 8) = make_uint4(pack_bf16x2(ov[8] * inv, ov[9] * inv), pack_bf16x2(ov[10] * inv, ov[11] * inv),
                                                                 pack_bf16x2(ov[12] * inv, ov[13] * inv), pack_bf16x2(ov[14] * inv, ov[15] * inv));
      }
      asm volatile("bar.sync 1, 256;\n" ::: "memory");                 // both halves of every row are staged
      // each warp copies 16 rows: 16 rows x D / 8 chunks of 16 B (the staged columns D..DM-1 are not stored)
      constexpr int kChunks = D / 8;
      __nv_bfloat16* dst = p.out + static_cast<size_t>(img) * T * W + head * D;
      const int row0 = quad * 32 + half * 16;
      const __nv_bfloat16* sw = reinterpret_cast<const __nv_bfloat16*>(sP) + row0 * (DM + 8);
      for (int i = lane; i < 16 * kChunks; i += 32) {
        const int rr = i / kChunks, cc = i - rr * kChunks;
        const int row = q0 + row0 + rr;
        if (row < T) *reinterpret_cast<uint4*>(dst + static_cast<size_t>(row) * W + cc * 8) = *reinterpret_cast<const uint4*>(sw + rr * (DM + 8) + cc * 8);
      }
      // the staging rows overlap the P rows of other warps: nobody writes the next item's P before everyone has copied
      asm volatile("bar.sync 1, 256;\n" ::: "memory");
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) tmem_dealloc<512>(tmem_base);
}

// ---------------------------------------------------------------------------------------------------------
// SigLIP MAP head (timm AttentionPoolLatent)
// ---------------------------------------------------------------------------------------------------------
// q[n] = latent . Wq[n, :] + bq[n] (fp32, once per set of weights: the latent query is the same for every image).  One warp per output.
__global__ void __launch_bounds__(256) siglip_latent_q_kernel(const float* __restrict__ latent, const float* __restrict__ wq, const float* __restrict__ bq,
                                                              float* __restrict__ q, int W) {
  const int n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (n >= W) return;
  const float* wr = wq + static_cast<size_t>(n) * W;
  float s = 0.f;
  for (int k = lane; k < W; k += 32) s = fmaf(__ldg(latent + k), __ldg(wr + k), s);
  s = warp_sum(s);
  if (lane == 0) q[n] = s + __ldg(bq + n);
}

// out[img, h * D + c] = softmax_t(q_h . k_t / sqrt(D)) v_t[c] over the T tokens of one image (bf16 out, fp32 throughout).
// kv: bf16 [images * T, 2 W] (k | v, head h at columns h * D).  One warp per (image, head): lanes in four groups of eight, each group
// one key (or value) row per step, each lane the 16-byte chunks c, c + 8, ... of the row's D / 8 (D = 64: one 128-byte row, one chunk
// per lane; D = 72: 144 bytes, the ninth chunk on the group's first lane); scores go through the warp's T floats of shared memory.
constexpr int kMapWarps = 4;
constexpr int kMapMaxTokens = 3072;       // the scores of kMapWarps warps stay within the 48 KB of default dynamic shared memory
template <int D>
__global__ void __launch_bounds__(kMapWarps * 32) siglip_map_attention_kernel(const __nv_bfloat16* __restrict__ kv, const float* __restrict__ q,
                                                                              __nv_bfloat16* __restrict__ out, int T, int W, int heads, int items, float scale_log2e) {
  static_assert(D % 8 == 0 && D >= 64 && D < 128, "one to two 16-byte chunks per lane");
  constexpr int kChunks = D / 8, kPer = (kChunks + 7) / 8;
  extern __shared__ float sm_map[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * kMapWarps + warp;
  if (item >= items) return;
  const int img = item / heads, head = item - img * heads;
  const int grp = lane >> 3, c0 = (lane & 7) * 8;
  const bool has2 = kPer > 1 && (lane & 7) + 8 < kChunks;      // lane's second chunk (D = 72: the group's first lane)
  float* sc = sm_map + warp * T;
  const __nv_bfloat16* krow = kv + static_cast<size_t>(img) * T * 2 * W + head * D + c0;
  const __nv_bfloat16* vrow = krow + W;
  float qv[kPer][8];
#pragma unroll
  for (int i = 0; i < kPer; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) qv[i][j] = i == 0 || has2 ? __ldg(q + head * D + c0 + i * 64 + j) * scale_log2e : 0.f;   // scores in log2 units
  for (int t0 = 0; t0 < T; t0 += 4) {
    const int t = t0 + grp;
    float s = 0.f;
    if (t < T) {
#pragma unroll
      for (int i = 0; i < kPer; ++i) {
        if (i > 0 && !has2) break;
        const uint4 u = __ldg(reinterpret_cast<const uint4*>(krow + static_cast<size_t>(t) * 2 * W + i * 64));
        const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = __bfloat1622float2(h2[j]);
          s = fmaf(qv[i][2 * j], f.x, fmaf(qv[i][2 * j + 1], f.y, s));
        }
      }
    }
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    if ((lane & 7) == 0 && t < T) sc[t] = s;
  }
  __syncwarp();
  float m = -INFINITY;
  for (int t = lane; t < T; t += 32) m = fmaxf(m, sc[t]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  float l = 0.f;
  for (int t = lane; t < T; t += 32) {
    const float e = exp2f(sc[t] - m);
    sc[t] = e;
    l += e;
  }
  l = warp_sum(l);
  __syncwarp();
  float acc[kPer][8];
#pragma unroll
  for (int i = 0; i < kPer; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  for (int t = grp; t < T; t += 4) {
    const float pt = sc[t];
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
      if (i > 0 && !has2) break;
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(vrow + static_cast<size_t>(t) * 2 * W + i * 64));
      const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = __bfloat1622float2(h2[j]);
        acc[i][2 * j] = fmaf(pt, f.x, acc[i][2 * j]);
        acc[i][2 * j + 1] = fmaf(pt, f.y, acc[i][2 * j + 1]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < kPer; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      acc[i][j] += __shfl_xor_sync(0xffffffffu, acc[i][j], 8);
      acc[i][j] += __shfl_xor_sync(0xffffffffu, acc[i][j], 16);
    }
  if (grp == 0) {
    const float inv = 1.0f / l;
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
      if (i > 0 && !has2) break;
      *reinterpret_cast<uint4*>(out + static_cast<size_t>(img) * W + head * D + c0 + i * 64) =
          make_uint4(pack_bf16x2(acc[i][0] * inv, acc[i][1] * inv), pack_bf16x2(acc[i][2] * inv, acc[i][3] * inv),
                     pack_bf16x2(acc[i][4] * inv, acc[i][5] * inv), pack_bf16x2(acc[i][6] * inv, acc[i][7] * inv));
    }
  }
}

// embed[b, :] /= ||embed[b, :]|| (fp32; embedders.py:764).  One warp per row.
__global__ void __launch_bounds__(256) vit_normalize_kernel(float* __restrict__ e, int rows, int F) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (row >= rows) return;
  float* r = e + static_cast<size_t>(row) * F;
  float s = 0.f;
  for (int i = lane; i < F; i += 32) s = fmaf(r[i], r[i], s);
  s = warp_sum(s);
  const float inv = 1.0f / fmaxf(sqrtf(s), 1e-12f);
  for (int i = lane; i < F; i += 32) r[i] *= inv;
}

}  // namespace novic
