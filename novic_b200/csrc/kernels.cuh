// Non-GEMM kernels of the decoder hot path: embedding normalisation, token-embedding gather + LayerNorm,
// KV-cache attention (decode / prefill / teacher-forced), greedy and beam selection over the vocabulary
// partials written by the logits epilogue, loss reduction, and the fused embedding-noise kernel.
// All of them are HBM/L2-bound byte shuffling: warp-per-row, 128-bit coalesced accesses, shuffles for the
// reductions, no shared-memory staging needed.
#pragma once

#include <curand_kernel.h>

#include "gemm.cuh"

namespace novic {

constexpr int kHeads = 8;
constexpr int kHeadDim = 64;
constexpr int kWarpsPerBlock = 4;

// ---------------------------------------------------------------------------------------------------------
// F.normalize(embed) -> bf16 (embedding_decoder.py:1276), warp per row
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
embed_prep_kernel(const float* __restrict__ embed, __nv_bfloat16* __restrict__ out, int B, int F) {
  pdl_trigger();
  pdl_wait();
  const int row = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (row >= B) return;
  const int lane = lane_id();
  const float4* src = reinterpret_cast<const float4*>(embed + static_cast<size_t>(row) * F);
  float ss = 0.f;
  for (int i = lane; i < F / 4; i += 32) {
    const float4 v = __ldg(src + i);
    ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  ss = warp_sum(ss);
  const float inv = 1.0f / fmaxf(sqrtf(ss), 1e-12f);
  uint2* dst = reinterpret_cast<uint2*>(out + static_cast<size_t>(row) * F);
  for (int i = lane; i < F / 4; i += 32) {
    const float4 v = __ldg(src + i);
    dst[i] = make_uint2(pack_bf16x2(v.x * inv, v.y * inv), pack_bf16x2(v.z * inv, v.w * inv));
  }
}

// ---------------------------------------------------------------------------------------------------------
// One residual-stream row from a token id: x = W_tied[tok] + pos[p]; xn = LayerNorm(x) * gain -> bf16.
// Executed by a full warp; lane owns columns [16*lane, 16*lane + 16).
// ---------------------------------------------------------------------------------------------------------
// xs != nullptr: the fp32 values go to a shared-memory image of the row's 32-row block of the blocked layout instead of to x -
// float4 unit (col4, r) at xs[col4 * 32 + (r ^ ((col4 >> 2) & 31))] (the XOR keeps both the row-wise writes here and the block-wise
// read-out of select_greedy_kernel free of bank conflicts) - and the caller writes the whole 64 KB block with coalesced stores.
__device__ __forceinline__ void embed_token_row(const float* __restrict__ wtok, const float* __restrict__ pos_row,
                                                const float* __restrict__ gain, long long tok, int out_row,
                                                float* __restrict__ x, __nv_bfloat16* __restrict__ xn, float eps, float4* xs = nullptr) {
  const int lane = lane_id();
  const float4* w4 = reinterpret_cast<const float4*>(wtok + static_cast<size_t>(tok) * kE) + lane * 4;
  const float4* p4 = reinterpret_cast<const float4*>(pos_row) + lane * 4;
  float v[16];
  float sum = 0.f, sumsq = 0.f;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float4 a = __ldg(w4 + q);
    const float4 b = __ldg(p4 + q);
    v[q * 4 + 0] = a.x + b.x; v[q * 4 + 1] = a.y + b.y; v[q * 4 + 2] = a.z + b.z; v[q * 4 + 3] = a.w + b.w;
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) { sum += v[i]; sumsq += v[i] * v[i]; }
  sum = warp_sum(sum);
  sumsq = warp_sum(sumsq);
  const float mean = sum * (1.0f / kE);
  const float rstd = rsqrtf(fmaxf(sumsq * (1.0f / kE) - mean * mean, 0.f) + eps);
  if (xs != nullptr) {
#pragma unroll
    for (int q = 0; q < 4; ++q)
      xs[(lane * 4 + q) * 32 + ((out_row & 31) ^ lane)] = make_float4(v[q * 4], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
  } else {
#pragma unroll
    for (int q = 0; q < 4; ++q)
      *reinterpret_cast<float4*>(x + xblk_off(out_row, lane * 4 + q)) =
          make_float4(v[q * 4], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
  }
  const float4* g4 = reinterpret_cast<const float4*>(gain) + lane * 4;
  uint32_t o[8];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float4 g = __ldg(g4 + q);
    o[q * 2 + 0] = pack_bf16x2((v[q * 4 + 0] - mean) * rstd * g.x, (v[q * 4 + 1] - mean) * rstd * g.y);
    o[q * 2 + 1] = pack_bf16x2((v[q * 4 + 2] - mean) * rstd * g.z, (v[q * 4 + 3] - mean) * rstd * g.w);
  }
  uint4* d = reinterpret_cast<uint4*>(xn + static_cast<size_t>(out_row) * kE) + lane * 2;
  d[0] = make_uint4(o[0], o[1], o[2], o[3]);
  d[1] = make_uint4(o[4], o[5], o[6], o[7]);
}

// Teacher-forced token rows (embedding_decoder.py:692-693): sequence a, token index i -> row a*S + P + i.
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
token_embed_kernel(const long long* __restrict__ target, int ld_target, int nseq, int ntok, int S, int P, int V,
                   const float* __restrict__ wtok, const float* __restrict__ pos, const float* __restrict__ gain,
                   float* __restrict__ x, __nv_bfloat16* __restrict__ xn, float eps) {
  const int w = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (w >= nseq * ntok) return;
  const int a = w / ntok, i = w - a * ntok;
  long long tok = target[static_cast<size_t>(a) * ld_target + i];
  tok = tok < 0 ? 0 : (tok >= V ? V - 1 : tok);
  embed_token_row(wtok, pos + static_cast<size_t>(P + i) * kE, gain, tok, a * S + P + i, x, xn, eps);
}

// ---------------------------------------------------------------------------------------------------------
// Attention over the KV cache.  One warp per (sequence, query position); lane owns 16 contiguous channels
// (head = lane / 4), K/V rows are read as 2 x 128-bit per lane (1 KB per row per warp, fully coalesced),
// scores are reduced over the 4 lanes of a head with shuffles, softmax is online in fp32.
// Visibility (embedding_decoder.py:651-654, :696-712): key j is visible to query s iff j <= s, or both are
// prefix positions (unless strictly causal); a key-padding byte masks key j > 0.
// KV pages: prefix positions live in the page of the first beam of the sequence's group; token position j
// lives in the page named by the ancestry table (beam search reorders by rewriting this table, never by
// moving K/V); the query's own position is always in the sequence's own page.
// ---------------------------------------------------------------------------------------------------------
struct AttnParams {
  const __nv_bfloat16* q;
  const __nv_bfloat16* kcache;
  const __nv_bfloat16* vcache;
  __nv_bfloat16* out;
  const unsigned char* keypad;  // optional [nseq, keypad_ld]
  const unsigned char* anc;     // optional [nseq, anc_ld]
  int nseq, nq, q0, smax, P, beams, slot_mul, prefix_bidir, keypad_ld, anc_ld;
  int early_loads;              // stream kernel: request chunks of older rows before griddepcontrol.wait
  int stream_hint;              // stream kernel: K/V rows are requested with an evict-first L2 policy (the decoder always sets it)
  DropCfg drop;                 // attention_tf_kernel<true> (training): dropout on the attention probabilities (thresh 0 = off)
  uint32_t drop_site;
  float scale_log2e;            // (1/sqrt(head_dim)) * log2(e)
};

__device__ __forceinline__ void bf16x8_to_f32(const uint4& u, float* f) {
  float2 t;
  t = unpack_bf16x2(u.x); f[0] = t.x; f[1] = t.y;
  t = unpack_bf16x2(u.y); f[2] = t.x; f[3] = t.y;
  t = unpack_bf16x2(u.z); f[4] = t.x; f[5] = t.y;
  t = unpack_bf16x2(u.w); f[6] = t.x; f[7] = t.y;
}

// ---------------------------------------------------------------------------------------------------------
// Attention, bulk-async version.  A warp-per-query kernel with register-staged loads (12 warps/SM; removed, see the history)
// kept too few bytes in flight: ncu showed 40 % of HBM peak.  Here a persistent CTA runs one producer warp
// that streams each sequence's K and V pages into a shared-memory ring with cp.async.bulk (TMA engine, no
// registers, completion on an mbarrier) while 8 consumer warps compute from shared memory: up to ~190 KB per SM
// are in flight at all times.  One ring stage = all the K rows then all the V rows one sequence needs
// (contiguous in its page unless beam search's ancestry table redirects token rows to sibling pages).
// ---------------------------------------------------------------------------------------------------------
constexpr int kAttnConsumers = 8;
constexpr int kAttnThreads = (kAttnConsumers + 1) * 32;
constexpr int kAttnMaxStages = 16;

// `ncons` consumer warps are active and nstages is a multiple of ncons: consumer c then owns ring stages c, c+ncons, ...
// and visits them in order, so it observes every phase of their mbarriers (a parity wait can only tell the current
// phase from the previous one - a waiter must never be a whole phase ahead).
__global__ void __launch_bounds__(kAttnThreads, 1) attention_bulk_kernel(const AttnParams p, int nstages, int stage_bytes, int ncons) {
  extern __shared__ __align__(128) uint8_t attn_smem[];
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(attn_smem);
  uint64_t* empty_bar = full_bar + kAttnMaxStages;
  uint8_t* ring = attn_smem + 2 * kAttnMaxStages * sizeof(uint64_t);

  const int warp = threadIdx.x >> 5;
  const int lane = lane_id();
  pdl_trigger();
  const int per_cta = (p.nseq + gridDim.x - 1) / gridDim.x;
  const int item0 = blockIdx.x * per_cta;
  const int item1 = min(p.nseq, item0 + per_cta);
  const int nk_max = max((p.prefix_bidir ? p.P : 1), p.q0 + p.nq);   // rows staged per sequence

  if (threadIdx.x == 0) {
    for (int s = 0; s < nstages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    fence_mbar_init();
  }
  __syncthreads();
  pdl_wait();

  if (warp == kAttnConsumers) {
    // ------------------------------ producer ------------------------------
    for (int it = item0, k = 0; it < item1; ++it, ++k) {
      const int stage = k % nstages;
      const uint32_t phase = static_cast<uint32_t>(k / nstages) & 1u;
      const int a = it;
      const int own_slot = a * p.slot_mul;
      const int group0 = (own_slot / p.beams) * p.beams;
      uint8_t* dst = ring + static_cast<size_t>(stage) * stage_bytes;
      if (lane == 0) {
        mbar_wait(&empty_bar[stage], phase ^ 1u, 4);
        mbar_arrive_expect_tx(&full_bar[stage], static_cast<uint32_t>(nk_max) * 2048u);
      }
      __syncwarp();
      const bool contiguous = (p.beams == 1);
      if (contiguous) {
        if (lane == 0) {
          const size_t off = static_cast<size_t>(own_slot) * p.smax * kE;
          bulk_load_1d(dst, p.kcache + off, static_cast<uint32_t>(nk_max) * 1024u, &full_bar[stage]);
          bulk_load_1d(dst + nk_max * 1024, p.vcache + off, static_cast<uint32_t>(nk_max) * 1024u, &full_bar[stage]);
        }
      } else {
        const int qlast = p.q0 + p.nq - 1;
        for (int j = lane; j < nk_max; j += 32) {
          int slot;
          if (j < p.P) slot = group0;
          else if (p.anc != nullptr && j < qlast) slot = group0 + p.anc[static_cast<size_t>(a) * p.anc_ld + (j - p.P)];
          else slot = own_slot;
          const size_t off = (static_cast<size_t>(slot) * p.smax + j) * kE;
          bulk_load_1d(dst + j * 1024, p.kcache + off, 1024u, &full_bar[stage]);
          bulk_load_1d(dst + (nk_max + j) * 1024, p.vcache + off, 1024u, &full_bar[stage]);
        }
      }
    }
  } else if (warp < ncons) {
    // ------------------------------ consumers ------------------------------
    for (int it = item0 + warp, k = warp; it < item1; it += ncons, k += ncons) {
      const int stage = k % nstages;
      const uint32_t phase = static_cast<uint32_t>(k / nstages) & 1u;
      const int a = it;
      const uint8_t* kbase = ring + static_cast<size_t>(stage) * stage_bytes;
      const uint8_t* vbase = kbase + nk_max * 1024;
      bool waited = false;
      for (int qi = 0; qi < p.nq; ++qi) {
        const int w = a * p.nq + qi;
        const int qpos = p.q0 + qi;
        const int nkeys = (p.prefix_bidir && qpos < p.P) ? p.P : qpos + 1;
        float qf[16];
        {
          const uint4* q4 = reinterpret_cast<const uint4*>(p.q + static_cast<size_t>(w) * kE) + lane * 2;
          const uint4 u0 = __ldg(q4), u1 = __ldg(q4 + 1);
          bf16x8_to_f32(u0, qf);
          bf16x8_to_f32(u1, qf + 8);
#pragma unroll
          for (int i = 0; i < 16; ++i) qf[i] *= p.scale_log2e;
        }
        if (!waited) { mbar_wait(&full_bar[stage], phase, 5); waited = true; }
        float m = -INFINITY, l = 0.f, acc[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) acc[i] = 0.f;
#pragma unroll 2
        for (int j = 0; j < nkeys; ++j) {
          if (p.keypad != nullptr && j > 0 && p.keypad[static_cast<size_t>(a) * p.keypad_ld + j]) continue;  // warp-uniform
          const uint4* k4 = reinterpret_cast<const uint4*>(kbase + j * 1024) + lane * 2;
          float kf[16];
          bf16x8_to_f32(k4[0], kf);
          bf16x8_to_f32(k4[1], kf + 8);
          float s = 0.f;
#pragma unroll
          for (int i = 0; i < 16; ++i) s = fmaf(qf[i], kf[i], s);
          s += __shfl_xor_sync(0xffffffffu, s, 1);
          s += __shfl_xor_sync(0xffffffffu, s, 2);
          const float m_new = fmaxf(m, s);
          const float corr = exp2f(m - m_new);
          const float pj = exp2f(s - m_new);
          l = l * corr + pj;
          const uint4* v4 = reinterpret_cast<const uint4*>(vbase + j * 1024) + lane * 2;
          float vf[16];
          bf16x8_to_f32(v4[0], vf);
          bf16x8_to_f32(v4[1], vf + 8);
#pragma unroll
          for (int i = 0; i < 16; ++i) acc[i] = fmaf(acc[i], corr, pj * vf[i]);
          m = m_new;
        }
        const float inv = 1.0f / l;
        uint32_t o[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = pack_bf16x2(acc[2 * i] * inv, acc[2 * i + 1] * inv);
        uint4* d = reinterpret_cast<uint4*>(p.out + static_cast<size_t>(w) * kE) + lane * 2;
        d[0] = make_uint4(o[0], o[1], o[2], o[3]);
        d[1] = make_uint4(o[4], o[5], o[6], o[7]);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty_bar[stage]);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// Attention, decode-step version (one query per sequence, no key padding): self-service streaming.
//
// ncu on the kernel above (profiles/r01_ncu_full_v3_summary.txt): 2.1 warps per scheduler, 6.7 cycles per issued
// instruction, issue slots 32 % busy - the 8 (or fewer: one per ring stage) consumer warps walk a serial
// online-softmax chain per key and are the bottleneck, not HBM.  Here 16 warps per CTA each stream their own
// sequences: a warp owns three 4 KB slots, lane 0 issues cp.async.bulk copies of up to four K rows (then the same
// four V rows) three copies ahead of consumption, and the four keys of a chunk are scored as independent chains
// before one softmax update (4x fewer dependent exp2 / max steps, 4x the ILP).  No producer warp, no empty
// barriers: a slot is refilled by the warp that just finished reading it.  Chunks that only hold rows written in
// earlier decode steps are requested before griddepcontrol.wait, so the stream starts under the previous kernel's tail.
// ---------------------------------------------------------------------------------------------------------
constexpr int kAsWarps = 16;
constexpr int kAsSlots = 3;
constexpr int kAsChunk = 4;                          // keys per chunk
constexpr int kAsSlotBytes = kAsChunk * 1024;        // one chunk of K rows or of V rows
constexpr int kAsThreads = kAsWarps * 32;
constexpr int kAsSmemBytes = kAsWarps * kAsSlots * kAsSlotBytes + kAsWarps * kAsSlots * 8 + 128;
__host__ __device__ constexpr int as_smem_bytes(int warps, int slots, int chunk) { return warps * slots * chunk * 1024 + warps * slots * 8 + 128; }

// WARPS x SLOTS x CHUNK KB of shared memory; the decoder instantiates <16, 3, 4> (other shapes were measured slower, DESIGN.md section 5).
template <int WARPS, int SLOTS, int CHUNK>
__global__ void __launch_bounds__(WARPS * 32, 1) attention_stream_kernel_t(const AttnParams p) {
  constexpr int kAsWarps = WARPS, kAsSlots = SLOTS, kAsChunk = CHUNK, kAsSlotBytes = CHUNK * 1024;
  extern __shared__ __align__(128) uint8_t as_smem[];
  const int warp = threadIdx.x >> 5;
  const int lane = lane_id();
  uint8_t* slots = as_smem + static_cast<size_t>(warp) * (kAsSlots * kAsSlotBytes);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(as_smem + kAsWarps * kAsSlots * kAsSlotBytes) + warp * kAsSlots;
  pdl_trigger();

  const int per_cta = (p.nseq + gridDim.x - 1) / gridDim.x;
  const int item0 = blockIdx.x * per_cta;
  const int item1 = min(p.nseq, item0 + per_cta);
  const int qpos = p.q0;
  const int nkeys = (p.prefix_bidir && qpos < p.P) ? p.P : qpos + 1;
  const int nchunks = (nkeys + kAsChunk - 1) / kAsChunk;
  const int per_item = 2 * nchunks;                                  // K chunk, V chunk, K chunk, ...
  const int nitems = (item0 + warp < item1) ? (item1 - item0 - warp + kAsWarps - 1) / kAsWarps : 0;
  const int nloads = nitems * per_item;
  const bool contiguous = p.beams == 1;

  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < kAsSlots; ++s) mbar_init(&full_bar[s], 1);
    fence_mbar_init();
  }
  __syncwarp();

  // request load n of this warp's stream into slot n % kAsSlots
  auto issue = [&](int n) {
    const int i = n / per_item, r = n - i * per_item;
    const int c = r >> 1, kv = r & 1;
    const int a = item0 + warp + i * kAsWarps;
    const int j0 = c * nkeys / nchunks, rows = (c + 1) * nkeys / nchunks - j0;
    const __nv_bfloat16* base = kv ? p.vcache : p.kcache;
    const int sl = n % kAsSlots;
    uint8_t* dst = slots + sl * kAsSlotBytes;
    const int own_slot = a * p.slot_mul;
    if (lane == 0) mbar_arrive_expect_tx(&full_bar[sl], static_cast<uint32_t>(rows) * 1024u);
    if (contiguous) {
      if (lane == 0) {
        const void* src = base + (static_cast<size_t>(own_slot) * p.smax + j0) * kE;
        if (p.stream_hint) bulk_load_1d_hint(dst, src, static_cast<uint32_t>(rows) * 1024u, &full_bar[sl], 0x12F0000000000000ull /* evict first */);
        else bulk_load_1d(dst, src, static_cast<uint32_t>(rows) * 1024u, &full_bar[sl]);
      }
    } else {
      __syncwarp();
      if (lane < rows) {
        const int j = j0 + lane;
        const int group0 = (own_slot / p.beams) * p.beams;
        int slot;
        if (j < p.P) slot = group0;
        else if (p.anc != nullptr && j < qpos) slot = group0 + p.anc[static_cast<size_t>(a) * p.anc_ld + (j - p.P)];
        else slot = own_slot;
        bulk_load_1d(dst + lane * 1024, base + (static_cast<size_t>(slot) * p.smax + j) * kE, 1024u, &full_bar[sl]);
      }
    }
  };

  // chunks other than an item's last hold only rows written by earlier decode steps: safe to request before the wait, because
  // select_greedy_kernel releases its dependents only after its own wait (no kernel of this step started before the previous step,
  // and with it the prefix pass, had completed)
  int issued = 0;
  if (p.early_loads == 1 && contiguous && nchunks >= 2) {
    const int early = min(min(nloads, kAsSlots), nchunks >= 3 ? 3 : 2);
    for (; issued < early; ++issued) issue(issued);
  } else if (p.early_loads == 3 && contiguous && nchunks >= 2 && nloads > 0) {   // diagnostic: generic-proxy probe of the same addresses
    const int a0 = item0 + warp;
    const uint4* probe = reinterpret_cast<const uint4*>(p.kcache + (static_cast<size_t>(a0 * p.slot_mul) * p.smax) * kE) + lane;
    const uint4 t = __ldcg(probe);
    if (t.x == 0x7fc12345u && t.y == 0x12345678u) as_smem[0] = 1;
  }
  pdl_wait();
  for (; issued < min(nloads, kAsSlots); ++issued) issue(issued);

  float qf[16], acc[16], pj[kAsChunk];
  float m = -INFINITY, l = 0.f, corr = 0.f;
  uint4 qa = make_uint4(0, 0, 0, 0), qb = qa;
  if (nitems > 0) {
    const uint4* q4 = reinterpret_cast<const uint4*>(p.q + static_cast<size_t>(item0 + warp) * kE) + lane * 2;
    qa = __ldg(q4); qb = __ldg(q4 + 1);
  }
  int i = 0, r = 0;
  for (int n = 0; n < nloads; ++n) {
    const int a = item0 + warp + i * kAsWarps;
    const int c = r >> 1;
    const int j0 = c * nkeys / nchunks, rows = (c + 1) * nkeys / nchunks - j0;
    if (r == 0) {
      bf16x8_to_f32(qa, qf);
      bf16x8_to_f32(qb, qf + 8);
#pragma unroll
      for (int k = 0; k < 16; ++k) { qf[k] *= p.scale_log2e; acc[k] = 0.f; }
      m = -INFINITY; l = 0.f;
      if (i + 1 < nitems) {   // next item's query: in flight while this item streams
        const uint4* q4 = reinterpret_cast<const uint4*>(p.q + static_cast<size_t>(a + kAsWarps) * kE) + lane * 2;
        qa = __ldg(q4); qb = __ldg(q4 + 1);
      }
    }
    const int sl = n % kAsSlots;
    const uint8_t* src = slots + sl * kAsSlotBytes + lane * 32;
    mbar_wait(&full_bar[sl], static_cast<uint32_t>(n / kAsSlots) & 1u, 5);
    if ((r & 1) == 0) {
      float s[kAsChunk];
#pragma unroll
      for (int u = 0; u < kAsChunk; ++u) {
        s[u] = -INFINITY;
        if (u < rows) {
          const uint4* k4 = reinterpret_cast<const uint4*>(src + u * 1024);
          float kf[16];
          bf16x8_to_f32(k4[0], kf);
          bf16x8_to_f32(k4[1], kf + 8);
          float d0 = 0.f, d1 = 0.f;
#pragma unroll
          for (int k = 0; k < 8; ++k) { d0 = fmaf(qf[k], kf[k], d0); d1 = fmaf(qf[8 + k], kf[8 + k], d1); }
          s[u] = d0 + d1;
        }
      }
#pragma unroll
      for (int u = 0; u < kAsChunk; ++u) {
        if (u < rows) {
          s[u] += __shfl_xor_sync(0xffffffffu, s[u], 1);
          s[u] += __shfl_xor_sync(0xffffffffu, s[u], 2);
        }
      }
      float m_new = m;
#pragma unroll
      for (int u = 0; u < kAsChunk; ++u) m_new = fmaxf(m_new, s[u]);
      corr = exp2f(m - m_new);
      float psum = 0.f;
#pragma unroll
      for (int u = 0; u < kAsChunk; ++u) { pj[u] = exp2f(s[u] - m_new); psum += pj[u]; }
      l = l * corr + psum;
      m = m_new;
    } else {
#pragma unroll
      for (int k = 0; k < 16; ++k) acc[k] *= corr;
#pragma unroll
      for (int u = 0; u < kAsChunk; ++u) {
        if (u < rows) {
          const uint4* v4 = reinterpret_cast<const uint4*>(src + u * 1024);
          float vf[16];
          bf16x8_to_f32(v4[0], vf);
          bf16x8_to_f32(v4[1], vf + 8);
#pragma unroll
          for (int k = 0; k < 16; ++k) acc[k] = fmaf(pj[u], vf[k], acc[k]);
        }
      }
    }
    __syncwarp();                       // every lane has consumed the slot: refill it
    if (issued < nloads) { issue(issued); ++issued; }
    if (++r == per_item) {
      const float inv = 1.0f / l;
      uint32_t o[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = pack_bf16x2(acc[2 * k] * inv, acc[2 * k + 1] * inv);
      uint4* d = reinterpret_cast<uint4*>(p.out + static_cast<size_t>(a) * kE) + lane * 2;
      d[0] = make_uint4(o[0], o[1], o[2], o[3]);
      d[1] = make_uint4(o[4], o[5], o[6], o[7]);
      r = 0;
      ++i;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// Attention, decode-step version for SMALL batches (at most 4 x #SMs sequences, at most 24 keys): the stream kernel above gives every
// sequence one warp, so 512 sequences occupy 32 CTAs and every warp walks its sequence's 2-5 chunks as a chain of HBM round trips (9 us
// per launch for 17 MB at 512 sequences).  Here a CTA takes four sequences and FOUR warps share a sequence's keys: each warp requests all
// its K rows and all its V rows at once (one round trip), computes a partial softmax (max, sum, weighted V) over its at most 6 keys, and
// the four partials are merged through shared memory (each warp's K slot, free by then, holds its partial).
// ---------------------------------------------------------------------------------------------------------
constexpr int kSpWarps = 16, kSpParts = 4, kSpSeqs = kSpWarps / kSpParts, kSpMaxRows = 6;
constexpr int kSpMaxKeys = kSpParts * kSpMaxRows;                       // 24
constexpr int kSpSlotBytes = kSpMaxRows * 1024;                         // K rows (later: the warp's partial), V rows
constexpr int kSpSmemBytes = kSpWarps * 2 * kSpSlotBytes + kSpWarps * 2 * 8 + 128;

__global__ void __launch_bounds__(kSpWarps * 32, 1) attention_split_kernel(const AttnParams p) {
  extern __shared__ __align__(128) uint8_t sp_smem[];
  const int warp = threadIdx.x >> 5;
  const int lane = lane_id();
  const int sq = warp / kSpParts, part = warp % kSpParts;
  uint8_t* kslot = sp_smem + static_cast<size_t>(warp) * (2 * kSpSlotBytes);
  uint8_t* vslot = kslot + kSpSlotBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sp_smem + kSpWarps * 2 * kSpSlotBytes) + warp * 2;
  pdl_trigger();

  const int a = blockIdx.x * kSpSeqs + sq;
  const bool valid = a < p.nseq;
  const int qpos = p.q0;
  const int nkeys = (p.prefix_bidir && qpos < p.P) ? p.P : qpos + 1;
  const int j0 = part * nkeys / kSpParts, rows = valid ? (part + 1) * nkeys / kSpParts - j0 : 0;
  const bool contiguous = p.beams == 1;
  const int own_slot = a * p.slot_mul;
  if (lane == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); fence_mbar_init(); }
  __syncwarp();

  auto request = [&](int kv) {
    const __nv_bfloat16* base = kv ? p.vcache : p.kcache;
    uint8_t* dst = kv ? vslot : kslot;
    if (lane == 0) mbar_arrive_expect_tx(&bars[kv], static_cast<uint32_t>(rows) * 1024u);
    if (contiguous) {
      if (lane == 0) {
        const void* src = base + (static_cast<size_t>(own_slot) * p.smax + j0) * kE;
        if (p.stream_hint) bulk_load_1d_hint(dst, src, static_cast<uint32_t>(rows) * 1024u, &bars[kv], 0x12F0000000000000ull /* evict first */);
        else bulk_load_1d(dst, src, static_cast<uint32_t>(rows) * 1024u, &bars[kv]);
      }
    } else {
      __syncwarp();
      if (lane < rows) {
        const int j = j0 + lane;
        const int group0 = (own_slot / p.beams) * p.beams;
        int slot;
        if (j < p.P) slot = group0;
        else if (p.anc != nullptr && j < qpos) slot = group0 + p.anc[static_cast<size_t>(a) * p.anc_ld + (j - p.P)];
        else slot = own_slot;
        bulk_load_1d(dst + lane * 1024, base + (static_cast<size_t>(slot) * p.smax + j) * kE, 1024u, &bars[kv]);
      }
    }
  };
  // rows written by earlier decode steps (every part but the one that holds the newest key) may be requested before the wait - see
  // attention_stream_kernel_t
  const bool early = p.early_loads == 1 && contiguous && rows > 0 && j0 + rows <= qpos;
  if (early) { request(0); request(1); }
  pdl_wait();
  if (!early && rows > 0) { request(0); request(1); }

  float acc[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) acc[k] = 0.f;
  float m = -INFINITY, l = 0.f;
  if (rows > 0) {
    float qf[16];
    {
      const uint4* q4 = reinterpret_cast<const uint4*>(p.q + static_cast<size_t>(a) * kE) + lane * 2;
      const uint4 qa = __ldg(q4), qb = __ldg(q4 + 1);
      bf16x8_to_f32(qa, qf);
      bf16x8_to_f32(qb, qf + 8);
#pragma unroll
      for (int k = 0; k < 16; ++k) qf[k] *= p.scale_log2e;
    }
    float s[kSpMaxRows];
    mbar_wait(&bars[0], 0, 5);
#pragma unroll
    for (int u = 0; u < kSpMaxRows; ++u) {
      s[u] = -INFINITY;
      if (u < rows) {
        const uint4* k4 = reinterpret_cast<const uint4*>(kslot + u * 1024 + lane * 32);
        float kf[16];
        bf16x8_to_f32(k4[0], kf);
        bf16x8_to_f32(k4[1], kf + 8);
        float d0 = 0.f, d1 = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) { d0 = fmaf(qf[k], kf[k], d0); d1 = fmaf(qf[8 + k], kf[8 + k], d1); }
        s[u] = d0 + d1;
      }
    }
#pragma unroll
    for (int u = 0; u < kSpMaxRows; ++u) {
      if (u < rows) {
        s[u] += __shfl_xor_sync(0xffffffffu, s[u], 1);
        s[u] += __shfl_xor_sync(0xffffffffu, s[u], 2);
      }
    }
#pragma unroll
    for (int u = 0; u < kSpMaxRows; ++u) m = fmaxf(m, s[u]);
    float pj[kSpMaxRows];
#pragma unroll
    for (int u = 0; u < kSpMaxRows; ++u) { pj[u] = exp2f(s[u] - m); l += pj[u]; }
    mbar_wait(&bars[1], 0, 5);
#pragma unroll
    for (int u = 0; u < kSpMaxRows; ++u) {
      if (u < rows) {
        const uint4* v4 = reinterpret_cast<const uint4*>(vslot + u * 1024 + lane * 32);
        float vf[16];
        bf16x8_to_f32(v4[0], vf);
        bf16x8_to_f32(v4[1], vf + 8);
#pragma unroll
        for (int k = 0; k < 16; ++k) acc[k] = fmaf(pj[u], vf[k], acc[k]);
      }
    }
  }
  // partial of this warp -> its K slot (every lane has read its K rows: the scores are complete): acc at lane * 64 B, (m, l) of head h at 2048 + 8 h
  __syncwarp();
  {
    float4* d = reinterpret_cast<float4*>(kslot + lane * 64);
#pragma unroll
    for (int k = 0; k < 4; ++k) d[k] = make_float4(acc[4 * k], acc[4 * k + 1], acc[4 * k + 2], acc[4 * k + 3]);
    if ((lane & 3) == 0) *reinterpret_cast<float2*>(kslot + 2048 + (lane >> 2) * 8) = make_float2(m, l);
  }
  __syncthreads();
  if (part == 0 && valid) {
    float mp[kSpParts], lp[kSpParts];
    float mx = -INFINITY;
#pragma unroll
    for (int q = 0; q < kSpParts; ++q) {
      const float2 t = *reinterpret_cast<const float2*>(sp_smem + static_cast<size_t>(sq * kSpParts + q) * (2 * kSpSlotBytes) + 2048 + (lane >> 2) * 8);
      mp[q] = t.x; lp[q] = t.y;
      mx = fmaxf(mx, t.x);
    }
    float out[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) out[k] = 0.f;
    float L = 0.f;
#pragma unroll
    for (int q = 0; q < kSpParts; ++q) {
      const float w = lp[q] > 0.f ? exp2f(mp[q] - mx) : 0.f;
      L = fmaf(lp[q], w, L);
      const float4* src = reinterpret_cast<const float4*>(sp_smem + static_cast<size_t>(sq * kSpParts + q) * (2 * kSpSlotBytes) + lane * 64);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float4 t = src[k];
        out[4 * k] = fmaf(t.x, w, out[4 * k]); out[4 * k + 1] = fmaf(t.y, w, out[4 * k + 1]);
        out[4 * k + 2] = fmaf(t.z, w, out[4 * k + 2]); out[4 * k + 3] = fmaf(t.w, w, out[4 * k + 3]);
      }
    }
    const float inv = 1.0f / L;
    uint32_t o[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) o[k] = pack_bf16x2(out[2 * k] * inv, out[2 * k + 1] * inv);
    uint4* d = reinterpret_cast<uint4*>(p.out + static_cast<size_t>(a) * kE) + lane * 2;
    d[0] = make_uint4(o[0], o[1], o[2], o[3]);
    d[1] = make_uint4(o[4], o[5], o[6], o[7]);
  }
}

// ---------------------------------------------------------------------------------------------------------
// Attention of the PREFIX pass (queries 0..P-1 of every sequence against keys 0..P-1, P <= 4): the bulk kernel above spends 29 us per
// launch on 67 MB at 4096 sequences (8 consumer warps walk query after query, key after key).  Here a warp owns a sequence: its P K rows
// and P V rows arrive as two bulk copies (two sequences in flight per warp: 12 warps x 2 x 8 KB = 192 KB per SM), the P queries are
// prefetched into registers, and each query's at most four scores need no online rescaling.
// ---------------------------------------------------------------------------------------------------------
constexpr int kApWarps = 12, kApSets = 2, kApMaxP = 4;
constexpr int kApSetBytes = 2 * kApMaxP * 1024;                        // K rows then V rows of one sequence
constexpr int kApSmemBytes = kApWarps * kApSets * kApSetBytes + kApWarps * kApSets * 2 * 8 + 128;

__global__ void __launch_bounds__(kApWarps * 32, 1) attention_prefix_kernel(const AttnParams p) {
  extern __shared__ __align__(128) uint8_t ap_smem[];
  const int warp = threadIdx.x >> 5;
  const int lane = lane_id();
  uint8_t* sets = ap_smem + static_cast<size_t>(warp) * (kApSets * kApSetBytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(ap_smem + kApWarps * kApSets * kApSetBytes) + warp * (kApSets * 2);   // [set][K, V]
  pdl_trigger();
  const int P = p.nq;                                                 // == p.P, q0 == 0 (checked by the launcher)
  const int per_cta = (p.nseq + gridDim.x - 1) / gridDim.x;
  const int item0 = blockIdx.x * per_cta;
  const int item1 = min(p.nseq, item0 + per_cta);
  const int nitems = (item0 + warp < item1) ? (item1 - item0 - warp + kApWarps - 1) / kApWarps : 0;
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < kApSets * 2; ++s) mbar_init(&bars[s], 1);
    fence_mbar_init();
  }
  __syncwarp();
  auto request = [&](int i) {
    if (lane != 0) return;
    const int a = item0 + warp + i * kApWarps;
    const int st = i % kApSets;
    uint8_t* dst = sets + st * kApSetBytes;
    // prefix rows live in the page of the first beam of the sequence's group, positions 0..P-1: contiguous
    const int own_slot = a * p.slot_mul;
    const size_t off = (static_cast<size_t>((own_slot / p.beams) * p.beams) * p.smax) * kE;
    const uint32_t bytes = static_cast<uint32_t>(P) * 1024u;
    mbar_arrive_expect_tx(&bars[st * 2], bytes);
    bulk_load_1d(dst, p.kcache + off, bytes, &bars[st * 2]);
    mbar_arrive_expect_tx(&bars[st * 2 + 1], bytes);
    bulk_load_1d(dst + kApMaxP * 1024, p.vcache + off, bytes, &bars[st * 2 + 1]);
  };
  pdl_wait();
  for (int i = 0; i < min(nitems, kApSets); ++i) request(i);
  for (int i = 0; i < nitems; ++i) {
    const int a = item0 + warp + i * kApWarps;
    const int st = i % kApSets;
    const uint32_t par = static_cast<uint32_t>(i / kApSets) & 1u;
    const uint8_t* kb = sets + st * kApSetBytes + lane * 32;
    const uint8_t* vb = kb + kApMaxP * 1024;
    uint4 qraw[kApMaxP][2];
#pragma unroll
    for (int qi = 0; qi < kApMaxP; ++qi) {
      if (qi < P) {
        const uint4* q4 = reinterpret_cast<const uint4*>(p.q + (static_cast<size_t>(a) * P + qi) * kE) + lane * 2;
        qraw[qi][0] = __ldg(q4); qraw[qi][1] = __ldg(q4 + 1);
      }
    }
    float pj[kApMaxP][kApMaxP], linv[kApMaxP];
    mbar_wait(&bars[st * 2], par, 5);
#pragma unroll
    for (int qi = 0; qi < kApMaxP; ++qi) {
      if (qi < P) {
        const int nkeys = p.prefix_bidir ? P : qi + 1;
        float qf[16];
        bf16x8_to_f32(qraw[qi][0], qf);
        bf16x8_to_f32(qraw[qi][1], qf + 8);
        float s[kApMaxP];
        float m = -INFINITY;
#pragma unroll
        for (int u = 0; u < kApMaxP; ++u) {
          s[u] = -INFINITY;
          if (u < nkeys) {
            const uint4* k4 = reinterpret_cast<const uint4*>(kb + u * 1024);
            float kf[16];
            bf16x8_to_f32(k4[0], kf);
            bf16x8_to_f32(k4[1], kf + 8);
            float d0 = 0.f, d1 = 0.f;
#pragma unroll
            for (int k = 0; k < 8; ++k) { d0 = fmaf(qf[k], kf[k], d0); d1 = fmaf(qf[8 + k], kf[8 + k], d1); }
            float t = (d0 + d1) * p.scale_log2e;
            t += __shfl_xor_sync(0xffffffffu, t, 1);
            t += __shfl_xor_sync(0xffffffffu, t, 2);
            s[u] = t;
            m = fmaxf(m, t);
          }
        }
        float l = 0.f;
#pragma unroll
        for (int u = 0; u < kApMaxP; ++u) { pj[qi][u] = exp2f(s[u] - m); l += pj[qi][u]; }
        linv[qi] = 1.0f / l;
      }
    }
    mbar_wait(&bars[st * 2 + 1], par, 5);
    float vf[kApMaxP][16];
#pragma unroll
    for (int u = 0; u < kApMaxP; ++u) {
      if (u < P) {
        const uint4* v4 = reinterpret_cast<const uint4*>(vb + u * 1024);
        bf16x8_to_f32(v4[0], vf[u]);
        bf16x8_to_f32(v4[1], vf[u] + 8);
      }
    }
    __syncwarp();                       // every lane has read the set: refill it with the sequence after next
    if (i + kApSets < nitems) request(i + kApSets);
#pragma unroll
    for (int qi = 0; qi < kApMaxP; ++qi) {
      if (qi < P) {
        float acc[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) acc[k] = 0.f;
#pragma unroll
        for (int u = 0; u < kApMaxP; ++u) {
          if (u < P) {
#pragma unroll
            for (int k = 0; k < 16; ++k) acc[k] = fmaf(pj[qi][u], vf[u][k], acc[k]);
          }
        }
        uint32_t o[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] = pack_bf16x2(acc[2 * k] * linv[qi], acc[2 * k + 1] * linv[qi]);
        uint4* d = reinterpret_cast<uint4*>(p.out + (static_cast<size_t>(a) * P + qi) * kE) + lane * 2;
        d[0] = make_uint4(o[0], o[1], o[2], o[3]);
        d[1] = make_uint4(o[4], o[5], o[6], o[7]);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// Merging the per-tile logits statistics of one row (executed by a full warp)
// ---------------------------------------------------------------------------------------------------------
struct RowStats {
  float max_all;   // natural-unit max over the vocabulary
  float lse_tau;   // log sum exp(x / tau)
  float lse_one;   // log sum exp(x)
  float sum_x;
  float best_val;
  int best_idx;
  float tgt_logit;
};

// masked = the partials come from the guided-decoding epilogue: the temperature sum has its own reference maximum (pad_)
__device__ __forceinline__ RowStats merge_partials(const LogitPartial* __restrict__ part, int ntiles, float inv_tau, bool masked = false) {
  const int lane = lane_id();
  float mx = -INFINITY, mxt = -INFINITY, best = -INFINITY, sum_x = 0.f, tgt = -INFINITY;
  int best_i = 0x7fffffff;
  for (int t = lane; t < ntiles; t += 32) {
    const LogitPartial q = part[t];
    mx = fmaxf(mx, q.max_all);
    mxt = fmaxf(mxt, masked ? __int_as_float(q.pad_) : q.max_all);
    sum_x += q.sum_x;
    tgt = fmaxf(tgt, q.tgt_logit);
    if (q.best_val > best || (q.best_val == best && q.best_idx < best_i)) { best = q.best_val; best_i = q.best_idx; }
  }
  mx = warp_max(mx);
  mxt = warp_max(mxt);
  float s_tau = 0.f, s_one = 0.f;
  for (int t = lane; t < ntiles; t += 32) {
    const LogitPartial q = part[t];
    s_one += q.sumexp_one * __expf(q.max_all - mx);
    const float mt = masked ? __int_as_float(q.pad_) : q.max_all;
    if (mt > -INFINITY) s_tau += q.sumexp_tau * __expf((mt - mxt) * inv_tau);
  }
  s_one = warp_sum(s_one);
  s_tau = warp_sum(s_tau);
  sum_x = warp_sum(sum_x);
  tgt = warp_max(tgt);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
    if (ov > best || (ov == best && oi < best_i)) { best = ov; best_i = oi; }
  }
  RowStats r;
  r.max_all = mx;
  r.lse_one = mx + __logf(s_one);
  r.lse_tau = mxt > -INFINITY ? mxt * inv_tau + __logf(s_tau) : -INFINITY;
  r.sum_x = sum_x;
  r.best_val = best;
  r.best_idx = best_i;
  r.tgt_logit = tgt;
  return r;
}

// ---------------------------------------------------------------------------------------------------------
// Guided decoding (embedding_decoder.py:802-813, :873-878, :915-920, :969-971).  The reference keeps a B x H x W
// mismatch mask over the W guide targets and scatters it into a B x H x (V+1) score tensor every step; here the guide
// targets are a token trie (novic_b200/guide.py) and every sequence carries one trie node id: the ids allowed next are
// the node's children.  guide_mask_kernel turns the node ids into one bit per (row, vocabulary id) for the logits
// epilogue; the selection kernels walk the trie with the chosen token.
// ---------------------------------------------------------------------------------------------------------
struct GuideTrie {
  const int* child_off;    // [num_nodes + 1] CSR offsets; node 0 = root (empty prefix)
  const int* child_tok;    // [num_edges] token id of each child edge, ascending within a node
  const int* child_node;   // [num_edges] node the edge leads to
  int num_nodes;
};

// node reached from `node` by `tok`, or -1 (no guide target continues that way)
__device__ __forceinline__ int guide_child(const GuideTrie& g, int node, int tok) {
  if (node < 0 || node >= g.num_nodes) return -1;
  int lo = g.child_off[node], hi = g.child_off[node + 1];
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    const int t = g.child_tok[mid];
    if (t == tok) return g.child_node[mid];
    if (t < tok) lo = mid + 1; else hi = mid;
  }
  return -1;
}

// allow[row, :] = bit set of the children tokens of node[row * node_stride].  One warp per row, bits assembled in shared memory.
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
guide_mask_kernel(GuideTrie g, const int* __restrict__ node, int node_stride, int rows, int words, uint32_t* __restrict__ allow,
                  int* __restrict__ edge0) {
  extern __shared__ uint32_t gm_smem[];
  pdl_trigger();
  pdl_wait();
  const int row = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = lane_id();
  uint32_t* bits = gm_smem + (threadIdx.x >> 5) * words;
  for (int i = lane; i < words; i += 32) bits[i] = 0u;
  __syncwarp();
  const int n = node[static_cast<size_t>(row) * node_stride];
  if (n >= 0 && n < g.num_nodes) {
    const int e0 = g.child_off[n], e1 = g.child_off[n + 1];
    for (int e = e0 + lane; e < e1; e += 32) {
      const int t = g.child_tok[e];
      atomicOr(&bits[t >> 5], 1u << (t & 31));
      // vocabulary prior: the logits epilogue finds an allowed id's edge as edge0[word] + (allowed ids below it in the word)
      if (edge0 != nullptr && (e == e0 || (g.child_tok[e - 1] >> 5) != (t >> 5))) edge0[static_cast<size_t>(row) * words + (t >> 5)] = e;
    }
  }
  __syncwarp();
  for (int i = lane; i < words; i += 32) allow[static_cast<size_t>(row) * words + i] = bits[i];
}

// Teacher-forced variant (generate_all with guide_renorm, embedding_decoder.py:1008-1018): sequence m is a given token
// row; the mask of position t holds the children of the node reached by its first t tokens.  One warp per sequence.
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
guide_path_mask_kernel(GuideTrie g, const long long* __restrict__ target, int ld_target, int M, int T, int words, uint32_t* __restrict__ allow) {
  extern __shared__ uint32_t gm_smem[];
  const int m = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (m >= M) return;
  const int lane = lane_id();
  uint32_t* bits = gm_smem + (threadIdx.x >> 5) * words;
  int n = 0;
  for (int t = 0; t < T; ++t) {
    for (int i = lane; i < words; i += 32) bits[i] = 0u;
    __syncwarp();
    if (n >= 0 && n < g.num_nodes) {
      const int e0 = g.child_off[n], e1 = g.child_off[n + 1];
      for (int e = e0 + lane; e < e1; e += 32) {
        const int tk = g.child_tok[e];
        atomicOr(&bits[tk >> 5], 1u << (tk & 31));
      }
    }
    __syncwarp();
    for (int i = lane; i < words; i += 32) allow[(static_cast<size_t>(m) * T + t) * words + i] = bits[i];
    __syncwarp();
    n = guide_child(g, n, static_cast<int>(target[static_cast<size_t>(m) * ld_target + t]));
  }
}

// score[a] = sum over the unpadded positions t of  logit[a, t, target] / tau - logsumexp(logits[a, t, support] / tau)
// (embedding_decoder.py:1067-1072).  One warp per sequence; target < 0 marks a padded position.
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
score_rows_kernel(const LogitPartial* __restrict__ part, int ntiles, int A, int T, float inv_tau, const long long* __restrict__ target,
                  int masked, float* __restrict__ score) {
  const int a = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (a >= A) return;
  float total = 0.f;
  for (int t = 0; t < T; ++t) {
    const size_t r = static_cast<size_t>(a) * T + t;
    if (target[r] < 0) continue;   // warp-uniform
    const RowStats st = merge_partials(part + r * ntiles, ntiles, inv_tau, masked != 0);
    total += st.tgt_logit * inv_tau - st.lse_tau;
  }
  if (lane_id() == 0) score[a] = total;
}

// ---------------------------------------------------------------------------------------------------------
// Greedy step (embedding_decoder.py:802-817): pick the arg-max token, update padding / done / score / loss
// accumulators and emit the next step's input row (token embedding + position + layer-0 LayerNorm).
// ---------------------------------------------------------------------------------------------------------
struct GreedyState {
  long long* tok;        // [B, G]
  unsigned char* pad;    // [B, G]
  unsigned char* done;   // [B]
  float* score;          // [B]  sum of log p_tau(token)
  float* nll;            // [B]  sum of -log p_1(token)  (+ label smoothing term)
  float* len;            // [B]  number of unpadded tokens
  int* alldone;          // [G + 1] per-step "every row finished" flags (host resets to 1)
};

// One CTA = 32 warps = the 32 consecutive rows of one block of the blocked fp32 layout of x: the warps stage their rows' values in a 64 KB
// shared-memory image of the block and the CTA writes it out as one contiguous run (the warp-per-row version wrote every row as 128
// scattered 16-byte pieces, half a sector each).
constexpr int kSelRows = 32;
constexpr int kSelSmemBytes = kSelRows * kE * 4;
__global__ void __launch_bounds__(kSelRows * 32, 1)
select_greedy_kernel(const LogitPartial* __restrict__ part, int ntiles, int B, int G, int step /*1-based*/, int V,
                     float inv_tau, float label_smoothing, GreedyState st, const float* __restrict__ wtok,
                     const float* __restrict__ pos_next, const float* __restrict__ gain0, float* __restrict__ x,
                     __nv_bfloat16* __restrict__ xn, float eps, GuideTrie guide, int* __restrict__ guide_node) {
  extern __shared__ __align__(16) uint8_t sel_smem[];
  float4* xs = reinterpret_cast<float4*>(sel_smem);
  // Wait BEFORE releasing the dependents: this kernel is the fence of a decode step.  Every other kernel releases its dependent at
  // entry, so with small grids a chain of prologues can run many launches ahead of the kernel that is actually executing; the
  // attention kernel's early K/V requests (rows written by earlier decode steps, issued before its own wait) are only safe because no
  // kernel of step t + 1 starts before this wait has passed, i.e. before every kernel of step t has completed.
  pdl_wait();
  pdl_trigger();
  const int b0 = blockIdx.x * kSelRows;
  const int b = b0 + (threadIdx.x >> 5);
  if (b < B) {
    const bool guided = guide_node != nullptr;
    const RowStats r = merge_partials(part + static_cast<size_t>(b) * ntiles, ntiles, inv_tau, guided);
    const bool was_done = st.done[b] != 0;
    const long long tok = r.best_idx < V ? r.best_idx : 0;   // no allowed id left: arg-max over all -inf = id 0 (the end token)
    if (guided && lane_id() == 0) guide_node[b] = guide_child(guide, guide_node[b], static_cast<int>(tok));
    if (lane_id() == 0) {
      st.pad[static_cast<size_t>(b) * G + (step - 1)] = was_done ? 1 : 0;
      st.tok[static_cast<size_t>(b) * G + (step - 1)] = was_done ? 0 : tok;
      if (!was_done) {
        st.score[b] += r.best_val * inv_tau - r.lse_tau;
        float nll = r.lse_one - r.best_val;
        if (label_smoothing != 0.f) nll = (1.f - label_smoothing) * nll + label_smoothing * (r.lse_one - r.sum_x / V);
        st.nll[b] += nll;
        st.len[b] += 1.f;
      }
      const bool now_done = was_done || tok == 0;
      st.done[b] = now_done ? 1 : 0;
      if (!now_done) st.alldone[step] = 0;
    }
    if (pos_next != nullptr) embed_token_row(wtok, pos_next, gain0, tok, b, x, xn, eps, xs);
  }
  if (pos_next == nullptr) return;
  __syncthreads();
  float4* dst = reinterpret_cast<float4*>(x + xblk_off(b0, 0));
#pragma unroll
  for (int i = 0; i < kSelRows * kE / 4 / (kSelRows * 32); ++i) {
    const int e = i * (kSelRows * 32) + threadIdx.x;     // float4 unit of the block: col4 = e / 32, row = e % 32
    const int col4 = e >> 5, r = e & 31;
    if (b0 + r < B) dst[e] = xs[col4 * 32 + (r ^ ((col4 >> 2) & 31))];
  }
}

// ---------------------------------------------------------------------------------------------------------
// Beam step (embedding_decoder.py:911-978; guide masks and the vocabulary prior are already folded into the top lists).  One warp per sample.  Every live
// candidate row contributes its per-tile top-HCAP logits (the H best continuations of a row are among the
// union of its tiles' H best); a finished candidate contributes exactly (its score, end token).  The H best
// totals are drawn in (score descending, flat index ascending) order.
// ---------------------------------------------------------------------------------------------------------
struct BeamState {
  const long long* tok_in;  long long* tok_out;          // [B, H, G]
  const unsigned char* pad_in; unsigned char* pad_out;   // [B, H, G]
  const unsigned char* anc_in; unsigned char* anc_out;   // [B, H, G]
  const float* score_in; float* score_out;               // [B, H] raw sum of log-probs
  float* score_norm_out;                                 // [B, H] length-normalised score of this step's ranking
  const float* len_in; float* len_out;                   // [B, H]
  const unsigned char* fin_in; unsigned char* fin_out;   // [B, H] candidate finished (its next position is padding)
  int* allfin;                                           // [G + 1]
  const int* node_in; int* node_out;                     // [B, H] guide trie node per candidate (nullptr = unguided)
};

template <int HCAP>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
select_beam_kernel(const LogitPartial* __restrict__ part, const float* __restrict__ topv, const int* __restrict__ topi,
                   int ntiles, int B, int H, int G, int step, int V, float inv_tau, float length_alpha, BeamState st,
                   const float* __restrict__ wtok, const float* __restrict__ pos_next, const float* __restrict__ gain0,
                   float* __restrict__ x, __nv_bfloat16* __restrict__ xn, float eps, GuideTrie guide) {
  pdl_trigger();
  pdl_wait();
  const int b = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (b >= B) return;
  const int lane = lane_id();
  const bool guided = st.node_in != nullptr;
  const int nrows = (step == 1) ? 1 : H;                 // logits rows available for this sample
  const size_t row0 = (step == 1) ? static_cast<size_t>(b) : static_cast<size_t>(b) * H;
  __shared__ float s_lse[kWarpsPerBlock][16], s_base[kWarpsPerBlock][16], s_scale[kWarpsPerBlock][16];
  __shared__ unsigned char s_fin[kWarpsPerBlock][16];
  float* lse = s_lse[threadIdx.x >> 5];
  float* base = s_base[threadIdx.x >> 5];
  float* scale = s_scale[threadIdx.x >> 5];
  unsigned char* fin = s_fin[threadIdx.x >> 5];
  for (int h = 0; h < H; ++h) {
    float l = 0.f;
    if (h < nrows) {
      const RowStats r = merge_partials(part + (row0 + h) * ntiles, ntiles, inv_tau, guided);
      l = r.lse_tau;
    }
    if (lane == 0) {
      lse[h] = l;
      base[h] = st.score_in[static_cast<size_t>(b) * H + h];
      fin[h] = st.fin_in[static_cast<size_t>(b) * H + h];
      scale[h] = (length_alpha != 0.f) ? __powf(fmaxf(st.len_in[static_cast<size_t>(b) * H + h], 1.f), -length_alpha) : 1.f;
    }
  }
  __syncwarp();
  const int per_row = ntiles * HCAP;
  // Candidate lists: one per (live row h, 64-column slice), sorted, ending at the first unused slot.  The k-th best total is always
  // the head of some list once the k-1 better ones have been popped, so the H winners are drawn by a tournament over the list heads:
  // every lane owns the lists L = h * ntiles + slice with L % 32 == lane and caches their heads; per winner one warp arg-max and one
  // pop.  (The first version rescanned all H * ntiles * HCAP entries for every winner: 10 x 17 280 entries per sample at H = 10.)
  constexpr int kSelMaxLists = 64;                         // lists per lane the tournament can hold: H * ntiles <= 2048
  const int nlists = H * ntiles;
  const bool tournament = nlists <= 32 * kSelMaxLists;
  float lraw[kSelMaxLists];
  int lidx[kSelMaxLists];
  unsigned char lpos[kSelMaxLists], lh[kSelMaxLists];
  int nmine = 0;
  unsigned fin_avail = 0;                                  // lane 0: finished / not yet existing rows, one end-token candidate each
  if (tournament) {
    for (int L = lane; L < nlists; L += 32) {
      const int h = L / ntiles, sl = L - h * ntiles;
      lpos[nmine] = 0; lh[nmine] = static_cast<unsigned char>(h); lidx[nmine] = -1; lraw[nmine] = -INFINITY;
      if (!(fin[h] || h >= nrows)) {
        const size_t e = (row0 + h) * per_row + static_cast<size_t>(sl) * HCAP;
        const int idx = topi[e];
        if (idx < V) { lidx[nmine] = idx; lraw[nmine] = base[h] + (topv[e] * inv_tau - lse[h]); }
      }
      ++nmine;
    }
    for (int h = 0; h < H; ++h) if (fin[h] || h >= nrows) fin_avail |= 1u << h;
  }
  float prev_v = INFINITY;
  long long prev_f = -1;
  for (int k = 0; k < H; ++k) {
    float bv = -INFINITY, braw = -INFINITY;
    long long bf = 0x7fffffffffffffffLL;
    if (tournament) {
      int bm = -1;
      for (int m = 0; m < nmine; ++m) {
        if (lidx[m] < 0) continue;
        const int h = lh[m];
        const float raw = lraw[m];
        const float v = (length_alpha != 0.f) ? raw * scale[h] : raw;
        const long long f = static_cast<long long>(h) * V + lidx[m];
        if (v > bv || (v == bv && f < bf)) { bv = v; bf = f; braw = raw; bm = m; }
      }
      if (lane == 0) {
        for (int h = 0; h < H; ++h) {
          if (!((fin_avail >> h) & 1u)) continue;
          const float raw = base[h];
          const float v = (length_alpha != 0.f) ? raw * scale[h] : raw;
          const long long f = static_cast<long long>(h) * V;
          if (v > bv || (v == bv && f < bf)) { bv = v; bf = f; braw = raw; bm = kSelMaxLists + h; }
        }
      }
      int owner = lane;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const float oraw = __shfl_xor_sync(0xffffffffu, braw, o);
        const long long of = __shfl_xor_sync(0xffffffffu, bf, o);
        const int oo = __shfl_xor_sync(0xffffffffu, owner, o);
        if (ov > bv || (ov == bv && of < bf)) { bv = ov; bf = of; braw = oraw; owner = oo; }
      }
      if (lane == owner && bm >= 0 && bf != 0x7fffffffffffffffLL) {   // pop the winner from its list
        if (bm >= kSelMaxLists) {
          fin_avail &= ~(1u << (bm - kSelMaxLists));
        } else {
          const int h = lh[bm], L = lane + 32 * bm, sl = L - h * ntiles;
          const int pos = ++lpos[bm];
          lidx[bm] = -1;
          if (pos < HCAP) {
            const size_t e = (row0 + h) * per_row + static_cast<size_t>(sl) * HCAP + pos;
            const int idx = topi[e];
            if (idx < V) { lidx[bm] = idx; lraw[bm] = base[h] + (topv[e] * inv_tau - lse[h]); }
          }
        }
      }
    } else {
    for (int h = 0; h < H; ++h) {
      if (fin[h] || h >= nrows) {
        // finished (or not yet existing) candidate: single continuation = end token at zero cost
        if (lane == 0) {
          const float raw = base[h];
          const float v = (length_alpha != 0.f) ? raw * scale[h] : raw;
          const long long f = static_cast<long long>(h) * V;
          const bool after_prev = (v < prev_v) || (v == prev_v && f > prev_f);
          if (after_prev && (v > bv || (v == bv && f < bf))) { bv = v; bf = f; braw = raw; }
        }
        continue;
      }
      const float* tvp = topv + (row0 + h) * per_row;
      const int* tip = topi + (row0 + h) * per_row;
      // one lane per 64-column slice; a slice's list is sorted and ends at its first unused slot (index >= V)
      for (int sl = lane; sl < ntiles; sl += 32) {
        const int4* ti4 = reinterpret_cast<const int4*>(tip + sl * HCAP);
        const float4* tv4 = reinterpret_cast<const float4*>(tvp + sl * HCAP);
        bool more = true;
#pragma unroll 1
        for (int q = 0; q < HCAP / 4 && more; ++q) {
          const int4 i4 = ti4[q];
          if (i4.x >= V) break;
          const float4 v4 = tv4[q];
          const int idx[4] = {i4.x, i4.y, i4.z, i4.w};
          const float val[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (idx[j] >= V) { more = false; break; }
            const float raw = base[h] + (val[j] * inv_tau - lse[h]);
            const float v = (length_alpha != 0.f) ? raw * scale[h] : raw;
            const long long f = static_cast<long long>(h) * V + idx[j];
            const bool after_prev = (v < prev_v) || (v == prev_v && f > prev_f);
            if (after_prev && (v > bv || (v == bv && f < bf))) { bv = v; bf = f; braw = raw; }
          }
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const float oraw = __shfl_xor_sync(0xffffffffu, braw, o);
      const long long of = __shfl_xor_sync(0xffffffffu, bf, o);
      if (ov > bv || (ov == bv && of < bf)) { bv = ov; bf = of; braw = oraw; }
    }
    }
    prev_v = bv;
    prev_f = bf;
    const bool dead = bf == 0x7fffffffffffffffLL;          // fewer than H continuations exist (tiny guide sets): a -inf, finished filler
    if (dead) { bf = 0; bv = -INFINITY; braw = -INFINITY; }
    const int parent = static_cast<int>(bf / V);
    const long long tok = bf - static_cast<long long>(parent) * V;
    const size_t o = static_cast<size_t>(b) * H + k;
    const size_t pi = static_cast<size_t>(b) * H + parent;
    const bool parent_fin = fin[parent] != 0 || dead;
    const bool nxt_fin = parent_fin || tok == 0;
    if (guided && lane == 0) st.node_out[o] = parent_fin ? st.node_in[pi] : guide_child(guide, st.node_in[pi], static_cast<int>(tok));
    // history: columns [0, step-1) come from the parent, column step-1 is the new token
    for (int j = lane; j < G; j += 32) {
      long long t = 0;
      unsigned char pd = 1, an = 0;
      if (j < step - 1) {
        t = st.tok_in[pi * G + j];
        pd = st.pad_in[pi * G + j];
        an = st.anc_in[pi * G + j];
      } else if (j == step - 1) {
        t = tok;
        pd = parent_fin ? 1 : 0;
      } else if (j == step) {
        pd = nxt_fin ? 1 : 0;
      }
      if (step >= 2 && j == step - 2) an = static_cast<unsigned char>(parent);
      st.tok_out[o * G + j] = pd ? 0 : t;
      st.pad_out[o * G + j] = pd;
      st.anc_out[o * G + j] = an;
    }
    if (lane == 0) {
      st.score_out[o] = braw;
      st.score_norm_out[o] = bv;
      st.len_out[o] = st.len_in[pi] + (nxt_fin ? 0.f : 1.f);
      st.fin_out[o] = nxt_fin ? 1 : 0;
      if (!nxt_fin) st.allfin[step] = 0;
    }
    if (pos_next != nullptr) embed_token_row(wtok, pos_next, gain0, tok, static_cast<int>(o), x, xn, eps);
  }
}

__global__ void beam_init_kernel(int B, int H, int G, long long* tok, unsigned char* pad, unsigned char* anc, float* score,
                                 float* len, unsigned char* fin, int* node) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * H) return;
  const int h = i % H;
  for (int j = 0; j < G; ++j) {
    tok[static_cast<size_t>(i) * G + j] = 0;
    pad[static_cast<size_t>(i) * G + j] = (h == 0 && j == 0) ? 0 : 1;   // embedding_decoder.py:861-862
    anc[static_cast<size_t>(i) * G + j] = 0;
  }
  score[i] = (h == 0) ? 0.f : -INFINITY;                                // :863-864
  len[i] = (h == 0) ? 1.f : 0.f;                                        // :898-899
  fin[i] = (h == 0) ? 0 : 1;
  node[i] = 0;                                                          // every candidate starts at the guide trie's root
}

// score * clamp(len, 1)^-alpha (embedding_decoder.py:836)
__global__ void greedy_finalize_kernel(int B, float length_alpha, const float* __restrict__ score_sum,
                                       const float* __restrict__ len, float* __restrict__ score_out) {
  pdl_trigger();
  pdl_wait();
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float s = score_sum[b];
  if (length_alpha != 0.f) s *= __powf(fmaxf(len[b], 1.f), -length_alpha);
  score_out[b] = s;
}

// ---------------------------------------------------------------------------------------------------------
// Teacher-forced loss / correctness per target position (embedding_decoder.py:729-761)
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
loss_rows_kernel(const LogitPartial* __restrict__ part, int ntiles, int nrows, int V, float label_smoothing,
                 const long long* __restrict__ target /*-1 = ignored*/, float* __restrict__ nll_out,
                 unsigned char* __restrict__ correct_out) {
  const int r = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (r >= nrows) return;
  const RowStats s = merge_partials(part + static_cast<size_t>(r) * ntiles, ntiles, 1.0f);
  if (lane_id() == 0) {
    const long long t = target[r];
    float nll = 0.f;
    if (t >= 0) {
      nll = s.lse_one - s.tgt_logit;
      if (label_smoothing != 0.f) nll = (1.f - label_smoothing) * nll + label_smoothing * (s.lse_one - s.sum_x / V);
    }
    nll_out[r] = nll;
    // guided evaluation with no allowed id left: the reference's arg-max over an all -inf row is id 0 (embedding_decoder.py:760)
    const long long pred = s.best_idx == 0x7fffffff ? 0 : s.best_idx;
    if (correct_out != nullptr) correct_out[r] = (t >= 0 && pred == t) ? 1 : 0;
  }
}

// Deterministic single-block reduction: loss_sum = sum_a w_a * sum_t nll[a, t]; basis = sum_a w_a * n_valid_a
__global__ void __launch_bounds__(1024)
loss_reduce_kernel(const float* __restrict__ nll, const long long* __restrict__ target, const float* __restrict__ weight,
                   int nseq, int C, float* __restrict__ out /*[2]*/) {
  __shared__ double s_loss[32], s_basis[32];
  double loss = 0.0, basis = 0.0;
  for (int a = threadIdx.x; a < nseq; a += blockDim.x) {
    float l = 0.f;
    int n = 0;
    for (int t = 0; t < C; ++t) {
      l += nll[static_cast<size_t>(a) * C + t];
      n += target[static_cast<size_t>(a) * C + t] >= 0;
    }
    const float w = weight != nullptr ? weight[a] : 1.f;
    loss += static_cast<double>(w) * l;
    basis += static_cast<double>(w) * n;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    loss += __shfl_xor_sync(0xffffffffu, loss, o);
    basis += __shfl_xor_sync(0xffffffffu, basis, o);
  }
  if (lane_id() == 0) { s_loss[threadIdx.x >> 5] = loss; s_basis[threadIdx.x >> 5] = basis; }
  __syncthreads();
  if (threadIdx.x < 32) {
    loss = threadIdx.x < (blockDim.x >> 5) ? s_loss[threadIdx.x] : 0.0;
    basis = threadIdx.x < (blockDim.x >> 5) ? s_basis[threadIdx.x] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      loss += __shfl_xor_sync(0xffffffffu, loss, o);
      basis += __shfl_xor_sync(0xffffffffu, basis, o);
    }
    if (threadIdx.x == 0) { out[0] = static_cast<float>(loss); out[1] = static_cast<float>(basis); }
  }
}

// Deterministic single-block reduction of two per-sample vectors (the tail of generate(), embedding_decoder.py:838-846):
// out_f[0] = sum_b w_b * a_b, out_f[1] = sum_b w_b * b_b (w = 1 without weights); out_i[0] = round(out_f[1]) as int64.
__global__ void __launch_bounds__(1024)
pair_reduce_kernel(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ weight, long long n,
                   float* __restrict__ out_f /*[2]*/, long long* __restrict__ out_i /*[1] or nullptr*/) {
  __shared__ double s_a[32], s_b[32];
  double sa = 0.0, sb = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) {
    const double w = weight != nullptr ? static_cast<double>(weight[i]) : 1.0;
    sa += w * a[i];
    sb += w * b[i];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sa += __shfl_xor_sync(0xffffffffu, sa, o);
    sb += __shfl_xor_sync(0xffffffffu, sb, o);
  }
  if (lane_id() == 0) { s_a[threadIdx.x >> 5] = sa; s_b[threadIdx.x >> 5] = sb; }
  __syncthreads();
  if (threadIdx.x < 32) {
    sa = threadIdx.x < (blockDim.x >> 5) ? s_a[threadIdx.x] : 0.0;
    sb = threadIdx.x < (blockDim.x >> 5) ? s_b[threadIdx.x] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      sa += __shfl_xor_sync(0xffffffffu, sa, o);
      sb += __shfl_xor_sync(0xffffffffu, sb, o);
    }
    if (threadIdx.x == 0) {
      out_f[0] = static_cast<float>(sa);
      out_f[1] = static_cast<float>(sb);
      if (out_i != nullptr) out_i[0] = llrint(sb);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// Embedding noise (embedding_noise.py), fused draw + perturb + renormalise, in place.  Warp per row.
// With `pre` pointers given the random draws are read instead of generated (deterministic parity mode).
// ---------------------------------------------------------------------------------------------------------
enum NoiseScheme : int { kGaussElem = 0, kGaussVec = 1, kGaussAngle = 2, kUniformAngle = 3, kGaussElemUniformAngle = 4 };

struct NoiseParams {
  int scheme, F;
  float vec_norm, angle_min_rad, angle_max_rad, angle_std_rad, mix_ratio;
  const float* pre_normals_a;  // [B, F] direction normals (angle schemes) or element normals (Gauss schemes)
  const float* pre_normals_b;  // [B, F] element normals of the mix scheme's Gaussian branch
  const float* pre_row_a;      // [B] angle draw (uniform [0,1) or standard normal) / GaussVec scalar normal
  const float* pre_row_b;      // [B] mix uniform
};

template <int MAXF_PER_LANE>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
noise_kernel(float* __restrict__ embed, int B, NoiseParams p, unsigned long long seed, unsigned long long offset) {
  const int row = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (row >= B) return;
  const int lane = lane_id();
  const int F = p.F;
  const int per = F / 32;  // host guarantees F % 128 == 0 and per <= MAXF_PER_LANE
  float* e = embed + static_cast<size_t>(row) * F;
  const bool pre = p.pre_normals_a != nullptr;

  curandStatePhilox4_32_10_t rng;
  if (!pre) curand_init(seed, static_cast<unsigned long long>(row) * 32 + lane, offset, &rng);

  float row_a = 0.f, row_b = 0.f;
  if (pre) {
    row_a = p.pre_row_a != nullptr ? p.pre_row_a[row] : 0.f;
    row_b = p.pre_row_b != nullptr ? p.pre_row_b[row] : 0.f;
  } else {
    // per-row scalars are drawn by lane 0 and broadcast
    float ua = 0.f, ub = 0.f;
    if (lane == 0) {
      const float4 n = curand_normal4(&rng);
      const float4 u = curand_uniform4(&rng);
      ua = (p.scheme == kGaussAngle || p.scheme == kGaussVec) ? n.x : (1.0f - u.x);  // curand uniform is (0,1]
      ub = 1.0f - u.y;
    } else {
      (void)curand_normal4(&rng);
      (void)curand_uniform4(&rng);
    }
    row_a = __shfl_sync(0xffffffffu, ua, 0);
    row_b = __shfl_sync(0xffffffffu, ub, 0);
  }
  const bool angle_branch = p.scheme == kGaussAngle || p.scheme == kUniformAngle ||
                            (p.scheme == kGaussElemUniformAngle && row_b < p.mix_ratio);

  float ev[MAXF_PER_LANE], nv[MAXF_PER_LANE];
#pragma unroll
  for (int i = 0; i < MAXF_PER_LANE; i += 4) {
    if (i < per) {
      const int col = (i / 4) * 128 + lane * 4;
      const float4 v = *reinterpret_cast<const float4*>(e + col);
      ev[i] = v.x; ev[i + 1] = v.y; ev[i + 2] = v.z; ev[i + 3] = v.w;
      float4 n;
      if (pre) {
        const float* src = (p.scheme == kGaussElemUniformAngle && !angle_branch) ? p.pre_normals_b : p.pre_normals_a;
        n = *reinterpret_cast<const float4*>(src + static_cast<size_t>(row) * F + col);
      } else {
        n = curand_normal4(&rng);
      }
      nv[i] = n.x; nv[i + 1] = n.y; nv[i + 2] = n.z; nv[i + 3] = n.w;
    }
  }
  float outv[MAXF_PER_LANE];
  if (angle_branch) {
    // d = unit(n - e (e.n)); e' = unit(e cos(a) + d sin(a))       (embedding_noise.py:105-112)
    float dot = 0.f;
#pragma unroll
    for (int i = 0; i < MAXF_PER_LANE; ++i) if (i < per) dot = fmaf(ev[i], nv[i], dot);
    dot = warp_sum(dot);
    float dd = 0.f;
#pragma unroll
    for (int i = 0; i < MAXF_PER_LANE; ++i) if (i < per) { nv[i] = fmaf(-ev[i], dot, nv[i]); dd = fmaf(nv[i], nv[i], dd); }
    dd = warp_sum(dd);
    const float dinv = 1.0f / fmaxf(sqrtf(dd), 1e-12f);
    float ang;
    if (p.scheme == kGaussAngle) ang = fminf(fmaxf(row_a * p.angle_std_rad, -p.angle_max_rad), p.angle_max_rad);
    else ang = p.angle_min_rad + (p.angle_max_rad - p.angle_min_rad) * row_a;
    float sn, cs;
    sincosf(ang, &sn, &cs);
#pragma unroll
    for (int i = 0; i < MAXF_PER_LANE; ++i) if (i < per) outv[i] = ev[i] * cs + nv[i] * dinv * sn;
  } else if (p.scheme == kGaussVec) {
    // e' = unit(e + vec_norm * g * unit(n))                         (embedding_noise.py:90-95)
    float nn = 0.f;
#pragma unroll
    for (int i = 0; i < MAXF_PER_LANE; ++i) if (i < per) nn = fmaf(nv[i], nv[i], nn);
    nn = warp_sum(nn);
    const float k = p.vec_norm * row_a / fmaxf(sqrtf(nn), 1e-12f);
#pragma unroll
    for (int i = 0; i < MAXF_PER_LANE; ++i) if (i < per) outv[i] = fmaf(k, nv[i], ev[i]);
  } else {
    // e' = unit(e + (vec_norm / sqrt(F)) * n)                       (embedding_noise.py:72-75)
    const float sigma = p.vec_norm * rsqrtf(static_cast<float>(F));
#pragma unroll
    for (int i = 0; i < MAXF_PER_LANE; ++i) if (i < per) outv[i] = fmaf(sigma, nv[i], ev[i]);
  }
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < MAXF_PER_LANE; ++i) if (i < per) ss = fmaf(outv[i], outv[i], ss);
  ss = warp_sum(ss);
  const float inv = 1.0f / fmaxf(sqrtf(ss), 1e-12f);
#pragma unroll
  for (int i = 0; i < MAXF_PER_LANE; i += 4) {
    if (i < per) {
      const int col = (i / 4) * 128 + lane * 4;
      *reinterpret_cast<float4*>(e + col) = make_float4(outv[i] * inv, outv[i + 1] * inv, outv[i + 2] * inv, outv[i + 3] * inv);
    }
  }
}

}  // namespace novic
