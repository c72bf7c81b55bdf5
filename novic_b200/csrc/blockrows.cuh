// Row-owner block kernel (decode path, inference): attention output -> next layer's LayerNorm rows, one CTA per 32 residual rows,
// no cluster.  Same arithmetic as outproj_ffn_kernel (embedding_decoder.py:1313-1322 = nn.TransformerEncoderLayer, norm_first):
//   r = x + ao * Wo^T;  y = LN2(r);  h = gelu(y * W1^T);  r += h * W2^T;  x = r;  xn = LN_next(r)
// but with the operands SWAPPED: the weights are the M = 128 operand of tcgen05.mma (128 output features per tile on the 128 TMEM
// lanes), the CTA's 32 rows are the N = 32 operand and stay resident in shared memory (32 KB), and the whole 768 KB of Wo / W1 / W2
// streams past them through a ring of three 64 KB slots (one TMA request each - the request size the L2 -> SM path delivers fastest,
// tools/tmabench.cu).  Every CTA owns whole rows, so the two LayerNorms need no exchange between CTAs: the cluster kernels spend 10 k of
// their 30 k cycles handing LN2 rows and hidden columns over DSMEM and another 3 k in cluster barriers.
//
// Feature permutation: tile t of Wo / W2 holds weight rows {4 i + t, i = 0..127} (a 4-D tensor map with the row index split into
// (i, t)), so the thread that reads TMEM lane i owns features 4 i .. 4 i + 3 after the four tiles - one float4 of the 32-row blocked
// residual layout per row, 8 contiguous bytes of the K-major LN2 operand and 8 contiguous bytes of the row-major xn row (a warp writes one
// 256-byte run per row and store).  No shuffles, no staging transposes.  The fp32 x tile leaves through one TMA tensor store.
//
// Warps: 0 = TMA producer, 1 = TMEM allocator + MMA issuer, 2..17 = epilogue (warp & 3 = TMEM lane quadrant, (warp - 2) >> 2 = which 8
// of the 32 rows).  TMEM columns: [0,128) out-proj (4 tiles x 32 rows), [128,160) hidden, [160,288) FFN2.
#pragma once

#include "gemm.cuh"
#include "kernels.cuh"

namespace novic {

constexpr int kBrRows = 32;                         // residual rows per CTA = UMMA N
constexpr int kBrSlotBytes = 64 * 1024;             // one weight request: 4 k-blocks of a 128-row tile (or 2 k-blocks of two tiles)
constexpr int kBrSlots = 3;
constexpr int kBrActBytes = kBrRows * kE * 2;       // resident operand: attention rows, then LN2 rows, then hidden rows, then the xn staging tile
constexpr int kBrKbBytes = kBrRows * kBlockK * 2;   // one k-block of the resident operand: 32 rows x 128 B
constexpr int kBrEpiWarps = 16;
constexpr int kBrThreads = 64 + 32 * kBrEpiWarps;   // 576
constexpr int kBrRequests = 12;                     // 8 x Wo, 2 x W1, 2 x W2
constexpr int kBrStatsBytes = kBrRows * 4 * 8;      // [row][quadrant] (sum, sum of squares)
constexpr int kBrBarBytes = 512;                    // pipeline barriers (the first 256 B are used)
__host__ __device__ constexpr int block_rows_smem_bytes() {
  return 1024 /*align*/ + kBrSlots * kBrSlotBytes + kBrActBytes + kBrBarBytes /*barriers*/ + kBrStatsBytes;
}
static_assert(block_rows_smem_bytes() <= 227 * 1024, "row-owner block kernel does not fit in shared memory");

// 4-D tiled load (c0 innermost)
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int32_t c0, int32_t c1, int32_t c2, int32_t c3,
                                            uint64_t cache_hint) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4, %5, %6}], [%2], %7;\n" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "l"(cache_hint)
      : "memory");
}

// TMEM -> registers: this warp's 32 lanes x 8 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld_32x8(uint32_t taddr, float (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
               : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
               : "r"(taddr)
               : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
}

// tcgen05.mma with both shared-memory descriptors given by their low words (start address >> 4; the high word - stride byte offset,
// version, 128-byte swizzle - is the same constant for every K-major SW128 operand): one 32-bit add per operand and MMA on the issuing
// thread.  With 64-bit descriptor arithmetic the single issuing thread needs 58-60 cycles per MMA, with precomputed descriptors 46
// (tools/ummabench.cu) - for N <= 64 that, not the tensor pipe, sets the MMA rate.
constexpr uint32_t kDescHiSw128 = (1024u >> 4) | (1u << 14) | (2u << 29);
template <bool ACC>
__device__ __forceinline__ void umma_lo(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 da, {%1, %3};\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t}\n" ::"r"(tmem_d),
      "r"(a_lo), "r"(b_lo), "r"(kDescHiSw128), "r"(idesc), "n"(ACC ? 1 : 0)
      : "memory");
}

// 256-bit global accesses (sm_100): two neighbouring rows of the blocked residual layout x 4 features = one full 32-byte sector
__device__ __forceinline__ void ld_global_v8(const float* p, float (&v)[8]) {
  asm volatile("ld.global.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
               : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
               : "l"(p));
}
__device__ __forceinline__ void st_global_v8(float* p, const float (&v)[8]) {
  asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};\n" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]),
               "f"(v[5]), "f"(v[6]), "f"(v[7])
               : "memory");
}

// Tiled store shared -> global (bulk async-group completion): the x tile leaves through the TMA unit instead of 64 KB of scattered per-thread stores
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, const void* smem_src, int32_t c0, int32_t c1, int32_t c2, int32_t c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];\n" ::"l"(reinterpret_cast<uint64_t>(map)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_group_read0() { asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory"); }

// named barrier over the 16 epilogue warps
__device__ __forceinline__ void br_epi_sync() { asm volatile("bar.sync 1, %0;\n" ::"n"(kBrEpiWarps * 32) : "memory"); }

// Sum 16 per-thread values over the 32 lanes of the warp in 16 shuffles (halving butterfly, fixed order): afterwards lanes 2 k and 2 k + 1
// both hold the warp total of val[k].
__device__ __forceinline__ float br_warp_reduce16(float (&val)[16], int lane) {
#pragma unroll
  for (int o = 16, n = 16; o >= 2; o >>= 1, n >>= 1) {
    const bool upper = (lane & o) != 0;
#pragma unroll
    for (int k = 0; k < n / 2; ++k) {
      const float send = upper ? val[k] : val[k + n / 2];
      const float keep = upper ? val[k + n / 2] : val[k];
      val[k] = keep + __shfl_xor_sync(0xffffffffu, send, o);
    }
  }
  return val[0] + __shfl_xor_sync(0xffffffffu, val[0], 1);
}


__global__ void __launch_bounds__(kBrThreads, 1)
block_rows_kernel(const __grid_constant__ CUtensorMap tmap_ao, const __grid_constant__ CUtensorMap tmap_wo, const __grid_constant__ CUtensorMap tmap_w1,
                  const __grid_constant__ CUtensorMap tmap_w2, const __grid_constant__ CUtensorMap tmap_x, int M,
                  FusedBlockParams ep) {
  constexpr uint32_t kIdesc = umma_idesc_bf16_f32(128, kBrRows);
  constexpr uint32_t kColHidden = 128, kColFfn2 = 160;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* ring = smem;
  uint8_t* act = ring + kBrSlots * kBrSlotBytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(act + kBrActBytes);   // [3]
  uint64_t* empty_bar = full_bar + kBrSlots;                            // [3]
  uint64_t* act_full = empty_bar + kBrSlots;
  uint64_t* acc0_full = act_full + 1;                                   // [4] out-proj tile t accumulated
  uint64_t* ln2_ready = acc0_full + 4;                                  // LN2 rows are in the resident operand (16 warp arrivals)
  uint64_t* acc1_full = ln2_ready + 1;
  uint64_t* h_ready = acc1_full + 1;                                    // hidden rows are in the resident operand
  uint64_t* acc2_full = h_ready + 1;                                    // [4]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc2_full + 4);
  static_assert((2 * kBrSlots + 1 + 4 + 3 + 4) * 8 + 4 <= 256, "barrier area");
  float2* s_stats = reinterpret_cast<float2*>(act + kBrActBytes + kBrBarBytes);  // [32 rows][4 quadrants]

  const int warp = threadIdx.x >> 5;
  const int lane = static_cast<int>(lane_id());
  const int m0 = blockIdx.x * kBrRows;
  __shared__ int s_trace;
  pdl_trigger();
  if (threadIdx.x == 0) { s_trace = trace_begin() ? 1 : 0; trace_point(s_trace != 0, 0); }

  // request i of the weight stream: 0..7 = Wo tile i / 2, k-blocks 4 (i & 1) .. + 3;  8, 9 = W1 k-blocks 0..3 / 4..7;  10, 11 = W2 tiles 0, 1 / 2, 3
  auto issue = [&](int i) {
    const int slot = i % kBrSlots;
    mbar_arrive_expect_tx(&full_bar[slot], kBrSlotBytes);
    uint8_t* dst = ring + slot * kBrSlotBytes;
    if (i < 8) tma_load_4d(dst, &tmap_wo, &full_bar[slot], 0, 0, i >> 1, (i & 1) * 4, kEvictLast);
    else if (i < 10) tma_load_3d(dst, &tmap_w1, &full_bar[slot], 0, (i - 8) * 4, kEvictLast);
    else tma_load_4d(dst, &tmap_w2, &full_bar[slot], 0, 0, (i - 10) * 2, 0, kEvictLast);
  };

  if (warp == 0) {
    if (elect_one()) {
      tma_prefetch_desc(&tmap_ao);
      tma_prefetch_desc(&tmap_wo); tma_prefetch_desc(&tmap_w1); tma_prefetch_desc(&tmap_w2);
      tma_prefetch_desc(&tmap_x);
      for (int st = 0; st < kBrSlots; ++st) { mbar_init(&full_bar[st], 1); mbar_init(&empty_bar[st], 1); }
      mbar_init(act_full, 1);
      for (int t = 0; t < 4; ++t) { mbar_init(&acc0_full[t], 1); mbar_init(&acc2_full[t], 1); }
      mbar_init(ln2_ready, kBrEpiWarps); mbar_init(acc1_full, 1); mbar_init(h_ready, kBrEpiWarps);
      fence_mbar_init();
      for (int i = 0; i < kBrSlots; ++i) issue(i);          // the weights do not depend on the previous kernel
      pdl_wait();
      mbar_arrive_expect_tx(act_full, kBrActBytes);
      tma_load_3d(act, &tmap_ao, act_full, m0, 0, kEvictFirst);
    }
  } else if (warp == 1) {
    tmem_alloc<512>(tmem_slot);
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  // phase trace: the buffer pointer is read once here (a trace_point() per phase would stall its thread for an L2 round trip each time)
  long long* const trp = (s_trace != 0 && (threadIdx.x == 64 || threadIdx.x == 32)) ? g_trace : nullptr;
  auto tp = [&](int idx) { if (trp != nullptr) trp[idx] = clock64(); };

  if (warp == 0) {
    if (elect_one()) {
      for (int i = kBrSlots; i < kBrRequests; ++i) {
        mbar_wait(&empty_bar[i % kBrSlots], ((i / kBrSlots) - 1) & 1, 1);
        issue(i);
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      // descriptors differ only in their 14-bit start-address field: low words = address >> 4, offsets added as constants
      const uint32_t lb = (smem_u32(act) & 0x3FFFFu) >> 4;
      auto lo = [](const void* p) { return (smem_u32(p) & 0x3FFFFu) >> 4; };
      constexpr uint32_t kKs = (kUmmaK * 2) >> 4, kAo = kABytes >> 4, kBo = kBrKbBytes >> 4;
      mbar_wait(act_full, 0, 2);
      tp(22);
      // ---- out-proj: tile t (features 4 i + t) = requests 2 t, 2 t + 1
      for (int i = 0; i < 8; ++i) {
        const int slot = i % kBrSlots;
        mbar_wait(&full_bar[slot], (i / kBrSlots) & 1, 3);
        tp(10 + i);
        tc_fence_after_sync();
        const uint32_t la = lo(ring + slot * kBrSlotBytes);
        const uint32_t lbi = lb + (i & 1) * 4 * kBo;
        const uint32_t d = tmem_base + (i >> 1) * kBrRows;
        if (i & 1) {
#pragma unroll
          for (int q = 0; q < 16; ++q) umma_lo<true>(d, la + (q >> 2) * kAo + (q & 3) * kKs, lbi + (q >> 2) * kBo + (q & 3) * kKs, kIdesc);
        } else {
          umma_lo<false>(d, la, lbi, kIdesc);
#pragma unroll
          for (int q = 1; q < 16; ++q) umma_lo<true>(d, la + (q >> 2) * kAo + (q & 3) * kKs, lbi + (q >> 2) * kBo + (q & 3) * kKs, kIdesc);
        }
        umma_commit(&empty_bar[slot]);
        if (i & 1) umma_commit(&acc0_full[i >> 1]);
      }
      // ---- FFN1: hidden (128 features, natural order) x 32 rows
      mbar_wait(ln2_ready, 0, 4);
      tp(23);
      tc_fence_after_sync();
      for (int i = 8; i < 10; ++i) {
        const int slot = i % kBrSlots;
        mbar_wait(&full_bar[slot], (i / kBrSlots) & 1, 5);
        tp(10 + i);
        tc_fence_after_sync();
        const uint32_t la = lo(ring + slot * kBrSlotBytes);
        const uint32_t lbi = lb + (i - 8) * 4 * kBo;
        const uint32_t d = tmem_base + kColHidden;
        if (i == 8) {
          umma_lo<false>(d, la, lbi, kIdesc);
#pragma unroll
          for (int q = 1; q < 16; ++q) umma_lo<true>(d, la + (q >> 2) * kAo + (q & 3) * kKs, lbi + (q >> 2) * kBo + (q & 3) * kKs, kIdesc);
        } else {
#pragma unroll
          for (int q = 0; q < 16; ++q) umma_lo<true>(d, la + (q >> 2) * kAo + (q & 3) * kKs, lbi + (q >> 2) * kBo + (q & 3) * kKs, kIdesc);
        }
        umma_commit(&empty_bar[slot]);
      }
      umma_commit(acc1_full);
      // ---- FFN2: K = 128 (two k-blocks); a request holds tiles 2 (i - 10), + 1 as [k-block][tile][128 rows][128 B]
      mbar_wait(h_ready, 0, 6);
      tp(24);
      tc_fence_after_sync();
      for (int i = 10; i < 12; ++i) {
        const int slot = i % kBrSlots;
        mbar_wait(&full_bar[slot], (i / kBrSlots) & 1, 7);
        tp(10 + i);
        tc_fence_after_sync();
        const uint32_t la = lo(ring + slot * kBrSlotBytes);
#pragma unroll
        for (int tt = 0; tt < 2; ++tt) {
          const uint32_t d = tmem_base + kColFfn2 + ((i - 10) * 2 + tt) * kBrRows;
          umma_lo<false>(d, la + tt * kAo, lb, kIdesc);
#pragma unroll
          for (int q = 1; q < 8; ++q) umma_lo<true>(d, la + (q >> 2) * (2 * kAo) + tt * kAo + (q & 3) * kKs, lb + (q >> 2) * kBo + (q & 3) * kKs, kIdesc);
          umma_commit(&acc2_full[(i - 10) * 2 + tt]);
        }
        umma_commit(&empty_bar[slot]);     // all MMAs that read the ring have completed once this one arrives: the ring becomes the x staging tile
      }
    }
  } else {
    // ---- epilogue warps: thread = (TMEM lane i = features 4 i .. 4 i + 3, rows 8 rg .. 8 rg + 7)
    const int ew = warp - 2;
    const int quad = warp & 3;
    const int rg = ew >> 2;
    const int fi = quad * 32 + lane;                         // TMEM lane = col4 index of the blocked residual layout
    const int r0 = rg * 8;
    const uint32_t tmem_lane = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + static_cast<uint32_t>(r0);
    const float* xrow = ep.x + (static_cast<size_t>(blockIdx.x) * (kE / 4) + fi) * (32 * 4) + r0 * 4;   // 8 rows x float4, contiguous
    const float4 g_mid = __ldg(reinterpret_cast<const float4*>(ep.gain_mid) + fi);
    const float4 g_out = __ldg(reinterpret_cast<const float4*>(ep.gain_out) + fi);
    float r[8][4];
    pdl_wait();
    tp(1);
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      float v[8];
      ld_global_v8(xrow + p * 8, v);
#pragma unroll
      for (int c = 0; c < 4; ++c) { r[2 * p][c] = v[c]; r[2 * p + 1][c] = v[4 + c]; }
    }
    // rows at or beyond M hold whatever the workspace holds: they are computed (finite or not, they stay in their own columns); the tiled
    // stores clip them at M (xn) or write them into the padding rows of the last 32-row block (x)
    // val[0..7] / val[8..15]: this thread's partial sum / sum of squares of rows r0 + j, accumulated as the tiles arrive (only the last
    // tile's share is on the critical path)
    float val[16];
    auto add_tiles = [&](uint64_t* bars, uint32_t col0) {
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        mbar_wait(&bars[t], 0, 8);
        if (t == 0) tp(col0 == 0 ? 25 : 26);
        tc_fence_after_sync();
        float v[8];
        tmem_ld_32x8(tmem_lane + col0 + t * kBrRows, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float x = r[j][t] + v[j];
          r[j][t] = x;
          val[j] = t == 0 ? x : val[j] + x;
          val[8 + j] = t == 0 ? x * x : fmaf(x, x, val[8 + j]);
        }
      }
    };
    // Per-row LayerNorm coefficients over the 512 features: thread partials -> warp totals (16 shuffles) -> [row][quadrant] in shared memory ->
    // lane j < 8 of every warp finishes row r0 + j -> broadcast by shuffle.  a[j] = rstd, b[j] = -mean * rstd: LN(v) = (v * a + b) * gain.
    auto row_stats = [&](float (&a)[8], float (&b)[8], bool store_x) {
      const float tot = br_warp_reduce16(val, lane);
      if ((lane & 1) == 0) {
        const int k = lane >> 1;                              // 0..7: sum of row k; 8..15: sum of squares of row k - 8
        reinterpret_cast<float*>(&s_stats[(r0 + (k & 7)) * 4 + quad])[k >> 3] = tot;
      }
      br_epi_sync();
      if (store_x && threadIdx.x == 64) {                     // the x tile is staged (fenced before the barrier): it drains while the xn tile is made
        tma_store_4d(&tmap_x, ring, 0, 0, 0, static_cast<int>(blockIdx.x));
        bulk_commit_group();
      }
      float ra = 0.f, rb = 0.f;
      if (lane < 8) {
        const float4 p = *reinterpret_cast<const float4*>(&s_stats[(r0 + lane) * 4]);
        const float4 q = *reinterpret_cast<const float4*>(&s_stats[(r0 + lane) * 4 + 2]);
        const float sum = (p.x + p.z) + (q.x + q.z), sumsq = (p.y + p.w) + (q.y + q.w);
        const float mean = sum * (1.0f / kE);
        ra = rsqrtf(fmaxf(sumsq * (1.0f / kE) - mean * mean, 0.f) + ep.eps);
        rb = -mean * ra;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) { a[j] = __shfl_sync(0xffffffffu, ra, j); b[j] = __shfl_sync(0xffffffffu, rb, j); }
    };

    // ---- phase A: residual + out-proj (tile by tile while the next tile streams), LN2 rows -> resident operand
    add_tiles(acc0_full, 0);
    tp(2);
    float ca[8], cb[8];
    row_stats(ca, cb, false);
    {
      // features 4 fi .. 4 fi + 3 = 8 bytes of k-block fi >> 4, 16-byte chunk (fi >> 1) & 7, half fi & 1 of row r (row & 7 = j)
      uint8_t* dst = act + (fi >> 4) * kBrKbBytes + r0 * 128 + (fi & 1) * 8;
      const int chunk = (fi >> 1) & 7;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float y0 = fmaf(r[j][0], ca[j], cb[j]) * g_mid.x, y1 = fmaf(r[j][1], ca[j], cb[j]) * g_mid.y;
        const float y2 = fmaf(r[j][2], ca[j], cb[j]) * g_mid.z, y3 = fmaf(r[j][3], ca[j], cb[j]) * g_mid.w;
        *reinterpret_cast<uint2*>(dst + j * 128 + ((chunk ^ j) << 4)) = make_uint2(pack_bf16x2(y0, y1), pack_bf16x2(y2, y3));
      }
    }
    fence_proxy_async_smem();
    tc_fence_before_sync();
    __syncwarp();
    if (lane == 0) mbar_arrive(ln2_ready);
    tp(3);

    // ---- phase B: GELU of this thread's hidden feature (TMEM lane fi, natural order) for its 8 rows -> resident operand (k-blocks 0, 1)
    mbar_wait(acc1_full, 0, 9);
    tc_fence_after_sync();
    tp(4);
    {
      float v[8];
      tmem_ld_32x8(tmem_lane + kColHidden, v);
      uint8_t* dst = act + (fi >> 6) * kBrKbBytes + r0 * 128 + (fi & 7) * 2;
      const int chunk = (fi >> 3) & 7;
#pragma unroll
      for (int j = 0; j < 8; ++j) *reinterpret_cast<__nv_bfloat16*>(dst + j * 128 + ((chunk ^ j) << 4)) = __float2bfloat16_rn(gelu_fast(v[j]));
    }
    fence_proxy_async_smem();
    tc_fence_before_sync();
    __syncwarp();
    if (lane == 0) mbar_arrive(h_ready);
    tp(5);

    // ---- phase C: residual + FFN2, final LayerNorm; the x tile leaves through the TMA unit, the xn rows straight from the registers
    add_tiles(acc2_full, kColFfn2);
    tp(6);
    // x tile, staged in ring slot 0 (every MMA has completed: acc2_full[3]) as [rg][col4 fi][8 rows x 16 B], 16-byte chunks XOR-swizzled by
    // fi & 7 (the 128-byte swizzle of tmap_x): conflict-free for the 8 lanes of a quarter-warp, which hold consecutive fi
    {
      uint8_t* line = ring + (rg * 128 + fi) * 128;
#pragma unroll
      for (int j = 0; j < 8; ++j) *reinterpret_cast<float4*>(line + ((j ^ (fi & 7)) << 4)) = make_float4(r[j][0], r[j][1], r[j][2], r[j][3]);
    }
    fence_proxy_async_smem();
    tp(27);
    row_stats(ca, cb, true);
    tp(28);
    // xn rows straight from the registers: a thread's four features are 8 contiguous bytes and a warp's 32 threads hold consecutive
    // feature quadruples - one 256-byte run per row and store instruction (no staging tile, no barrier, nothing for the exit to wait for)
    {
      const bool remap = ep.remap_rows_in > 0;      // last layer of a prefix / teacher-forced pass: rows are renumbered, leading rows of a sequence dropped
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float y0 = fmaf(r[j][0], ca[j], cb[j]) * g_out.x, y1 = fmaf(r[j][1], ca[j], cb[j]) * g_out.y;
        const float y2 = fmaf(r[j][2], ca[j], cb[j]) * g_out.z, y3 = fmaf(r[j][3], ca[j], cb[j]) * g_out.w;
        const int grow = m0 + r0 + j;
        int nrow = grow;
        bool keep = grow < M;
        if (remap) {
          const int seq = grow / ep.remap_rows_in;
          const int k = grow - seq * ep.remap_rows_in;
          keep = keep && k >= ep.remap_skip;
          nrow = seq * ep.remap_rows_out + (k - ep.remap_skip);
        }
        if (keep) *reinterpret_cast<uint2*>(ep.xn + static_cast<size_t>(nrow) * kE + fi * 4) = make_uint2(pack_bf16x2(y0, y1), pack_bf16x2(y2, y3));
      }
    }
    tp(29);
    if (threadIdx.x == 64) bulk_wait_group_read0();          // the staged x tile must stay in place until the TMA unit has read it
    tp(7);
  }
  tc_fence_before_sync();
  __syncthreads();
  if (threadIdx.x == 64) tp(8);
  if (warp == 1) tmem_dealloc<512>(tmem_base);
}

// ---------------------------------------------------------------------------------------------------------
// The same kernel on 64 rows per CTA, for passes of more rows than one wave of 32-row CTAs covers (beam search, prefix / teacher-forced
// passes, 8192-embedding batches).  A tcgen05.mma costs the same 60 cycles for N = 64 as for N = 32 and the weight stream per CTA is the
// same 768 KB, so a CTA handles twice the rows in the same stream time: half the waves.  What changes: two 64 KB weight slots (the resident
// operand takes 64 KB), and the fp32 residual rows live in TMEM instead of registers - the x tile is written into the out-proj accumulator
// columns before the first MMA (tcgen05.st), every out-proj and FFN2 MMA accumulates onto it, and the epilogue reads it back once for
// the LayerNorm statistics and once to normalise (64 values per thread would not fit beside the statistics in 112 registers).
// TMEM columns: [0, 256) residual rows (4 tiles x 64 rows), [256, 320) hidden.  Thread = (TMEM lane i = features 4 i .. 4 i + 3,
// rows 32 h + 8 rg .. + 7 for h = 0, 1).
// ---------------------------------------------------------------------------------------------------------
constexpr int kB64Rows = 64;
constexpr int kB64Slots = 2;
constexpr int kB64ActBytes = kB64Rows * kE * 2;      // 64 KB
constexpr int kB64KbBytes = kB64Rows * kBlockK * 2;  // 8 KB
constexpr int kB64StatsBytes = kB64Rows * 4 * 8;
__host__ __device__ constexpr int block_rows64_smem_bytes() { return 1024 + kB64Slots * kBrSlotBytes + kB64ActBytes + 256 + kB64StatsBytes; }
static_assert(block_rows64_smem_bytes() <= 227 * 1024, "64-row row-owner block kernel does not fit in shared memory");

__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const float (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};\n" ::"r"(taddr), "r"(__float_as_uint(v[0])),
               "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
               "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
               : "memory");
}

__global__ void __launch_bounds__(kBrThreads, 1)
block_rows64_kernel(const __grid_constant__ CUtensorMap tmap_ao, const __grid_constant__ CUtensorMap tmap_wo, const __grid_constant__ CUtensorMap tmap_w1,
                    const __grid_constant__ CUtensorMap tmap_w2, const __grid_constant__ CUtensorMap tmap_x, int M,
                    FusedBlockParams ep) {
  constexpr uint32_t kIdesc = umma_idesc_bf16_f32(128, kB64Rows);
  constexpr uint32_t kColHidden = 256;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* ring = smem;
  uint8_t* act = ring + kB64Slots * kBrSlotBytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(act + kB64ActBytes);  // [2]
  uint64_t* empty_bar = full_bar + kB64Slots;                            // [2]
  uint64_t* act_full = empty_bar + kB64Slots;
  uint64_t* x_ready = act_full + 1;                                      // the residual rows are in TMEM (16 warp arrivals)
  uint64_t* acc0_full = x_ready + 1;                                     // [4]
  uint64_t* ln2_ready = acc0_full + 4;
  uint64_t* acc1_full = ln2_ready + 1;
  uint64_t* h_ready = acc1_full + 1;
  uint64_t* acc2_full = h_ready + 1;                                     // [4]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc2_full + 4);
  static_assert((2 * kB64Slots + 2 + 4 + 3 + 4) * 8 + 4 <= 256, "barrier area");
  float2* s_stats = reinterpret_cast<float2*>(act + kB64ActBytes + 256);  // [64 rows][4 quadrants]

  const int warp = threadIdx.x >> 5;
  const int lane = static_cast<int>(lane_id());
  const int m0 = blockIdx.x * kB64Rows;
  pdl_trigger();

  auto issue = [&](int i) {
    const int slot = i % kB64Slots;
    mbar_arrive_expect_tx(&full_bar[slot], kBrSlotBytes);
    uint8_t* dst = ring + slot * kBrSlotBytes;
    if (i < 8) tma_load_4d(dst, &tmap_wo, &full_bar[slot], 0, 0, i >> 1, (i & 1) * 4, kEvictLast);
    else if (i < 10) tma_load_3d(dst, &tmap_w1, &full_bar[slot], 0, (i - 8) * 4, kEvictLast);
    else tma_load_4d(dst, &tmap_w2, &full_bar[slot], 0, 0, (i - 10) * 2, 0, kEvictLast);
  };

  if (warp == 0) {
    if (elect_one()) {
      tma_prefetch_desc(&tmap_ao); tma_prefetch_desc(&tmap_wo); tma_prefetch_desc(&tmap_w1); tma_prefetch_desc(&tmap_w2);
      tma_prefetch_desc(&tmap_x);
      for (int st = 0; st < kB64Slots; ++st) { mbar_init(&full_bar[st], 1); mbar_init(&empty_bar[st], 1); }
      mbar_init(act_full, 1); mbar_init(x_ready, kBrEpiWarps);
      for (int t = 0; t < 4; ++t) { mbar_init(&acc0_full[t], 1); mbar_init(&acc2_full[t], 1); }
      mbar_init(ln2_ready, kBrEpiWarps); mbar_init(acc1_full, 1); mbar_init(h_ready, kBrEpiWarps);
      fence_mbar_init();
      for (int i = 0; i < kB64Slots; ++i) issue(i);
      pdl_wait();
      mbar_arrive_expect_tx(act_full, kB64ActBytes);
      tma_load_3d(act, &tmap_ao, act_full, m0, 0, kEvictFirst);
    }
  } else if (warp == 1) {
    tmem_alloc<512>(tmem_slot);
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      for (int i = kB64Slots; i < kBrRequests; ++i) {
        mbar_wait(&empty_bar[i % kB64Slots], ((i / kB64Slots) - 1) & 1, 1);
        issue(i);
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      const uint32_t lb = (smem_u32(act) & 0x3FFFFu) >> 4;
      auto lo = [](const void* p) { return (smem_u32(p) & 0x3FFFFu) >> 4; };
      constexpr uint32_t kKs = (kUmmaK * 2) >> 4, kAo = kABytes >> 4, kBo = kB64KbBytes >> 4;
      mbar_wait(act_full, 0, 2);
      mbar_wait(x_ready, 0, 2);
      tc_fence_after_sync();
      for (int i = 0; i < 8; ++i) {                      // out-proj, accumulated onto the residual rows
        const int slot = i % kB64Slots;
        mbar_wait(&full_bar[slot], (i / kB64Slots) & 1, 3);
        tc_fence_after_sync();
        const uint32_t la = lo(ring + slot * kBrSlotBytes);
        const uint32_t lbi = lb + (i & 1) * 4 * kBo;
        const uint32_t d = tmem_base + (i >> 1) * kB64Rows;
#pragma unroll
        for (int q = 0; q < 16; ++q) umma_lo<true>(d, la + (q >> 2) * kAo + (q & 3) * kKs, lbi + (q >> 2) * kBo + (q & 3) * kKs, kIdesc);
        umma_commit(&empty_bar[slot]);
        if (i & 1) umma_commit(&acc0_full[i >> 1]);
      }
      mbar_wait(ln2_ready, 0, 4);
      tc_fence_after_sync();
      for (int i = 8; i < 10; ++i) {                     // FFN1
        const int slot = i % kB64Slots;
        mbar_wait(&full_bar[slot], (i / kB64Slots) & 1, 5);
        tc_fence_after_sync();
        const uint32_t la = lo(ring + slot * kBrSlotBytes);
        const uint32_t lbi = lb + (i - 8) * 4 * kBo;
        const uint32_t d = tmem_base + kColHidden;
        if (i == 8) {
          umma_lo<false>(d, la, lbi, kIdesc);
#pragma unroll
          for (int q = 1; q < 16; ++q) umma_lo<true>(d, la + (q >> 2) * kAo + (q & 3) * kKs, lbi + (q >> 2) * kBo + (q & 3) * kKs, kIdesc);
        } else {
#pragma unroll
          for (int q = 0; q < 16; ++q) umma_lo<true>(d, la + (q >> 2) * kAo + (q & 3) * kKs, lbi + (q >> 2) * kBo + (q & 3) * kKs, kIdesc);
        }
        umma_commit(&empty_bar[slot]);
      }
      umma_commit(acc1_full);
      mbar_wait(h_ready, 0, 6);
      tc_fence_after_sync();
      for (int i = 10; i < 12; ++i) {                    // FFN2, accumulated onto the residual rows
        const int slot = i % kB64Slots;
        mbar_wait(&full_bar[slot], (i / kB64Slots) & 1, 7);
        tc_fence_after_sync();
        const uint32_t la = lo(ring + slot * kBrSlotBytes);
#pragma unroll
        for (int tt = 0; tt < 2; ++tt) {
          const uint32_t d = tmem_base + ((i - 10) * 2 + tt) * kB64Rows;
#pragma unroll
          for (int q = 0; q < 8; ++q) umma_lo<true>(d, la + (q >> 2) * (2 * kAo) + tt * kAo + (q & 3) * kKs, lb + (q >> 2) * kBo + (q & 3) * kKs, kIdesc);
          umma_commit(&acc2_full[(i - 10) * 2 + tt]);
        }
      }
    }
  } else {
    const int ew = warp - 2;
    const int quad = warp & 3;
    const int rg = ew >> 2;
    const int fi = quad * 32 + lane;
    const int r0 = rg * 8;
    const uint32_t tl = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + static_cast<uint32_t>(r0);
    const float4 g_mid = __ldg(reinterpret_cast<const float4*>(ep.gain_mid) + fi);
    const float4 g_out = __ldg(reinterpret_cast<const float4*>(ep.gain_out) + fi);
    pdl_wait();
    // ---- residual rows -> TMEM (column 64 t + 32 h + row of tile t = feature 4 fi + t)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float v[4][8];
      if (m0 + 32 * h < M) {
        const float* xrow = ep.x + (static_cast<size_t>(blockIdx.x * 2 + h) * (kE / 4) + fi) * (32 * 4) + r0 * 4;
#pragma unroll
        for (int p = 0; p < 4; ++p) ld_global_v8(xrow + p * 8, v[p]);
      } else {
#pragma unroll
        for (int p = 0; p < 4; ++p)
#pragma unroll
          for (int c = 0; c < 8; ++c) v[p][c] = 0.f;
      }
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        float c[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) c[j] = v[j >> 1][(j & 1) * 4 + t];
        tmem_st_32x8(tl + t * kB64Rows + 32 * h, c);
      }
    }
    tmem_st_wait();
    tc_fence_before_sync();
    __syncwarp();
    if (lane == 0) mbar_arrive(x_ready);

    float val[32];      // [h][0..7 sums, 8..15 sums of squares] of rows 32 h + r0 + j
    auto stat_tiles = [&](uint64_t* bars) {
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        mbar_wait(&bars[t], 0, 8);
        tc_fence_after_sync();
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float v[8];
          tmem_ld_32x8(tl + t * kB64Rows + 32 * h, v);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            val[h * 16 + j] = t == 0 ? v[j] : val[h * 16 + j] + v[j];
            val[h * 16 + 8 + j] = t == 0 ? v[j] * v[j] : fmaf(v[j], v[j], val[h * 16 + 8 + j]);
          }
        }
      }
    };
    float ca[2][8], cb[2][8];
    auto row_stats = [&]() {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        float part[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) part[k] = val[h * 16 + k];
        const float tot = br_warp_reduce16(part, lane);
        if ((lane & 1) == 0) {
          const int k = lane >> 1;
          reinterpret_cast<float*>(&s_stats[(32 * h + r0 + (k & 7)) * 4 + quad])[k >> 3] = tot;
        }
      }
      br_epi_sync();
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        float ra = 0.f, rb = 0.f;
        if (lane < 8) {
          const float4 p = *reinterpret_cast<const float4*>(&s_stats[(32 * h + r0 + lane) * 4]);
          const float4 q = *reinterpret_cast<const float4*>(&s_stats[(32 * h + r0 + lane) * 4 + 2]);
          const float sum = (p.x + p.z) + (q.x + q.z), sumsq = (p.y + p.w) + (q.y + q.w);
          const float mean = sum * (1.0f / kE);
          ra = rsqrtf(fmaxf(sumsq * (1.0f / kE) - mean * mean, 0.f) + ep.eps);
          rb = -mean * ra;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) { ca[h][j] = __shfl_sync(0xffffffffu, ra, j); cb[h][j] = __shfl_sync(0xffffffffu, rb, j); }
      }
    };
    // this thread's residual values of half h: r[j][t]
    auto load_rows = [&](int h, float (&r)[8][4]) {
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        float v[8];
        tmem_ld_32x8(tl + t * kB64Rows + 32 * h, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j][t] = v[j];
      }
    };

    // ---- phase A: statistics of x + out-proj, LN2 rows -> resident operand
    stat_tiles(acc0_full);
    row_stats();
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float r[8][4];
      load_rows(h, r);
      uint8_t* dst = act + (fi >> 4) * kB64KbBytes + (32 * h + r0) * 128 + (fi & 1) * 8;
      const int chunk = (fi >> 1) & 7;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float y0 = fmaf(r[j][0], ca[h][j], cb[h][j]) * g_mid.x, y1 = fmaf(r[j][1], ca[h][j], cb[h][j]) * g_mid.y;
        const float y2 = fmaf(r[j][2], ca[h][j], cb[h][j]) * g_mid.z, y3 = fmaf(r[j][3], ca[h][j], cb[h][j]) * g_mid.w;
        *reinterpret_cast<uint2*>(dst + j * 128 + ((chunk ^ j) << 4)) = make_uint2(pack_bf16x2(y0, y1), pack_bf16x2(y2, y3));
      }
    }
    fence_proxy_async_smem();
    tc_fence_before_sync();
    __syncwarp();
    if (lane == 0) mbar_arrive(ln2_ready);

    // ---- phase B: GELU -> hidden rows in the resident operand (k-blocks 0, 1)
    mbar_wait(acc1_full, 0, 9);
    tc_fence_after_sync();
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float v[8];
      tmem_ld_32x8(tl + kColHidden + 32 * h, v);
      uint8_t* dst = act + (fi >> 6) * kB64KbBytes + (32 * h + r0) * 128 + (fi & 7) * 2;
      const int chunk = (fi >> 3) & 7;
#pragma unroll
      for (int j = 0; j < 8; ++j) *reinterpret_cast<__nv_bfloat16*>(dst + j * 128 + ((chunk ^ j) << 4)) = __float2bfloat16_rn(gelu_fast(v[j]));
    }
    fence_proxy_async_smem();
    tc_fence_before_sync();
    __syncwarp();
    if (lane == 0) mbar_arrive(h_ready);

    // ---- phase C: statistics of the block's output rows; the x tiles leave through the TMA unit, the xn rows straight from the registers
    stat_tiles(acc2_full);
    row_stats();
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float r[8][4];
      load_rows(h, r);
      uint8_t* line = ring + h * kBrSlotBytes + (rg * 128 + fi) * 128;                 // x tile of 32-row block h: [rg][col4][8 rows x 16 B], swizzled
      const bool remap = ep.remap_rows_in > 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        *reinterpret_cast<float4*>(line + ((j ^ (fi & 7)) << 4)) = make_float4(r[j][0], r[j][1], r[j][2], r[j][3]);
        const float y0 = fmaf(r[j][0], ca[h][j], cb[h][j]) * g_out.x, y1 = fmaf(r[j][1], ca[h][j], cb[h][j]) * g_out.y;
        const float y2 = fmaf(r[j][2], ca[h][j], cb[h][j]) * g_out.z, y3 = fmaf(r[j][3], ca[h][j], cb[h][j]) * g_out.w;
        // xn rows straight from the registers (8 contiguous bytes per thread, 256 per warp and row), renumbered in a pass's last layer
        const int grow = m0 + 32 * h + r0 + j;
        int nrow = grow;
        bool keep = grow < M;
        if (remap) {
          const int seq = grow / ep.remap_rows_in;
          const int k = grow - seq * ep.remap_rows_in;
          keep = keep && k >= ep.remap_skip;
          nrow = seq * ep.remap_rows_out + (k - ep.remap_skip);
        }
        if (keep) *reinterpret_cast<uint2*>(ep.xn + static_cast<size_t>(nrow) * kE + fi * 4) = make_uint2(pack_bf16x2(y0, y1), pack_bf16x2(y2, y3));
      }
    }
    fence_proxy_async_smem();
    br_epi_sync();
    if (threadIdx.x == 64) {
#pragma unroll
      for (int h = 0; h < 2; ++h) tma_store_4d(&tmap_x, ring + h * kBrSlotBytes, 0, 0, 0, static_cast<int>(blockIdx.x) * 2 + h);   // a block beyond the allocation is clipped
      bulk_commit_group();
    }
    if (threadIdx.x == 64) bulk_wait_group_read0();
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) tmem_dealloc<512>(tmem_base);
}

}  // namespace novic
