// tcgen05 GEMMs for the decoder: D[M, N] = A[M, K] * W[N, K]^T with bf16 operands (both K-major), fp32
// accumulation in TMEM, operands staged by TMA into 128B-swizzled shared memory, and the layer's
// elementwise work fused into the epilogue (SURVEY.md §2 kernel inventory rows: QKV, out-proj + residual +
// LayerNorm, FFN1 + GELU, FFN2 + residual + LayerNorm, prefix projection + positions + LayerNorm,
// logits + max / argmax / log-sum-exp / top-k).
//
// One CTA computes one 128 x 128 output tile.  Warp roles:
//   warp 0      : barrier init + TMA producer (one elected lane; the first stages are issued before the CTA-wide
//                 setup barrier so the TMEM allocation overlaps the first loads' latency)
//   warp 1      : TMEM allocator + tcgen05.mma issuer (one elected lane)
//   warps 2..   : epilogue (4 or 8 warps); warp w owns TMEM lanes [32*(w%4), +32), thread = one output row
// Pipelines: smem full/empty mbarriers between TMA and MMA; one tmem_full mbarrier MMA -> epilogue.
// bf16 outputs are staged per warp in shared memory (the drained pipeline stages) and written with lanes covering
// contiguous row segments: "thread = row" direct stores touch 32 cache lines per instruction and were measured at
// 5-6k cycles per tile (profiles/r01_phase_trace.txt).
#pragma once

#include "ptx.cuh"

namespace novic {

constexpr int kE = 512;           // hidden dim (config/train.yaml:256)
constexpr int kBlockM = 128;
constexpr int kBlockK = 64;       // 64 bf16 = 128 B = one swizzle row
constexpr int kUmmaK = 16;
constexpr int kTileN = 128;
constexpr int kABytes = kBlockM * kBlockK * 2;
constexpr int kBBytes = kTileN * kBlockK * 2;
constexpr int kStageBytes = kABytes + kBBytes;           // 32 KB
constexpr int kStagePitch = kTileN * 2 + 16;             // staged bf16 row: 256 B + 16 B pad (conflict-free 16 B accesses)
constexpr int kWarpStageBytes = 32 * kStagePitch;        // 8704 B per epilogue warp

// fp32 residual stream `x` lives in a 32-row blocked layout so that "thread = row" epilogue accesses are
// coalesced: element (row, col) is at (((row >> 5) * (kE / 4) + (col >> 2)) * 32 + (row & 31)) * 4 + (col & 3).
__host__ __device__ __forceinline__ size_t xblk_off(int row, int col4) {
  return ((static_cast<size_t>(row >> 5) * (kE / 4) + col4) * 32 + (row & 31)) * 4;
}

__host__ __device__ constexpr int gemm_smem_bytes(int stages) { return stages * kStageBytes + 1024 /*align*/ + 256 /*barriers*/ + 1536 /*scratch*/; }

struct EpiCtx {
  uint32_t tmem_row;   // TMEM address of this thread's lane, first column of the thread's column range
  int row;             // global output row of this thread
  int warp_row0;       // global output row of lane 0 of this warp
  int n0;              // first output column of this thread's column range
  int ncols;           // columns per thread: 64 (128-column tiles; what every decoder epilogue assumes) or 128 (256-column tiles)
  int M;
  int part;            // partial index: tile * 2 + half
  uint8_t* stage;      // warp-private staging memory (kEpiStageBytes)
};

// Every epilogue of the persistent kernel runs on 8 warps: two per TMEM lane quadrant, 64 columns per thread.
constexpr int kEpiWarps = 8;
constexpr int kEpiCols = kTileN / 2;                 // 64
constexpr int kEpiStagePitch = kEpiCols * 2;         // staged bf16 row: 128 B, 16-byte chunks XOR-swizzled by the row (conflict-free)
constexpr int kEpiStageBytes = 32 * kEpiStagePitch;  // 4096 B per epilogue warp

// 16-byte chunk `chunk` (0..7) of staged row `row` (0..31)
__device__ __forceinline__ uint4* stage_chunk(uint8_t* stage, int row, int chunk) {
  return reinterpret_cast<uint4*>(stage + row * kEpiStagePitch + ((chunk ^ (row & 7)) << 4));
}
__device__ __forceinline__ const uint4* stage_chunk(const uint8_t* stage, int row, int chunk) {
  return reinterpret_cast<const uint4*>(stage + row * kEpiStagePitch + ((chunk ^ (row & 7)) << 4));
}

// 4 packed uint4 (32 bf16) of this thread's row -> staging row (columns [c0, c0 + 32) of the thread's 64)
__device__ __forceinline__ void stage_put32(uint8_t* stage, int lane, int c0, const float (&v)[32]) {
#pragma unroll
  for (int q = 0; q < 4; ++q)
    *stage_chunk(stage, lane, (c0 >> 3) + q) = make_uint4(pack_bf16x2(v[q * 8 + 0], v[q * 8 + 1]), pack_bf16x2(v[q * 8 + 2], v[q * 8 + 3]),
                      pack_bf16x2(v[q * 8 + 4], v[q * 8 + 5]), pack_bf16x2(v[q * 8 + 6], v[q * 8 + 7]));
}

// Write the warp's staged 32 x 64 bf16 block: per instruction the 32 lanes cover 4 rows x 128 contiguous bytes.
// row_ptr(r) -> global address of the block's first column for warp-local row r, or nullptr to skip the row.
// l2_hint != 0: the stores carry that L2 eviction-priority policy.
template <class RowPtr>
__device__ __forceinline__ void stage_copy_out(const uint8_t* stage, int lane, RowPtr row_ptr, uint64_t l2_hint = 0) {
  __syncwarp();
  const int sub = lane >> 3, chunk = lane & 7;
#pragma unroll 4
  for (int i = 0; i < 8; ++i) {
    const int r = i * 4 + sub;
    const uint4 v = *stage_chunk(stage, r, chunk);
    __nv_bfloat16* dst = row_ptr(r);
    if (dst != nullptr) {
      if (l2_hint != 0) st_global_v4_hint(dst + chunk * 8, v, l2_hint);
      else *reinterpret_cast<uint4*>(dst + chunk * 8) = v;
    }
  }
  __syncwarp();
}

// ---------------------------------------------------------------------------------------------------------
// Epilogues of the generic kernel.  run(params, ctx, release): `release()` must be called (by all lanes) right after
// the thread's last tcgen05.ld of the tile - it hands the TMEM accumulator stage back to the MMA warp.
// ---------------------------------------------------------------------------------------------------------

// q / k / v split (nn.MultiheadAttention in_proj, rows [Wq;Wk;Wv]): q -> q buffer, k and v -> KV cache page
// of the row's sequence at the row's position.
struct EpiQKV {
  struct Params {
    __nv_bfloat16* q;       // [M, 512]
    __nv_bfloat16* kcache;  // this layer: [slots, smax, 512]
    __nv_bfloat16* vcache;
    int rows_per_seq, pos0, slot_mul, smax;
    int kv_hint;            // K/V rows are stored with an evict-last L2 policy (decode steps: the next step reads them back)
  };
  // A thread owns c.ncols = 64 columns (128-column tiles) or 128 (256-column tiles; a 256-column tile lies inside one of q / K / V):
  // 64 columns are staged and written at a time.
  template <class Release>
  __device__ static __forceinline__ void run(const Params& p, const EpiCtx& c, Release release) {
    const int lane = lane_id();
    const int nparts = c.ncols / kEpiCols;
    if (c.stage == nullptr) {
      // No staging tile (the three-stage weight-stationary kernel spends those 32 KB on a third activation stage): the thread's 64 columns
      // are 128 contiguous bytes of its row of q / K / V and leave as four 256-bit stores - full 32-byte sectors, where 16-byte stores
      // wrote half sectors (measured slower than the staged copy-out, gemm_ws_smem_bytes)
      for (int part = 0; part < nparts; ++part) {
        const int n0 = c.n0 + part * kEpiCols;
        __nv_bfloat16* dst = nullptr;
        if (c.row < c.M) {
          if (n0 < kE) dst = p.q + static_cast<size_t>(c.row) * kE + n0;
          else {
            const int seq = c.row / p.rows_per_seq;
            const int pos = p.pos0 + (c.row - seq * p.rows_per_seq);
            const size_t page = (static_cast<size_t>(seq) * p.slot_mul * p.smax + pos) * kE;
            dst = (n0 < 2 * kE) ? p.kcache + page + (n0 - kE) : p.vcache + page + (n0 - 2 * kE);
          }
        }
#pragma unroll
        for (int ch = 0; ch < kEpiCols / 32; ++ch) {
          float v[32];
          tmem_ld_32x32(c.tmem_row + part * kEpiCols + ch * 32, v);
          if (part == nparts - 1 && ch == kEpiCols / 32 - 1) release();
          if (dst != nullptr) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              uint32_t w[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) w[i] = pack_bf16x2(v[h * 16 + 2 * i], v[h * 16 + 2 * i + 1]);
              asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};\n" ::"l"(dst + ch * 32 + h * 16), "r"(w[0]), "r"(w[1]), "r"(w[2]),
                           "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7])
                           : "memory");
            }
          }
        }
      }
      return;
    }
    for (int part = 0; part < nparts; ++part) {
#pragma unroll
      for (int ch = 0; ch < kEpiCols / 32; ++ch) {
        float v[32];
        tmem_ld_32x32(c.tmem_row + part * kEpiCols + ch * 32, v);
        if (part == nparts - 1 && ch == kEpiCols / 32 - 1) release();
        stage_put32(c.stage, lane, ch * 32, v);
      }
      const int n0 = c.n0 + part * kEpiCols;
      stage_copy_out(c.stage, lane, [&](int r) -> __nv_bfloat16* {
        const int row = c.warp_row0 + r;
        if (row >= c.M) return nullptr;
        if (n0 < kE) return p.q + static_cast<size_t>(row) * kE + n0;
        const int seq = row / p.rows_per_seq;
        const int pos = p.pos0 + (row - seq * p.rows_per_seq);
        const size_t page = (static_cast<size_t>(seq) * p.slot_mul * p.smax + pos) * kE;
        return (n0 < 2 * kE) ? p.kcache + page + (n0 - kE) : p.vcache + page + (n0 - 2 * kE);
      }, (n0 >= kE && p.kv_hint) ? kEvictLast : 0ull);   // new K/V rows: keep them in L2 for the next step's attention
    }
  }
};

// exact-GELU with erf from Abramowitz & Stegun 7.1.26 (|error| < 1.5e-7, far below the bf16 output resolution)
__device__ __forceinline__ float gelu_fast(float x) {
  const float ax = fabsf(x) * 0.70710678118654752440f;
  const float t = __fdividef(1.0f, fmaf(0.3275911f, ax, 1.0f));
  float poly = fmaf(t, 1.061405429f, -1.453152027f);
  poly = fmaf(poly, t, 1.421413741f);
  poly = fmaf(poly, t, -0.284496736f);
  poly = fmaf(poly, t, 0.254829592f);
  const float erf_abs = 1.0f - poly * t * __expf(-ax * ax);
  return 0.5f * x * (1.0f + copysignf(erf_abs, x));
}

// Per (row, 64-column vocabulary slice) statistics written by the logits epilogue and merged by the selection kernels.
struct __align__(32) LogitPartial {
  float max_all;     // max over the slice's valid columns (natural units)
  float sumexp_tau;  // sum exp((x - max_all) / tau)
  float sumexp_one;  // sum exp(x - max_all)
  float sum_x;       // sum of x (label smoothing term; 0 unless requested)
  float best_val;    // best selectable logit (column 0 excluded when the end token is banned)
  int best_idx;      // its vocabulary index (lowest index wins ties)
  float tgt_logit;   // logit of this row's target id if it falls in this slice, else -inf
  int pad_;
};

constexpr int kLogitSlice = kEpiCols;     // columns per epilogue thread

// Vocabulary logits (tied weights, embedding_decoder.py:725): never materialised unless asked for.
// MASKED = guided decoding (embedding_decoder.py:806-810, :915-920, :942-943): `allow` holds one bit per (row, vocabulary id);
// only allowed ids can be selected (best / top-H), and with mask_lse (guide_renorm) the temperature log-sum-exp runs over
// the allowed ids only.  The tau = 1 log-sum-exp (cross-entropy of the raw logits) and the optional logits copy are never masked.
// BIAS (beam search with a vocabulary prior, embedding_decoder.py:924-936; implies MASKED): every allowed id is a trie edge with
// an additive score; the top-H lists rank and store  logit + tau * bias  so that the selection kernel's
// (value / tau - logsumexp) is the reference's  log_softmax - vocab_scaler * log p_vocab.  `edge0` names the edge of the lowest
// allowed id of each 32-id mask word; the others follow in id order.
template <int HCAP, bool MASKED = false, bool BIAS = false>
struct EpiLogits {
  struct Params {
    float* logits;              // optional [M, ld_logits] fp32
    long long ld_logits;
    LogitPartial* part;         // [M, nparts]
    float* topv;                // optional [M, nparts, HCAP]
    int* topi;
    const long long* target;    // optional [M] target ids (-1 = ignore)
    int n_valid;                // V
    int nparts;                 // 2 * number of 128-column tiles
    float inv_tau;
    int ban_eos;                // exclude id 0 from best / top-k (first generated token)
    int want_sumx;              // label smoothing needs sum of logits
    const uint32_t* allow;      // MASKED: [M, allow_ld] bit masks (bit c & 31 of word c >> 5 = id c allowed)
    int allow_ld;
    int allow_mod;              // MASKED: mask row = row % allow_mod when > 0 (teacher forcing: masks shared by all embeddings)
    int mask_lse;               // MASKED: renormalise the temperature softmax over the allowed ids
    const int* edge0;           // BIAS: [M, allow_ld] trie edge of the lowest allowed id of each mask word
    const float* bias;          // BIAS: [num_edges]
    float tau;
  };
  // A thread owns c.ncols = 64 columns (128-column tiles) or 128 (256-column tiles): one 64-column vocabulary slice at a time, each with
  // its own partial record; the accumulator stage is released after the last load of the last slice.
  template <class Release>
  __device__ static __forceinline__ void run(const Params& p, const EpiCtx& c0, Release release) {
    const int nslices = c0.ncols / kLogitSlice;
#pragma unroll 1
    for (int sl = 0; sl < nslices; ++sl) {
      EpiCtx c = c0;
      c.tmem_row = c0.tmem_row + sl * kLogitSlice;
      c.n0 = c0.n0 + sl * kLogitSlice;
      c.part = c0.part + sl;
      if (sl == nslices - 1) slice(p, c, release);
      else slice(p, c, []() {});
    }
  }
  template <class Release>
  __device__ static __forceinline__ void slice(const Params& p, const EpiCtx& c, Release release) {
    constexpr float kLog2e = 1.4426950408889634f;
    float m = -INFINITY, s_tau = 0.f, s_one = 0.f, sum_x = 0.f, best = -INFINITY, tgt_logit = -INFINITY;
    float m_t = -INFINITY;       // MASKED: running max of the temperature softmax's support
    int best_i = 0x7fffffff;
    float tv[HCAP > 0 ? HCAP : 1];
    int ti[HCAP > 0 ? HCAP : 1];
#pragma unroll
    for (int i = 0; i < (HCAP > 0 ? HCAP : 1); ++i) { tv[i] = -INFINITY; ti[i] = 0x7fffffff; }
    const bool in_range = c.row < c.M;
    const long long tgt = (p.target != nullptr && in_range) ? p.target[c.row] : -1;
    const bool tau_is_one = (p.inv_tau == 1.0f);
    const float tau_l2e = p.inv_tau * kLog2e;
#pragma unroll 1
    for (int ch = 0; ch < kLogitSlice / 32; ++ch) {
      const int col0 = c.n0 + ch * 32;
      if (col0 >= p.n_valid) { if (ch == 0) release(); break; }  // uniform over the warp; the release still has to happen
      float v[32];
      tmem_ld_32x32(c.tmem_row + ch * 32, v);
      if (ch == kLogitSlice / 32 - 1 || col0 + 32 >= p.n_valid) release();
      if (col0 + 32 > p.n_valid) {   // ragged last chunk of the vocabulary: neutralise the invalid columns
#pragma unroll
        for (int j = 0; j < 32; ++j) if (col0 + j >= p.n_valid) v[j] = -INFINITY;
      }
      if (p.logits != nullptr && in_range) {
        float* lp = p.logits + static_cast<size_t>(c.row) * p.ld_logits + col0;
        if ((p.ld_logits & 3) == 0 && col0 + 32 <= p.n_valid) {
#pragma unroll
          for (int q = 0; q < 8; ++q) reinterpret_cast<float4*>(lp)[q] = make_float4(v[q * 4], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) if (col0 + j < p.n_valid) lp[j] = v[j];
        }
      }
      if (p.want_sumx) {
#pragma unroll
        for (int j = 0; j < 32; ++j) if (col0 + j < p.n_valid) sum_x += v[j];
      }
      if (tgt >= col0 && tgt < col0 + 32) {
#pragma unroll
        for (int j = 0; j < 32; ++j) if (col0 + j == tgt) tgt_logit = v[j];
      }
      if (!MASKED) {
        // (a) chunk max and arg-max; ascending scan with strict '>' keeps the lowest index on ties
        const float v0 = v[0];
        if (p.ban_eos && col0 == 0) v[0] = -INFINITY;
        float cm = v[0];
        int ci = 0;
#pragma unroll
        for (int j = 1; j < 32; ++j) if (v[j] > cm) { cm = v[j]; ci = j; }
        if (cm > best) { best = cm; best_i = col0 + ci; }
        if (HCAP > 0) {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            if (v[j] > tv[HCAP > 0 ? HCAP - 1 : 0]) {
              float cv = v[j]; int cidx = col0 + j;
#pragma unroll
              for (int i = 0; i < (HCAP > 0 ? HCAP : 1); ++i)
                if (cv > tv[i]) { const float tf = tv[i]; const int tI = ti[i]; tv[i] = cv; ti[i] = cidx; cv = tf; cidx = tI; }
            }
          }
        }
        v[0] = v0;
        // (b) online log-sum-exp in base 2: exp(x - m) = ex2(x * log2e - m * log2e)
        const float m_new = fmaxf(m, fmaxf(cm, v0));
        const float mb = m_new * kLog2e;
        float a_one = 0.f;
#pragma unroll
        for (int j = 0; j < 32; ++j) a_one += exp2f(fmaf(v[j], kLog2e, -mb));
        s_one = s_one * exp2f((m - m_new) * kLog2e) + a_one;
        if (!tau_is_one) {
          const float mbt = m_new * tau_l2e;
          float a_tau = 0.f;
#pragma unroll
          for (int j = 0; j < 32; ++j) a_tau += exp2f(fmaf(v[j], tau_l2e, -mbt));
          s_tau = s_tau * exp2f((m - m_new) * tau_l2e) + a_tau;
        }
        m = m_new;
      } else {
        const int mrow = p.allow_mod > 0 ? c.row % p.allow_mod : c.row;
        uint32_t bits = in_range ? p.allow[static_cast<size_t>(mrow) * p.allow_ld + (col0 >> 5)] : 0u;
        uint32_t sel = bits;
        if (p.ban_eos && col0 == 0) sel &= ~1u;
        // (a) best / top-H over the selectable ids only
        float cm = -INFINITY, call = -INFINITY;
        int ci = 0;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          call = fmaxf(call, v[j]);
          if (((sel >> j) & 1u) && v[j] > cm) { cm = v[j]; ci = j; }
        }
        if (cm > best) { best = cm; best_i = col0 + ci; }
        if (HCAP > 0) {
          const float* eb = nullptr;
          if (BIAS && bits != 0u) eb = p.bias + p.edge0[static_cast<size_t>(mrow) * p.allow_ld + (col0 >> 5)];
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            if (!((sel >> j) & 1u)) continue;
            float key = v[j];
            if (BIAS) key = fmaf(eb[__popc(bits & ((1u << j) - 1u))], p.tau, key);
            if (key > tv[HCAP > 0 ? HCAP - 1 : 0]) {
              float cv = key; int cidx = col0 + j;
#pragma unroll
              for (int i = 0; i < (HCAP > 0 ? HCAP : 1); ++i)
                if (cv > tv[i]) { const float tf = tv[i]; const int tI = ti[i]; tv[i] = cv; ti[i] = cidx; cv = tf; cidx = tI; }
            }
          }
        }
        // (b) tau = 1 log-sum-exp over every id; temperature log-sum-exp over its support (allowed ids when renormalising)
        const float m_new = fmaxf(m, call);
        const float mb = m_new * kLog2e;
        float a_one = 0.f;
#pragma unroll
        for (int j = 0; j < 32; ++j) a_one += exp2f(fmaf(v[j], kLog2e, -mb));
        s_one = s_one * exp2f((m - m_new) * kLog2e) + a_one;
        m = m_new;
        const uint32_t sup = p.mask_lse ? bits : 0xffffffffu;
        float cmt = -INFINITY;
#pragma unroll
        for (int j = 0; j < 32; ++j) if ((sup >> j) & 1u) cmt = fmaxf(cmt, v[j]);
        if (cmt > -INFINITY) {
          const float mt_new = fmaxf(m_t, cmt);
          const float mbt = mt_new * tau_l2e;
          float a_tau = 0.f;
#pragma unroll
          for (int j = 0; j < 32; ++j) if ((sup >> j) & 1u) a_tau += exp2f(fmaf(v[j], tau_l2e, -mbt));
          s_tau = s_tau * exp2f((m_t - mt_new) * tau_l2e) + a_tau;   // m_t = -inf on the first contribution: factor 0
          m_t = mt_new;
        }
      }
    }
    if (in_range) {
      LogitPartial o;
      o.max_all = m; o.sumexp_tau = tau_is_one ? s_one : s_tau; o.sumexp_one = s_one; o.sum_x = sum_x;
      o.best_val = best; o.best_idx = best_i; o.tgt_logit = tgt_logit; o.pad_ = 0;
      if (MASKED) { o.sumexp_tau = s_tau; o.pad_ = __float_as_int(m_t); }   // the temperature sum has its own reference maximum
      p.part[static_cast<size_t>(c.row) * p.nparts + c.part] = o;
      if (HCAP > 0) {
        const size_t base = (static_cast<size_t>(c.row) * p.nparts + c.part) * (HCAP > 0 ? HCAP : 1);
        // the list is sorted, unused slots (index 0x7fffffff) come last: store up to and including the first unused slot - the
        // selection kernel stops there.  Guided rows have a handful of allowed ids, so most slices store one terminator only.
        bool live = true;
#pragma unroll
        for (int i = 0; i < (HCAP > 0 ? HCAP : 1); ++i) {
          if (live) { p.topv[base + i] = tv[i]; p.topi[base + i] = ti[i]; }
          live = live && ti[i] != 0x7fffffff;
        }
      }
    }
  }
};

// ---------------------------------------------------------------------------------------------------------
// Shared mainloop pieces
// ---------------------------------------------------------------------------------------------------------
struct GemmSmemView {
  uint8_t* stages;
  uint64_t* full_bar;
  uint64_t* empty_bar;
  uint64_t* tmem_full_bar;
  uint32_t* tmem_slot;
  uint8_t* scratch;
};

template <int STAGES>
__device__ __forceinline__ GemmSmemView carve_smem(uint8_t* smem_raw) {
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  GemmSmemView v;
  v.stages = smem;
  v.full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * kStageBytes);
  v.empty_bar = v.full_bar + STAGES;
  v.tmem_full_bar = v.empty_bar + STAGES;
  v.tmem_slot = reinterpret_cast<uint32_t*>(v.tmem_full_bar + 1);
  v.scratch = smem + STAGES * kStageBytes + 256;
  return v;
}

__device__ __forceinline__ void tma_issue_stage(const GemmSmemView& sv, int stage, const CUtensorMap* ta, const CUtensorMap* tb,
                                                int kb, int m0, int n0, uint32_t stage_tx = kStageBytes) {
  uint8_t* sa = sv.stages + stage * kStageBytes;
  mbar_arrive_expect_tx(&sv.full_bar[stage], stage_tx);
  tma_load_2d(sa, ta, &sv.full_bar[stage], kb * kBlockK, m0, kEvictNormal);
  tma_load_2d(sa + kABytes, tb, &sv.full_bar[stage], kb * kBlockK, n0, kEvictLast);
}

// warp 0, one lane: init barriers, start the first loads (before the CTA-wide setup barrier)
template <int STAGES>
__device__ __forceinline__ void producer_prologue(const GemmSmemView& sv, const CUtensorMap* ta, const CUtensorMap* tb, int nkb, int m0, int n0) {
  for (int s = 0; s < STAGES; ++s) { mbar_init(&sv.full_bar[s], 1); mbar_init(&sv.empty_bar[s], 1); }
  mbar_init(sv.tmem_full_bar, 1);
  fence_mbar_init();
  const int pre = nkb < STAGES ? nkb : STAGES;
  for (int kb = 0; kb < pre; ++kb) tma_issue_stage(sv, kb, ta, tb, kb, m0, n0);
}

template <int STAGES>
__device__ __forceinline__ void producer_rest(const GemmSmemView& sv, const CUtensorMap* ta, const CUtensorMap* tb, int nkb, int m0, int n0,
                                              uint32_t stage_tx = kStageBytes) {
  int stage = 0; uint32_t phase = 0;   // k-block kb = STAGES + i reuses stage i % STAGES, whose first use must have drained
  for (int kb = STAGES; kb < nkb; ++kb) {
    mbar_wait(&sv.empty_bar[stage], phase, 1);
    tma_issue_stage(sv, stage, ta, tb, kb, m0, n0, stage_tx);
    if (++stage == STAGES) { stage = 0; phase ^= 1; }
  }
}

template <int STAGES, int BN = kTileN>
__device__ __forceinline__ void mma_mainloop(const GemmSmemView& sv, uint32_t tmem_base, int nkb, bool tr) {
  constexpr uint32_t kIdesc = umma_idesc_bf16_f32(kBlockM, BN);
  int stage = 0; uint32_t phase = 0;
  for (int kb = 0; kb < nkb; ++kb) {
    mbar_wait(&sv.full_bar[stage], phase, 2);
    if (kb == 0) trace_point(tr, 4);
    tc_fence_after_sync();
    const uint32_t sa = smem_u32(sv.stages + stage * kStageBytes);
    const uint32_t sb = sa + kABytes;
#pragma unroll
    for (int k = 0; k < kBlockK / kUmmaK; ++k)
      umma_bf16_ss(tmem_base, umma_desc_sw128_kmajor(sa + k * (kUmmaK * 2)), umma_desc_sw128_kmajor(sb + k * (kUmmaK * 2)), kIdesc,
                   (kb | k) != 0 ? 1u : 0u);
    umma_commit(&sv.empty_bar[stage]);  // frees this smem stage once the MMAs above have read it
    if (++stage == STAGES) { stage = 0; phase ^= 1; }
  }
  umma_commit(sv.tmem_full_bar);        // accumulator complete
  trace_point(tr, 5);
}

// ---------------------------------------------------------------------------------------------------------
// The generic kernel: 128 x 128 tile, epilogue from a policy class
// ---------------------------------------------------------------------------------------------------------
constexpr int kGemmThreads = 64 + 32 * kEpiWarps;   // 320
constexpr int kAccStages = 2;                       // TMEM accumulator double buffering: 2 x 128 columns

// ew = epilogue warps: 8 (with their 4 KB staging tiles) or 16 (no staging memory: only for epilogues that do not use EpiCtx::stage)
__host__ __device__ constexpr int gemm_persistent_smem_bytes(int stages, int kbs = 1, int bn = kTileN, int ew = kEpiWarps) {
  return stages * kbs * (kABytes + bn * kBlockK * 2) + (ew == kEpiWarps ? kEpiWarps * kEpiStageBytes : 0) + 1024 /*align*/ + 256 /*barriers*/;
}

// Persistent: grid = min(#tiles, #SMs); CTA b walks tiles b, b + grid, ... (n fastest, so neighbouring CTAs share A).
// The TMA producer runs ahead across tile boundaries, the MMA warp alternates between two TMEM accumulator stages,
// and the 8 epilogue warps drain stage i while the tensor core fills stage i ^ 1.
// KBS = k-blocks per pipeline stage.  KBS > 1 takes 3-D tensor maps (make_tmap3): one TMA request then brings KBS k-block tiles of
// an operand.  The TMA unit serves ~2 requests at a time at ~0.4-0.5 k cycles each regardless of their size (tools/tmabench.cu),
// so with 16 KB requests a 128 x 128 x 512 tile takes ~6 k cycles to load against 2 k cycles of MMA; 32 KB requests halve that.
// BN = output columns per tile: 128, or 256 (one UMMA of N = 256 per k-slice: 48 KB of operands per 128 x 256 x 64 block instead of 64 KB for
// two 128 x 128 ones, i.e. 0.75 of the L2 -> SM traffic per FLOP - the large GEMMs of the image encoder are bound by exactly that; the
// two accumulator stages then fill all 512 TMEM columns and every epilogue thread owns 128 columns).  Only epilogues that honour
// EpiCtx::ncols may be instantiated with BN = 256.
// EW = epilogue warps: 8, or 16 (BN = 256 only: four warps per TMEM lane quadrant, 64 columns per thread).  The logits epilogue is bound by
// issue latency - 32 k exponentials, compares and FMAs per tile on two warps per scheduler take 1.6 x the tile's MMA time - so twice the
// warps make the kernel MMA-bound.  Such epilogues get no staging memory (EpiCtx::stage is null).
// MN (bit 0: operand A, bit 1: operand B): that operand is a ROW-major matrix whose rows are the contraction index - A[K, M] or
// B[K, N] - given as a 3-D map (64 columns, K rows, column blocks) with boxes of [64, 64, 2]: one request per k-block lands as two
// [64 K rows][128 B] blocks, which the MMAs read through MN-major descriptors.  MN = 3: the weight-gradient GEMMs, out[M, N] =
// A[K, M]^T * B[K, N], straight from the activations; MN = 2: the data-gradient GEMMs, out[M, N] = A[M, K] * B[K, N], straight from the
// forward weights.  No transposed copies.
template <class Epi, int STAGES, int KBS = 1, int BN = kTileN, int EW = kEpiWarps, int MN = 0>
__global__ void __launch_bounds__(64 + 32 * EW, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, int M, int n_tiles,
            int num_k_blocks, int k_splits, int b_is_static, typename Epi::Params ep) {
  static_assert(BN == 128 || BN == 256, "tile width");
  static_assert(!MN || (KBS == 1 && BN == 128), "MN-major operands: one k-block per stage, 128-wide tiles");
  static_assert(EW == kEpiWarps || (EW == 16 && BN == 256), "epilogue warps");
  constexpr int kSubs = EW / 4;                            // column groups of the tile: 2 or 4
  constexpr int kColsPerThread = BN / kSubs;
  constexpr int kTileN = BN;                               // shadows the namespace constant inside this kernel
  constexpr int kBBytes = BN * kBlockK * 2;
  constexpr int kStageBytes = KBS * (kABytes + kBBytes);   // this kernel's stage: [A: KBS k-blocks][B: KBS k-blocks]
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stages = smem;
  uint8_t* epi_stage = smem + STAGES * kStageBytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(epi_stage + (EW == kEpiWarps ? kEpiWarps * kEpiStageBytes : 0));
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;        // [kAccStages]
  uint64_t* tmem_empty_bar = tmem_full_bar + kAccStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + kAccStages);
  __shared__ int s_trace;

  const int warp = threadIdx.x >> 5;
  const int mn_tiles = n_tiles * ((M + kBlockM - 1) / kBlockM);
  const int total_tiles = mn_tiles * k_splits;                       // split-K: tile t covers k-blocks [kb0, kb1) of (t % mn_tiles)
  const int kb_per_split = (num_k_blocks + k_splits - 1) / k_splits;
  pdl_trigger();
  if (threadIdx.x == 0) { s_trace = trace_begin() ? 1 : 0; trace_point(s_trace != 0, 0); }
  // The B operand (weights) does not depend on the previous kernel: the first pipeline fill's weight halves are requested
  // before griddepcontrol.wait (the whole fill belongs to this CTA's first tile), the activation halves after it.
  const int first_loads = (min(num_k_blocks, kb_per_split) + KBS - 1) / KBS;
  const int early_b = (b_is_static && static_cast<int>(blockIdx.x) < total_tiles) ? min(STAGES, first_loads) : 0;

  if (warp == 0) {
    if (elect_one()) {
      tma_prefetch_desc(&tmap_a);
      tma_prefetch_desc(&tmap_b);
      for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
      for (int a = 0; a < kAccStages; ++a) { mbar_init(&tmem_full_bar[a], 1); mbar_init(&tmem_empty_bar[a], EW); }
      fence_mbar_init();
      if (early_b > 0) {
        const int tt = blockIdx.x % mn_tiles, sp = blockIdx.x / mn_tiles;
        const int n0 = (tt % n_tiles) * kTileN, kb0 = sp * kb_per_split;
        for (int i = 0; i < early_b; ++i) {
          uint8_t* sa = stages + i * kStageBytes;
          mbar_arrive_expect_tx(&full_bar[i], kStageBytes);
          if (KBS == 1) tma_load_2d(sa + kABytes, &tmap_b, &full_bar[i], (kb0 + i) * kBlockK, n0, kEvictLast);
          else tma_load_3d(sa + KBS * kABytes, &tmap_b, &full_bar[i], n0, kb0 + i * KBS, kEvictLast);
        }
      }
    }
  } else if (warp == 1) {
    tmem_alloc<kAccStages * kTileN>(tmem_slot);
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  const bool tr = s_trace != 0;
  pdl_wait();   // everything above (barriers, TMEM, descriptors, first weight tiles) overlapped the previous kernel's tail
  if (threadIdx.x == 0) trace_point(tr, 1);

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0; uint32_t phase = 0;
      int nload = 0;                      // loads issued so far; the B halves of the first `early_b` were issued before the wait
      for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
        const int tt = t % mn_tiles, sp = t / mn_tiles;
        const int m0 = (tt / n_tiles) * kBlockM, n0 = (tt % n_tiles) * kTileN;
        const int kb0 = sp * kb_per_split, kb1 = min(num_k_blocks, kb0 + kb_per_split);
        for (int kb = kb0; kb < kb1; kb += KBS, ++nload) {
          uint8_t* sa = stages + stage * kStageBytes;
          if (nload >= early_b) {
            mbar_wait(&empty_bar[stage], phase ^ 1, 1);
            mbar_arrive_expect_tx(&full_bar[stage], kStageBytes);
          }
          if (MN) {
            if (MN & 1) tma_load_3d_at(sa, &tmap_a, &full_bar[stage], 0, kb * kBlockK, m0 / 64, kEvictNormal);
            else tma_load_2d(sa, &tmap_a, &full_bar[stage], kb * kBlockK, m0, kEvictNormal);
            if (MN & 2) tma_load_3d_at(sa + kABytes, &tmap_b, &full_bar[stage], 0, kb * kBlockK, n0 / 64, (MN & 1) ? kEvictNormal : kEvictLast);
            else tma_load_2d(sa + kABytes, &tmap_b, &full_bar[stage], kb * kBlockK, n0, kEvictLast);
          } else if (KBS == 1) {
            tma_load_2d(sa, &tmap_a, &full_bar[stage], kb * kBlockK, m0, kEvictNormal);
            if (nload >= early_b) tma_load_2d(sa + kABytes, &tmap_b, &full_bar[stage], kb * kBlockK, n0, kEvictLast);
          } else {
            tma_load_3d(sa, &tmap_a, &full_bar[stage], m0, kb, kEvictNormal);
            if (nload >= early_b) tma_load_3d(sa + KBS * kABytes, &tmap_b, &full_bar[stage], n0, kb, kEvictLast);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
      trace_point(tr, 3);
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t kIdesc = MN ? umma_idesc_bf16_f32_mn(kBlockM, kTileN, (MN & 1) != 0, (MN & 2) != 0) : umma_idesc_bf16_f32(kBlockM, kTileN);
      int stage = 0; uint32_t phase = 0;
      int i = 0;
      for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++i) {
        const int as = i & 1;
        mbar_wait(&tmem_empty_bar[as], ((i >> 1) & 1) ^ 1, 9);   // epilogue has drained this accumulator stage
        tc_fence_after_sync();
        const uint32_t acc = tmem_base + as * kTileN;
        const int sp = t / mn_tiles;
        const int kb0 = sp * kb_per_split, kb1 = min(num_k_blocks, kb0 + kb_per_split);
        for (int kb = kb0; kb < kb1; kb += KBS) {
          mbar_wait(&full_bar[stage], phase, 2);
          if (i == 0 && kb == kb0) trace_point(tr, 4);
          tc_fence_after_sync();
          const uint32_t sa = smem_u32(stages + stage * kStageBytes);
          const uint32_t sb = sa + KBS * kABytes;
          if (MN) {
#pragma unroll
            for (int k = 0; k < kBlockK / kUmmaK; ++k)     // 16 K rows = two 1024-byte groups of every 64-element block
              umma_bf16_ss(acc, (MN & 1) ? umma_desc_sw128_mnmajor(sa + k * (kUmmaK * 128), kBlockK * 128) : umma_desc_sw128_kmajor(sa + k * (kUmmaK * 2)),
                           (MN & 2) ? umma_desc_sw128_mnmajor(sb + k * (kUmmaK * 128), kBlockK * 128) : umma_desc_sw128_kmajor(sb + k * (kUmmaK * 2)),
                           kIdesc, (kb > kb0 || k != 0) ? 1u : 0u);
          } else {
#pragma unroll
            for (int j = 0; j < KBS; ++j)
#pragma unroll
              for (int k = 0; k < kBlockK / kUmmaK; ++k)
                umma_bf16_ss(acc, umma_desc_sw128_kmajor(sa + j * kABytes + k * (kUmmaK * 2)),
                             umma_desc_sw128_kmajor(sb + j * kBBytes + k * (kUmmaK * 2)), kIdesc, (kb > kb0 || (j | k) != 0) ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tmem_full_bar[as]);
        if (i == 0) trace_point(tr, 5);
      }
    }
  } else {
    const int ew = warp - 2;
    const int quad = warp & 3;           // TMEM lane quadrant this warp may read
    const int half = ew >> 2;            // which column group of the tile
    const int lane = static_cast<int>(lane_id());
    int i = 0;
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++i) {
      const int as = i & 1;
      const int tt = t % mn_tiles;
      const int m0 = (tt / n_tiles) * kBlockM, nt = tt % n_tiles;
      mbar_wait(&tmem_full_bar[as], (i >> 1) & 1, 3);
      if (i == 0 && threadIdx.x == 64) trace_point(tr, 6);
      if (i < 8 && threadIdx.x == 64) trace_point(tr, 16 + 2 * i);   // per-tile: accumulator ready / epilogue done
      tc_fence_after_sync();
      EpiCtx c;
      c.tmem_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * kTileN + half * kColsPerThread;
      c.warp_row0 = m0 + quad * 32;
      c.row = c.warp_row0 + lane;
      c.n0 = nt * kTileN + half * kColsPerThread;
      c.ncols = kColsPerThread;
      c.M = M;
      c.part = nt * (kTileN / 64) + half * (kColsPerThread / 64);   // index of the thread's first 64-column slice
      c.stage = EW == kEpiWarps ? epi_stage + ew * kEpiStageBytes : nullptr;
      uint64_t* rel = &tmem_empty_bar[as];
      Epi::run(ep, c, [rel, lane]() {
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(rel);
      });
      if (i == 0 && threadIdx.x == 64) trace_point(tr, 8);
      if (i < 8 && threadIdx.x == 64) trace_point(tr, 17 + 2 * i);
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (threadIdx.x == 0) trace_point(tr, 10);
  if (warp == 1) tmem_dealloc<kAccStages * kTileN>(tmem_base);
}

// ---------------------------------------------------------------------------------------------------------
// Weight-stationary variant of the persistent kernel for GEMMs with few column tiles and K = 512 (the decoder's QKV projection: 12 column
// tiles, 32+ row blocks).  The generic kernel moves 256 KB of operands per 128 x 128 x 512 tile - 4.4 k cycles at what the L2 delivers when all
// SMs pull, against 2.1 k cycles of MMA - and half of those bytes are the same 128 KB weight tile every time.  Here CTA b owns ONE column
// tile (b % n_tiles) for the whole launch: its weight tile (8 k-blocks, 128 KB) is loaded once - before griddepcontrol.wait, i.e. under the
// previous kernel's tail, since weights do not depend on it - and stays in shared memory; the CTA then walks the row blocks
// b / n_tiles, + gridDim.x / n_tiles, ... streaming only the activation tiles through three 32 KB stages.  Grid = n_tiles x floor(#SMs / n_tiles).
// Same accumulation order as gemm_kernel: results are bit-identical.
// ---------------------------------------------------------------------------------------------------------
constexpr int kWsKb = 8;                                   // k-blocks of the stationary weight tile (K = 512)
constexpr int kWsABytes = 2 * kABytes;                     // activation stage: two k-blocks (32 KB)
constexpr int kWsStages = 3;                               // activation stages
// Three activation stages and no epilogue staging tile: q / K / V leave straight from the registers as 256-bit stores (st.global.v8.b32: a
// thread's 64 columns are four full 32-byte sectors of its row).  With 16-byte stores - half-sector writes - the third stage cost more than
// it gained (5.5 k instead of 4.5 k cycles per tile); with full sectors the QKV class dropped from 1.10 to 0.99 ms per decode against two
// stages plus the staging tile.
__host__ __device__ constexpr int gemm_ws_smem_bytes() { return kWsKb * kBBytes + kWsStages * kWsABytes + 1024 + 256; }

template <class Epi>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_ws_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, int M, int n_tiles, int b_is_static,
               typename Epi::Params ep) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* b_smem = smem;                                   // [8 k-blocks][128 rows x 128 B]
  uint8_t* a_ring = b_smem + kWsKb * kBBytes;
  uint64_t* b_full = reinterpret_cast<uint64_t*>(a_ring + kWsStages * kWsABytes);   // [4] one per pair of k-blocks
  uint64_t* a_full = b_full + kWsKb / 2;
  uint64_t* a_empty = a_full + kWsStages;
  uint64_t* tmem_full_bar = a_empty + kWsStages;
  uint64_t* tmem_empty_bar = tmem_full_bar + kAccStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + kAccStages);
  __shared__ int s_trace;

  const int warp = threadIdx.x >> 5;
  const int m_blocks = (M + kBlockM - 1) / kBlockM;
  const int nt = blockIdx.x % n_tiles, g0 = blockIdx.x / n_tiles, gstep = gridDim.x / n_tiles;
  const int n0 = nt * kTileN;
  pdl_trigger();
  if (threadIdx.x == 0) { s_trace = trace_begin() ? 1 : 0; trace_point(s_trace != 0, 0); }

  if (warp == 0) {
    if (elect_one()) {
      tma_prefetch_desc(&tmap_a);
      tma_prefetch_desc(&tmap_b);
      for (int j = 0; j < kWsKb / 2; ++j) mbar_init(&b_full[j], 1);
      for (int s = 0; s < kWsStages; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], 1); }
      for (int a = 0; a < kAccStages; ++a) { mbar_init(&tmem_full_bar[a], 1); mbar_init(&tmem_empty_bar[a], kEpiWarps); }
      fence_mbar_init();
      if (b_is_static && g0 < m_blocks) {
        for (int j = 0; j < kWsKb / 2; ++j) {
          mbar_arrive_expect_tx(&b_full[j], 2 * kBBytes);
          tma_load_3d(b_smem + j * 2 * kBBytes, &tmap_b, &b_full[j], n0, 2 * j, kEvictLast);
        }
      }
    }
  } else if (warp == 1) {
    tmem_alloc<kAccStages * kTileN>(tmem_slot);
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  const bool tr = s_trace != 0;
  pdl_wait();
  if (threadIdx.x == 0) trace_point(tr, 1);

  if (warp == 0) {
    if (elect_one()) {
      if (!b_is_static && g0 < m_blocks) {
        for (int j = 0; j < kWsKb / 2; ++j) {
          mbar_arrive_expect_tx(&b_full[j], 2 * kBBytes);
          tma_load_3d(b_smem + j * 2 * kBBytes, &tmap_b, &b_full[j], n0, 2 * j, kEvictLast);
        }
      }
      int stage = 0; uint32_t phase = 0;
      for (int mb = g0; mb < m_blocks; mb += gstep) {
        for (int j = 0; j < kWsKb / 2; ++j) {
          mbar_wait(&a_empty[stage], phase ^ 1, 1);
          mbar_arrive_expect_tx(&a_full[stage], kWsABytes);
          tma_load_3d(a_ring + stage * kWsABytes, &tmap_a, &a_full[stage], mb * kBlockM, 2 * j, kEvictNormal);
          if (++stage == kWsStages) { stage = 0; phase ^= 1; }
        }
      }
      trace_point(tr, 3);
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t kIdesc = umma_idesc_bf16_f32(kBlockM, kTileN);
      int stage = 0; uint32_t phase = 0;
      int i = 0;
      for (int mb = g0; mb < m_blocks; mb += gstep, ++i) {
        const int as = i & 1;
        mbar_wait(&tmem_empty_bar[as], ((i >> 1) & 1) ^ 1, 9);
        tc_fence_after_sync();
        const uint32_t acc = tmem_base + as * kTileN;
        for (int j = 0; j < kWsKb / 2; ++j) {
          if (i == 0) mbar_wait(&b_full[j], 0, 4);
          mbar_wait(&a_full[stage], phase, 2);
          if (i == 0 && j == 0) trace_point(tr, 4);
          tc_fence_after_sync();
          const uint32_t sa = smem_u32(a_ring + stage * kWsABytes);
          const uint32_t sb = smem_u32(b_smem + j * 2 * kBBytes);
#pragma unroll
          for (int jj = 0; jj < 2; ++jj)
#pragma unroll
            for (int k = 0; k < kBlockK / kUmmaK; ++k)
              umma_bf16_ss(acc, umma_desc_sw128_kmajor(sa + jj * kABytes + k * (kUmmaK * 2)),
                           umma_desc_sw128_kmajor(sb + jj * kBBytes + k * (kUmmaK * 2)), kIdesc, (j | jj | k) != 0 ? 1u : 0u);
          umma_commit(&a_empty[stage]);
          if (++stage == kWsStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tmem_full_bar[as]);
        if (i == 0) trace_point(tr, 5);
      }
    }
  } else {
    const int ew = warp - 2;
    const int quad = warp & 3;
    const int half = ew >> 2;
    const int lane = static_cast<int>(lane_id());
    int i = 0;
    for (int mb = g0; mb < m_blocks; mb += gstep, ++i) {
      const int as = i & 1;
      mbar_wait(&tmem_full_bar[as], (i >> 1) & 1, 3);
      if (i < 8 && threadIdx.x == 64) trace_point(tr, 16 + 2 * i);
      tc_fence_after_sync();
      EpiCtx c;
      c.tmem_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * kTileN + half * (kTileN / 2);
      c.warp_row0 = mb * kBlockM + quad * 32;
      c.row = c.warp_row0 + lane;
      c.n0 = n0 + half * (kTileN / 2);
      c.ncols = kTileN / 2;
      c.M = M;
      c.part = nt * 2 + half;
      c.stage = nullptr;
      uint64_t* rel = &tmem_empty_bar[as];
      Epi::run(ep, c, [rel, lane]() {
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(rel);
      });
      if (i < 8 && threadIdx.x == 64) trace_point(tr, 17 + 2 * i);
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (threadIdx.x == 0) trace_point(tr, 10);
  if (warp == 1) tmem_dealloc<kAccStages * kTileN>(tmem_base);
}

// ---------------------------------------------------------------------------------------------------------
// Full-row GEMM + residual + LayerNorm, split over a 4-CTA cluster.
//
// The 512-wide output row of a 128-row tile is split across the 4 CTAs of a cluster (128 columns each), so a
// decode step over 4096 sequences fills 128 SMs instead of 32.  Each epilogue thread keeps its 128 row values in
// registers (single pass): the residual slice is prefetched while the MMAs run, the accumulator is added from
// TMEM, the per-row (sum, sum of squares) partials are exchanged through distributed shared memory, and every
// CTA then normalises and writes its own 128 columns of x (fp32, blocked layout) and LayerNorm(x) (bf16).
// Used for out-proj, FFN2 and the prefix projection (positions instead of a residual).
// ---------------------------------------------------------------------------------------------------------
constexpr int kRowBN = kTileN;
constexpr int kRowCluster = kE / kRowBN;  // 4
constexpr int kRowEpiWarps = 8;           // two warps per TMEM lane quadrant, 64 columns per thread
constexpr int kRowThreads = 64 + 32 * kRowEpiWarps;
constexpr int kRowCols = kRowBN / 2;      // columns per epilogue thread
constexpr int kRowStagePitch = kRowCols * 2 + 16;  // staged bf16 row of 64 columns: 128 B + 16 B pad
constexpr int kFfnDim = 128;              // FFN hidden size (config/train.yaml: feedfwd_scale 1/4)

struct RowParams {
  float* x;               // blocked fp32 residual stream, output
  const float* x_in;      // residual input (nullptr: same buffer as x, i.e. in place; ignored in prefix mode)
  __nv_bfloat16* xn;      // [rows, 512] bf16 LayerNorm output
  const float* gain;      // LayerNorm weight of the *consumer* (norm2 / next layer's norm1 / final norm)
  const float* pos;       // prefix mode: positional table [smax, 512]; else nullptr
  int prefix_rep;         // prefix mode: sequences per embedding (multi-target M or 1)
  int prefix_rows_per_seq;// prefix mode: rows per sequence in x / xn (P for decode prefill, S for teacher forcing)
  int remap_rows_in;      // xn row remap (0 = identity): rows per sequence in,
  int remap_skip;         //   leading rows per sequence to drop,
  int remap_rows_out;     //   rows per sequence out
  float eps;
  DropCfg drop;           // training: dropout on the GEMM result before the residual add (thresh 0 = off; not in prefix mode)
  uint32_t drop_site;
};

__host__ __device__ constexpr int rowln_smem_bytes(int stages, bool fuse_ffn) {
  return stages * kStageBytes + (fuse_ffn ? 2 * 2 * kABytes : 0) + 1024 /*align*/ + 256 /*barriers*/ + 2 * 128 * 8 /*stats*/ + kRowBN * 4 /*gain*/;
}

// FUSE_FFN = false:  x += A * W^T (tmap_a, tmap_b)                          -> LayerNorm      (out-proj, prefix projection)
// FUSE_FFN = true :  h = gelu(A * W1^T) (tmap_a = LN2(x), tmap_w1), kept in shared memory as the next A operand;
//                    x += h * W2^T (tmap_b = this CTA's 128 rows of W2)     -> LayerNorm      (whole feed-forward block)
// In the fused variant every CTA of the cluster recomputes the full 128 x 128 hidden tile (4x redundant FFN1, 2048
// tensor cycles) - far cheaper than a separate kernel plus a global round trip of h.
// FFN = 2 (split hidden tile): CTA r of the cluster computes only hidden columns [32 r, 32 r + 32) (tmap_w1 has a 32-row box),
// applies GELU and stores the bf16 values into the h operand of all four CTAs through distributed shared memory; one cluster
// barrier later every CTA holds the complete 128 x 128 hidden tile.  4x less GELU work, W1 traffic and FFN1 MMA per CTA
// (the phase trace of the redundant variant shows 5.1 k cycles of GELU per CTA, profiles/r01_phase_trace_v6.txt).
// DROP (training only): dropout on the GEMM result before the residual add (a separate instantiation: the mask arithmetic in the
// accumulation loop costs the inference kernels 0.5 ms per decode when it is merely branched around).
template <int STAGES, int FFN, bool DROP = false>
__global__ void __cluster_dims__(kRowCluster, 1, 1) __launch_bounds__(kRowThreads, 1)
gemm_rowln_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                  const __grid_constant__ CUtensorMap tmap_w1, int M, int num_k_blocks, RowParams ep) {
  constexpr bool FUSE_FFN = FFN != 0;
  constexpr bool SPLIT_H = FFN == 2;
  constexpr int kHSplit = kFfnDim / kRowCluster;                                  // 32 hidden columns per CTA
  constexpr uint32_t kStageTx = SPLIT_H ? kABytes + kHSplit * kBlockK * 2 : kStageBytes;
  constexpr int BN = kRowBN;
  constexpr uint32_t kTmemCols = FUSE_FFN ? 256 : 128;
  constexpr uint32_t kIdesc = umma_idesc_bf16_f32(kBlockM, BN);
  extern __shared__ uint8_t smem_raw[];
  const GemmSmemView sv0 = carve_smem<STAGES>(smem_raw);
  // layout: [stages][h: 2 k-blocks][w2: 2 k-blocks][barriers][stats][gain]
  uint8_t* h_smem = sv0.stages + STAGES * kStageBytes;
  uint8_t* w2_smem = h_smem + (FUSE_FFN ? 2 * kABytes : 0);
  uint8_t* after = w2_smem + (FUSE_FFN ? 2 * kABytes : 0);
  GemmSmemView sv = sv0;
  sv.full_bar = reinterpret_cast<uint64_t*>(after);
  sv.empty_bar = sv.full_bar + STAGES;
  sv.tmem_full_bar = sv.empty_bar + STAGES;
  uint64_t* w2_full_bar = sv.tmem_full_bar + 1;
  uint64_t* h_ready_bar = sv.tmem_full_bar + 2;
  uint64_t* tmem_full2_bar = sv.tmem_full_bar + 3;
  sv.tmem_slot = reinterpret_cast<uint32_t*>(sv.tmem_full_bar + 4);
  float2* s_stats = reinterpret_cast<float2*>(after + 256);                  // [2 halves][128 rows] (sum, sumsq)
  float* s_gain = reinterpret_cast<float*>(after + 256 + 2 * 128 * 8);       // [128]
  __shared__ int s_trace;

  const int warp = threadIdx.x >> 5;
  const int lane = static_cast<int>(lane_id());
  const int m0 = blockIdx.y * kBlockM;
  const int n0 = blockIdx.x * BN;               // column in the [*, P*512] / [*, 512] output
  const uint32_t crank = cluster_ctarank();     // == blockIdx.x % 4
  const int coff = static_cast<int>(crank) * BN;  // column offset inside the 512-wide row
  const int ptok = blockIdx.x / kRowCluster;    // prefix mode: which prefix position
  pdl_trigger();
  if (threadIdx.x == 0) { s_trace = trace_begin() ? 1 : 0; trace_point(s_trace != 0, 0); }

  const CUtensorMap* tb1 = FUSE_FFN ? &tmap_w1 : &tmap_b;   // B operand of the first (pipelined) GEMM
  const int bn0 = SPLIT_H ? static_cast<int>(crank) * kHSplit : (FUSE_FFN ? 0 : n0);   // its row offset (W1 has exactly 128 rows)
  if (warp == 0) {
    if (elect_one()) {
      tma_prefetch_desc(&tmap_a);
      tma_prefetch_desc(tb1);
      if (FUSE_FFN) {
        mbar_init(w2_full_bar, 1);
        mbar_init(h_ready_bar, kRowEpiWarps);
        mbar_init(tmem_full2_bar, 1);
      }
      // weights do not depend on the previous kernel: start their loads, then wait for it, then load activations
      for (int st = 0; st < STAGES; ++st) { mbar_init(&sv.full_bar[st], 1); mbar_init(&sv.empty_bar[st], 1); }
      mbar_init(sv.tmem_full_bar, 1);
      fence_mbar_init();
      const int pre = num_k_blocks < STAGES ? num_k_blocks : STAGES;
      for (int kb = 0; kb < pre; ++kb) {
        mbar_arrive_expect_tx(&sv.full_bar[kb], kStageTx);
        tma_load_2d(sv.stages + kb * kStageBytes + kABytes, tb1, &sv.full_bar[kb], kb * kBlockK, bn0, kEvictLast);
      }
      if (FUSE_FFN) {   // this CTA's 128 rows of W2, both k-blocks
        mbar_arrive_expect_tx(w2_full_bar, 2 * kBBytes);
        tma_load_2d(w2_smem, &tmap_b, w2_full_bar, 0, n0, kEvictLast);
        tma_load_2d(w2_smem + kBBytes, &tmap_b, w2_full_bar, kBlockK, n0, kEvictLast);
      }
      pdl_wait();
      for (int kb = 0; kb < pre; ++kb)
        tma_load_2d(sv.stages + kb * kStageBytes, &tmap_a, &sv.full_bar[kb], kb * kBlockK, m0, kEvictNormal);
    }
  } else if (warp == 1) {
    tmem_alloc<kTmemCols>(sv.tmem_slot);
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *sv.tmem_slot;
  const bool tr = s_trace != 0;
  pdl_wait();
  if (threadIdx.x == 0) trace_point(tr, 1);

  // second GEMM of the fused feed-forward block: x_delta = h * W2^T from shared memory (issued by one thread of warp 1)
  auto issue_ffn2 = [&]() {
    mbar_wait(w2_full_bar, 0, 6);
    if (!SPLIT_H) mbar_wait(h_ready_bar, 0, 7);
    tc_fence_after_sync();
    const uint32_t sa = smem_u32(h_smem), sb = smem_u32(w2_smem);
#pragma unroll
    for (int kb = 0; kb < kFfnDim / kBlockK; ++kb)
#pragma unroll
      for (int k = 0; k < kBlockK / kUmmaK; ++k)
        umma_bf16_ss(tmem_base + BN, umma_desc_sw128_kmajor(sa + kb * kABytes + k * (kUmmaK * 2)),
                     umma_desc_sw128_kmajor(sb + kb * kBBytes + k * (kUmmaK * 2)), kIdesc, (kb | k) != 0 ? 1u : 0u);
    umma_commit(tmem_full2_bar);
    trace_point(tr, 12);
  };
  if (warp == 0) {
    if (elect_one()) {
      producer_rest<STAGES>(sv, &tmap_a, tb1, num_k_blocks, m0, bn0, kStageTx);
      trace_point(tr, 3);
    }
  } else if (warp == 1) {
    if (elect_one()) {
      mma_mainloop<STAGES, SPLIT_H ? kHSplit : kTileN>(sv, tmem_base, num_k_blocks, tr);
      if (FUSE_FFN && !SPLIT_H) issue_ffn2();
    }
  }

  // ---- epilogue part 1 (warps 2..9): residual prefetch (+ fused FFN hidden tile) + accumulator + partial row statistics
  const bool is_epi = warp >= 2;
  const int ew = warp - 2;
  const int quad = warp & 3;
  const int half = ew >> 2;                       // which 64 of this CTA's 128 columns
  const int row_in_tile = quad * 32 + lane;
  const int row = m0 + row_in_tile;
  const int c0 = coff + half * kRowCols;          // first column (within the 512-wide row) this thread owns
  const bool prefix = ep.pos != nullptr;
  const int reps = prefix ? ep.prefix_rep : 1;
  float r[kRowCols];
  if (is_epi) {
    if (ew < 4) s_gain[threadIdx.x - 64] = __ldg(ep.gain + coff + (threadIdx.x - 64));
    if (row < M) {
      if (prefix) {
        const float4* p4 = reinterpret_cast<const float4*>(ep.pos + static_cast<size_t>(ptok) * kE + c0);
#pragma unroll
        for (int q = 0; q < kRowCols / 4; ++q) { const float4 t = __ldg(p4 + q); r[q * 4] = t.x; r[q * 4 + 1] = t.y; r[q * 4 + 2] = t.z; r[q * 4 + 3] = t.w; }
      } else {
#pragma unroll
        for (int q = 0; q < kRowCols / 4; ++q) {
          const float4 t = *reinterpret_cast<const float4*>((ep.x_in != nullptr ? ep.x_in : ep.x) + xblk_off(row, (c0 >> 2) + q));
          r[q * 4] = t.x; r[q * 4 + 1] = t.y; r[q * 4 + 2] = t.z; r[q * 4 + 3] = t.w;
        }
      }
    } else {
#pragma unroll
      for (int i = 0; i < kRowCols; ++i) r[i] = 0.f;
    }
    if (threadIdx.x == 64) trace_point(tr, 11);
    const uint32_t tmem_lane = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    mbar_wait(sv.tmem_full_bar, 0, 3);
    if (threadIdx.x == 64) trace_point(tr, 6);
    tc_fence_after_sync();
    if (SPLIT_H) {
      // this CTA's 32 hidden columns: the thread's 16 (two 16-byte chunks of the row) go to the h operand of all four CTAs
      float v[16];
      tmem_ld_32x16(tmem_lane + half * 16, v);
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = gelu_fast(v[j]);
      const int hcol = static_cast<int>(crank) * kHSplit + half * 16;              // first hidden column of this thread
      uint8_t* hrow = h_smem + (hcol >> 6) * kABytes + row_in_tile * 128;
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int chunk = ((hcol & 63) >> 3) + q;
        const uint4 pk = make_uint4(pack_bf16x2(v[q * 8 + 0], v[q * 8 + 1]), pack_bf16x2(v[q * 8 + 2], v[q * 8 + 3]),
                                    pack_bf16x2(v[q * 8 + 4], v[q * 8 + 5]), pack_bf16x2(v[q * 8 + 6], v[q * 8 + 7]));
        uint8_t* dst = hrow + ((chunk ^ (row_in_tile & 7)) << 4);
#pragma unroll
        for (uint32_t pr = 0; pr < kRowCluster; ++pr) dsmem_st_v4(dsmem_addr(dst, pr), pk);
      }
      fence_proxy_async_any();       // generic-proxy writes into the peers' shared memory -> visible to their tensor cores
      tc_fence_before_sync();
      if (threadIdx.x == 64) trace_point(tr, 13);
    } else if (FUSE_FFN) {
      // hidden tile: gelu(acc1) -> bf16 -> K-major 128B-swizzled A operand of the second GEMM; this thread's 64 columns
      // are exactly k-block `half`, its row is 128 B there, 16-byte chunk c lands at chunk (c ^ (row & 7)).
      uint8_t* hrow = h_smem + half * kABytes + row_in_tile * 128;
#pragma unroll
      for (int c = 0; c < kRowCols / 16; ++c) {
        float v[16];
        tmem_ld_32x16(tmem_lane + half * kRowCols + c * 16, v);
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = gelu_fast(v[j]);
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const int chunk = c * 2 + q;
          *reinterpret_cast<uint4*>(hrow + ((chunk ^ (row_in_tile & 7)) << 4)) =
              make_uint4(pack_bf16x2(v[q * 8 + 0], v[q * 8 + 1]), pack_bf16x2(v[q * 8 + 2], v[q * 8 + 3]),
                         pack_bf16x2(v[q * 8 + 4], v[q * 8 + 5]), pack_bf16x2(v[q * 8 + 6], v[q * 8 + 7]));
        }
      }
      fence_proxy_async_smem();      // generic-proxy smem writes -> visible to the tensor core's async-proxy reads
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(h_ready_bar);
      if (threadIdx.x == 64) trace_point(tr, 13);
      mbar_wait(tmem_full2_bar, 0, 8);
      tc_fence_after_sync();
    }
  }
  if (SPLIT_H) {
    __syncwarp();
    cluster_sync_all();              // the whole hidden tile now sits in every CTA's h operand
    if (warp == 1) {
      if (elect_one()) { fence_proxy_async_any(); issue_ffn2(); }
    }
    __syncwarp();
    if (is_epi) {
      mbar_wait(tmem_full2_bar, 0, 8);
      tc_fence_after_sync();
    }
  }
  if (is_epi) {
    const uint32_t tmem_lane = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    const uint32_t acc = tmem_lane + (FUSE_FFN ? BN : 0) + half * kRowCols;
    float sum = 0.f, sumsq = 0.f;
#pragma unroll
    for (int c = 0; c < kRowCols / 16; ++c) {
      float v[16];
      tmem_ld_32x16(acc + c * 16, v);
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        float b = v[j];
        if (DROP) b *= drop_factor(ep.drop, ep.drop_site, static_cast<uint32_t>(row) * kE + static_cast<uint32_t>(c0 + c * 16 + j));
        const float t = r[c * 16 + j] + b;
        r[c * 16 + j] = t;
        sum += t;
        sumsq = fmaf(t, t, sumsq);
      }
    }
    s_stats[half * 128 + row_in_tile] = make_float2(sum, sumsq);
    // (measured: issuing the 64 KB of residual stores here, before the cluster barrier, is SLOWER - 6.01 vs 5.92 ms per decode;
    //  barrier.cluster.arrive.release has to wait for them)
    if (threadIdx.x == 64) trace_point(tr, 7);
  }
  __syncwarp();
  cluster_sync_all();   // every thread of the 4 CTAs: partial statistics are now visible cluster-wide
  if (threadIdx.x == 64) trace_point(tr, 8);

  // ---- epilogue part 2: combine the 8 partials (fixed order -> identical mean/rstd everywhere), normalise, store
  if (is_epi) {
    float mean = 0.f, rstd = 0.f;
    if (row < M) {
      float2 part[kRowCluster * 2];   // issue all remote loads first, then reduce in a fixed order
#pragma unroll
      for (uint32_t pr = 0; pr < kRowCluster; ++pr) {
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) part[pr * 2 + hh] = dsmem_ld_f32x2_addr(dsmem_addr(&s_stats[hh * 128 + row_in_tile], pr));
      }
      float sum = 0.f, sumsq = 0.f;
#pragma unroll
      for (int i = 0; i < kRowCluster * 2; ++i) { sum += part[i].x; sumsq += part[i].y; }
      mean = sum * (1.0f / kE);
      rstd = rsqrtf(fmaxf(sumsq * (1.0f / kE) - mean * mean, 0.f) + ep.eps);
    }
    // LayerNorm output -> warp-private staging (drained pipeline stages) -> coalesced row-major stores
    uint8_t* stage = sv.stages + ew * (32 * kRowStagePitch);
    {
      uint4* d = reinterpret_cast<uint4*>(stage + lane * kRowStagePitch);
#pragma unroll
      for (int q = 0; q < kRowCols / 8; ++q) {
        float y[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) y[i] = (r[q * 8 + i] - mean) * rstd * s_gain[half * kRowCols + q * 8 + i];
        d[q] = make_uint4(pack_bf16x2(y[0], y[1]), pack_bf16x2(y[2], y[3]), pack_bf16x2(y[4], y[5]), pack_bf16x2(y[6], y[7]));
      }
    }
    const int warp_row0 = m0 + quad * 32;
    for (int j = 0; j < reps; ++j) {
      if (row < M) {
        const int orow = prefix ? ((row * reps + j) * ep.prefix_rows_per_seq + ptok) : row;
#pragma unroll
        for (int q = 0; q < kRowCols / 4; ++q)
          *reinterpret_cast<float4*>(ep.x + xblk_off(orow, (c0 >> 2) + q)) = make_float4(r[q * 4], r[q * 4 + 1], r[q * 4 + 2], r[q * 4 + 3]);
      }
      // 32 rows x 128 B: per instruction the lanes cover 4 rows x 128 contiguous bytes
      __syncwarp();
      const int sub = lane >> 3, chunk = lane & 7;
#pragma unroll 4
      for (int i = 0; i < 8; ++i) {
        const int rr = i * 4 + sub;
        const int grow = warp_row0 + rr;
        if (grow < M) {
          const int orow = prefix ? ((grow * reps + j) * ep.prefix_rows_per_seq + ptok) : grow;
          int nrow = orow;
          bool keep = true;
          if (ep.remap_rows_in > 0) {
            const int seq = orow / ep.remap_rows_in;
            const int k = orow - seq * ep.remap_rows_in;
            keep = k >= ep.remap_skip;
            nrow = seq * ep.remap_rows_out + (k - ep.remap_skip);
          }
          if (keep)
            *reinterpret_cast<uint4*>(ep.xn + static_cast<size_t>(nrow) * kE + c0 + chunk * 8) =
                *reinterpret_cast<const uint4*>(stage + rr * kRowStagePitch + chunk * 16);
        }
      }
      __syncwarp();
    }
  }

  if (threadIdx.x == 64) trace_point(tr, 9);
  tc_fence_before_sync();
  __syncwarp();
  cluster_sync_relaxed();   // peers may still be reading this CTA's s_stats; no data hand-over, so no fence
  if (threadIdx.x == 0) trace_point(tr, 10);
  if (warp == 1) tmem_dealloc<kTmemCols>(tmem_base);
}

// ---------------------------------------------------------------------------------------------------------
// Attention output -> next layer's LayerNorm rows in ONE cluster kernel (decode path): out-proj + residual + LN2, then the whole
// feed-forward block + residual + LN, without the round trip of x_mid (fp32) and LN2(x_mid) (bf16) through L2 that the two separate
// row kernels need - 12 MB of stores at the L2's ~5 TB/s write rate plus a 128 KB TMA reload per CTA and one kernel ramp per layer.
//   phase A  acc0 = ao * Wo^T (this CTA's 128 columns, pipelined over K = 512);  r = x + acc0;  LN2 statistics over the cluster
//   hand-over  y = LN2(r) in bf16: the thread's 64 columns are exactly one 128-byte row of k-block (2 * rank + half) of the K-major
//            swizzled A operand of FFN1, and are stored into the operand buffer of all four CTAs through DSMEM.  The buffer is the
//            out-proj ring itself (dead once every CTA's phase-A MMAs have completed, which the statistics barrier guarantees).
//   phase B  acc1 = y * W1[32 r : 32 r + 32]^T (UMMA N = 32, A resident);  GELU;  the CTA's 8 KB of hidden columns go to the peers as bulk
//            copies too, and every CTA assembles the swizzled FFN2 operand locally (in the W1 region, dead by then)
//   phase C  acc2 = h * W2^T;  r += acc2;  LN statistics over the cluster;  store x (fp32) and LayerNorm(x) (bf16)
// The residual values r never leave the registers between the two LayerNorms.  Results are bit-identical to the separate kernels.
// ---------------------------------------------------------------------------------------------------------
constexpr int kFbRing = 4;      // 32 KB stages that later hold the FFN1 A operand (128 KB)
constexpr int kFbStages = 7;    // phase-A pipeline depth: the W1 / W2 / h regions (3 x 32 KB) are idle during phase A and serve as stages 4..6,
                                // so 7 of the 8 k-block loads are in flight at once; W1 and W2 are loaded once stages 4 and 5 have been consumed
__host__ __device__ constexpr int outproj_ffn_smem_bytes() {
  return kFbRing * kStageBytes /*ring = FFN1 A operand*/ + (kFfnDim / kRowCluster) * kE * 2 /*W1 slice*/ + 2 * kBBytes /*W2*/ + 2 * kABytes /*h*/ +
         1024 /*align*/ + 256 /*barriers*/ + 2 * kRowBN * 4 /*gains*/;
}
static_assert((kFfnDim / kRowCluster) * kE * 2 == kStageBytes && 2 * kBBytes == kStageBytes && 2 * kABytes == kStageBytes, "regions double as pipeline stages");
struct FusedBlockParams {
  float* x;                 // blocked fp32 residual stream, in and out (in place)
  __nv_bfloat16* xn;        // [rows, 512] LayerNorm output of the block (next layer's LN1 / final LN)
  const float* gain_mid;    // LN2 weight
  const float* gain_out;    // weight of the LayerNorm that follows the block
  int remap_rows_in, remap_skip, remap_rows_out;   // xn row remap of the last layer (0 = identity)
  float eps;
};

__global__ void __cluster_dims__(kRowCluster, 1, 1) __launch_bounds__(kRowThreads, 1)
outproj_ffn_kernel(const __grid_constant__ CUtensorMap tmap_ao, const __grid_constant__ CUtensorMap tmap_wo, const __grid_constant__ CUtensorMap tmap_w1q,
                   const __grid_constant__ CUtensorMap tmap_w2, int M, FusedBlockParams ep) {
  constexpr int BN = kRowBN;
  constexpr int kHSplit = kFfnDim / kRowCluster;              // 32 hidden columns per CTA
  constexpr int kW1kb = kHSplit * kBlockK * 2;                // bytes of one k-block of the W1 slice: 4 KB
  constexpr uint32_t kIdesc = umma_idesc_bf16_f32(kBlockM, BN);
  constexpr uint32_t kIdescH = umma_idesc_bf16_f32(kBlockM, kHSplit);
  constexpr int kNkb = kE / kBlockK;                          // 8
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* ring = smem;                                       // phase A pipeline; afterwards the 8 k-block tiles of LN2(x_mid)
  uint8_t* w1_smem = ring + kFbRing * kStageBytes;
  uint8_t* w2_smem = w1_smem + kNkb * kW1kb;
  uint8_t* h_smem = w2_smem + 2 * kBBytes;
  uint8_t* after = h_smem + 2 * kABytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(after);
  uint64_t* empty_bar = full_bar + kFbStages;
  uint64_t* tmem_full0 = empty_bar + kFbStages;
  uint64_t* w1_full = tmem_full0 + 1;
  uint64_t* w2_full = tmem_full0 + 2;
  uint64_t* tmem_full1 = tmem_full0 + 3;
  uint64_t* tmem_full2 = tmem_full0 + 4;
  uint64_t* affn_full = tmem_full0 + 5;                       // the three peers' LN2 slices have landed in this CTA's FFN1 operand
  uint64_t* hx_full = tmem_full0 + 6;                         // the three peers' hidden-column slices have landed in the h region
  uint64_t* hop_ready = tmem_full0 + 7;                       // the epilogue warps have assembled the FFN2 A operand
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full0 + 8);
  static_assert((2 * kFbStages + 8) * 8 + 4 <= 256, "barrier area");
  constexpr int kHSlice = kBlockM * kHSplit * 2;              // one CTA's hidden columns: 128 rows x 64 B = 8 KB
  float* s_gain_mid = reinterpret_cast<float*>(after + 256);
  float* s_gain_out = s_gain_mid + BN;
  // LayerNorm partials [2 halves][128 rows]: the first exchange uses the start of the h region (no hidden slice exists yet), the second
  // the start of the W2 region (FFN2 has read it; the h region may still be the source of this CTA's outgoing slice copies)
  float2* s_stats = reinterpret_cast<float2*>(h_smem);

  const int warp = threadIdx.x >> 5;
  const int lane = static_cast<int>(lane_id());
  const int m0 = blockIdx.y * kBlockM;
  const uint32_t crank = cluster_ctarank();
  const int coff = static_cast<int>(crank) * BN;
  const int n0 = coff;
  __shared__ int s_trace;
  pdl_trigger();
  if (threadIdx.x == 0) { s_trace = trace_begin() ? 1 : 0; trace_point(s_trace != 0, 0); }

  GemmSmemView sv;
  sv.stages = ring; sv.full_bar = full_bar; sv.empty_bar = empty_bar; sv.tmem_full_bar = tmem_full0; sv.tmem_slot = tmem_slot; sv.scratch = nullptr;

  if (warp == 0) {
    if (elect_one()) {
      tma_prefetch_desc(&tmap_ao); tma_prefetch_desc(&tmap_wo); tma_prefetch_desc(&tmap_w1q); tma_prefetch_desc(&tmap_w2);
      for (int st = 0; st < kFbStages; ++st) { mbar_init(&full_bar[st], 1); mbar_init(&empty_bar[st], 1); }
      mbar_init(tmem_full0, 1); mbar_init(w1_full, 1); mbar_init(w2_full, 1); mbar_init(tmem_full1, 1); mbar_init(tmem_full2, 1);
      mbar_init(affn_full, 1); mbar_init(hx_full, 1); mbar_init(hop_ready, kRowEpiWarps);
      fence_mbar_init();
      mbar_arrive_expect_tx(affn_full, (kRowCluster - 1) * 2 * kABytes);   // the peers' copies can only start after cluster barrier #1
      mbar_arrive_expect_tx(hx_full, (kRowCluster - 1) * kHSlice);
      // all weights first (they do not depend on the previous kernel), then wait, then the activation tiles
      for (int kb = 0; kb < kFbStages; ++kb) {
        mbar_arrive_expect_tx(&full_bar[kb], kStageBytes);
        tma_load_2d(ring + kb * kStageBytes + kABytes, &tmap_wo, &full_bar[kb], kb * kBlockK, n0, kEvictLast);
      }
      pdl_wait();
      for (int kb = 0; kb < kFbStages; ++kb)
        tma_load_2d(ring + kb * kStageBytes, &tmap_ao, &full_bar[kb], kb * kBlockK, m0, kEvictNormal);
    }
  } else if (warp == 1) {
    tmem_alloc<512>(tmem_slot);
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  const bool tr = s_trace != 0;
  pdl_wait();
  if (threadIdx.x == 0) trace_point(tr, 1);

  if (warp == 0) {
    if (elect_one()) {
      producer_rest<kFbStages>(sv, &tmap_ao, &tmap_wo, kNkb, m0, n0);
      // stages 4 and 5 are the W1 / W2 regions: load the feed-forward weights as soon as the out-proj MMAs have read them
      mbar_wait(&empty_bar[kFbRing], 0, 1);
      mbar_arrive_expect_tx(w1_full, kNkb * kW1kb);
      for (int kb = 0; kb < kNkb; ++kb) tma_load_2d(w1_smem + kb * kW1kb, &tmap_w1q, w1_full, kb * kBlockK, static_cast<int>(crank) * kHSplit, kEvictLast);
      mbar_wait(&empty_bar[kFbRing + 1], 0, 1);
      mbar_arrive_expect_tx(w2_full, 2 * kBBytes);
      tma_load_2d(w2_smem, &tmap_w2, w2_full, 0, n0, kEvictLast);
      tma_load_2d(w2_smem + kBBytes, &tmap_w2, w2_full, kBlockK, n0, kEvictLast);
    }
  } else if (warp == 1) {
    if (elect_one()) mma_mainloop<kFbStages>(sv, tmem_base, kNkb, false);      // acc0 -> TMEM columns [0, 128)
  }

  // ---- phase A epilogue: residual + accumulator, LN2 statistics
  const bool is_epi = warp >= 2;
  const int ew = warp - 2;
  const int quad = warp & 3;
  const int half = ew >> 2;
  const int row_in_tile = quad * 32 + lane;
  const int row = m0 + row_in_tile;
  const int c0 = coff + half * kRowCols;
  const uint32_t tmem_lane = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
  float r[kRowCols];
  auto add_acc_and_stats = [&](uint32_t acc_col) {
    float sum = 0.f, sumsq = 0.f;
#pragma unroll
    for (int c = 0; c < kRowCols / 16; ++c) {
      float v[16];
      tmem_ld_32x16(tmem_lane + acc_col + half * kRowCols + c * 16, v);
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const float t = r[c * 16 + j] + v[j];
        r[c * 16 + j] = t;
        sum += t;
        sumsq = fmaf(t, t, sumsq);
      }
    }
    s_stats[half * 128 + row_in_tile] = make_float2(sum, sumsq);
  };
  auto gather_stats = [&](float& mean, float& rstd) {
    float2 part[kRowCluster * 2];
#pragma unroll
    for (uint32_t pr = 0; pr < kRowCluster; ++pr) {
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) part[pr * 2 + hh] = dsmem_ld_f32x2_addr(dsmem_addr(&s_stats[hh * 128 + row_in_tile], pr));
    }
    float sum = 0.f, sumsq = 0.f;
#pragma unroll
    for (int i = 0; i < kRowCluster * 2; ++i) { sum += part[i].x; sumsq += part[i].y; }
    mean = sum * (1.0f / kE);
    rstd = rsqrtf(fmaxf(sumsq * (1.0f / kE) - mean * mean, 0.f) + ep.eps);
  };
  if (is_epi) {
    if (ew < 4) {
      s_gain_mid[threadIdx.x - 64] = __ldg(ep.gain_mid + coff + (threadIdx.x - 64));
      s_gain_out[threadIdx.x - 64] = __ldg(ep.gain_out + coff + (threadIdx.x - 64));
    }
    if (row < M) {
#pragma unroll
      for (int q = 0; q < kRowCols / 4; ++q) {
        const float4 t = *reinterpret_cast<const float4*>(ep.x + xblk_off(row, (c0 >> 2) + q));
        r[q * 4] = t.x; r[q * 4 + 1] = t.y; r[q * 4 + 2] = t.z; r[q * 4 + 3] = t.w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < kRowCols; ++i) r[i] = 0.f;
    }
    mbar_wait(tmem_full0, 0, 3);
    if (threadIdx.x == 64) trace_point(tr, 2);
    tc_fence_after_sync();
    add_acc_and_stats(0);
    if (threadIdx.x == 64) trace_point(tr, 3);
  }
  __syncthreads();          // s_gain visible to all epilogue warps
  cluster_sync_all();       // #1: LN2 partials visible; every CTA's phase-A MMAs have completed (their accumulators were read)
  if (threadIdx.x == 64) trace_point(tr, 4);

  // ---- hand-over: LN2 rows -> FFN1 operand of all four CTAs.  Every thread writes its 128-byte row into the LOCAL operand buffer; one
  // thread then pushes the CTA's two k-block tiles (32 KB) to each peer with a TMA shared->shared bulk copy that completes on the peer's
  // mbarrier (per-thread st.shared::cluster stores took 11 k cycles for the same bytes).
  if (is_epi) {
    float mean = 0.f, rstd = 0.f;
    if (row < M) gather_stats(mean, rstd);
    const int kb = static_cast<int>(crank) * 2 + half;                       // this thread's 64 columns = one row of that k-block
    uint8_t* arow = ring + kb * kABytes + row_in_tile * 128;
#pragma unroll
    for (int q = 0; q < kRowCols / 8; ++q) {
      float y[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) y[i] = (r[q * 8 + i] - mean) * rstd * s_gain_mid[half * kRowCols + q * 8 + i];
      *reinterpret_cast<uint4*>(arow + ((q ^ (row_in_tile & 7)) << 4)) =
          make_uint4(pack_bf16x2(y[0], y[1]), pack_bf16x2(y[2], y[3]), pack_bf16x2(y[4], y[5]), pack_bf16x2(y[6], y[7]));
    }
    fence_proxy_async_smem();      // generic-proxy writes -> visible to the async proxy (the bulk copies and this CTA's own MMAs)
    if (threadIdx.x == 64) trace_point(tr, 5);
  }
  __syncthreads();
  if (warp == 0) {
    if (elect_one()) {
      const uint8_t* src = ring + static_cast<int>(crank) * 2 * kABytes;
#pragma unroll
      for (uint32_t d = 1; d < kRowCluster; ++d) {
        const uint32_t pr = (crank + d) % kRowCluster;
        dsmem_bulk_copy(dsmem_addr(src, pr), src, 2 * kABytes, dsmem_addr(affn_full, pr));
      }
    }
  }
  __syncwarp();
  if (threadIdx.x == 64) trace_point(tr, 6);

  // ---- phase B: this CTA's 32 hidden columns
  if (warp == 1) {
    if (elect_one()) {
      mbar_wait(affn_full, 0, 5);
      trace_point(tr, 15);
      mbar_wait(w1_full, 0, 6);
      tc_fence_after_sync();
      const uint32_t sa = smem_u32(ring), sb = smem_u32(w1_smem);
#pragma unroll
      for (int kb = 0; kb < kNkb; ++kb)
#pragma unroll
        for (int k = 0; k < kBlockK / kUmmaK; ++k)
          umma_bf16_ss(tmem_base + 128, umma_desc_sw128_kmajor(sa + kb * kABytes + k * (kUmmaK * 2)),
                       umma_desc_sw128_kmajor(sb + kb * kW1kb + k * (kUmmaK * 2)), kIdescH, (kb | k) != 0 ? 1u : 0u);
      umma_commit(tmem_full1);
    }
  }
  __syncwarp();
  if (is_epi) {
    mbar_wait(tmem_full1, 0, 7);
    if (threadIdx.x == 64) trace_point(tr, 7);
    tc_fence_after_sync();
    float v[16];
    tmem_ld_32x16(tmem_lane + 128 + half * 16, v);
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = gelu_fast(v[j]);
    // hidden-column exchange: the h region holds four 8 KB slices [source CTA][128 rows][64 B]; this thread's 16 columns go into the
    // local slice, which one thread then pushes to the peers with bulk copies (per-thread st.shared::cluster stores: 4.2 k cycles)
    uint4* mine = reinterpret_cast<uint4*>(h_smem + static_cast<int>(crank) * kHSlice + row_in_tile * 64 + half * 32);
#pragma unroll
    for (int q = 0; q < 2; ++q)
      mine[q] = make_uint4(pack_bf16x2(v[q * 8 + 0], v[q * 8 + 1]), pack_bf16x2(v[q * 8 + 2], v[q * 8 + 3]),
                           pack_bf16x2(v[q * 8 + 4], v[q * 8 + 5]), pack_bf16x2(v[q * 8 + 6], v[q * 8 + 7]));
    fence_proxy_async_smem();
  }
  __syncthreads();
  if (warp == 0) {
    if (elect_one()) {
      const uint8_t* src = h_smem + static_cast<int>(crank) * kHSlice;
#pragma unroll
      for (uint32_t d = 1; d < kRowCluster; ++d) {
        const uint32_t pr = (crank + d) % kRowCluster;
        dsmem_bulk_copy(dsmem_addr(src, pr), src, kHSlice, dsmem_addr(hx_full, pr));
      }
    }
  }
  __syncwarp();
  if (threadIdx.x == 64) trace_point(tr, 8);
  if (is_epi) {
    // assemble the K-major swizzled A operand of FFN2 in the (now dead) W1 region: this thread's row, k-block `half` = the slices of
    // source CTAs 2 * half and 2 * half + 1
    mbar_wait(hx_full, 0, 10);
    uint8_t* hrow = w1_smem + half * kABytes + row_in_tile * 128;
#pragma unroll
    for (int sidx = 0; sidx < 2; ++sidx) {
      const uint4* src = reinterpret_cast<const uint4*>(h_smem + (2 * half + sidx) * kHSlice + row_in_tile * 64);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int chunk = sidx * 4 + c;
        *reinterpret_cast<uint4*>(hrow + ((chunk ^ (row_in_tile & 7)) << 4)) = src[c];
      }
    }
    fence_proxy_async_smem();
    tc_fence_before_sync();
    __syncwarp();
    if (lane == 0) mbar_arrive(hop_ready);
  }
  if (threadIdx.x == 64) trace_point(tr, 9);

  // ---- phase C: second feed-forward GEMM, residual, LayerNorm
  if (warp == 1) {
    if (elect_one()) {
      mbar_wait(hop_ready, 0, 11);
      mbar_wait(w2_full, 0, 8);
      tc_fence_after_sync();
      const uint32_t sa = smem_u32(w1_smem), sb = smem_u32(w2_smem);
#pragma unroll
      for (int kb = 0; kb < kFfnDim / kBlockK; ++kb)
#pragma unroll
        for (int k = 0; k < kBlockK / kUmmaK; ++k)
          umma_bf16_ss(tmem_base + 256, umma_desc_sw128_kmajor(sa + kb * kABytes + k * (kUmmaK * 2)),
                       umma_desc_sw128_kmajor(sb + kb * kBBytes + k * (kUmmaK * 2)), kIdesc, (kb | k) != 0 ? 1u : 0u);
      umma_commit(tmem_full2);
    }
  }
  __syncwarp();
  if (is_epi) {
    mbar_wait(tmem_full2, 0, 9);     // FFN2 has read W2: its first 2 KB hold the second round of statistics
    if (threadIdx.x == 64) trace_point(tr, 10);
    tc_fence_after_sync();
    s_stats = reinterpret_cast<float2*>(w2_smem);
    add_acc_and_stats(256);
    if (threadIdx.x == 64) trace_point(tr, 11);
  }
  __syncwarp();
  cluster_sync_all();       // #4
  if (threadIdx.x == 64) trace_point(tr, 12);
  if (is_epi) {
    float mean = 0.f, rstd = 0.f;
    s_stats = reinterpret_cast<float2*>(w2_smem);
    if (row < M) gather_stats(mean, rstd);
    uint8_t* stage = ring + ew * (32 * kRowStagePitch);      // the FFN1 operand is dead: every CTA's phase-B MMAs completed before #3
    {
      uint4* d = reinterpret_cast<uint4*>(stage + lane * kRowStagePitch);
#pragma unroll
      for (int q = 0; q < kRowCols / 8; ++q) {
        float y[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) y[i] = (r[q * 8 + i] - mean) * rstd * s_gain_out[half * kRowCols + q * 8 + i];
        d[q] = make_uint4(pack_bf16x2(y[0], y[1]), pack_bf16x2(y[2], y[3]), pack_bf16x2(y[4], y[5]), pack_bf16x2(y[6], y[7]));
      }
    }
    if (row < M) {
#pragma unroll
      for (int q = 0; q < kRowCols / 4; ++q)
        *reinterpret_cast<float4*>(ep.x + xblk_off(row, (c0 >> 2) + q)) = make_float4(r[q * 4], r[q * 4 + 1], r[q * 4 + 2], r[q * 4 + 3]);
    }
    __syncwarp();
    const int warp_row0 = m0 + quad * 32;
    const int sub = lane >> 3, chunk = lane & 7;
#pragma unroll 4
    for (int i = 0; i < 8; ++i) {
      const int rr = i * 4 + sub;
      const int grow = warp_row0 + rr;
      if (grow < M) {
        int nrow = grow;
        bool keep = true;
        if (ep.remap_rows_in > 0) {
          const int seq = grow / ep.remap_rows_in;
          const int k = grow - seq * ep.remap_rows_in;
          keep = k >= ep.remap_skip;
          nrow = seq * ep.remap_rows_out + (k - ep.remap_skip);
        }
        if (keep)
          *reinterpret_cast<uint4*>(ep.xn + static_cast<size_t>(nrow) * kE + c0 + chunk * 8) =
              *reinterpret_cast<const uint4*>(stage + rr * kRowStagePitch + chunk * 16);
      }
    }
  }
  if (threadIdx.x == 64) trace_point(tr, 13);
  tc_fence_before_sync();
  __syncwarp();
  cluster_sync_relaxed();   // peers may still be reading this CTA's statistics / operand tiles
  if (threadIdx.x == 0) trace_point(tr, 14);
  if (warp == 1) tmem_dealloc<512>(tmem_base);
}

// ---------------------------------------------------------------------------------------------------------
// The persistent GEMM on CTA PAIRS: 256 x 256 output tiles, one tcgen05.mma.cta_group::2 of M = 256, N = 256 per k-slice.
// Why: the 128 x 128 single-CTA tile takes in 256 KB of operands per 33.5 MFLOP - 4.4 k cycles per tile at the ~58 B/clk per SM that the L2
// delivers when all 148 SMs pull (phase trace of the QKV GEMM; the chip-wide L2 output cap is ~6300 B/clk), against 2.1 k cycles of
// MMA.  A pair moves HALF the bytes per FLOP: each CTA loads its own 128 rows of A and 128 of the tile's 256 rows of B (the tensor
// cores of both SMs read both shared memories), and owns the 128 x 256 accumulator rows of its half in its own TMEM.
//   * cluster (2, 1, 1); rank 0 = leader: its MMA warp waits on ITS full barrier - both CTAs' TMA loads count their bytes there
//     (cp.async.bulk.tensor ... .cta_group::2 with the leader's barrier address) - and issues the MMAs; tcgen05.commit multicasts the
//     "stage free" and "accumulator ready" arrivals to the barriers of both CTAs
//   * both CTAs run the 8 epilogue warps on their own accumulator half (any epilogue that honours EpiCtx::ncols = 128); the leader's
//     "accumulator drained" barrier counts the warps of both CTAs (the peer arrives through the cluster address)
//   * stages: KBS = 2 k-blocks of [A 128 x 64 | B-half 128 x 64] = 64 KB per CTA, 3-D tensor maps with 128-row boxes (the same maps as
//     gemm_kernel<.., KBS = 2>), two accumulator stages of 256 columns = all 512 TMEM columns.
// ---------------------------------------------------------------------------------------------------------
constexpr int kPairKbs = 2;
// PN = columns of the pair's tile: 256 (64 KB stages, the big GEMMs of the image encoder) or 128 (48 KB stages; keeps the 128 x 128 tile count
// per CTA - and with it the wave quantisation - of the single-CTA kernel at 0.75 of its operand bytes: the decoder's QKV projection).
__host__ __device__ constexpr int pair_stage_bytes(int pn) { return kPairKbs * (kABytes + (pn / 2) * kBlockK * 2); }
__host__ __device__ constexpr int gemm2_smem_bytes(int stages, int pn = 256) { return stages * pair_stage_bytes(pn) + kEpiWarps * kEpiStageBytes + 1024 + 256; }

template <class Epi, int STAGES, int PN = 256>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemmThreads, 1)
gemm2_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, int M, int n_tiles /* of PN columns */,
             int num_k_blocks, int b_is_static, typename Epi::Params ep) {
  static_assert(PN == 256 || PN == 128, "pair tile width");
  constexpr int KBS = kPairKbs;
  constexpr int kPairTileN = PN;
  constexpr int kHalfN = PN / 2;                              // rows of B (= output columns) this CTA loads
  constexpr int kBBytes = kHalfN * kBlockK * 2;               // shadows the namespace constant: one k-block of this CTA's B half
  constexpr int kPairStageBytes = pair_stage_bytes(PN);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stages = smem;
  uint8_t* epi_stage = smem + STAGES * kPairStageBytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(epi_stage + kEpiWarps * kEpiStageBytes);   // used in the leader only
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;        // [kAccStages]
  uint64_t* tmem_empty_bar = tmem_full_bar + kAccStages;   // used in the leader only: 2 x kEpiWarps arrivals
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + kAccStages);

  const int warp = threadIdx.x >> 5;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int m_tiles = (M + 2 * kBlockM - 1) / (2 * kBlockM);
  const int total_tiles = m_tiles * n_tiles;
  const int loads_per_tile = num_k_blocks / KBS;
  pdl_trigger();

  if (warp == 0) {
    if (elect_one()) {
      tma_prefetch_desc(&tmap_a);
      tma_prefetch_desc(&tmap_b);
      for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
      for (int a = 0; a < kAccStages; ++a) { mbar_init(&tmem_full_bar[a], 1); mbar_init(&tmem_empty_bar[a], 2 * kEpiWarps); }
      fence_mbar_init();
    }
  } else if (warp == 1) {
    tmem_alloc2<kAccStages * kPairTileN>(tmem_slot);
  }
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();       // the peer's barriers are initialised before anything arrives on them
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t leader_full0 = dsmem_addr(&full_bar[0], 0);

  if (warp == 0) {
    if (elect_one()) {
      // weight halves of the first pipeline fill before griddepcontrol.wait (they do not depend on the previous kernel)
      const int early_b = (b_is_static && pair < total_tiles) ? min(STAGES, loads_per_tile) : 0;
      if (early_b > 0) {
        const int n0 = (pair % n_tiles) * kPairTileN + static_cast<int>(rank) * kHalfN;
        for (int i = 0; i < early_b; ++i) {
          if (leader) mbar_arrive_expect_tx(&full_bar[i], 2 * kPairStageBytes);
          tma_load_3d_2sm(stages + i * kPairStageBytes + KBS * kABytes, &tmap_b, leader_full0 + i * 8, n0, i * KBS, kEvictLast);
        }
      }
      pdl_wait();
      int stage = 0; uint32_t phase = 0;
      int nload = 0;
      for (int t = pair; t < total_tiles; t += npairs) {
        const int m0 = (t / n_tiles) * (2 * kBlockM) + static_cast<int>(rank) * kBlockM;
        const int n0 = (t % n_tiles) * kPairTileN + static_cast<int>(rank) * kHalfN;
        for (int kb = 0; kb < num_k_blocks; kb += KBS, ++nload) {
          uint8_t* sa = stages + stage * kPairStageBytes;
          if (nload >= early_b) {
            mbar_wait(&empty_bar[stage], phase ^ 1, 1);
            if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * kPairStageBytes);
          }
          tma_load_3d_2sm(sa, &tmap_a, leader_full0 + stage * 8, m0, kb, kEvictNormal);
          if (nload >= early_b) tma_load_3d_2sm(sa + KBS * kABytes, &tmap_b, leader_full0 + stage * 8, n0, kb, kEvictLast);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    pdl_wait();
    if (leader && elect_one()) {
      constexpr uint32_t kIdesc = umma_idesc_bf16_f32(2 * kBlockM, kPairTileN);
      int stage = 0; uint32_t phase = 0;
      int i = 0;
      for (int t = pair; t < total_tiles; t += npairs, ++i) {
        const int as = i & 1;
        mbar_wait(&tmem_empty_bar[as], ((i >> 1) & 1) ^ 1, 9);   // both CTAs' epilogues have drained this accumulator stage
        tc_fence_after_sync();
        const uint32_t acc = tmem_base + as * kPairTileN;
        for (int kb = 0; kb < num_k_blocks; kb += KBS) {
          mbar_wait(&full_bar[stage], phase, 2);
          tc_fence_after_sync();
          const uint32_t sa = smem_u32(stages + stage * kPairStageBytes);
          const uint32_t sb = sa + KBS * kABytes;
#pragma unroll
          for (int j = 0; j < KBS; ++j)
#pragma unroll
            for (int k = 0; k < kBlockK / kUmmaK; ++k)
              umma2_bf16_ss(acc, umma_desc_sw128_kmajor(sa + j * kABytes + k * (kUmmaK * 2)),
                            umma_desc_sw128_kmajor(sb + j * kBBytes + k * (kUmmaK * 2)), kIdesc, (kb > 0 || (j | k) != 0) ? 1u : 0u);
          umma2_commit_mc(&empty_bar[stage], 0x3);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma2_commit_mc(&tmem_full_bar[as], 0x3);
      }
    }
    __syncwarp();
  } else {
    pdl_wait();
    const int ew = warp - 2;
    const int quad = warp & 3;
    const int half = ew >> 2;            // which half of the tile's columns
    const int lane = static_cast<int>(lane_id());
    const uint32_t leader_tmem_empty0 = dsmem_addr(&tmem_empty_bar[0], 0);
    int i = 0;
    for (int t = pair; t < total_tiles; t += npairs, ++i) {
      const int as = i & 1;
      const int m0 = (t / n_tiles) * (2 * kBlockM) + static_cast<int>(rank) * kBlockM, nt = t % n_tiles;
      mbar_wait(&tmem_full_bar[as], (i >> 1) & 1, 3);
      tc_fence_after_sync();
      EpiCtx c;
      c.tmem_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * kPairTileN + half * (kPairTileN / 2);
      c.warp_row0 = m0 + quad * 32;
      c.row = c.warp_row0 + lane;
      c.n0 = nt * kPairTileN + half * (kPairTileN / 2);
      c.ncols = kPairTileN / 2;
      c.M = M;
      c.part = (nt * 2 + half) * (kPairTileN / 128);
      c.stage = epi_stage + ew * kEpiStageBytes;
      const uint32_t rel = leader_tmem_empty0 + as * 8;
      Epi::run(ep, c, [rel, lane]() {
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(rel);
      });
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();       // the leader's MMAs have read the peer's shared memory; the peer's arrivals have landed in the leader
  if (warp == 1) tmem_dealloc2<kAccStages * kPairTileN>(tmem_base);
}


}  // namespace novic
