// Full-catalogue logits  D[M,V] = out[M,64] . E[V,64]^T  on the 5th-gen tensor cores (tcgen05),
// with the consumer fused into the TMEM epilogue so the [M,V] logits never reach HBM:
//   MODE_STORE : plain scores (full_sort_predict)                  acsasrec.py:162-163
//   MODE_CE    : per-row running (max, sum exp) -> cross entropy   acsasrec.py:118-120
//   MODE_GRAD  : Gt[V,M] = ((softmax - onehot) * row_scale)^T (CE backward)
//   MODE_TOPK  : streaming per-row top-k, column 0 excluded         trainer.py:941-942, collector.py:147
//
// Warp-specialised persistent CTA (320 threads, one per SM):
//   warp 0      producer : 1-D bulk async copies (TMA engine, cp.async.bulk -> UBLKCP) of 64-row
//                          fp32 tiles of the item table into a shared-memory ring, mbarrier tx-count
//   warps 2-5   splitter : fp32 tile -> (hi, lo) TF32 operands written in the canonical no-swizzle
//                          K-major UMMA layout (8x16B core matrices); diagonal chunk rotation keeps
//                          both the LDS and the STS bank-conflict free
//   warp 1      MMA      : one thread issues tcgen05.mma.kind::tf32 128x64x8, 8 k-steps x {lo.hi,
//                          hi.lo, hi.hi} (3xTF32: fp32-level accuracy) or 1 pass; accumulator in
//                          TMEM, double buffered (2 x 64 columns); completion via tcgen05.commit
//   warps 6-9   epilogue : tcgen05.ld 32 lanes x 32 columns -> one thread owns one logits row, so the
//                          online softmax / top-k state is thread-private (no shuffles)
// The activation tile A (128 x 64, hi and lo) is stationary in shared memory.
#include "logits_common.cuh"
#include "../../include/acsr.h"

namespace acsr {

template <int MODE>
struct TcCfg {
  static constexpr bool kTopkMode = MODE == MODE_TOPK || MODE == MODE_TOPK_RANK;
  static constexpr int kStages = kTopkMode ? 2 : 4;
  static constexpr int kAbytes = kBM * kD * 4;          // 32 KB per (hi|lo)
  static constexpr int kBbytes = kBN * kD * 4;          // 16 KB per (hi|lo) per buffer
  // MODE_TOPK keeps the stationary tile of `out` in TENSOR MEMORY (hi / lo halves written once with tcgen05.st; the MMAs take
  // it as their A operand, TS form): its shared memory goes to a second set of candidate lists, so that the top-k epilogue --
  // the bottleneck of the kernel, one thread per logits row -- runs on eight warps like the CE epilogue.
  static constexpr bool kATmem = kTopkMode;
  static constexpr int kOffAhi = 0;
  static constexpr int kOffAlo = kOffAhi + (kATmem ? 0 : kAbytes);
  static constexpr int kOffBhi = kOffAlo + (kATmem ? 0 : kAbytes);      // [2]
  static constexpr int kOffBlo = kOffBhi + 2 * kBbytes;  // [2]
  static constexpr int kOffStg = kOffBlo + 2 * kBbytes;  // [kStages]
  static constexpr int kOffTopk = kOffStg + kStages * kBbytes;
  static constexpr int kListBytes = 2 * kMaxTopK * kBM * 4;              // values + indices of one warp set: 64 KB
  static constexpr int kTopkBytes = kTopkMode ? 2 * kListBytes : 0;
  // MODE_CE / MODE_TOPK: the epilogue is instruction-issue / latency bound (one thread per logits row), so it runs on EIGHT warps,
  // two per TMEM lane quarter, each owning one 32-column half of every tile; the halves meet once, at the end, through kOffPair
  static constexpr int kEpiWarps = (MODE == MODE_CE || kTopkMode) ? 8 : 4;
  // Two MMA-issuing threads (warp 1: even tiles, the last warp: odd tiles -- each owns one operand buffer and one accumulator
  // stage): a thread issues one 128 x 64 x 8 TF32 MMA every ~90 cycles against a 32-cycle tensor floor (scripts/umma_rate.py)
  static constexpr int kIssuer2 = 6 + kEpiWarps;
  static constexpr int kThreads = 192 + 32 * kEpiWarps + 32;
  static constexpr int kOffPair = kOffTopk + kTopkBytes;
  // MODE_TOPK_RANK also hands the upper warp set's two rank counts over: [128] candidate counts, then [128] int2
  static constexpr int kPairBytes = MODE == MODE_TOPK_RANK ? kBM * 12 : (MODE == MODE_CE || kTopkMode) ? kBM * 8 : 0;
  static constexpr int kOffBar = kOffPair + kPairBytes;
  static constexpr int kNumBars = 2 * kStages + 2 + 2 + 2 + 2;
  static constexpr int kSmemBytes = kOffBar + kNumBars * 8 + 16;
  static constexpr int kTmem = kATmem ? 256 : kTmemCols;                 // 2 accumulator stages (+ out hi / lo at columns 128 / 192)
};

// Thread-private top-k candidate set kept UNSORTED with a cached minimum (slot-major in shared memory so
// lane == bank for every slot).  A new score replaces the current minimum and the k slots are rescanned
// with independent loads -- no dependent shift chain as in a sorted insert; acsr_topk_merge sorts at the end.
// (A binary min-heap with one sift-down per insert was measured too: 720 vs 734 us at 1M items, slower at k = 10 -- the cost
// of an insertion is the lockstep drain round around it, not the rescan.)
__device__ __noinline__ void topk_insert(float x, int col, float* lval, int* lidx, int row, int k, int& cnt, float& thr,
                                         int& minpos) {
  if (cnt < k) {
    lval[cnt * kBM + row] = x;
    lidx[cnt * kBM + row] = col;
    if (++cnt < k) return;
  } else {
    lval[minpos * kBM + row] = x;
    lidx[minpos * kBM + row] = col;
  }
  float m = lval[row];
  int mp = 0;
#pragma unroll 8
  for (int s = 1; s < k; ++s) {
    const float v = lval[s * kBM + row];
    if (v < m) { m = v; mp = s; }
  }
  thr = m;
  minpos = mp;
}

// order-preserving int image of a float (signed integer compare == float compare), for atomicMax on a shared lower bound
__device__ __forceinline__ int bound_enc(float x) { const int b = __float_as_int(x); return b >= 0 ? b : b ^ 0x7fffffff; }
__device__ __forceinline__ float bound_dec(int k) { return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff); }

template <int MODE>
__global__ void __launch_bounds__(TcCfg<MODE>::kThreads, 1) logits_tc_kernel(const LogitsParams p) {
  pdl_launch_dependents();
  pdl_wait();
  using Cfg = TcCfg<MODE>;
  constexpr bool kTopk = Cfg::kTopkMode, kRank = MODE == MODE_TOPK_RANK;
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tile = blockIdx.x % p.m_tiles;
  const int chunk = blockIdx.x / p.m_tiles;
  const float* out_p = p.out + (MODE == MODE_LINEAR ? blockIdx.y * p.b_out : 0);
  const float* table_p = p.table + (MODE == MODE_LINEAR ? blockIdx.y * p.b_table : 0);
  float* C_p = p.C + (MODE == MODE_LINEAR ? blockIdx.y * p.b_C : 0);
  const int my_tiles = chunk < p.n_tiles ? (p.n_tiles - chunk + p.n_chunks - 1) / p.n_chunks : 0;

  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kOffBar);
  uint64_t* stg_full = bars;
  uint64_t* stg_empty = bars + Cfg::kStages;
  uint64_t* op_full = bars + 2 * Cfg::kStages;
  uint64_t* op_empty = op_full + 2;
  uint64_t* tm_full = op_empty + 2;
  uint64_t* tm_empty = tm_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + Cfg::kNumBars);

  if (threadIdx.x == 0) {
    for (int s = 0; s < Cfg::kStages; ++s) { mbar_init(stg_full + s, 1); mbar_init(stg_empty + s, 128); }
    for (int s = 0; s < 2; ++s) {
      mbar_init(op_full + s, 128); mbar_init(op_empty + s, 1);
      mbar_init(tm_full + s, 1); mbar_init(tm_empty + s, 32 * Cfg::kEpiWarps);
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc<Cfg::kTmem>(tmem_slot);

  // stationary A tile: rows of `out`, split into hi/lo TF32, canonical K-major layout
  if (!Cfg::kATmem) {
    float* Ahi = reinterpret_cast<float*>(smem + Cfg::kOffAhi);
    float* Alo = reinterpret_cast<float*>(smem + Cfg::kOffAlo);
    for (int item = threadIdx.x; item < kBM * kKC; item += Cfg::kThreads) {
      const int r = item / kKC, kc = item % kKC;
      const int grow = m_tile * kBM + r;
      float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
      if (grow < p.M) {
        if (MODE != MODE_LINEAR) x = *reinterpret_cast<const float4*>(out_p + (long long)grow * kD + kc * 4);
        else if (p.out_sk == 1 && (p.out_sn & 3) == 0) x = *reinterpret_cast<const float4*>(out_p + grow * p.out_sn + kc * 4);
        else {                         // transposed / strided weight (input-gradient GEMMs)
          const float* w = out_p + grow * p.out_sn + (long long)(kc * 4) * p.out_sk;
          x = make_float4(w[0], w[p.out_sk], w[2 * p.out_sk], w[3 * p.out_sk]);
        }
      }
      float4 hi = make_float4(to_tf32(x.x), to_tf32(x.y), to_tf32(x.z), to_tf32(x.w));
      float4 lo = make_float4(x.x - hi.x, x.y - hi.y, x.z - hi.z, x.w - hi.w);
      const int off = kc * (kBM * 4) + r * 4;      // floats: chunk plane of kBM rows x 16 B
      *reinterpret_cast<float4*>(Ahi + off) = hi;
      *reinterpret_cast<float4*>(Alo + off) = lo;
    }
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (Cfg::kATmem) {
    // the thread's row of `out` (its 32 columns) -> TMEM columns 128.. (hi) and 192.. (lo): the A operand of every MMA
    if (warp >= 6 && warp < Cfg::kIssuer2) {
      const int quarter = warp & 3, half = (warp - 6) >> 2;
      const int grow = m_tile * kBM + quarter * 32 + lane;
      float hi[32], lo[32];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        if (grow < p.M) x = *reinterpret_cast<const float4*>(out_p + (long long)grow * kD + half * 32 + 4 * j);
        hi[4 * j + 0] = to_tf32(x.x); hi[4 * j + 1] = to_tf32(x.y); hi[4 * j + 2] = to_tf32(x.z); hi[4 * j + 3] = to_tf32(x.w);
        lo[4 * j + 0] = x.x - hi[4 * j + 0]; lo[4 * j + 1] = x.y - hi[4 * j + 1]; lo[4 * j + 2] = x.z - hi[4 * j + 2]; lo[4 * j + 3] = x.w - hi[4 * j + 3];
      }
      const uint32_t t_row = tmem_base + ((uint32_t)(quarter * 32) << 16) + half * 32;
      tmem_st32(t_row + 128, hi);
      tmem_st32(t_row + 192, lo);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
  }

  if (warp == 0) {
    // ------------------------------ producer ------------------------------
    if (lane == 0) {
      for (int it = 0; it < my_tiles; ++it) {
        const int s = it % Cfg::kStages;
        const uint32_t ph = (it / Cfg::kStages) & 1;
        const long long n0 = (long long)(chunk + it * p.n_chunks) * kBN;
        const long long rows = (p.V - n0) < kBN ? (p.V - n0) : kBN;
        mbar_wait(stg_empty + s, ph ^ 1);
        mbar_arrive_expect_tx(stg_full + s, (uint32_t)(rows * kD * 4));
        bulk_g2s(smem + Cfg::kOffStg + s * Cfg::kBbytes, table_p + n0 * kD, (uint32_t)(rows * kD * 4), stg_full + s);
      }
    }
  } else if (warp == 1 || warp == Cfg::kIssuer2) {
    // ------------------------------ MMA issuers ------------------------------
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_tf32(kBM, kBN);
      const uint32_t a_hi = smem_u32(smem + Cfg::kOffAhi), a_lo = smem_u32(smem + Cfg::kOffAlo);
      constexpr uint32_t kALbo = kBM * 16, kBLbo = kBN * 16, kSbo = 128;
      for (int it = (warp == 1 ? 0 : 1); it < my_tiles; it += 2) {
        const int ob = it & 1;
        const uint32_t ph = (it >> 1) & 1;
        mbar_wait(op_full + ob, ph);
        mbar_wait(tm_empty + ob, ph ^ 1);
        tc_fence_after();
        const uint32_t b_hi = smem_u32(smem + Cfg::kOffBhi + ob * Cfg::kBbytes);
        const uint32_t b_lo = smem_u32(smem + Cfg::kOffBlo + ob * Cfg::kBbytes);
        const uint32_t d_tmem = tmem_base + ob * kBN;
        uint32_t acc = 0;
        const int npass = p.passes == 3 ? 3 : 1;
        for (int ps = 0; ps < npass; ++ps) {
          // small cross terms first, the dominant hi.hi product last
          const uint32_t a_base = (npass == 3 && ps == 0) ? a_lo : a_hi;
          const uint32_t b_base = (npass == 3 && ps == 1) ? b_lo : b_hi;
#pragma unroll
          for (int ks = 0; ks < kD / 8; ++ks) {
            const uint64_t bd = umma_desc_kmajor(b_base + ks * 2 * kBLbo, kBLbo, kSbo);
            if (Cfg::kATmem) {
              const uint32_t at = tmem_base + ((npass == 3 && ps == 0) ? 192 : 128) + ks * 8;
              umma_tf32_ts(d_tmem, at, bd, idesc, acc);
            } else {
              const uint64_t ad = umma_desc_kmajor(a_base + ks * 2 * kALbo, kALbo, kSbo);
              umma_tf32(d_tmem, ad, bd, idesc, acc);
            }
            acc = 1;
          }
        }
        umma_commit(op_empty + ob);     // operand buffer may be overwritten once these MMAs retire
        umma_commit(tm_full + ob);      // accumulator stage ready for the epilogue
      }
    }
  } else if (warp < 6) {
    // ------------------------------ hi/lo splitter ------------------------------
    const int tid = threadIdx.x - 64;   // 0..127
    for (int it = 0; it < my_tiles; ++it) {
      const int s = it % Cfg::kStages;
      const uint32_t sph = (it / Cfg::kStages) & 1;
      const int ob = it & 1;
      const uint32_t oph = (it >> 1) & 1;
      const long long n0 = (long long)(chunk + it * p.n_chunks) * kBN;
      const int rows = (int)((p.V - n0) < kBN ? (p.V - n0) : kBN);
      mbar_wait(stg_full + s, sph);
      mbar_wait(op_empty + ob, oph ^ 1);
      const float* stg = reinterpret_cast<const float*>(smem + Cfg::kOffStg + s * Cfg::kBbytes);
      float* Bhi = reinterpret_cast<float*>(smem + Cfg::kOffBhi + ob * Cfg::kBbytes);
      float* Blo = reinterpret_cast<float*>(smem + Cfg::kOffBlo + ob * Cfg::kBbytes);
#pragma unroll
      for (int q = 0; q < (kBN * kKC) / 128; ++q) {
        const int item = q * 128 + tid;
        const int r = item % kBN;
        const int kc = (item / kBN + r) % kKC;      // diagonal rotation: conflict-free LDS and STS
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < rows) x = *reinterpret_cast<const float4*>(stg + r * kD + kc * 4);
        float4 hi = make_float4(to_tf32(x.x), to_tf32(x.y), to_tf32(x.z), to_tf32(x.w));
        float4 lo = make_float4(x.x - hi.x, x.y - hi.y, x.z - hi.z, x.w - hi.w);
        const int off = kc * (kBN * 4) + r * 4;
        *reinterpret_cast<float4*>(Bhi + off) = hi;
        *reinterpret_cast<float4*>(Blo + off) = lo;
      }
      fence_proxy_async();               // generic-proxy stores -> visible to the tensor-core (async) proxy
      mbar_arrive(op_full + ob);
      mbar_arrive(stg_empty + s);
    }
  } else if (warp < Cfg::kIssuer2) {
    // ------------------------------ epilogue ------------------------------
    const int quarter = warp & 3;                 // TMEM lane quarter this warp may access
    const int half = (warp - 6) >> 2;             // MODE_CE: the 32-column half of every tile this warp owns
    const int row = quarter * 32 + lane;
    const int grow = m_tile * kBM + row;
    const bool row_ok = grow < p.M;
    const uint32_t t_lane = tmem_base + ((uint32_t)(quarter * 32) << 16);
    float run_m = -INFINITY, run_s = 0.f;         // MODE_CE
    float g_lse = 0.f, g_scale = 0.f;             // MODE_GRAD
    long long g_tgt = -1;
    const int lhalf = kTopk ? half : 0;                          // MODE_TOPK: each warp set keeps its own candidate lists
    float* lval = reinterpret_cast<float*>(smem + Cfg::kOffTopk + lhalf * Cfg::kListBytes);           // [k][128]
    int* lidx = reinterpret_cast<int*>(smem + Cfg::kOffTopk + lhalf * Cfg::kListBytes + kMaxTopK * kBM * 4);
    int cnt = 0, minpos = 0, npend = 0;
    float thr = -INFINITY;
    float gb = -INFINITY;                         // MODE_TOPK: lower bound of the row's overall k-th best score, from p.row_bound
    float rmax = -INFINITY, rmax_pub = -INFINITY;  // best score of this CTA's stream for the row, and the value last published
    // MODE_TOPK_RANK: the positive's score (+inf on rows past M: nothing counted), its local column, and this stream's counts
    float r_s = INFINITY;
    long long r_pl = -1;
    int r_gt = 0, r_eq = 0;
    if (kRank && row_ok) { r_s = p.rank_score[grow]; r_pl = p.rank_pos[grow] - p.idx_offset; }
    if (MODE == MODE_GRAD && row_ok) { g_lse = p.lse[grow]; g_scale = p.row_scale[grow]; g_tgt = p.target[grow]; }
    float lin_bias = 0.f;
    if (MODE == MODE_LINEAR && row_ok && p.bias != nullptr) lin_bias = p.bias[blockIdx.y * p.b_bias + grow];
    for (int it = 0; it < my_tiles; ++it) {
      const int ob = it & 1;
      const uint32_t ph = (it >> 1) & 1;
      const long long n0 = (long long)(chunk + it * p.n_chunks) * kBN;
      mbar_wait(tm_full + ob, ph);
      tc_fence_after();
      if (kTopk && p.row_bound != nullptr && row_ok && (it < 8 ? (it & 3) == 1 : (it & 31) == 9)) {
        // Every warp set of every CTA of this row tile publishes the best score of its own stream (slot [2 chunk + half][row]).
        // Those are 2 n_chunks DIFFERENT catalogue items, so once >= k of them are known, their minimum is a lower bound of the row's overall k-th best:
        // a score at or below it cannot make the top-k and never touches the candidate list.  (Each stream's own k-th best is a far
        // weaker bound: all streams are equally long, so sharing THAT gains nothing -- measured.)
        int mn = 0x7fffffff;                 // (the encoding is order preserving: take the minimum on the integer images)
        const int* rb = p.row_bound + grow;
        int c = 0;
        const int n_streams = 2 * p.n_chunks;
        for (; c + 8 <= n_streams; c += 8) {
          int t[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) t[u] = __ldcg(rb + (long long)(c + u) * p.M);      // eight independent loads in flight
#pragma unroll
          for (int u = 0; u < 8; ++u) mn = min(mn, t[u]);
        }
        for (; c < n_streams; ++c) mn = min(mn, __ldcg(rb + (long long)c * p.M));
        gb = fmaxf(gb, bound_dec(mn));
      }
#pragma unroll 1
      for (int cc = (Cfg::kEpiWarps == 8 ? half : 0); cc < (Cfg::kEpiWarps == 8 ? half + 1 : kBN / 32); ++cc) {
        float v[32];
        tmem_ld32(t_lane + ob * kBN + cc * 32, v);
        const long long c0 = n0 + cc * 32;
        const int nvalid = (int)((p.V - c0) < 32 ? ((p.V - c0) > 0 ? (p.V - c0) : 0) : 32);
        if (MODE == MODE_LINEAR) {
          // Y[token][feature]: a warp's 32 features are 32 consecutive floats of one token row -> coalesced
          if (row_ok) {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              if (i < nvalid) {
                float* dst = C_p + (c0 + i) * p.ldc + grow;
                float y = v[i] + lin_bias;
                if (p.accumulate) y += *dst;
                *dst = y;
              }
            }
          }
        } else if (MODE == MODE_GRAD) {
          // transposed store Gt[v][m]: a warp's 32 rows are 32 consecutive floats -> coalesced 128-byte lines
          if (row_ok) {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              if (i < nvalid) {
                float g = __expf(v[i] - g_lse);
                if (c0 + i == g_tgt) g -= 1.0f;
                C_p[(c0 + i) * p.ldc + grow] = g * g_scale;
              }
            }
          }
        } else if (MODE == MODE_STORE) {
          if (row_ok) {
            float* dst = C_p + (long long)grow * p.ldc + c0;
            if (nvalid == 32 && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) {
#pragma unroll
              for (int i = 0; i < 32; i += 4) *reinterpret_cast<float4*>(dst + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i) if (i < nvalid) dst[i] = v[i];
            }
          }
        } else if (MODE == MODE_CE) {
          // running (max, sum exp) of this warp's column half: one max and three instructions (fma, ex2, add) per logit
          constexpr float kL2e = 1.4426950408889634f;
          if (nvalid == 32) {
            float cm = v[0];
#pragma unroll
            for (int i = 1; i < 32; ++i) cm = fmaxf(cm, v[i]);
            const float nm = fmaxf(run_m, cm);
            const float off = -nm * kL2e;
            float s0 = 0.f, s1 = 0.f;
#pragma unroll
            for (int i = 0; i < 32; i += 2) {
              float e0, e1;
              asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(fmaf(v[i], kL2e, off)));
              asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(fmaf(v[i + 1], kL2e, off)));
              s0 += e0; s1 += e1;
            }
            float rs;
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(rs) : "f"(fmaf(run_m, kL2e, off)));     // ex2(-inf) = 0 on the first tile
            run_s = run_s * rs + (s0 + s1);
            run_m = nm;
          } else if (nvalid > 0) {
            float cm = -INFINITY;
#pragma unroll
            for (int i = 0; i < 32; ++i) if (i < nvalid) cm = fmaxf(cm, v[i]);
            const float nm = fmaxf(run_m, cm);
            float s = 0.f;
#pragma unroll
            for (int i = 0; i < 32; ++i) if (i < nvalid) s += __expf(v[i] - nm);
            run_s = run_s * __expf(run_m - nm) + s;
            run_m = nm;
          }
        } else {   // MODE_TOPK
          // Thread-private k-best list (unsorted, cached minimum `thr`).  The 32 rows of a warp beat their thresholds at
          // different columns, so inserting on the spot would serialise the warp (one active lane per insert) and the
          // per-score bookkeeping would dominate the kernel.  Instead: a score that beats the row's threshold is PARKED in
          // the row's spare slots [k, kMaxTopK) (one compare + predicated stores per score), and the warp drains the parked
          // scores in lockstep -- the number of insert rounds is the maximum over the lanes, not the sum.
          const int k = p.k;
          const int pcap = kMaxTopK - k;
          if (nvalid < 32 || (p.skip_col0 && c0 == 0)) {       // ragged last tile / excluded column 0: never candidates
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (i >= nvalid || (p.skip_col0 && c0 + i == 0)) v[i] = -INFINITY;
          }
          // A score at or below `gb` cannot be among the row's k best of the WHOLE catalogue (see the refresh above).  Without it
          // every CTA's stream pays k (1 + ln(n/k)) list insertions per row, each a rescan of the k slots.
          float cmax = v[0];                                     // best score of this chunk for the row
#pragma unroll
          for (int i = 1; i < 32; ++i) cmax = fmaxf(cmax, v[i]);
          rmax = fmaxf(rmax, cmax);
          if (kRank && cmax >= r_s) {
            // every score of every tile is counted here, before the bound / threshold tests below may skip the tile; excluded
            // columns are -inf already.  A chunk whose maximum is below s_pos holds nothing to count.
#pragma unroll
            for (int i = 0; i < 32; ++i) { r_gt += v[i] > r_s; r_eq += v[i] == r_s; }
            if (r_pl >= c0 && r_pl < c0 + 32) {                  // the positive's own score, however this path rounded it
#pragma unroll
              for (int i = 0; i < 32; ++i)
                if (c0 + i == r_pl) { r_gt -= v[i] > r_s; r_eq -= v[i] == r_s; }
            }
          }
          auto drain = [&]() {
            while (__any_sync(0xffffffffu, npend > 0)) {
              if (npend > 0) {
                --npend;
                const float y = lval[(k + npend) * kBM + row];
                if (y > gb && (cnt < k || y > thr)) topk_insert(y, lidx[(k + npend) * kBM + row], lval, lidx, row, k, cnt, thr, minpos);
              }
            }
          };
          if (__any_sync(0xffffffffu, cnt < k && !(gb > -INFINITY)) || pcap < 8) {
            // filling the list (first tile, no bound yet) or no room to park: insert on the spot
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const float x = v[i];
              if (x != -INFINITY && x > gb && (cnt < k || x > thr)) topk_insert(x, (int)(c0 + i), lval, lidx, row, k, cnt, thr, minpos);
            }
          } else {
            const float eff = fmaxf(thr, gb);
            // most chunks hold no candidate for any of the warp's 32 rows once the bounds are tight: the chunk maximum decides
            // that, and the parking loop (whose slot index is a serial dependency) is skipped altogether
            if (__any_sync(0xffffffffu, cmax > eff))
#pragma unroll
            for (int i0 = 0; i0 < 32; i0 += 8) {
              // at most 8 scores are parked per row before the next check: drain when some row has fewer than 8 free slots
              if (__any_sync(0xffffffffu, npend > pcap - 8)) drain();
#pragma unroll
              for (int i = i0; i < i0 + 8; ++i) {
                const float x = v[i];
                if (x > eff) {
                  lval[(k + npend) * kBM + row] = x;
                  lidx[(k + npend) * kBM + row] = (int)c0 + i;
                  ++npend;
                }
              }
            }
            drain();
          }
        }
      }
      tc_fence_before();
      mbar_arrive(tm_empty + ob);
      if (kTopk && p.row_bound != nullptr && row_ok && rmax > rmax_pub) {
        __stcg(p.row_bound + (long long)(2 * chunk + half) * p.M + grow, bound_enc(rmax));
        rmax_pub = rmax;
      }
    }
    if (MODE == MODE_CE) {
      // the two column halves of a row meet once: the upper warp parks its pair, the lower one combines and stores
      float2* pair = reinterpret_cast<float2*>(smem + Cfg::kOffPair);
      if (half == 1) pair[row] = make_float2(run_m, run_s);
      asm volatile("bar.sync 1, %0;" ::"n"(32 * Cfg::kEpiWarps) : "memory");
      if (half == 0 && row_ok) {
        const float2 o2 = pair[row];
        const float nm = fmaxf(run_m, o2.x);
        float s = 0.f;
        if (run_s > 0.f) s += run_s * __expf(run_m - nm);
        if (o2.y > 0.f) s += o2.y * __expf(o2.x - nm);
        float* o = p.partial + ((long long)grow * p.n_chunks + chunk) * 2;
        o[0] = nm; o[1] = s;
      }
    }
    if (kTopk) {
      // the two warp sets of a row meet once: the upper set's candidates are inserted into the lower set's list
      int* pcnt = reinterpret_cast<int*>(smem + Cfg::kOffPair);
      int2* prank = reinterpret_cast<int2*>(smem + Cfg::kOffPair + kBM * 4);
      if (half == 1) {
        pcnt[row] = cnt;
        if (kRank) prank[row] = make_int2(r_gt, r_eq);
      }
      asm volatile("bar.sync 1, %0;" ::"n"(32 * Cfg::kEpiWarps) : "memory");
      if (half == 0) {
        if (kRank) { const int2 o = prank[row]; r_gt += o.x; r_eq += o.y; }
        const int cnt1 = pcnt[row];
        const float* oval = reinterpret_cast<const float*>(smem + Cfg::kOffTopk + Cfg::kListBytes);
        const int* oidx = reinterpret_cast<const int*>(smem + Cfg::kOffTopk + Cfg::kListBytes + kMaxTopK * kBM * 4);
        for (int s2 = 0; s2 < cnt1; ++s2) {
          const float y = oval[s2 * kBM + row];
          if (cnt < p.k || y > thr) topk_insert(y, oidx[s2 * kBM + row], lval, lidx, row, p.k, cnt, thr, minpos);
        }
      }
    }
    if (kTopk && row_ok && half == 0) {
      float* ov = p.pval + ((long long)grow * p.n_slots + chunk) * p.k;
      long long* oi = p.pidx + ((long long)grow * p.n_slots + chunk) * p.k;
      for (int s = 0; s < p.k; ++s) {
        const bool ok = s < cnt;
        ov[s] = ok ? lval[s * kBM + row] : -INFINITY;
        oi[s] = ok ? (long long)lidx[s * kBM + row] + p.idx_offset : -1;
      }
      // the partial layout has n_slots >= n_chunks lists per row: pad the ones no CTA produces
      for (int c = p.n_chunks + chunk; c < p.n_slots; c += p.n_chunks) {
        float* pv = p.pval + ((long long)grow * p.n_slots + c) * p.k;
        long long* pi = p.pidx + ((long long)grow * p.n_slots + c) * p.k;
        for (int s = 0; s < p.k; ++s) { pv[s] = -INFINITY; pi[s] = -1; }
      }
      if (kRank) {                                   // plain stores, one slot per (row, chunk): no atomics, deterministic
        int* rc = p.rank_counts + (long long)grow * p.n_slots * 2;
        rc[2 * chunk] = r_gt;
        rc[2 * chunk + 1] = r_eq;
        for (int c = p.n_chunks + chunk; c < p.n_slots; c += p.n_chunks) { rc[2 * c] = 0; rc[2 * c + 1] = 0; }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<Cfg::kTmem>(tmem_base);
  }
}

// ---- CE finalize: warp per row over the whole GPU, then one small CTA for the group means ---------
__global__ void __launch_bounds__(256) ce_rows_kernel(const float* __restrict__ partial, int n_parts, const float* __restrict__ out,
                                                      const float* __restrict__ table, const long long* __restrict__ target, int M,
                                                      int d, long long V, long long idx_offset, float* __restrict__ lse,
                                                      float* __restrict__ tgt_logit, float* __restrict__ row_loss) {
  pdl_launch_dependents();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * (blockDim.x >> 5) + warp;
  if (m >= M) return;
  float mx = -INFINITY;
  for (int i = lane; i < n_parts; i += 32) mx = fmaxf(mx, partial[((long long)m * n_parts + i) * 2]);
  mx = warp_max(mx);
  float s = 0.f;
  for (int i = lane; i < n_parts; i += 32) {
    const float pm = partial[((long long)m * n_parts + i) * 2], ps = partial[((long long)m * n_parts + i) * 2 + 1];
    if (ps > 0.f) s += ps * expf(pm - mx);
  }
  s = warp_sum(s);
  const float l = mx + logf(s);
  const long long t = target[m] - idx_offset;
  float dot = 0.f;
  if (t >= 0 && t < V)
    for (int j = lane; j < d; j += 32) dot = fmaf(out[(long long)m * d + j], table[t * d + j], dot);
  dot = warp_sum(dot);
  if (lane == 0) { lse[m] = l; tgt_logit[m] = dot; row_loss[m] = l - dot; }
}

// dot[m] = out[m] . table[ids[m] - idx_offset] when that row lives in this table (shard), else 0: the target logit of ce_rows_kernel
// on its own, in the same fixed fp32 order (lane-strided FMAs, then the warp sum), so the shards' answers can be summed
__global__ void __launch_bounds__(256) row_dot_kernel(const float* __restrict__ out, const float* __restrict__ table,
                                                      const long long* __restrict__ ids, int M, int d, long long V, long long idx_offset,
                                                      float* __restrict__ dot) {
  pdl_launch_dependents();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * (blockDim.x >> 5) + warp;
  if (m >= M) return;
  const long long t = ids[m] - idx_offset;
  float acc = 0.f;
  if (t >= 0 && t < V)
    for (int j = lane; j < d; j += 32) acc = fmaf(out[(long long)m * d + j], table[t * d + j], acc);
  acc = warp_sum(acc);
  if (lane == 0) dot[m] = acc;
}

__global__ void __launch_bounds__(256) ce_mean_kernel(const float* __restrict__ row_loss, int M, int n_groups, float* __restrict__ loss) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ double red[8];
  const int per_group = M / n_groups;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int g = 0; g < n_groups; ++g) {          // fixed summation order: deterministic
    double s = 0.0;
    for (int i = threadIdx.x; i < per_group; i += blockDim.x) s += (double)row_loss[g * per_group + i];
    s = warp_sum_d(s);
    if (lane == 0) red[warp] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
      loss[g] = (float)(t / per_group);
    }
    __syncthreads();
  }
}

// ---- scalar glue of the adversarial losses (acsasrec.py:129-142): pen_l = sqrt(pen_sq_l);
// loss_att = -ce_att + w * mean_l pen_l ; d loss_att / d pen_sq_l = w / (2 N pen_l) -------------------
__global__ void loss_combine_kernel(const double* __restrict__ pen_sq, int n_layers, const float* __restrict__ ce, const float* w_ptr,
                                    float w_val, float* __restrict__ loss_att, float* __restrict__ d_pen_sq) {
  pdl_launch_dependents();
  pdl_wait();
  if (threadIdx.x != 0) return;
  const float w = w_ptr ? w_ptr[0] : w_val;
  float acc = 0.f;
  for (int l = 0; l < n_layers; ++l) {
    const float pn = sqrtf((float)pen_sq[l]);
    acc += pn;
    if (d_pen_sq) d_pen_sq[l] = (w / (2.0f * n_layers)) / pn;
  }
  loss_att[0] = -ce[0] + (acc / n_layers) * w;
}

// ---- the three kernels above in ONE launch (the step's critical path runs through them): warp per row over the whole GPU ->
// lse / target logit / row loss; the LAST CTA to finish (device-scope counter, reset for the next launch) then takes the group
// means in a fixed order and evaluates the adversarial-loss glue -----------------------------------------------------------
__global__ void __launch_bounds__(256) ce_finalize_losses_kernel(const float* __restrict__ partial, int n_parts, const float* __restrict__ out,
                                                                 const float* __restrict__ table, const long long* __restrict__ target,
                                                                 int M, int d, long long V, long long idx_offset, int n_groups,
                                                                 float* __restrict__ lse, float* __restrict__ tgt_logit,
                                                                 float* row_loss, float* __restrict__ loss,
                                                                 const double* __restrict__ pen_sq, int n_layers, const float* w_ptr,
                                                                 float w_val, float* __restrict__ loss_att, float* __restrict__ d_pen_sq,
                                                                 unsigned int* counter) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ double red[8];
  __shared__ float s_loss[8];
  __shared__ bool s_last;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * (blockDim.x >> 5) + warp;
  if (m < M) {
    float mx = -INFINITY;
    for (int i = lane; i < n_parts; i += 32) mx = fmaxf(mx, partial[((long long)m * n_parts + i) * 2]);
    mx = warp_max(mx);
    float s = 0.f;
    for (int i = lane; i < n_parts; i += 32) {
      const float pm = partial[((long long)m * n_parts + i) * 2], ps = partial[((long long)m * n_parts + i) * 2 + 1];
      if (ps > 0.f) s += ps * expf(pm - mx);
    }
    s = warp_sum(s);
    const float l = mx + logf(s);
    const long long t = target[m] - idx_offset;
    float dot = 0.f;
    if (t >= 0 && t < V)
      for (int j = lane; j < d; j += 32) dot = fmaf(out[(long long)m * d + j], table[t * d + j], dot);
    dot = warp_sum(dot);
    if (lane == 0) { lse[m] = l; tgt_logit[m] = dot; row_loss[m] = l - dot; }
  }
  __threadfence();                                  // this CTA's row losses are visible device-wide before it checks in
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(counter, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  const volatile float* rl = row_loss;
  const int per_group = M / n_groups;
  for (int g = 0; g < n_groups; ++g) {              // fixed summation order: deterministic
    double s = 0.0;
    for (int i = threadIdx.x; i < per_group; i += blockDim.x) s += (double)rl[g * per_group + i];
    s = warp_sum_d(s);
    if (lane == 0) red[warp] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
      const float lg = (float)(t / per_group);
      loss[g] = lg;
      s_loss[g] = lg;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    *counter = 0u;                                  // ready for the next launch (graph replays included)
    if (loss_att != nullptr) {
      const float w = w_ptr ? w_ptr[0] : w_val;
      float acc = 0.f;
      for (int l = 0; l < n_layers; ++l) {
        const float pn = sqrtf((float)pen_sq[l]);
        acc += pn;
        if (d_pen_sq) d_pen_sq[l] = (w / (2.0f * n_layers)) / pn;
      }
      loss_att[0] = -s_loss[n_groups - 1] + (acc / n_layers) * w;
    }
  }
}

template <int MODE>
static int launch_tc(LogitsParams& p, cudaStream_t st, const char* who, int batch = 1) {
  using Cfg = TcCfg<MODE>;
  static_assert(Cfg::kSmemBytes <= 227 * 1024, "shared memory budget");
  logits_plan(p, batch);
  if (Cfg::kTopkMode) logits_plan_topk(p);
  cudaError_t e = cudaFuncSetAttribute(logits_tc_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
  if (e != cudaSuccess) { set_error("%s: smem attr: %s", who, cudaGetErrorString(e)); return ACSR_ERR_CUDA; }
  launch_pdl(logits_tc_kernel<MODE>, dim3(p.m_tiles * p.n_chunks, batch), dim3(Cfg::kThreads), Cfg::kSmemBytes, st, p);
  return check_launch(who);
}

static int validate_common(const float* out, const float* table, int M, long long V, int d, int passes, const char* who) {
  ACSR_REQUIRE(out && table, "%s: NULL input", who);
  ACSR_REQUIRE(M > 0 && V > 0, "%s: bad sizes M=%d V=%lld", who, M, V);
  if (d != kD && (d < 4 || d > 1024 || (d & 3))) {
    set_error("%s: hidden size %d unsupported (64 on the tensor-core path; multiples of 4 up to 1024 on the fp32 path)", who, d);
    return ACSR_ERR_UNSUPPORTED;
  }
  ACSR_REQUIRE(passes == 1 || passes == 3, "%s: passes must be 1 (TF32) or 3 (3xTF32)", who);
  ACSR_REQUIRE(V < (1ll << 31), "%s: V too large", who);
  return ACSR_OK;
}

}  // namespace acsr

using namespace acsr;

extern "C" {

int acsr_logits_num_chunks(int M, int64_t V) {
  LogitsParams p = {};
  p.M = M; p.V = V;
  if (M <= 0 || V <= 0) return 0;
  logits_plan(p);
  return p.n_chunks;
}

int acsr_logits_num_chunks_d(int M, int64_t V, int d) {
  if (d == kD) return acsr_logits_num_chunks(M, V);
  return acsr_gemm_ce_parts(V);
}

int acsr_logits_store(const float* out, const float* table, int M, int64_t V, int d, int passes, float* scores, int64_t ldc,
                      void* stream) {
  int rc = validate_common(out, table, M, V, d, passes, "logits_store");
  if (rc) return rc;
  ACSR_REQUIRE(scores && ldc >= V, "logits_store: bad output");
  LogitsParams p = {};
  p.out = out; p.table = table; p.M = M; p.V = V; p.passes = passes; p.C = scores; p.ldc = ldc;
  // other hidden sizes: the K-streamed tcgen05 GEMM (gemm_ks.cu), rows of `out` on M, table rows on N
  if (d != kD) return gemm_logits(ACSR_EPI_STORE, out, table, M, V, d, passes, scores, ldc, nullptr, nullptr, nullptr, nullptr, (cudaStream_t)stream);
  return launch_tc<MODE_STORE>(p, (cudaStream_t)stream, "logits_store");
}

int acsr_logits_ce_partial(const float* out, const float* table, int M, int64_t V, int d, int passes, float* partial, void* stream) {
  int rc = validate_common(out, table, M, V, d, passes, "logits_ce_partial");
  if (rc) return rc;
  ACSR_REQUIRE(partial, "logits_ce_partial: NULL output");
  LogitsParams p = {};
  p.out = out; p.table = table; p.M = M; p.V = V; p.passes = passes; p.partial = partial;
  // other hidden sizes: K-streamed tcgen05 GEMM with the (max, sum exp) epilogue; partial is [M, acsr_logits_num_chunks_d(M, V, d), 2]
  if (d != kD) return gemm_logits(ACSR_EPI_CE, out, table, M, V, d, passes, nullptr, V, partial, nullptr, nullptr, nullptr, (cudaStream_t)stream);
  return launch_tc<MODE_CE>(p, (cudaStream_t)stream, "logits_ce_partial");
}

int acsr_ce_finalize(const float* partial, int n_parts, const float* out, const float* table, const int64_t* target, int M, int d,
                     int64_t V, int64_t idx_offset, int n_groups, float* lse, float* tgt_logit, float* row_loss, float* loss,
                     void* stream) {
  ACSR_REQUIRE(partial && out && table && target && lse && tgt_logit && row_loss && loss, "ce_finalize: NULL pointer");
  ACSR_REQUIRE(M > 0 && n_parts > 0 && n_groups > 0 && n_groups <= 8 && M % n_groups == 0, "ce_finalize: bad sizes");
  launch_pdl(ce_rows_kernel, dim3((M + 7) / 8), dim3(256), 0, (cudaStream_t)stream, partial, n_parts, out, table,
             (const long long*)target, M, d, (long long)V, (long long)idx_offset, lse, tgt_logit, row_loss);
  launch_pdl(ce_mean_kernel, dim3(1), dim3(256), 0, (cudaStream_t)stream, (const float*)row_loss, M, n_groups, loss);
  return check_launch("ce_finalize");
}

int acsr_ce_finalize_losses(const float* partial, int n_parts, const float* out, const float* table, const int64_t* target, int M, int d,
                            int64_t V, int64_t idx_offset, int n_groups, float* lse, float* tgt_logit, float* row_loss, float* loss,
                            const double* pen_sq, int n_layers, const float* mask_loss_weight, float mask_loss_weight_value,
                            float* loss_attacked, float* d_pen_sq, uint32_t* counter, void* stream) {
  ACSR_REQUIRE(partial && out && table && target && lse && tgt_logit && row_loss && loss && counter, "ce_finalize_losses: NULL pointer");
  ACSR_REQUIRE(M > 0 && n_parts > 0 && n_groups > 0 && n_groups <= 8 && M % n_groups == 0, "ce_finalize_losses: bad sizes");
  ACSR_REQUIRE(loss_attacked == nullptr || (pen_sq != nullptr && n_layers > 0), "ce_finalize_losses: penalty inputs missing");
  launch_pdl(ce_finalize_losses_kernel, dim3((M + 7) / 8), dim3(256), 0, (cudaStream_t)stream, partial, n_parts, out, table,
             (const long long*)target, M, d, (long long)V, (long long)idx_offset, n_groups, lse, tgt_logit, row_loss, loss, pen_sq, n_layers,
             mask_loss_weight, mask_loss_weight_value, loss_attacked, d_pen_sq, (unsigned int*)counter);
  return check_launch("ce_finalize_losses");
}

int acsr_loss_combine(const double* pen_sq, int n_layers, const float* ce_attacked, const float* mask_loss_weight, float mask_loss_weight_value,
                      float* loss_attacked, float* d_pen_sq, void* stream) {
  ACSR_REQUIRE(pen_sq && ce_attacked && loss_attacked && n_layers > 0, "loss_combine: bad arguments");
  launch_pdl(loss_combine_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, pen_sq, n_layers, ce_attacked, mask_loss_weight,
             mask_loss_weight_value, loss_attacked, d_pen_sq);
  return check_launch("loss_combine");
}

int acsr_logits_ce_grad(const float* out, const float* table, const float* lse, const int64_t* target, const float* row_scale, int M,
                        int64_t V, int d, int passes, float* G, int64_t ldg, void* stream) {
  int rc = validate_common(out, table, M, V, d, passes, "logits_ce_grad");
  if (rc) return rc;
  ACSR_REQUIRE(lse && target && row_scale && G && ldg >= M, "logits_ce_grad: bad arguments");
  LogitsParams p = {};
  p.out = out; p.table = table; p.M = M; p.V = V; p.passes = passes; p.C = G; p.ldc = ldg;
  p.lse = lse; p.target = (const long long*)target; p.row_scale = row_scale;
  if (d != kD) return gemm_logits(ACSR_EPI_CE_GRAD, out, table, M, V, d, passes, G, ldg, nullptr, lse, (const long long*)target, row_scale, (cudaStream_t)stream);
  return launch_tc<MODE_GRAD>(p, (cudaStream_t)stream, "logits_ce_grad");
}

int acsr_linear_tc(const float* X, int64_t rows, int K, const float* W, int N, int64_t w_stride_n, int64_t w_stride_k,
                   const float* bias, int accumulate, float* Y, int64_t ldy, int batch, int64_t stride_x, int64_t stride_w,
                   int64_t stride_bias, int64_t stride_y, int passes, void* stream) {
  ACSR_REQUIRE(X && W && Y, "linear_tc: NULL pointer");
  ACSR_REQUIRE(rows >= 0 && N > 0 && batch > 0 && batch < 65536 && ldy >= N, "linear_tc: bad sizes");
  if (K != kD) { set_error("linear_tc: K=%d unsupported by the tensor-core path in ABI v1 (64)", K); return ACSR_ERR_UNSUPPORTED; }
  ACSR_REQUIRE(passes == 1 || passes == 3, "linear_tc: passes must be 1 or 3");
  if (rows == 0) return ACSR_OK;
  LogitsParams p = {};
  p.out = W; p.table = X; p.M = N; p.V = rows; p.passes = passes; p.C = Y; p.ldc = ldy;
  p.out_sn = w_stride_n; p.out_sk = w_stride_k; p.bias = bias; p.accumulate = accumulate;
  p.b_out = stride_w; p.b_table = stride_x; p.b_bias = stride_bias; p.b_C = stride_y;
  return launch_tc<MODE_LINEAR>(p, (cudaStream_t)stream, "linear_tc", batch);
}

int acsr_logits_topk_partial(const float* out, const float* table, int M, int64_t V, int d, int passes, int k, int64_t idx_offset,
                             int skip_col0, float* partial_val, int64_t* partial_idx, void* stream) {
  return acsr_logits_topk_partial_ws(out, table, M, V, d, passes, k, idx_offset, skip_col0, partial_val, partial_idx, nullptr, stream);
}

int acsr_logits_topk_partial_ws(const float* out, const float* table, int M, int64_t V, int d, int passes, int k, int64_t idx_offset,
                                int skip_col0, float* partial_val, int64_t* partial_idx, int32_t* row_bound, void* stream) {
  int rc = validate_common(out, table, M, V, d, passes, "logits_topk_partial");
  if (rc) return rc;
  ACSR_REQUIRE(partial_val && partial_idx, "logits_topk_partial: NULL output");
  if (k < 1 || k > kMaxTopK) { set_error("logits_topk_partial: k=%d unsupported (1..%d)", k, kMaxTopK); return ACSR_ERR_UNSUPPORTED; }
  LogitsParams p = {};
  p.out = out; p.table = table; p.M = M; p.V = V; p.passes = passes;
  p.k = k; p.idx_offset = idx_offset; p.skip_col0 = skip_col0; p.pval = partial_val; p.pidx = (long long*)partial_idx;
  if (d != kD) return launch_logits_simt(MODE_TOPK, p, d, (cudaStream_t)stream, "logits_topk_partial");   // fp32 FMA path (logits_simt.cu)
  {
    LogitsParams q = p;                    // the plan decides how many CTAs share a row tile: the bound needs at least k of them
    logits_plan(q);
    logits_plan_topk(q);
    p.row_bound = (row_bound != nullptr && 2 * q.n_chunks >= k) ? row_bound : nullptr;     // two streams (warp sets) per CTA
    if (p.row_bound != nullptr) {
      // every byte 0x80: a very negative score (-3.4e38) in the order-preserving int encoding = "nothing published yet"
      cudaError_t e = cudaMemsetAsync(row_bound, 0x80, (size_t)M * 2 * q.n_chunks * sizeof(int32_t), (cudaStream_t)stream);
      if (e != cudaSuccess) { set_error("logits_topk_partial: memset: %s", cudaGetErrorString(e)); return ACSR_ERR_CUDA; }
    }
  }
  return launch_tc<MODE_TOPK>(p, (cudaStream_t)stream, "logits_topk_partial");
}

int acsr_row_dot(const float* out, const float* table, const int64_t* ids, int M, int d, int64_t V, int64_t idx_offset, float* dot,
                 void* stream) {
  ACSR_REQUIRE(out && table && ids && dot, "row_dot: NULL pointer");
  ACSR_REQUIRE(M > 0 && V > 0 && d > 0, "row_dot: bad sizes M=%d V=%lld d=%d", M, (long long)V, d);
  launch_pdl(row_dot_kernel, dim3((M + 7) / 8), dim3(256), 0, (cudaStream_t)stream, out, table, (const long long*)ids, M, d, (long long)V,
             (long long)idx_offset, dot);
  return check_launch("row_dot");
}

int acsr_logits_topk_rank_partial(const float* out, const float* table, int M, int64_t V, int d, int passes, int k, int64_t idx_offset,
                                  int skip_col0, const int64_t* positive, const float* pos_score, float* partial_val,
                                  int64_t* partial_idx, int32_t* partial_counts, int32_t* row_bound, void* stream) {
  int rc = validate_common(out, table, M, V, d, passes, "logits_topk_rank_partial");
  if (rc) return rc;
  ACSR_REQUIRE(partial_val && partial_idx && positive && pos_score && partial_counts, "logits_topk_rank_partial: NULL pointer");
  if (k < 1 || k > kMaxTopK) { set_error("logits_topk_rank_partial: k=%d unsupported (1..%d)", k, kMaxTopK); return ACSR_ERR_UNSUPPORTED; }
  LogitsParams p = {};
  p.out = out; p.table = table; p.M = M; p.V = V; p.passes = passes;
  p.k = k; p.idx_offset = idx_offset; p.skip_col0 = skip_col0; p.pval = partial_val; p.pidx = (long long*)partial_idx;
  p.rank_pos = (const long long*)positive; p.rank_score = pos_score; p.rank_counts = partial_counts;
  if (d != kD) return launch_logits_simt(MODE_TOPK_RANK, p, d, (cudaStream_t)stream, "logits_topk_rank_partial");
  {
    LogitsParams q = p;                    // the shared bound as in acsr_logits_topk_partial_ws
    logits_plan(q);
    logits_plan_topk(q);
    p.row_bound = (row_bound != nullptr && 2 * q.n_chunks >= k) ? row_bound : nullptr;
    if (p.row_bound != nullptr) {
      cudaError_t e = cudaMemsetAsync(row_bound, 0x80, (size_t)M * 2 * q.n_chunks * sizeof(int32_t), (cudaStream_t)stream);
      if (e != cudaSuccess) { set_error("logits_topk_rank_partial: memset: %s", cudaGetErrorString(e)); return ACSR_ERR_CUDA; }
    }
  }
  return launch_tc<MODE_TOPK_RANK>(p, (cudaStream_t)stream, "logits_topk_rank_partial");
}

}  // extern "C"
