// Backward of an encoder layer's dense part after its attention (layers.py:676-684, 790-798) as ONE tcgen05 launch,
// hidden size 64, inner size a multiple of 64 up to 256.  Per 128-token tile:
//   1. FFN LayerNorm backward: d_out -> d_pre_f (the residual part of d_h) and d_z2 = d_pre_f * mask_f
//   2. per 64-wide chunk c of the inner axis: acc_c = d_z2.W2[:, c] ; d_z1_c = acc_c * act'(z1_c + b1_c) ; acc_h += d_z1_c.W1[c, :]
//   3. attention LayerNorm backward of d_h = acc_h + d_pre_f: d_xres (written) and d_hz = d_pre_a * mask_a
//   4. d_ctx = d_hz.Wo
// As six launches (two row-wise LayerNorm backwards, three acsr_linear_tok GEMMs, the activation backward) the chain sat on the
// critical path of every non-last layer's backward, and d_a1 / d_z1 ([rows, I] each) made round trips through L2 although only
// rows < param_rows of d_z2 / d_z1 / d_hz are read afterwards (by the weight gradients).  Here the intermediates stay in TENSOR
// MEMORY: each epilogue leaves its result split into hi / lo TF32 halves with tcgen05.st and the next MMA reads it as its A
// operand (TS form, as in logits_bwd.cu / proj_bwd.cu).  Bias gradients are not computed here: the weight-gradient launch takes
// them as column sums of its left operand (d_z2, d_z1, d_hz).
//
// TMEM columns (128 lanes x 512, one CTA per SM):
//   [0,128)   A: d_z2 hi / lo, later d_hz hi / lo           [128,256) C[2]: chunk accumulators, overwritten IN PLACE by d_z1 hi
//   [256,384) L[2]: d_z1 lo                                  [384,448) acc_h          [448,512) acc_ctx
// Weights arrive pre-split (acsr_dense_bwd_prep, once per step): Wo^T, the W2 column chunks and the W1 row chunks as (hi, lo) TF32
// operands in the canonical K-major UMMA layout, so staging one is a 32 KB bulk copy.  Wo^T stays resident, the chunks stream
// through two 2-slot rings (288 KB at I = 256 would not fit).
// Roles (352 threads, persistent over tiles): warp 0 bulk-copy producer; warp 1 issues the d_z2.W2 chunk MMAs and d_hz.Wo, warp 2
// the acc_h MMAs, so chunk c+1's first GEMM runs under chunk c's epilogue; warps 3-10 are row workers, two per TMEM lane quarter:
// one thread owns 32 columns of one token row (the LayerNorm row sums are exchanged between the two threads of a row through
// shared memory), so the activation derivative of a chunk and the Philox masks are spread over all eight warps.
#include "acsr_common.cuh"
#include "../../include/acsr.h"

namespace acsr {

constexpr int kDbThreads = 352;
constexpr int kDbD = 64;
constexpr int kDbBM = 128;
constexpr int kDbOpFloats = 64 * 64;              // one 64 x 64 operand (hi or lo)
constexpr int kDbBlkBytes = 2 * kDbOpFloats * 4;  // hi + lo: 32 KB
constexpr int kDbMaxI = 256;

struct DbParams {
  const float* d_out; long long rows, act_rows, res_rows, param_rows; int I, act, passes;
  const float* ops;
  const float *z2, *b2, *h, *lnF_w, *st_f, *z1, *b1, *hz, *bo, *x_res, *lnA_w, *st_a;
  float p_drop; const float *mask_a, *mask_f; const RngState* rng; uint32_t stream_a, stream_f;
  float *d_z2, *d_z1, *d_hz, *d_xres, *d_ctx;
  float *g_lnF_w, *g_lnF_b, *g_lnA_w, *g_lnA_b;
  int m_tiles, w_static;
};

// ---- weights -> (hi, lo) TF32 operands B(n, k), canonical K-major layout: block 0 = Wo^T (n, k) = Wo[k][n]; 1..nc: W2 column
// chunk c, (n, k) = W2[k][c*64 + n]; nc+1..2nc: W1 row chunk c, (n, k) = W1[c*64 + k][n] ----
__global__ void __launch_bounds__(256) dense_bwd_prep_kernel(const float* __restrict__ Wo, const float* __restrict__ W1,
                                                             const float* __restrict__ W2, int I, float* __restrict__ ops) {
  pdl_wait();
  const int nc = I / 64, blk = blockIdx.x;
  float* hi = ops + (long long)blk * 2 * kDbOpFloats;
  float* lo = hi + kDbOpFloats;
  for (int e = threadIdx.x; e < 64 * 16; e += blockDim.x) {
    const int kc = e >> 6, n = e & 63;               // consecutive threads: consecutive n (coalesced source rows)
    float x[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = kc * 4 + j;
      if (blk == 0) x[j] = Wo[k * 64 + n];
      else if (blk <= nc) x[j] = W2[(long long)k * I + (blk - 1) * 64 + n];
      else x[j] = W1[(long long)((blk - 1 - nc) * 64 + k) * 64 + n];
    }
    const float4 h4 = make_float4(to_tf32(x[0]), to_tf32(x[1]), to_tf32(x[2]), to_tf32(x[3]));
    const int off = kc * 256 + n * 4;
    *reinterpret_cast<float4*>(hi + off) = h4;
    *reinterpret_cast<float4*>(lo + off) = make_float4(x[0] - h4.x, x[1] - h4.y, x[2] - h4.z, x[3] - h4.w);
  }
}

struct DbCfg {
  static constexpr int kOffWo = 0;
  static constexpr int kOffW2 = kOffWo + kDbBlkBytes;          // [2] W2 column chunks
  static constexpr int kOffW1 = kOffW2 + 2 * kDbBlkBytes;      // [2] W1 row chunks
  static constexpr int kOffPar = kOffW1 + 2 * kDbBlkBytes;     // b2, lnF_w, bo, lnA_w [64 each], b1 [256]
  static constexpr int kParFloats = 4 * 64 + kDbMaxI;
  static constexpr int kOffLn = kOffPar + kParFloats * 4;      // per-CTA LayerNorm parameter-gradient sums [4][64]
  static constexpr int kOffXch = kOffLn + 4 * 64 * 4;          // row-sum exchange [2 norms][2 halves][128 rows] float2
  static constexpr int kOffBar = kOffXch + 2 * 2 * kDbBM * 8;
  static constexpr int kNumBars = 24;
  static constexpr int kSmemBytes = kOffBar + kNumBars * 8 + 16;
  static constexpr int kColA = 0, kColC = 128, kColL = 256, kColH = 384, kColX = 448;
};

// dropout multipliers of columns c0..c0+31 of saved row `row`: the Philox counters of bdrl_{fwd,bwd}_kernel (element e -> call
// e>>2, word e&3), or the explicit mask
__device__ __forceinline__ void db_drop32(const DbParams& p, const float* mask, uint32_t stream, long long row, int c0, bool ok,
                                          float* m) {
  if (!ok || (mask == nullptr && !(p.p_drop > 0.f && p.rng != nullptr))) {
#pragma unroll
    for (int i = 0; i < 32; ++i) m[i] = 1.0f;
  } else if (mask != nullptr) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const float4 mm = __ldg(reinterpret_cast<const float4*>(mask + row * kDbD + c0) + q);
      m[4 * q] = mm.x; m[4 * q + 1] = mm.y; m[4 * q + 2] = mm.z; m[4 * q + 3] = mm.w;
    }
  } else {
    const float inv_keep = 1.0f / (1.0f - p.p_drop);
    const unsigned long long seed = p.rng->seed, step = p.rng->step;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const uint4 w = philox4x32(seed, step, stream, (unsigned long long)row * 16 + (c0 >> 2) + q);
      m[4 * q] = drop_mult(w.x, p.p_drop, inv_keep); m[4 * q + 1] = drop_mult(w.y, p.p_drop, inv_keep);
      m[4 * q + 2] = drop_mult(w.z, p.p_drop, inv_keep); m[4 * q + 3] = drop_mult(w.w, p.p_drop, inv_keep);
    }
  }
}

__device__ __forceinline__ void db_load32(const float* src, bool ok, float* v) {
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const float4 x = ok ? __ldg(reinterpret_cast<const float4*>(src) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
    v[4 * q] = x.x; v[4 * q + 1] = x.y; v[4 * q + 2] = x.z; v[4 * q + 3] = x.w;
  }
}

__device__ __forceinline__ void db_store32(float* dst, const float* v) {
#pragma unroll
  for (int q = 0; q < 8; ++q) reinterpret_cast<float4*>(dst)[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
}

// 32 columns of one row -> TMEM (hi at column c, lo at c + lo_off)
__device__ __forceinline__ void db_store_split(uint32_t taddr, uint32_t lo_off, float* v) {
  float lo[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) { const float hi = to_tf32(v[i]); lo[i] = v[i] - hi; v[i] = hi; }
  tmem_st32(taddr, v);
  tmem_st32(taddr + lo_off, lo);
}

// column sums of a warp's 32 rows x 32 columns (destroys v): lane j ends with column j in v[0] (butterfly reduce-scatter)
__device__ __forceinline__ float db_warp_colsum32(float* v, int lane) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const bool up = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < off; ++i) {
      const float send = up ? v[i] : v[i + off];
      const float keep = up ? v[i + off] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}

__device__ __forceinline__ void db_pair_sync(int quarter) {   // the two row-worker warps of one TMEM lane quarter
  asm volatile("bar.sync %0, 64;" ::"r"(1 + quarter) : "memory");
}

// LayerNorm backward of 32 columns of a row, given xhat and g = d_out.  Accumulates the gamma / beta gradient column sums
// (rows < param_rows) into sLn, exchanges the row sums with the partner thread (other half of the row) and returns
// d_pre = rstd (g w - mean(g w) - xhat mean(g w xhat)) in g.
__device__ __forceinline__ void db_ln_bwd(float* g, const float* xh, const float* w, float rstd, bool keep, float* sLn_w,
                                          float* sLn_b, float2* xch, int half, int row, int quarter, int lane) {
  float t[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) t[i] = keep ? g[i] * xh[i] : 0.f;
  atomicAdd(sLn_w + lane, db_warp_colsum32(t, lane));
#pragma unroll
  for (int i = 0; i < 32; ++i) t[i] = keep ? g[i] : 0.f;
  atomicAdd(sLn_b + lane, db_warp_colsum32(t, lane));
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    g[i] *= w[i];
    s1 += g[i];
    s2 += g[i] * xh[i];
  }
  xch[half * kDbBM + row] = make_float2(s1, s2);
  db_pair_sync(quarter);
  const float2 o = xch[(half ^ 1) * kDbBM + row];
  // the same order of the two partial sums in both threads of the row
  s1 = (half == 0 ? s1 + o.x : o.x + s1) * (1.0f / kDbD);
  s2 = (half == 0 ? s2 + o.y : o.y + s2) * (1.0f / kDbD);
#pragma unroll
  for (int i = 0; i < 32; ++i) g[i] = rstd * (g[i] - s1 - xh[i] * s2);
}

template <int ACT>
__device__ __forceinline__ void db_act_bwd32(float* v, const float* z, const float* b) {
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] *= act_bwd(ACT, z[i] + b[i]);
}

__global__ void __launch_bounds__(kDbThreads, 1) dense_bwd_kernel(const DbParams p) {
  using Cfg = DbCfg;
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nc = p.I / 64;
  float* sPar = reinterpret_cast<float*>(smem + Cfg::kOffPar);
  float *s_b2 = sPar, *s_lnFw = sPar + 64, *s_bo = sPar + 128, *s_lnAw = sPar + 192, *s_b1 = sPar + 256;
  float* sLn = reinterpret_cast<float*>(smem + Cfg::kOffLn);     // lnF_w, lnF_b, lnA_w, lnA_b gradients
  float2* xch = reinterpret_cast<float2*>(smem + Cfg::kOffXch);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kOffBar);
  uint64_t* wo_full = bars;
  uint64_t* w2_full = bars + 1;      // [2]
  uint64_t* w2_empty = bars + 3;     // [2]
  uint64_t* w1_full = bars + 5;      // [2]
  uint64_t* w1_empty = bars + 7;     // [2]
  uint64_t* a_full = bars + 9;       // d_z2 (hi, lo) sits in TMEM
  uint64_t* c_full = bars + 10;      // [2] chunk accumulator ready
  uint64_t* c_empty = bars + 12;     // [2] acc_h MMA of the chunk retired: its C / L columns are free
  uint64_t* a_ready = bars + 14;     // [2] d_z1 chunk (hi, lo) sits in TMEM
  uint64_t* h_full = bars + 16;      // acc_h ready
  uint64_t* hz_full = bars + 17;     // d_hz (hi, lo) sits in TMEM
  uint64_t* x_full = bars + 18;      // acc_ctx ready
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + Cfg::kNumBars);

  pdl_launch_dependents();
  if (threadIdx.x == 0) {
    mbar_init(wo_full, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(w2_full + s, 1); mbar_init(w2_empty + s, 1); mbar_init(w1_full + s, 1); mbar_init(w1_empty + s, 1);
      mbar_init(c_full + s, 1); mbar_init(c_empty + s, 1); mbar_init(a_ready + s, 256);
    }
    mbar_init(a_full, 256); mbar_init(h_full, 1); mbar_init(hz_full, 256); mbar_init(x_full, 1);
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  // parameters (never written inside a step): staged before the dependency wait
  for (int i = threadIdx.x; i < 64; i += kDbThreads) { s_b2[i] = p.b2[i]; s_lnFw[i] = p.lnF_w[i]; s_bo[i] = p.bo[i]; s_lnAw[i] = p.lnA_w[i]; }
  for (int i = threadIdx.x; i < p.I; i += kDbThreads) s_b1[i] = p.b1[i];
  for (int i = threadIdx.x; i < 4 * 64; i += kDbThreads) sLn[i] = 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int my_tiles = (int)blockIdx.x < p.m_tiles ? (p.m_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;

  if (warp == 0) {
    // ------------------------------ producer: prepared weight blocks, one bulk copy each ------------------------------
    if (lane == 0 && my_tiles > 0) {
      if (!p.w_static) pdl_wait();
      mbar_arrive_expect_tx(wo_full, kDbBlkBytes);
      bulk_g2s(smem + Cfg::kOffWo, p.ops, kDbBlkBytes, wo_full);
      for (int it = 0; it < my_tiles; ++it)
        for (int c = 0; c < nc; ++c) {
          const int g = it * nc + c, b = g & 1;
          const uint32_t ph = (g >> 1) & 1;
          mbar_wait(w2_empty + b, ph ^ 1);
          mbar_arrive_expect_tx(w2_full + b, kDbBlkBytes);
          bulk_g2s(smem + Cfg::kOffW2 + b * kDbBlkBytes, p.ops + (long long)(1 + c) * 2 * kDbOpFloats, kDbBlkBytes, w2_full + b);
          mbar_wait(w1_empty + b, ph ^ 1);
          mbar_arrive_expect_tx(w1_full + b, kDbBlkBytes);
          bulk_g2s(smem + Cfg::kOffW1 + b * kDbBlkBytes, p.ops + (long long)(1 + nc + c) * 2 * kDbOpFloats, kDbBlkBytes, w1_full + b);
        }
    }
  } else if (warp == 1 || warp == 2) {
    if (lane == 0 && my_tiles > 0) {
      const uint32_t idesc = umma_idesc_tf32(kDbBM, 64);
      constexpr uint32_t kLbo = 64 * 16, kSbo = 128;
      const int npass = p.passes == 3 ? 3 : 1;
      // d (+)= A[tmem ahi (hi), alo (lo)] . B^T over K = 64; 3xTF32: small cross terms first, hi.hi last
      auto mma24 = [&](uint32_t d_tmem, uint32_t ahi, uint32_t alo, uint32_t bsm, bool first_zero) {
        uint32_t acc = first_zero ? 0u : 1u;
        for (int ps = 0; ps < npass; ++ps) {
          const uint32_t a_base = (npass == 3 && ps == 0) ? alo : ahi;
          const uint32_t b_base = bsm + ((npass == 3 && ps == 1) ? kDbOpFloats * 4 : 0);
#pragma unroll
          for (int ks = 0; ks < 8; ++ks) {
            umma_tf32_ts(d_tmem, a_base + ks * 8, umma_desc_kmajor(b_base + ks * 2 * kLbo, kLbo, kSbo), idesc, acc);
            acc = 1;
          }
        }
      };
      const uint32_t a_hi = tmem_base + Cfg::kColA, a_lo = a_hi + 64;
      if (warp == 1) {
        // ---- issuer A: chunk accumulators acc_c = d_z2 . W2[:, c], then acc_ctx = d_hz . Wo ----
        for (int it = 0; it < my_tiles; ++it) {
          mbar_wait(a_full, it & 1);
          tc_fence_after();
          for (int c = 0; c < nc; ++c) {
            const int g = it * nc + c, b = g & 1;
            const uint32_t ph = (g >> 1) & 1;
            mbar_wait(w2_full + b, ph);
            mbar_wait(c_empty + b, ph ^ 1);
            tc_fence_after();
            mma24(tmem_base + Cfg::kColC + b * 64, a_hi, a_lo, smem_u32(smem + Cfg::kOffW2 + b * kDbBlkBytes), true);
            umma_commit(w2_empty + b);
            umma_commit(c_full + b);
          }
          mbar_wait(hz_full, it & 1);         // (d_hz replaced d_z2 in A after every chunk MMA of the tile had completed)
          if (it == 0) mbar_wait(wo_full, 0);
          tc_fence_after();
          mma24(tmem_base + Cfg::kColX, a_hi, a_lo, smem_u32(smem + Cfg::kOffWo), true);
          umma_commit(x_full);
        }
      } else {
        // ---- issuer B: acc_h (+)= d_z1 chunk . W1[c, :] ----
        for (int it = 0; it < my_tiles; ++it) {
          for (int c = 0; c < nc; ++c) {
            const int g = it * nc + c, b = g & 1;
            const uint32_t ph = (g >> 1) & 1;
            mbar_wait(a_ready + b, ph);
            mbar_wait(w1_full + b, ph);
            tc_fence_after();
            mma24(tmem_base + Cfg::kColH, tmem_base + Cfg::kColC + b * 64, tmem_base + Cfg::kColL + b * 64,
                  smem_u32(smem + Cfg::kOffW1 + b * kDbBlkBytes), c == 0);
            umma_commit(w1_empty + b);
            umma_commit(c_empty + b);
          }
          umma_commit(h_full);
        }
      }
    }
  } else {
    // ------------------------------ row workers: one thread = 32 columns of one token row ------------------------------
    pdl_wait();
    const int quarter = warp & 3;
    const int half = (warp - 3) >> 2;
    const int c0 = half * 32;
    const int row = quarter * 32 + lane;
    const uint32_t t_lane = tmem_base + ((uint32_t)(quarter * 32) << 16);
    float2* xchF = xch;
    float2* xchA = xch + 2 * kDbBM;
    for (int it = 0; it < my_tiles; ++it) {
      const long long grow = (long long)(blockIdx.x + it * gridDim.x) * kDbBM + row;
      const bool row_ok = grow < p.rows, keep = grow < p.param_rows;
      const long long ta = row_ok ? grow % p.act_rows : 0, tr = row_ok ? grow % p.res_rows : 0;
      // ---- 1. FFN LayerNorm backward: d_pre_f (kept for d_h) and d_z2 -> TMEM (and global, rows < param_rows) ----
      float dpre[32];
      {
        float xh[32], m[32];
        db_load32(p.d_out + grow * kDbD + c0, row_ok, dpre);
        db_load32(p.z2 + ta * kDbD + c0, row_ok, xh);
        db_load32(p.h + ta * kDbD + c0, row_ok, m);
        const float mean = row_ok ? p.st_f[2 * ta] : 0.f, rstd = row_ok ? p.st_f[2 * ta + 1] : 0.f;
#pragma unroll
        for (int i = 0; i < 32; ++i) xh[i] += s_b2[c0 + i];
        {
          float mk[32];
          db_drop32(p, p.mask_f, p.stream_f, ta, c0, row_ok, mk);
#pragma unroll
          for (int i = 0; i < 32; ++i) xh[i] = (xh[i] * mk[i] + m[i] - mean) * rstd;
#pragma unroll
          for (int i = 0; i < 32; ++i) m[i] = mk[i];
        }
        db_ln_bwd(dpre, xh, s_lnFw + c0, rstd, keep, sLn + c0, sLn + 64 + c0, xchF, half, row, quarter, lane);
        float v[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = dpre[i] * m[i];
        if (keep) db_store32(p.d_z2 + grow * kDbD + c0, v);
        db_store_split(t_lane + Cfg::kColA + c0, 64, v);
        tc_fence_before();
        mbar_arrive(a_full);
      }
      // ---- 2. chunks: d_z1 = acc_c * act'(z1 + b1) -> TMEM (hi in place, lo in L) and global (rows < param_rows) ----
      for (int c = 0; c < nc; ++c) {
        const int g = it * nc + c, b = g & 1;
        const uint32_t ph = (g >> 1) & 1;
        float z[32], v[32];
        db_load32(p.z1 + ta * p.I + c * 64 + c0, row_ok, z);
        mbar_wait(c_full + b, ph);
        tc_fence_after();
        tmem_ld32(t_lane + Cfg::kColC + b * 64 + c0, v);
        const float* bb = s_b1 + c * 64 + c0;
        switch (p.act) {
          case ACT_GELU: db_act_bwd32<ACT_GELU>(v, z, bb); break;
          case ACT_RELU: db_act_bwd32<ACT_RELU>(v, z, bb); break;
          case ACT_SWISH: db_act_bwd32<ACT_SWISH>(v, z, bb); break;
          case ACT_TANH: db_act_bwd32<ACT_TANH>(v, z, bb); break;
          default: db_act_bwd32<ACT_SIGMOID>(v, z, bb); break;
        }
        if (keep) db_store32(p.d_z1 + grow * p.I + c * 64 + c0, v);
        db_store_split(t_lane + Cfg::kColC + b * 64 + c0, Cfg::kColL - Cfg::kColC, v);
        tc_fence_before();
        mbar_arrive(a_ready + b);
      }
      // ---- 3. attention LayerNorm backward of d_h = acc_h + d_pre_f: d_xres, d_hz -> TMEM (and global, rows < param_rows) ----
      {
        float xh[32], m[32], r[32];
        db_load32(p.hz + ta * kDbD + c0, row_ok, xh);
        db_load32(p.x_res + tr * kDbD + c0, row_ok, r);
        const float mean = row_ok ? p.st_a[2 * ta] : 0.f, rstd = row_ok ? p.st_a[2 * ta + 1] : 0.f;
        db_drop32(p, p.mask_a, p.stream_a, ta, c0, row_ok, m);
#pragma unroll
        for (int i = 0; i < 32; ++i) xh[i] = ((xh[i] + s_bo[c0 + i]) * m[i] + r[i] - mean) * rstd;
        mbar_wait(h_full, it & 1);
        tc_fence_after();
        tmem_ld32(t_lane + Cfg::kColH + c0, r);
#pragma unroll
        for (int i = 0; i < 32; ++i) dpre[i] += r[i];
        db_ln_bwd(dpre, xh, s_lnAw + c0, rstd, keep, sLn + 128 + c0, sLn + 192 + c0, xchA, half, row, quarter, lane);
        if (row_ok) db_store32(p.d_xres + grow * kDbD + c0, dpre);
#pragma unroll
        for (int i = 0; i < 32; ++i) dpre[i] *= m[i];
        if (keep) db_store32(p.d_hz + grow * kDbD + c0, dpre);
        db_store_split(t_lane + Cfg::kColA + c0, 64, dpre);
        tc_fence_before();
        mbar_arrive(hz_full);
      }
      // ---- 4. d_ctx = acc_ctx ----
      {
        float v[32];
        mbar_wait(x_full, it & 1);
        tc_fence_after();
        tmem_ld32(t_lane + Cfg::kColX + c0, v);
        if (row_ok) db_store32(p.d_ctx + grow * kDbD + c0, v);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (my_tiles > 0 && (long long)blockIdx.x * kDbBM < p.param_rows) {
    // (row workers passed griddepcontrol.wait; the barrier above orders this after it for every thread)
    float* dst[4] = {p.g_lnF_w, p.g_lnF_b, p.g_lnA_w, p.g_lnA_b};
    for (int i = threadIdx.x; i < 4 * 64; i += kDbThreads) atomicAdd(dst[i >> 6] + (i & 63), sLn[i]);
  }
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

}  // namespace acsr

using namespace acsr;

extern "C" {

int64_t acsr_dense_bwd_prep_floats(int I) { return (I > 0 && I % 64 == 0) ? (int64_t)(1 + 2 * (I / 64)) * 2 * kDbOpFloats : 0; }

int acsr_dense_bwd_prep(const float* Wo, const float* W1, const float* W2, int d, int I, float* ops, void* stream) {
  if (d != kDbD || I <= 0 || I > kDbMaxI || (I & 63)) {
    set_error("dense_bwd_prep: hidden size %d / inner size %d unsupported (64; multiples of 64 up to %d)", d, I, kDbMaxI);
    return ACSR_ERR_UNSUPPORTED;
  }
  ACSR_REQUIRE(Wo && W1 && W2 && ops, "dense_bwd_prep: NULL pointer");
  launch_pdl(dense_bwd_prep_kernel, dim3(1 + 2 * (I / 64)), dim3(256), 0, (cudaStream_t)stream, Wo, W1, W2, I, ops);
  return check_launch("dense_bwd_prep");
}

int acsr_dense_bwd(const float* d_out, int64_t rows, int64_t act_rows, int64_t res_rows, int64_t param_rows, int d, int I, int act,
                   const float* ops, const float* z2, const float* b2, const float* h, const float* lnF_w, const float* st_f,
                   const float* z1, const float* b1, const float* hz, const float* bo, const float* x_res, const float* lnA_w,
                   const float* st_a, float p_drop, const float* mask_a, const float* mask_f, const void* rng, uint32_t stream_a,
                   uint32_t stream_f, float* d_z2, float* d_z1, float* d_hz, float* d_xres, float* d_ctx, float* g_lnF_w,
                   float* g_lnF_b, float* g_lnA_w, float* g_lnA_b, int passes, void* stream) {
  if (d != kDbD || I <= 0 || I > kDbMaxI || (I & 63)) {
    set_error("dense_bwd: hidden size %d / inner size %d unsupported (64; multiples of 64 up to %d)", d, I, kDbMaxI);
    return ACSR_ERR_UNSUPPORTED;
  }
  ACSR_REQUIRE(d_out && ops && z2 && b2 && h && lnF_w && st_f && z1 && b1 && hz && bo && x_res && lnA_w && st_a, "dense_bwd: NULL input");
  ACSR_REQUIRE(d_z2 && d_z1 && d_hz && d_xres && d_ctx && g_lnF_w && g_lnF_b && g_lnA_w && g_lnA_b, "dense_bwd: NULL output");
  ACSR_REQUIRE(rows >= 0 && act_rows > 0 && res_rows > 0 && param_rows >= 0 && param_rows <= rows && act >= 0 && act <= 4,
               "dense_bwd: bad sizes");
  ACSR_REQUIRE(passes == 1 || passes == 3, "dense_bwd: passes must be 1 or 3");
  ACSR_REQUIRE(p_drop >= 0.f && p_drop < 1.f, "dense_bwd: dropout p=%f", p_drop);
  ACSR_REQUIRE(!(p_drop > 0.f && rng == nullptr && (mask_a == nullptr || mask_f == nullptr)), "dense_bwd: p>0 needs masks or rng");
  if (rows == 0) return ACSR_OK;
  DbParams p = {};
  p.d_out = d_out; p.rows = rows; p.act_rows = act_rows; p.res_rows = res_rows; p.param_rows = param_rows; p.I = I; p.act = act;
  p.passes = passes; p.ops = ops;
  p.z2 = z2; p.b2 = b2; p.h = h; p.lnF_w = lnF_w; p.st_f = st_f; p.z1 = z1; p.b1 = b1; p.hz = hz; p.bo = bo; p.x_res = x_res;
  p.lnA_w = lnA_w; p.st_a = st_a;
  p.p_drop = p_drop; p.mask_a = mask_a; p.mask_f = mask_f; p.rng = (const RngState*)rng; p.stream_a = stream_a; p.stream_f = stream_f;
  p.d_z2 = d_z2; p.d_z1 = d_z1; p.d_hz = d_hz; p.d_xres = d_xres; p.d_ctx = d_ctx;
  p.g_lnF_w = g_lnF_w; p.g_lnF_b = g_lnF_b; p.g_lnA_w = g_lnA_w; p.g_lnA_b = g_lnA_b;
  p.m_tiles = (int)((rows + kDbBM - 1) / kDbBM);
  p.w_static = is_static_memory(ops);
  static_assert(DbCfg::kSmemBytes <= 227 * 1024, "shared memory budget");
  cudaError_t e = cudaFuncSetAttribute(dense_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DbCfg::kSmemBytes);
  if (e != cudaSuccess) { set_error("dense_bwd: smem attr: %s", cudaGetErrorString(e)); return ACSR_ERR_CUDA; }
  const int grid = p.m_tiles < kNumSMs ? p.m_tiles : kNumSMs;
  launch_pdl(dense_bwd_kernel, dim3(grid), dim3(kDbThreads), DbCfg::kSmemBytes, (cudaStream_t)stream, p);
  return check_launch("dense_bwd");
}

}  // extern "C"
