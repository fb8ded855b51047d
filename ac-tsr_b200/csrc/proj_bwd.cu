// Input gradient of a layer's Q / K / V projections, attack transforms and gate (the backward of layers.py:658-659, 687-689,
// 887) as ONE tcgen05 launch, hidden size 64:
//   d_mq += d_aq.Waq (+ d_gl.Wg) ; d_mk += d_ak.Wak ; d_x += [d_mq d_mk d_mv] . [Wq; Wk; Wv]
// As three acsr_linear_tok launches this chain sits on the critical path of every layer's backward, right after the attention
// backward; each launch pays the fixed cost of a tcgen05 launch (barrier init, TMEM allocation, weight staging, pipeline
// handshakes: about 6 us, profiles/r02_linear_tok_phase_ablation.txt) and the summed d_mq / d_mk make two round trips through
// L2.  Their epilogues are plain adds, so nothing serial is gained by fusing them.  Here a 128-token tile goes through both
// stages on one SM:
//   stage 1: acc_q = d_aq.Waq (+ d_gl.Wg), acc_k = d_ak.Wak (3xTF32, in TMEM); the epilogue adds d_mq / d_mk in exact fp32 (the
//            add of linear_tok's accumulate epilogue), writes rows < rows_keep back into d_qkv (the Q / K weight gradients read
//            them) and leaves the sums, split into hi / lo, in TMEM with tcgen05.st;
//   stage 2: d_x += [d_mq | d_mk | d_mv] . [Wq; Wk; Wv], the A operand read from TMEM (TS form, as in logits_bwd.cu / dense_bwd.cu).
// The A operands of stage 1 are streamed through TMEM too: the six weight blocks (read transposed, split into hi / lo, canonical
// K-major UMMA layout) fill 192 KB of shared memory and leave no room for an A tile there.
//
// TMEM columns (128 lanes x 512, one CTA per SM):
//   [0,128)   A_q: d_aq hi / lo, then the summed d_mq     [128,256) A_k: d_ak, then the summed d_mk     [256,384) A_g: d_gl, then d_mv
//   [384,448) acc_q, then acc_x1 = d_mq.Wq + d_mv.Wv (k < 32)    [448,512) acc_k, then acc_x2 = d_mk.Wk + d_mv.Wv (k >= 32)
// Roles (320 threads, persistent over tiles): warps 0 and 1 each have one thread issuing MMAs (warp 0: acc_q, acc_x1; warp 1:
// acc_k, acc_x2) -- two issuing threads keep the tensor pipe busier than one (43 against 78 cycles per TS-form 128x64x8 MMA,
// profiles/r02_ce_backward.txt); warps 2-9 are the row workers, two per TMEM lane quarter: one thread owns 32 columns of one
// token row through loads, hi / lo splits, both epilogues and the read-modify-write of d_x.
#include "acsr_common.cuh"
#include "../../include/acsr.h"

namespace acsr {

constexpr int kPbThreads = 320;
constexpr int kPbD = 64;
constexpr int kPbBM = 128;                          // tokens per tile (UMMA M)
constexpr int kPbOpFloats = 64 * 64;                // one 64 x 64 operand (hi or lo)
constexpr int kPbBlkBytes = 2 * kPbOpFloats * 4;    // hi + lo: 32 KB
constexpr int kPbNumBlk = 6;                        // Waq, Wak, Wg, Wq, Wk, Wv
constexpr int kPbOffBar = kPbNumBlk * kPbBlkBytes;
constexpr int kPbNumBars = 8;
constexpr int kPbSmemBytes = kPbOffBar + kPbNumBars * 8 + 16;
constexpr int kColAq = 0, kColAk = 128, kColAg = 256, kColAccQ = 384, kColAccK = 448;
enum { PB_WAQ = 0, PB_WAK = 1, PB_WG = 2, PB_WQ = 3, PB_WK = 4, PB_WV = 5 };

struct PbParams {
  float* d_qkv; const float* d_aqk; long long plane;    // [3, plane, 64] (d_mq, d_mk, d_mv) and [2, plane, 64] (d_aq, d_ak)
  const float* d_gl; int L;                              // [plane, L], NULL without the gate
  const float *Wqkv, *Waqk, *Wg;                         // [3,64,64], [2,64,64], [L,64] (row-major [out, in])
  float* d_x; long long rows, rows_keep;
  int passes, m_tiles, w_static;
};

// 32 columns of one row -> TMEM (hi at column c, lo at c + 64)
__device__ __forceinline__ void pb_store_split(uint32_t taddr, float* v) {
  float lo[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) { const float hi = to_tf32(v[i]); lo[i] = v[i] - hi; v[i] = hi; }
  tmem_st32(taddr, v);
  tmem_st32(taddr + 64, lo);
}

__device__ __forceinline__ void pb_load32(const float* p, bool ok, float* v) {
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const float4 x = ok ? __ldg(reinterpret_cast<const float4*>(p) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
    v[4 * q] = x.x; v[4 * q + 1] = x.y; v[4 * q + 2] = x.z; v[4 * q + 3] = x.w;
  }
}

__global__ void __launch_bounds__(kPbThreads, 1) proj_bwd_kernel(const PbParams p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool gate = p.d_gl != nullptr;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kPbOffBar);
  uint64_t* a1_full = bars;        // stage-1 A operands sit in TMEM (and the previous tile's acc_x has been read)
  uint64_t* s1q_full = bars + 1;   // acc_q ready, A_q / A_g free
  uint64_t* s1k_full = bars + 2;   // acc_k ready, A_k free
  uint64_t* k_ready = bars + 3;    // summed d_mk in A_k, acc_k columns free
  uint64_t* q_ready = bars + 4;    // summed d_mq in A_q and d_mv in A_g, acc_q columns free
  uint64_t* s2a_full = bars + 5;   // acc_x1 ready
  uint64_t* s2b_full = bars + 6;   // acc_x2 ready
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kPbNumBars);

  pdl_launch_dependents();
  if (threadIdx.x == 0) {
    mbar_init(a1_full, 256); mbar_init(k_ready, 256); mbar_init(q_ready, 256);
    mbar_init(s1q_full, 1); mbar_init(s1k_full, 1); mbar_init(s2a_full, 1); mbar_init(s2b_full, 1);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc<512>(tmem_slot);
  // Weights: registered parameters are staged before waiting for the previous kernel (as linear_tok's w_static).  Block b holds
  // B(n, k) = W_b[k][n] (the input gradient reads the weight transposed); rows k >= L of the gate block are zero.
  if (!p.w_static) pdl_wait();
  {
    constexpr int kItems = kPbNumBlk * 64 * 16;     // (block, 16-byte chunk along k, n)
    // all loads of the 192 KB in flight at once: one L2 round trip (the launch of layer 0 runs one tile per CTA)
    constexpr int kU = (kItems + kPbThreads - 1) / kPbThreads;
    for (int item0 = threadIdx.x; item0 < kItems; item0 += kPbThreads * kU) {
      float4 xs[kU];
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        const int item = item0 + u * kPbThreads;
        xs[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (item >= kItems) continue;
        const int blk = item >> 10, kc = (item >> 6) & 15, n = item & 63;
        const float* src = blk < PB_WG ? p.Waqk + blk * kPbOpFloats : (blk == PB_WG ? p.Wg : p.Wqkv + (blk - PB_WQ) * kPbOpFloats);
        const int kmax = blk == PB_WG ? (gate ? p.L : 0) : kPbD;
        const int k0 = kc * 4;
        if (k0 + 0 < kmax) xs[u].x = __ldg(src + (k0 + 0) * kPbD + n);     // consecutive threads: consecutive n (coalesced)
        if (k0 + 1 < kmax) xs[u].y = __ldg(src + (k0 + 1) * kPbD + n);
        if (k0 + 2 < kmax) xs[u].z = __ldg(src + (k0 + 2) * kPbD + n);
        if (k0 + 3 < kmax) xs[u].w = __ldg(src + (k0 + 3) * kPbD + n);
      }
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        const int item = item0 + u * kPbThreads;
        if (item >= kItems) continue;
        const int blk = item >> 10, kc = (item >> 6) & 15, n = item & 63;
        float* hi = reinterpret_cast<float*>(smem + blk * kPbBlkBytes) + kc * 256 + n * 4;
        const float4 x = xs[u];
        const float4 h4 = make_float4(to_tf32(x.x), to_tf32(x.y), to_tf32(x.z), to_tf32(x.w));
        *reinterpret_cast<float4*>(hi) = h4;
        *reinterpret_cast<float4*>(hi + kPbOpFloats) = make_float4(x.x - h4.x, x.y - h4.y, x.z - h4.z, x.w - h4.w);
      }
    }
  }
  if (p.w_static) pdl_wait();
  fence_proxy_async();               // generic-proxy stores -> visible to the tensor-core (async) proxy
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 2) {
    // ------------------------------ MMA issuers ------------------------------
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_tf32(kPbBM, 64);
      constexpr uint32_t kLbo = 64 * 16, kSbo = 128;
      const int npass = p.passes == 3 ? 3 : 1;
      const uint32_t w0 = smem_u32(smem);
      // d (+)= A[tmem a_hi (hi), a_hi + 64 (lo)] . W_blk^T over k in [8 ks0, 8 ks1); 3xTF32: small cross terms first, hi.hi last
      auto mma = [&](uint32_t d_tmem, uint32_t a_hi, int ks0, int ks1, int blk, uint32_t acc) {
        for (int ps = 0; ps < npass; ++ps) {
          const uint32_t a_base = (npass == 3 && ps == 0) ? a_hi + 64 : a_hi;
          const uint32_t b_base = w0 + blk * kPbBlkBytes + ((npass == 3 && ps == 1) ? kPbOpFloats * 4 : 0);
          for (int ks = ks0; ks < ks1; ++ks) {
            umma_tf32_ts(d_tmem, a_base + ks * 8, umma_desc_kmajor(b_base + ks * 2 * kLbo, kLbo, kSbo), idesc, acc);
            acc = 1;
          }
        }
      };
      const int kg = (p.L + 7) / 8;
      int it = 0;
      for (int tile = blockIdx.x; tile < p.m_tiles; tile += gridDim.x, ++it) {
        const uint32_t ph = it & 1;
        mbar_wait(a1_full, ph);
        tc_fence_after();
        // d_mv.Wv is split along K between the two accumulators: after q_ready each issuer has 36 MMAs (3xTF32) left, not 24 / 48
        if (warp == 0) {
          mma(tmem_base + kColAccQ, tmem_base + kColAq, 0, 8, PB_WAQ, 0);
          if (gate) mma(tmem_base + kColAccQ, tmem_base + kColAg, 0, kg, PB_WG, 1);
          umma_commit(s1q_full);
          mbar_wait(q_ready, ph);
          tc_fence_after();
          mma(tmem_base + kColAccQ, tmem_base + kColAq, 0, 8, PB_WQ, 0);
          mma(tmem_base + kColAccQ, tmem_base + kColAg, 0, 4, PB_WV, 1);
          umma_commit(s2a_full);
        } else {
          mma(tmem_base + kColAccK, tmem_base + kColAk, 0, 8, PB_WAK, 0);
          umma_commit(s1k_full);
          mbar_wait(k_ready, ph);
          tc_fence_after();
          mma(tmem_base + kColAccK, tmem_base + kColAk, 0, 8, PB_WK, 0);
          mbar_wait(q_ready, ph);
          tc_fence_after();
          mma(tmem_base + kColAccK, tmem_base + kColAg, 4, 8, PB_WV, 1);
          umma_commit(s2b_full);
        }
      }
    }
  } else {
    // ------------------------------ row workers: one thread = 32 columns of one token row ------------------------------
    const int quarter = warp & 3;                 // TMEM lane quarter this warp may access
    const int c0 = ((warp - 2) >> 2) * 32;        // column half of the row
    const int row = quarter * 32 + lane;
    const uint32_t t_lane = tmem_base + ((uint32_t)(quarter * 32) << 16);
    float* d_mq = p.d_qkv;
    float* d_mk = p.d_qkv + p.plane * kPbD;
    const float* d_mv = p.d_qkv + 2 * p.plane * kPbD;
    const float* d_aq = p.d_aqk;
    const float* d_ak = p.d_aqk + p.plane * kPbD;
    int it = 0;
    for (int tile = blockIdx.x; tile < p.m_tiles; tile += gridDim.x, ++it) {
      const uint32_t ph = it & 1;
      const long long grow = (long long)tile * kPbBM + row;
      const bool row_ok = grow < p.rows, keep = grow < p.rows_keep;
      const long long off = grow * kPbD + c0;
      {
        // ---- stage-1 A operands -> TMEM (the previous tile's stage 2 has retired: its A columns are free) ----
        float aq[32], ak[32];
        pb_load32(d_aq + off, row_ok, aq);
        pb_load32(d_ak + off, row_ok, ak);
        pb_store_split(t_lane + kColAq + c0, aq);
        if (gate) {
          float* g = aq;
#pragma unroll
          for (int i = 0; i < 32; ++i) g[i] = (row_ok && c0 + i < p.L) ? __ldg(p.d_gl + grow * p.L + c0 + i) : 0.f;
          pb_store_split(t_lane + kColAk + c0, ak);
          pb_store_split(t_lane + kColAg + c0, g);
        } else {
          pb_store_split(t_lane + kColAk + c0, ak);
        }
        tc_fence_before();
        mbar_arrive(a1_full);
      }
      // the epilogue operands are loaded while the MMAs they wait for run
      float mq[32], mk[32];
      pb_load32(d_mq + off, row_ok, mq);
      pb_load32(d_mk + off, row_ok, mk);
      {
        // ---- acc_k + d_mk -> d_mk (rows < rows_keep) and, split, the stage-2 A operand ----
        float v[32];
        mbar_wait(s1k_full, ph);
        tc_fence_after();
        tmem_ld32(t_lane + kColAccK + c0, v);
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] += mk[i];
        if (keep) {
#pragma unroll
          for (int i = 0; i < 32; i += 4) *reinterpret_cast<float4*>(d_mk + off + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
        }
        pb_store_split(t_lane + kColAk + c0, v);
        tc_fence_before();
        mbar_arrive(k_ready);
      }
      {
        float mv[32];
        pb_load32(d_mv + off, row_ok, mv);
        // ---- acc_q + d_mq likewise; d_mv into the gate's A columns ----
        float v[32];
        mbar_wait(s1q_full, ph);
        tc_fence_after();
        tmem_ld32(t_lane + kColAccQ + c0, v);
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] += mq[i];
        if (keep) {
#pragma unroll
          for (int i = 0; i < 32; i += 4) *reinterpret_cast<float4*>(d_mq + off + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
        }
        pb_store_split(t_lane + kColAq + c0, v);
        pb_store_split(t_lane + kColAg + c0, mv);
        tc_fence_before();
        mbar_arrive(q_ready);
      }
      {
        // ---- d_x += acc_x1 + acc_x2 ----
        float x[32], x1[32], x2[32];
        pb_load32(p.d_x + off, row_ok, x);
        mbar_wait(s2a_full, ph);
        mbar_wait(s2b_full, ph);
        tc_fence_after();
        tmem_ld32(t_lane + kColAccQ + c0, x1);
        tmem_ld32(t_lane + kColAccK + c0, x2);
        if (row_ok) {
          float* y = p.d_x + off;
#pragma unroll
          for (int i = 0; i < 32; i += 4)
            *reinterpret_cast<float4*>(y + i) = make_float4(x[i] + (x1[i] + x2[i]), x[i + 1] + (x1[i + 1] + x2[i + 1]),
                                                            x[i + 2] + (x1[i + 2] + x2[i + 2]), x[i + 3] + (x1[i + 3] + x2[i + 3]));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

}  // namespace acsr

using namespace acsr;

extern "C" {

int acsr_proj_input_grad(float* d_qkv, const float* d_aqk, int64_t plane_rows, const float* d_gl, int L, const float* Wqkv,
                         const float* Waqk, const float* Wg, int d, int64_t rows, int64_t rows_keep, float* d_x, int passes,
                         void* stream) {
  if (d != kPbD) { set_error("proj_input_grad: hidden size %d unsupported (64)", d); return ACSR_ERR_UNSUPPORTED; }
  ACSR_REQUIRE(d_qkv && d_aqk && Wqkv && Waqk && d_x, "proj_input_grad: NULL pointer");
  ACSR_REQUIRE((d_gl == nullptr) == (Wg == nullptr), "proj_input_grad: d_gl and Wg go together");
  ACSR_REQUIRE(d_gl == nullptr || (L >= 1 && L <= kPbD), "proj_input_grad: gate width L=%d out of range (1..64)", L);
  ACSR_REQUIRE(rows >= 0 && rows <= plane_rows && rows_keep >= 0 && rows_keep <= rows, "proj_input_grad: bad row counts");
  ACSR_REQUIRE(passes == 1 || passes == 3, "proj_input_grad: passes must be 1 or 3");
  ACSR_REQUIRE(((reinterpret_cast<uintptr_t>(d_qkv) | reinterpret_cast<uintptr_t>(d_aqk) | reinterpret_cast<uintptr_t>(d_x)) & 15) == 0,
               "proj_input_grad: d_qkv / d_aqk / d_x must be 16-byte aligned");
  if (rows == 0) return ACSR_OK;
  PbParams p = {};
  p.d_qkv = d_qkv; p.d_aqk = d_aqk; p.plane = plane_rows; p.d_gl = d_gl; p.L = d_gl ? L : 0;
  p.Wqkv = Wqkv; p.Waqk = Waqk; p.Wg = Wg;
  p.d_x = d_x; p.rows = rows; p.rows_keep = rows_keep; p.passes = passes;
  p.m_tiles = (int)((rows + kPbBM - 1) / kPbBM);
  p.w_static = is_static_memory(Wqkv) && is_static_memory(Waqk) && (Wg == nullptr || is_static_memory(Wg));
  static_assert(kPbSmemBytes <= 227 * 1024, "shared memory budget");
  cudaError_t e = cudaFuncSetAttribute(proj_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPbSmemBytes);
  if (e != cudaSuccess) { set_error("proj_input_grad: smem attr: %s", cudaGetErrorString(e)); return ACSR_ERR_CUDA; }
  const int grid = p.m_tiles < kNumSMs ? p.m_tiles : kNumSMs;
  launch_pdl(proj_bwd_kernel, dim3(grid), dim3(kPbThreads), kPbSmemBytes, (cudaStream_t)stream, p);
  return check_launch("proj_input_grad");
}

}  // extern "C"
