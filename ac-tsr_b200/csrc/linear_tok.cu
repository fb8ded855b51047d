// Encoder GEMMs  Y[T,N] = epilogue(X[T,K] . W^T)  on the 5th-gen tensor cores (tcgen05), 3xTF32.
//
// Replaces the nn.Linear forward / input-gradient GEMMs of layers.py:658-659, 680, 687-689, 791-794, 887
// and fuses what follows them in the reference: the bias add and
// bias + dropout + residual + LayerNorm (layers.py:681-683, 794-796).
//
// Token rows are the UMMA M axis: a 128-token tile of X is split by four loader warps into (hi, lo)
// TF32 operands (fp32 -> hi = rna(x), lo = x - hi) written straight in the canonical no-swizzle K-major
// UMMA layout (each thread owns one token row and walks its 16-byte chunks on a rotated diagonal so
// the shared-memory stores are bank-conflict free); the weight block (<= 128 output features, K <= 256)
// is split once per CTA and stays in shared memory.  One thread issues tcgen05.mma.kind::tf32
// 128 x N x 8 for {lo.hi, hi.lo, hi.hi} (3xTF32: fp32-level accuracy) into a double-buffered TMEM
// accumulator; four epilogue warps read it back with tcgen05.ld 32x32b, so ONE THREAD OWNS ONE TOKEN
// ROW: bias, dropout, residual and the LayerNorm statistics are thread-private (no
// shuffles), and the row is written with 16-byte stores.  CTAs are persistent over token tiles; the
// X operand is double buffered when shared memory allows, so loading/splitting tile t+1 overlaps the
// MMAs and the epilogue of tile t.
#include "acsr_common.cuh"
#include "../../include/acsr.h"

namespace acsr {

constexpr int kLtThreads = 320;      // warp 0: spare, warp 1: MMA issuer, warps 2-5: loaders, warps 6-9: epilogue
constexpr int kLtBM = 128;           // tokens per tile (UMMA M)
constexpr int kLtKB = 64;            // K block (floats) held per A buffer
constexpr int kLtABytes = kLtBM * kLtKB * 4;     // 32 KB per (hi | lo)
constexpr int kLtTmemCols = 256;     // 2 accumulator stages x <= 128 columns

enum { EPI_PLAIN = 0, EPI_BDRL = 2 };

struct LinTokParams {
  const float* X; long long ldx, xkb; long long rows; int K;       // element (r, k) = X[(k / 64) * xkb + r * ldx + k % 64]
  const float* W; long long w_sn, w_sk, wkb; int N;                 // element (n, k) = W[(k / 64) * wkb + n * w_sn + (k % 64) * w_sk]
  const float* bias;
  float* Y; long long ldy; int accumulate;
  int batch; long long bx, bw, bb, by;                               // per-problem strides of a batched launch (blockIdx.z)
  int passes, epi;
  // EPI_BDRL
  const float* res; long long res_rows; const float *ln_w, *ln_b; float eps, p; const float* mask;
  const RngState* rng; uint32_t rng_stream; float* out; float* stats;
  // plan
  int m_tiles, n_blocks, NB, KBn, nbuf;                              // NB: features per CTA (multiple of 16), KBn = ceil(K/64)
  int w_static;                                                      // W / bias are registered parameters (acsr_register_static): staged before griddepcontrol.wait
};

struct LtSmem {
  uint32_t b_hi, b_lo, a0;      // shared-space byte addresses
  int b_bytes;                  // bytes of one (hi | lo) weight operand
};

__device__ __forceinline__ float4 lt_load4(const float* base, long long off, int k0, int kvalid, bool vec_ok) {
  // 4 consecutive k of one row, zero beyond kvalid
  if (vec_ok && k0 + 4 <= kvalid) return __ldg(reinterpret_cast<const float4*>(base + off));
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (k0 + 0 < kvalid) v.x = __ldg(base + off + 0);
  if (k0 + 1 < kvalid) v.y = __ldg(base + off + 1);
  if (k0 + 2 < kvalid) v.z = __ldg(base + off + 2);
  if (k0 + 3 < kvalid) v.w = __ldg(base + off + 3);
  return v;
}

__device__ __forceinline__ void lt_split_store(float* hi_p, float* lo_p, const float4 x) {
  const float4 hi = make_float4(to_tf32(x.x), to_tf32(x.y), to_tf32(x.z), to_tf32(x.w));
  const float4 lo = make_float4(x.x - hi.x, x.y - hi.y, x.z - hi.z, x.w - hi.w);
  *reinterpret_cast<float4*>(hi_p) = hi;
  *reinterpret_cast<float4*>(lo_p) = lo;
}

template <int EPI>
__global__ void __launch_bounds__(kLtThreads, 1) linear_tok_kernel(const LinTokParams p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nb_idx = blockIdx.y, bz = blockIdx.z;
  const int n0 = nb_idx * p.NB;
  const float* Xp = p.X + bz * p.bx;
  const float* Wp = p.W + bz * p.bw;
  const float* biasp = p.bias ? p.bias + bz * p.bb : nullptr;
  float* Yp = p.Y + bz * p.by;
  const int NB = p.NB, KBn = p.KBn, nbuf = p.nbuf;
  const int b_bytes = NB * KBn * kLtKB * 4;
  uint8_t* sBhi = smem;
  uint8_t* sBlo = smem + b_bytes;
  uint8_t* sA = smem + 2 * b_bytes;                        // [nbuf][hi | lo]
  float* sBias = reinterpret_cast<float*>(sA + nbuf * 2 * kLtABytes);     // [128]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sBias + 128);
  uint64_t* a_full = bars;          // [2]
  uint64_t* a_empty = bars + 2;     // [2]
  uint64_t* tm_full = bars + 4;     // [2]
  uint64_t* tm_empty = bars + 6;    // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

  pdl_launch_dependents();
  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(a_full + s, 128); mbar_init(a_empty + s, 1);
      mbar_init(tm_full + s, 1); mbar_init(tm_empty + s, 128);
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc<kLtTmemCols>(tmem_slot);
  // Everything above overlaps the tail of the previous kernel.  When the weights are registered parameters (nothing but the
  // optimizer, the last node of a step, writes them) the warps that stage them do so BEFORE waiting for the previous kernel too:
  // measured on B200 (profiles/r02_linear_tok_phase_ablation.txt) the weight staging is 1.9 us of an 8.5 us launch.
  const bool is_loader = warp >= 2 && warp < 6;
  const bool stage_early = p.w_static && !is_loader;
  if (!stage_early) pdl_wait();
  const int lr = threadIdx.x - 64;            // loader: token row of the tile owned by this thread (0..127)
  const bool x_vec_ok = (p.ldx & 3) == 0 && (p.xkb & 3) == 0 && ((reinterpret_cast<uintptr_t>(Xp) & 15) == 0);
  // the loader warps put the loads of their first tile in flight while the other warps stage the weights
  float4 xpre[kLtKB / 4];
  if (is_loader && (int)blockIdx.x < p.m_tiles) {
    const long long grow = (long long)blockIdx.x * kLtBM + lr;
    const int kvalid = min(kLtKB, p.K);
    const float* xrow = Xp + grow * p.ldx;
#pragma unroll
    for (int q = 0; q < kLtKB / 4; ++q) {
      const int kc = (q + lr) & (kLtKB / 4 - 1);
      xpre[q] = grow < p.rows ? lt_load4(xrow, kc * 4, kc * 4, kvalid, x_vec_ok) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }

  // stationary weight block: rows n0 .. n0+NB of W (zero beyond N / K), split into hi/lo, canonical K-major layout
  if (!is_loader) {
    constexpr int kStagers = kLtThreads - 128;
    const int sid = threadIdx.x < 64 ? threadIdx.x : threadIdx.x - 128;
    const int KC = KBn * (kLtKB / 4);                      // 16-byte chunks along K
    float* Bhi = reinterpret_cast<float*>(sBhi);
    float* Blo = reinterpret_cast<float*>(sBlo);
    const bool vec_ok = p.w_sk == 1 && (p.w_sn & 3) == 0 && (p.wkb & 3) == 0 && ((reinterpret_cast<uintptr_t>(Wp) & 15) == 0);
    constexpr int kU = 4;                                  // loads in flight per thread
    for (int item0 = sid; item0 < NB * KC; item0 += kStagers * kU) {
      float4 xs[kU];
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        const int item = item0 + u * kStagers;
        xs[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (item >= NB * KC) continue;
        const int n = item % NB, kc = item / NB;
        const int kb = kc / (kLtKB / 4), kcl = kc % (kLtKB / 4);
        const int k0 = kb * kLtKB + kcl * 4;
        if (n0 + n < p.N && k0 < p.K) {
          const float* w = Wp + kb * p.wkb + (long long)(n0 + n) * p.w_sn + (long long)(kcl * 4) * p.w_sk;
          if (vec_ok && k0 + 4 <= p.K) xs[u] = __ldg(reinterpret_cast<const float4*>(w));
          else {
            xs[u].x = __ldg(w);
            if (k0 + 1 < p.K) xs[u].y = __ldg(w + p.w_sk);
            if (k0 + 2 < p.K) xs[u].z = __ldg(w + 2 * p.w_sk);
            if (k0 + 3 < p.K) xs[u].w = __ldg(w + 3 * p.w_sk);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        const int item = item0 + u * kStagers;
        if (item >= NB * KC) continue;
        const int n = item % NB, kc = item / NB;
        const int off = kc * (NB * 4) + n * 4;             // floats: chunk plane of NB rows x 16 B
        lt_split_store(Bhi + off, Blo + off, xs[u]);
      }
    }
    for (int i = sid; i < 128; i += kStagers) sBias[i] = (biasp != nullptr && n0 + i < p.N) ? biasp[n0 + i] : 0.f;
  }
  if (stage_early) pdl_wait();
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 1) {
    // ------------------------------ MMA issuer ------------------------------
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_tf32(kLtBM, NB);
      const uint32_t b_hi = smem_u32(sBhi), b_lo = smem_u32(sBlo);
      constexpr uint32_t kALbo = kLtBM * 16, kSbo = 128;
      const uint32_t kBLbo = NB * 16;
      const int npass = p.passes == 3 ? 3 : 1;
      int it = 0;
      for (int tile = blockIdx.x; tile < p.m_tiles; tile += gridDim.x, ++it) {
        const int ts = it & 1;
        mbar_wait(tm_empty + ts, ((it >> 1) & 1) ^ 1);
        const uint32_t d_tmem = tmem_base + ts * NB;
        uint32_t acc = 0;
        for (int kb = 0; kb < KBn; ++kb) {
          const int it2 = it * KBn + kb;
          const int buf = it2 % nbuf;
          mbar_wait(a_full + buf, (it2 / nbuf) & 1);
          tc_fence_after();
          const uint32_t a_hi = smem_u32(sA + buf * 2 * kLtABytes), a_lo = a_hi + kLtABytes;
          for (int ps = 0; ps < npass; ++ps) {
            // small cross terms first, the dominant hi.hi product last
            const uint32_t a_base = (npass == 3 && ps == 0) ? a_lo : a_hi;
            const uint32_t b_base = ((npass == 3 && ps == 1) ? b_lo : b_hi) + kb * (kLtKB / 4) * kBLbo;
#pragma unroll
            for (int ks = 0; ks < kLtKB / 8; ++ks) {
              const uint64_t ad = umma_desc_kmajor(a_base + ks * 2 * kALbo, kALbo, kSbo);
              const uint64_t bd = umma_desc_kmajor(b_base + ks * 2 * kBLbo, kBLbo, kSbo);
              umma_tf32(d_tmem, ad, bd, idesc, acc);
              acc = 1;
            }
          }
          umma_commit(a_empty + buf);     // the X buffer may be overwritten once these MMAs retire
        }
        umma_commit(tm_full + ts);        // accumulator stage ready for the epilogue
      }
    }
  } else if (warp >= 2 && warp < 6) {
    // ------------------------------ loader / hi-lo splitter ------------------------------
    const int r = lr;
    const bool vec_ok = x_vec_ok;
    int it = 0;
    for (int tile = blockIdx.x; tile < p.m_tiles; tile += gridDim.x, ++it) {
      const long long grow = (long long)tile * kLtBM + r;
      const bool row_ok = grow < p.rows;
      for (int kb = 0; kb < KBn; ++kb) {
        const int it2 = it * KBn + kb;
        const int buf = it2 % nbuf;
        const int kvalid = min(kLtKB, p.K - kb * kLtKB);
        const float* xrow = Xp + kb * p.xkb + grow * p.ldx;
        // issue the 16 loads of this row first (independent), then wait for the buffer and split
        float4 x[kLtKB / 4];
        if (it2 == 0) {
#pragma unroll
          for (int q = 0; q < kLtKB / 4; ++q) x[q] = xpre[q];
        } else {
#pragma unroll
          for (int q = 0; q < kLtKB / 4; ++q) {
            const int kc = (q + r) & (kLtKB / 4 - 1);          // rotated diagonal
            x[q] = row_ok ? lt_load4(xrow, kc * 4, kc * 4, kvalid, vec_ok) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
        mbar_wait(a_empty + buf, ((it2 / nbuf) & 1) ^ 1);
        float* Ahi = reinterpret_cast<float*>(sA + buf * 2 * kLtABytes);
        float* Alo = Ahi + kLtABytes / 4;
#pragma unroll
        for (int q = 0; q < kLtKB / 4; ++q) {
          const int kc = (q + r) & (kLtKB / 4 - 1);
          const int off = kc * (kLtBM * 4) + r * 4;
          lt_split_store(Ahi + off, Alo + off, x[q]);
        }
        fence_proxy_async();               // generic-proxy stores -> visible to the tensor-core (async) proxy
        mbar_arrive(a_full + buf);
      }
    }
  } else if (warp >= 6) {
    // ------------------------------ epilogue: one thread = one token row ------------------------------
    const int quarter = warp & 3;                 // TMEM lane quarter this warp may access
    const int row = quarter * 32 + lane;
    const uint32_t t_lane = tmem_base + ((uint32_t)(quarter * 32) << 16);
    const int ncols = min(NB, p.N - n0);          // valid features of this block
    int it = 0;
    for (int tile = blockIdx.x; tile < p.m_tiles; tile += gridDim.x, ++it) {
      const int ts = it & 1;
      const long long grow = (long long)tile * kLtBM + row;
      const bool row_ok = grow < p.rows;
      mbar_wait(tm_full + ts, (it >> 1) & 1);
      tc_fence_after();
      if (EPI == EPI_BDRL) {
        // N == 64: hz = acc ; out = LN(dropout(acc + bias) * m + res) ; stats = (mean, rstd)
        float x[64];
        tmem_ld32(t_lane + ts * NB, x);
        tmem_ld32(t_lane + ts * NB + 32, x + 32);
        tc_fence_before();
        mbar_arrive(tm_empty + ts);               // accumulator stage is free as soon as it sits in registers
        if (row_ok) {
          float* hz = Yp + grow * p.ldy;
#pragma unroll
          for (int i = 0; i < 64; i += 4) *reinterpret_cast<float4*>(hz + i) = make_float4(x[i], x[i + 1], x[i + 2], x[i + 3]);
          const float* rr = p.res + (grow % p.res_rows) * 64;
          const float inv_keep = p.p > 0.f ? 1.0f / (1.0f - p.p) : 1.0f;
          const bool philox = p.p > 0.f && p.mask == nullptr && p.rng != nullptr;
          unsigned long long seed = 0, step = 0;
          if (philox) { seed = p.rng->seed; step = p.rng->step; }
          float s = 0.f;
#pragma unroll
          for (int q = 0; q < 16; ++q) {
            float m[4] = {1.f, 1.f, 1.f, 1.f};
            if (p.mask != nullptr) {
              const float4 mm = __ldg(reinterpret_cast<const float4*>(p.mask + grow * 64 + q * 4));
              m[0] = mm.x; m[1] = mm.y; m[2] = mm.z; m[3] = mm.w;
            } else if (philox) {           // same counters as bdrl_{fwd,bwd}_kernel (rowwise.cu): element e -> call e>>2, word e&3
              const uint4 w = philox4x32(seed, step, p.rng_stream, (unsigned long long)grow * 16 + q);
              m[0] = drop_mult(w.x, p.p, inv_keep); m[1] = drop_mult(w.y, p.p, inv_keep);
              m[2] = drop_mult(w.z, p.p, inv_keep); m[3] = drop_mult(w.w, p.p, inv_keep);
            }
            const float4 r4 = __ldg(reinterpret_cast<const float4*>(rr + q * 4));
            const float rv[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
            for (int v = 0; v < 4; ++v) {
              const int c = q * 4 + v;
              x[c] = (x[c] + sBias[c]) * m[v] + rv[v];
              s += x[c];
            }
          }
          const float mean = s * (1.0f / 64);
          float var = 0.f;
#pragma unroll
          for (int c = 0; c < 64; ++c) { const float t = x[c] - mean; var = fmaf(t, t, var); }
          const float rstd = 1.0f / sqrtf(var * (1.0f / 64) + p.eps);
          float* o = p.out + grow * 64;
#pragma unroll
          for (int c = 0; c < 64; c += 4) {
            const float4 w4 = __ldg(reinterpret_cast<const float4*>(p.ln_w + c));
            const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.ln_b + c));
            *reinterpret_cast<float4*>(o + c) = make_float4((x[c] - mean) * rstd * w4.x + b4.x, (x[c + 1] - mean) * rstd * w4.y + b4.y,
                                                            (x[c + 2] - mean) * rstd * w4.z + b4.z, (x[c + 3] - mean) * rstd * w4.w + b4.w);
          }
          p.stats[2 * grow] = mean;
          p.stats[2 * grow + 1] = rstd;
        }
      } else {
#pragma unroll 1
        for (int cc = 0; cc < NB / 32 + ((NB & 31) ? 1 : 0); ++cc) {
          if (cc * 32 >= ncols) break;
          float v[32];
          tmem_ld32(t_lane + ts * NB + cc * 32, v);
          const int nvalid = min(32, ncols - cc * 32);
          if (row_ok) {
            float* y = Yp + grow * p.ldy + n0 + cc * 32;
            const bool vec = nvalid == 32 && ((reinterpret_cast<uintptr_t>(y) & 15) == 0);
            if (vec) {
              float4 old[8];
              if (p.accumulate) {
#pragma unroll
                for (int i = 0; i < 8; ++i) old[i] = *reinterpret_cast<const float4*>(y + 4 * i);
              }
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                float4 o = make_float4(v[4 * i] + sBias[cc * 32 + 4 * i], v[4 * i + 1] + sBias[cc * 32 + 4 * i + 1],
                                       v[4 * i + 2] + sBias[cc * 32 + 4 * i + 2], v[4 * i + 3] + sBias[cc * 32 + 4 * i + 3]);
                if (p.accumulate) { o.x += old[i].x; o.y += old[i].y; o.z += old[i].z; o.w += old[i].w; }
                *reinterpret_cast<float4*>(y + 4 * i) = o;
              }
            } else {
              float old[32];
              if (p.accumulate) {
#pragma unroll
                for (int i = 0; i < 32; ++i) old[i] = i < nvalid ? y[i] : 0.f;
              }
#pragma unroll
              for (int i = 0; i < 32; ++i)
                if (i < nvalid) y[i] = v[i] + sBias[cc * 32 + i] + (p.accumulate ? old[i] : 0.f);
            }
          }
        }
        tc_fence_before();
        mbar_arrive(tm_empty + ts);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<kLtTmemCols>(tmem_base);
  }
}

static int lt_plan(LinTokParams& p, size_t& smem, const char* who) {
  p.KBn = (p.K + kLtKB - 1) / kLtKB;
  if (p.KBn < 1 || p.KBn > 4) { set_error("%s: K=%d unsupported (1..256)", who, p.K); return ACSR_ERR_UNSUPPORTED; }
  // features per CTA: as wide as shared memory allows (weights hi+lo + at least one X buffer)
  const int n16 = (p.N + 15) & ~15;
  int NB = n16 < 128 ? n16 : 128;
  const size_t fixed = 128 * 4 + 9 * 8 + 64;
  while (NB > 16 && (size_t)2 * NB * p.KBn * kLtKB * 4 + 2 * kLtABytes + fixed > 227 * 1024) NB -= 16;
  p.NB = NB;
  p.n_blocks = (p.N + NB - 1) / NB;
  const size_t bw = (size_t)2 * NB * p.KBn * kLtKB * 4;
  p.nbuf = (bw + 4 * kLtABytes + fixed <= 227 * 1024) ? 2 : 1;
  smem = bw + (size_t)p.nbuf * 2 * kLtABytes + fixed;
  p.m_tiles = (int)((p.rows + kLtBM - 1) / kLtBM);
  return ACSR_OK;
}

template <int EPI>
static int lt_launch(LinTokParams& p, cudaStream_t st, const char* who) {
  size_t smem = 0;
  int rc = lt_plan(p, smem, who);
  if (rc) return rc;
  cudaError_t e = cudaFuncSetAttribute(linear_tok_kernel<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) { set_error("%s: smem attr %zu: %s", who, smem, cudaGetErrorString(e)); return ACSR_ERR_CUDA; }
  int gx = kNumSMs / (p.n_blocks * p.batch);
  if (gx < 1) gx = 1;
  if (gx > p.m_tiles) gx = p.m_tiles;
  launch_pdl(linear_tok_kernel<EPI>, dim3(gx, p.n_blocks, p.batch), dim3(kLtThreads), smem, st, p);
  return check_launch(who);
}

}  // namespace acsr

using namespace acsr;

extern "C" {

int acsr_linear_tok(const float* X, int64_t ldx, int64_t x_kblock_stride, int64_t rows, int K, const float* W, int64_t w_stride_n,
                    int64_t w_stride_k, int64_t w_kblock_stride, int N, const float* bias, int accumulate, float* Y, int64_t ldy,
                    int batch, int64_t stride_x, int64_t stride_w, int64_t stride_bias, int64_t stride_y, int passes, void* stream) {
  ACSR_REQUIRE(X && W && Y, "linear_tok: NULL pointer");
  ACSR_REQUIRE(rows >= 0 && N > 0 && K > 0 && batch > 0 && batch < 65536 && ldy >= N, "linear_tok: bad sizes");
  ACSR_REQUIRE(passes == 1 || passes == 3, "linear_tok: passes must be 1 or 3");
  if (rows == 0) return ACSR_OK;
  LinTokParams p = {};
  p.X = X; p.ldx = ldx; p.xkb = x_kblock_stride; p.rows = rows; p.K = K;
  p.W = W; p.w_sn = w_stride_n; p.w_sk = w_stride_k; p.wkb = w_kblock_stride; p.N = N;
  p.bias = bias; p.accumulate = accumulate; p.Y = Y; p.ldy = ldy;
  p.batch = batch; p.bx = stride_x; p.bw = stride_w; p.bb = stride_bias; p.by = stride_y;
  p.passes = passes; p.epi = EPI_PLAIN;
  p.w_static = is_static_memory(p.W) && (p.bias == nullptr || is_static_memory(p.bias));
  return lt_launch<EPI_PLAIN>(p, (cudaStream_t)stream, "linear_tok");
}

int acsr_linear_tok_bdrl(const float* X, int64_t ldx, int64_t rows, int K, const float* W, const float* bias, const float* res,
                         int64_t res_rows, const float* ln_w, const float* ln_b, float eps, float p_drop, const float* mask,
                         const void* rng, uint32_t rng_stream, float* HZ, float* out, float* stats, int passes, void* stream) {
  ACSR_REQUIRE(X && W && res && ln_w && ln_b && HZ && out && stats, "linear_tok_bdrl: NULL pointer");
  ACSR_REQUIRE(rows >= 0 && K > 0 && res_rows > 0, "linear_tok_bdrl: bad sizes");
  ACSR_REQUIRE(p_drop >= 0.f && p_drop < 1.f, "linear_tok_bdrl: dropout p=%f", p_drop);
  ACSR_REQUIRE(!(p_drop > 0.f && mask == nullptr && rng == nullptr), "linear_tok_bdrl: p>0 needs mask or rng");
  ACSR_REQUIRE(passes == 1 || passes == 3, "linear_tok_bdrl: passes must be 1 or 3");
  if (rows == 0) return ACSR_OK;
  LinTokParams p = {};
  p.X = X; p.ldx = ldx; p.xkb = kLtKB; p.rows = rows; p.K = K;
  p.W = W; p.w_sn = K; p.w_sk = 1; p.wkb = kLtKB; p.N = 64;
  p.bias = bias; p.Y = HZ; p.ldy = 64;
  p.batch = 1; p.passes = passes; p.epi = EPI_BDRL;
  p.w_static = is_static_memory(p.W) && (p.bias == nullptr || is_static_memory(p.bias));
  p.res = res; p.res_rows = res_rows; p.ln_w = ln_w; p.ln_b = ln_b; p.eps = eps; p.p = p_drop; p.mask = mask;
  p.rng = (const RngState*)rng; p.rng_stream = rng_stream; p.out = out; p.stats = stats;
  return lt_launch<EPI_BDRL>(p, (cudaStream_t)stream, "linear_tok_bdrl");
}

}  // extern "C"
