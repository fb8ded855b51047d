// Full-catalogue logits  D[M,V] = out[M,d] . E[V,d]^T  for hidden sizes the tcgen05 path (logits_tc.cu, d = 64)
// does not take (d = 128 of config/yelp.yaml:39, d = 256 of the long-sequence stress configuration): plain fp32
// FMA, the consumer fused into the register epilogue exactly as in the tensor-core path, so the [M,V] logits
// never reach HBM in the CE / top-k modes.  Same modes, same [m_tile(128), n_chunk] CTA plan, same partial layouts.
//
// CTA = 256 threads = 128 logits rows x 2 column halves: thread (row, half) owns row `row` of the m-tile and the
// 32 columns [half*32, half*32+32) of every 64-row catalogue tile, so the online softmax / top-k state is
// thread-private; the two halves of a row are merged through shared memory when the CTA is done.  The K axis is
// walked in 32-wide chunks: out^T chunk [32][128] and table^T chunk [32][64] in shared memory (register-prefetched
// from global/L2 one chunk ahead); per k one conflict-free LDS of the row's activation and eight broadcast float4
// LDS of the table chunk feed 32 FMAs.
#include "logits_common.cuh"

namespace acsr {

constexpr int kSimtThreads = 256;
constexpr int kSimtKC = 32;            // K chunk

struct SimtSmem {
  float* As;        // [kSimtKC][kBM]
  float* Bs;        // [kSimtKC][kBN]
  float* pair;      // [kBM][2]   half 1 -> half 0 hand-over (CE)
  int* cnts;        // [kBM]      half 1's candidate count (TOPK)
  float* lval;      // [k][256]
  int* lidx;        // [k][256]
};

__device__ __forceinline__ void simt_topk_insert(float x, int col, float* lval, int* lidx, int slot0, int k, int& cnt, float& thr,
                                                 int& minpos) {
  if (cnt < k) {
    lval[cnt * kSimtThreads + slot0] = x;
    lidx[cnt * kSimtThreads + slot0] = col;
    if (++cnt < k) return;
  } else {
    lval[minpos * kSimtThreads + slot0] = x;
    lidx[minpos * kSimtThreads + slot0] = col;
  }
  float m = lval[slot0];
  int mp = 0;
  for (int s = 1; s < k; ++s) {
    const float v = lval[s * kSimtThreads + slot0];
    if (v < m) { m = v; mp = s; }
  }
  thr = m;
  minpos = mp;
}

template <int MODE>
__global__ void __launch_bounds__(kSimtThreads, 1) logits_simt_kernel(const LogitsParams p, const int d) {
  pdl_launch_dependents();
  pdl_wait();
  constexpr bool kTopk = MODE == MODE_TOPK || MODE == MODE_TOPK_RANK, kRank = MODE == MODE_TOPK_RANK;
  extern __shared__ __align__(16) float smem_f[];
  SimtSmem sm;
  sm.As = smem_f;
  sm.Bs = sm.As + kSimtKC * kBM;
  sm.pair = sm.Bs + kSimtKC * kBN;
  sm.cnts = reinterpret_cast<int*>(sm.pair + 2 * kBM);
  sm.lval = reinterpret_cast<float*>(sm.cnts + kBM);
  sm.lidx = reinterpret_cast<int*>(sm.lval + (kTopk ? p.k * kSimtThreads : 0));

  const int tid = threadIdx.x;
  const int row = tid & (kBM - 1), half = tid >> 7;
  const int m_tile = blockIdx.x % p.m_tiles;
  const int chunk = blockIdx.x / p.m_tiles;
  const int my_tiles = chunk < p.n_tiles ? (p.n_tiles - chunk + p.n_chunks - 1) / p.n_chunks : 0;
  const int nkc = (d + kSimtKC - 1) / kSimtKC;
  const int total = my_tiles * nkc;
  const int m0 = m_tile * kBM;
  const int grow = m0 + row;
  const bool row_ok = grow < p.M;

  float run_m = -INFINITY, run_s = 0.f;         // MODE_CE
  float g_lse = 0.f, g_scale = 0.f;             // MODE_GRAD
  long long g_tgt = -1;
  int cnt = 0, minpos = 0;                      // MODE_TOPK
  float thr = -INFINITY;
  float r_s = INFINITY;                         // MODE_TOPK_RANK: the positive's score, its local column, this thread's counts
  long long r_pl = -1;
  int r_gt = 0, r_eq = 0;
  if (kRank && row_ok) { r_s = p.rank_score[grow]; r_pl = p.rank_pos[grow] - p.idx_offset; }
  if (MODE == MODE_GRAD && row_ok) { g_lse = p.lse[grow]; g_scale = p.row_scale[grow]; g_tgt = p.target[grow]; }

  float4 pa[4], pb[2];
  auto prefetch = [&](int step) {
    const int it = step / nkc, kc = step - it * nkc;
    const long long n0 = (long long)(chunk + it * p.n_chunks) * kBN;
    const int k0 = kc * kSimtKC;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int idx = q * kSimtThreads + tid;
      const int r = idx & (kBM - 1), k = k0 + (idx >> 7) * 4;
      pa[q] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (m0 + r < p.M && k < d) pa[q] = *reinterpret_cast<const float4*>(p.out + (long long)(m0 + r) * d + k);
    }
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int idx = q * kSimtThreads + tid;
      const int n = idx & (kBN - 1), k = k0 + (idx >> 6) * 4;
      pb[q] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (n0 + n < p.V && k < d) pb[q] = *reinterpret_cast<const float4*>(p.table + (n0 + n) * d + k);
    }
  };
  auto commit = [&]() {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int idx = q * kSimtThreads + tid;
      const int r = idx & (kBM - 1), k = (idx >> 7) * 4;
      sm.As[(k + 0) * kBM + r] = pa[q].x; sm.As[(k + 1) * kBM + r] = pa[q].y;
      sm.As[(k + 2) * kBM + r] = pa[q].z; sm.As[(k + 3) * kBM + r] = pa[q].w;
    }
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int idx = q * kSimtThreads + tid;
      const int n = idx & (kBN - 1), k = (idx >> 6) * 4;
      sm.Bs[(k + 0) * kBN + n] = pb[q].x; sm.Bs[(k + 1) * kBN + n] = pb[q].y;
      sm.Bs[(k + 2) * kBN + n] = pb[q].z; sm.Bs[(k + 3) * kBN + n] = pb[q].w;
    }
  };

  float acc[32];
  if (total > 0) prefetch(0);
  for (int step = 0; step < total; ++step) {
    const int it = step / nkc, kc = step - it * nkc;
    __syncthreads();                     // the previous chunk has been consumed
    commit();
    __syncthreads();
    if (step + 1 < total) prefetch(step + 1);
    if (kc == 0) {
#pragma unroll
      for (int i = 0; i < 32; ++i) acc[i] = 0.f;
    }
    const float4* b4 = reinterpret_cast<const float4*>(sm.Bs) + half * 8;
#pragma unroll 8
    for (int k = 0; k < kSimtKC; ++k) {
      const float a = sm.As[k * kBM + row];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float4 b = b4[k * (kBN / 4) + q];
        acc[4 * q + 0] = fmaf(a, b.x, acc[4 * q + 0]);
        acc[4 * q + 1] = fmaf(a, b.y, acc[4 * q + 1]);
        acc[4 * q + 2] = fmaf(a, b.z, acc[4 * q + 2]);
        acc[4 * q + 3] = fmaf(a, b.w, acc[4 * q + 3]);
      }
    }
    if (kc != nkc - 1) continue;
    // ---------------- epilogue of tile `it`: this thread's 32 logits of row `grow` ----------------
    const long long c0 = (long long)(chunk + it * p.n_chunks) * kBN + half * 32;
    const int nvalid = (int)((p.V - c0) < 32 ? ((p.V - c0) > 0 ? (p.V - c0) : 0) : 32);
    if (MODE == MODE_GRAD) {
      // transposed store Gt[v][m]: a warp's 32 rows are 32 consecutive floats -> coalesced 128-byte lines
      if (row_ok) {
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          if (i < nvalid) {
            float g = __expf(acc[i] - g_lse);
            if (c0 + i == g_tgt) g -= 1.0f;
            p.C[(c0 + i) * p.ldc + grow] = g * g_scale;
          }
        }
      }
    } else if (MODE == MODE_STORE) {
      if (row_ok) {
        float* dst = p.C + (long long)grow * p.ldc + c0;
        if (nvalid == 32 && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) {
#pragma unroll
          for (int i = 0; i < 32; i += 4) *reinterpret_cast<float4*>(dst + i) = make_float4(acc[i], acc[i + 1], acc[i + 2], acc[i + 3]);
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) if (i < nvalid) dst[i] = acc[i];
        }
      }
    } else if (MODE == MODE_CE) {
      if (nvalid > 0) {
        float cm = -INFINITY;
#pragma unroll
        for (int i = 0; i < 32; ++i) if (i < nvalid) cm = fmaxf(cm, acc[i]);
        const float nm = fmaxf(run_m, cm);
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 32; ++i) if (i < nvalid) s += __expf(acc[i] - nm);
        run_s = run_s * __expf(run_m - nm) + s;
        run_m = nm;
      }
    } else {   // MODE_TOPK / MODE_TOPK_RANK
      const int k = p.k;
      if (kRank) {
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const bool ok = i < nvalid && !(p.skip_col0 && c0 + i == 0) && c0 + i != r_pl;
          r_gt += ok && acc[i] > r_s;
          r_eq += ok && acc[i] == r_s;
        }
      }
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const float x = acc[i];
        if (i < nvalid && !(p.skip_col0 && c0 + i == 0) && (cnt < k || x > thr))
          simt_topk_insert(x, (int)(c0 + i), sm.lval, sm.lidx, tid, k, cnt, thr, minpos);
      }
    }
  }
  // ---------------- merge the two column halves of every row, write the chunk's partial ----------------
  if (MODE == MODE_CE) {
    if (half == 1) { sm.pair[2 * row] = run_m; sm.pair[2 * row + 1] = run_s; }
    __syncthreads();
    if (half == 0 && row_ok) {
      const float om = sm.pair[2 * row], os = sm.pair[2 * row + 1];
      const float nm = fmaxf(run_m, om);
      float s = 0.f;
      if (run_s > 0.f) s += run_s * __expf(run_m - nm);
      if (os > 0.f) s += os * __expf(om - nm);
      float* o = p.partial + ((long long)grow * p.n_chunks + chunk) * 2;
      o[0] = nm; o[1] = s;
    }
  }
  if (kTopk) {
    int* rpair = reinterpret_cast<int*>(sm.pair);   // MODE_TOPK_RANK: half 1's two counts (the CE hand-over slots are free here)
    if (half == 1) {
      sm.cnts[row] = cnt;
      if (kRank) { rpair[2 * row] = r_gt; rpair[2 * row + 1] = r_eq; }
    }
    __syncthreads();
    if (half == 0) {
      if (kRank) { r_gt += rpair[2 * row]; r_eq += rpair[2 * row + 1]; }
      const int k = p.k, oc = sm.cnts[row], oslot = tid + kBM;
      for (int s = 0; s < oc; ++s) {
        const float x = sm.lval[s * kSimtThreads + oslot];
        if (cnt < k || x > thr) simt_topk_insert(x, sm.lidx[s * kSimtThreads + oslot], sm.lval, sm.lidx, tid, k, cnt, thr, minpos);
      }
      if (row_ok) {
        float* ov = p.pval + ((long long)grow * p.n_slots + chunk) * k;
        long long* oi = p.pidx + ((long long)grow * p.n_slots + chunk) * k;
        for (int s = 0; s < k; ++s) {
          const bool ok = s < cnt;
          ov[s] = ok ? sm.lval[s * kSimtThreads + tid] : -INFINITY;
          oi[s] = ok ? (long long)sm.lidx[s * kSimtThreads + tid] + p.idx_offset : -1;
        }
        for (int c = p.n_chunks + chunk; c < p.n_slots; c += p.n_chunks) {     // lists no CTA produces
          float* pv = p.pval + ((long long)grow * p.n_slots + c) * k;
          long long* pi = p.pidx + ((long long)grow * p.n_slots + c) * k;
          for (int s = 0; s < k; ++s) { pv[s] = -INFINITY; pi[s] = -1; }
        }
        if (kRank) {
          int* rc = p.rank_counts + (long long)grow * p.n_slots * 2;
          rc[2 * chunk] = r_gt;
          rc[2 * chunk + 1] = r_eq;
          for (int c = p.n_chunks + chunk; c < p.n_slots; c += p.n_chunks) { rc[2 * c] = 0; rc[2 * c + 1] = 0; }
        }
      }
    }
  }
}

template <int MODE>
static int launch_simt(LogitsParams& p, int d, cudaStream_t st, const char* who) {
  logits_plan(p);
  constexpr bool kTopk = MODE == MODE_TOPK || MODE == MODE_TOPK_RANK;
  if (kTopk) logits_plan_topk(p);
  size_t smem = (size_t)(kSimtKC * kBM + kSimtKC * kBN + 2 * kBM + kBM) * 4;
  if (kTopk) smem += (size_t)2 * p.k * kSimtThreads * 4;
  cudaError_t e = cudaFuncSetAttribute(logits_simt_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) { set_error("%s: smem attr: %s", who, cudaGetErrorString(e)); return ACSR_ERR_CUDA; }
  launch_pdl(logits_simt_kernel<MODE>, dim3(p.m_tiles * p.n_chunks), dim3(kSimtThreads), smem, st, p, d);
  return check_launch(who);
}

int launch_logits_simt(int mode, LogitsParams& p, int d, cudaStream_t st, const char* who) {
  if (d < 4 || d > 1024 || (d & 3)) {
    set_error("%s: hidden size %d unsupported (multiple of 4, 4..1024)", who, d);
    return ACSR_ERR_UNSUPPORTED;
  }
  switch (mode) {
    case MODE_STORE: return launch_simt<MODE_STORE>(p, d, st, who);
    case MODE_CE: return launch_simt<MODE_CE>(p, d, st, who);
    case MODE_GRAD: return launch_simt<MODE_GRAD>(p, d, st, who);
    case MODE_TOPK: return launch_simt<MODE_TOPK>(p, d, st, who);
    case MODE_TOPK_RANK: return launch_simt<MODE_TOPK_RANK>(p, d, st, who);
  }
  set_error("%s: bad mode", who);
  return ACSR_ERR_ARG;
}

}  // namespace acsr
