// Merge of the per-chunk (and per-vocab-shard) partial top-k lists: one CTA per user row.  The n_parts*k candidates
// are turned into order-preserving 32-bit keys in shared memory, the k-th largest key is found with a 4-pass radix
// select (256-bin shared-memory histograms), the k winners are gathered (ties on the k-th key: lowest candidate slot
// first) and only those k are sorted (descending score, ascending slot on ties) before the final item ids, scores and the
// hit flags the collector needs are written (evaluator/collector.py:147-153: pos_matrix gather -> [B,k] flags + pos_len).
#include "acsr_common.cuh"
#include "../../include/acsr.h"

namespace acsr {

constexpr int kMergeThreads = 256;
constexpr int kMergeMaxK = 64;
constexpr int kFastCap = 512;        // candidates the fast path sorts (P/2 <= 256 threads)
// The 32-bit keys of one row (dynamic shared memory) and the kernel's static arrays (histograms, scan, fast-path candidates:
// 15,904 bytes by ptxas -v) share the 227 KB a block may use; a key count beyond that cannot be launched at all.
constexpr int kMergeStaticBytes = 16 * 1024;
constexpr int kMergeMaxCand = (227 * 1024 - kMergeStaticBytes) / 4;     // 54,016 keys

__device__ __forceinline__ unsigned f2key(float v) {        // larger float <-> larger unsigned
  const unsigned u = __float_as_uint(v);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// RANK: counts[row] = (#items scoring > s_pos, #items scoring == s_pos) with s_pos = pos_score[row].  Dense rows count their own
// scores, the excluded position 0 and the positive's own column left out; candidate lists sum the n_count_parts (greater, equal)
// pairs pcounts[row, :] the producers of the lists counted.
template <bool RANK>
__global__ void __launch_bounds__(kMergeThreads)
topk_merge_kernel(const float* __restrict__ pval, const long long* __restrict__ pidx, int n_cand, long long ld, int k,
                  int skip_first, long long idx_offset, const long long* __restrict__ positive, float* __restrict__ oval,
                  long long* __restrict__ oidx, int* __restrict__ rec, const float* __restrict__ pos_score,
                  const int* __restrict__ pcounts, int n_count_parts, int* __restrict__ counts) {
  // pidx != NULL: candidate lists (value, item id; id < 0 = padding).  pidx == NULL: a dense score row, item id = position +
  // idx_offset, position 0 excluded when skip_first (trainer.py:942: scores[:, 0] = -inf).
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ unsigned smem_k[];
  unsigned* keys = smem_k;                               // [n_cand]
  __shared__ int hist[256];
  __shared__ int whist[kMergeThreads / 32][256];      // per-warp histograms of the first (most skewed) pass
  __shared__ int scan[kMergeThreads];
  __shared__ unsigned long long sel[kMergeMaxK];         // (key << 32) | ~slot : sorts descending as (score desc, slot asc)
  __shared__ unsigned s_prefix;
  __shared__ int s_need, s_cnt;
  const int row = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* rv = pval + (long long)row * ld;
  const long long* ri = pidx ? pidx + (long long)row * ld : nullptr;
  int r_gt = 0, r_eq = 0;                                // RANK: this thread's share of the row's counts
  __shared__ int s_gt, s_eq;
  const float r_s = RANK && pidx == nullptr ? pos_score[row] : 0.f;
  const long long r_pl = RANK && pidx == nullptr ? positive[row] - idx_offset : -1;
  if (RANK && pidx == nullptr) {                         // dense row: each score is read once for its key and its count
    for (int i = tid; i < n_cand; i += kMergeThreads) {
      const bool valid = !(skip_first && i == 0);
      const float x = rv[i];
      keys[i] = valid ? f2key(x) : 0u;
      if (valid && i != r_pl) { r_gt += x > r_s; r_eq += x == r_s; }
    }
  } else {
    for (int i = tid; i < n_cand; i += kMergeThreads) {
      const bool valid = ri ? ri[i] >= 0 : !(skip_first && i == 0);
      keys[i] = valid ? f2key(rv[i]) : 0u;                // padding entries sort last
    }
  }
  if (RANK && pidx != nullptr)
    for (int i = tid; i < n_count_parts; i += kMergeThreads) {
      r_gt += pcounts[((long long)row * n_count_parts + i) * 2];
      r_eq += pcounts[((long long)row * n_count_parts + i) * 2 + 1];
    }
  if (RANK && tid == 0) { s_gt = 0; s_eq = 0; }
  if (tid == 0) { s_prefix = 0u; s_need = k; s_cnt = 0; }
  if (tid < kMergeMaxK) sel[tid] = 0ull;
  // ---- fast path: a lower bound T0 of the k-th largest key from the threads' local maxima (at least k keys are >= the k-th
  // largest of the 256 local maxima), then only the handful of keys >= T0 are gathered and sorted.  Exact, ties included
  // (every key equal to the k-th largest is >= T0); rows with more than kFastCap such keys (heavy ties) take the radix select.
  __shared__ unsigned lmax[kMergeThreads];
  __shared__ unsigned long long cand[kFastCap];
  __shared__ int s_ncand;
  bool fast_done = false;
  {
    unsigned m = 0u;
    for (int i = tid; i < n_cand; i += kMergeThreads) m = max(m, keys[i]);     // own writes: no barrier needed yet
    lmax[tid] = m;
    if (tid == 0) s_ncand = 0;
    __syncthreads();
    for (int size = 2; size <= kMergeThreads; size <<= 1) {                    // bitonic sort of the 256 maxima, descending
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        if (tid < kMergeThreads / 2) {
          const int l = 2 * tid - (tid & (stride - 1)), h = l + stride;
          const bool desc = (l & size) == 0;
          const unsigned a = lmax[l], b = lmax[h];
          if ((a > b) != desc) { lmax[l] = b; lmax[h] = a; }
        }
        __syncthreads();
      }
    }
    const unsigned T0 = lmax[k - 1];
    if (T0 != 0u) {
      for (int i = tid; i < n_cand; i += kMergeThreads) {
        const unsigned key = keys[i];
        if (key >= T0) {
          const int pos = atomicAdd(&s_ncand, 1);
          if (pos < kFastCap) cand[pos] = ((unsigned long long)key << 32) | (unsigned)(~(unsigned)i);
        }
      }
    }
    __syncthreads();
    const int nc = T0 != 0u ? s_ncand : kFastCap + 1;
    if (nc <= kFastCap) {                                                       // uniform over the CTA
      int P = 64;
      while (P < nc) P <<= 1;
      for (int i = nc + tid; i < P; i += kMergeThreads) cand[i] = 0ull;
      __syncthreads();
      for (int size = 2; size <= P; size <<= 1) {                               // sort the candidates: (score desc, slot asc)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
          if (tid < P / 2) {
            const int l = 2 * tid - (tid & (stride - 1)), h = l + stride;
            const bool desc = (l & size) == 0;
            const unsigned long long a = cand[l], b = cand[h];
            if ((a > b) != desc) { cand[l] = b; cand[h] = a; }
          }
          __syncthreads();
        }
      }
      if (tid < k) sel[tid] = cand[tid];
      fast_done = true;
    }
  }
  if (!fast_done) {
  unsigned mask = 0u;
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    hist[tid] = 0;
    if (pass == 0) {
#pragma unroll
      for (int w = 0; w < kMergeThreads / 32; ++w) whist[w][tid] = 0;
    }
    __syncthreads();
    const unsigned prefix = s_prefix;
    if (pass == 0) {
      // sign + exponent bits: a handful of bins take almost every key.  Lanes with the same bin elect a leader that adds
      // their count to the warp's private histogram.
      for (int i0 = 0; i0 < n_cand; i0 += kMergeThreads) {
        const int i = i0 + tid;
        const bool in = i < n_cand;
        const unsigned bin = in ? (keys[i] >> 24) : 0x100u + lane;
        const unsigned peers = __match_any_sync(0xffffffffu, bin);
        if (in && lane == __ffs(peers) - 1) atomicAdd(&whist[warp][bin], __popc(peers));
      }
      __syncthreads();
      int t = 0;
#pragma unroll
      for (int w = 0; w < kMergeThreads / 32; ++w) t += whist[w][tid];
      hist[tid] = t;
    } else {
      for (int i = tid; i < n_cand; i += kMergeThreads) {
        const unsigned key = keys[i];
        if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1);
      }
    }
    __syncthreads();
    if (warp == 0) {
      // lane l owns the 8 bins [248-8l, 255-8l]; walk the bins from the top until `need` keys are covered
      const int need = s_need;
      int mine = 0;
#pragma unroll
      for (int q = 0; q < 8; ++q) mine += hist[255 - 8 * lane - q];
      int incl = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
      const unsigned hit = __ballot_sync(0xffffffffu, incl >= need);
      const int owner = __ffs(hit) - 1;                   // always found: the matching keys number at least `need`
      if (lane == owner) {
        int cum = incl - mine;
        for (int q = 0; q < 8; ++q) {
          const int bin = 255 - 8 * lane - q;
          const int c = hist[bin];
          if (cum + c >= need) { s_prefix = prefix | ((unsigned)bin << shift); s_need = need - cum; break; }
          cum += c;
        }
      }
    }
    mask |= 0xffu << shift;
    __syncthreads();
  }
  const unsigned T = s_prefix;           // the k-th largest key
  const int need = s_need;               // how many candidates equal to T are taken (lowest slots first)
  const int n_gt = k - need;
  // winners above the threshold: any order (sorted below)
  for (int i = tid; i < n_cand; i += kMergeThreads) {
    const unsigned key = keys[i];
    if (key > T) sel[atomicAdd(&s_cnt, 1)] = ((unsigned long long)key << 32) | (unsigned)(~(unsigned)i);
  }
  // ties on the threshold, in slot order: contiguous index ranges per thread + an exclusive scan of the tie counts
  const int per = (n_cand + kMergeThreads - 1) / kMergeThreads;
  const int lo = tid * per, hi = min(n_cand, lo + per);
  int ties = 0;
  for (int i = lo; i < hi; ++i) ties += keys[i] == T;
  scan[tid] = ties;
  __syncthreads();
  for (int o = 1; o < kMergeThreads; o <<= 1) {
    const int t = tid >= o ? scan[tid - o] : 0;
    __syncthreads();
    scan[tid] += t;
    __syncthreads();
  }
  int rank = scan[tid] - ties;
  for (int i = lo; i < hi && rank < need; ++i)
    if (keys[i] == T) { sel[n_gt + rank] = ((unsigned long long)T << 32) | (unsigned)(~(unsigned)i); ++rank; }
  __syncthreads();
  // bitonic sort of the 64 selected entries, descending
  if (tid < kMergeMaxK / 2 * 2) {
    for (int size = 2; size <= kMergeMaxK; size <<= 1) {
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        if (tid < kMergeMaxK / 2) {
          const int l = 2 * tid - (tid & (stride - 1)), h = l + stride;
          const bool desc = (l & size) == 0;
          const unsigned long long a = sel[l], b = sel[h];
          if ((a > b) != desc) { sel[l] = b; sel[h] = a; }
        }
        __syncwarp();
      }
    }
  }
  }   // radix-select path
  __syncthreads();
  if (RANK) {                                            // s_gt / s_eq were zeroed before the barriers above
    r_gt = __reduce_add_sync(0xffffffffu, r_gt);
    r_eq = __reduce_add_sync(0xffffffffu, r_eq);
    if (lane == 0) { atomicAdd(&s_gt, r_gt); atomicAdd(&s_eq, r_eq); }
    __syncthreads();
    if (tid == 0) { counts[2 * row] = s_gt; counts[2 * row + 1] = s_eq; }
  }
  const long long pos_item = positive ? positive[row] : -1;
  for (int j = tid; j < k; j += kMergeThreads) {
    const unsigned long long e = sel[j];
    const int slot = (int)(~(unsigned)(e & 0xffffffffull));
    const bool ok = e != 0ull && (e >> 32) != 0ull && slot >= 0 && slot < n_cand;
    const long long id = ok ? (ri ? ri[slot] : slot + idx_offset) : -1;
    oval[(long long)row * k + j] = ok ? rv[slot] : -INFINITY;
    oidx[(long long)row * k + j] = id;
    if (rec) rec[(long long)row * (k + 1) + j] = (id == pos_item && id >= 0) ? 1 : 0;
  }
  if (rec && tid == 0) rec[(long long)row * (k + 1) + k] = 1;   // pos_len: one held-out item per user
}

}  // namespace acsr

using namespace acsr;

extern "C" int acsr_topk_merge(const float* partial_val, const int64_t* partial_idx, int M, int n_parts, int k,
                               const int64_t* positive, float* topk_val, int64_t* topk_idx, int32_t* rec_topk, void* stream) {
  ACSR_REQUIRE(partial_val && partial_idx && topk_val && topk_idx, "topk_merge: NULL pointer");
  ACSR_REQUIRE(M > 0 && n_parts > 0 && k > 0, "topk_merge: bad sizes");
  const int n_cand = n_parts * k;
  if (n_cand > kMergeMaxCand) { set_error("topk_merge: %d candidates per row exceed %d", n_cand, kMergeMaxCand); return ACSR_ERR_UNSUPPORTED; }
  ACSR_REQUIRE(n_cand >= k, "topk_merge: fewer candidates than k");
  if (k > kMergeMaxK) { set_error("topk_merge: k=%d unsupported (1..%d)", k, kMergeMaxK); return ACSR_ERR_UNSUPPORTED; }
  const size_t smem = (size_t)n_cand * 4;
  cudaError_t e = cudaFuncSetAttribute(topk_merge_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) { set_error("topk_merge: smem attr: %s", cudaGetErrorString(e)); return ACSR_ERR_CUDA; }
  launch_pdl(topk_merge_kernel<false>, dim3(M), dim3(kMergeThreads), smem, (cudaStream_t)stream, partial_val, (const long long*)partial_idx, n_cand,
             (long long)n_cand, k, 0, 0ll, (const long long*)positive, topk_val, (long long*)topk_idx, rec_topk, (const float*)nullptr,
             (const int*)nullptr, 0, (int*)nullptr);
  return check_launch("topk_merge");
}

extern "C" int acsr_topk_merge_rank(const float* partial_val, const int64_t* partial_idx, int M, int n_parts, int k,
                                    const int64_t* positive, const int32_t* partial_counts, int n_count_parts, float* topk_val,
                                    int64_t* topk_idx, int32_t* rec_topk, int32_t* counts, void* stream) {
  ACSR_REQUIRE(partial_val && partial_idx && topk_val && topk_idx && partial_counts && counts, "topk_merge_rank: NULL pointer");
  ACSR_REQUIRE(M > 0 && n_parts > 0 && k > 0 && n_count_parts > 0, "topk_merge_rank: bad sizes");
  const int n_cand = n_parts * k;
  if (n_cand > kMergeMaxCand) { set_error("topk_merge_rank: %d candidates per row exceed %d", n_cand, kMergeMaxCand); return ACSR_ERR_UNSUPPORTED; }
  if (k > kMergeMaxK) { set_error("topk_merge_rank: k=%d unsupported (1..%d)", k, kMergeMaxK); return ACSR_ERR_UNSUPPORTED; }
  const size_t smem = (size_t)n_cand * 4;
  cudaError_t e = cudaFuncSetAttribute(topk_merge_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) { set_error("topk_merge_rank: smem attr: %s", cudaGetErrorString(e)); return ACSR_ERR_CUDA; }
  launch_pdl(topk_merge_kernel<true>, dim3(M), dim3(kMergeThreads), smem, (cudaStream_t)stream, partial_val, (const long long*)partial_idx,
             n_cand, (long long)n_cand, k, 0, 0ll, (const long long*)positive, topk_val, (long long*)topk_idx, rec_topk,
             (const float*)nullptr, (const int*)partial_counts, n_count_parts, (int*)counts);
  return check_launch("topk_merge_rank");
}

extern "C" int acsr_topk_select_max_items(void) { return kMergeMaxCand; }

extern "C" int acsr_topk_select(const float* scores, int M, int64_t V, int64_t ld, int k, int skip_col0, int64_t idx_offset,
                                const int64_t* positive, float* topk_val, int64_t* topk_idx, int32_t* rec_topk, void* stream) {
  ACSR_REQUIRE(scores && topk_val && topk_idx, "topk_select: NULL pointer");
  ACSR_REQUIRE(M > 0 && V > 0 && k > 0 && ld >= V, "topk_select: bad sizes");
  if (V > kMergeMaxCand) { set_error("topk_select: %lld items per row exceed %d (use the fused top-k)", (long long)V, kMergeMaxCand); return ACSR_ERR_UNSUPPORTED; }
  if (k > kMergeMaxK) { set_error("topk_select: k=%d unsupported (1..%d)", k, kMergeMaxK); return ACSR_ERR_UNSUPPORTED; }
  ACSR_REQUIRE(V - (skip_col0 ? 1 : 0) >= k, "topk_select: fewer items than k");
  const size_t smem = (size_t)V * 4;
  cudaError_t e = cudaFuncSetAttribute(topk_merge_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) { set_error("topk_select: smem attr: %s", cudaGetErrorString(e)); return ACSR_ERR_CUDA; }
  launch_pdl(topk_merge_kernel<false>, dim3(M), dim3(kMergeThreads), smem, (cudaStream_t)stream, scores, (const long long*)nullptr, (int)V, (long long)ld, k,
             skip_col0 ? 1 : 0, (long long)idx_offset, (const long long*)positive, topk_val, (long long*)topk_idx, rec_topk,
             (const float*)nullptr, (const int*)nullptr, 0, (int*)nullptr);
  return check_launch("topk_select");
}

extern "C" int acsr_topk_select_rank(const float* scores, int M, int64_t V, int64_t ld, int k, int skip_col0, int64_t idx_offset,
                                     const int64_t* positive, const float* pos_score, float* topk_val, int64_t* topk_idx,
                                     int32_t* rec_topk, int32_t* counts, void* stream) {
  ACSR_REQUIRE(scores && topk_val && topk_idx && positive && pos_score && counts, "topk_select_rank: NULL pointer");
  ACSR_REQUIRE(M > 0 && V > 0 && k > 0 && ld >= V, "topk_select_rank: bad sizes");
  if (V > kMergeMaxCand) { set_error("topk_select_rank: %lld items per row exceed %d (use the fused top-k)", (long long)V, kMergeMaxCand); return ACSR_ERR_UNSUPPORTED; }
  if (k > kMergeMaxK) { set_error("topk_select_rank: k=%d unsupported (1..%d)", k, kMergeMaxK); return ACSR_ERR_UNSUPPORTED; }
  ACSR_REQUIRE(V - (skip_col0 ? 1 : 0) >= k, "topk_select_rank: fewer items than k");
  const size_t smem = (size_t)V * 4;
  cudaError_t e = cudaFuncSetAttribute(topk_merge_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) { set_error("topk_select_rank: smem attr: %s", cudaGetErrorString(e)); return ACSR_ERR_CUDA; }
  launch_pdl(topk_merge_kernel<true>, dim3(M), dim3(kMergeThreads), smem, (cudaStream_t)stream, scores, (const long long*)nullptr, (int)V,
             (long long)ld, k, skip_col0 ? 1 : 0, (long long)idx_offset, (const long long*)positive, topk_val, (long long*)topk_idx,
             rec_topk, pos_score, (const int*)nullptr, 0, (int*)counts);
  return check_launch("topk_select_rank");
}
