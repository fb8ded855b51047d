// Negative sampling on the device and the ranking of sampled candidates.
//
// RecBole draws negatives on the host (recbole/sampler/sampler.py sample_by_user_ids: numpy draws, rejected while they hit
// the user's used ids) and ranks a test user's positive among them by scattering 1+N candidate scores into a -inf [B, n_items]
// matrix and running topk over it (trainer/trainer.py _neg_sample_batch_eval, evaluator/collector.py eval_batch_collect).
// Here both are one kernel each:
//   acsr_neg_sample      one warp per row.  Uniform: r ~ U[0, |complement|), mapped to the r-th item not in the user's sorted
//                        used set by a binary search -- exact, bounded cost, no rejection loop.  Popularity: alias draw, rejected
//                        while it hits the used set, at most kPopTries times, then the uniform-complement draw.
//   acsr_candidate_rank  one CTA per row: fp32 gather-dots of out[m] with the candidates' table rows, and the rank of the
//                        positive = number of DISTINCT negatives scoring strictly higher (a shared-memory hash set de-duplicates
//                        only those), written as the [M, kmax+1] hit-flag matrix the evaluator consumes.
#include "acsr_common.cuh"
#include "../../include/acsr.h"

namespace acsr {

constexpr int kPopTries = 16;            // alias draws per negative before the uniform-complement draw takes over
constexpr int kRankMaxCand = 8192;       // 1 + N of acsr_candidate_rank
constexpr int kRankMaxK = 1024;          // kmax of acsr_candidate_rank
constexpr int kRankThreads = 256;
constexpr unsigned kNegRngStreamBits = 5;   // counter = (row * N + j) << 5 | attempt (0: uniform draw, 1..16: alias draws)

// number of entries of the sorted set u[0, n) that are <= x
__device__ __forceinline__ long long count_le(const long long* __restrict__ u, long long n, long long x) {
  long long lo = 0, hi = n;
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    if (__ldg(u + mid) <= x) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// the r-th (0-based) item of [1, n_items) that is not in the sorted set u[0, n): with f(j) = u[j] - 1 - j (complement items
// below u[j], non-decreasing) and c = #{j : f(j) <= r}, the answer is 1 + r + c
__device__ __forceinline__ long long select_complement(const long long* __restrict__ u, long long n, long long r) {
  long long lo = 0, hi = n;
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    if (__ldg(u + mid) - 1 - mid <= r) lo = mid + 1; else hi = mid;
  }
  return 1 + r + lo;
}

__device__ __forceinline__ unsigned long long bits64(uint4 b, int half) {
  return half ? (((unsigned long long)b.w << 32) | b.z) : (((unsigned long long)b.y << 32) | b.x);
}

__global__ void __launch_bounds__(256) neg_sample_kernel(const long long* __restrict__ users, const long long* __restrict__ positives,
                                                         const long long* __restrict__ perm, const long long* __restrict__ cursor,
                                                         long long n_rows, int M, int N, const long long* __restrict__ offsets,
                                                         const long long* __restrict__ used, long long n_users, long long n_items,
                                                         const float* __restrict__ prob, const long long* __restrict__ alias,
                                                         const RngState* __restrict__ rng, unsigned rng_stream,
                                                         long long* __restrict__ negs, long long ld) {
  pdl_launch_dependents();
  pdl_wait();
  const unsigned long long seed = rng->seed, step = rng->step;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long base = perm != nullptr ? cursor[0] * (long long)M : 0;
  for (int r = blockIdx.x * 8 + warp; r < M; r += gridDim.x * 8) {
    long long src = r;
    if (perm != nullptr) {
      src = base + r;
      src = perm[src < n_rows ? src : n_rows - 1];            // (a cursor past the end repeats the last row, as batch_gather does)
    }
    const long long u = users[src];
    if (u < 0 || u >= n_users) {                               // no used set to exclude: item 0, which no valid draw returns
      for (int j = lane; j < N; j += 32) negs[(long long)r * ld + j] = 0;
      continue;
    }
    const long long* U = used + offsets[u];
    const long long nu = offsets[u + 1] - offsets[u];
    // the positive joins the excluded set when it is a real item outside the used set (it is always inside on RecBole's splits)
    long long p = positives != nullptr ? positives[src] : 0;
    if (p <= 0 || p >= n_items || (nu > 0 && count_le(U, nu, p) != count_le(U, nu, p - 1))) p = 0;
    const long long n_comp = (n_items - 1) - nu - (p > 0 ? 1 : 0);
    for (int j = lane; j < N; j += 32) {
      const unsigned long long ctr = ((unsigned long long)r * N + j) << kNegRngStreamBits;
      long long item = -1;
      if (prob != nullptr) {
        for (int t = 0; t < kPopTries && item < 0; ++t) {
          const uint4 b = philox4x32(seed, step, rng_stream, ctr | (unsigned long long)(t + 1));
          const long long col = (long long)__umul64hi(bits64(b, 0), (unsigned long long)n_items);
          const long long cand = u32_to_unit(b.z) <= __ldg(prob + col) ? col : __ldg(alias + col);
          if (cand <= 0 || cand >= n_items || cand == p) continue;
          if (nu > 0 && count_le(U, nu, cand) != count_le(U, nu, cand - 1)) continue;
          item = cand;
        }
      }
      if (item < 0) {
        if (n_comp <= 0) {
          item = 0;                                            // no item left to draw (the host rejects such users up front)
        } else {
          const uint4 b = philox4x32(seed, step, rng_stream, ctr);
          const long long rr = (long long)__umul64hi(bits64(b, 0), (unsigned long long)n_comp);
          item = select_complement(U, nu, rr);
          if (p > 0 && item >= p) item = select_complement(U, nu, rr + 1);
        }
      }
      negs[(long long)r * ld + j] = item;
    }
  }
}

__device__ __forceinline__ unsigned hash_slot(long long id, unsigned mask) {
  return (unsigned)(((unsigned long long)id * 0x9E3779B97F4A7C15ull) >> 40) & mask;
}

// dot of out (shared, d floats) with table row `row`, over a group of G lanes (float4 loads); every lane of the group gets it
template <int G>
__device__ __forceinline__ float group_dot(const float4* __restrict__ o4, const float4* __restrict__ t4, int d4, int sub) {
  float acc = 0.f;
  for (int j = sub; j < d4; j += G) {
    const float4 a = o4[j], b = __ldg(t4 + j);
    acc = fmaf(a.x, b.x, acc);
    acc = fmaf(a.y, b.y, acc);
    acc = fmaf(a.z, b.z, acc);
    acc = fmaf(a.w, b.w, acc);
  }
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o, G);
  return acc;
}

// COUNT: every candidate id enters the hash set (the positive's first), and counts[m] = (distinct negatives scoring above the
// positive = the rank, distinct negatives tied with it, distinct candidates = the finite entries of the scattered score row)
template <int G, bool COUNT>
__global__ void __launch_bounds__(kRankThreads) candidate_rank_kernel(const float* __restrict__ out, const float* __restrict__ table,
                                                                      long long V, int d, const long long* __restrict__ cand, int C,
                                                                      int kmax, int hash_size, int* __restrict__ rec,
                                                                      float* __restrict__ scores, int* __restrict__ counts) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float4* o4 = reinterpret_cast<float4*>(smem_raw);
  long long* hset = reinterpret_cast<long long*>(smem_raw + (size_t)d * 4);
  __shared__ float s_pos;
  __shared__ int s_rank, s_eq, s_distinct;
  pdl_launch_dependents();
  const int m = blockIdx.x, tid = threadIdx.x;
  for (int i = tid; i < hash_size; i += kRankThreads) hset[i] = -1;
  if (tid == 0) { s_rank = 0; s_eq = 0; s_distinct = 1; }
  pdl_wait();
  const int d4 = d >> 2;
  const float4* orow = reinterpret_cast<const float4*>(out + (long long)m * d);
  for (int i = tid; i < d4; i += kRankThreads) o4[i] = orow[i];
  __syncthreads();
  const long long* crow = cand + (long long)m * C;
  const int lane = tid & 31, sub = lane & (G - 1);
  if (tid < 32) {
    long long id = crow[0];
    id = id < 0 ? 0 : (id >= V ? V - 1 : id);
    const float s = group_dot<G>(o4, reinterpret_cast<const float4*>(table + id * d), d4, sub);
    if (tid == 0) {
      s_pos = s;
      if (scores != nullptr) scores[(long long)m * C] = s;
    }
  }
  const unsigned mask = (unsigned)hash_size - 1;
  long long pos_id = crow[0];
  pos_id = pos_id < 0 ? 0 : (pos_id >= V ? V - 1 : pos_id);
  if (COUNT && tid == 0) hset[hash_slot(pos_id, mask)] = pos_id;     // a negative equal to the positive collapses into it
  __syncthreads();
  const float s0 = s_pos;
  const int groups = kRankThreads / G;
  for (int c = 1 + tid / G; c - (tid / G) < C; c += groups) {          // every lane of a warp iterates the same number of times
    const bool live = c < C;
    long long id = live ? crow[c] : 0;
    id = id < 0 ? 0 : (id >= V ? V - 1 : id);
    const float s = group_dot<G>(o4, reinterpret_cast<const float4*>(table + id * d), d4, sub);
    if (live && sub == 0) {
      if (scores != nullptr) scores[(long long)m * C + c] = s;
      if (COUNT) {
        unsigned h = hash_slot(id, mask);
        while (true) {
          const long long prev = (long long)atomicCAS(reinterpret_cast<unsigned long long*>(hset + h), (unsigned long long)-1ll,
                                                      (unsigned long long)id);
          if (prev == -1) {                                            // first copy of this item among all candidates
            atomicAdd(&s_distinct, 1);
            if (s > s0) atomicAdd(&s_rank, 1);
            else if (s == s0) atomicAdd(&s_eq, 1);
            break;
          }
          if (prev == id) break;
          h = (h + 1) & mask;
        }
      } else if (s > s0) {                                             // ties count in the positive's favour
        unsigned h = hash_slot(id, mask);
        while (true) {
          const long long prev = (long long)atomicCAS(reinterpret_cast<unsigned long long*>(hset + h), (unsigned long long)-1ll,
                                                      (unsigned long long)id);
          if (prev == -1) { atomicAdd(&s_rank, 1); break; }          // first copy of this item among the higher-scoring ones
          if (prev == id) break;                                       // a duplicate negative: counted once
          h = (h + 1) & mask;
        }
      }
    }
  }
  __syncthreads();
  const int rank = s_rank;
  int* rrow = rec + (long long)m * (kmax + 1);
  for (int i = tid; i <= kmax; i += kRankThreads) rrow[i] = (i == kmax) ? 1 : (i == rank ? 1 : 0);
  if (COUNT && tid == 0) {
    counts[3 * m] = rank;
    counts[3 * m + 1] = s_eq;
    counts[3 * m + 2] = s_distinct;
  }
}

}  // namespace acsr

using namespace acsr;

extern "C" {

int acsr_neg_sample(const int64_t* users, const int64_t* positives, const int64_t* perm, const int64_t* cursor, int64_t n_rows, int M,
                    int N, const int64_t* used_offsets, const int64_t* used_items, int64_t n_users, int64_t n_items,
                    const float* alias_prob, const int64_t* alias_idx, const void* rng, uint32_t rng_stream, int64_t* negs,
                    int64_t ld_negs, void* stream) {
  ACSR_REQUIRE(users && used_offsets && used_items && rng && negs, "neg_sample: NULL pointer");
  ACSR_REQUIRE(M > 0 && N > 0 && ld_negs >= N, "neg_sample: bad sizes (M=%d N=%d ld=%lld)", M, N, (long long)ld_negs);
  ACSR_REQUIRE(n_items >= 2 && n_users > 0, "neg_sample: need n_items >= 2 and n_users >= 1");
  ACSR_REQUIRE((perm == nullptr) == (cursor == nullptr), "neg_sample: perm and cursor go together");
  ACSR_REQUIRE(perm == nullptr || n_rows > 0, "neg_sample: n_rows must be positive with a row permutation");
  ACSR_REQUIRE((alias_prob == nullptr) == (alias_idx == nullptr), "neg_sample: alias_prob and alias_idx go together");
  if ((long long)N * M > (1ll << 58)) { set_error("neg_sample: M*N=%lld too large", (long long)N * M); return ACSR_ERR_UNSUPPORTED; }
  int blocks = (M + 7) / 8;
  if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
  launch_pdl(neg_sample_kernel, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, (const long long*)users, (const long long*)positives,
             (const long long*)perm, (const long long*)cursor, (long long)n_rows, M, N, (const long long*)used_offsets,
             (const long long*)used_items, (long long)n_users, (long long)n_items, alias_prob, (const long long*)alias_idx,
             (const RngState*)rng, (unsigned)rng_stream, (long long*)negs, (long long)ld_negs);
  return check_launch("neg_sample");
}

int acsr_candidate_rank_max_candidates(void) { return kRankMaxCand; }

static int candidate_rank_impl(const float* out, const float* table, int64_t V, int d, const int64_t* cand, int M, int n_cand, int kmax,
                               int32_t* rec, float* scores, int32_t* counts, void* stream) {
  ACSR_REQUIRE(out && table && cand && rec, "candidate_rank: NULL pointer");
  ACSR_REQUIRE(M > 0 && V > 0 && n_cand >= 1 && kmax >= 1, "candidate_rank: bad sizes");
  ACSR_REQUIRE(d > 0 && d % 4 == 0, "candidate_rank: hidden size %d must be a positive multiple of 4", d);
  if (d > 1024) { set_error("candidate_rank: hidden size %d unsupported (at most 1024)", d); return ACSR_ERR_UNSUPPORTED; }
  if (n_cand > kRankMaxCand) {
    set_error("candidate_rank: %d candidates per row unsupported (1 + N <= %d, i.e. at most %d negatives)", n_cand, kRankMaxCand,
              kRankMaxCand - 1);
    return ACSR_ERR_UNSUPPORTED;
  }
  if (kmax > kRankMaxK) { set_error("candidate_rank: kmax=%d unsupported (1..%d)", kmax, kRankMaxK); return ACSR_ERR_UNSUPPORTED; }
  ACSR_REQUIRE(((uintptr_t)out & 15) == 0 && ((uintptr_t)table & 15) == 0, "candidate_rank: out / table must be 16-byte aligned");
  int hash_size = 64;
  while (hash_size < 2 * n_cand) hash_size <<= 1;
  const size_t smem = (size_t)d * 4 + (size_t)hash_size * 8;
  const int d4 = d / 4;
  cudaStream_t st = (cudaStream_t)stream;
#define ACSR_RANK_LAUNCH(G)                                                                                                  \
  do {                                                                                                                       \
    if (counts != nullptr) {                                                                                                 \
      cudaError_t e = cudaFuncSetAttribute(candidate_rank_kernel<G, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
      if (e != cudaSuccess) { set_error("candidate_rank: smem attr: %s", cudaGetErrorString(e)); return ACSR_ERR_CUDA; }    \
      launch_pdl(candidate_rank_kernel<G, true>, dim3(M), dim3(kRankThreads), smem, st, out, table, (long long)V, d,       \
                 (const long long*)cand, n_cand, kmax, hash_size, (int*)rec, scores, (int*)counts);                         \
    } else {                                                                                                                 \
      cudaError_t e = cudaFuncSetAttribute(candidate_rank_kernel<G, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
      if (e != cudaSuccess) { set_error("candidate_rank: smem attr: %s", cudaGetErrorString(e)); return ACSR_ERR_CUDA; }    \
      launch_pdl(candidate_rank_kernel<G, false>, dim3(M), dim3(kRankThreads), smem, st, out, table, (long long)V, d,      \
                 (const long long*)cand, n_cand, kmax, hash_size, (int*)rec, scores, (int*)nullptr);                        \
    }                                                                                                                        \
  } while (0)
  if (d4 > 16) ACSR_RANK_LAUNCH(32);
  else if (d4 > 8) ACSR_RANK_LAUNCH(16);
  else if (d4 > 4) ACSR_RANK_LAUNCH(8);
  else ACSR_RANK_LAUNCH(4);
#undef ACSR_RANK_LAUNCH
  return check_launch("candidate_rank");
}

int acsr_candidate_rank(const float* out, const float* table, int64_t V, int d, const int64_t* cand, int M, int n_cand, int kmax,
                        int32_t* rec, float* scores, void* stream) {
  return candidate_rank_impl(out, table, V, d, cand, M, n_cand, kmax, rec, scores, nullptr, stream);
}

int acsr_candidate_rank_counts(const float* out, const float* table, int64_t V, int d, const int64_t* cand, int M, int n_cand, int kmax,
                               int32_t* rec, float* scores, int32_t* counts, void* stream) {
  ACSR_REQUIRE(counts, "candidate_rank_counts: NULL counts");
  return candidate_rank_impl(out, table, V, d, cand, M, n_cand, kmax, rec, scores, counts, stream);
}

}  // extern "C"
