// Gradient clipping by global norm (torch.nn.utils.clip_grad_norm_) over the flat gradient buffer: the partial sum of |g|^q
// (or max |g| for q = inf) of one or more ranges of the buffer, in fp64.  The clip itself is applied by acsr_adam_step_clipped
// (rowwise.cu), which combines the partials of this kernel -- one per launch, and one per rank of a sharded item table -- in a
// fixed order, so the coefficient costs no launch of its own and is the same on every rank.
#include "acsr_common.cuh"
#include "../../include/acsr.h"

namespace acsr {

constexpr int kNormThreads = 256;
constexpr int kNormMaxBlocks = kNumSMs * 4;       // persistent grid; also the length of the caller's block_partials scratch
constexpr int kNormMaxRanges = 8;

enum NormKind { kNormL1 = 0, kNormL2 = 1, kNormLp = 2, kNormInf = 3 };

struct NormRanges {                                // passed by value: the launch (and a captured graph node) owns the copy
  long long begin[kNormMaxRanges];
  long long end[kNormMaxRanges];
  int n;
};

// max that propagates NaN (fmax would drop it): torch's inf-norm of a buffer holding a NaN is NaN
__device__ __forceinline__ double nan_max(double a, double b) { return (b > a || b != b) ? b : a; }

template <int K>
__device__ __forceinline__ double norm_combine(double a, double b) { return K == kNormInf ? nan_max(a, b) : a + b; }

template <int K>
__device__ __forceinline__ double norm_term(double acc, float x, double q) {
  const double a = fabs((double)x);
  if (K == kNormL1) return acc + a;
  if (K == kNormL2) return fma(a, a, acc);
  if (K == kNormLp) return acc + pow(a, q);
  return nan_max(acc, a);
}

// fixed-order block reduction (butterfly per warp, then the warps' results in warp order); the result is valid in thread 0
template <int K>
__device__ __forceinline__ double block_combine(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = norm_combine<K>(v, __shfl_xor_sync(0xffffffffu, v, o));
  const int warp = threadIdx.x >> 5;
  __syncthreads();                                 // red may still be read by an earlier call
  if ((threadIdx.x & 31) == 0) red[warp] = v;
  __syncthreads();
  if (threadIdx.x == 0)
    for (int w = 1; w < kNormThreads / 32; ++w) v = norm_combine<K>(v, red[w]);
  return v;
}

template <int K>
__global__ void __launch_bounds__(kNormThreads) grad_norm_partial_kernel(const float* __restrict__ grad, NormRanges rg, double q,
                                                                         double* block_partials, unsigned int* counter,
                                                                         double* __restrict__ out) {
  pdl_wait();
  __shared__ double red[kNormThreads / 32];
  __shared__ bool s_last;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  double acc = 0.0;
  for (int r = 0; r < rg.n; ++r) {
    const float* p = grad + rg.begin[r];
    const long long len = rg.end[r] - rg.begin[r];
    long long head = (long long)(((16u - ((uintptr_t)p & 15u)) & 15u) >> 2);     // scalars before the first 16-byte boundary
    head = head < len ? head : len;
    const long long nv = (len - head) >> 2;
    const long long tail = head + 4 * nv;
    if (tid < head) acc = norm_term<K>(acc, p[tid], q);
    const float4* v = reinterpret_cast<const float4*>(p + head);
    for (long long i = tid; i < nv; i += stride) {
      const float4 x = v[i];
      acc = norm_term<K>(acc, x.x, q);
      acc = norm_term<K>(acc, x.y, q);
      acc = norm_term<K>(acc, x.z, q);
      acc = norm_term<K>(acc, x.w, q);
    }
    if (tid < len - tail) acc = norm_term<K>(acc, p[tail + tid], q);
  }
  acc = block_combine<K>(acc, red);
  if (threadIdx.x == 0) block_partials[blockIdx.x] = acc;
  __threadfence();                                 // this CTA's partial is visible device-wide before it checks in
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(counter, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  // the last CTA combines the per-CTA partials: thread t takes CTAs t, t + 256, ... in order, then the fixed block reduction --
  // the same order on every launch of the same sizes, so the result is bit-identical from run to run and under graph replay
  const volatile double* bp = block_partials;
  double s = 0.0;
  for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) s = norm_combine<K>(s, bp[i]);
  s = block_combine<K>(s, red);
  if (threadIdx.x == 0) {
    out[0] = s;
    *counter = 0u;                                 // ready for the next launch (graph replays included)
  }
}

}  // namespace acsr

using namespace acsr;

extern "C" {

int acsr_grad_norm_max_blocks(void) { return kNormMaxBlocks; }

int acsr_grad_norm_partial(const float* grad, int64_t n, const int64_t* ranges, int n_ranges, double norm_type,
                           double* block_partials, uint32_t* counter, double* out, void* stream) {
  ACSR_REQUIRE(grad && ranges && block_partials && counter && out, "grad_norm_partial: NULL pointer");
  ACSR_REQUIRE(n >= 0, "grad_norm_partial: n=%lld", (long long)n);
  ACSR_REQUIRE(n_ranges >= 1 && n_ranges <= kNormMaxRanges, "grad_norm_partial: n_ranges=%d (need 1..%d)", n_ranges, kNormMaxRanges);
  ACSR_REQUIRE(norm_type > 0.0, "grad_norm_partial: norm_type=%f (need a positive number or inf)", norm_type);
  NormRanges rg = {};
  rg.n = n_ranges;
  long long nv = 0;
  for (int r = 0; r < n_ranges; ++r) {
    ACSR_REQUIRE(ranges[2 * r] >= 0 && ranges[2 * r + 1] >= ranges[2 * r] && ranges[2 * r + 1] <= n,
                 "grad_norm_partial: range %d is [%lld, %lld) of %lld elements", r, (long long)ranges[2 * r],
                 (long long)ranges[2 * r + 1], (long long)n);
    rg.begin[r] = ranges[2 * r];
    rg.end[r] = ranges[2 * r + 1];
    nv += (rg.end[r] - rg.begin[r] + 3) / 4;
  }
  const long long need = (nv + kNormThreads - 1) / kNormThreads;
  const int grid = (int)(need < kNormMaxBlocks ? (need > 0 ? need : 1) : kNormMaxBlocks);
  const int kind = isinf(norm_type) ? kNormInf : norm_type == 1.0 ? kNormL1 : norm_type == 2.0 ? kNormL2 : kNormLp;
  const cudaStream_t st = (cudaStream_t)stream;
  unsigned int* cnt = (unsigned int*)counter;
  switch (kind) {
    case kNormL1: launch_pdl(grad_norm_partial_kernel<kNormL1>, dim3(grid), dim3(kNormThreads), 0, st, grad, rg, norm_type, block_partials, cnt, out); break;
    case kNormL2: launch_pdl(grad_norm_partial_kernel<kNormL2>, dim3(grid), dim3(kNormThreads), 0, st, grad, rg, norm_type, block_partials, cnt, out); break;
    case kNormLp: launch_pdl(grad_norm_partial_kernel<kNormLp>, dim3(grid), dim3(kNormThreads), 0, st, grad, rg, norm_type, block_partials, cnt, out); break;
    default: launch_pdl(grad_norm_partial_kernel<kNormInf>, dim3(grid), dim3(kNormThreads), 0, st, grad, rg, norm_type, block_partials, cnt, out); break;
  }
  return check_launch("grad_norm_partial");
}

}  // extern "C"
