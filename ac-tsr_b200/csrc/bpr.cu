// loss_type BPR (acsasrec.py:109-116, recbole/model/loss.py:21-47):
//   x_m = out_m . (E[pos_m] - E[neg_m]) ;  loss = mean_m -log(gamma + sigmoid(x_m))
// forward and backward as two warp-per-row kernels; both the attacked and the calibrated rows ([2B, d], two groups)
// go through one launch.  The table gradient is a scatter of +-g_m * out_m into the rows pos_m / neg_m (atomics).
// Over a vocab-sharded table (dist.VocabParallel) every rank runs the shard kernels on all ranks' rows: the dot partials of the
// ids it owns (bpr_fwd_kernel's arithmetic, 0 elsewhere, so the sum over ranks is the unsharded (s_pos, s_neg) bit for bit), the
// loss from the summed dots, and a backward whose d_out and table gradient touch only the owned rows.
#include "acsr_common.cuh"
#include "../../include/acsr.h"

namespace acsr {

__global__ void __launch_bounds__(256) bpr_fwd_kernel(const float* __restrict__ out, const float* __restrict__ table,
                                                      const long long* __restrict__ pos, const long long* __restrict__ neg, int M, int d,
                                                      float gamma, float* __restrict__ row_x, float* __restrict__ row_loss) {
  pdl_launch_dependents();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * (blockDim.x >> 5) + warp;
  if (m >= M) return;
  const float* o = out + (long long)m * d;
  const float* ep = table + pos[m] * d;
  const float* en = table + neg[m] * d;
  float sp = 0.f, sn = 0.f;                       // the reference forms the two scores separately, then subtracts
  for (int j = lane; j < d; j += 32) {
    const float v = o[j];
    sp = fmaf(v, ep[j], sp);
    sn = fmaf(v, en[j], sn);
  }
  sp = warp_sum(sp);
  sn = warp_sum(sn);
  if (lane == 0) {
    const float x = sp - sn;
    row_x[m] = x;
    row_loss[m] = -logf(gamma + sigmoidf_(x));
  }
}

__global__ void __launch_bounds__(256) bpr_mean_kernel(const float* __restrict__ row_loss, int M, int n_groups, float* __restrict__ loss) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ double red[8];
  const int per_group = M / n_groups;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int g = 0; g < n_groups; ++g) {            // fixed summation order: deterministic
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

__global__ void __launch_bounds__(256) bpr_bwd_kernel(const float* __restrict__ out, const float* __restrict__ table,
                                                      const long long* __restrict__ pos, const long long* __restrict__ neg,
                                                      const float* __restrict__ row_x, const float* __restrict__ row_scale, int M, int d,
                                                      float gamma, int table_row_begin, int table_row_end, float* __restrict__ d_out,
                                                      float* __restrict__ d_table) {
  pdl_launch_dependents();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * (blockDim.x >> 5) + warp;
  if (m >= M) return;
  const float s = sigmoidf_(row_x[m]);
  const float g = -row_scale[m] * s * (1.0f - s) / (gamma + s);      // d loss / d x, scaled by the row's cotangent
  const long long ip = pos[m], in = neg[m];
  const float* o = out + (long long)m * d;
  const float* ep = table + ip * d;
  const float* en = table + in * d;
  const bool to_table = d_table != nullptr && m >= table_row_begin && m < table_row_end;
  for (int j = lane; j < d; j += 32) {
    if (d_out != nullptr) d_out[(long long)m * d + j] = g * (ep[j] - en[j]);
    if (to_table) {
      const float v = g * o[j];
      atomicAdd(d_table + ip * d + j, v);
      atomicAdd(d_table + in * d + j, -v);
    }
  }
}

// dots[m] = (out_m . E[pos_m], out_m . E[neg_m]) with E[i] = shard[i - lo] for owned ids i in [lo, hi), 0 for the others
__global__ void __launch_bounds__(256) bpr_dots_shard_kernel(const float* __restrict__ out, const float* __restrict__ shard,
                                                             long long lo, long long hi, const long long* __restrict__ pos,
                                                             const long long* __restrict__ neg, int M, int d,
                                                             float* __restrict__ dots) {
  pdl_launch_dependents();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * (blockDim.x >> 5) + warp;
  if (m >= M) return;
  const long long ip = pos[m], in = neg[m];
  const bool op = ip >= lo && ip < hi, on = in >= lo && in < hi;
  const float* o = out + (long long)m * d;
  const float* ep = shard + (op ? ip - lo : 0) * d;
  const float* en = shard + (on ? in - lo : 0) * d;
  float sp = 0.f, sn = 0.f;
  for (int j = lane; j < d; j += 32) {
    const float v = o[j];
    if (op) sp = fmaf(v, ep[j], sp);
    if (on) sn = fmaf(v, en[j], sn);
  }
  sp = warp_sum(sp);
  sn = warp_sum(sn);
  if (lane == 0) {
    dots[2 * m] = sp;
    dots[2 * m + 1] = sn;
  }
}

__global__ void __launch_bounds__(256) bpr_rows_from_dots_kernel(const float* __restrict__ dots, int M, float gamma,
                                                                 float* __restrict__ row_x, float* __restrict__ row_loss) {
  pdl_launch_dependents();
  pdl_wait();
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  const float x = dots[2 * m] - dots[2 * m + 1];
  row_x[m] = x;
  row_loss[m] = -logf(gamma + sigmoidf_(x));
}

// bpr_bwd_kernel over owned ids: d_out[m] = g * (E[pos] - E[neg]) with an unowned row read as 0 (g * (ep - en) when this rank
// owns both), and +-g * out_m into the shard gradient rows of owned ids
__global__ void __launch_bounds__(256) bpr_bwd_shard_kernel(const float* __restrict__ out, const float* __restrict__ shard,
                                                            long long lo, long long hi, const long long* __restrict__ pos,
                                                            const long long* __restrict__ neg, const float* __restrict__ row_x,
                                                            const float* __restrict__ row_scale, int M, int d, float gamma,
                                                            int table_row_begin, int table_row_end, float* __restrict__ d_out,
                                                            float* __restrict__ d_shard) {
  pdl_launch_dependents();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * (blockDim.x >> 5) + warp;
  if (m >= M) return;
  const float s = sigmoidf_(row_x[m]);
  const float g = -row_scale[m] * s * (1.0f - s) / (gamma + s);
  const long long ip = pos[m], in = neg[m];
  const bool op = ip >= lo && ip < hi, on = in >= lo && in < hi;
  const float* o = out + (long long)m * d;
  const float* ep = shard + (op ? ip - lo : 0) * d;
  const float* en = shard + (on ? in - lo : 0) * d;
  const bool to_table = d_shard != nullptr && m >= table_row_begin && m < table_row_end;
  for (int j = lane; j < d; j += 32) {
    if (d_out != nullptr) d_out[(long long)m * d + j] = g * ((op ? ep[j] : 0.f) - (on ? en[j] : 0.f));
    if (to_table) {
      const float v = g * o[j];
      if (op) atomicAdd(d_shard + (ip - lo) * d + j, v);
      if (on) atomicAdd(d_shard + (in - lo) * d + j, -v);
    }
  }
}

}  // namespace acsr

using namespace acsr;

extern "C" {

int acsr_bpr_loss_fwd(const float* out, const float* table, const int64_t* pos_items, const int64_t* neg_items, int M, int d,
                      int n_groups, float gamma, float* row_x, float* row_loss, float* loss, void* stream) {
  ACSR_REQUIRE(out && table && pos_items && neg_items && row_x && row_loss && loss, "bpr_loss_fwd: NULL pointer");
  ACSR_REQUIRE(M > 0 && d > 0 && n_groups > 0 && n_groups <= 8 && M % n_groups == 0, "bpr_loss_fwd: bad sizes");
  launch_pdl(bpr_fwd_kernel, dim3((M + 7) / 8), dim3(256), 0, (cudaStream_t)stream, out, table, (const long long*)pos_items,
             (const long long*)neg_items, M, d, gamma, row_x, row_loss);
  launch_pdl(bpr_mean_kernel, dim3(1), dim3(256), 0, (cudaStream_t)stream, (const float*)row_loss, M, n_groups, loss);
  return check_launch("bpr_loss_fwd");
}

int acsr_bpr_loss_bwd(const float* out, const float* table, const int64_t* pos_items, const int64_t* neg_items, const float* row_x,
                      const float* row_scale, int M, int d, float gamma, int table_row_begin, int table_row_end, float* d_out,
                      float* d_table, void* stream) {
  ACSR_REQUIRE(out && table && pos_items && neg_items && row_x && row_scale, "bpr_loss_bwd: NULL pointer");
  ACSR_REQUIRE(M > 0 && d > 0 && (d_out != nullptr || d_table != nullptr), "bpr_loss_bwd: bad arguments");
  launch_pdl(bpr_bwd_kernel, dim3((M + 7) / 8), dim3(256), 0, (cudaStream_t)stream, out, table, (const long long*)pos_items,
             (const long long*)neg_items, row_x, row_scale, M, d, gamma, table_row_begin, table_row_end, d_out, d_table);
  return check_launch("bpr_loss_bwd");
}

#define ACSR_SHARD_RANGE_OK(who)                                                                                          \
  ACSR_REQUIRE(lo >= 0 && lo < hi && hi <= V, who ": rows [%lld, %lld) not a non-empty range of [0, %lld)", (long long)lo, \
               (long long)hi, (long long)V)

int acsr_bpr_dots_shard(const float* out, const float* shard, int64_t lo, int64_t hi, int64_t V, const int64_t* pos_items,
                        const int64_t* neg_items, int M, int d, float* dots, void* stream) {
  ACSR_REQUIRE(out && shard && pos_items && neg_items && dots, "bpr_dots_shard: NULL pointer");
  ACSR_REQUIRE(M > 0 && d > 0, "bpr_dots_shard: bad sizes (M=%d d=%d)", M, d);
  ACSR_SHARD_RANGE_OK("bpr_dots_shard");
  launch_pdl(bpr_dots_shard_kernel, dim3((M + 7) / 8), dim3(256), 0, (cudaStream_t)stream, out, shard, (long long)lo, (long long)hi,
             (const long long*)pos_items, (const long long*)neg_items, M, d, dots);
  return check_launch("bpr_dots_shard");
}

int acsr_bpr_loss_from_dots(const float* dots, int M, int n_groups, float gamma, float* row_x, float* row_loss, float* loss,
                            void* stream) {
  ACSR_REQUIRE(dots && row_x && row_loss && loss, "bpr_loss_from_dots: NULL pointer");
  ACSR_REQUIRE(M > 0 && n_groups > 0 && n_groups <= 8 && M % n_groups == 0, "bpr_loss_from_dots: bad sizes");
  launch_pdl(bpr_rows_from_dots_kernel, dim3((M + 255) / 256), dim3(256), 0, (cudaStream_t)stream, dots, M, gamma, row_x, row_loss);
  launch_pdl(bpr_mean_kernel, dim3(1), dim3(256), 0, (cudaStream_t)stream, (const float*)row_loss, M, n_groups, loss);
  return check_launch("bpr_loss_from_dots");
}

int acsr_bpr_loss_bwd_shard(const float* out, const float* shard, int64_t lo, int64_t hi, int64_t V, const int64_t* pos_items,
                            const int64_t* neg_items, const float* row_x, const float* row_scale, int M, int d, float gamma,
                            int table_row_begin, int table_row_end, float* d_out, float* d_shard_grad, void* stream) {
  ACSR_REQUIRE(out && shard && pos_items && neg_items && row_x && row_scale, "bpr_loss_bwd_shard: NULL pointer");
  ACSR_REQUIRE(M > 0 && d > 0 && (d_out != nullptr || d_shard_grad != nullptr), "bpr_loss_bwd_shard: bad arguments");
  ACSR_SHARD_RANGE_OK("bpr_loss_bwd_shard");
  launch_pdl(bpr_bwd_shard_kernel, dim3((M + 7) / 8), dim3(256), 0, (cudaStream_t)stream, out, shard, (long long)lo, (long long)hi,
             (const long long*)pos_items, (const long long*)neg_items, row_x, row_scale, M, d, gamma, table_row_begin, table_row_end,
             d_out, d_shard_grad);
  return check_launch("bpr_loss_bwd_shard");
}

#undef ACSR_SHARD_RANGE_OK

}  // extern "C"
