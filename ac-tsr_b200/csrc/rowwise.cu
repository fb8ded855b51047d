// Memory-bound row-wise kernels: K1 (gather + pos + LayerNorm + dropout), the
// bias+dropout+residual+LayerNorm epilogue, bias+activation, last-position gather, fused Adam (optionally with the
// gradient clipped by global norm).
// One warp owns one token row; every lane reads/writes 16-byte (or 8-byte at d=64) vectors so a
// warp touches whole 128-byte lines; grids are persistent (a multiple of the 148 SMs) and
// grid-stride over rows so LayerNorm weight/bias gradients are reduced in registers first.
#include <type_traits>
#include "acsr_common.cuh"
#include "../../include/acsr.h"

namespace acsr {

constexpr int kWarpsPerBlock = 8;
constexpr int kRowBlocksPerSM = 4;

template <int D>
struct RowVec {
  static constexpr int VPT = D / 32;                 // elements per lane
  static constexpr int VEC = VPT >= 4 ? 4 : VPT;     // vector width of one access
  static constexpr int NCH = VPT / VEC;              // accesses per lane
  __device__ static __forceinline__ int col(int c, int lane, int v) { return c * 32 * VEC + lane * VEC + v; }

  __device__ static __forceinline__ void load(const float* __restrict__ row, int lane, float* x) {
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const float* p = row + col(c, lane, 0);
      if (VEC == 4) {
        float4 t = *reinterpret_cast<const float4*>(p);
        x[c * 4 + 0] = t.x; x[c * 4 + 1] = t.y; x[c * 4 + 2] = t.z; x[c * 4 + 3] = t.w;
      } else if (VEC == 2) {
        float2 t = *reinterpret_cast<const float2*>(p);
        x[c * 2 + 0] = t.x; x[c * 2 + 1] = t.y;
      } else {
        x[c] = p[0];
      }
    }
  }
  __device__ static __forceinline__ void store(float* __restrict__ row, int lane, const float* x) {
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      float* p = row + col(c, lane, 0);
      if (VEC == 4) {
        *reinterpret_cast<float4*>(p) = make_float4(x[c * 4 + 0], x[c * 4 + 1], x[c * 4 + 2], x[c * 4 + 3]);
      } else if (VEC == 2) {
        *reinterpret_cast<float2*>(p) = make_float2(x[c * 2 + 0], x[c * 2 + 1]);
      } else {
        p[0] = x[c];
      }
    }
  }
  // multiplicative dropout mask for this lane's elements of row `row_idx`
  __device__ static __forceinline__ void dropmask(float p, const float* __restrict__ mask, const RngState* rng,
                                                  uint32_t stream, long long row_idx, int lane, float* m) {
    if (mask != nullptr) {
      load(mask + row_idx * D, lane, m);
      return;
    }
    if (p <= 0.0f || rng == nullptr) {
#pragma unroll
      for (int i = 0; i < VPT; ++i) m[i] = 1.0f;
      return;
    }
    const float inv_keep = 1.0f / (1.0f - p);
    const unsigned long long seed = rng->seed, step = rng->step;
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      unsigned long long e = (unsigned long long)row_idx * D + col(c, lane, 0);
      uint4 r = philox4x32(seed, step, stream, e >> 2);
      uint32_t bits[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
      for (int v = 0; v < VEC; ++v) m[c * VEC + v] = drop_mult(bits[(e + v) & 3], p, inv_keep);
    }
  }
};

template <int D>
__device__ __forceinline__ void ln_stats(const float* x, float& mean, float& rstd, float eps) {
  constexpr int VPT = D / 32;
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < VPT; ++i) s += x[i];
  mean = warp_sum(s) * (1.0f / D);
  float v = 0.f;
#pragma unroll
  for (int i = 0; i < VPT; ++i) { float t = x[i] - mean; v += t * t; }
  v = warp_sum(v) * (1.0f / D);
  rstd = 1.0f / sqrtf(v + eps);
}

// reduce per-lane column partials across the warps of a block, then one atomic per column per block
template <int D, int NACC>
__device__ __forceinline__ void block_col_reduce(float (*acc)[D / 32], float* const* dst, float* smem) {
  using RV = RowVec<D>;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int a = 0; a < NACC; ++a) {
    if (dst[a] == nullptr) continue;
    __syncthreads();
#pragma unroll
    for (int c = 0; c < RV::NCH; ++c)
#pragma unroll
      for (int v = 0; v < RV::VEC; ++v) smem[warp * D + RV::col(c, lane, v)] = acc[a][c * RV::VEC + v];
    __syncthreads();
    for (int j = threadIdx.x; j < D; j += blockDim.x) {
      float s = 0.f;
      for (int w = 0; w < kWarpsPerBlock; ++w) s += smem[w * D + j];
      atomicAdd(dst[a] + j, s);
    }
  }
}

// ------------------------------------------------------------------------------------------
// K1 forward / backward
// ------------------------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
embed_ln_fwd_kernel(const int64_t* __restrict__ item_seq, const float* __restrict__ table, const float* __restrict__ pos_emb,
                    const float* __restrict__ ln_w, const float* __restrict__ ln_b, float eps, int T, int L, long long V,
                    float p, const float* __restrict__ mask, const RngState* rng, uint32_t stream,
                    float* __restrict__ out, float* __restrict__ stats) {
  pdl_launch_dependents();
  pdl_wait();
  using RV = RowVec<D>;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float w[RV::VPT], b[RV::VPT];
  RV::load(ln_w, lane, w);
  RV::load(ln_b, lane, b);
  for (long long t = (long long)blockIdx.x * kWarpsPerBlock + warp; t < T; t += (long long)gridDim.x * kWarpsPerBlock) {
    int64_t idx = item_seq[t];
    if (idx < 0 || idx >= V) idx = 0;       // an id outside the table reads (and trains) nothing: treated as padding, never out of bounds
    float x[RV::VPT], m[RV::VPT];
    RV::load(table + idx * D, lane, x);
    if (pos_emb != nullptr) {
      float pe[RV::VPT];
      RV::load(pos_emb + (t % L) * D, lane, pe);
#pragma unroll
      for (int i = 0; i < RV::VPT; ++i) x[i] += pe[i];
    }
    float mean, rstd;
    ln_stats<D>(x, mean, rstd, eps);
    RV::dropmask(p, mask, rng, stream, t, lane, m);
#pragma unroll
    for (int i = 0; i < RV::VPT; ++i) x[i] = ((x[i] - mean) * rstd * w[i] + b[i]) * m[i];
    RV::store(out + t * D, lane, x);
    if (lane == 0) { stats[2 * t] = mean; stats[2 * t + 1] = rstd; }
  }
}

template <int D>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
embed_ln_bwd_kernel(const float* __restrict__ d_out, const int64_t* __restrict__ item_seq, const float* __restrict__ table,
                    const float* __restrict__ pos_emb, const float* __restrict__ ln_w, const float* __restrict__ stats,
                    int T, int L, long long V, float p, const float* __restrict__ mask, const RngState* rng, uint32_t stream,
                    float* __restrict__ d_table, float* __restrict__ d_pos, float* __restrict__ d_ln_w, float* __restrict__ d_ln_b) {
  pdl_launch_dependents();
  pdl_wait();
  using RV = RowVec<D>;
  __shared__ float red[kWarpsPerBlock * D];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float w[RV::VPT];
  RV::load(ln_w, lane, w);
  float acc[2][RV::VPT];
#pragma unroll
  for (int i = 0; i < RV::VPT; ++i) acc[0][i] = acc[1][i] = 0.f;
  for (long long t = (long long)blockIdx.x * kWarpsPerBlock + warp; t < T; t += (long long)gridDim.x * kWarpsPerBlock) {
    int64_t idx = item_seq[t];
    if (idx < 0 || idx >= V) idx = 0;       // an id outside the table reads (and trains) nothing: treated as padding, never out of bounds
    float x[RV::VPT], g[RV::VPT], m[RV::VPT];
    RV::load(table + idx * D, lane, x);
    if (pos_emb != nullptr) {
      float pe[RV::VPT];
      RV::load(pos_emb + (t % L) * D, lane, pe);
#pragma unroll
      for (int i = 0; i < RV::VPT; ++i) x[i] += pe[i];
    }
    const float mean = stats[2 * t], rstd = stats[2 * t + 1];
    RV::load(d_out + t * D, lane, g);
    RV::dropmask(p, mask, rng, stream, t, lane, m);
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < RV::VPT; ++i) {
      x[i] = (x[i] - mean) * rstd;          // xhat
      g[i] *= m[i];                         // grad wrt LN output
      acc[0][i] += g[i] * x[i];
      acc[1][i] += g[i];
      g[i] *= w[i];                         // grad wrt xhat
      s1 += g[i];
      s2 += g[i] * x[i];
    }
    s1 = warp_sum(s1) * (1.0f / D);
    s2 = warp_sum(s2) * (1.0f / D);
#pragma unroll
    for (int i = 0; i < RV::VPT; ++i) g[i] = rstd * (g[i] - s1 - x[i] * s2);
    if (idx != 0) {                         // nn.Embedding(padding_idx=0): no gradient through the gather of row 0
#pragma unroll
      for (int c = 0; c < RV::NCH; ++c)
#pragma unroll
        for (int v = 0; v < RV::VEC; ++v) atomicAdd(d_table + idx * D + RV::col(c, lane, v), g[c * RV::VEC + v]);
    }
    if (d_pos != nullptr) {
#pragma unroll
      for (int c = 0; c < RV::NCH; ++c)
#pragma unroll
        for (int v = 0; v < RV::VEC; ++v) atomicAdd(d_pos + (t % L) * D + RV::col(c, lane, v), g[c * RV::VEC + v]);
    }
  }
  float* dst[2] = {d_ln_w, d_ln_b};
  block_col_reduce<D, 2>(acc, dst, red);
}

// ------------------------------------------------------------------------------------------
// LN(dropout(h + bias) + res)
// ------------------------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
bdrl_fwd_kernel(const float* __restrict__ h, const float* __restrict__ bias, const float* __restrict__ res,
                const float* __restrict__ ln_w, const float* __restrict__ ln_b, float eps, int T, int res_rows,
                float p, const float* __restrict__ mask, const RngState* rng, uint32_t stream,
                float* __restrict__ out, float* __restrict__ stats) {
  pdl_launch_dependents();
  pdl_wait();
  using RV = RowVec<D>;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float w[RV::VPT], b[RV::VPT], bi[RV::VPT];
  RV::load(ln_w, lane, w);
  RV::load(ln_b, lane, b);
  if (bias != nullptr) RV::load(bias, lane, bi);
  else {
#pragma unroll
    for (int i = 0; i < RV::VPT; ++i) bi[i] = 0.f;
  }
  for (long long t = (long long)blockIdx.x * kWarpsPerBlock + warp; t < T; t += (long long)gridDim.x * kWarpsPerBlock) {
    float x[RV::VPT], r[RV::VPT], m[RV::VPT];
    RV::load(h + t * D, lane, x);
    RV::load(res + (t % res_rows) * D, lane, r);
    RV::dropmask(p, mask, rng, stream, t, lane, m);
#pragma unroll
    for (int i = 0; i < RV::VPT; ++i) x[i] = (x[i] + bi[i]) * m[i] + r[i];
    float mean, rstd;
    ln_stats<D>(x, mean, rstd, eps);
#pragma unroll
    for (int i = 0; i < RV::VPT; ++i) x[i] = (x[i] - mean) * rstd * w[i] + b[i];
    RV::store(out + t * D, lane, x);
    if (lane == 0) { stats[2 * t] = mean; stats[2 * t + 1] = rstd; }
  }
}

template <int D>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
bdrl_bwd_kernel(const float* __restrict__ d_out, const float* __restrict__ h, const float* __restrict__ bias,
                const float* __restrict__ res, const float* __restrict__ ln_w, const float* __restrict__ stats, int T,
                int act_rows, int res_rows, int param_rows,
                float p, const float* __restrict__ mask, const RngState* rng, uint32_t stream,
                float* __restrict__ d_h, float* __restrict__ d_res, float* __restrict__ d_bias,
                float* __restrict__ d_ln_w, float* __restrict__ d_ln_b) {
  pdl_launch_dependents();
  pdl_wait();
  using RV = RowVec<D>;
  __shared__ float red[kWarpsPerBlock * D];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float w[RV::VPT], bi[RV::VPT];
  RV::load(ln_w, lane, w);
  if (bias != nullptr) RV::load(bias, lane, bi);
  else {
#pragma unroll
    for (int i = 0; i < RV::VPT; ++i) bi[i] = 0.f;
  }
  float acc[3][RV::VPT];
#pragma unroll
  for (int i = 0; i < RV::VPT; ++i) acc[0][i] = acc[1][i] = acc[2][i] = 0.f;
  for (long long t = (long long)blockIdx.x * kWarpsPerBlock + warp; t < T; t += (long long)gridDim.x * kWarpsPerBlock) {
    float x[RV::VPT], r[RV::VPT], m[RV::VPT], g[RV::VPT];
    // saved forward tensors repeat with period act_rows (both cotangent streams of a shared activation)
    const long long ta = t % act_rows;
    const float keep = t < param_rows ? 1.0f : 0.0f;       // only these rows feed the parameter gradients
    RV::load(h + ta * D, lane, x);
    RV::load(res + (t % res_rows) * D, lane, r);
    RV::load(d_out + t * D, lane, g);
    RV::dropmask(p, mask, rng, stream, ta, lane, m);
    const float mean = stats[2 * ta], rstd = stats[2 * ta + 1];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < RV::VPT; ++i) {
      x[i] = ((x[i] + bi[i]) * m[i] + r[i] - mean) * rstd;   // xhat
      acc[0][i] += keep * g[i] * x[i];
      acc[1][i] += keep * g[i];
      g[i] *= w[i];
      s1 += g[i];
      s2 += g[i] * x[i];
    }
    s1 = warp_sum(s1) * (1.0f / D);
    s2 = warp_sum(s2) * (1.0f / D);
#pragma unroll
    for (int i = 0; i < RV::VPT; ++i) {
      g[i] = rstd * (g[i] - s1 - x[i] * s2);   // grad wrt (dropout(h+bias) + res)
      r[i] = g[i] * m[i];                      // grad wrt h (and bias)
      acc[2][i] += keep * r[i];
    }
    RV::store(d_res + t * D, lane, g);
    RV::store(d_h + t * D, lane, r);
  }
  float* dst[3] = {d_ln_w, d_ln_b, d_bias};
  block_col_reduce<D, 3>(acc, dst, red);
}

// ------------------------------------------------------------------------------------------
// out = act(h + bias)   [T,n]; thread x-dim = float4 column group, y-dim = rows
// ------------------------------------------------------------------------------------------
constexpr int kActTX = 64, kActTY = 4, kActMaxK = 8;   // n <= 64*4*8 = 2048

__global__ void __launch_bounds__(kActTX * kActTY)
bias_act_fwd_kernel(const float4* __restrict__ h, const float4* __restrict__ bias, int T, int ncv, int act, float4* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  for (int cv = threadIdx.x; cv < ncv; cv += kActTX) {
    const float4 b = bias != nullptr ? bias[cv] : make_float4(0.f, 0.f, 0.f, 0.f);
    for (long long t = (long long)blockIdx.x * kActTY + threadIdx.y; t < T; t += (long long)gridDim.x * kActTY) {
      float4 x = h[t * ncv + cv];
      x.x = act_fwd(act, x.x + b.x); x.y = act_fwd(act, x.y + b.y);
      x.z = act_fwd(act, x.z + b.z); x.w = act_fwd(act, x.w + b.w);
      out[t * ncv + cv] = x;
    }
  }
}

__global__ void __launch_bounds__(kActTX * kActTY)
bias_act_bwd_kernel(const float4* __restrict__ d_out, const float4* __restrict__ h, const float4* __restrict__ bias,
                    int T, int ncv, int act, int act_rows, int param_rows, float4* __restrict__ d_h, float* __restrict__ d_bias) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float4 red[kActTY][kActTX];
  for (int cv0 = 0; cv0 < ncv; cv0 += kActTX) {      // uniform trip count across the block (syncthreads inside)
    const int cv = cv0 + threadIdx.x;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (cv < ncv) {
      const float4 b = bias != nullptr ? bias[cv] : make_float4(0.f, 0.f, 0.f, 0.f);
      for (long long t = (long long)blockIdx.x * kActTY + threadIdx.y; t < T; t += (long long)gridDim.x * kActTY) {
        float4 x = h[(t % act_rows) * ncv + cv];
        float4 g = d_out[t * ncv + cv];
        g.x *= act_bwd(act, x.x + b.x); g.y *= act_bwd(act, x.y + b.y);
        g.z *= act_bwd(act, x.z + b.z); g.w *= act_bwd(act, x.w + b.w);
        d_h[t * ncv + cv] = g;
        if (t < param_rows) { acc.x += g.x; acc.y += g.y; acc.z += g.z; acc.w += g.w; }
      }
    }
    red[threadIdx.y][threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.y == 0 && cv < ncv && d_bias != nullptr) {
      float4 s = red[0][threadIdx.x];
#pragma unroll
      for (int y = 1; y < kActTY; ++y) {
        float4 o = red[y][threadIdx.x];
        s.x += o.x; s.y += o.y; s.z += o.z; s.w += o.w;
      }
      atomicAdd(d_bias + 4 * cv + 0, s.x); atomicAdd(d_bias + 4 * cv + 1, s.y);
      atomicAdd(d_bias + 4 * cv + 2, s.z); atomicAdd(d_bias + 4 * cv + 3, s.w);
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// K9 gather of position len-1
// ------------------------------------------------------------------------------------------
__global__ void gather_last_fwd_kernel(const float* __restrict__ x_att, const float* __restrict__ x_cal,
                                       const int64_t* __restrict__ item_len, int B, int L, int d, float* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  const int row = blockIdx.x;                 // [0, 2B) or [0,B)
  const bool has_att = x_att != nullptr;
  const int b = has_att ? (row % B) : row;
  const float* src = (has_att && row < B) ? x_att : x_cal;
  const long long pos = item_len[b] - 1;
  for (int j = threadIdx.x; j < d; j += blockDim.x) out[(long long)row * d + j] = src[((long long)b * L + pos) * d + j];
}

__global__ void gather_last_bwd_kernel(const float* __restrict__ d_out, const int64_t* __restrict__ item_len, int B, int L, int d,
                                       float* __restrict__ d_x_att, float* __restrict__ d_x_cal) {
  pdl_launch_dependents();
  pdl_wait();
  const int row = blockIdx.x;
  const bool has_att = d_x_att != nullptr;
  const int b = has_att ? (row % B) : row;
  float* dst = (has_att && row < B) ? d_x_att : d_x_cal;
  const long long pos = item_len[b] - 1;
  for (int j = threadIdx.x; j < d; j += blockDim.x) dst[((long long)b * L + pos) * d + j] = d_out[(long long)row * d + j];
}

// ------------------------------------------------------------------------------------------
// fused Adam (torch.optim.Adam, amsgrad=False, maximize=False)
// kClip: torch.nn.utils.clip_grad_norm_ folded in.  Every CTA combines the norm partials of acsr_grad_norm_partial in index
// order (so every CTA, and every rank, derives the same coefficient), scales the gradient, writes the clipped gradient back
// (p.grad after clip_grad_norm_) and runs the same update on it.
// ------------------------------------------------------------------------------------------
template <bool kClip>
__global__ void adam_kernel(float* __restrict__ param, std::conditional_t<kClip, float, const float>* __restrict__ grad,
                            float* __restrict__ m, float* __restrict__ v, long long n, float lr, float b1, float b2, float eps,
                            float wd, const long long* __restrict__ step_count, const double* __restrict__ partials,
                            int n_partials, double norm_type, float max_norm, float* __restrict__ total_out) {
  // (no early programmatic-launch trigger: this kernel WRITES the parameters, which later kernels may read ahead of their
  // griddepcontrol.wait -- acsr_register_static -- so nothing that follows may start before it has completed)
  pdl_wait();
  float coef = 1.f;
  if constexpr (kClip) {
    __shared__ float s_coef;
    if (threadIdx.x == 0) {
      const bool inf_norm = isinf(norm_type);
      double s = partials[0];
      for (int i = 1; i < n_partials; ++i) {
        const double p = partials[i];
        s = inf_norm ? ((p > s || p != p) ? p : s) : s + p;         // the max keeps a NaN, as torch's inf-norm does
      }
      const float total = (float)(inf_norm || norm_type == 1.0 ? s : norm_type == 2.0 ? sqrt(s) : pow(s, 1.0 / norm_type));
      // torch: clamp(max_norm / (total + 1e-6), max=1), the division as reciprocal * max_norm; a NaN coefficient propagates
      const float c = (1.f / (total + 1e-6f)) * max_norm;
      s_coef = c > 1.f ? 1.f : c;
      if (blockIdx.x == 0) total_out[0] = total;
    }
    __syncthreads();
    coef = s_coef;
  }
  const double step = (double)(step_count[0] + 1);
  const float bc1 = (float)(1.0 - pow((double)b1, step));
  const float bc2_sqrt = (float)sqrt(1.0 - pow((double)b2, step));
  const float step_size = lr / bc1;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float g = grad[i], pm = param[i];
    if constexpr (kClip) {
      g *= coef;
      grad[i] = g;
    }
    if (wd != 0.f) g += wd * pm;
    float mi = b1 * m[i] + (1.f - b1) * g;
    float vi = b2 * v[i] + (1.f - b2) * g * g;
    m[i] = mi; v[i] = vi;
    param[i] = pm - step_size * mi / (sqrtf(vi) / bc2_sqrt + eps);
  }
}
__global__ void step_inc_kernel(long long* step_count) {
  pdl_launch_dependents();
  pdl_wait(); step_count[0] += 1; }

static int row_grid(long long T) {
  long long need = (T + kWarpsPerBlock - 1) / kWarpsPerBlock;
  long long cap = (long long)kNumSMs * kRowBlocksPerSM;
  return (int)(need < cap ? (need > 0 ? need : 1) : cap);
}

}  // namespace acsr

using namespace acsr;

#define DISPATCH_D(d, CALL)                                                        \
  switch (d) {                                                                     \
    case 32: { constexpr int D_ = 32; CALL; } break;                               \
    case 64: { constexpr int D_ = 64; CALL; } break;                               \
    case 128: { constexpr int D_ = 128; CALL; } break;                             \
    case 256: { constexpr int D_ = 256; CALL; } break;                             \
    default: set_error("hidden size %d unsupported (need 32/64/128/256)", d); return ACSR_ERR_UNSUPPORTED; \
  }

extern "C" {

int acsr_embed_ln_dropout_fwd(const int64_t* item_seq, const float* table, const float* pos_emb, const float* ln_w,
                              const float* ln_b, float eps, int T, int L, int d, int64_t V, float p, const float* mask,
                              const void* rng, uint32_t rng_stream, float* out, float* stats, void* stream) {
  ACSR_REQUIRE(item_seq && table && ln_w && ln_b && out && stats, "embed_ln_dropout_fwd: NULL pointer");
  ACSR_REQUIRE(T >= 0 && L > 0 && V > 0, "embed_ln_dropout_fwd: bad sizes T=%d L=%d", T, L);
  ACSR_REQUIRE(p >= 0.f && p < 1.f, "embed_ln_dropout_fwd: dropout p=%f", p);
  ACSR_REQUIRE(!(p > 0.f && mask == nullptr && rng == nullptr), "embed_ln_dropout_fwd: p>0 needs mask or rng");
  if (T == 0) return ACSR_OK;
  DISPATCH_D(d, (launch_pdl(embed_ln_fwd_kernel<D_>, dim3(row_grid(T)), dim3(kWarpsPerBlock * 32), 0, (cudaStream_t)stream, 
                    item_seq, table, pos_emb, ln_w, ln_b, eps, T, L, (long long)V, p, mask, (const RngState*)rng, rng_stream, out, stats)));
  return check_launch("embed_ln_dropout_fwd");
}

int acsr_embed_ln_dropout_bwd(const float* d_out, const int64_t* item_seq, const float* table, const float* pos_emb,
                              const float* ln_w, const float* stats, int T, int L, int d, int64_t V, float p, const float* mask,
                              const void* rng, uint32_t rng_stream, float* d_table, float* d_pos, float* d_ln_w, float* d_ln_b,
                              void* stream) {
  ACSR_REQUIRE(d_out && item_seq && table && ln_w && stats && d_table, "embed_ln_dropout_bwd: NULL pointer");
  ACSR_REQUIRE((pos_emb == nullptr) == (d_pos == nullptr), "embed_ln_dropout_bwd: pos_emb/d_pos mismatch");
  if (T == 0) return ACSR_OK;
  DISPATCH_D(d, (launch_pdl(embed_ln_bwd_kernel<D_>, dim3(row_grid(T)), dim3(kWarpsPerBlock * 32), 0, (cudaStream_t)stream, 
                    d_out, item_seq, table, pos_emb, ln_w, stats, T, L, (long long)V, p, mask, (const RngState*)rng, rng_stream, d_table,
                    d_pos, d_ln_w, d_ln_b)));
  return check_launch("embed_ln_dropout_bwd");
}

int acsr_bias_dropout_res_ln_fwd(const float* h, const float* bias, const float* res, const float* ln_w, const float* ln_b,
                                 float eps, int T, int d, int res_rows, float p, const float* mask, const void* rng,
                                 uint32_t rng_stream, float* out, float* stats, void* stream) {
  ACSR_REQUIRE(h && res && ln_w && ln_b && out && stats, "bias_dropout_res_ln_fwd: NULL pointer");
  ACSR_REQUIRE(res_rows > 0 && res_rows <= T || T == 0, "bias_dropout_res_ln_fwd: res_rows=%d", res_rows);
  ACSR_REQUIRE(p >= 0.f && p < 1.f, "bias_dropout_res_ln_fwd: dropout p=%f", p);
  ACSR_REQUIRE(!(p > 0.f && mask == nullptr && rng == nullptr), "bias_dropout_res_ln_fwd: p>0 needs mask or rng");
  if (T == 0) return ACSR_OK;
  DISPATCH_D(d, (launch_pdl(bdrl_fwd_kernel<D_>, dim3(row_grid(T)), dim3(kWarpsPerBlock * 32), 0, (cudaStream_t)stream, 
                    h, bias, res, ln_w, ln_b, eps, T, res_rows, p, mask, (const RngState*)rng, rng_stream, out, stats)));
  return check_launch("bias_dropout_res_ln_fwd");
}

int acsr_bias_dropout_res_ln_bwd(const float* d_out, const float* h, const float* bias, const float* res, const float* ln_w,
                                 const float* stats, int T, int d, int act_rows, int res_rows, int param_rows, float p,
                                 const float* mask, const void* rng, uint32_t rng_stream, float* d_h, float* d_res,
                                 float* d_bias, float* d_ln_w, float* d_ln_b, void* stream) {
  ACSR_REQUIRE(d_out && h && res && ln_w && stats && d_h && d_res, "bias_dropout_res_ln_bwd: NULL pointer");
  ACSR_REQUIRE(T == 0 || (act_rows > 0 && res_rows > 0 && param_rows >= 0), "bias_dropout_res_ln_bwd: bad row periods");
  if (T == 0) return ACSR_OK;
  DISPATCH_D(d, (launch_pdl(bdrl_bwd_kernel<D_>, dim3(row_grid(T)), dim3(kWarpsPerBlock * 32), 0, (cudaStream_t)stream, 
                    d_out, h, bias, res, ln_w, stats, T, act_rows, res_rows, param_rows, p, mask, (const RngState*)rng,
                    rng_stream, d_h, d_res, d_bias, d_ln_w, d_ln_b)));
  return check_launch("bias_dropout_res_ln_bwd");
}

int acsr_bias_act_fwd(const float* h, const float* bias, int T, int n, int act, float* out, void* stream) {
  ACSR_REQUIRE(h && out, "bias_act_fwd: NULL pointer");
  ACSR_REQUIRE(n % 4 == 0 && n > 0 && n <= kActTX * 4 * kActMaxK, "bias_act_fwd: n=%d must be a multiple of 4, <= 2048", n);
  ACSR_REQUIRE(act >= 0 && act <= 4, "bias_act_fwd: unknown activation %d", act);
  if (T == 0) return ACSR_OK;
  long long need = (T + kActTY - 1) / kActTY, cap = kNumSMs * 8;
  dim3 blk(kActTX, kActTY);
  launch_pdl(bias_act_fwd_kernel, dim3((int)(need < cap ? need : cap)), blk, 0, (cudaStream_t)stream, 
      (const float4*)h, (const float4*)bias, T, n / 4, act, (float4*)out);
  return check_launch("bias_act_fwd");
}

int acsr_bias_act_bwd(const float* d_out, const float* h, const float* bias, int T, int n, int act, int act_rows,
                      int param_rows, float* d_h, float* d_bias, void* stream) {
  ACSR_REQUIRE(d_out && h && d_h, "bias_act_bwd: NULL pointer");
  ACSR_REQUIRE(n % 4 == 0 && n > 0 && n <= kActTX * 4 * kActMaxK, "bias_act_bwd: n=%d must be a multiple of 4, <= 2048", n);
  ACSR_REQUIRE(act >= 0 && act <= 4, "bias_act_bwd: unknown activation %d", act);
  ACSR_REQUIRE(T == 0 || (act_rows > 0 && param_rows >= 0), "bias_act_bwd: bad row periods");
  if (T == 0) return ACSR_OK;
  long long need = (T + kActTY - 1) / kActTY, cap = kNumSMs * 4;
  dim3 blk(kActTX, kActTY);
  launch_pdl(bias_act_bwd_kernel, dim3((int)(need < cap ? need : cap)), blk, 0, (cudaStream_t)stream, 
      (const float4*)d_out, (const float4*)h, (const float4*)bias, T, n / 4, act, act_rows, param_rows, (float4*)d_h, d_bias);
  return check_launch("bias_act_bwd");
}

int acsr_gather_last_fwd(const float* x_att, const float* x_cal, const int64_t* item_len, int B, int L, int d, float* out,
                         void* stream) {
  ACSR_REQUIRE(x_cal && item_len && out, "gather_last_fwd: NULL pointer");
  if (B == 0) return ACSR_OK;
  launch_pdl(gather_last_fwd_kernel, dim3(x_att ? 2 * B : B), dim3(64), 0, (cudaStream_t)stream, x_att, x_cal, item_len, B, L, d, out);
  return check_launch("gather_last_fwd");
}

int acsr_gather_last_bwd(const float* d_out, const int64_t* item_len, int B, int L, int d, float* d_x_att, float* d_x_cal,
                         void* stream) {
  ACSR_REQUIRE(d_out && item_len && d_x_cal, "gather_last_bwd: NULL pointer");
  if (B == 0) return ACSR_OK;
  launch_pdl(gather_last_bwd_kernel, dim3(d_x_att ? 2 * B : B), dim3(64), 0, (cudaStream_t)stream, d_out, item_len, B, L, d, d_x_att, d_x_cal);
  return check_launch("gather_last_bwd");
}

int acsr_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                   float beta2, float eps, float weight_decay, int64_t* step_count, void* stream) {
  ACSR_REQUIRE(param && grad && exp_avg && exp_avg_sq && step_count, "adam_step: NULL pointer");
  if (n > 0) {
    long long need = (n + 255) / 256, cap = kNumSMs * 8;
    launch_pdl(adam_kernel<false>, dim3((int)(need < cap ? need : cap)), dim3(256), 0, (cudaStream_t)stream,
        param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay, (const long long*)step_count,
        (const double*)nullptr, 0, 0.0, 0.f, (float*)nullptr);
  }
  launch_pdl(step_inc_kernel, dim3(1), dim3(1), 0, (cudaStream_t)stream, (long long*)step_count);
  return check_launch("adam_step");
}

int acsr_adam_step_clipped(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                           float beta2, float eps, float weight_decay, int64_t* step_count, const double* partials, int n_partials,
                           double norm_type, float max_norm, float* total_out, void* stream) {
  ACSR_REQUIRE(param && grad && exp_avg && exp_avg_sq && step_count && partials && total_out, "adam_step_clipped: NULL pointer");
  ACSR_REQUIRE(n >= 0, "adam_step_clipped: n=%lld", (long long)n);
  ACSR_REQUIRE(n_partials >= 1 && n_partials <= 1024, "adam_step_clipped: n_partials=%d (need 1..1024)", n_partials);
  ACSR_REQUIRE(norm_type > 0.0, "adam_step_clipped: norm_type=%f (need a positive number or inf)", norm_type);
  ACSR_REQUIRE(max_norm > 0.f, "adam_step_clipped: max_norm=%f (need > 0)", max_norm);
  // one CTA even for n == 0: the norm is still reported
  long long need = (n + 255) / 256, cap = kNumSMs * 8;
  launch_pdl(adam_kernel<true>, dim3((int)(need < cap ? (need > 0 ? need : 1) : cap)), dim3(256), 0, (cudaStream_t)stream,
      param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay, (const long long*)step_count,
      partials, n_partials, norm_type, max_norm, total_out);
  launch_pdl(step_inc_kernel, dim3(1), dim3(1), 0, (cudaStream_t)stream, (long long*)step_count);
  return check_launch("adam_step_clipped");
}

}  // extern "C"
