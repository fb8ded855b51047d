// Weight / bias gradient of a token-parallel linear layer:  dW[N,K] += dY[T,N]^T . X[T,K],  db[N] += sum_t dY.
// T (tokens) is the long axis (12,800 per step) and the output is tiny (64x64 ... 256x64), the
// shape library GEMMs handle worst (one split-K CTA per output tile, ~40 us each on B200).
// Decomposition: the output is cut into small (8R x 8R) tiles and the token axis into `splits`
// ranges so that ~4 CTAs per SM are busy while the number of atomics (N*K*splits) stays small.
// Inside a CTA four 64-thread groups take every fourth token of a 64-token shared-memory slab,
// each thread accumulates an R x R register tile in exact fp32 FMAs, the four partial tiles are
// summed through shared memory and one atomic per output element lands the result directly in the
// caller's (flat) gradient buffer.  Also used for d_out = G.E of the CE backward (reduction over V).
#include "acsr_common.cuh"
#include "../../include/acsr.h"

namespace acsr {

constexpr int kWgThreads = 256;
constexpr int kWgSlab = 64;        // tokens per shared-memory slab

template <int R>
__global__ void __launch_bounds__(kWgThreads)
linear_wgrad_kernel(const float* __restrict__ dY, const float* __restrict__ X, int T, int N, int K, int tok_per_cta,
                    int tiles_k, float* __restrict__ dW, float* __restrict__ db, long long strY, long long strX, long long strW,
                    long long strB) {
  pdl_launch_dependents();
  pdl_wait();
  constexpr int TILE = 8 * R;
  // batched launch: blockIdx.z selects one independent (dY, X, dW, db) problem
  dY += blockIdx.z * strY; X += blockIdx.z * strX; dW += blockIdx.z * strW;
  if (db != nullptr) db += blockIdx.z * strB;
  __shared__ __align__(16) float sY[kWgSlab][TILE];
  __shared__ __align__(16) float sX[kWgSlab][TILE];
  __shared__ float sRed[3][64][R * R + R];
  const int tile_n = blockIdx.y / tiles_k, tile_k = blockIdx.y % tiles_k;
  const int n0 = tile_n * TILE, k0 = tile_k * TILE;
  const int grp = threadIdx.x >> 6, u = threadIdx.x & 63;
  const int ty = u >> 3, tx = u & 7;                 // ty -> n sub-tile, tx -> k sub-tile
  const int t_begin = blockIdx.x * tok_per_cta;
  const int t_end = min(T, t_begin + tok_per_cta);
  const bool vecY = (N % 4 == 0) && (n0 + TILE <= N), vecX = (K % 4 == 0) && (k0 + TILE <= K);
  float acc[R][R], accb[R];
#pragma unroll
  for (int a = 0; a < R; ++a) {
    accb[a] = 0.f;
#pragma unroll
    for (int c = 0; c < R; ++c) acc[a][c] = 0.f;
  }
  // software pipeline: the next 64-token slab is fetched into registers while the current one is consumed
  constexpr int NV = kWgSlab * TILE / 4 / kWgThreads;      // float4 per thread per matrix per slab
  float4 ry[NV], rx[NV];
  auto fetch = [&](int t0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int e = threadIdx.x + i * kWgThreads;
      const int tt = e / (TILE / 4), q = e % (TILE / 4), t = t0 + tt;
      ry[i] = rx[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (t < t_end) {
        const float* py = dY + (long long)t * N + n0 + 4 * q;
        const float* px = X + (long long)t * K + k0 + 4 * q;
        if (vecY) ry[i] = *reinterpret_cast<const float4*>(py);
        else {
          if (n0 + 4 * q + 0 < N) ry[i].x = py[0];
          if (n0 + 4 * q + 1 < N) ry[i].y = py[1];
          if (n0 + 4 * q + 2 < N) ry[i].z = py[2];
          if (n0 + 4 * q + 3 < N) ry[i].w = py[3];
        }
        if (vecX) rx[i] = *reinterpret_cast<const float4*>(px);
        else {
          if (k0 + 4 * q + 0 < K) rx[i].x = px[0];
          if (k0 + 4 * q + 1 < K) rx[i].y = px[1];
          if (k0 + 4 * q + 2 < K) rx[i].z = px[2];
          if (k0 + 4 * q + 3 < K) rx[i].w = px[3];
        }
      }
    }
  };
  if (t_begin < t_end) fetch(t_begin);
  for (int t0 = t_begin; t0 < t_end; t0 += kWgSlab) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int e = threadIdx.x + i * kWgThreads;
      const int tt = e / (TILE / 4), q = e % (TILE / 4);
      *reinterpret_cast<float4*>(&sY[tt][4 * q]) = ry[i];
      *reinterpret_cast<float4*>(&sX[tt][4 * q]) = rx[i];
    }
    __syncthreads();
    if (t0 + kWgSlab < t_end) fetch(t0 + kWgSlab);
#pragma unroll 4
    for (int tt = grp; tt < kWgSlab; tt += 4) {
      float y[R], x[R];
#pragma unroll
      for (int a = 0; a < R; ++a) { y[a] = sY[tt][ty * R + a]; x[a] = sX[tt][tx * R + a]; }
#pragma unroll
      for (int a = 0; a < R; ++a) {
        accb[a] += y[a];
#pragma unroll
        for (int c = 0; c < R; ++c) acc[a][c] = fmaf(y[a], x[c], acc[a][c]);
      }
    }
    __syncthreads();
  }
  // sum the four token groups, then one atomic per output element
  if (grp > 0) {
#pragma unroll
    for (int a = 0; a < R; ++a) {
      sRed[grp - 1][u][R * R + a] = accb[a];
#pragma unroll
      for (int c = 0; c < R; ++c) sRed[grp - 1][u][a * R + c] = acc[a][c];
    }
  }
  __syncthreads();
  if (grp == 0) {
#pragma unroll
    for (int a = 0; a < R; ++a) {
      const int n = n0 + ty * R + a;
      float bsum = accb[a] + sRed[0][u][R * R + a] + sRed[1][u][R * R + a] + sRed[2][u][R * R + a];
#pragma unroll
      for (int c = 0; c < R; ++c) {
        const int k = k0 + tx * R + c;
        const float v = acc[a][c] + sRed[0][u][a * R + c] + sRed[1][u][a * R + c] + sRed[2][u][a * R + c];
        if (n < N && k < K) atomicAdd(dW + (long long)n * K + k, v);
      }
      if (db != nullptr && tx == 0 && tile_k == 0 && n < N) atomicAdd(db + n, bsum);
    }
  }
}

// ---- projection weights of one AC layer folded for ONE batched forward GEMM -------------------------------------------------
// layers.py:658-659, 687-689: mixed_q/k/v = x.Wq/k/v^T + b ; attack_q = mixed_q.Waq^T + baq ; attack_k = mixed_k.Wak^T + bak.
// attack_q = x.(Waq.Wq)^T + (Waq.bq + baq), so with the folded weights all five projections read the same x and run as one
// batched launch.  Slots 0-2 of out_W [5,d,d] / out_b [5,d] are copies of Wq, Wk, Wv; slots 3, 4 the folded attack pair.
// One CTA per slot; parameters only (read before the dependency wait), a few microseconds next to the embedding kernel.
constexpr int kFoldRows = 8;       // output rows per CTA
__global__ void __launch_bounds__(256) fold_attack_weights_kernel(const float* __restrict__ Wqkv, const float* __restrict__ bqkv,
                                                                  const float* __restrict__ Waqk, const float* __restrict__ baqk, int d,
                                                                  float* __restrict__ out_W, float* __restrict__ out_b) {
  extern __shared__ float fsm[];                    // B [d][d], A rows [kFoldRows][d], b1 [d]
  // (no early programmatic-launch trigger: the folded weights it writes are registered as static, see acsr_register_static)
  pdl_wait();
  const int slot = blockIdx.y, r0 = blockIdx.x * kFoldRows;
  const int nr = min(kFoldRows, d - r0);
  if (nr <= 0) return;
  float* oW = out_W + (long long)slot * d * d + (long long)r0 * d;
  float* ob = out_b + (long long)slot * d + r0;
  if (slot < 3) {
    for (int e = threadIdx.x; e < nr * d; e += blockDim.x) oW[e] = Wqkv[(long long)slot * d * d + (long long)r0 * d + e];
    for (int e = threadIdx.x; e < nr; e += blockDim.x) ob[e] = bqkv[slot * d + r0 + e];
    return;
  }
  float* sB = fsm;
  float* sA = sB + d * d;
  float* sb1 = sA + kFoldRows * d;
  const int first = slot - 3;                                                     // the projection folded in: Wq (slot 3) or Wk (slot 4)
  const float* A = Waqk + (long long)first * d * d + (long long)r0 * d;           // rows r0.. of the second linear map
  const float* b2 = baqk + first * d;
  const float* Bm = Wqkv + (long long)first * d * d;
  for (int e = threadIdx.x; e < d * d; e += blockDim.x) sB[e] = Bm[e];
  for (int e = threadIdx.x; e < nr * d; e += blockDim.x) sA[e] = A[e];
  for (int e = threadIdx.x; e < d; e += blockDim.x) sb1[e] = bqkv[first * d + e];
  __syncthreads();
  for (int e = threadIdx.x; e < nr * d; e += blockDim.x) {
    const int r = e / d, c = e - r * d;             // out[r][c] = sum_k A[r][k] * B[k][c]: lanes walk c (conflict-free), A broadcast
    float s = 0.f;
#pragma unroll 8
    for (int k = 0; k < d; ++k) s = fmaf(sA[r * d + k], sB[k * d + c], s);
    oW[e] = s;
  }
  for (int r = threadIdx.x; r < nr; r += blockDim.x) {
    float s = b2[r0 + r];
    for (int k = 0; k < d; ++k) s = fmaf(sA[r * d + k], sb1[k], s);
    ob[r] = s;
  }
}

}  // namespace acsr

using namespace acsr;

extern "C" int acsr_fold_attack_weights(const float* Wqkv, const float* bqkv, const float* Waqk, const float* baqk, int d, float* out_W,
                                        float* out_b, void* stream) {
  ACSR_REQUIRE(Wqkv && bqkv && Waqk && baqk && out_W && out_b && d > 0 && d <= 1024, "fold_attack_weights: bad arguments");
  ACSR_REQUIRE(d <= 128, "fold_attack_weights: hidden size %d > 128", d);
  const size_t smem = (size_t)(d * d + kFoldRows * d + d) * sizeof(float);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(fold_attack_weights_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { set_error("fold_attack_weights: smem attr: %s", cudaGetErrorString(e)); return ACSR_ERR_CUDA; }
  }
  launch_pdl(fold_attack_weights_kernel, dim3((d + kFoldRows - 1) / kFoldRows, 5), dim3(256), smem, (cudaStream_t)stream, Wqkv, bqkv,
             Waqk, baqk, d, out_W, out_b);
  return check_launch("fold_attack_weights");
}

static int launch_wgrad(const float* dY, const float* X, int T, int N, int K, float* dW, float* db, int batch, long long sY,
                        long long sX, long long sW, long long sB, cudaStream_t stream, const char* who) {
  ACSR_REQUIRE(dY && X && dW, "%s: NULL pointer", who);
  ACSR_REQUIRE(T >= 0 && N > 0 && K > 0 && batch > 0 && batch < 65536, "%s: bad sizes", who);
  if (T == 0) return ACSR_OK;
  const bool big = (long long)N * K > 8192;
  const int tile = big ? 32 : 16;
  const int tiles_n = (N + tile - 1) / tile, tiles_k = (K + tile - 1) / tile;
  int splits = (4 * kNumSMs) / (tiles_n * tiles_k * batch);
  if (splits < 1) splits = 1;
  int tok = (T + splits - 1) / splits;
  tok = (tok + kWgSlab - 1) / kWgSlab * kWgSlab;
  dim3 grid((T + tok - 1) / tok, tiles_n * tiles_k, batch);
  if (big)
    launch_pdl(linear_wgrad_kernel<4>, dim3(grid), dim3(kWgThreads), 0, stream, dY, X, T, N, K, tok, tiles_k, dW, db, sY, sX, sW, sB);
  else
    launch_pdl(linear_wgrad_kernel<2>, dim3(grid), dim3(kWgThreads), 0, stream, dY, X, T, N, K, tok, tiles_k, dW, db, sY, sX, sW, sB);
  return check_launch(who);
}

extern "C" int acsr_linear_wgrad(const float* dY, const float* X, int T, int N, int K, float* dW, float* db, void* stream) {
  return launch_wgrad(dY, X, T, N, K, dW, db, 1, 0, 0, 0, 0, (cudaStream_t)stream, "linear_wgrad");
}

extern "C" int acsr_linear_wgrad_batched(const float* dY, const float* X, int T, int N, int K, float* dW, float* db, int batch,
                                         int64_t stride_dy, int64_t stride_x, int64_t stride_dw, int64_t stride_db, void* stream) {
  return launch_wgrad(dY, X, T, N, K, dW, db, batch, stride_dy, stride_x, stride_dw, stride_db, (cudaStream_t)stream,
                      "linear_wgrad_batched");
}
