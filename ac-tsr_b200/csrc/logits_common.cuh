// Declarations shared by the two full-catalogue logits paths: logits_tc.cu (tcgen05, hidden size 64) and
// logits_simt.cu (fp32 FMA, any other hidden size).
#pragma once
#include "acsr_common.cuh"
#include <cstdlib>

namespace acsr {

constexpr int kD = 64;                 // hidden size handled by ABI v1 of the tensor-core path
constexpr int kBM = 128;               // rows per CTA tile  (UMMA M)
constexpr int kBN = 64;                // catalogue rows per tile (UMMA N)
constexpr int kKC = kD / 4;            // 16-byte K chunks per row
constexpr int kTcThreads = 320;
constexpr int kTmemCols = 128;         // 2 accumulator stages x 64 columns
constexpr int kMaxTopK = 64;

// MODE_TOPK_RANK: MODE_TOPK that also counts, per row, the scores above and equal to the positive's (GAUC's average rank)
enum { MODE_STORE = 0, MODE_CE = 1, MODE_GRAD = 2, MODE_TOPK = 3, MODE_LINEAR = 4, MODE_TOPK_RANK = 5 };

struct LogitsParams {
  const float* out;      // [M,64]
  const float* table;    // [V,64]
  int M;
  long long V;
  int passes;
  int m_tiles, n_tiles, n_chunks;
  // STORE / GRAD
  float* C;
  long long ldc;
  const float* lse;
  const long long* target;
  const float* row_scale;
  // CE
  float* partial;        // [M, n_chunks, 2]
  // TOPK
  int k;
  int n_slots;           // lists per row in pval / pidx (= acsr_logits_num_chunks); the kernel fills n_chunks <= n_slots of them
  long long idx_offset;
  int skip_col0;
  float* pval;           // [M, n_chunks, k]
  long long* pidx;
  int* row_bound;        // [M] or NULL: order-preserving int image of a lower bound of each row's k-th best score, shared by the CTAs of a launch
  // LINEAR: stationary operand element (r,k) = out[r*out_sn + k*out_sk]; Y[v*ldc + r] (+)= D[r][v] + bias[r]
  long long out_sn, out_sk;
  const float* bias;
  int accumulate;
  long long b_out, b_table, b_bias, b_C;   // per-problem strides of a batched launch (blockIdx.y)
  // TOPK_RANK: per (row, chunk) the number of items scoring > rank_score[row] and == rank_score[row], columns 0 (when skipped) and
  // rank_pos[row] - idx_offset excluded -> rank_counts [M, n_slots, 2]
  const long long* rank_pos;
  const float* rank_score;
  int* rank_counts;
};

// grid plan shared by both paths: [m_tile(128 rows), n_chunk] CTAs, about one per SM
static inline void logits_plan(LogitsParams& p, int batch = 1) {
  p.m_tiles = (p.M + kBM - 1) / kBM;
  p.n_tiles = (int)((p.V + kBN - 1) / kBN);
  int nc = kNumSMs / ((p.m_tiles > 0 ? p.m_tiles : 1) * batch);
  if (nc < 1) nc = 1;
  if (nc > p.n_tiles) nc = p.n_tiles;
  p.n_chunks = nc;
}

// top-k mode: pval / pidx hold n_slots = acsr_logits_num_chunks lists per row, one per CTA of the row tile.  The CTAs spread over
// all SMs even when that leaves few catalogue tiles each: measured on B200 (scripts/topk_micro.py), a CTA's first tile (filling the
// k-best lists) costs as much as many later ones, so fewer, longer CTAs lose at every size.
static inline void logits_plan_topk(LogitsParams& p) { p.n_slots = p.n_chunks; }

// gemm_ks.cu: logits for hidden sizes other than 64 on the K-streamed tcgen05 GEMM (mode = ACSR_EPI_STORE / _CE / _CE_GRAD)
int gemm_logits(int mode, const float* out, const float* table, int M, long long V, int d, int passes, float* C, long long ldc,
                float* partial, const float* lse, const long long* target, const float* row_scale, cudaStream_t st);

// logits_simt.cu: same modes, same partial layouts, hidden size d (multiple of 4, <= 1024)
int launch_logits_simt(int mode, LogitsParams& p, int d, cudaStream_t st, const char* who);

}  // namespace acsr
