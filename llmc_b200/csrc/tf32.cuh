// tf32.cuh — host entry points of the fp32-accurate 3xTF32 tensor-core update (tf32.cu), used by
// the blocked Cholesky (chol.cu) and the GPTQ / SpQR column sweeps (gptq.cu).
#pragma once

#include "common.cuh"

namespace llmc {

// hi = tf32(x), lo = tf32(x - hi) for a rows x cols fp32 matrix with row stride ld (outputs: ld_out).
int split_tf32(const float* x, int64_t rows, int64_t cols, int64_t ld, float* hi, float* lo,
               int64_t ld_out, cudaStream_t st);

// C[m][n] <- C[m][n] - sum_k A(m,k) B(n,k) (mode 0) or C[m][n] <- sum_k A(m,k) B(n,k) (mode 1),
// m < M, n < N, k < K, for fp32 operands given as tf32 splits (hi, lo).  Operand layout: K-major
// (element (i, k) at base[i*ld + k]) or, with a_mn / b_mn set, MN-major (at base[k*ld + i]).
struct Tf32x3Update {
  const float* Ahi;
  const float* Alo;
  int a_mn;
  int64_t lda;
  const float* Bhi;
  const float* Blo;
  int b_mn;
  int64_t ldb;
  float* C;
  int64_t ldc;
  int64_t M, N;
  int K;
  int mode;
  // Optional tf32 split of the result (same ld as C), written only in rows [0, split_rows) and
  // columns [0, split_cols) of C (multiples of 32).  The blocked Cholesky uses this to get the
  // split of the *next* panel for free from the trailing update.
  float* Chi = nullptr;
  float* Clo = nullptr;
  int64_t split_rows = INT64_MAX;
  int64_t split_cols = INT64_MAX;
  // tri != 0: only the tiles touching the lower triangle (global col <= global row), where
  // (row_off, col_off) is the global position of C[0][0].
  int tri = 0;
  int64_t row_off = 0;
  int64_t col_off = 0;
  // one_tile_per_cta != 0: grid = number of tiles, every CTA computes one tile and exits.  Bulk
  // updates launched on a LOW-priority stream this way give their SMs back at tile granularity
  // (~20 us), so the short kernels of a latency-bound chain on a high-priority stream (blocked
  // Cholesky look-ahead, chol.cu) never wait behind a persistent 148-CTA grid.
  int one_tile_per_cta = 0;
};
int tf32x3_update(const Tf32x3Update& u, cudaStream_t st);

}  // namespace llmc
