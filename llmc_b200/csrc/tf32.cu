// tf32.cu — fp32-accurate rank-K updates on tcgen05 tensor cores ("3xTF32").
//
//   C[M,N]  <-  C - A * B      (mode 0)      or      C <- A * B      (mode 1)
//
// with fp32 A, B given as pre-split pairs (hi = tf32(x), lo = tf32(x - hi)) and the product
// evaluated as  A_hi*B_hi + A_lo*B_hi + A_hi*B_lo  (three kind::tf32 MMAs accumulating into the
// same fp32 TMEM tile; the dropped A_lo*B_lo term is ~2^-22 relative).  This is the workhorse for
// every fp32 GEMM-shaped step of GPTQ that the reference runs as cuBLAS SGEMM / cuSOLVER:
//   * W[:, i2:] -= Err1 @ Hinv[i1:i2, i2:]                        (gptq.py:244)
//   * the trailing updates of the blocked Cholesky and of the triangular inverse that replace
//     torch.linalg.cholesky / cholesky_inverse / cholesky(upper) (gptq.py:172-174).
// K is small (128 per call), so these are HBM-bound read-modify-write sweeps over C; the three
// MMAs per k-step are free under that roof.
//
// Operand layouts (per operand flag):
//   K-major : element (i, k) at base[i*ld + k]   (rows = M or N index, K contiguous)
//   MN-major: element (i, k) at base[k*ld + i]   (rows = K index, M or N contiguous)
// Same warp-specialised structure as gemm.cu (TMA producer / MMA issuer / 4 epilogue warps,
// double-buffered 2 x 256-column TMEM accumulators, scaffolding from tc.cuh), tile 128 x 256,
// 32 k per stage, 2 stages.  Host entry point: tf32x3_update(const Tf32x3Update&) in tf32.cuh.
#include "tc.cuh"
#include "tf32.cuh"

namespace llmc {

using namespace tc;

namespace t3 {

constexpr int BM = 128, BN = 256, BK = 32;     // BK tf32 elements = 128 bytes
constexpr int kStages = 2;
constexpr int kABytes = BM * BK * 4;             // 16 KB (per hi / lo)
constexpr int kBBytes = BN * BK * 4;             // 32 KB
constexpr int kStageBytes = 2 * (kABytes + kBBytes);   // 96 KB
constexpr int kBoxBytes = 32 * BK * 4;           // MN-major box: 32 MN x 32 K rows = 4 KB
constexpr int kSmemBytes = kStages * kStageBytes + 1024 + 256;
constexpr int kThreads = 192;
constexpr int kTmemCols = 512;

struct Params {
  int64_t M, N;
  int K;
  float* C;
  int64_t ldc;
  float* Chi;            // optional: tf32 split of the result (same ld)
  float* Clo;
  int mode;              // 0: C -= A*B ; 1: C = A*B
  int tri;               // 0 all tiles; 1 only tiles touching the lower triangle (col <= row)
  int n_tiles_n, n_tiles_m;
  int num_units;
  int64_t row_off, col_off;   // global (row, col) of C[0][0] for the triangle test
  int64_t split_rows, split_cols;   // Chi/Clo are written where row < split_rows or col < split_cols
};

__device__ __forceinline__ void decode(const Params& p, int u, int& m_blk, int& n_blk) {
  if (!p.tri) {
    n_blk = u % p.n_tiles_n;
    m_blk = u / p.n_tiles_n;
    return;
  }
  // lower-triangle tiles of row-block mi: n_blk in [0, cnt(mi)) with
  // cnt = number of 256-wide column tiles whose first column <= last row of the block
  int mi = 0;
  for (;; ++mi) {
    const int64_t last_row = p.row_off + static_cast<int64_t>(mi) * BM + BM - 1;
    int64_t cnt = (last_row - p.col_off) / BN + 1;
    if (last_row < p.col_off) cnt = 0;
    if (cnt > p.n_tiles_n) cnt = p.n_tiles_n;
    if (u < cnt) break;
    u -= static_cast<int>(cnt);
  }
  m_blk = mi;
  n_blk = u;
}

__device__ __forceinline__ float to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

template <bool kAmn, bool kBmn>
__global__ void __launch_bounds__(kThreads, 1)
tf32x3_kernel(const __grid_constant__ CUtensorMap tmAhi, const __grid_constant__ CUtensorMap tmAlo,
              const __grid_constant__ CUtensorMap tmBhi, const __grid_constant__ CUtensorMap tmBlo,
              const Params p) {
  uint8_t* smem = smem_align1024();
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full = empty_bar + kStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kb_total = (p.K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmAhi); prefetch_tmap(&tmAlo); prefetch_tmap(&tmBhi); prefetch_tmap(&tmBlo);
    for (int s = 0; s < kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], 4); }
    fence_barrier_init();
  }
  const uint32_t tmem_base = tmem_setup(warp, tmem_ptr, kTmemCols);

  if (warp == 0) {
    if (lane == 0) {
      Ring<kStages> s;
      for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
        int m_blk, n_blk;
        decode(p, u, m_blk, n_blk);
        for (int kb = 0; kb < kb_total; ++kb) {
          mbar_wait(&empty_bar[s.idx], s.phase ^ 1);
          uint8_t* ahi = smem + s.idx * kStageBytes;
          uint8_t* alo = ahi + kABytes;
          uint8_t* bhi = alo + kABytes;
          uint8_t* blo = bhi + kBBytes;
          uint64_t* bar = &full_bar[s.idx];
          mbar_expect_tx(bar, kStageBytes);
          if constexpr (!kAmn) {
            tma_load_2d(ahi, &tmAhi, bar, kb * BK, m_blk * BM);
            tma_load_2d(alo, &tmAlo, bar, kb * BK, m_blk * BM);
          } else {
#pragma unroll
            for (int i = 0; i < BM / 32; ++i) {
              tma_load_2d(ahi + i * kBoxBytes, &tmAhi, bar, m_blk * BM + i * 32, kb * BK);
              tma_load_2d(alo + i * kBoxBytes, &tmAlo, bar, m_blk * BM + i * 32, kb * BK);
            }
          }
          if constexpr (!kBmn) {
            tma_load_2d(bhi, &tmBhi, bar, kb * BK, n_blk * BN);
            tma_load_2d(blo, &tmBlo, bar, kb * BK, n_blk * BN);
          } else {
#pragma unroll
            for (int i = 0; i < BN / 32; ++i) {
              tma_load_2d(bhi + i * kBoxBytes, &tmBhi, bar, n_blk * BN + i * 32, kb * BK);
              tma_load_2d(blo + i * kBoxBytes, &tmBlo, bar, n_blk * BN + i * 32, kb * BK);
            }
          }
          s.advance();
        }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc(2, 2, kAmn, kBmn, BM, BN);    // tf32 x tf32
    Ring<kStages> s;
    Ring<2> acc;
    for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
      mbar_wait(&tmem_empty[acc.idx], acc.phase ^ 1);
      tcgen05_fence_after();
      const uint32_t d_tmem = tmem_base + acc.idx * BN;
      for (int kb = 0; kb < kb_total; ++kb) {
        mbar_wait(&full_bar[s.idx], s.phase);
        tcgen05_fence_after();
        if (lane == 0) {
          const uint32_t ahi = smem_u32(smem + s.idx * kStageBytes);
          const uint32_t alo = ahi + kABytes;
          const uint32_t bhi = alo + kABytes;
          const uint32_t blo = bhi + kBBytes;
#pragma unroll
          for (int k = 0; k < BK / 8; ++k) {
            // K-major: 8 tf32 = 32 B along the swizzled 128-B row; MN-major: one 8-row atom
            const uint32_t aoff = kAmn ? k * 1024 : k * 32;
            const uint32_t boff = kBmn ? k * 1024 : k * 32;
            const uint32_t albo = kAmn ? kBoxBytes : 16, blbo = kBmn ? kBoxBytes : 16;
            // MN-major tf32: SWIZZLE_128B_BASE32B, K groups of 4 rows (512 B)
            const uint32_t asbo = kAmn ? 512 : 1024, bsbo = kBmn ? 512 : 1024;
            const uint32_t alay = kAmn ? 1 : 2, blay = kBmn ? 1 : 2;
            const uint64_t dah = make_smem_desc(ahi + aoff, albo, asbo, alay);
            const uint64_t dal = make_smem_desc(alo + aoff, albo, asbo, alay);
            const uint64_t dbh = make_smem_desc(bhi + boff, blbo, bsbo, blay);
            const uint64_t dbl = make_smem_desc(blo + boff, blbo, bsbo, blay);
            umma_tf32(d_tmem, dah, dbh, idesc, (kb > 0 || k > 0) ? 1u : 0u);
            umma_tf32(d_tmem, dal, dbh, idesc, 1u);
            umma_tf32(d_tmem, dah, dbl, idesc, 1u);
          }
          umma_commit(&empty_bar[s.idx]);
          if (kb == kb_total - 1) umma_commit(&tmem_full[acc.idx]);
        }
        __syncwarp();
        s.advance();
      }
      acc.advance();
    }
  } else {
    const int q = warp & 3;
    Ring<2> acc;
    for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
      int m_blk, n_blk;
      decode(p, u, m_blk, n_blk);
      mbar_wait(&tmem_full[acc.idx], acc.phase);
      tcgen05_fence_after();
      const int64_t row = static_cast<int64_t>(m_blk) * BM + q * 32 + lane;
      const uint32_t taddr0 = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc.idx * BN;
#pragma unroll 1
      for (int c = 0; c < BN; c += 32) {
        uint32_t r[32];
        tmem_ld_32x32b_x32(taddr0 + c, r);
        tmem_ld_wait();
        const int64_t col0 = static_cast<int64_t>(n_blk) * BN + c;
        if (row < p.M && col0 < p.N) {
          float* cp = p.C + row * p.ldc + col0;
          const bool vec = (col0 + 32 <= p.N) && ((reinterpret_cast<uintptr_t>(cp) & 15) == 0);
          float v[32];
          if (p.mode == 0) {
            if (vec) {
#pragma unroll
              for (int i = 0; i < 32; i += 4) {
                const float4 o = *reinterpret_cast<const float4*>(cp + i);
                v[i] = o.x - __uint_as_float(r[i]);
                v[i + 1] = o.y - __uint_as_float(r[i + 1]);
                v[i + 2] = o.z - __uint_as_float(r[i + 2]);
                v[i + 3] = o.w - __uint_as_float(r[i + 3]);
              }
            } else {
              for (int i = 0; i < 32; ++i)
                v[i] = (col0 + i < p.N) ? cp[i] - __uint_as_float(r[i]) : 0.f;
            }
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
          }
          if (vec) {
#pragma unroll
            for (int i = 0; i < 32; i += 4)
              *reinterpret_cast<float4*>(cp + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
          } else {
            for (int i = 0; i < 32 && col0 + i < p.N; ++i) cp[i] = v[i];
          }
          if (p.Chi != nullptr && (row < p.split_rows || col0 < p.split_cols)) {
            float* hp = p.Chi + row * p.ldc + col0;
            float* lp = p.Clo + row * p.ldc + col0;
            if (vec && ((reinterpret_cast<uintptr_t>(hp) | reinterpret_cast<uintptr_t>(lp)) & 15) == 0) {
#pragma unroll
              for (int i = 0; i < 32; i += 4) {
                const float4 h = make_float4(to_tf32(v[i]), to_tf32(v[i + 1]), to_tf32(v[i + 2]), to_tf32(v[i + 3]));
                *reinterpret_cast<float4*>(hp + i) = h;
                *reinterpret_cast<float4*>(lp + i) = make_float4(to_tf32(v[i] - h.x), to_tf32(v[i + 1] - h.y),
                                                                 to_tf32(v[i + 2] - h.z), to_tf32(v[i + 3] - h.w));
              }
            } else {
              for (int i = 0; i < 32 && col0 + i < p.N; ++i) {
                const float h = to_tf32(v[i]);
                hp[i] = h;
                lp[i] = to_tf32(v[i] - h);
              }
            }
          }
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc.idx]);
      acc.advance();
    }
  }
  tmem_teardown(warp, tmem_base, kTmemCols);
}

__global__ void __launch_bounds__(256)
split_tf32_kernel(const float* __restrict__ x, int64_t rows, int64_t cols, int64_t ld,
                  float* __restrict__ hi, float* __restrict__ lo, int64_t ld_out) {
  const int64_t total = rows * cols;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t r = i / cols, c = i - r * cols;
    const float v = x[r * ld + c];
    const float h = to_tf32(v);
    hi[r * ld_out + c] = h;
    lo[r * ld_out + c] = to_tf32(v - h);
  }
}

}  // namespace t3

int tf32x3_update(const Tf32x3Update& u, cudaStream_t st) {
  using namespace t3;
  const int64_t M = u.M, N = u.N;
  const int K = u.K;
  if (M <= 0 || N <= 0 || K <= 0) return LLMC_OK;
  if ((u.lda % 4) || (u.ldb % 4) || !aligned16(u.Ahi) || !aligned16(u.Alo) || !aligned16(u.Bhi) ||
      !aligned16(u.Blo)) {
    set_last_error("tf32x3_update: operands need 16-byte aligned bases and ld %% 4 == 0");
    return LLMC_EALIGN;
  }
  // K-major: [rows, K] boxes of BK fp32 = 128 B, 128B swizzle; MN-major: [K, rows] boxes of
  // 32 fp32, 128B swizzle with 32-byte atoms (SWIZZLE_128B_BASE32B in the smem descriptor)
  auto encode = [&](CUtensorMap* m, const float* base, int mn, int64_t rows, int64_t ld,
                    uint32_t box_rows) {
    return mn ? encode_tmap_2d(m, base, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, K, rows, ld, BK, 32,
                               CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)
              : encode_tmap_2d(m, base, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, rows, K, ld, box_rows,
                               BK, CU_TENSOR_MAP_SWIZZLE_128B);
  };
  CUtensorMap tah, tal, tbh, tbl;
  if (int rc = encode(&tah, u.Ahi, u.a_mn, M, u.lda, BM)) return rc;
  if (int rc = encode(&tal, u.Alo, u.a_mn, M, u.lda, BM)) return rc;
  if (int rc = encode(&tbh, u.Bhi, u.b_mn, N, u.ldb, BN)) return rc;
  if (int rc = encode(&tbl, u.Blo, u.b_mn, N, u.ldb, BN)) return rc;
  Params p{};
  p.M = M; p.N = N; p.K = K; p.C = u.C; p.ldc = u.ldc; p.Chi = u.Chi; p.Clo = u.Clo;
  p.mode = u.mode; p.tri = u.tri; p.row_off = u.row_off; p.col_off = u.col_off;
  p.split_rows = u.split_rows; p.split_cols = u.split_cols;
  p.n_tiles_m = static_cast<int>((M + BM - 1) / BM);
  p.n_tiles_n = static_cast<int>((N + BN - 1) / BN);
  if (!u.tri) {
    p.num_units = p.n_tiles_m * p.n_tiles_n;
  } else {
    long units = 0;
    for (int mi = 0; mi < p.n_tiles_m; ++mi) {
      const int64_t last_row = u.row_off + static_cast<int64_t>(mi) * BM + BM - 1;
      int64_t cnt = last_row < u.col_off ? 0 : (last_row - u.col_off) / BN + 1;
      if (cnt > p.n_tiles_n) cnt = p.n_tiles_n;
      units += cnt;
    }
    p.num_units = static_cast<int>(units);
  }
  if (p.num_units == 0) return LLMC_OK;
  const int grid = (u.one_tile_per_cta || p.num_units < kNumSMs) ? p.num_units : kNumSMs;
  if (!u.a_mn && !u.b_mn) return launch_tc<tf32x3_kernel<false, false>>(grid, kThreads, kSmemBytes, st, tah, tal, tbh, tbl, p);
  if (!u.a_mn && u.b_mn) return launch_tc<tf32x3_kernel<false, true>>(grid, kThreads, kSmemBytes, st, tah, tal, tbh, tbl, p);
  if (u.a_mn && !u.b_mn) return launch_tc<tf32x3_kernel<true, false>>(grid, kThreads, kSmemBytes, st, tah, tal, tbh, tbl, p);
  return launch_tc<tf32x3_kernel<true, true>>(grid, kThreads, kSmemBytes, st, tah, tal, tbh, tbl, p);
}

int split_tf32(const float* x, int64_t rows, int64_t cols, int64_t ld, float* hi, float* lo,
               int64_t ld_out, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return LLMC_OK;
  int64_t blocks = (rows * cols + 255) / 256;
  if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
  t3::split_tf32_kernel<<<(int)blocks, 256, 0, st>>>(x, rows, cols, ld, hi, lo, ld_out);
  LLMC_CHECK_LAUNCH();
  return LLMC_OK;
}

}  // namespace llmc

using namespace llmc;

// Exported for unit tests and as a general fp32-accurate tensor-core GEMM building block.
extern "C" int llmc_split_tf32(const float* x, int64_t rows, int64_t cols, int64_t ld, float* hi,
                               float* lo, void* stream) {
  LLMC_CHECK_ARG(x && hi && lo && rows >= 0 && cols >= 0 && ld >= cols, "split_tf32: bad argument");
  return split_tf32(x, rows, cols, ld, hi, lo, ld, static_cast<cudaStream_t>(stream));
}

extern "C" int llmc_gemm_f32x3(const float* a_hi, const float* a_lo, int a_mn, int64_t lda,
                               const float* b_hi, const float* b_lo, int b_mn, int64_t ldb,
                               float* c, int64_t ldc, int64_t M, int64_t N, int64_t K, int mode,
                               int lower_only, void* stream) {
  LLMC_CHECK_ARG(a_hi && a_lo && b_hi && b_lo && c, "gemm_f32x3: null pointer");
  LLMC_CHECK_ARG(M >= 0 && N >= 0 && K > 0 && K % 8 == 0 && K <= (1 << 20), "gemm_f32x3: bad shape (K %% 8 == 0)");
  LLMC_CHECK_ARG(mode == 0 || mode == 1, "gemm_f32x3: mode must be 0 (C -= AB) or 1 (C = AB)");
  return tf32x3_update({.Ahi = a_hi, .Alo = a_lo, .a_mn = a_mn, .lda = lda,
                        .Bhi = b_hi, .Blo = b_lo, .b_mn = b_mn, .ldb = ldb,
                        .C = c, .ldc = ldc, .M = M, .N = N, .K = (int)K, .mode = mode,
                        .tri = lower_only},
                       static_cast<cudaStream_t>(stream));
}
