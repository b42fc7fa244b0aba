// gemm.cu — K3 (Hessian SYRK) and K6 (fake-quant forward GEMM) on tcgen05 tensor cores.
//
// One persistent, warp-specialised kernel template (1 CTA per SM):
//   warp 0     TMA producer  (cp.async.bulk.tensor -> 128B-swizzled smem ring, mbarrier tx)
//   warp 1     MMA issuer    (one elected thread, tcgen05.mma kind::f16, fp32 accum in TMEM)
//   warps 2-5  epilogue      (tcgen05.ld TMEM -> registers -> global), double-buffered TMEM
// Tile 128(M) x 256(N) x 64(K), 4-stage ring (48 KB / stage), 2 x 256 TMEM columns.  The
// scaffolding (TMEM setup, rings, rasterisation, epilogue stores, launch) comes from tc.cuh; this
// file also defines the tensor-map encoder declared there.
//
//  * GEMM  (llmc_gemm_bf16):  Y[M,N] = X[M,K] . W[N,K]^T (+bias) — both operands K-major.
//      Replaces F.linear in FakeQuantLinear / EffcientFakeQuantLinear.forward
//      (llmc/compression/quantization/module_utils.py:643, 719).
//  * SYRK  (llmc_syrk_accum): H <- H*n/(n+b) + 2/(n+b) * X^T X, X[T,C] row-major so BOTH
//      operands are MN-major views of the same tensor (no transpose pass).  Only tiles touching
//      the upper triangle are computed; split-K partial slabs + a finalize kernel that applies
//      the running-mean scaling and mirrors.  Replaces GPTQ.add_batch (gptq.py:283-290), whose
//      fp32 SGEMM on X.float() has exactly representable bf16/fp16 operands, so an fp32-
//      accumulating tensor-core product differs only by summation order.
#include "tc.cuh"

namespace llmc {

using namespace tc;

constexpr int BM = 128, BN = 256, BK = 64;
constexpr int kStages = 4;
constexpr int kABytes = BM * BK * 2;                 // 16 KB
constexpr int kBBytes = BN * BK * 2;                 // 32 KB
constexpr int kStageBytes = kABytes + kBBytes;       // 48 KB
constexpr int kBoxBytes = 64 * 64 * 2;               // SYRK box: 64 tokens x 64 channels
constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/;
constexpr int kThreads = 192;
constexpr int kTmemCols = 512;

struct GemmParams {
  int64_t M, N, K;          // GEMM: Y[M,N]; SYRK: M = N = C, K = T
  void* out;                // GEMM: Y (bf16/fp16) ; SYRK: partial slabs fp32 [splits][C][C]
  const void* bias;         // GEMM only, may be null (dtype = out dtype)
  int64_t ld_out;
  int n_tiles_n;            // tiles along N
  int num_units;            // GEMM: tiles ; SYRK: upper tiles * splits
  int num_tiles;            // SYRK: upper tiles
  int splits;               // SYRK split-K factor
  int kb_total;             // k-blocks in K
  int kb_per_split;
  int gn;                   // rasterisation group: n-tiles (GEMM) / m-blocks (SYRK) per group
};

struct Unit {
  int m_blk, n_blk, kb0, kb1, split;
};

template <bool kSyrk>
__device__ __forceinline__ Unit decode_unit(const GemmParams& p, int u) {
  Unit t;
  if constexpr (!kSyrk) {
    // (a 14336-row weight is 117 MB: n-fastest order would stream all of it per 148-tile wave)
    grouped_tile(u, p.num_tiles / p.n_tiles_n, p.n_tiles_n, p.gn, t.m_blk, t.n_blk);
    t.kb0 = 0;
    t.kb1 = p.kb_total;
    t.split = 0;
  } else {
    // tile fastest, split slowest: concurrent CTAs stream the same token range (L2 reuse).
    // Tiles are visited in super-rows of `gn` m-blocks, n-major inside a super-row, so the 148
    // tiles of a wave form a compact patch of H and touch ~4.6K channels of X per k-block instead
    // of all C (X is streamed from HBM once per wave).
    int tile = u % p.num_tiles;
    t.split = u / p.num_tiles;
    const int m_tiles = (static_cast<int>(p.M) + BM - 1) / BM;
    int m0 = 0;
    for (;; m0 += p.gn) {
      const int m1 = min(m0 + p.gn, m_tiles);
      int cnt = 0;
      for (int mi = m0; mi < m1; ++mi) cnt += p.n_tiles_n - (mi >> 1);
      if (tile < cnt) break;
      tile -= cnt;
    }
    const int m1 = min(m0 + p.gn, m_tiles);
    int n = m0 >> 1;
    for (;; ++n) {
      const int cnt = min(m1, 2 * n + 2) - m0;     // m-blocks of the group with m/2 <= n
      if (tile < cnt) break;
      tile -= cnt;
    }
    t.m_blk = m0 + tile;
    t.n_blk = n;
    t.kb0 = t.split * p.kb_per_split;
    t.kb1 = min(t.kb0 + p.kb_per_split, p.kb_total);
  }
  return t;
}

template <bool kSyrk, bool kBf16>
__global__ void __launch_bounds__(kThreads, 1)
umma_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const GemmParams p) {
  uint8_t* smem = smem_align1024();
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full = empty_bar + kStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], 4);   // one arrive per epilogue warp
    }
    fence_barrier_init();
  }
  const uint32_t tmem_base = tmem_setup(warp, tmem_ptr, kTmemCols);

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      Ring<kStages> s;
      for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
        const Unit t = decode_unit<kSyrk>(p, u);
        for (int kb = t.kb0; kb < t.kb1; ++kb) {
          mbar_wait(&empty_bar[s.idx], s.phase ^ 1);
          uint8_t* a_dst = smem + s.idx * kStageBytes;
          uint8_t* b_dst = a_dst + kABytes;
          uint64_t* bar = &full_bar[s.idx];
          mbar_expect_tx(bar, kStageBytes);
          if constexpr (!kSyrk) {
            tma_load_2d(a_dst, &tmA, bar, kb * BK, t.m_blk * BM);
            tma_load_2d(b_dst, &tmB, bar, kb * BK, t.n_blk * BN);
          } else {
            // X[T, C]: coordinate 0 = channel, coordinate 1 = token; box = 64 ch x 64 tok
#pragma unroll
            for (int i = 0; i < BM / 64; ++i)
              tma_load_2d(a_dst + i * kBoxBytes, &tmA, bar, t.m_blk * BM + i * 64, kb * BK);
#pragma unroll
            for (int i = 0; i < BN / 64; ++i)
              tma_load_2d(b_dst + i * kBoxBytes, &tmA, bar, t.n_blk * BN + i * 64, kb * BK);
          }
          s.advance();
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc = make_idesc(kBf16, kBf16, kSyrk, kSyrk, BM, BN);
    Ring<kStages> s;
    Ring<2> acc;
    for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
      const Unit t = decode_unit<kSyrk>(p, u);
      mbar_wait(&tmem_empty[acc.idx], acc.phase ^ 1);
      tcgen05_fence_after();
      const uint32_t d_tmem = tmem_base + acc.idx * BN;
      for (int kb = t.kb0; kb < t.kb1; ++kb) {
        mbar_wait(&full_bar[s.idx], s.phase);
        tcgen05_fence_after();
        if (lane == 0) {
          const uint32_t a_addr = smem_u32(smem + s.idx * kStageBytes);
          const uint32_t b_addr = a_addr + kABytes;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            uint64_t adesc, bdesc;
            if constexpr (!kSyrk) {
              adesc = make_smem_desc(a_addr + k * 32, 16, 1024);
              bdesc = make_smem_desc(b_addr + k * 32, 16, 1024);
            } else {
              adesc = make_smem_desc(a_addr + k * 2048, kBoxBytes, 1024);
              bdesc = make_smem_desc(b_addr + k * 2048, kBoxBytes, 1024);
            }
            umma_f16(d_tmem, adesc, bdesc, idesc, (kb > t.kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty_bar[s.idx]);                         // frees the smem slot
          if (kb == t.kb1 - 1) umma_commit(&tmem_full[acc.idx]);  // accumulator complete
        }
        __syncwarp();
        s.advance();
      }
      if (t.kb1 <= t.kb0 && lane == 0) umma_commit(&tmem_full[acc.idx]);  // empty K range (never)
      acc.advance();
    }
  } else {
    // ===================== epilogue (warps 2..5) =====================
    const int q = warp & 3;                       // TMEM lane quarter this warp may access
    Ring<2> acc;
    for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
      const Unit t = decode_unit<kSyrk>(p, u);
      mbar_wait(&tmem_full[acc.idx], acc.phase);
      tcgen05_fence_after();
      const int64_t row = static_cast<int64_t>(t.m_blk) * BM + q * 32 + lane;
      const uint32_t taddr0 = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc.idx * BN;
#pragma unroll 1
      for (int c = 0; c < BN; c += 32) {
        uint32_t r[32];
        tmem_ld_32x32b_x32(taddr0 + c, r);
        tmem_ld_wait();
        const int64_t col0 = static_cast<int64_t>(t.n_blk) * BN + c;
        if (row < p.M && col0 < p.N) {
          if constexpr (kSyrk) {
            float* o = reinterpret_cast<float*>(p.out) +
                       (static_cast<int64_t>(t.split) * p.M + row) * p.ld_out + col0;
            if (col0 + 32 <= p.N) {
#pragma unroll
              for (int i = 0; i < 32; i += 4)
                *reinterpret_cast<uint4*>(o + i) = make_uint4(r[i], r[i + 1], r[i + 2], r[i + 3]);
            } else {
              for (int i = 0; i < 32 && col0 + i < p.N; ++i) o[i] = __uint_as_float(r[i]);
            }
          } else {
            store_chunk_bias<kBf16>(reinterpret_cast<uint16_t*>(p.out) + row * p.ld_out + col0, r,
                                    reinterpret_cast<const uint16_t*>(p.bias), col0, p.N,
                                    (p.ld_out & 7) == 0);
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

// ---- SYRK finalize: H = a*H + b*sum_s P_s on the upper triangle, mirrored -----------------------
__global__ void __launch_bounds__(256)
syrk_finalize_kernel(float* __restrict__ H, const float* __restrict__ P, int64_t C, int splits,
                     float a, float b) {
  // 32x32 tiles; block (bx, by) with bx >= by handles tile rows by, cols bx and its mirror.
  __shared__ float tile[32][33];
  const int bx = blockIdx.x, by = blockIdx.y;
  if (bx < by) return;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    const int64_t r = static_cast<int64_t>(by) * 32 + i, c = static_cast<int64_t>(bx) * 32 + tx;
    float v = 0.f;
    if (r < C && c < C) {
      float acc = 0.f;
      for (int s = 0; s < splits; ++s) acc += P[(static_cast<int64_t>(s) * C + r) * C + c];
      // for diagonal tiles take the upper-triangle value for both (r,c) and (c,r)
      if (bx == by && c < r) {
        acc = 0.f;
        for (int s = 0; s < splits; ++s) acc += P[(static_cast<int64_t>(s) * C + c) * C + r];
        v = a * H[c * C + r] + b * acc;
      } else {
        v = a * H[r * C + c] + b * acc;
      }
    }
    tile[i][tx] = v;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int64_t r = static_cast<int64_t>(by) * 32 + i, c = static_cast<int64_t>(bx) * 32 + tx;
    if (r < C && c < C) H[r * C + c] = tile[i][tx];
    if (bx != by) {
      const int64_t r2 = static_cast<int64_t>(bx) * 32 + i, c2 = static_cast<int64_t>(by) * 32 + tx;
      if (r2 < C && c2 < C) H[r2 * C + c2] = tile[tx][i];
    }
  }
}

// ---- host side -------------------------------------------------------------------------------------
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                        const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                        const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion,
                                        CUtensorMapFloatOOBfill);

static PFN_tmapEncodeTiled get_encode_fn() {
  static PFN_tmapEncodeTiled fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || p == nullptr) {
    set_last_error("cudaGetDriverEntryPoint(cuTensorMapEncodeTiled) failed: %s",
                   cudaGetErrorString(e));
    return nullptr;
  }
  fn = reinterpret_cast<PFN_tmapEncodeTiled>(p);
  return fn;
}

int encode_tmap_2d(CUtensorMap* out, const void* base, CUtensorMapDataType dtype,
                   uint32_t elem_bytes, uint64_t rows, uint64_t cols, uint64_t ld_elems,
                   uint32_t box_rows, uint32_t box_cols, CUtensorMapSwizzle swizzle) {
  PFN_tmapEncodeTiled fn = get_encode_fn();
  if (!fn) return LLMC_ECUDA;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld_elems * elem_bytes};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, dtype, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_last_error("cuTensorMapEncodeTiled failed with CUresult %d (dtype %d rows %llu cols %llu "
                   "ld %llu box %ux%u)", (int)r, (int)dtype, (unsigned long long)rows,
                   (unsigned long long)cols, (unsigned long long)ld_elems, box_rows, box_cols);
    return LLMC_ECUDA;
  }
  return LLMC_OK;
}

template <bool kSyrk, bool kBf16>
static int launch_umma(const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmParams& p,
                       cudaStream_t st) {
  const int grid = p.num_units < kNumSMs ? p.num_units : kNumSMs;
  return launch_tc<umma_gemm_kernel<kSyrk, kBf16>>(grid, kThreads, kSmemBytes, st, tmA, tmB, p);
}

struct SyrkPlan {
  int n_tiles_n, num_tiles, splits, kb_total, kb_per_split;
};

static SyrkPlan plan_syrk(int64_t T, int64_t C) {
  SyrkPlan s;
  const int mt = static_cast<int>((C + BM - 1) / BM);
  s.n_tiles_n = static_cast<int>((C + BN - 1) / BN);
  int tiles = 0;
  for (int mi = 0; mi < mt; ++mi) {
    int cnt = s.n_tiles_n - (mi >> 1);
    if (cnt > 0) tiles += cnt;
  }
  s.num_tiles = tiles;
  s.kb_total = static_cast<int>((T + BK - 1) / BK);
  // choose the split-K factor that best fills whole waves of 148 CTAs
  int best = 1;
  double best_eff = 0.0;
  for (int sp = 1; sp <= 16; ++sp) {
    if (sp > 1 && s.kb_total / sp < 16) break;
    const long units = static_cast<long>(tiles) * sp;
    const long waves = (units + kNumSMs - 1) / kNumSMs;
    const double eff = static_cast<double>(units) / (waves * kNumSMs) - 0.004 * (sp - 1);
    if (eff > best_eff + 1e-9) { best_eff = eff; best = sp; }
  }
  s.splits = best;
  s.kb_per_split = (s.kb_total + best - 1) / best;
  s.splits = (s.kb_total + s.kb_per_split - 1) / s.kb_per_split;
  return s;
}

}  // namespace llmc

using namespace llmc;

extern "C" int llmc_gemm_bf16(const void* x, const void* w, const void* bias, void* y, int64_t M,
                              int64_t N, int64_t K, int dtype, void* stream) {
  LLMC_CHECK_ARG(M >= 0 && N >= 0 && K > 0, "gemm: bad shape");
  if (M == 0 || N == 0) return LLMC_OK;
  LLMC_CHECK_ARG(x && w && y, "gemm: null pointer");
  LLMC_CHECK_ARG(dtype == LLMC_BF16 || dtype == LLMC_F16, "gemm: dtype must be bf16 or fp16");
  if (K % 8 != 0 || !aligned16(x) || !aligned16(w) || !aligned16(y)) {
    set_last_error("gemm: K=%lld must be a multiple of 8 and pointers 16-byte aligned", (long long)K);
    return LLMC_EALIGN;
  }
  CUtensorMap tmA, tmB;
  if (int rc = encode_tmap_2d(&tmA, x, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, M, K, K, BM, BK,
                              CU_TENSOR_MAP_SWIZZLE_128B))
    return rc;
  if (int rc = encode_tmap_2d(&tmB, w, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, N, K, K, BN, BK,
                              CU_TENSOR_MAP_SWIZZLE_128B))
    return rc;
  GemmParams p{};
  p.M = M; p.N = N; p.K = K;
  p.out = y; p.bias = bias; p.ld_out = N;
  p.n_tiles_n = static_cast<int>((N + BN - 1) / BN);
  const int64_t mt = (M + BM - 1) / BM;
  LLMC_CHECK_ARG(mt * p.n_tiles_n < (1ll << 31), "gemm: too many tiles");
  p.num_units = static_cast<int>(mt * p.n_tiles_n);
  p.num_tiles = p.num_units;
  p.splits = 1;
  p.kb_total = static_cast<int>((K + BK - 1) / BK);
  p.kb_per_split = p.kb_total;
  p.gn = raster_group_n(static_cast<int64_t>(BN) * K * 2, p.n_tiles_n);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return dtype == LLMC_BF16 ? launch_umma<false, true>(tmA, tmB, p, st)
                            : launch_umma<false, false>(tmA, tmB, p, st);
}

extern "C" int64_t llmc_syrk_workspace_bytes(int64_t T, int64_t C) {
  if (T <= 0 || C <= 0) return 0;
  const SyrkPlan s = plan_syrk(T, C);
  return static_cast<int64_t>(s.splits) * C * C * 4;
}

extern "C" int llmc_syrk_accum(const void* x, int64_t T, int64_t C, int dtype, float* H, double n,
                               double b, void* workspace, int64_t workspace_bytes, void* stream) {
  LLMC_CHECK_ARG(T > 0 && C > 0 && x && H && workspace, "syrk: bad argument");
  LLMC_CHECK_ARG(dtype == LLMC_BF16 || dtype == LLMC_F16, "syrk: X must be bf16 or fp16");
  LLMC_CHECK_ARG(n >= 0 && b > 0, "syrk: need n >= 0 and b > 0");
  if (C % 8 != 0 || !aligned16(x) || !aligned16(H) || !aligned16(workspace)) {
    set_last_error("syrk: C=%lld must be a multiple of 8 and pointers 16-byte aligned", (long long)C);
    return LLMC_EALIGN;
  }
  const SyrkPlan s = plan_syrk(T, C);
  LLMC_CHECK_ARG(workspace_bytes >= static_cast<int64_t>(s.splits) * C * C * 4,
                 "syrk: workspace too small (%lld < %lld)", (long long)workspace_bytes,
                 (long long)(static_cast<int64_t>(s.splits) * C * C * 4));
  CUtensorMap tmX;
  if (int rc = encode_tmap_2d(&tmX, x, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, T, C, C, 64, 64,
                              CU_TENSOR_MAP_SWIZZLE_128B))
    return rc;
  GemmParams p{};
  p.M = C; p.N = C; p.K = T;
  p.out = workspace; p.bias = nullptr; p.ld_out = C;
  p.n_tiles_n = s.n_tiles_n;
  p.num_tiles = s.num_tiles;
  p.splits = s.splits;
  p.num_units = s.num_tiles * s.splits;
  p.kb_total = s.kb_total;
  p.kb_per_split = s.kb_per_split;
  p.gn = 12;                      // 12 m-blocks (1536 rows) x ~12 n-tiles ~ one wave of 148 tiles
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = dtype == LLMC_BF16 ? launch_umma<true, true>(tmX, tmX, p, st)
                              : launch_umma<true, false>(tmX, tmX, p, st);
  if (rc) return rc;
  // gptq.py:283-290: H *= n/(n+b); H += (sqrt(2/(n+b)) X)^T (sqrt(2/(n+b)) X)
  const float fa = static_cast<float>(n / (n + b));
  const float fb = static_cast<float>(2.0 / (n + b));
  const unsigned nb = static_cast<unsigned>((C + 31) / 32);
  syrk_finalize_kernel<<<dim3(nb, nb), 256, 0, st>>>(H, reinterpret_cast<const float*>(workspace),
                                                     C, s.splits, fa, fb);
  LLMC_CHECK_LAUNCH();
  return LLMC_OK;
}
