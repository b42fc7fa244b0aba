// gemm.cu — K3 (Hessian SYRK) and K6 (fake-quant forward GEMM) on tcgen05 tensor cores.
//
// One persistent, warp-specialised kernel template (1 CTA per SM):
//   warp 0     TMA producer  (cp.async.bulk.tensor -> 128B-swizzled smem ring, mbarrier tx)
//   warp 1     MMA issuer    (one elected thread, tcgen05.mma kind::f16, fp32 accum in TMEM)
//   warps 2-5  epilogue      (tcgen05.ld TMEM -> registers -> global), double-buffered TMEM
// Tile 128(M) x 256(N) x 64(K), 4-stage ring (48 KB / stage), 2 x 256 TMEM columns.
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
    // Grouped rasterisation: weights are swept in groups of `gn` n-tiles (<= ~32 MB, L2 resident),
    // all m-tiles per group, n fastest inside the group.  Activations are re-read N/(256*gn)
    // times from HBM, weights once; n-fastest over a 14336-row weight would instead stream the
    // whole 117 MB weight through L2 once per 148-tile wave.
    const int m_tiles = p.num_tiles / p.n_tiles_n;
    const int per_group = p.gn * m_tiles;
    const int g = u / per_group;
    const int rem = u - g * per_group;
    const int gsz = min(p.gn, p.n_tiles_n - g * p.gn);
    t.m_blk = rem / gsz;
    t.n_blk = g * p.gn + (rem - t.m_blk * gsz);
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
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
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
  if (warp == 1) tmem_alloc(tmem_ptr, kTmemCols);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
        const Unit t = decode_unit<kSyrk>(p, u);
        for (int kb = t.kb0; kb < t.kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* a_dst = smem + stage * kStageBytes;
          uint8_t* b_dst = a_dst + kABytes;
          mbar_expect_tx(&full_bar[stage], kStageBytes);
          if constexpr (!kSyrk) {
            tma_load_2d(a_dst, &tmA, &full_bar[stage], kb * BK, t.m_blk * BM);
            tma_load_2d(b_dst, &tmB, &full_bar[stage], kb * BK, t.n_blk * BN);
          } else {
            // X[T, C]: coordinate 0 = channel, coordinate 1 = token; box = 64 ch x 64 tok
#pragma unroll
            for (int i = 0; i < BM / 64; ++i)
              tma_load_2d(a_dst + i * kBoxBytes, &tmA, &full_bar[stage], t.m_blk * BM + i * 64,
                          kb * BK);
#pragma unroll
            for (int i = 0; i < BN / 64; ++i)
              tma_load_2d(b_dst + i * kBoxBytes, &tmA, &full_bar[stage], t.n_blk * BN + i * 64,
                          kb * BK);
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc = make_idesc_f16(kBf16 ? 1 : 0, kSyrk ? 1 : 0, kSyrk ? 1 : 0, BM, BN);
    int stage = 0;
    uint32_t phase = 0;
    int as = 0;
    uint32_t aphase = 0;
    for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
      const Unit t = decode_unit<kSyrk>(p, u);
      mbar_wait(&tmem_empty[as], aphase ^ 1);
      tcgen05_fence_after();
      const uint32_t d_tmem = tmem_base + as * BN;
      for (int kb = t.kb0; kb < t.kb1; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tcgen05_fence_after();
        if (lane == 0) {
          const uint32_t a_addr = smem_u32(smem + stage * kStageBytes);
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
          umma_commit(&empty_bar[stage]);                    // frees the smem slot
          if (kb == t.kb1 - 1) umma_commit(&tmem_full[as]);  // accumulator complete
        }
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
      if (t.kb1 <= t.kb0 && lane == 0) umma_commit(&tmem_full[as]);  // empty K range (never)
      as ^= 1;
      if (as == 0) aphase ^= 1;
    }
  } else {
    // ===================== epilogue (warps 2..5) =====================
    const int q = warp & 3;                       // TMEM lane quarter this warp may access
    int as = 0;
    uint32_t aphase = 0;
    for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
      const Unit t = decode_unit<kSyrk>(p, u);
      mbar_wait(&tmem_full[as], aphase);
      tcgen05_fence_after();
      const int64_t row = static_cast<int64_t>(t.m_blk) * BM + q * 32 + lane;
      const uint32_t taddr0 = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * BN;
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
            uint16_t* o = reinterpret_cast<uint16_t*>(p.out) + row * p.ld_out + col0;
            const uint16_t* bs = reinterpret_cast<const uint16_t*>(p.bias);
            const bool full = (col0 + 32 <= p.N) && ((p.ld_out & 7) == 0);
            uint32_t pk[16];
#pragma unroll
            for (int i = 0; i < 32; i += 2) {
              float v0 = __uint_as_float(r[i]), v1 = __uint_as_float(r[i + 1]);
              if (bs != nullptr) {
                // F.linear adds the bias in fp32 before the single rounding to the out dtype
                if (col0 + i < p.N) v0 += kBf16 ? __uint_as_float(static_cast<uint32_t>(bs[col0 + i]) << 16)
                                                : __half2float(__ushort_as_half(bs[col0 + i]));
                if (col0 + i + 1 < p.N) v1 += kBf16 ? __uint_as_float(static_cast<uint32_t>(bs[col0 + i + 1]) << 16)
                                                    : __half2float(__ushort_as_half(bs[col0 + i + 1]));
              }
              if constexpr (kBf16) {
                __nv_bfloat162 h = __floats2bfloat162_rn(v0, v1);
                pk[i >> 1] = *reinterpret_cast<uint32_t*>(&h);
              } else {
                __half2 h = __floats2half2_rn(v0, v1);
                pk[i >> 1] = *reinterpret_cast<uint32_t*>(&h);
              }
            }
            if (full) {
#pragma unroll
              for (int i = 0; i < 16; i += 4)
                *reinterpret_cast<uint4*>(o + 2 * i) = make_uint4(pk[i], pk[i + 1], pk[i + 2], pk[i + 3]);
            } else {
              for (int i = 0; i < 32 && col0 + i < p.N; ++i)
                o[i] = static_cast<uint16_t>((i & 1) ? (pk[i >> 1] >> 16) : (pk[i >> 1] & 0xffffu));
            }
          }
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[as]);
      as ^= 1;
      if (as == 0) aphase ^= 1;
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, kTmemCols);
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

int encode_tmap_2d_b16(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols,
                       uint64_t ld_elems, uint32_t box_rows, uint32_t box_cols) {
  PFN_tmapEncodeTiled fn = get_encode_fn();
  if (!fn) return LLMC_ECUDA;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld_elems * 2};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides,
                  box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_last_error("cuTensorMapEncodeTiled failed with CUresult %d (rows %llu cols %llu ld %llu)",
                   (int)r, (unsigned long long)rows, (unsigned long long)cols,
                   (unsigned long long)ld_elems);
    return LLMC_ECUDA;
  }
  return LLMC_OK;
}

int encode_tmap_2d_u8(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols,
                      uint64_t ld_elems, uint32_t box_rows, uint32_t box_cols) {
  PFN_tmapEncodeTiled fn = get_encode_fn();
  if (!fn) return LLMC_ECUDA;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld_elems};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides,
                  box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_last_error("cuTensorMapEncodeTiled(u8) failed with CUresult %d (rows %llu cols %llu ld %llu)",
                   (int)r, (unsigned long long)rows, (unsigned long long)cols,
                   (unsigned long long)ld_elems);
    return LLMC_ECUDA;
  }
  return LLMC_OK;
}

int encode_tmap_2d_f32(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols,
                       uint64_t ld_elems, uint32_t box_rows, uint32_t box_cols, int atom32b) {
  PFN_tmapEncodeTiled fn = get_encode_fn();
  if (!fn) return LLMC_ECUDA;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld_elems * 4};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides,
                  box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  atom32b ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_last_error("cuTensorMapEncodeTiled(f32) failed with CUresult %d (rows %llu cols %llu ld %llu)",
                   (int)r, (unsigned long long)rows, (unsigned long long)cols,
                   (unsigned long long)ld_elems);
    return LLMC_ECUDA;
  }
  return LLMC_OK;
}

// swizzle32: CU_TENSOR_MAP_SWIZZLE_32B (box_cols must be 8 = 32 bytes): the 16-byte half of a
// 32-byte row is XORed with bit 2 of the row index, which makes one-row-per-thread 16-byte
// shared-memory loads conflict free.
int encode_tmap_2d_i32_noswizzle(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols,
                                 uint64_t ld_elems, uint32_t box_rows, uint32_t box_cols,
                                 int swizzle32) {
  PFN_tmapEncodeTiled fn = get_encode_fn();
  if (!fn) return LLMC_ECUDA;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld_elems * 4};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_INT32, 2, const_cast<void*>(base), dims, strides, box,
                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  swizzle32 == 2 ? CU_TENSOR_MAP_SWIZZLE_64B
                                 : (swizzle32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE),
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_last_error("cuTensorMapEncodeTiled(i32) failed with CUresult %d", (int)r);
    return LLMC_ECUDA;
  }
  return LLMC_OK;
}

template <bool kSyrk, bool kBf16>
static int launch_umma(const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmParams& p,
                       cudaStream_t st) {
  auto kern = umma_gemm_kernel<kSyrk, kBf16>;
  LLMC_ONCE_PER_DEVICE({
    LLMC_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
  });
  int grid = p.num_units < kNumSMs ? p.num_units : kNumSMs;
  kern<<<grid, kThreads, kSmemBytes, st>>>(tmA, tmB, p);
  LLMC_CHECK_LAUNCH();
  return LLMC_OK;
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
  if (int rc = encode_tmap_2d_b16(&tmA, x, M, K, K, BM, BK)) return rc;
  if (int rc = encode_tmap_2d_b16(&tmB, w, N, K, K, BN, BK)) return rc;
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
  {
    const int64_t tile_bytes = static_cast<int64_t>(BN) * K * 2;      // one n-tile of weights
    int64_t gn = (32ll << 20) / (tile_bytes > 0 ? tile_bytes : 1);
    if (gn < 1) gn = 1;
    if (gn > p.n_tiles_n) gn = p.n_tiles_n;
    p.gn = static_cast<int>(gn);
  }
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
  if (int rc = encode_tmap_2d_b16(&tmX, x, T, C, C, 64, 64)) return rc;
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
