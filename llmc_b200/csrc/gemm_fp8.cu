// gemm_fp8.cu — K7-fp8: block-scaled FP8 forward of 128x128 FP8 checkpoints (DeepSeek-V3 / R1),
// the pair the reference runs on Hopper and Blackwell (kernel.py:31-53, 141-242; module_utils.py
// block_wise_fp8_forward_func).
//
//  * llmc_fp8_act_quant: per 1x128 block of the last dimension, s = absmax / 448 and
//      y = e4m3(x / s).  Both divisions are `div.full.f32` and the conversion is
//      `cvt.rn.satfinite.e4m3x2.f32`, the instructions the reference's Triton kernel compiles to,
//      so codes and scales match it bit for bit on the same GPU (IEEE division would differ by
//      up to 2 ulp in the scale).  An all-zero block gives s = 0 and NaN codes, as there.
//      One warp per block, 4 elements per lane; HBM-bound.
//
//  * llmc_fp8_gemm: C[M,N] = sum_kb (A_kb . B_kb^T) * a_s[m,kb] * b_s[n/128,kb] with A [M,K] and
//      B [N,K] e4m3, both K-major, and fp32 scales.  Persistent, warp-specialised, 1 CTA per SM:
//        warp 0     TMA producer: one 128x128-byte box of A and of B per K-block (128 fp8 = one
//                   128-byte swizzle row = one scale block), 6-stage ring
//        warp 1     MMA issuer: four tcgen05.mma kind::f8f6f4 (K = 32) per K-block into a FRESH
//                   128-column TMEM slot (4 slots), then commit
//        warps 2-5  promotion + epilogue: tcgen05.ld the slot, acc = fma(dot * a_s, b_s, acc) in
//                   registers (packed f32x2; the reference's PTX issues mul.f32x2 then
//                   fma.rn.f32x2 in this order), then one rounding to the output dtype.
//      Tile 128(M) x 128(N): a tile's columns share one weight-scale row, as the reference's
//      `n // 128` indexing assumes.  Ragged M and N: TMA zero-fill and masked stores.
//      Optional bias (bf16 output only) follows block_wise_fp8_forward_func: the fp32 result is
//      rounded to bf16 and then `y += bias` rounds bf16(float(y) + float(bias)) once more.
//      The scaffolding (TMEM setup, rings, rasterisation, 16-bit stores, launch) comes from tc.cuh.
#include "tc.cuh"

namespace llmc {

using namespace tc;

namespace fp8g {

constexpr int BM = 128, BN = 128, BK = 128;          // BK in elements = bytes
constexpr int kStages = 6;
constexpr int kTileBytes = BM * BK;                  // 16 KB (A) = 16 KB (B)
constexpr int kStageBytes = 2 * kTileBytes;
constexpr int kSlots = 4;                            // TMEM accumulator slots of BN columns
constexpr int kTmemCols = kSlots * BN;               // 512
constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/;
constexpr int kThreads = 192;

struct Params {
  int64_t M, N, K;
  const float* a_s;         // [M, kb_total]
  const float* b_s;         // [ceil(N/128), kb_total]
  void* out;                // [M, N] out_dtype
  const void* bias;         // [N] bias_dtype, bf16 output only; may be null
  int out_dtype, bias_dtype;
  int kb_total;
  int n_tiles_n, m_tiles, num_tiles;
  int gn;                   // rasterisation group (n-tiles)
};

__device__ __forceinline__ float bias_at(const Params& p, int64_t col) {
  if (p.bias_dtype == LLMC_F32) return reinterpret_cast<const float*>(p.bias)[col];
  return __uint_as_float(static_cast<uint32_t>(reinterpret_cast<const uint16_t*>(p.bias)[col]) << 16);
}

// one 32-column chunk of a finished row -> global
__device__ __forceinline__ void store_chunk(const Params& p, int64_t row, int64_t col0,
                                            const float* v) {
  const int64_t n_valid = p.N - col0;
  if (p.out_dtype == LLMC_F32) {
    float* o = reinterpret_cast<float*>(p.out) + row * p.N + col0;
    if (n_valid >= 32 && (p.N & 3) == 0) {
#pragma unroll
      for (int i = 0; i < 32; i += 4) *reinterpret_cast<float4*>(o + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i)
        if (i < n_valid) o[i] = v[i];
    }
    return;
  }
  uint32_t pk[16];
  if (p.out_dtype == LLMC_BF16) {
#pragma unroll
    for (int i = 0; i < 32; i += 2) {
      pk[i >> 1] = pack2<true>(v[i], v[i + 1]);
      if (p.bias != nullptr) {
        // `y += bias`: bf16 y and fp32 / bf16 bias meet in fp32, one more rounding to bf16
        const float b0 = i < n_valid ? bias_at(p, col0 + i) : 0.f;
        const float b1 = i + 1 < n_valid ? bias_at(p, col0 + i + 1) : 0.f;
        pk[i >> 1] = pack2<true>(__uint_as_float(pk[i >> 1] << 16) + b0,
                                 __uint_as_float(pk[i >> 1] & 0xffff0000u) + b1);
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < 32; i += 2) pk[i >> 1] = pack2<false>(v[i], v[i + 1]);
  }
  // columns counted from the chunk's start: the first n_valid are inside the row
  store_row32_b16(reinterpret_cast<uint16_t*>(p.out) + row * p.N + col0, pk,
                  n_valid >= 32 && (p.N & 7) == 0, 0, n_valid);
}

__global__ void __launch_bounds__(kThreads, 1)
fp8_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const Params p) {
  uint8_t* smem = smem_align1024();
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full = empty_bar + kStages;
  uint64_t* tmem_empty = tmem_full + kSlots;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + kSlots);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < kSlots; ++s) {
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
      for (int u = blockIdx.x; u < p.num_tiles; u += gridDim.x) {
        int m_blk, n_blk;
        grouped_tile(u, p.m_tiles, p.n_tiles_n, p.gn, m_blk, n_blk);
        for (int kb = 0; kb < p.kb_total; ++kb) {
          mbar_wait(&empty_bar[s.idx], s.phase ^ 1);
          uint8_t* a_dst = smem + s.idx * kStageBytes;
          mbar_expect_tx(&full_bar[s.idx], kStageBytes);
          tma_load_2d(a_dst, &tmA, &full_bar[s.idx], kb * BK, m_blk * BM);
          tma_load_2d(a_dst + kTileBytes, &tmB, &full_bar[s.idx], kb * BK, n_blk * BN);
          s.advance();
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc = make_idesc(0, 0, 0, 0, BM, BN);     // e4m3 x e4m3, both K-major
    Ring<kStages> s;
    Ring<kSlots> slot;
    for (int u = blockIdx.x; u < p.num_tiles; u += gridDim.x) {
      for (int kb = 0; kb < p.kb_total; ++kb) {
        mbar_wait(&tmem_empty[slot.idx], slot.phase ^ 1);
        mbar_wait(&full_bar[s.idx], s.phase);
        tcgen05_fence_after();
        if (lane == 0) {
          const uint32_t a_addr = smem_u32(smem + s.idx * kStageBytes);
          const uint32_t b_addr = a_addr + kTileBytes;
          const uint32_t d_tmem = tmem_base + slot.idx * BN;
#pragma unroll
          for (int k = 0; k < BK / 32; ++k)
            umma_f8f6f4(d_tmem, make_smem_desc(a_addr + k * 32, 16, 1024),
                        make_smem_desc(b_addr + k * 32, 16, 1024), idesc, k > 0 ? 1u : 0u);
          umma_commit(&empty_bar[s.idx]);     // frees the smem slot
          umma_commit(&tmem_full[slot.idx]);  // this K-block's partial product is ready
        }
        __syncwarp();
        s.advance();
        slot.advance();
      }
    }
  } else {
    // ===================== promotion + epilogue (warps 2..5) =====================
    const int q = warp & 3;                       // TMEM lane quarter this warp may access
    Ring<kSlots> slot;
    for (int u = blockIdx.x; u < p.num_tiles; u += gridDim.x) {
      int m_blk, n_blk;
      grouped_tile(u, p.m_tiles, p.n_tiles_n, p.gn, m_blk, n_blk);
      const int64_t row = static_cast<int64_t>(m_blk) * BM + q * 32 + lane;
      const bool row_ok = row < p.M;
      const float* as_row = p.a_s + (row_ok ? row : 0) * p.kb_total;
      const float* bs_row = p.b_s + static_cast<int64_t>(n_blk) * p.kb_total;
      float acc[BN];
#pragma unroll
      for (int i = 0; i < BN; ++i) acc[i] = 0.f;
      float sa = row_ok ? __ldg(as_row) : 0.f;
      float sb = __ldg(bs_row);
      for (int kb = 0; kb < p.kb_total; ++kb) {
        // next K-block's scales are fetched while this one waits on the tensor core
        const int kn = kb + 1 < p.kb_total ? kb + 1 : kb;
        const float sa_next = row_ok ? __ldg(as_row + kn) : 0.f;
        const float sb_next = __ldg(bs_row + kn);
        mbar_wait(&tmem_full[slot.idx], slot.phase);
        tcgen05_fence_after();
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + slot.idx * BN;
#pragma unroll
        for (int c = 0; c < BN; c += 32) {
          uint32_t r[32];
          tmem_ld_32x32b_x32(taddr + c, r);
          tmem_ld_wait();
          if (c == BN - 32) {
            // the slot has been read out: hand it back before the last promotion
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[slot.idx]);
          }
#pragma unroll
          for (int i = 0; i < 32; i += 2)
            promote2(acc[c + i], acc[c + i + 1], __uint_as_float(r[i]), __uint_as_float(r[i + 1]),
                     sa, sb);
        }
        sa = sa_next;
        sb = sb_next;
        slot.advance();
      }
      const int64_t colt = static_cast<int64_t>(n_blk) * BN;
      if (row_ok) {
#pragma unroll
        for (int c = 0; c < BN; c += 32)
          if (colt + c < p.N) store_chunk(p, row, colt + c, acc + c);
      }
    }
  }

  tmem_teardown(warp, tmem_base, kTmemCols);
}

// ---- act_quant ------------------------------------------------------------------------------
__device__ __forceinline__ float div_full(float a, float b) {
  float r;
  asm("div.full.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
// two floats -> two e4m3 bytes (lo in the low byte)
__device__ __forceinline__ uint32_t cvt_e4m3x2(float lo, float hi) {
  uint16_t r;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(r) : "f"(hi), "f"(lo));
  return r;
}

template <int DT>
__global__ void __launch_bounds__(256)
act_quant_kernel(const void* __restrict__ x, uint8_t* __restrict__ y, float* __restrict__ s,
                 int64_t nblocks) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
  for (int64_t b = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
       b < nblocks; b += nwarps) {
    const int64_t idx = b * 128 + lane * 4;
    float v[4];
    if constexpr (DT == LLMC_F32) {
      const float4 f = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(x) + idx));
      v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
    } else {
      const uint2 u = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const uint16_t*>(x) + idx));
      const uint32_t w[2] = {u.x, u.y};
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        if constexpr (DT == LLMC_BF16) {
          v[2 * i] = __uint_as_float(w[i] << 16);
          v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
        } else {
          const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
          v[2 * i] = f.x;
          v[2 * i + 1] = f.y;
        }
      }
    }
    float amax = fmaxf(fmaxf(fabsf(v[0]), fabsf(v[1])), fmaxf(fabsf(v[2]), fabsf(v[3])));
    amax = warp_max(amax);
    const float sc = div_full(amax, 448.f);
    const uint32_t lo = cvt_e4m3x2(div_full(v[0], sc), div_full(v[1], sc));
    const uint32_t hi = cvt_e4m3x2(div_full(v[2], sc), div_full(v[3], sc));
    *reinterpret_cast<uint32_t*>(y + idx) = lo | (hi << 16);
    if (lane == 0) s[b] = sc;
  }
}

}  // namespace fp8g
}  // namespace llmc

using namespace llmc;

extern "C" int llmc_fp8_act_quant(const void* x, int64_t M, int64_t K, int dtype, void* y,
                                  float* s, void* stream) {
  LLMC_CHECK_ARG(M >= 0 && K > 0, "fp8_act_quant: bad shape (M=%lld K=%lld)", (long long)M,
                 (long long)K);
  LLMC_CHECK_ARG(K % 128 == 0, "fp8_act_quant: K=%lld must be a multiple of 128", (long long)K);
  LLMC_CHECK_ARG(dtype == LLMC_F32 || dtype == LLMC_F16 || dtype == LLMC_BF16,
                 "fp8_act_quant: dtype must be fp32, fp16 or bf16");
  if (M == 0) return LLMC_OK;
  LLMC_CHECK_ARG(x && y && s, "fp8_act_quant: null pointer");
  if (!aligned16(x) || (reinterpret_cast<uintptr_t>(y) & 3u) != 0) {
    set_last_error("fp8_act_quant: x must be 16-byte and y 4-byte aligned");
    return LLMC_EALIGN;
  }
  const int64_t nblocks = M * (K / 128);
  int64_t grid = (nblocks + 7) / 8;
  if (grid > 16 * kNumSMs) grid = 16 * kNumSMs;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* yb = static_cast<uint8_t*>(y);
  if (dtype == LLMC_F32)
    fp8g::act_quant_kernel<LLMC_F32><<<(unsigned)grid, 256, 0, st>>>(x, yb, s, nblocks);
  else if (dtype == LLMC_F16)
    fp8g::act_quant_kernel<LLMC_F16><<<(unsigned)grid, 256, 0, st>>>(x, yb, s, nblocks);
  else
    fp8g::act_quant_kernel<LLMC_BF16><<<(unsigned)grid, 256, 0, st>>>(x, yb, s, nblocks);
  LLMC_CHECK_LAUNCH();
  return LLMC_OK;
}

extern "C" int llmc_fp8_gemm(const void* a, const float* a_s, const void* b, const float* b_s,
                             const void* bias, int bias_dtype, void* c, int out_dtype, int64_t M,
                             int64_t N, int64_t K, void* stream) {
  using namespace fp8g;
  LLMC_CHECK_ARG(M >= 0 && N >= 0 && K > 0, "fp8_gemm: bad shape (M=%lld N=%lld K=%lld)",
                 (long long)M, (long long)N, (long long)K);
  LLMC_CHECK_ARG(K % 128 == 0, "fp8_gemm: K=%lld must be a multiple of 128", (long long)K);
  LLMC_CHECK_ARG(out_dtype == LLMC_F32 || out_dtype == LLMC_F16 || out_dtype == LLMC_BF16,
                 "fp8_gemm: out_dtype must be fp32, fp16 or bf16");
  LLMC_CHECK_ARG(bias == nullptr || out_dtype == LLMC_BF16,
                 "fp8_gemm: bias needs a bf16 output (y = bf16(acc); y += bias)");
  LLMC_CHECK_ARG(bias == nullptr || bias_dtype == LLMC_F32 || bias_dtype == LLMC_BF16,
                 "fp8_gemm: bias_dtype must be fp32 or bf16");
  if (M == 0 || N == 0) return LLMC_OK;
  LLMC_CHECK_ARG(a && a_s && b && b_s && c, "fp8_gemm: null pointer");
  if (!aligned16(a) || !aligned16(b)) {
    set_last_error("fp8_gemm: A and B must be 16-byte aligned");
    return LLMC_EALIGN;
  }
  CUtensorMap tmA, tmB;
  if (int rc = encode_tmap_2d(&tmA, a, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, M, K, K, BM, BK,
                              CU_TENSOR_MAP_SWIZZLE_128B))
    return rc;
  if (int rc = encode_tmap_2d(&tmB, b, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, N, K, K, BN, BK,
                              CU_TENSOR_MAP_SWIZZLE_128B))
    return rc;
  Params p{};
  p.M = M; p.N = N; p.K = K;
  p.a_s = a_s; p.b_s = b_s; p.out = c; p.bias = bias;
  p.out_dtype = out_dtype; p.bias_dtype = bias_dtype;
  p.kb_total = static_cast<int>(K / BK);
  p.n_tiles_n = static_cast<int>((N + BN - 1) / BN);
  const int64_t mt = (M + BM - 1) / BM;
  LLMC_CHECK_ARG(mt * p.n_tiles_n < (1ll << 31), "fp8_gemm: too many tiles");
  p.m_tiles = static_cast<int>(mt);
  p.num_tiles = static_cast<int>(mt * p.n_tiles_n);
  p.gn = raster_group_n(static_cast<int64_t>(BN) * K, p.n_tiles_n);
  const int grid = p.num_tiles < kNumSMs ? p.num_tiles : kNumSMs;
  return launch_tc<fp8_gemm_kernel>(grid, kThreads, kSmemBytes, static_cast<cudaStream_t>(stream),
                                    tmA, tmB, p);
}
