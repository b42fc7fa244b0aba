// gemm_w4.cu — K6: fake-quant forward on PACKED INT4 weights, dequantisation fused into the
// tcgen05 operand pipeline.
//
//   Y[M,N] = X[M,K] . dequant(Wq)[N,K]^T (+ bias),   dequant(n,k) = rT( fp32((code - zero) * scale) )
//
// which is bit-for-bit the bf16/fp16 weight the reference materialises in FakeQuantLinear /
// EffcientFakeQuantLinear (llmc/compression/quantization/module_utils.py:626-643, 722-741) before
// F.linear — so the result equals llmc_gemm_bf16 on that materialised weight exactly (same tile
// shape, same K order), while the weight stream from HBM is 4.25 bits instead of 16 per element.
//
// Pipeline per 64-deep K step, TWO rings so that the TMA latency is covered by a deep, cheap ring
// and the dequantised tile by a short one:
//   ring L (4 x 24 KB): X tile [128 x 64] bf16 (swizzle 128B) + packed W tile [256 x 8] int32
//   ring B (3 x 32 KB): the dequantised, 128B-swizzled UMMA B tile
//   warp 0       TMA into ring L
//   warps 6..13  dequant, two groups of four warps on alternate K steps (two weight rows per
//                thread): nibble -> fp32 via the 2^23 magic constant,
//                (q - z) * s in fp32, round to bf16/fp16, 16-byte stores into ring B,
//                fence.proxy.async; the group's scale/zero for the NEXT step is prefetched
//   warp 1       MMA issuer (tcgen05.mma kind::f16, 128 x 256 x 16, fp32 accumulators in TMEM);
//                its commit frees the ring-L stage (X consumed) and the ring-B stage
//   warps 2..5   epilogue (tcgen05.ld -> bias -> bf16/fp16 -> global, the store of gemm.cu),
//                double-buffered TMEM
// The scaffolding (TMEM setup, rings, rasterisation, epilogue stores, launch) comes from tc.cuh.
// Weight layout: LLMC_OUT_PACK_VLLM of UNSIGNED codes — 8 nibbles per int32 along K, nibble i =
// element 8*w + i; scales / zeros fp32 [N, K/group] (zeros NULL => 2^(bit-1), the symmetric
// +8 offset of module_utils.py:842-844).
#include <stdlib.h>

#include "tc.cuh"

namespace llmc {

using namespace tc;

namespace w4 {

constexpr int BM = 128, BN = 256, BK = 64;
// Two groups of four dequant warps take alternate K steps (see the kernel).  (A four-group
// variant was tried in round 2 on the theory that the per-thread unpack chain, not issue
// bandwidth, limits the kernel: it was slower, 728 vs 871 TFLOP/s, and was removed.)
constexpr int NG = 2;
constexpr int kThreads = (6 + 4 * NG) * 32;
constexpr int kBStages = 3;                    // ring B (dequantised W tile)
constexpr int kABytes = BM * BK * 2;          // 16 KB
constexpr int kBBytes = BN * BK * 2;          // 32 KB dequantised
constexpr int kTmemCols = 512;
// per weight width: INT4 -> 8 KB packed tile, 4-deep ring L; INT8 -> 16 KB packed tile, 3-deep
template <int kBits> struct Cfg {
  static constexpr int kPBytes = BN * BK * kBits / 8;
  static constexpr int kLBytes = kABytes + kPBytes;
  static constexpr int kLStages = kBits == 4 ? 4 : 3;
  static constexpr int kSmemBytes = kLStages * kLBytes + kBStages * kBBytes + 1024 + 256;
  static constexpr int kWordsPerRow = BK * kBits / 32;      // int32 per row of the packed tile
};

struct Params {
  int64_t M, N, K;
  void* out;
  const void* bias;
  const void* scales;       // [N, ng] fp32, or `dtype` when qparam_native
  const void* zeros;        // [N, ng] or null
  int qparam_native;        // qparams are in the activation dtype: packed half2 / bf16x2 dequant
  int q_transposed;         // qparams stored [ng, N] (a warp's 32 rows = one coalesced segment)
  int64_t group;
  int ng;
  float zero_default;
  int n_tiles_n, num_units, kb_total, gn;
};

__device__ __forceinline__ void decode(const Params& p, int u, int& m_blk, int& n_blk) {
  grouped_tile(u, p.num_units / p.n_tiles_n, p.n_tiles_n, p.gn, m_blk, n_blk);
}

// (a & b) | c in one LOP3
__device__ __forceinline__ uint32_t and_or(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}

// ((x2 - zm2) * s2) on two packed 16-bit floats; the subtraction is exact (small integers), the
// product of two T values rounds once — the same value as rT(fp32((q - z) * s)).
template <bool kBf16>
__device__ __forceinline__ uint32_t sub_mul2(uint32_t x2, uint32_t zm2, uint32_t s2) {
  if constexpr (kBf16) {
    const __nv_bfloat162 r = __hmul2(__hsub2(*reinterpret_cast<__nv_bfloat162*>(&x2),
                                             *reinterpret_cast<__nv_bfloat162*>(&zm2)),
                                     *reinterpret_cast<__nv_bfloat162*>(&s2));
    return *reinterpret_cast<const uint32_t*>(&r);
  } else {
    const __half2 r = __hmul2(__hsub2(*reinterpret_cast<__half2*>(&x2), *reinterpret_cast<__half2*>(&zm2)),
                              *reinterpret_cast<__half2*>(&s2));
    return *reinterpret_cast<const uint32_t*>(&r);
  }
}

template <bool kBf16, int kBits>
__global__ void __launch_bounds__(kThreads, 1)
w4a16_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmP,
                  const Params p) {
  using C = Cfg<kBits>;
  constexpr int kLStages = C::kLStages;
  constexpr int kLBytes = C::kLBytes;
  uint8_t* smem = smem_align1024();
  uint8_t* ringL = smem;
  uint8_t* ringB = smem + kLStages * kLBytes;
  uint64_t* fullL = reinterpret_cast<uint64_t*>(ringB + kBStages * kBBytes);
  uint64_t* emptyL = fullL + kLStages;
  uint64_t* readyB = emptyL + kLStages;          // dequantised B tile written
  uint64_t* emptyB = readyB + kBStages;
  uint64_t* tmem_full = emptyB + kBStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmP);
    for (int s = 0; s < kLStages; ++s) {
      mbar_init(&fullL[s], 1);
      mbar_init(&emptyL[s], 1 + 4);                   // MMA commit (X) + the step's dequant group (4 warps)
    }
    for (int s = 0; s < kBStages; ++s) {
      mbar_init(&readyB[s], 4);
      mbar_init(&emptyB[s], 1);
    }
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], 4); }
    fence_barrier_init();
  }
  const uint32_t tmem_base = tmem_setup(warp, tmem_ptr, kTmemCols);

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      Ring<kLStages> sl;
      for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
        int m_blk, n_blk;
        decode(p, u, m_blk, n_blk);
        for (int kb = 0; kb < p.kb_total; ++kb) {
          mbar_wait(&emptyL[sl.idx], sl.phase ^ 1);
          uint8_t* a_dst = ringL + sl.idx * kLBytes;
          uint8_t* p_dst = a_dst + kABytes;
          mbar_expect_tx(&fullL[sl.idx], kLBytes);
          tma_load_2d(a_dst, &tmA, &fullL[sl.idx], kb * BK, m_blk * BM);
          tma_load_2d(p_dst, &tmP, &fullL[sl.idx], kb * C::kWordsPerRow, n_blk * BN);
          sl.advance();
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc = make_idesc(kBf16, kBf16, 0, 0, BM, BN);
    Ring<kLStages> sl;
    Ring<kBStages> sb;
    Ring<2> acc;
    for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
      mbar_wait(&tmem_empty[acc.idx], acc.phase ^ 1);
      tcgen05_fence_after();
      const uint32_t d_tmem = tmem_base + acc.idx * BN;
      for (int kb = 0; kb < p.kb_total; ++kb) {
        mbar_wait(&fullL[sl.idx], sl.phase);     // X tile landed
        mbar_wait(&readyB[sb.idx], sb.phase);    // W tile dequantised
        tcgen05_fence_after();
        if (lane == 0) {
          const uint32_t a_addr = smem_u32(ringL + sl.idx * kLBytes);
          const uint32_t b_addr = smem_u32(ringB + sb.idx * kBBytes);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint64_t adesc = make_smem_desc(a_addr + k * 32, 16, 1024);
            const uint64_t bdesc = make_smem_desc(b_addr + k * 32, 16, 1024);
            umma_f16(d_tmem, adesc, bdesc, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&emptyL[sl.idx]);
          umma_commit(&emptyB[sb.idx]);
          if (kb == p.kb_total - 1) umma_commit(&tmem_full[acc.idx]);
        }
        __syncwarp();
        sl.advance();
        sb.advance();
      }
      acc.advance();
    }
  } else if (warp >= 6) {
    // ===================== dequant warps (4 * NG): two weight rows per thread =====================
    // NG groups of four warps take every NG-th K step.  A thread's unpack -> convert -> store chain
    // for its 128 weights of a tile is ~2300 cycles of dependent latency (round-2 finding: with two
    // groups the kernel ran at exactly one tile per two such chains, tensor pipe 44 % active, while
    // only half of the issue slots were used) — more groups in flight, not more instructions per
    // clock, is what hides it.
    const int grp = (warp - 6) % NG;
    const int tig = ((warp - 6) / NG) * 32 + lane;   // 0..127 inside the group
    uint32_t it = 0;                                 // K steps issued so far (all tiles)
    // raw group qparams of row n, group gi (no arithmetic on the loaded values here: the loads
    // must stay in flight while the current step is dequantised)
    // RAW bits of (scale, zero) — widening / arithmetic happens at use (widen below), so the two
    // loads stay in flight across a whole K step
    auto load_qparams = [&](int64_t n, int gi, uint32_t& s, uint32_t& z) {
      s = 0u; z = 0u;
      if (n >= p.N) return;
      const int64_t qi = p.q_transposed ? static_cast<int64_t>(gi) * p.N + n : n * p.ng + gi;
      if (p.qparam_native) {
        s = __ldg(&reinterpret_cast<const uint16_t*>(p.scales)[qi]);
        if (p.zeros != nullptr) z = __ldg(&reinterpret_cast<const uint16_t*>(p.zeros)[qi]);
      } else {
        s = __ldg(&reinterpret_cast<const uint32_t*>(p.scales)[qi]);
        if (p.zeros != nullptr) z = __ldg(&reinterpret_cast<const uint32_t*>(p.zeros)[qi]);
      }
    };
    auto widen = [&](uint32_t raw) -> float {
      if (!p.qparam_native) return __uint_as_float(raw);
      return kBf16 ? __uint_as_float(raw << 16) : __half2float(__ushort_as_half(static_cast<uint16_t>(raw)));
    };
    const bool have_zeros = p.zeros != nullptr;
    const int steps_per_group = static_cast<int>(p.group / BK);
    for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
      int m_blk, n_blk;
      decode(p, u, m_blk, n_blk);
      const int64_t n0 = static_cast<int64_t>(n_blk) * BN + tig;
      // first K step of this tile that belongs to this group: (it + kb) % NG == grp
      int kb = (grp + NG - static_cast<int>(it % NG)) % NG;
      uint32_t s_cur[2] = {0u, 0u}, z_cur[2] = {0u, 0u};
      if (kb < p.kb_total) {
#pragma unroll
        for (int h = 0; h < 2; ++h) load_qparams(n0 + h * 128, kb / steps_per_group, s_cur[h], z_cur[h]);
      }
      for (; kb < p.kb_total; kb += NG) {
        const uint32_t my = it + kb;
        const int sl = my % kLStages, sb = my % kBStages;
        const uint32_t phl = (my / kLStages) & 1u, phb = (my / kBStages) & 1u;
        // qparams of this group's NEXT step are requested now and consumed next iteration
        uint32_t s_nxt[2] = {s_cur[0], s_cur[1]}, z_nxt[2] = {z_cur[0], z_cur[1]};
        if (kb + NG < p.kb_total && (kb + NG) / steps_per_group != kb / steps_per_group) {
#pragma unroll
          for (int h = 0; h < 2; ++h)
            load_qparams(n0 + h * 128, (kb + NG) / steps_per_group, s_nxt[h], z_nxt[h]);
        }
        mbar_wait(&fullL[sl], phl);
        mbar_wait(&emptyB[sb], phb ^ 1);
        const uint8_t* pk = ringL + sl * kLBytes + kABytes;
        uint8_t* bt = ringB + sb * kBBytes;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int row = tig + h * 128;
          const float z_c = have_zeros ? widen(z_cur[h]) : p.zero_default;
          const float zm_cur = 8388608.0f + z_c;        // (2^23 + q) - (2^23 + z) = q - z exactly
          const float s_c = (n0 + h * 128 < p.N) ? widen(s_cur[h]) : 0.f;
          if constexpr (kBits == 8) {
            // INT8: 64-byte rows, TMA SWIZZLE_64B: 16-byte chunk c of row r sits at c ^ ((r >> 1) & 3).
            // byte -> fp32 through the 2^23 magic (0x4B0000nn), (q - z) * s in fp32, one rounding;
            // bf16 has no exact packed form for 8-bit codes (128 + q needs 9 bits), so both qparam
            // flavours take this path (same value: the product of two T numbers rounds once).
            const int sw8 = (row >> 1) & 3;
#pragma unroll
            for (int c4 = 0; c4 < 4; ++c4) {
              const uint4 wv = *reinterpret_cast<const uint4*>(pk + row * 64 + ((c4 ^ sw8) << 4));
              const uint32_t wd[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
              for (int hh = 0; hh < 2; ++hh) {
                float v[8];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  v[j] = fmul_rn(__uint_as_float(__byte_perm(wd[2 * hh], 0x4B000000u, 0x7650u + j)) - zm_cur, s_c);
                  v[4 + j] = fmul_rn(__uint_as_float(__byte_perm(wd[2 * hh + 1], 0x4B000000u, 0x7650u + j)) - zm_cur, s_c);
                }
                const uint4 o = make_uint4(pack2<kBf16>(v[0], v[1]), pack2<kBf16>(v[2], v[3]),
                                           pack2<kBf16>(v[4], v[5]), pack2<kBf16>(v[6], v[7]));
                const int c = c4 * 2 + hh;
                *reinterpret_cast<uint4*>(bt + row * 128 + ((c ^ (row & 7)) << 4)) = o;
              }
            }
            continue;
          }
          // packed tile is TMA-swizzled (32B): half h of row r sits at half h ^ ((r >> 2) & 1)
          const int sw = ((row >> 2) & 1) << 4;
          const uint4 w0 = *reinterpret_cast<const uint4*>(pk + row * 32 + sw);
          const uint4 w1 = *reinterpret_cast<const uint4*>(pk + row * 32 + (sw ^ 16));
          const uint32_t words[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
          if (p.qparam_native) {
            // packed path: 0x6400|q = 1024+q (fp16) / 0x4300|q = 128+q (bf16), two weights per
            // register; (magic+q) - (magic+z) and * s are one HSUB2 + one HMUL2 per pair
            constexpr uint32_t kMagic2 = kBf16 ? 0x43004300u : 0x64006400u;
            const uint32_t s2 = pack2<kBf16>(s_c, s_c);                          // exact: s is a T value
            const uint32_t zm2 = pack2<kBf16>((kBf16 ? 128.f : 1024.f) + z_c,
                                              (kBf16 ? 128.f : 1024.f) + z_c);        // exact: <= 8 bits
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              const uint32_t w = words[c];
              // element pairs (0,4) (1,5) (2,6) (3,7): nibble i in the low half, nibble i+4 in the high
              const uint32_t r04 = sub_mul2<kBf16>(and_or(w, 0x000F000Fu, kMagic2), zm2, s2);
              const uint32_t r15 = sub_mul2<kBf16>(and_or(w >> 4, 0x000F000Fu, kMagic2), zm2, s2);
              const uint32_t r26 = sub_mul2<kBf16>(and_or(w >> 8, 0x000F000Fu, kMagic2), zm2, s2);
              const uint32_t r37 = sub_mul2<kBf16>(and_or(w >> 12, 0x000F000Fu, kMagic2), zm2, s2);
              const uint4 o = make_uint4(__byte_perm(r04, r15, 0x5410), __byte_perm(r26, r37, 0x5410),
                                         __byte_perm(r04, r15, 0x7632), __byte_perm(r26, r37, 0x7632));
              // K-major SWIZZLE_128B: 16-byte chunk c of row r lives at chunk (c ^ (r & 7))
              *reinterpret_cast<uint4*>(bt + row * 128 + ((c ^ (row & 7)) << 4)) = o;
            }
          } else {
#pragma unroll
            for (int c = 0; c < 8; ++c) {            // one 16-byte chunk = 8 elements = one word
              // The integer pipe is the scarce resource (64 lanes vs 128 fp32 lanes per SM and
              // clock): split the word into even / odd nibbles once, then ONE byte-permute per
              // element builds the fp32 bit pattern 0x4B0000nn = 2^23 + nibble.
              const uint32_t w = words[c];
              const uint32_t ev = w & 0x0F0F0F0Fu;           // nibbles 0,2,4,6 in bytes 0..3
              const uint32_t od = (w >> 4) & 0x0F0F0F0Fu;    // nibbles 1,3,5,7
              float v[8];
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const uint32_t be = __byte_perm(ev, 0x4B000000u, 0x7650u + j);
                const uint32_t bo = __byte_perm(od, 0x4B000000u, 0x7650u + j);
                v[2 * j] = fmul_rn(__uint_as_float(be) - zm_cur, s_c);
                v[2 * j + 1] = fmul_rn(__uint_as_float(bo) - zm_cur, s_c);
              }
              const uint4 o = make_uint4(pack2<kBf16>(v[0], v[1]), pack2<kBf16>(v[2], v[3]),
                                         pack2<kBf16>(v[4], v[5]), pack2<kBf16>(v[6], v[7]));
              *reinterpret_cast<uint4*>(bt + row * 128 + ((c ^ (row & 7)) << 4)) = o;
            }
          }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(&readyB[sb]);
          mbar_arrive(&emptyL[sl]);                // packed tile consumed
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) { s_cur[h] = s_nxt[h]; z_cur[h] = z_nxt[h]; }
      }
      it += static_cast<uint32_t>(p.kb_total);
    }
  } else {
    // ===================== epilogue (warps 2..5) =====================
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
        if (row < p.M && col0 < p.N)
          store_chunk_bias<kBf16>(reinterpret_cast<uint16_t*>(p.out) + row * p.N + col0, r,
                                  reinterpret_cast<const uint16_t*>(p.bias), col0, p.N,
                                  (p.N & 7) == 0);
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc.idx]);
      acc.advance();
    }
  }
  tmem_teardown(warp, tmem_base, kTmemCols);
}

}  // namespace w4
}  // namespace llmc

using namespace llmc;

template <int kBits>
static int gemm_wNa16(const void* x, const int32_t* wq, const void* scales, const void* zeros,
                      int qparam_dtype, const void* bias, void* y, int64_t M, int64_t N, int64_t K,
                      int64_t group, int dtype, int q_transposed, void* stream, const char* name) {
  using namespace w4;
  LLMC_CHECK_ARG(M >= 0 && N >= 0 && K > 0, "%s: bad shape", name);
  if (M == 0 || N == 0) return LLMC_OK;
  LLMC_CHECK_ARG(x && wq && scales && y, "%s: null pointer", name);
  LLMC_CHECK_ARG(dtype == LLMC_BF16 || dtype == LLMC_F16, "%s: dtype must be bf16 or fp16", name);
  LLMC_CHECK_ARG(qparam_dtype == LLMC_F32 || qparam_dtype == dtype,
                 "%s: qparam_dtype must be fp32 or the activation dtype", name);
  LLMC_CHECK_ARG(group > 0 && K % group == 0 && group % BK == 0,
                 "%s: group %lld must divide K=%lld and be a multiple of %d", name, (long long)group,
                 (long long)K, BK);
  if (K % 64 != 0 || !aligned16(x) || !aligned16(wq) || !aligned16(y)) {
    set_last_error("%s: K=%lld must be a multiple of 64 and pointers 16-byte aligned", name, (long long)K);
    return LLMC_EALIGN;
  }
  using C = Cfg<kBits>;
  CUtensorMap tmA, tmP;
  if (int rc = encode_tmap_2d(&tmA, x, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, M, K, K, BM, BK,
                              CU_TENSOR_MAP_SWIZZLE_128B))
    return rc;
  // packed rows of 32 B (INT4) / 64 B (INT8): the 32B / 64B swizzle makes the dequant warps'
  // one-row-per-thread 16-byte shared-memory loads conflict free
  if (int rc = encode_tmap_2d(&tmP, wq, CU_TENSOR_MAP_DATA_TYPE_INT32, 4, N, K * kBits / 32,
                              K * kBits / 32, BN, C::kWordsPerRow,
                              kBits == 4 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_64B))
    return rc;
  Params p{};
  p.M = M; p.N = N; p.K = K; p.out = y; p.bias = bias;
  p.scales = scales; p.zeros = zeros;
  // packed half2 / bf16x2 dequant exists for INT4 only; INT8 widens native qparams to fp32
  p.qparam_native = (qparam_dtype != LLMC_F32) ? 1 : 0;
  p.q_transposed = q_transposed ? 1 : 0;
  p.group = group; p.ng = static_cast<int>(K / group);
  p.zero_default = static_cast<float>(1 << (kBits - 1));
  p.n_tiles_n = static_cast<int>((N + BN - 1) / BN);
  const int64_t mt = (M + BM - 1) / BM;
  LLMC_CHECK_ARG(mt * p.n_tiles_n < (1ll << 31), "%s: too many tiles", name);
  p.num_units = static_cast<int>(mt * p.n_tiles_n);
  p.kb_total = static_cast<int>(K / BK);
  p.gn = raster_group_n(static_cast<int64_t>(BN) * K * kBits / 8, p.n_tiles_n);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  constexpr int smem = C::kSmemBytes;
  static_assert(smem <= 227 * 1024, "shared memory budget");
  const int grid = p.num_units < kNumSMs ? p.num_units : kNumSMs;
  return dtype == LLMC_BF16 ? launch_tc<w4a16_gemm_kernel<true, kBits>>(grid, kThreads, smem, st, tmA, tmP, p)
                            : launch_tc<w4a16_gemm_kernel<false, kBits>>(grid, kThreads, smem, st, tmA, tmP, p);
}


extern "C" int llmc_gemm_w4a16(const void* x, const int32_t* wq, const void* scales,
                               const void* zeros, int qparam_dtype, const void* bias, void* y,
                               int64_t M, int64_t N, int64_t K, int64_t group, int dtype,
                               void* stream) {
  // `group` < 0 selects the TRANSPOSED qparam layout [K/|group|, N] (coalesced per-warp loads)
  return gemm_wNa16<4>(x, wq, scales, zeros, qparam_dtype, bias, y, M, N, K, group < 0 ? -group : group,
                       dtype, group < 0, stream, "gemm_w4a16");
}

// INT8 weights: wq [N, K/4] int32, 4 UNSIGNED codes per word along K (code + 128 for symmetric,
// zeros NULL => 128), otherwise as llmc_gemm_w4a16.
extern "C" int llmc_gemm_w8a16(const void* x, const int32_t* wq, const void* scales,
                               const void* zeros, int qparam_dtype, const void* bias, void* y,
                               int64_t M, int64_t N, int64_t K, int64_t group, int dtype,
                               void* stream) {
  return gemm_wNa16<8>(x, wq, scales, zeros, qparam_dtype, bias, y, M, N, K, group < 0 ? -group : group,
                       dtype, group < 0, stream, "gemm_w8a16");
}
