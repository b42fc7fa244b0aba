// tc.cuh — sm_100a building blocks: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (UMMA +
// TMEM).  Hand-written inline PTX; bit layouts follow the PTX ISA "tcgen05" chapter
// (cross-checked against cute/arch/mma_sm100_desc.hpp field tables).  Also the scaffolding the
// persistent warp-specialised kernels share (gemm.cu, tf32.cu, gemm_w4.cu, gemm_fp8.cu): smem
// alignment, TMEM setup / teardown, ring positions, grouped rasterisation, the bf16 / fp16
// epilogue stores, the tensor-map encoder and the launch helper.
#pragma once

#include <cuda.h>  // CUtensorMap (types only; the driver entry point is resolved at run time)

#include "common.cuh"

namespace llmc {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n"
      ".reg .b32 rx;\n"
      ".reg .pred px;\n"
      "elect.sync rx|px, 0xffffffff;\n"
      "selp.b32 %0, 1, 0, px;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---- mbarrier ---------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Bounded wait: a protocol bug must trap (kernel error) instead of hanging the GPU.
__device__ __forceinline__ bool mbar_try_wait(uint32_t addr, uint32_t parity) {
  uint32_t done = 0;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.b32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(done)
      : "r"(addr), "r"(parity)
      : "memory");
  return done != 0;
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  if (mbar_try_wait(addr, parity)) return;
  const uint64_t t0 = globaltimer_ns();
  while (!mbar_try_wait(addr, parity)) {
    if (globaltimer_ns() - t0 > 5000000000ull) {  // 5 s: far beyond any legitimate wait
      printf("llmc_b200: mbarrier wait timed out (block %d thread %d bar %u parity %u)\n",
             blockIdx.x, threadIdx.x, addr, parity);
      __trap();
    }
  }
}

// generic-proxy writes to smem -> visible to the async proxy (UMMA / TMA reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---- TMA ----------------------------------------------------------------------------------
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tile load, completion counted in bytes on `bar`.  c0 = innermost coordinate.
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar,
                                            int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0),
        "r"(c1)
      : "memory");
}

// ---- TMEM ---------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// MMA completion -> mbarrier (implies fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::
                   "r"(smem_u32(bar))
               : "memory");
}

// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread = lane = row)
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
        "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
        "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---- UMMA descriptors ------------------------------------------------------------------------
// Shared-memory matrix descriptor (64 bit):
//   [0,14)  start address >> 4        [16,30) leading-dim byte offset >> 4
//   [32,46) stride-dim byte offset >> 4   [46,48) version = 1 (Blackwell)
//   [49,52) base offset = 0           [61,64) layout: 0 none, 2 = SWIZZLE_128B
// K-major, SWIZZLE_128B (rows of 128 B, 8-row 1024-B atoms, as written by TMA):
//   SBO = 1024 (next 8 rows), LBO unused (encoded 1).
// MN-major, SWIZZLE_128B (128-B rows hold 64 MN-contiguous elements of one K index):
//   SBO = 1024 (next 8 K indices), LBO = byte distance between 64-element MN atoms.
// 32-bit MN-major operands (tf32) are the exception: the only supported swizzled layout is
// layout type 1 = SWIZZLE_128B_BASE32B (32-byte swizzle atoms, 4-row K groups -> SBO = 512),
// written by TMA with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes,
                                                   uint32_t sbo_bytes, uint32_t layout = 2) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr >> 4) & 0x3fffu);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3fffu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3fffu) << 32;
  d |= static_cast<uint64_t>(1) << 46;  // version
  d |= static_cast<uint64_t>(layout) << 61;  // 2 = SWIZZLE_128B, 1 = SWIZZLE_128B_BASE32B
  return d;
}

// Instruction descriptor (fp32 accumulate), the same field layout for every MMA kind:
//   [4,6) D format: 1 = f32      [7,10) A format      [10,13) B format
//   [15] A major: 0 = K, 1 = MN  [16] B major         [17,23) N >> 3        [24,29) M >> 4
// Format codes per kind: kind::f16 0 = f16, 1 = bf16; kind::tf32 2 = tf32; kind::f8f6f4 0 = e4m3.
__host__ __device__ constexpr uint32_t make_idesc(int a_fmt, int b_fmt, int a_mn, int b_mn, int M,
                                                  int N) {
  return (1u << 4) | (static_cast<uint32_t>(a_fmt) << 7) | (static_cast<uint32_t>(b_fmt) << 10) |
         (static_cast<uint32_t>(a_mn) << 15) | (static_cast<uint32_t>(b_mn) << 16) |
         (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem], issued by ONE thread.  K per instruction: 16 (f16 / bf16),
// 8 (tf32), 32 (8-bit operands).
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                         uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_f8f6f4(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                            uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// ---- persistent-kernel scaffolding -------------------------------------------------------------
// Dynamic shared memory, rounded up to the 1024-byte alignment of 128B-swizzle atoms (kernels
// reserve 1024 bytes of slack for it).
__device__ __forceinline__ uint8_t* smem_align1024() {
  extern __shared__ uint8_t smem_raw[];
  return reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                    ~static_cast<uintptr_t>(1023));
}

// Called by every thread after the barriers are initialised: warp 1 allocates `ncols` TMEM
// columns, the barrier initialisation and the allocation become visible to all threads, and the
// TMEM base address is returned.  `warp` = threadIdx.x / 32.
__device__ __forceinline__ uint32_t tmem_setup(int warp, uint32_t* tmem_ptr, uint32_t ncols) {
  if (warp == 1) tmem_alloc(tmem_ptr, ncols);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  return *tmem_ptr;
}
// Called by every thread at the end: warp 1 frees the columns once all TMEM traffic is done.
__device__ __forceinline__ void tmem_teardown(int warp, uint32_t tmem_base, uint32_t ncols) {
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, ncols);
}

// Position in a ring of kN mbarrier-guarded slots: slot index and the parity of the current pass.
template <int kN>
struct Ring {
  int idx = 0;
  uint32_t phase = 0;
  __device__ __forceinline__ void advance() {
    if (++idx == kN) { idx = 0; phase ^= 1; }
  }
};

// Grouped rasterisation of an m_tiles x n_tiles output: the weights (n) are swept in groups of
// `gn` n-tiles sized to stay L2-resident (raster_group_n), all m-tiles per group, n fastest
// inside the group.  Activations are re-read once per group from HBM, weights once; n-fastest
// over the whole N would instead stream every weight through L2 once per wave of tiles.
__device__ __forceinline__ void grouped_tile(int u, int m_tiles, int n_tiles, int gn, int& m_blk,
                                             int& n_blk) {
  const int per_group = gn * m_tiles;
  const int g = u / per_group;
  const int rem = u - g * per_group;
  const int gsz = min(gn, n_tiles - g * gn);
  m_blk = rem / gsz;
  n_blk = g * gn + (rem - m_blk * gsz);
}

// ---- bf16 / fp16 epilogue ---------------------------------------------------------------------
template <bool kBf16>
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  if constexpr (kBf16) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  } else {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
}

// Columns [col0, col0 + 32) of a row of 16-bit outputs (`o` points at column col0), packed in
// pairs: four 16-byte stores when `full` (all 32 columns inside the row and the row 16-byte
// aligned), else the columns below N one by one.
__device__ __forceinline__ void store_row32_b16(uint16_t* o, const uint32_t (&pk)[16], bool full,
                                                int64_t col0, int64_t N) {
  if (full) {
#pragma unroll
    for (int i = 0; i < 16; i += 4)
      *reinterpret_cast<uint4*>(o + 2 * i) = make_uint4(pk[i], pk[i + 1], pk[i + 2], pk[i + 3]);
  } else {
#pragma unroll
    for (int i = 0; i < 32 && col0 + i < N; ++i)
      o[i] = static_cast<uint16_t>((i & 1) ? (pk[i >> 1] >> 16) : (pk[i >> 1] & 0xffffu));
  }
}

// One 32-column chunk of fp32 accumulators -> T (bf16 / fp16): columns [col0, col0 + 32) of a row
// at `o`, masked to col < N.  bias[col] (T, may be null) is added in fp32 before the single
// rounding, as F.linear does.  `ld_aligned`: rows start 16-byte aligned.
template <bool kBf16>
__device__ __forceinline__ void store_chunk_bias(uint16_t* o, const uint32_t (&r)[32],
                                                 const uint16_t* bias, int64_t col0, int64_t N,
                                                 bool ld_aligned) {
  uint32_t pk[16];
#pragma unroll
  for (int i = 0; i < 32; i += 2) {
    float v0 = __uint_as_float(r[i]), v1 = __uint_as_float(r[i + 1]);
    if (bias != nullptr) {
      if (col0 + i < N) v0 += kBf16 ? __uint_as_float(static_cast<uint32_t>(bias[col0 + i]) << 16)
                                    : __half2float(__ushort_as_half(bias[col0 + i]));
      if (col0 + i + 1 < N) v1 += kBf16 ? __uint_as_float(static_cast<uint32_t>(bias[col0 + i + 1]) << 16)
                                        : __half2float(__ushort_as_half(bias[col0 + i + 1]));
    }
    pk[i >> 1] = pack2<kBf16>(v0, v1);
  }
  store_row32_b16(o, pk, col0 + 32 <= N && ld_aligned, col0, N);
}

// Packed fp32 pair arithmetic (sm_100): (c0, c1) = fma((d0, d1) * sa, sb, (c0, c1)), with the
// product d * sa rounded on its own (mul.rn then fma.rn, never contracted into one fma).
__device__ __forceinline__ void promote2(float& c0, float& c1, float d0, float d1, float sa,
                                         float sb) {
  asm("{\n"
      ".reg .b64 d, a, b, c;\n"
      "mov.b64 d, {%2, %3};\n"
      "mov.b64 a, {%4, %4};\n"
      "mov.b64 b, {%5, %5};\n"
      "mov.b64 c, {%0, %1};\n"
      "mul.rn.f32x2 d, a, d;\n"
      "fma.rn.f32x2 c, d, b, c;\n"
      "mov.b64 {%0, %1}, c;\n"
      "}\n"
      : "+f"(c0), "+f"(c1)
      : "f"(d0), "f"(d1), "f"(sa), "f"(sb));
}

}  // namespace tc

// ---- host ------------------------------------------------------------------------------------
// Tensor map of a row-major rows x cols matrix of `elem_bytes`-byte elements with row stride
// ld_elems; box = box_cols (inner) x box_rows.  The swizzle span bounds the box's inner extent:
// box_cols * elem_bytes must be 128 for SWIZZLE_128B(_ATOM_32B), 64 for 64B, 32 for 32B.
// Encoded through the driver entry point resolved at run time (the library links no libcuda).
int encode_tmap_2d(CUtensorMap* out, const void* base, CUtensorMapDataType dtype,
                   uint32_t elem_bytes, uint64_t rows, uint64_t cols, uint64_t ld_elems,
                   uint32_t box_rows, uint32_t box_cols, CUtensorMapSwizzle swizzle);

// Weight-group width of grouped_tile: as many n-tiles as fit in ~32 MiB (L2-resident), at least
// one and at most all of them.
inline int raster_group_n(int64_t n_tile_bytes, int n_tiles_n) {
  int64_t gn = (32ll << 20) / n_tile_bytes;
  if (gn < 1) gn = 1;
  if (gn > n_tiles_n) gn = n_tiles_n;
  return static_cast<int>(gn);
}

// Launch a tcgen05 kernel on `grid` CTAs: the first launch on each device opts in to `smem` bytes
// of dynamic shared memory (one flag per kernel instantiation), and every launch is counted.
template <auto kKernel, typename... Args>
int launch_tc(int grid, int threads, int smem, cudaStream_t st, const Args&... args) {
  LLMC_ONCE_PER_DEVICE({
    LLMC_CHECK_CUDA(cudaFuncSetAttribute(kKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  });
  kKernel<<<grid, threads, smem, st>>>(args...);
  LLMC_CHECK_LAUNCH();
  return LLMC_OK;
}

}  // namespace llmc
