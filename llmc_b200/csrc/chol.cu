// chol.cu — K4: U = cholesky(cholesky_inverse(cholesky(H)), upper)  (gptq.py:172-174) as ONE
// reverse-ordered blocked factorisation + ONE blocked triangular inverse.
//
// Identity used (DESIGN.md §K4): let J be the index reversal and G = J H J = L L^T (lower
// Cholesky).  Then H = (J L J)(J L J)^T with R = J L J upper triangular, so H^-1 = R^-T R^-1 and
// the unique upper factor with positive diagonal is U = R^-1 = J L^-1 J, i.e.
//        U[i][j] = (L^-1)[n-1-i][n-1-j].
// Work: C^3/3 (factor) + C^3/3 (inverse) flops instead of the reference's potrf + potri + potrf
// (4/3 C^3), and every O(C^3) part is a 128-deep rank update executed by the 3xTF32 tensor-core
// kernel of tf32.cu (fp32-accurate); only the 128x128 diagonal blocks run on CUDA cores.
#include <vector>

#include "tc.cuh"
#include "tf32.cuh"

namespace llmc {
namespace ch {

constexpr int NB = 128;
constexpr int LDS = NB + 1;

__device__ __forceinline__ float tf32r(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

// G[i][j] = H[n-1-i][n-1-j]
__global__ void __launch_bounds__(256)
reverse_kernel(const float* __restrict__ H, float* __restrict__ G, int64_t n) {
  const int64_t total = n * n;
  for (int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    G[idx] = H[total - 1 - idx];
  }
}

// U[i][j] = j >= i ? Y[n-1-i][n-1-j] : 0
__global__ void __launch_bounds__(256)
reverse_upper_kernel(const float* __restrict__ Y, float* __restrict__ U, int64_t n) {
  const int64_t total = n * n;
  for (int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t i = idx / n, j = idx - i * n;
    U[idx] = (j >= i) ? Y[total - 1 - idx] : 0.f;
  }
}

// One CTA: factor the nb x nb diagonal block at G[k0][k0] (lower), invert the factor.
//   G block <- L_kk (lower part), D <- L_kk^-1 (nb x nb, row-major, ld NB, zero above the diagonal
//   and zero padded to 128), Dhi/Dlo its tf32 split.  info[0] = k0 + j + 1 on a non-positive pivot.
__global__ void __launch_bounds__(256, 1)
diag_kernel(float* __restrict__ G, int64_t n, int64_t k0, int nb, float* __restrict__ D,
            float* __restrict__ Dhi, float* __restrict__ Dlo, int* __restrict__ info) {
  extern __shared__ float sm[];
  float* S = sm;                 // [NB][LDS] the block / L
  float* X = sm + NB * LDS;      // [NB][LDS] L^-1
  const int tid = threadIdx.x;
  for (int idx = tid; idx < NB * NB; idx += 256) {
    const int i = idx >> 7, j = idx & 127;
    float v = 0.f;
    if (i < nb && j < nb && j <= i) v = G[(k0 + i) * n + k0 + j];
    S[i * LDS + j] = v;
    X[i * LDS + j] = 0.f;
  }
  __syncthreads();
  // Left-looking column Cholesky: thread i owns row i (conflict-free padded rows, row j is a
  // broadcast read).  L[i][j] = (A[i][j] - sum_{k<j} L[i][k] L[j][k]) / L[j][j].
  {
    const int i = tid;
    for (int j = 0; j < nb; ++j) {
      float v = 0.f;
      if (i >= j && i < nb) {
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        const float* ri = S + i * LDS;
        const float* rj = S + j * LDS;
        int k = 0;
        for (; k + 3 < j; k += 4) {
          a0 = fmaf(ri[k], rj[k], a0);
          a1 = fmaf(ri[k + 1], rj[k + 1], a1);
          a2 = fmaf(ri[k + 2], rj[k + 2], a2);
          a3 = fmaf(ri[k + 3], rj[k + 3], a3);
        }
        for (; k < j; ++k) a0 = fmaf(ri[k], rj[k], a0);
        v = ri[j] - ((a0 + a1) + (a2 + a3));
      }
      // (column j is only written below; the dot products above read columns < j, final already)
      if (i == j) {
        if (!(v > 0.f) && info[0] == 0) info[0] = static_cast<int>(k0) + j + 1;
        S[j * LDS + j] = sqrtf(fmaxf(v, 1e-30f));
      }
      __syncthreads();
      if (i > j && i < nb) S[i * LDS + j] = v / S[j * LDS + j];
      // row j+1's column j is written by thread j+1 and read by all in the next iteration
      __syncthreads();
    }
  }
  // X = L^-1: thread c owns column c (unit-stride across threads), forward substitution with
  // four partial sums per entry to break the FMA dependency chain
  if (tid < nb) {
    const int c = tid;
    X[c * LDS + c] = 1.0f / S[c * LDS + c];
    for (int i = c + 1; i < nb; ++i) {
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
      const float* ri = S + i * LDS;
      int k = c;
      for (; k + 3 < i; k += 4) {
        a0 = fmaf(ri[k], X[k * LDS + c], a0);
        a1 = fmaf(ri[k + 1], X[(k + 1) * LDS + c], a1);
        a2 = fmaf(ri[k + 2], X[(k + 2) * LDS + c], a2);
        a3 = fmaf(ri[k + 3], X[(k + 3) * LDS + c], a3);
      }
      for (; k < i; ++k) a0 = fmaf(ri[k], X[k * LDS + c], a0);
      X[i * LDS + c] = -((a0 + a1) + (a2 + a3)) / ri[i];
    }
  }
  __syncthreads();
  for (int idx = tid; idx < NB * NB; idx += 256) {
    const int i = idx >> 7, j = idx & 127;
    if (i < nb && j < nb && j <= i) G[(k0 + i) * n + k0 + j] = S[i * LDS + j];
    const float x = X[i * LDS + j];
    D[idx] = x;
    const float h = tf32r(x);
    Dhi[idx] = h;
    Dlo[idx] = tf32r(x - h);
  }
}

// ---- diag_kernel_v2: the same contract as diag_kernel, blocked by 32 ------------------------------
// The v1 kernel above is one long sequential sweep whose shared-memory traffic (two LDS per FMA,
// 2-way conflicts in the inverse) made it 180 us per block — 11 % of a calibration step.  v2 factors
// 32x32 diagonal sub-blocks in registers (warp shuffles), solves the sub-panel with one thread per
// row in registers, applies the trailing update with 4x4 register tiles, and builds L^-1 from 32x32
// block products (X_ij = -X_ii * sum_k L_ik X_kj).  Rows/cols >= nb are padded with the identity so
// every loop runs at the full 128.
constexpr int SBK = 32;

__global__ void __launch_bounds__(256, 1)
diag_kernel_v2(float* __restrict__ G, int64_t n, int64_t k0, int nb, float* __restrict__ Y,
               float* __restrict__ Yhi, float* __restrict__ Ylo, int* __restrict__ info) {
  extern __shared__ float sm[];
  float* S = sm;                 // [NB][LDS]
  float* X = sm + NB * LDS;      // [NB][LDS]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  __shared__ __align__(16) float colbuf[SBK];
  __shared__ float rinv[NB];
  {
    // 64 elements per thread, 16 independent loads in flight at a time (the block was just
    // written by the trailing update: L2 latency, not bandwidth, is what this costs)
    const int j = tid & 127;
#pragma unroll 1
    for (int t0 = 0; t0 < NB / 2; t0 += 16) {
      float v[16];
#pragma unroll
      for (int t = 0; t < 16; ++t) {
        const int i = (tid >> 7) + 2 * (t0 + t);
        v[t] = (i == j) ? 1.f : 0.f;
        if (i < nb && j < nb) v[t] = (j <= i) ? __ldcg(G + (k0 + i) * n + k0 + j) : 0.f;
      }
#pragma unroll
      for (int t = 0; t < 16; ++t) {
        const int i = (tid >> 7) + 2 * (t0 + t);
        S[i * LDS + j] = v[t];
        X[i * LDS + j] = 0.f;
      }
    }
  }
  __syncthreads();

  // ---------------- phase A: L = chol(S), panels of 32 columns ----------------
  for (int b0 = 0; b0 < NB; b0 += SBK) {
    if (warp == 0) {                      // A1: 32x32 diagonal block, lane i = row i, in registers
      float a[SBK];
#pragma unroll
      for (int k = 0; k < SBK; ++k) a[k] = (k <= lane) ? S[(b0 + lane) * LDS + b0 + k] : 0.f;
      // Per column j the dependent chain is: broadcast a[j][j] -> rsqrt (+ one Newton step) ->
      // scale -> broadcast L[j+1][j] -> update a[j+1].  The updates of columns >= j+2 go through
      // shared memory (8 broadcast LDS.128 instead of 30 shuffles) and are consumed one
      // iteration later, so their latency is off the chain.
      float4 pend[SBK / 4];
      float lprev = 0.f;
#pragma unroll
      for (int j = 0; j < SBK; ++j) {
        const float ajj = __shfl_sync(0xffffffffu, a[j], j);
        if (!(ajj > 0.f) && lane == j && (b0 + j) < nb && info[0] == 0)
          info[0] = static_cast<int>(k0) + b0 + j + 1;
        const float ac = fmaxf(ajj, 1e-30f);
        float r = rsqrtf(ac);
        r = r * fmaf(-0.5f * ac * r, r, 1.5f);            // 1/sqrt(a), ~1 ulp
        float d = ac * r;
        d = fmaf(fmaf(-d, d, ac), 0.5f * r, d);           // sqrt(a), ~1 ulp
        const float lij = (lane > j) ? a[j] * r : ((lane == j) ? d : 0.f);
        a[j] = lij;
        if (lane == j) rinv[b0 + j] = r;                  // 1 / L[j][j] for A2 and B1
        if (j + 1 < SBK) {
          const float lnext = __shfl_sync(0xffffffffu, lij, j + 1);
          a[j + 1] = fmaf(-lij, lnext, a[j + 1]);
        }
        if (j > 0) {                                       // deferred updates of column j-1: k >= j+1
#pragma unroll
          for (int k4 = (j + 1) & ~3; k4 < SBK; k4 += 4) {
            const float4 l4 = pend[k4 / 4];
            if (k4 + 0 > j) a[k4 + 0] = fmaf(-lprev, l4.x, a[k4 + 0]);
            if (k4 + 1 > j) a[k4 + 1] = fmaf(-lprev, l4.y, a[k4 + 1]);
            if (k4 + 2 > j) a[k4 + 2] = fmaf(-lprev, l4.z, a[k4 + 2]);
            if (k4 + 3 > j) a[k4 + 3] = fmaf(-lprev, l4.w, a[k4 + 3]);
          }
        }
        if (j + 2 < SBK) {                                 // publish column j, fetch it for k >= j+2
          __syncwarp();
          colbuf[lane] = lij;
          __syncwarp();
#pragma unroll
          for (int k4 = (j + 2) & ~3; k4 < SBK; k4 += 4)
            pend[k4 / 4] = *reinterpret_cast<const float4*>(colbuf + k4);
          lprev = lij;
        }
      }
#pragma unroll
      for (int k = 0; k < SBK; ++k)
        if (k <= lane) S[(b0 + lane) * LDS + b0 + k] = a[k];
    }
    __syncthreads();
    const int nrem = NB - b0 - SBK;       // rows below the diagonal sub-block
    if (tid < nrem) {                     // A2: P = A_panel * L_kk^-T by forward substitution
      const int i = b0 + SBK + tid;
      float p[SBK];
#pragma unroll
      for (int j = 0; j < SBK; ++j) p[j] = S[i * LDS + b0 + j];
#pragma unroll
      for (int j = 0; j < SBK; ++j) {
        float acc = p[j];
#pragma unroll
        for (int k = 0; k < j; ++k) acc = fmaf(-p[k], S[(b0 + j) * LDS + b0 + k], acc);
        p[j] = acc * rinv[b0 + j];
      }
#pragma unroll
      for (int j = 0; j < SBK; ++j) S[i * LDS + b0 + j] = p[j];
    } else if (warp == 7) {
      // B1, overlapped with A2 (which occupies warps 0-2 at most): the inverse of this panel's
      // 32x32 diagonal block, lane c = column c, forward substitution in registers
      float x[SBK];
#pragma unroll
      for (int i = 0; i < SBK; ++i) {
        float acc = (i == lane) ? 1.f : 0.f;
#pragma unroll
        for (int k = 0; k < i; ++k) acc = fmaf(-S[(b0 + i) * LDS + b0 + k], x[k], acc);
        x[i] = acc * rinv[b0 + i];                        // zero for i < c (acc stays 0)
      }
#pragma unroll
      for (int i = 0; i < SBK; ++i) X[(b0 + i) * LDS + b0 + lane] = x[i];
    }
    __syncthreads();
    if (nrem > 0) {                       // A3: trailing S[i][j] -= sum_k P[i][k] P[j][k], j <= i
      const int nt = nrem >> 2;           // 4x4 tiles per side
      const int ntiles = nt * (nt + 1) / 2;
      for (int t = tid; t < ntiles; t += 256) {
        // unrank the lower-triangular tile index t -> (ti >= tj)
        int ti = static_cast<int>((sqrtf(8.f * t + 1.f) - 1.f) * 0.5f);
        while ((ti + 1) * (ti + 2) / 2 <= t) ++ti;
        while (ti * (ti + 1) / 2 > t) --ti;
        const int tj = t - ti * (ti + 1) / 2;
        const int r0 = b0 + SBK + ti * 4, c0 = b0 + SBK + tj * 4;
        float acc[4][4];
#pragma unroll
        for (int x = 0; x < 4; ++x)
#pragma unroll
          for (int y = 0; y < 4; ++y) acc[x][y] = 0.f;
#pragma unroll 8
        for (int k = 0; k < SBK; ++k) {
          float pr[4], pc[4];
#pragma unroll
          for (int x = 0; x < 4; ++x) { pr[x] = S[(r0 + x) * LDS + b0 + k]; pc[x] = S[(c0 + x) * LDS + b0 + k]; }
#pragma unroll
          for (int x = 0; x < 4; ++x)
#pragma unroll
            for (int y = 0; y < 4; ++y) acc[x][y] = fmaf(pr[x], pc[y], acc[x][y]);
        }
#pragma unroll
        for (int x = 0; x < 4; ++x)
#pragma unroll
          for (int y = 0; y < 4; ++y)
            if (c0 + y <= r0 + x) S[(r0 + x) * LDS + c0 + y] -= acc[x][y];
      }
    }
    __syncthreads();
  }

  // ---------------- phase B: X = L^-1 (the diagonal 32x32 inverses were built in phase A) ------
  // B2: off-diagonal blocks by distance d = i - j; thread (ty, tx) of a 16x16 grid owns a 2x2 patch
  {
    const int tx = tid & 15, ty = tid >> 4;
    for (int d = 1; d < NB / SBK; ++d) {
      for (int bi = d; bi < NB / SBK; ++bi) {
        const int bj = bi - d;
        const int ri = bi * SBK, cj = bj * SBK;
        // T = sum_{k=bj}^{bi-1} L[bi][k] X[k][bj]   (X[k][bj] for k > bj was produced at smaller d)
        float t00 = 0.f, t01 = 0.f, t10 = 0.f, t11 = 0.f;
        for (int kk = cj; kk < ri; ++kk) {
          const float l0 = S[(ri + 2 * ty) * LDS + kk], l1 = S[(ri + 2 * ty + 1) * LDS + kk];
          const float x0 = X[kk * LDS + cj + 2 * tx], x1 = X[kk * LDS + cj + 2 * tx + 1];
          t00 = fmaf(l0, x0, t00); t01 = fmaf(l0, x1, t01);
          t10 = fmaf(l1, x0, t10); t11 = fmaf(l1, x1, t11);
        }
        // stash T in the (still unused) X[bi][bj] block
        X[(ri + 2 * ty) * LDS + cj + 2 * tx] = t00;
        X[(ri + 2 * ty) * LDS + cj + 2 * tx + 1] = t01;
        X[(ri + 2 * ty + 1) * LDS + cj + 2 * tx] = t10;
        X[(ri + 2 * ty + 1) * LDS + cj + 2 * tx + 1] = t11;
        __syncthreads();
        // X[bi][bj] = -X[bi][bi] * T
        float o00 = 0.f, o01 = 0.f, o10 = 0.f, o11 = 0.f;
        for (int m = 0; m < SBK; ++m) {
          const float a0 = X[(ri + 2 * ty) * LDS + ri + m], a1 = X[(ri + 2 * ty + 1) * LDS + ri + m];
          const float b0v = X[(ri + m) * LDS + cj + 2 * tx], b1v = X[(ri + m) * LDS + cj + 2 * tx + 1];
          o00 = fmaf(a0, b0v, o00); o01 = fmaf(a0, b1v, o01);
          o10 = fmaf(a1, b0v, o10); o11 = fmaf(a1, b1v, o11);
        }
        __syncthreads();
        X[(ri + 2 * ty) * LDS + cj + 2 * tx] = -o00;
        X[(ri + 2 * ty) * LDS + cj + 2 * tx + 1] = -o01;
        X[(ri + 2 * ty + 1) * LDS + cj + 2 * tx] = -o10;
        X[(ri + 2 * ty + 1) * LDS + cj + 2 * tx + 1] = -o11;
        __syncthreads();
      }
    }
  }
  for (int idx = tid; idx < NB * NB; idx += 256) {
    const int i = idx >> 7, j = idx & 127;
    if (i < nb && j <= i) {
      // L_kk, and the diagonal block of Y = L^-1 with its tf32 split.  The GEMMs that multiply by
      // L_kk^-1 read it from Yhi/Ylo in place (ld n); the part above the diagonal is zero from
      // the memsets at the start of llmc_chol_inv_upper.
      const int64_t o = (k0 + i) * n + k0 + j;
      G[o] = S[i * LDS + j];
      const float x = X[i * LDS + j];
      const float h = tf32r(x);
      Y[o] = x;
      Yhi[o] = h;
      Ylo[o] = tf32r(x - h);
    }
  }
}

// copy the nb x nb block D (ld NB) into Y / Yhi / Ylo at (k0, k0)
__global__ void __launch_bounds__(256)
place_diag_kernel(const float* __restrict__ D, const float* __restrict__ Dhi,
                  const float* __restrict__ Dlo, float* __restrict__ Y, float* __restrict__ Yhi,
                  float* __restrict__ Ylo, int64_t n, int64_t k0, int nb) {
  for (int idx = threadIdx.x + blockIdx.x * blockDim.x; idx < nb * nb; idx += blockDim.x * gridDim.x) {
    const int i = idx / nb, j = idx - i * nb;
    const int64_t o = (k0 + i) * n + k0 + j;
    Y[o] = D[i * NB + j];
    Yhi[o] = Dhi[i * NB + j];
    Ylo[o] = Dlo[i * NB + j];
  }
}

}  // namespace ch
}  // namespace llmc

using namespace llmc;

extern "C" int64_t llmc_chol_workspace_bytes(int64_t C) {
  if (C <= 0) return 0;
  const int64_t nbk = (C + ch::NB - 1) / ch::NB;
  // G, Lhi, Llo, Y, Yhi, Ylo (C^2 each) + per-block D, Dhi, Dlo (128^2 each)
  return (6 * C * C + 3 * nbk * ch::NB * ch::NB) * 4 + 256;
}

extern "C" int llmc_chol_inv_upper(float* A, int64_t C, void* workspace, int64_t workspace_bytes,
                                   int* info, void* stream) {
  using namespace ch;
  LLMC_CHECK_ARG(A && workspace && info && C > 0, "chol_inv_upper: bad argument");
  LLMC_CHECK_ARG(C % 8 == 0, "chol_inv_upper: C=%lld must be a multiple of 8", (long long)C);
  LLMC_CHECK_ARG(workspace_bytes >= llmc_chol_workspace_bytes(C), "chol_inv_upper: workspace too small");
  LLMC_CHECK_ARG(aligned16(A) && aligned16(workspace), "chol_inv_upper: 16-byte alignment required");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t n = C, nn = C * C;
  const int64_t nbk = (n + NB - 1) / NB;
  float* G = reinterpret_cast<float*>(workspace);
  float* Lhi = G + nn;
  float* Llo = Lhi + nn;
  float* Y = Llo + nn;
  float* Yhi = Y + nn;
  float* Ylo = Yhi + nn;
  float* D = Ylo + nn;
  float* Dhi = D + nbk * NB * NB;
  float* Dlo = Dhi + nbk * NB * NB;
  const int diag_smem = 2 * NB * LDS * 4;
  LLMC_ONCE_PER_DEVICE({
    LLMC_CHECK_CUDA(cudaFuncSetAttribute(diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, diag_smem));
    LLMC_CHECK_CUDA(cudaFuncSetAttribute(diag_kernel_v2, cudaFuncAttributeMaxDynamicSharedMemorySize, diag_smem));
  });
  // LLMC_B200_CHOL_DIAG_V1=1: the unblocked diagonal kernel, for A/B runs
  const char* v1_env = getenv("LLMC_B200_CHOL_DIAG_V1");
  const bool use_v1 = (v1_env != nullptr && v1_env[0] == '1');
  // Side stream + events for the inverse chain (process-wide, created once; the call stays
  // asynchronous with respect to the host and ordered on `stream` through the final join).
  // (per device; one host thread per device is assumed, like everywhere in this library)
  constexpr int kMaxDev = 64;
  static cudaStream_t side_of[kMaxDev] = {};
  static cudaEvent_t join_of[kMaxDev] = {};
  static std::vector<cudaEvent_t> ev_of[kMaxDev];
  int dev_id = 0;
  LLMC_CHECK_CUDA(cudaGetDevice(&dev_id));
  dev_id &= kMaxDev - 1;
  if (side_of[dev_id] == nullptr) {
    LLMC_CHECK_CUDA(cudaStreamCreateWithFlags(&side_of[dev_id], cudaStreamNonBlocking));
    LLMC_CHECK_CUDA(cudaEventCreateWithFlags(&join_of[dev_id], cudaEventDisableTiming));
  }
  std::vector<cudaEvent_t>& ev = ev_of[dev_id];
  while (static_cast<int64_t>(ev.size()) < nbk) {
    cudaEvent_t e;
    LLMC_CHECK_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    ev.push_back(e);
  }
  cudaStream_t side = side_of[dev_id];
  cudaEvent_t ev_join = join_of[dev_id];
  // LLMC_B200_CHOL_ONE_STREAM=1 keeps the inverse chain on the caller's stream (A/B runs only)
  const char* one_env = getenv("LLMC_B200_CHOL_ONE_STREAM");
  const bool one_stream = one_env != nullptr && one_env[0] == '1';
  cudaStream_t s2 = one_stream ? st : side;
  while (static_cast<int64_t>(ev.size()) < nbk) {
    cudaEvent_t e;
    LLMC_CHECK_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    ev.push_back(e);
  }
  // super-panel width for the lazy trailing updates (LLMC_B200_CHOL_SP=1..8 blocks, default 4)
  int64_t spw = 4 * NB;
  if (const char* e = getenv("LLMC_B200_CHOL_SP")) {
    const int v = atoi(e);
    if (v >= 1 && v <= 8) spw = static_cast<int64_t>(v) * NB;
  }
  LLMC_CHECK_CUDA(cudaMemsetAsync(info, 0, sizeof(int), st));
  LLMC_CHECK_CUDA(cudaMemsetAsync(Y, 0, nn * sizeof(float), st));
  // the rank-512 inverse update reads Yhi/Ylo over whole super-panel rows: the part above the
  // diagonal blocks inside each super-panel square is never written, so it must be zero
  for (int64_t s0 = 0; s0 < n; s0 += spw) {
    const int64_t w = (s0 + spw < n) ? spw : n - s0;
    LLMC_CHECK_CUDA(cudaMemset2DAsync(Yhi + s0 * n + s0, n * sizeof(float), 0, w * sizeof(float), w, st));
    LLMC_CHECK_CUDA(cudaMemset2DAsync(Ylo + s0 * n + s0, n * sizeof(float), 0, w * sizeof(float), w, st));
  }
  int64_t blocks = (nn + 255) / 256;
  if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
  reverse_kernel<<<(int)blocks, 256, 0, st>>>(A, G, n);
  LLMC_CHECK_LAUNCH();

  // LLMC_B200_CHOL_LOOKAHEAD=0 selects the round-1 schedule below (A/B runs only)
  const char* la_env = getenv("LLMC_B200_CHOL_LOOKAHEAD");
  const bool lookahead = !(la_env != nullptr && la_env[0] == '0') && !use_v1 && !one_stream && n > spw;
  if (lookahead) {
    // ================= look-ahead schedule (round 2) ==========================================
    // The factorisation's dependent chain is  diag(k) -> panel solve(k) -> update of column block
    // k+1  (~100 us per 128 columns, 1..112 CTAs wide); everything else — 90 % of the flops — is
    // off that chain.  Streams (created once per device):
    //   hi    highest priority : the chain.  Inside a super-panel of 4 blocks it is LEFT-looking
    //                            (column block j receives the rank-128*(j-j0) update of its
    //                            super-panel's earlier panels right before it is factored); at a
    //                            super-panel boundary it applies the rank-512 update to the next
    //                            column block only.
    //   bulk  lowest priority  : the rest of each rank-512 trailing update, first the part the
    //                            chain needs next (A': the following 512 columns, event evA), then
    //                            everything beyond (B).  One tile per CTA, so SMs return to the
    //                            chain within a tile time.
    //   s2    middle priority  : the inverse chain (needs panel k of L only), with its own bulk
    //                            stream s3 for the rows beyond the next super-panel.
    // Every column block receives its updates in a fixed order (events), so the result does not
    // depend on timing.
    static cudaStream_t hi_of[kMaxDev] = {}, bulk_of[kMaxDev] = {}, s3_of[kMaxDev] = {}, s2p_of[kMaxDev] = {};
    static cudaEvent_t fork_of[kMaxDev] = {}, j_of[kMaxDev][4] = {};
    static std::vector<cudaEvent_t> evA_of[kMaxDev], evI_of[kMaxDev], evIB_of[kMaxDev];
    if (hi_of[dev_id] == nullptr) {
      int least = 0, greatest = 0;
      LLMC_CHECK_CUDA(cudaDeviceGetStreamPriorityRange(&least, &greatest));
      const int mid = (greatest < least) ? greatest + 1 : greatest;
      LLMC_CHECK_CUDA(cudaStreamCreateWithPriority(&hi_of[dev_id], cudaStreamNonBlocking, greatest));
      LLMC_CHECK_CUDA(cudaStreamCreateWithPriority(&s2p_of[dev_id], cudaStreamNonBlocking, mid));
      LLMC_CHECK_CUDA(cudaStreamCreateWithPriority(&bulk_of[dev_id], cudaStreamNonBlocking, least));
      LLMC_CHECK_CUDA(cudaStreamCreateWithPriority(&s3_of[dev_id], cudaStreamNonBlocking, least));
      LLMC_CHECK_CUDA(cudaEventCreateWithFlags(&fork_of[dev_id], cudaEventDisableTiming));
      for (int i = 0; i < 4; ++i) LLMC_CHECK_CUDA(cudaEventCreateWithFlags(&j_of[dev_id][i], cudaEventDisableTiming));
    }
    auto grow = [&](std::vector<cudaEvent_t>& v) -> int {
      while (static_cast<int64_t>(v.size()) < nbk + 1) {
        cudaEvent_t e;
        LLMC_CHECK_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        v.push_back(e);
      }
      return LLMC_OK;
    };
    if (int rc = grow(evA_of[dev_id])) return rc;
    if (int rc = grow(evI_of[dev_id])) return rc;
    if (int rc = grow(evIB_of[dev_id])) return rc;
    cudaStream_t hi = hi_of[dev_id], bulk = bulk_of[dev_id], si = s2p_of[dev_id], s3 = s3_of[dev_id];
    std::vector<cudaEvent_t>& evA = evA_of[dev_id];     // A' of super-panel s done (bulk)
    std::vector<cudaEvent_t>& evI = evI_of[dev_id];     // inverse chain reached the end of super-panel s
    std::vector<cudaEvent_t>& evIB = evIB_of[dev_id];   // inverse bulk of super-panel s done (s3)
    LLMC_CHECK_CUDA(cudaEventRecord(fork_of[dev_id], st));
    LLMC_CHECK_CUDA(cudaStreamWaitEvent(hi, fork_of[dev_id], 0));
    const int64_t nsp = (n + spw - 1) / spw;
    for (int64_t kb = 0; kb < nbk; ++kb) {
      const int64_t k0 = kb * NB;
      const int nb = static_cast<int>((n - k0) < NB ? (n - k0) : NB);
      const int64_t sidx = k0 / spw;
      const int64_t sp0 = sidx * spw;
      const int64_t sp1 = (sp0 + spw < n) ? sp0 + spw : n;
      const int64_t r0 = k0 + nb;
      const int64_t m = n - r0;
      // ---- chain (hi): bring column block kb up to date ----
      if (k0 > sp0) {
        if (sidx > 0 && k0 == sp0 + NB)      // columns sp0+128.. of this super-panel come from A' of the previous one
          LLMC_CHECK_CUDA(cudaStreamWaitEvent(hi, evA[sidx - 1], 0));
        // G[k0:, k0:k0+nb] -= L[k0:, sp0:k0] L[k0:k0+nb, sp0:k0]^T ; emits the split of the block
        if (int rc = tf32x3_update({.Ahi = Lhi + k0 * n + sp0, .Alo = Llo + k0 * n + sp0, .lda = n,
                                    .Bhi = Lhi + k0 * n + sp0, .Blo = Llo + k0 * n + sp0, .ldb = n,
                                    .C = G + k0 * n + k0, .ldc = n, .M = n - k0, .N = nb,
                                    .K = static_cast<int>(k0 - sp0), .mode = 0,
                                    .Chi = Lhi + k0 * n + k0, .Clo = Llo + k0 * n + k0},
                                   hi))
          return rc;
      }
      diag_kernel_v2<<<1, 256, diag_smem, hi>>>(G, n, k0, nb, Y, Yhi, Ylo, info);
      LLMC_CHECK_LAUNCH();
      const float* Xh = Yhi + k0 * n + k0;
      const float* Xl = Ylo + k0 * n + k0;
      float* P = G + r0 * n + k0;
      float* Ph = Lhi + r0 * n + k0;
      float* Pl = Llo + r0 * n + k0;
      if (m > 0) {
        if (kb == 0)
          if (int rc = split_tf32(P, m, nb, n, Ph, Pl, n, hi)) return rc;
        if (int rc = tf32x3_update({.Ahi = Ph, .Alo = Pl, .lda = n, .Bhi = Xh, .Blo = Xl, .ldb = n,
                                    .C = P, .ldc = n, .M = m, .N = nb, .K = nb, .mode = 1,
                                    .Chi = Ph, .Clo = Pl},
                                   hi))
          return rc;
      }
      LLMC_CHECK_CUDA(cudaEventRecord(ev[kb], hi));        // L panel kb, Y_kk final
      if (m > 0 && r0 == sp1) {
        // ---- super-panel boundary: rank-(sp1-sp0) update of G[sp1:, sp1:] in three pieces ----
        const int kk = static_cast<int>(sp1 - sp0);
        const float* Ah = Lhi + sp1 * n + sp0;
        const float* Al = Llo + sp1 * n + sp0;
        const int64_t w1 = (n - sp1) < NB ? (n - sp1) : NB;
        // chain: the next column block (also waits for what earlier bulk pieces wrote there)
        if (sidx > 0) LLMC_CHECK_CUDA(cudaStreamWaitEvent(hi, evA[sidx - 1], 0));
        if (int rc = tf32x3_update({.Ahi = Ah, .Alo = Al, .lda = n, .Bhi = Ah, .Blo = Al, .ldb = n,
                                    .C = G + sp1 * n + sp1, .ldc = n, .M = n - sp1, .N = w1,
                                    .K = kk, .mode = 0,
                                    .Chi = Lhi + sp1 * n + sp1, .Clo = Llo + sp1 * n + sp1},
                                   hi))
          return rc;
        // bulk: A' = columns [sp1+128, sp1+128+spw), then B = the rest; lower tiles only
        LLMC_CHECK_CUDA(cudaStreamWaitEvent(bulk, ev[kb], 0));
        const int64_t ca = sp1 + NB;
        const int64_t cb = (ca + spw < n) ? ca + spw : n;
        if (ca < n) {
          if (int rc = tf32x3_update({.Ahi = Ah, .Alo = Al, .lda = n,
                                      .Bhi = Lhi + ca * n + sp0, .Blo = Llo + ca * n + sp0, .ldb = n,
                                      .C = G + sp1 * n + ca, .ldc = n, .M = n - sp1, .N = cb - ca,
                                      .K = kk, .mode = 0, .tri = 1, .row_off = sp1, .col_off = ca,
                                      .one_tile_per_cta = 1},
                                     bulk))
            return rc;
        }
        LLMC_CHECK_CUDA(cudaEventRecord(evA[sidx], bulk));
        if (cb < n) {
          if (int rc = tf32x3_update({.Ahi = Ah, .Alo = Al, .lda = n,
                                      .Bhi = Lhi + cb * n + sp0, .Blo = Llo + cb * n + sp0, .ldb = n,
                                      .C = G + sp1 * n + cb, .ldc = n, .M = n - sp1, .N = n - cb,
                                      .K = kk, .mode = 0, .tri = 1, .row_off = sp1, .col_off = cb,
                                      .one_tile_per_cta = 1},
                                     bulk))
            return rc;
        }
      }
      // ---- inverse chain (si): Y = L^-1, one block row per panel ----
      LLMC_CHECK_CUDA(cudaStreamWaitEvent(si, ev[kb], 0));
      if (kb > 0) {
        float* T = Y + k0 * n;
        float* Th = Yhi + k0 * n;
        float* Tl = Ylo + k0 * n;
        if (int rc = tf32x3_update({.Ahi = Xh, .Alo = Xl, .lda = n,
                                    .Bhi = Th, .Blo = Tl, .b_mn = 1, .ldb = n,
                                    .C = T, .ldc = n, .M = nb, .N = k0, .K = nb, .mode = 1,
                                    .Chi = Th, .Clo = Tl},
                                   si))
          return rc;
      }
      if (m > 0 && r0 < sp1) {
        if (int rc = tf32x3_update({.Ahi = Lhi + r0 * n + k0, .Alo = Llo + r0 * n + k0, .lda = n,
                                    .Bhi = Yhi + k0 * n, .Blo = Ylo + k0 * n, .b_mn = 1, .ldb = n,
                                    .C = Y + r0 * n, .ldc = n, .M = sp1 - r0, .N = r0, .K = nb,
                                    .mode = 0, .Chi = Yhi + r0 * n, .Clo = Ylo + r0 * n,
                                    .split_rows = NB, .split_cols = 0},
                                   si))
          return rc;
      } else if (m > 0) {
        // T'[sp1:, 0:sp1] -= L[sp1:, sp0:sp1] Y[sp0:sp1, 0:sp1]: the next super-panel's rows on the
        // chain, the rows beyond on s3 (they are next touched by the following boundary's pieces,
        // which wait for evIB)
        const int kk = static_cast<int>(sp1 - sp0);
        const int64_t ra = (sp1 + spw < n) ? sp1 + spw : n;
        if (sidx > 0) LLMC_CHECK_CUDA(cudaStreamWaitEvent(si, evIB[sidx - 1], 0));
        if (int rc = tf32x3_update({.Ahi = Lhi + sp1 * n + sp0, .Alo = Llo + sp1 * n + sp0, .lda = n,
                                    .Bhi = Yhi + sp0 * n, .Blo = Ylo + sp0 * n, .b_mn = 1, .ldb = n,
                                    .C = Y + sp1 * n, .ldc = n, .M = ra - sp1, .N = sp1, .K = kk,
                                    .mode = 0, .Chi = Yhi + sp1 * n, .Clo = Ylo + sp1 * n,
                                    .split_rows = NB, .split_cols = 0},
                                   si))
          return rc;
        LLMC_CHECK_CUDA(cudaEventRecord(evI[sidx], si));
        LLMC_CHECK_CUDA(cudaStreamWaitEvent(s3, evI[sidx], 0));
        if (ra < n) {
          if (int rc = tf32x3_update({.Ahi = Lhi + ra * n + sp0, .Alo = Llo + ra * n + sp0, .lda = n,
                                      .Bhi = Yhi + sp0 * n, .Blo = Ylo + sp0 * n, .b_mn = 1, .ldb = n,
                                      .C = Y + ra * n, .ldc = n, .M = n - ra, .N = sp1, .K = kk,
                                      .mode = 0, .one_tile_per_cta = 1},
                                     s3))
            return rc;
        }
        LLMC_CHECK_CUDA(cudaEventRecord(evIB[sidx], s3));
      }
    }
    (void)nsp;
    cudaStream_t all[4] = {hi, bulk, si, s3};
    for (int i = 0; i < 4; ++i) {
      LLMC_CHECK_CUDA(cudaEventRecord(j_of[dev_id][i], all[i]));
      LLMC_CHECK_CUDA(cudaStreamWaitEvent(st, j_of[dev_id][i], 0));
    }
    reverse_upper_kernel<<<(int)blocks, 256, 0, st>>>(Y, A, n);
    LLMC_CHECK_LAUNCH();
    return LLMC_OK;
  }

  // ---- factor: G = L L^T (lower, in place), Lhi/Llo = split of the sub-diagonal panels ----
  for (int64_t kb = 0; kb < nbk; ++kb) {
    const int64_t k0 = kb * NB;
    const int nb = static_cast<int>((n - k0) < NB ? (n - k0) : NB);
    float* Dk = D + kb * NB * NB;
    float* Dkh = Dhi + kb * NB * NB;
    float* Dkl = Dlo + kb * NB * NB;
    if (use_v1) {
      diag_kernel<<<1, 256, diag_smem, st>>>(G, n, k0, nb, Dk, Dkh, Dkl, info);
      LLMC_CHECK_LAUNCH();
      place_diag_kernel<<<16, 256, 0, st>>>(Dk, Dkh, Dkl, Y, Yhi, Ylo, n, k0, nb);
    } else {
      diag_kernel_v2<<<1, 256, diag_smem, st>>>(G, n, k0, nb, Y, Yhi, Ylo, info);
    }
    LLMC_CHECK_LAUNCH();
    // L_kk^-1 as a GEMM operand: v2 leaves it in the diagonal block of Yhi/Ylo (ld n)
    const float* Xh = use_v1 ? Dkh : Yhi + k0 * n + k0;
    const float* Xl = use_v1 ? Dkl : Ylo + k0 * n + k0;
    const int64_t ldx = use_v1 ? NB : n;
    const int64_t r0 = k0 + nb;
    const int64_t m = n - r0;
    float* P = G + r0 * n + k0;          // panel [m x nb], ld n
    float* Ph = Lhi + r0 * n + k0;
    float* Pl = Llo + r0 * n + k0;
    if (m > 0) {
      // the split of panel 0 is made here; later panels get theirs from the trailing update below
      if (kb == 0)
        if (int rc = split_tf32(P, m, nb, n, Ph, Pl, n, st)) return rc;
      // P <- P * L_kk^-T : out[i][j] = sum_k P[i][k] * Dk[j][k]   (both K-major), + split
      if (int rc = tf32x3_update({.Ahi = Ph, .Alo = Pl, .lda = n, .Bhi = Xh, .Blo = Xl, .ldb = ldx,
                                  .C = P, .ldc = n, .M = m, .N = nb, .K = nb, .mode = 1,
                                  .Chi = Ph, .Clo = Pl},
                                 st))
        return rc;
    }
    LLMC_CHECK_CUDA(cudaEventRecord(ev[kb], st));          // L panel kb, D_kb and Y_kk are final
    // Trailing updates are lazy per super-panel [sp0, sp1) of kSuperBlocks blocks: a block updates
    // only the super-panel's remaining columns (rank 128); everything beyond the super-panel
    // gets one rank-512 update when its last block is done — a quarter of the read-modify-write
    // traffic.  Both emit the tf32 split of the next panel (their first 128 columns).
    const int64_t sp0 = (k0 / spw) * spw;
    const int64_t sp1 = (sp0 + spw < n) ? sp0 + spw : n;
    if (m > 0 && r0 < sp1) {
      // G[r0:, r0:sp1] -= P P[r0:sp1]^T  (lower tiles only)
      if (int rc = tf32x3_update({.Ahi = Ph, .Alo = Pl, .lda = n, .Bhi = Ph, .Blo = Pl, .ldb = n,
                                  .C = G + r0 * n + r0, .ldc = n, .M = m, .N = sp1 - r0, .K = nb,
                                  .mode = 0, .Chi = Lhi + r0 * n + r0, .Clo = Llo + r0 * n + r0,
                                  .split_rows = 0, .split_cols = NB, .tri = 1},
                                 st))
        return rc;
    } else if (m > 0) {
      // G[sp1:, sp1:] -= L[sp1:, sp0:sp1] L[sp1:, sp0:sp1]^T
      const float* Ah = Lhi + sp1 * n + sp0;
      const float* Al = Llo + sp1 * n + sp0;
      if (int rc = tf32x3_update({.Ahi = Ah, .Alo = Al, .lda = n, .Bhi = Ah, .Blo = Al, .ldb = n,
                                  .C = G + sp1 * n + sp1, .ldc = n, .M = n - sp1, .N = n - sp1,
                                  .K = static_cast<int>(sp1 - sp0), .mode = 0,
                                  .Chi = Lhi + sp1 * n + sp1, .Clo = Llo + sp1 * n + sp1,
                                  .split_rows = 0, .split_cols = NB, .tri = 1},
                                 st))
        return rc;
    }

    // ---- inverse step kb on the side stream: Y = L^-1 (lower).  T' (stored in Y below the
    //      diagonal blocks) accumulates -sum_{k<i} L_ik Y_k ;  Y_i = D_i T'_i.  It needs panel kb
    //      of L only, so it overlaps the factorisation's trailing update and later steps. ----
    LLMC_CHECK_CUDA(cudaStreamWaitEvent(s2, ev[kb], 0));
    if (kb > 0) {
      float* T = Y + k0 * n;             // rows k0..k0+nb, cols 0..k0; split emitted by step kb-1
      float* Th = Yhi + k0 * n;
      float* Tl = Ylo + k0 * n;
      // Y[k rows, 0:k0] = D_k (K-major: D[m][kk]) * T' (MN-major: element (col, kk) at T[kk*n + col])
      if (int rc = tf32x3_update({.Ahi = Xh, .Alo = Xl, .lda = ldx,
                                  .Bhi = Th, .Blo = Tl, .b_mn = 1, .ldb = n,
                                  .C = T, .ldc = n, .M = nb, .N = k0, .K = nb, .mode = 1,
                                  .Chi = Th, .Clo = Tl},
                                 s2))
        return rc;
    }
    if (m > 0 && r0 < sp1) {
      // T'[r0:sp1, 0:r0] -= L[r0:sp1, kblock] * Y[k rows, 0:r0]; emits the split of the next T' rows
      if (int rc = tf32x3_update({.Ahi = Lhi + r0 * n + k0, .Alo = Llo + r0 * n + k0, .lda = n,
                                  .Bhi = Yhi + k0 * n, .Blo = Ylo + k0 * n, .b_mn = 1, .ldb = n,
                                  .C = Y + r0 * n, .ldc = n, .M = sp1 - r0, .N = r0, .K = nb,
                                  .mode = 0, .Chi = Yhi + r0 * n, .Clo = Ylo + r0 * n,
                                  .split_rows = NB, .split_cols = 0},
                                 s2))
        return rc;
    } else if (m > 0) {
      // T'[sp1:, 0:sp1] -= L[sp1:, sp0:sp1] * Y[sp0:sp1, 0:sp1]
      if (int rc = tf32x3_update({.Ahi = Lhi + sp1 * n + sp0, .Alo = Llo + sp1 * n + sp0, .lda = n,
                                  .Bhi = Yhi + sp0 * n, .Blo = Ylo + sp0 * n, .b_mn = 1, .ldb = n,
                                  .C = Y + sp1 * n, .ldc = n, .M = n - sp1, .N = sp1,
                                  .K = static_cast<int>(sp1 - sp0), .mode = 0,
                                  .Chi = Yhi + sp1 * n, .Clo = Ylo + sp1 * n,
                                  .split_rows = NB, .split_cols = 0},
                                 s2))
        return rc;
    }
  }
  LLMC_CHECK_CUDA(cudaEventRecord(ev_join, s2));
  LLMC_CHECK_CUDA(cudaStreamWaitEvent(st, ev_join, 0));
  reverse_upper_kernel<<<(int)blocks, 256, 0, st>>>(Y, A, n);
  LLMC_CHECK_LAUNCH();
  return LLMC_OK;
}
