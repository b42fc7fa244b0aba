// gptq.cu — K5: GPTQ column-block update, plus the gathers around it.
//
// Replaces GPTQ.process_hessian_and_weights (dead columns, act-order gather, damping;
// llmc/compression/quantization/gptq.py:128-171) and GPTQ.weight_transform (:198-244) with
// search_column_qparams (:358-366).  The reference spends ~15 tiny launches per COLUMN; here a
// 128-column block is one launch of `gptq_inblock_kernel` (rows are independent: one thread
// owns one weight row, the 128x128 Hinv block and the row tile live in shared memory) followed
// by one fp32 `trailing_update_kernel` (W[:, i2:] -= Err1 @ Hinv[i1:i2, i2:], :244).
//
// Numerics: fp32 throughout like the reference (gptq.py:135).  Inside a block every op is
// rounded exactly like torch (separate multiply and subtract for the rank-1 updates, :240;
// IEEE divides), so single-block problems are bit-exact; across blocks only the summation
// order of the 128-deep trailing dot products differs from the CPU BLAS.
#include "common.cuh"
#include "spqr_row.cuh"
#include "tf32.cuh"

namespace llmc {

constexpr int GB = 128;          // gptq blocksize (gptq_w_only.yml: blocksize 128)
// Trailing updates are applied lazily per super-panel of 4 blocks: inside the super-panel each
// block updates only the super-panel's remaining columns (rank 128), and the columns beyond it get
// ONE rank-512 update.  Same terms as gptq.py:244 block by block, grouped differently (fp32
// summation order only), and a quarter of the read-modify-write traffic over W.
constexpr int kSuperPanel = 4 * GB;
constexpr int SB = 16;           // register sub-block inside the 128-column block
constexpr int kPad = GB + 1;
constexpr int HP = GB + 4;       // pitch of the transposed Hinv block (16-byte aligned rows)

// ---- prepare -----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
diag_mean_kernel(const float* __restrict__ H, int64_t C, float percdamp, float* __restrict__ out) {
  // out[0] = percdamp * mean(diag(H) with zeros replaced by 1)   (gptq.py:139-140, 169)
  __shared__ float red[8];
  float acc = 0.f;
  for (int64_t i = threadIdx.x; i < C; i += blockDim.x) {
    const float d = H[i * C + i];
    acc += (d == 0.f) ? 1.f : d;
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < 8 ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) out[0] = percdamp * (v / static_cast<float>(C));
  }
}

__global__ void __launch_bounds__(256)
gather_h_kernel(const float* __restrict__ H, int64_t C, const int64_t* __restrict__ perm,
                const float* __restrict__ damp, float* __restrict__ Hp) {
  extern __shared__ float row[];
  const int64_t i = blockIdx.x;
  const int64_t pi = perm ? perm[i] : i;
  for (int64_t j = threadIdx.x; j < C; j += blockDim.x) row[j] = H[pi * C + j];
  __syncthreads();
  const float dmp = damp[0];
  for (int64_t j = threadIdx.x; j < C; j += blockDim.x) {
    const int64_t pj = perm ? perm[j] : j;
    float v = row[pj];
    if (i == j) v = ((v == 0.f) ? 1.f : v) + dmp;
    Hp[i * C + j] = v;
  }
}

template <int WT>
__global__ void __launch_bounds__(256)
gather_w_kernel(const void* __restrict__ W, int64_t R, int64_t C, const float* __restrict__ H,
                const int64_t* __restrict__ perm, float* __restrict__ Wp) {
  extern __shared__ float row[];
  const int64_t r = blockIdx.x;
  for (int64_t j = threadIdx.x; j < C; j += blockDim.x) row[j] = DType<WT>::load(W, r * C + j);
  __syncthreads();
  for (int64_t j = threadIdx.x; j < C; j += blockDim.x) {
    const int64_t pj = perm ? perm[j] : j;
    const bool dead = H[pj * C + pj] == 0.f;
    Wp[r * C + j] = dead ? 0.f : row[pj];
  }
}

// ---- in-block column loop ------------------------------------------------------------------------------
struct InblockArgs {
  float* W;              // [R, C] fp32 working copy (permuted)
  const float* Hinv;     // [C, C] upper factor
  int64_t R, C;
  int i1, count;         // block start, columns in this block (<= 128)
  int64_t group;         // elements per group (C for per_channel)
  int64_t ng;
  int sym;
  float qmin, qmax;
  int static_groups;     // qparams are inputs
  const int32_t* gmap;   // static: column -> group index (perm[idx]/g), may be null
  void* scales;          // dynamic: fp32 out [R, ng]; static: q_dtype in
  void* zeros;
  int q_dtype;
  float* tmp;            // [R, C] out
  const int64_t* out_perm;  // optional: scatter tmp columns back to the original order
  float* losses;         // [R] accumulated
  float* err;            // [128, Rpad] out (Err1 transposed)
  float* err_hi;         // tf32 split of err
  float* err_lo;
  int64_t Rpad;          // R rounded up to 128
};

__device__ __forceinline__ float load_q(const void* p, int dt, int64_t i) {
  if (dt == LLMC_F32) return DType<LLMC_F32>::load(p, i);
  if (dt == LLMC_F16) return DType<LLMC_F16>::load(p, i);
  return DType<LLMC_BF16>::load(p, i);
}

// fp32-faithful quant-dequant of one value (quant.py:699-717 on fp32 tensors).
__device__ __forceinline__ float qdq_f32(float w, float s, float z, float qmin, float qmax) {
  float q = rintf(fdiv_rn(w, s)) + z;
  q = fminf(fmaxf(q, qmin), qmax);
  return fmul_rn(q - z, s);
}

__device__ __forceinline__ void qparams_f32(float mn, float mx, int sym, float qmin, float qmax,
                                            float& s, float& z) {
  if (sym) {
    float a = fmaxf(fmaxf(fabsf(mx), fabsf(mn)), 1e-5f);
    s = fdiv_rn(a, qmax);
    z = 0.f;
  } else {
    float d = fmaxf(fsub_rn(mx, mn), 1e-5f);
    s = fdiv_rn(d, fsub_rn(qmax, qmin));
    z = fsub_rn(qmin, rintf(fdiv_rn(mn, s)));
    z = fminf(fmaxf(z, qmin), qmax);
  }
}

__global__ void __launch_bounds__(GB, 1)
gptq_inblock_kernel(InblockArgs a) {
  extern __shared__ float sm[];
  float* Wt = sm;                        // [128 cols][129]  current (lazily updated) weights
  float* Et = Wt + GB * kPad;            // [128 cols][129]  err (Err1 transposed)
  float* Ht = Et + GB * kPad;            // [128 j][HP]      Ht[j][i] = Hinv1[i][j]
  const int tid = threadIdx.x;
  const int64_t r0 = static_cast<int64_t>(blockIdx.x) * GB;
  const int64_t row = r0 + tid;
  const int cnt = a.count;

  // Tile loads: 16-byte coalesced loads, eight in flight per thread (the scalar one-at-a-time
  // version spent ~47 % of the kernel stalled on global latency), transposed into shared memory.
  {
    const bool vec = (cnt == GB) && ((a.C & 3) == 0) && ((reinterpret_cast<uintptr_t>(a.W) & 15) == 0) &&
                     ((reinterpret_cast<uintptr_t>(a.Hinv) & 15) == 0);
    if (vec) {
      constexpr int kBatch = 8;
      // W tile: 128 rows x 32 float4; item = row * 32 + c4
      for (int base = 0; base < GB * 32; base += GB * kBatch) {
        float4 v[kBatch];
#pragma unroll
        for (int b = 0; b < kBatch; ++b) {
          const int item = base + b * GB + tid;
          const int rr = item >> 5, c4 = item & 31;
          const int64_t r = r0 + rr;
          v[b] = (r < a.R) ? *reinterpret_cast<const float4*>(&a.W[r * a.C + a.i1 + c4 * 4])
                           : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int b = 0; b < kBatch; ++b) {
          const int item = base + b * GB + tid;
          const int rr = item >> 5, c = (item & 31) * 4;
          Wt[(c + 0) * kPad + rr] = v[b].x;
          Wt[(c + 1) * kPad + rr] = v[b].y;
          Wt[(c + 2) * kPad + rr] = v[b].z;
          Wt[(c + 3) * kPad + rr] = v[b].w;
        }
      }
      // Hinv block: row i, float4 over j -> Ht[j][i], upper triangle only
      for (int base = 0; base < GB * 32; base += GB * kBatch) {
        float4 v[kBatch];
#pragma unroll
        for (int b = 0; b < kBatch; ++b) {
          const int item = base + b * GB + tid;
          const int i = item >> 5, j4 = item & 31;
          v[b] = *reinterpret_cast<const float4*>(
              &a.Hinv[(static_cast<int64_t>(a.i1) + i) * a.C + a.i1 + j4 * 4]);
        }
#pragma unroll
        for (int b = 0; b < kBatch; ++b) {
          const int item = base + b * GB + tid;
          const int i = item >> 5, j = (item & 31) * 4;
          Ht[(j + 0) * HP + i] = (j + 0 >= i) ? v[b].x : 0.f;
          Ht[(j + 1) * HP + i] = (j + 1 >= i) ? v[b].y : 0.f;
          Ht[(j + 2) * HP + i] = (j + 2 >= i) ? v[b].z : 0.f;
          Ht[(j + 3) * HP + i] = (j + 3 >= i) ? v[b].w : 0.f;
        }
      }
    } else {
      const int warp = tid >> 5, lane = tid & 31;
      for (int rr = warp; rr < GB; rr += 4) {
        const int64_t r = r0 + rr;
        for (int c = lane; c < GB; c += 32) {
          float v = 0.f;
          if (r < a.R && c < cnt) v = a.W[r * a.C + a.i1 + c];
          Wt[c * kPad + rr] = v;
        }
      }
      for (int i = warp; i < GB; i += 4)
        for (int j = lane; j < GB; j += 32) {
          float v = 0.f;
          if (i < cnt && j < cnt && j >= i)
            v = a.Hinv[(static_cast<int64_t>(a.i1) + i) * a.C + a.i1 + j];
          Ht[j * HP + i] = v;
        }
    }
  }
  __syncthreads();
  const bool live = row < a.R;

  // ---- qparams of the groups that start inside this block (gptq.py:215-223) ----
  // searched on W as it stands at block entry (the reference indexes the global W, not the
  // in-block clone W1).  Kept in registers for group >= 128, recomputed per group otherwise.
  float s_cur = 1.f, z_cur = 0.f;
  const bool dynamic = !a.static_groups;
  const int gsz = static_cast<int>(a.group < GB ? a.group : GB);   // columns per group inside the block
  if (dynamic && live) {
    if (a.group >= GB) {
      if ((a.i1 % a.group) == 0) {
        float mn = INFINITY, mx = -INFINITY;
        const int64_t gend = min(static_cast<int64_t>(a.i1) + a.group, a.C);
        if (gend - a.i1 <= cnt) {
          for (int c = 0; c < cnt; ++c) { const float v = Wt[c * kPad + tid]; mn = fminf(mn, v); mx = fmaxf(mx, v); }
        } else {
          for (int64_t c = a.i1; c < gend; ++c) { const float v = a.W[row * a.C + c]; mn = fminf(mn, v); mx = fmaxf(mx, v); }
        }
        qparams_f32(mn, mx, a.sym, a.qmin, a.qmax, s_cur, z_cur);
        const int64_t gi = a.i1 / a.group;
        reinterpret_cast<float*>(a.scales)[row * a.ng + gi] = s_cur;
        if (!a.sym) reinterpret_cast<float*>(a.zeros)[row * a.ng + gi] = z_cur;
      } else {
        const int64_t gi = a.i1 / a.group;    // group opened by an earlier block
        s_cur = reinterpret_cast<const float*>(a.scales)[row * a.ng + gi];
        z_cur = a.sym ? 0.f : reinterpret_cast<const float*>(a.zeros)[row * a.ng + gi];
      }
    }
  } else if (!dynamic && live && a.group >= a.C) {
    s_cur = load_q(a.scales, a.q_dtype, row);                 // per_channel
    z_cur = a.zeros ? load_q(a.zeros, a.q_dtype, row) : 0.f;
  }
  // small groups: compute all in-block group qparams up front into registers (<= 8 groups)
  float s_small[8], z_small[8];
  if (dynamic && a.group < GB) {
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      s_small[g] = 1.f; z_small[g] = 0.f;
      if (g * gsz < cnt && live) {
        float mn = INFINITY, mx = -INFINITY;
        const int cend = min((g + 1) * gsz, cnt);
        for (int c = g * gsz; c < cend; ++c) { const float v = Wt[c * kPad + tid]; mn = fminf(mn, v); mx = fmaxf(mx, v); }
        qparams_f32(mn, mx, a.sym, a.qmin, a.qmax, s_small[g], z_small[g]);
        const int64_t gi = (a.i1 + g * gsz) / a.group;
        reinterpret_cast<float*>(a.scales)[row * a.ng + gi] = s_small[g];
        if (!a.sym) reinterpret_cast<float*>(a.zeros)[row * a.ng + gi] = z_small[g];
      }
    }
  }

  float loss = 0.f;
  for (int sb = 0; sb < cnt; sb += SB) {
    float w[SB], e[SB], ss[SB], zz[SB];
    // qparams for the sub-block's columns
#pragma unroll
    for (int k = 0; k < SB; ++k) {
      const int c = sb + k;
      ss[k] = s_cur; zz[k] = z_cur;
      if (dynamic && a.group < GB) {
        const int g = c / gsz;
        // static register indexing through a switch-free select (g <= 7)
        float sv = s_small[0], zv = z_small[0];
#pragma unroll
        for (int t = 1; t < 8; ++t) { if (g == t) { sv = s_small[t]; zv = z_small[t]; } }
        ss[k] = sv; zz[k] = zv;
      } else if (!dynamic && a.group < a.C && live && c < cnt) {
        const int64_t idx = static_cast<int64_t>(a.i1) + c;
        const int64_t gi = a.gmap ? a.gmap[idx] : idx / a.group;     // gptq.py:225-227
        ss[k] = load_q(a.scales, a.q_dtype, row * a.ng + gi);
        zz[k] = a.zeros ? load_q(a.zeros, a.q_dtype, row * a.ng + gi) : 0.f;
      }
      w[k] = Wt[c * kPad + tid];
    }
    // sequential part: quantise column, propagate inside the sub-block (registers)
#pragma unroll
    for (int k = 0; k < SB; ++k) {
      const int c = sb + k;
      const float d = Ht[c * HP + c];                      // Hinv1[c][c]
      const float q = qdq_f32(w[k], ss[k], zz[k], a.qmin, a.qmax);
      const float diff = fsub_rn(w[k], q);
      float err = 0.f;
      if (c < cnt) {
        loss += fdiv_rn(fmul_rn(diff, diff), fmul_rn(2.f, fmul_rn(d, d)));   // :238
        err = fdiv_rn(diff, d);                                               // :239
      }
      e[k] = err;
#pragma unroll
      for (int k2 = k + 1; k2 < SB; ++k2)
        w[k2] = fsub_rn(w[k2], fmul_rn(err, Ht[(sb + k2) * HP + c]));          // :240
    }
    // record tmp (pre-rounding compensated weight, :237) and Err1 (:241)
#pragma unroll
    for (int k = 0; k < SB; ++k) {
      const int c = sb + k;
      Wt[c * kPad + tid] = w[k];
      Et[c * kPad + tid] = e[k];
    }
    // lazy propagation to the remaining columns of the block, in the reference's order
    // (each column's 16 updates are a dependent chain by definition; four columns are kept in
    // flight so the chains overlap)
    int j = sb + SB;
    for (; j + 3 < cnt; j += 4) {
      float v0 = Wt[(j + 0) * kPad + tid], v1 = Wt[(j + 1) * kPad + tid];
      float v2 = Wt[(j + 2) * kPad + tid], v3 = Wt[(j + 3) * kPad + tid];
      const float4* h0 = reinterpret_cast<const float4*>(&Ht[(j + 0) * HP + sb]);
      const float4* h1 = reinterpret_cast<const float4*>(&Ht[(j + 1) * HP + sb]);
      const float4* h2 = reinterpret_cast<const float4*>(&Ht[(j + 2) * HP + sb]);
      const float4* h3 = reinterpret_cast<const float4*>(&Ht[(j + 3) * HP + sb]);
#pragma unroll
      for (int k4 = 0; k4 < SB / 4; ++k4) {
        const float4 a = h0[k4], b = h1[k4], c = h2[k4], d = h3[k4];
        v0 = fsub_rn(v0, fmul_rn(e[4 * k4 + 0], a.x)); v1 = fsub_rn(v1, fmul_rn(e[4 * k4 + 0], b.x));
        v2 = fsub_rn(v2, fmul_rn(e[4 * k4 + 0], c.x)); v3 = fsub_rn(v3, fmul_rn(e[4 * k4 + 0], d.x));
        v0 = fsub_rn(v0, fmul_rn(e[4 * k4 + 1], a.y)); v1 = fsub_rn(v1, fmul_rn(e[4 * k4 + 1], b.y));
        v2 = fsub_rn(v2, fmul_rn(e[4 * k4 + 1], c.y)); v3 = fsub_rn(v3, fmul_rn(e[4 * k4 + 1], d.y));
        v0 = fsub_rn(v0, fmul_rn(e[4 * k4 + 2], a.z)); v1 = fsub_rn(v1, fmul_rn(e[4 * k4 + 2], b.z));
        v2 = fsub_rn(v2, fmul_rn(e[4 * k4 + 2], c.z)); v3 = fsub_rn(v3, fmul_rn(e[4 * k4 + 2], d.z));
        v0 = fsub_rn(v0, fmul_rn(e[4 * k4 + 3], a.w)); v1 = fsub_rn(v1, fmul_rn(e[4 * k4 + 3], b.w));
        v2 = fsub_rn(v2, fmul_rn(e[4 * k4 + 3], c.w)); v3 = fsub_rn(v3, fmul_rn(e[4 * k4 + 3], d.w));
      }
      Wt[(j + 0) * kPad + tid] = v0; Wt[(j + 1) * kPad + tid] = v1;
      Wt[(j + 2) * kPad + tid] = v2; Wt[(j + 3) * kPad + tid] = v3;
    }
    for (; j < cnt; ++j) {
      float v = Wt[j * kPad + tid];
      const float4* hp = reinterpret_cast<const float4*>(&Ht[j * HP + sb]);
#pragma unroll
      for (int k4 = 0; k4 < SB / 4; ++k4) {
        const float4 h = hp[k4];
        v = fsub_rn(v, fmul_rn(e[4 * k4 + 0], h.x));
        v = fsub_rn(v, fmul_rn(e[4 * k4 + 1], h.y));
        v = fsub_rn(v, fmul_rn(e[4 * k4 + 2], h.z));
        v = fsub_rn(v, fmul_rn(e[4 * k4 + 3], h.w));
      }
      Wt[j * kPad + tid] = v;
    }
  }
  if (live) a.losses[row] += loss;
  __syncthreads();
  // coalesced write-back: tmp[:, i1:i2] (row-major) and Err1 transposed ([k][row], k-major so
  // the trailing GEMM reads its A operand with unit stride)
  {
    const int warp = tid >> 5, lane = tid & 31;
    for (int rr = warp; rr < GB; rr += 4) {
      const int64_t r = r0 + rr;
      if (r >= a.R) break;
      for (int c = lane; c < cnt; c += 32) {
        // tmp[:, invperm] (gptq.py:186-188) fused as a scatter: permuted column i1+c goes back
        // to original column perm[i1+c]
        const int64_t oc = a.out_perm ? a.out_perm[a.i1 + c] : static_cast<int64_t>(a.i1) + c;
        a.tmp[r * a.C + oc] = Wt[c * kPad + rr];
      }
    }
    for (int c = warp; c < GB; c += 4)
      for (int rr = lane; rr < GB; rr += 32) {
        const float ev = (c < cnt) ? Et[c * kPad + rr] : 0.f;
        const int64_t o = static_cast<int64_t>(c) * a.Rpad + r0 + rr;
        a.err[o] = ev;
        uint32_t hb;                                   // tf32 split for the 3xTF32 trailing GEMM
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(ev));
        const float h = __uint_as_float(hb);
        uint32_t lb;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(lb) : "f"(ev - h));
        a.err_hi[o] = h;
        a.err_lo[o] = __uint_as_float(lb);
      }
  }
}

// ---- in-block column loop, v2: eight lanes per weight row ----------------------------------------------
// v1 above gives one thread a whole row: 128 CTAs' worth of parallelism does not exist for
// R = 4096 (32 CTAs on 148 SMs, one warp per scheduler, IPC 0.23 per warp, 85 us per block).
// v2 spreads a row over 8 lanes (lane l owns columns l, l+8, ...), 32 rows per CTA, 256 threads,
// two CTAs per SM:
//   * per 8-column sub-block each lane keeps ITS column in a register; the eight sequential
//     quantise -> err -> rank-1 steps exchange `err` with one width-8 shuffle each;
//   * the other columns of the row stay in shared memory and receive the sub-block's eight
//     updates lazily, in the reference's order (same op sequence per element as gptq.py:240, so
//     results are bit-identical to v1);
//   * x / s with s fixed is evaluated as a reciprocal multiply plus two FMA corrections
//     (div_by below), which is the correctly rounded quotient, at a third of div.rn's cost.
constexpr int IR = 32;            // rows per CTA
constexpr int IL = 8;             // lanes per row
constexpr int WP = GB + 8;        // pitch of the row-major W tile: 4 rows x 8 lanes hit 32 banks
constexpr int EP = IR + 1;        // pitch of the transposed err tile
constexpr int HP2 = GB + 4;       // pitch of the row-major Hinv block
constexpr int kInblockV2Smem = (IR * WP + GB * EP + GB * HP2 + 2 * GB) * 4;

// RN(x / s) given r = RN(1 / s).  q1 is a faithful quotient (residual-corrected once), and the
// second correction of a faithful quotient with a correctly rounded reciprocal is the correctly
// rounded quotient (Markstein), provided nothing under/overflows: x, s and r with exponents in
// [2^-40, 2^41) keep q and both residuals normal (x = 0 is exact as well).  Anything else takes
// div.rn, kept OUT of line: inlined, its ~10-instruction sequence sat on the dependent chain of
// every column step whether or not it was needed (profiles/r01c_hot_gptq_inblock_v2.md).
__device__ __noinline__ float div_exact_slow(float x, float s) { return fdiv_rn(x, s); }

__device__ __forceinline__ bool exp_mid(float v) {
  return (((__float_as_uint(v) >> 23) & 0xffu) - 87u) <= 80u;
}

// sr_ok = exp_mid(s) && exp_mid(r): a property of the divisor, evaluated once by the caller
__device__ __forceinline__ float div_by(float x, float s, float r, bool sr_ok) {
  const float q0 = fmul_rn(x, r);
  float rem = fma_rn(-q0, s, x);
  const float q1 = fma_rn(rem, r, q0);
  rem = fma_rn(-q1, s, x);
  float q2 = fma_rn(rem, r, q1);
  if (!(sr_ok && (exp_mid(x) || x == 0.f))) q2 = div_exact_slow(x, s);
  return q2;
}

__device__ __forceinline__ float qdq_f32_r(float w, float s, float rs, bool s_ok, float z, float qmin,
                                           float qmax) {
  float q = rintf(div_by(w, s, rs, s_ok)) + z;
  q = fminf(fmaxf(q, qmin), qmax);
  return fmul_rn(q - z, s);
}

__device__ __forceinline__ float group8_min(float v) {
  v = fminf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  v = fminf(v, __shfl_xor_sync(0xffffffffu, v, 2));
  return fminf(v, __shfl_xor_sync(0xffffffffu, v, 4));
}
__device__ __forceinline__ float group8_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 4));
}

__global__ void __launch_bounds__(IR * IL, 2)
gptq_inblock_kernel_v2(InblockArgs a) {
  extern __shared__ float sm[];
  float* Wr = sm;                        // [32 rows][136]   current (lazily updated) weights
  float* Et = Wr + IR * WP;              // [128 cols][33]   err (Err1 transposed)
  float* Hs = Et + GB * EP;              // [128 j][132]     Hs[j][k] = Hinv1[j][k]
  float* dd = Hs + GB * HP2;             // [128] Hinv1[c][c]
  float* rd = dd + GB;                   // [128] RN(1 / Hinv1[c][c])
  const int tid = threadIdx.x, rg = tid >> 3, l = tid & 7;
  const int warp = tid >> 5, lane = tid & 31;
  const int64_t r0 = static_cast<int64_t>(blockIdx.x) * IR;
  const int64_t row = r0 + rg;
  const bool live = row < a.R;
  const int cnt = a.count;

  {
    const bool vec = (cnt == GB) && ((a.C & 3) == 0) && ((reinterpret_cast<uintptr_t>(a.W) & 15) == 0) &&
                     ((reinterpret_cast<uintptr_t>(a.Hinv) & 15) == 0);
    if (vec) {
      float4 v[8];
#pragma unroll
      for (int b = 0; b < 4; ++b) {        // W tile: 32 rows x 32 float4
        const int item = b * (IR * IL) + tid;
        const int rr = item >> 5, c4 = item & 31;
        const int64_t r = r0 + rr;
        v[b] = (r < a.R) ? *reinterpret_cast<const float4*>(&a.W[r * a.C + a.i1 + c4 * 4])
                         : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int item = b * (IR * IL) + tid;
        const int rr = item >> 5, c4 = item & 31;
        *reinterpret_cast<float4*>(&Wr[rr * WP + c4 * 4]) = v[b];
      }
#pragma unroll 1
      for (int base = 0; base < GB * 32; base += 8 * IR * IL) {   // Hinv block: 128 rows x 32 float4
#pragma unroll
        for (int b = 0; b < 8; ++b) {
          const int item = base + b * (IR * IL) + tid;
          const int i = item >> 5, j4 = item & 31;
          v[b] = *reinterpret_cast<const float4*>(
              &a.Hinv[(static_cast<int64_t>(a.i1) + i) * a.C + a.i1 + j4 * 4]);
        }
#pragma unroll
        for (int b = 0; b < 8; ++b) {
          const int item = base + b * (IR * IL) + tid;
          const int i = item >> 5, j4 = item & 31;
          *reinterpret_cast<float4*>(&Hs[i * HP2 + j4 * 4]) = v[b];
        }
      }
    } else {
      for (int idx = tid; idx < IR * GB; idx += IR * IL) {
        const int rr = idx >> 7, c = idx & 127;
        const int64_t r = r0 + rr;
        Wr[rr * WP + c] = (r < a.R && c < cnt) ? a.W[r * a.C + a.i1 + c] : 0.f;
      }
      for (int idx = tid; idx < GB * GB; idx += IR * IL) {
        const int i = idx >> 7, j = idx & 127;
        Hs[i * HP2 + j] = (i < cnt && j < cnt) ? a.Hinv[(static_cast<int64_t>(a.i1) + i) * a.C + a.i1 + j]
                                               : 0.f;
      }
    }
  }
  __syncthreads();
  if (tid < GB) {
    const float d = (tid < cnt) ? Hs[tid * HP2 + tid] : 1.f;
    dd[tid] = d;
    rd[tid] = __frcp_rn(d);
  }

  // ---- qparams of the groups that start inside this block (gptq.py:215-223), searched on W as
  //      it stands at block entry (the reference indexes the global W, not the in-block clone)
  float s_cur = 1.f, z_cur = 0.f;
  const bool dynamic = !a.static_groups;
  const int gsz = static_cast<int>(a.group < GB ? a.group : GB);
  float s_small[8], z_small[8];
#pragma unroll
  for (int g = 0; g < 8; ++g) { s_small[g] = 1.f; z_small[g] = 0.f; }
  if (dynamic) {
    if (a.group >= GB) {
      const int64_t gi = a.i1 / a.group;
      if ((a.i1 % a.group) == 0) {
        float mn = INFINITY, mx = -INFINITY;
        const int64_t gend = min(static_cast<int64_t>(a.i1) + a.group, a.C);
        if (gend - a.i1 <= cnt) {
          for (int c = l; c < cnt; c += IL) { const float v = Wr[rg * WP + c]; mn = fminf(mn, v); mx = fmaxf(mx, v); }
        } else if (live) {
          for (int64_t c = a.i1 + l; c < gend; c += IL) { const float v = a.W[row * a.C + c]; mn = fminf(mn, v); mx = fmaxf(mx, v); }
        } else {
          mn = 0.f; mx = 0.f;
        }
        mn = group8_min(mn); mx = group8_max(mx);
        qparams_f32(mn, mx, a.sym, a.qmin, a.qmax, s_cur, z_cur);
        if (live && l == 0) {
          reinterpret_cast<float*>(a.scales)[row * a.ng + gi] = s_cur;
          if (!a.sym) reinterpret_cast<float*>(a.zeros)[row * a.ng + gi] = z_cur;
        }
      } else if (live) {                   // group opened by an earlier block
        s_cur = reinterpret_cast<const float*>(a.scales)[row * a.ng + gi];
        z_cur = a.sym ? 0.f : reinterpret_cast<const float*>(a.zeros)[row * a.ng + gi];
      }
    } else {
#pragma unroll
      for (int g = 0; g < 8; ++g) {
        if (g * gsz < cnt) {               // uniform across the CTA
          float mn = INFINITY, mx = -INFINITY;
          const int cend = min((g + 1) * gsz, cnt);
          for (int c = g * gsz + l; c < cend; c += IL) { const float v = Wr[rg * WP + c]; mn = fminf(mn, v); mx = fmaxf(mx, v); }
          mn = group8_min(mn); mx = group8_max(mx);
          qparams_f32(mn, mx, a.sym, a.qmin, a.qmax, s_small[g], z_small[g]);
          if (live && l == 0) {
            const int64_t gi = (a.i1 + g * gsz) / a.group;
            reinterpret_cast<float*>(a.scales)[row * a.ng + gi] = s_small[g];
            if (!a.sym) reinterpret_cast<float*>(a.zeros)[row * a.ng + gi] = z_small[g];
          }
        }
      }
    }
  } else if (live && a.group >= a.C) {
    s_cur = load_q(a.scales, a.q_dtype, row);                 // per_channel
    z_cur = a.zeros ? load_q(a.zeros, a.q_dtype, row) : 0.f;
  }
  __syncthreads();                         // dd / rd

  float loss = 0.f;
  const int nsb = (cnt + IL - 1) / IL;
#pragma unroll 1
  for (int m = 0; m < nsb; ++m) {
    const int cb = m * IL, c_own = cb + l;
    const bool col_live = c_own < cnt;
    float s = s_cur, z = z_cur;
    if (dynamic && a.group < GB) {
      const int g = cb / gsz;              // a sub-block of 8 never straddles a group (group >= 16)
#pragma unroll
      for (int t = 0; t < 8; ++t) { if (g == t) { s = s_small[t]; z = z_small[t]; } }
    } else if (!dynamic && a.group < a.C && live && col_live) {
      const int64_t idx = static_cast<int64_t>(a.i1) + c_own;
      const int64_t gi = a.gmap ? a.gmap[idx] : idx / a.group;     // gptq.py:225-227
      s = load_q(a.scales, a.q_dtype, row * a.ng + gi);
      z = a.zeros ? load_q(a.zeros, a.q_dtype, row * a.ng + gi) : 0.f;
    }
    const float rs = __frcp_rn(s);
    const bool s_ok = exp_mid(s) && exp_mid(rs);
    float wc = Wr[rg * WP + c_own];
    float hd[IL];
#pragma unroll
    for (int jj = 0; jj < IL; ++jj) hd[jj] = Hs[(cb + jj) * HP2 + c_own];
    const float d = dd[c_own], rdv = rd[c_own];
    const bool d_ok = exp_mid(d) && exp_mid(rdv);
    float ev[IL];
    float my_err = 0.f, my_diff = 0.f;
    // the eight sequential columns of the sub-block: lane jj's column is final at step jj
#pragma unroll
    for (int jj = 0; jj < IL; ++jj) {
      const float q = qdq_f32_r(wc, s, rs, s_ok, z, a.qmin, a.qmax);
      const float diff = fsub_rn(wc, q);
      float err = div_by(diff, d, rdv, d_ok);                                       // :239
      if (!col_live) err = 0.f;
      const float e = __shfl_sync(0xffffffffu, err, jj, IL);
      ev[jj] = e;
      if (l == jj) { my_err = err; my_diff = diff; }
      if (l > jj) wc = fsub_rn(wc, fmul_rn(e, hd[jj]));                       // :240
    }
    if (col_live) loss += fdiv_rn(fmul_rn(my_diff, my_diff), fmul_rn(2.f, fmul_rn(d, d)));   // :238
    Wr[rg * WP + c_own] = wc;              // tmp: the compensated, not yet rounded weight (:237)
    Et[c_own * EP + rg] = my_err;          // Err1 (:241)
    // lazy propagation of the sub-block's eight errors to the later columns this lane owns
    int mp = m + 1;
    for (; mp + 3 < nsb; mp += 4) {
      float w0 = Wr[rg * WP + (mp + 0) * IL + l], w1 = Wr[rg * WP + (mp + 1) * IL + l];
      float w2 = Wr[rg * WP + (mp + 2) * IL + l], w3 = Wr[rg * WP + (mp + 3) * IL + l];
      const float* hp = Hs + cb * HP2 + mp * IL + l;
#pragma unroll
      for (int jj = 0; jj < IL; ++jj) {
        w0 = fsub_rn(w0, fmul_rn(ev[jj], hp[jj * HP2]));
        w1 = fsub_rn(w1, fmul_rn(ev[jj], hp[jj * HP2 + IL]));
        w2 = fsub_rn(w2, fmul_rn(ev[jj], hp[jj * HP2 + 2 * IL]));
        w3 = fsub_rn(w3, fmul_rn(ev[jj], hp[jj * HP2 + 3 * IL]));
      }
      Wr[rg * WP + (mp + 0) * IL + l] = w0; Wr[rg * WP + (mp + 1) * IL + l] = w1;
      Wr[rg * WP + (mp + 2) * IL + l] = w2; Wr[rg * WP + (mp + 3) * IL + l] = w3;
    }
    for (; mp < nsb; ++mp) {
      float w0 = Wr[rg * WP + mp * IL + l];
      const float* hp = Hs + cb * HP2 + mp * IL + l;
#pragma unroll
      for (int jj = 0; jj < IL; ++jj) w0 = fsub_rn(w0, fmul_rn(ev[jj], hp[jj * HP2]));
      Wr[rg * WP + mp * IL + l] = w0;
    }
  }
  loss += __shfl_xor_sync(0xffffffffu, loss, 4);
  loss += __shfl_xor_sync(0xffffffffu, loss, 2);
  loss += __shfl_xor_sync(0xffffffffu, loss, 1);
  if (live && l == 0) a.losses[row] += loss;
  __syncthreads();
  // write-back: tmp[:, invperm] (gptq.py:186-188) fused as a scatter — permuted column i1+c goes
  // back to original column perm[i1+c] — and Err1 transposed ([k][row], so the trailing GEMM
  // reads its A operand with unit stride) with its tf32 split
  for (int rr = warp; rr < IR; rr += (IR * IL) / 32) {
    const int64_t r = r0 + rr;
    if (r >= a.R) break;
    for (int c = lane; c < cnt; c += 32) {
      const int64_t oc = a.out_perm ? a.out_perm[a.i1 + c] : static_cast<int64_t>(a.i1) + c;
      a.tmp[r * a.C + oc] = Wr[rr * WP + c];
    }
  }
  if (r0 + lane < a.Rpad) {
    for (int c = warp; c < GB; c += (IR * IL) / 32) {
      const float evv = (c < cnt) ? Et[c * EP + lane] : 0.f;
      const int64_t o = static_cast<int64_t>(c) * a.Rpad + r0 + lane;
      a.err[o] = evv;
      uint32_t hb, lb;                                   // tf32 split for the 3xTF32 trailing GEMM
      asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(evv));
      const float h = __uint_as_float(hb);
      asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(lb) : "f"(evv - h));
      a.err_hi[o] = h;
      a.err_lo[o] = __uint_as_float(lb);
    }
  }
}


// ---- SpQR in-block kernel (spqr.py:215-268) ------------------------------------------------------------------
// Same role as gptq_inblock_kernel for the SpQR sweep: one thread owns one weight row of the
// 128-column block (rows are independent), the row tile / Hinv block / Err1 / outlier mask live in
// shared memory, and ALL arithmetic is spqr::row_block() of spqr_row.cuh — the function the CPU tests
// run on the host against the oracle.  Per group of `gs` columns: leave-one-out outlier search
// (gs * (gs - 1) quantise-dequantise evaluations per row), bilevel (scale / zero) quantisation; per
// column: quantise, unstructured outlier mask, rank-1 update of the block's remaining columns.
struct SpqrArgs {
  float* W;
  const float* Hinv;
  int64_t R, C, Rpad;
  int i1, count;
  int64_t ng;
  spqr::Cfg cfg;             // thr / has_thr / outliers are filled in by the kernel from `thr`
  const float* thr;          // device scalar: relative_threshold * outlier_scale (may be +inf)
  int simplified;
  float* scales;             // [R, ng] out
  float* zeros;              // [R, ng] out
  float* tmp;                // [R, C] out
  uint8_t* mask;             // [R, C] out
  const int64_t* out_perm;
  float* losses;
  float* err; float* err_hi; float* err_lo;
};

constexpr int kSpqrMaskPitch = GB + 16;
constexpr int kSpqrSmem = (2 * GB * kPad + GB * HP) * 4 + GB * kSpqrMaskPitch;

__global__ void __launch_bounds__(GB, 1)
spqr_inblock_kernel(SpqrArgs a) {
  extern __shared__ float sm[];
  float* Wt = sm;                       // [col][row]  pitch kPad
  float* Et = Wt + GB * kPad;           // [col][row]
  float* Ht = Et + GB * kPad;           // Ht[j * HP + i] = Hinv1[i][j], upper triangle
  uint8_t* Mt = reinterpret_cast<uint8_t*>(Ht + GB * HP);   // [col][row] pitch kSpqrMaskPitch
  const int tid = threadIdx.x;
  const int64_t r0 = static_cast<int64_t>(blockIdx.x) * GB;
  const int64_t row = r0 + tid;
  const int cnt = a.count;
  {
    const int warp = tid >> 5, lane = tid & 31;
    for (int rr = warp; rr < GB; rr += 4) {
      const int64_t r = r0 + rr;
      for (int c = lane; c < GB; c += 32) {
        float v = 0.f;
        if (r < a.R && c < cnt) v = a.W[r * a.C + a.i1 + c];
        Wt[c * kPad + rr] = v;
      }
    }
    for (int i = warp; i < GB; i += 4)
      for (int j = lane; j < GB; j += 32) {
        float v = (i == j) ? 1.f : 0.f;
        if (i < cnt && j < cnt && j >= i)
          v = a.Hinv[(static_cast<int64_t>(a.i1) + i) * a.C + a.i1 + j];
        Ht[j * HP + i] = v;
      }
    for (int idx = tid; idx < GB * kSpqrMaskPitch; idx += GB) Mt[idx] = 0;
    for (int idx = tid; idx < GB * kPad; idx += GB) Et[idx] = 0.f;
  }
  __syncthreads();
  if (row < a.R) {
    spqr::Cfg cfg = a.cfg;
    cfg.thr = a.thr[0];
    cfg.has_thr = !isinf(cfg.thr);
    cfg.outliers = (!a.simplified && cfg.has_thr) ? 1 : 0;
    float s_out[GB / 16], z_out[GB / 16];
    const float loss = spqr::row_block(Wt + tid, kPad, Ht, 1, HP, cnt, cfg, Et + tid, kPad,
                                       Mt + tid, kSpqrMaskPitch, s_out, z_out);
    a.losses[row] += loss;
    const int64_t g0 = a.i1 / cfg.gs;
    for (int g = 0; g * cfg.gs < cnt; ++g) {
      a.scales[row * a.ng + g0 + g] = s_out[g];
      a.zeros[row * a.ng + g0 + g] = z_out[g];
    }
  }
  __syncthreads();
  {
    const int warp = tid >> 5, lane = tid & 31;
    for (int rr = warp; rr < GB; rr += 4) {
      const int64_t r = r0 + rr;
      if (r >= a.R) break;
      for (int c = lane; c < cnt; c += 32) {
        // tmp[:, invperm] / mask[:, invperm] (spqr.py:163-165) fused as a scatter
        const int64_t oc = a.out_perm ? a.out_perm[a.i1 + c] : static_cast<int64_t>(a.i1) + c;
        a.tmp[r * a.C + oc] = Wt[c * kPad + rr];
        a.mask[r * a.C + oc] = Mt[c * kSpqrMaskPitch + rr];
      }
    }
    for (int c = warp; c < GB; c += 4)
      for (int rr = lane; rr < GB; rr += 32) {
        const float ev = (c < cnt) ? Et[c * kPad + rr] : 0.f;
        const int64_t o = static_cast<int64_t>(c) * a.Rpad + r0 + rr;
        a.err[o] = ev;
        uint32_t hb, lb;                                   // tf32 split for the 3xTF32 trailing GEMM
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(ev));
        const float h = __uint_as_float(hb);
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(lb) : "f"(ev - h));
        a.err_hi[o] = h;
        a.err_lo[o] = __uint_as_float(lb);
      }
  }
}


// ---- SpQR in-block kernel, 16 lanes per weight row ----------------------------------------------------------
// spqr_inblock_kernel above gives a row to ONE thread: 32 CTAs for R = 4096, one warp per scheduler,
// 887 us per 128-column block (profiles/r02_microbench_spqr.txt).  Here a row is spread over 16 lanes
// (16 rows per CTA, 256 threads, two CTAs per SM): lane j evaluates the leave-one-out cases j,
// j + 16, ... of a group, every lane recomputes the cheap group statistics, and after the (redundant)
// quantise -> err step of a column each lane applies the rank-1 update to the later columns it owns.
// The three phases are spqr::lanes_* of spqr_row.cuh — bit-identical to row_block() by construction,
// checked on the host (lock-step emulation) by the CPU tests and on the GPU against the kernel above
// (1000 x 1024, g16: 6.8 -> 1.2 ms).  Lanes talk through the row's
// shared-memory storage, with __syncwarp() between phases.
constexpr int SL = 16;            // lanes per row
constexpr int SR = 16;            // rows per CTA
constexpr int SWP = GB + 16;      // pitch of a W row: the two rows of a warp sit 16 banks apart
constexpr int SHP = GB + 4;       // pitch of the row-major Hinv block
constexpr int SEP = SR + 1;       // pitch of the transposed err tile
constexpr int kSpqrLanesSmem = (SR * SWP + GB * SHP + GB * SEP) * 4 + 2 * SR * GB;

__global__ void __launch_bounds__(SR * SL, 2)
spqr_inblock_lanes_kernel(SpqrArgs a) {
  extern __shared__ float sm[];
  float* Ws = sm;                        // [row][col]   current (in place updated) weights
  float* Hs = Ws + SR * SWP;             // [i][j]       Hinv1, upper triangle
  float* Et = Hs + GB * SHP;             // [col][row]   Err1 transposed
  uint8_t* Ms = reinterpret_cast<uint8_t*>(Et + GB * SEP);   // [row][col] outlier mask
  uint8_t* Fl = Ms + SR * GB;                                // [row][k]   leave-one-out flags of the group
  const int tid = threadIdx.x, rr = tid / SL, lane = tid % SL;
  const int64_t r0 = static_cast<int64_t>(blockIdx.x) * SR;
  const int64_t row = r0 + rr;
  const int cnt = a.count;
  for (int idx = tid; idx < SR * GB; idx += SR * SL) {
    const int r = idx >> 7, c = idx & 127;
    float v = 0.f;
    if (r0 + r < a.R && c < cnt) v = a.W[(r0 + r) * a.C + a.i1 + c];
    Ws[r * SWP + c] = v;
    Ms[idx] = 0;
    Fl[idx] = 0;
  }
  for (int idx = tid; idx < GB * GB; idx += SR * SL) {
    const int i = idx >> 7, j = idx & 127;
    float v = (i == j) ? 1.f : 0.f;
    if (i < cnt && j < cnt && j >= i) v = a.Hinv[(static_cast<int64_t>(a.i1) + i) * a.C + a.i1 + j];
    Hs[i * SHP + j] = v;
  }
  for (int idx = tid; idx < GB * SEP; idx += SR * SL) Et[idx] = 0.f;
  __syncthreads();
  const bool live = row < a.R;
  spqr::Cfg cfg = a.cfg;
  cfg.thr = a.thr[0];
  cfg.has_thr = !isinf(cfg.thr);
  cfg.outliers = (!a.simplified && cfg.has_thr) ? 1 : 0;
  float* w = Ws + rr * SWP;
  uint8_t* fl = Fl + rr * GB;
  float loss = 0.f, s = 1.f, z = 0.f;
  for (int col = 0; col < cnt; ++col) {
    if (col % cfg.gs == 0) {
      if (live) spqr::lanes_group_flags(w + col, 1, Hs + col * SHP + col, SHP + 1, cfg, lane, SL, fl);
      __syncwarp();
      if (live) {
        spqr::lanes_group_qparams(w + col, 1, fl, cfg, s, z);
        if (lane == 0) {
          const int64_t gi = (static_cast<int64_t>(a.i1) + col) / cfg.gs;
          a.scales[row * a.ng + gi] = s;
          a.zeros[row * a.ng + gi] = z;
        }
      }
      __syncwarp();
    }
    float err = 0.f;
    uint8_t m = 0;
    if (live) err = spqr::lanes_column(w, 1, Hs, SHP, 1, cnt, col, s, z, cfg, lane, SL, m);
    if (live && lane == 0) {
      Et[col * SEP + rr] = err;
      Ms[rr * GB + col] = m;
      loss = spqr::add(loss, spqr::mul(err, err));
    }
    __syncwarp();
  }
  if (live && lane == 0) a.losses[row] += loss;
  __syncthreads();
  for (int idx = tid; idx < SR * GB; idx += SR * SL) {
    const int r = idx >> 7, c = idx & 127;
    if (r0 + r < a.R && c < cnt) {
      const int64_t oc = a.out_perm ? a.out_perm[a.i1 + c] : static_cast<int64_t>(a.i1) + c;
      a.tmp[(r0 + r) * a.C + oc] = Ws[r * SWP + c];
      a.mask[(r0 + r) * a.C + oc] = Ms[idx];
    }
  }
  for (int idx = tid; idx < GB * SR; idx += SR * SL) {
    const int c = idx / SR, r = idx % SR;
    const float ev = (c < cnt) ? Et[c * SEP + r] : 0.f;
    const int64_t o = static_cast<int64_t>(c) * a.Rpad + r0 + r;
    a.err[o] = ev;
    uint32_t hb, lb;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(ev));
    const float h = __uint_as_float(hb);
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(lb) : "f"(ev - h));
    a.err_hi[o] = h;
    a.err_lo[o] = __uint_as_float(lb);
  }
}

// ---- trailing update: W[:, n0:] -= Err[R,128] @ Hinv[i1:i1+128, n0:] ---------------------------------------
// fp32 SIMT GEMM, 128x128 tile, 8x8 per thread, K = 128 resident in shared memory.
constexpr int TT = 128;
__global__ void __launch_bounds__(256, 1)
trailing_update_kernel(float* __restrict__ W, int64_t R, int64_t Rpad, int64_t C, const float* __restrict__ Err,
                       const float* __restrict__ Hinv, int i1, int kcount, int64_t n0) {
  extern __shared__ float sm[];
  float* As = sm;               // [k][m]  (Err transposed), 128 x 128
  float* Bs = sm + TT * TT;     // [k][n]
  const int tid = threadIdx.x;
  const int64_t m0 = static_cast<int64_t>(blockIdx.y) * TT;
  const int64_t nb0 = n0 + static_cast<int64_t>(blockIdx.x) * TT;
  // load A: ErrT[k][Rpad] (k-major) -> As[k][m], unit stride both sides (Rpad % 128 == 0)
  for (int idx = tid; idx < TT * TT / 4; idx += 256) {
    const int k = idx >> 5;            // 32 float4 per k row
    const int m4 = (idx & 31) << 2;
    *reinterpret_cast<float4*>(&As[k * TT + m4]) =
        *reinterpret_cast<const float4*>(&Err[static_cast<int64_t>(k) * Rpad + m0 + m4]);
  }
  // load B: Hinv rows i1..i1+kcount-1, cols nb0..nb0+127
  for (int idx = tid; idx < TT * TT; idx += 256) {
    const int k = idx >> 7, n = idx & 127;
    float v = 0.f;
    if (k < kcount && nb0 + n < C) v = Hinv[(static_cast<int64_t>(i1) + k) * C + nb0 + n];
    Bs[k * TT + n] = v;
  }
  __syncthreads();
  const int tx = tid & 15, ty = tid >> 4;       // 16 x 16 threads; thread tile 8 x 8
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
#pragma unroll 4
  for (int k = 0; k < TT; ++k) {
    const float4 a0 = *reinterpret_cast<const float4*>(&As[k * TT + ty * 4]);
    const float4 a1 = *reinterpret_cast<const float4*>(&As[k * TT + 64 + ty * 4]);
    const float4 b0 = *reinterpret_cast<const float4*>(&Bs[k * TT + tx * 4]);
    const float4 b1 = *reinterpret_cast<const float4*>(&Bs[k * TT + 64 + tx * 4]);
    const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
    const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    if (m >= R) continue;
#pragma unroll
    for (int jh = 0; jh < 2; ++jh) {
      const int64_t n = nb0 + jh * 64 + tx * 4;
      float* wp = &W[m * C + n];
      if (n + 3 < C && ((reinterpret_cast<uintptr_t>(wp) & 15) == 0)) {
        float4 v = *reinterpret_cast<float4*>(wp);
        v.x -= acc[i][jh * 4 + 0]; v.y -= acc[i][jh * 4 + 1];
        v.z -= acc[i][jh * 4 + 2]; v.w -= acc[i][jh * 4 + 3];
        *reinterpret_cast<float4*>(wp) = v;
      } else {
        for (int j = 0; j < 4; ++j)
          if (n + j < C) wp[j] -= acc[i][jh * 4 + j];
      }
    }
  }
}

}  // namespace llmc

using namespace llmc;

extern "C" int llmc_gptq_prepare(const float* H, int64_t C, const int64_t* perm, float percdamp,
                                 float* Hp, const void* W, int64_t R, int w_dtype, float* Wp,
                                 float* diag_scratch, void* stream) {
  // Hp == NULL skips the Hessian gather, W == NULL the weight gather (linears that share one
  // Hessian need Hp once and one Wp each)
  LLMC_CHECK_ARG(H && (Hp || W) && (!W || (Wp && R > 0)) && diag_scratch && C > 0, "gptq_prepare: bad argument");
  LLMC_CHECK_ARG(C * 4 <= 200 * 1024, "gptq_prepare: C=%lld exceeds the shared-memory row buffer",
                 (long long)C);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int smem = static_cast<int>(C * 4);
  LLMC_ONCE_PER_DEVICE({
    LLMC_CHECK_CUDA(cudaFuncSetAttribute(gather_h_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    LLMC_CHECK_CUDA(cudaFuncSetAttribute(gather_w_kernel<LLMC_F32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    LLMC_CHECK_CUDA(cudaFuncSetAttribute(gather_w_kernel<LLMC_F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    LLMC_CHECK_CUDA(cudaFuncSetAttribute(gather_w_kernel<LLMC_BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  });
  diag_mean_kernel<<<1, 256, 0, st>>>(H, C, percdamp, diag_scratch);
  LLMC_CHECK_LAUNCH();
  // W first: it reads the ORIGINAL diagonal of H (dead test), Hp may alias neither H nor W
  if (W != nullptr) {
    if (w_dtype == LLMC_F32) gather_w_kernel<LLMC_F32><<<(unsigned)R, 256, smem, st>>>(W, R, C, H, perm, Wp);
    else if (w_dtype == LLMC_F16) gather_w_kernel<LLMC_F16><<<(unsigned)R, 256, smem, st>>>(W, R, C, H, perm, Wp);
    else if (w_dtype == LLMC_BF16) gather_w_kernel<LLMC_BF16><<<(unsigned)R, 256, smem, st>>>(W, R, C, H, perm, Wp);
    else { set_last_error("gptq_prepare: bad dtype %d", w_dtype); return LLMC_EINVAL; }
    LLMC_CHECK_LAUNCH();
  }
  if (Hp != nullptr) {
    gather_h_kernel<<<(unsigned)C, 256, smem, st>>>(H, C, perm, diag_scratch, Hp);
    LLMC_CHECK_LAUNCH();
  }
  return LLMC_OK;
}

// The schedule shared by the GPTQ and SpQR sweeps: in-block kernel per 128 columns (launched by
// `launch_inblock(i1, count, err, err_hi, err_lo, stream)`), lazy trailing updates per super-panel
// and the look-ahead split of the bulk update.  `wide_dynamic_group`: the in-block kernel reads
// columns beyond its super-panel (a dynamic group wider than 512), which the look-ahead cannot
// order.
template <class F>
static int sweep_schedule(float* W, const float* Hinv, int64_t R, int64_t C, int64_t group,
                          bool wide_dynamic_group, void* workspace, cudaStream_t st, F&& launch_inblock) {
  const int tr_smem = 2 * TT * TT * 4;                     // 131,072 B
  const int64_t Rpad = ((R + GB - 1) / GB) * GB;
  // [512][Rpad] x {err, hi, lo}, two sets selected by the parity of the super-panel
  float* const err_set[2] = {reinterpret_cast<float*>(workspace),
                             reinterpret_cast<float*>(workspace) + 3 * kSuperPanel * Rpad};
  float* Hh = err_set[1] + 3 * kSuperPanel * Rpad;
  float* Hl = Hh + C * C;
  // trailing updates on tensor cores (3xTF32) when the shapes allow TMA; fp32 SIMT otherwise
  // LLMC_B200_SIMT_TRAILING=1 forces the fp32 CUDA-core kernel (A/B comparisons in tests only)
  static const bool force_simt = getenv("LLMC_B200_SIMT_TRAILING") != nullptr;
  const bool tensor_trailing = !force_simt && (C % 8 == 0) && aligned16(W) && aligned16(Hinv) &&
                               aligned16(workspace);
  if (tensor_trailing && C > GB) {
    if (int rc = split_tf32(Hinv, C, C, C, Hh, Hl, C, st)) return rc;
  }
  // super-panel width: 512 on the tensor path, one block (the reference's schedule) otherwise
  // (a dynamic group is searched on W[:, start : start+group] at its first column, so a group
  // must never reach past the super-panel it starts in unless it starts with it)
  const bool groups_fit = group <= GB || kSuperPanel % group == 0 || group % kSuperPanel == 0;
  const int64_t sp_width = (tensor_trailing && groups_fit) ? kSuperPanel : GB;
  // ---- look-ahead schedule ------------------------------------------------------------------
  // The sweep's dependent chain is  in-block kernel -> in-panel update -> next in-block kernel
  // (~90 us per 128 columns); the rank-512 update of everything beyond a super-panel is 25-35 % of
  // the sweep's time at R >= 4096 and is NOT on that chain beyond the next 512 columns.  So at a
  // super-panel boundary the chain (high-priority stream) updates the next super-panel's columns
  // only, and the rest goes to a low-priority stream, one tile per CTA, overlapping the next
  // panel's chain.  Every column receives its panel updates in the same order as before (events),
  // and a 3xTF32 tile's value does not depend on how the N range is cut, so results are
  // bit-identical to the serial schedule (LLMC_B200_SWEEP_LOOKAHEAD=0 selects it).
  const char* la_env = getenv("LLMC_B200_SWEEP_LOOKAHEAD");      // read per call: tests toggle it
  const bool la_off = la_env != nullptr && la_env[0] == '0';
  // (a dynamic group wider than a super-panel is searched on columns a bulk piece may still be
  //  updating: those sweeps keep the serial schedule)
  const bool lookahead = !la_off && tensor_trailing && sp_width == kSuperPanel && C > 2 * kSuperPanel &&
                         !wide_dynamic_group;
  constexpr int kMaxDev = 64;
  static cudaStream_t hi_of[kMaxDev] = {}, bulk_of[kMaxDev] = {};
  static cudaEvent_t fork_of[kMaxDev] = {}, join_of[kMaxDev][2] = {}, panel_of[kMaxDev][2] = {}, bulkdone_of[kMaxDev][2] = {};
  cudaStream_t chain = st, bulk = st;
  int dev_id = 0;
  if (lookahead) {
    LLMC_CHECK_CUDA(cudaGetDevice(&dev_id));
    dev_id &= kMaxDev - 1;
    if (hi_of[dev_id] == nullptr) {
      int least = 0, greatest = 0;
      LLMC_CHECK_CUDA(cudaDeviceGetStreamPriorityRange(&least, &greatest));
      LLMC_CHECK_CUDA(cudaStreamCreateWithPriority(&hi_of[dev_id], cudaStreamNonBlocking, greatest));
      LLMC_CHECK_CUDA(cudaStreamCreateWithPriority(&bulk_of[dev_id], cudaStreamNonBlocking, least));
      LLMC_CHECK_CUDA(cudaEventCreateWithFlags(&fork_of[dev_id], cudaEventDisableTiming));
      for (int i = 0; i < 2; ++i) {
        LLMC_CHECK_CUDA(cudaEventCreateWithFlags(&join_of[dev_id][i], cudaEventDisableTiming));
        LLMC_CHECK_CUDA(cudaEventCreateWithFlags(&panel_of[dev_id][i], cudaEventDisableTiming));
        LLMC_CHECK_CUDA(cudaEventCreateWithFlags(&bulkdone_of[dev_id][i], cudaEventDisableTiming));
      }
    }
    chain = hi_of[dev_id];
    bulk = bulk_of[dev_id];
    LLMC_CHECK_CUDA(cudaEventRecord(fork_of[dev_id], st));
    LLMC_CHECK_CUDA(cudaStreamWaitEvent(chain, fork_of[dev_id], 0));
  }
  bool bulk_pending[2] = {false, false};        // a bulk update of that parity has been enqueued
  for (int64_t i1 = 0; i1 < C; i1 += GB) {
    const int64_t i2 = (i1 + GB < C) ? i1 + GB : C;
    const int64_t sp0 = (i1 / sp_width) * sp_width;
    const int64_t sp1 = (sp0 + sp_width < C) ? sp0 + sp_width : C;
    const int par = static_cast<int>((i1 / sp_width) & 1);
    float* err_base = err_set[par];
    float* errh_base = err_base + kSuperPanel * Rpad;
    float* errl_base = errh_base + kSuperPanel * Rpad;
    const int b_i1 = static_cast<int>(i1);
    const int b_count = static_cast<int>(i2 - i1);
    float* const b_err = err_base + (i1 - sp0) * Rpad;
    float* const b_err_hi = errh_base + (i1 - sp0) * Rpad;
    float* const b_err_lo = errl_base + (i1 - sp0) * Rpad;
    if (int rc = launch_inblock(b_i1, b_count, b_err, b_err_hi, b_err_lo, chain)) return rc;
    if (i2 < C && tensor_trailing) {
      // W[:, i2:] -= Err1 @ Hinv[i1:i2, i2:]   (gptq.py:244): A = Err1^T (MN-major, ld Rpad),
      // B = Hinv rows (MN-major, ld C).  Inside the super-panel: this block's errors onto the
      // super-panel's remaining columns; at its end: all of its errors onto everything beyond.
      if (i2 < sp1) {
        if (int rc = tf32x3_update({.Ahi = b_err_hi, .Alo = b_err_lo, .a_mn = 1, .lda = Rpad,
                                    .Bhi = Hh + i1 * C + i2, .Blo = Hl + i1 * C + i2, .b_mn = 1, .ldb = C,
                                    .C = W + i2, .ldc = C, .M = R, .N = sp1 - i2, .K = b_count,
                                    .mode = 0},
                                   chain))
          return rc;
      } else if (!lookahead) {
        if (int rc = tf32x3_update({.Ahi = errh_base, .Alo = errl_base, .a_mn = 1, .lda = Rpad,
                                    .Bhi = Hh + sp0 * C + sp1, .Blo = Hl + sp0 * C + sp1, .b_mn = 1, .ldb = C,
                                    .C = W + sp1, .ldc = C, .M = R, .N = C - sp1,
                                    .K = static_cast<int>(sp1 - sp0), .mode = 0},
                                   chain))
          return rc;
      } else {
        const int kk = static_cast<int>(sp1 - sp0);
        const int64_t nx1 = (sp1 + sp_width < C) ? sp1 + sp_width : C;
        // the errors of this panel are complete: the bulk piece may start (after the previous one)
        LLMC_CHECK_CUDA(cudaEventRecord(panel_of[dev_id][par], chain));
        // chain: the next super-panel's columns, last written by the previous panel's bulk piece
        if (bulk_pending[par ^ 1]) LLMC_CHECK_CUDA(cudaStreamWaitEvent(chain, bulkdone_of[dev_id][par ^ 1], 0));
        if (int rc = tf32x3_update({.Ahi = errh_base, .Alo = errl_base, .a_mn = 1, .lda = Rpad,
                                    .Bhi = Hh + sp0 * C + sp1, .Blo = Hl + sp0 * C + sp1, .b_mn = 1, .ldb = C,
                                    .C = W + sp1, .ldc = C, .M = R, .N = nx1 - sp1, .K = kk, .mode = 0},
                                   chain))
          return rc;
        // bulk: everything beyond.  After this wait the chain goes on to write the OTHER error set,
        // which the previous bulk piece (just waited for) was the last reader of.
        if (nx1 < C) {
          LLMC_CHECK_CUDA(cudaStreamWaitEvent(bulk, panel_of[dev_id][par], 0));
          if (int rc = tf32x3_update({.Ahi = errh_base, .Alo = errl_base, .a_mn = 1, .lda = Rpad,
                                      .Bhi = Hh + sp0 * C + nx1, .Blo = Hl + sp0 * C + nx1, .b_mn = 1, .ldb = C,
                                      .C = W + nx1, .ldc = C, .M = R, .N = C - nx1, .K = kk, .mode = 0,
                                      .one_tile_per_cta = 1},
                                     bulk))
            return rc;
          LLMC_CHECK_CUDA(cudaEventRecord(bulkdone_of[dev_id][par], bulk));
          bulk_pending[par] = true;
        }
      }
    } else if (i2 < C) {
      dim3 grid(static_cast<unsigned>((C - i2 + TT - 1) / TT), static_cast<unsigned>((R + TT - 1) / TT));
      trailing_update_kernel<<<grid, 256, tr_smem, chain>>>(W, R, Rpad, C, b_err, Hinv, b_i1, b_count, i2);
      LLMC_CHECK_LAUNCH();
    }
  }
  if (lookahead) {
    LLMC_CHECK_CUDA(cudaEventRecord(join_of[dev_id][0], chain));
    LLMC_CHECK_CUDA(cudaEventRecord(join_of[dev_id][1], bulk));
    LLMC_CHECK_CUDA(cudaStreamWaitEvent(st, join_of[dev_id][0], 0));
    LLMC_CHECK_CUDA(cudaStreamWaitEvent(st, join_of[dev_id][1], 0));
  }
  return LLMC_OK;
}

extern "C" int64_t llmc_gptq_workspace_bytes(int64_t R, int64_t C) {
  // Err1^T + its tf32 split for TWO super-panels ([512, Rpad] x 3 each: the bulk trailing update
  // of panel p reads its errors while the chain of panel p+1 writes the other set) and the tf32
  // split of Hinv ([C, C] x 2)
  const int64_t rpad = ((R + GB - 1) / GB) * GB;
  return (6 * kSuperPanel * rpad + 2 * C * C) * 4;
}

extern "C" int llmc_gptq_colblock(float* W, const float* Hinv, int64_t R, int64_t C, int64_t group,
                                  int bit, int sym, int static_groups, const int32_t* gmap,
                                  void* scales, void* zeros, int q_dtype, float* tmp,
                                  const int64_t* out_perm, float* losses, void* workspace,
                                  int64_t workspace_bytes, void* stream) {
  LLMC_CHECK_ARG(W && Hinv && tmp && losses && workspace && R > 0 && C > 0, "gptq_colblock: bad argument");
  LLMC_CHECK_ARG(bit >= 2 && bit <= 8, "gptq_colblock: bit %d outside 2..8", bit);
  LLMC_CHECK_ARG(group > 0 && group <= C && C % group == 0, "gptq_colblock: C=%lld %% group=%lld != 0",
                 (long long)C, (long long)group);
  LLMC_CHECK_ARG((group >= C) || (group >= GB ? group % GB == 0 : (GB % group == 0 && GB / group <= 8)),
                 "gptq_colblock: group %lld must divide or be a multiple of the block size 128 "
                 "(and be >= 16)", (long long)group);
  LLMC_CHECK_ARG(scales, "gptq_colblock: scales is NULL");
  LLMC_CHECK_ARG(sym || zeros, "gptq_colblock: zeros is NULL for asymmetric quantisation");
  LLMC_CHECK_ARG(static_groups || q_dtype == LLMC_F32, "gptq_colblock: dynamic groups write fp32 qparams");
  LLMC_CHECK_ARG(workspace_bytes >= llmc_gptq_workspace_bytes(R, C), "gptq_colblock: workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int in_smem = (2 * GB * kPad + GB * HP) * 4;       // 199,680 B
  const int tr_smem = 2 * TT * TT * 4;                     // 131,072 B
  LLMC_ONCE_PER_DEVICE({
    LLMC_CHECK_CUDA(cudaFuncSetAttribute(gptq_inblock_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, in_smem));
    LLMC_CHECK_CUDA(cudaFuncSetAttribute(trailing_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tr_smem));
    LLMC_CHECK_CUDA(cudaFuncSetAttribute(gptq_inblock_kernel_v2, cudaFuncAttributeMaxDynamicSharedMemorySize, kInblockV2Smem));
  });
  // LLMC_B200_INBLOCK_V1=1 selects the thread-per-row kernel (A/B comparisons in tests only)
  const char* v1env = getenv("LLMC_B200_INBLOCK_V1");
  const bool inblock_v1 = v1env != nullptr && v1env[0] == '1';
  LLMC_CHECK_CUDA(cudaMemsetAsync(losses, 0, R * sizeof(float), st));
  InblockArgs a{};
  a.W = W; a.Hinv = Hinv; a.R = R; a.C = C;
  a.group = group; a.ng = C / group; a.sym = sym;
  if (sym) { a.qmin = -(float)(1 << (bit - 1)); a.qmax = (float)((1 << (bit - 1)) - 1); }
  else { a.qmin = 0.f; a.qmax = (float)((1 << bit) - 1); }
  a.static_groups = static_groups; a.gmap = gmap;
  a.scales = scales; a.zeros = sym ? nullptr : zeros; a.q_dtype = q_dtype;
  a.tmp = tmp; a.out_perm = out_perm; a.losses = losses;
  const unsigned row_blocks = static_cast<unsigned>((R + GB - 1) / GB);
  a.Rpad = static_cast<int64_t>(row_blocks) * GB;
  const bool wide = !static_groups && group > kSuperPanel;
  return sweep_schedule(W, Hinv, R, C, group, wide, workspace, st,
                        [&](int i1, int count, float* err, float* err_hi, float* err_lo, cudaStream_t cs) -> int {
    a.i1 = i1; a.count = count; a.err = err; a.err_hi = err_hi; a.err_lo = err_lo;
    if (inblock_v1) gptq_inblock_kernel<<<row_blocks, GB, in_smem, cs>>>(a);
    else gptq_inblock_kernel_v2<<<static_cast<unsigned>(a.Rpad / IR), IR * IL, kInblockV2Smem, cs>>>(a);
    LLMC_CHECK_LAUNCH();
    return LLMC_OK;
  });
}

static spqr::QCfg spqr_qcfg(int bit, int sym, int round_zp) {
  spqr::QCfg q{};
  if (sym) { q.qmin = -static_cast<float>(1 << (bit - 1)); q.qmax = static_cast<float>((1 << (bit - 1)) - 1); }
  else { q.qmin = 0.f; q.qmax = static_cast<float>((1 << bit) - 1); }
  q.sym = sym; q.round_zp = round_zp;
  return q;
}

extern "C" int llmc_spqr_colblock(float* W, const float* Hinv, int64_t R, int64_t C, int64_t group,
                                  int bit, int sym, int round_zp, int s_bit, int s_sym, int s_round_zp,
                                  int z_bit, int z_sym, int z_round_zp, const float* threshold,
                                  int simplified_outliers, float* scales, float* zeros, float* tmp,
                                  uint8_t* mask, const int64_t* out_perm, float* losses, void* workspace,
                                  int64_t workspace_bytes, void* stream) {
  LLMC_CHECK_ARG(W && Hinv && tmp && mask && losses && workspace && threshold && scales && zeros && R > 0 && C > 0,
                 "spqr_colblock: bad argument");
  LLMC_CHECK_ARG(bit >= 2 && bit <= 8 && s_bit >= 2 && s_bit <= 8 && z_bit >= 2 && z_bit <= 8,
                 "spqr_colblock: bit widths outside 2..8");
  LLMC_CHECK_ARG(!sym, "spqr_colblock: symmetric weights (the reference fails on them, spqr.py:334)");
  LLMC_CHECK_ARG((group == 16 || group == 32 || group == 64 || group == 128) && C % group == 0,
                 "spqr_colblock: group %lld must be 16, 32, 64 or 128 and divide C=%lld",
                 (long long)group, (long long)C);
  LLMC_CHECK_ARG(workspace_bytes >= llmc_gptq_workspace_bytes(R, C), "spqr_colblock: workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int tr_smem = 2 * TT * TT * 4;
  LLMC_ONCE_PER_DEVICE({
    LLMC_CHECK_CUDA(cudaFuncSetAttribute(spqr_inblock_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSpqrSmem));
    LLMC_CHECK_CUDA(cudaFuncSetAttribute(spqr_inblock_lanes_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSpqrLanesSmem));
    LLMC_CHECK_CUDA(cudaFuncSetAttribute(trailing_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tr_smem));
  });
  LLMC_CHECK_CUDA(cudaMemsetAsync(losses, 0, R * sizeof(float), st));
  SpqrArgs a{};
  a.W = W; a.Hinv = Hinv; a.R = R; a.C = C; a.ng = C / group;
  a.cfg.w = spqr_qcfg(bit, sym, round_zp);
  a.cfg.loo = spqr_qcfg(bit, sym, 0);                   // spqr.py:56-58
  a.cfg.sc = spqr_qcfg(s_bit, s_sym, s_round_zp);
  a.cfg.zc = spqr_qcfg(z_bit, z_sym, z_round_zp);
  a.cfg.gs = static_cast<int>(group);
  a.thr = threshold; a.simplified = simplified_outliers;
  a.scales = scales; a.zeros = zeros; a.tmp = tmp; a.mask = mask; a.out_perm = out_perm; a.losses = losses;
  const unsigned row_blocks = static_cast<unsigned>((R + GB - 1) / GB);
  a.Rpad = static_cast<int64_t>(row_blocks) * GB;
  // the 16-lanes-per-row kernel is the default (bit-identical to the thread-per-row kernel and
  // 5-6x faster: tests/test_gpu_spqr.py::test_lane_kernel_bit_identical_to_row_kernel);
  // LLMC_B200_SPQR_KERNEL=row selects the thread-per-row kernel (A/B comparisons in tests only)
  const char* kenv = getenv("LLMC_B200_SPQR_KERNEL");
  const bool row_kernel = kenv != nullptr && kenv[0] == 'r';
  return sweep_schedule(W, Hinv, R, C, group, false, workspace, st,
                        [&](int i1, int count, float* err, float* err_hi, float* err_lo, cudaStream_t cs) -> int {
    a.i1 = i1; a.count = count; a.err = err; a.err_hi = err_hi; a.err_lo = err_lo;
    if (row_kernel) spqr_inblock_kernel<<<row_blocks, GB, kSpqrSmem, cs>>>(a);
    else spqr_inblock_lanes_kernel<<<static_cast<unsigned>(a.Rpad / SR), SR * SL, kSpqrLanesSmem, cs>>>(a);
    LLMC_CHECK_LAUNCH();
    return LLMC_OK;
  });
}
