/*
 * llmc_b200.h — C ABI of libllmc_b200.so: the B200 (sm_100a) kernels behind llmc's
 * weight-quantization hot path (SURVEY.md §8).
 *
 * The reference (ModelTC/llmc) has no FFI: its plug-in boundary is the Python object
 * protocol of `llmc/compression/quantization/{quant,module_utils,gptq,awq,auto_clip}.py`.
 * Each entry point below names the reference function (file:line, relative to the llmc
 * tree) whose arithmetic it replaces; `llmc_b200/*.py` mirrors the reference classes and
 * calls these through ctypes (see INTEGRATION.md for the binding a maintainer would add).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to caller-owned, contiguous memory (16-byte aligned
 *     base); nothing is allocated, nothing is retained after return;
 *   - every call is asynchronous on `stream` (a cudaStream_t / CUstream handle passed as
 *     void*; NULL = legacy default stream) and never synchronises the host;
 *   - return value: 0 on success, a negative LLMC_E* code otherwise
 *     (llmc_b200_error_string() explains it, llmc_b200_last_error() adds detail);
 *   - dtype enums: LLMC_F32 / LLMC_F16 / LLMC_BF16.  "T-faithful" below means: computed
 *     like torch eager does for a tensor of dtype T — every elementwise op is evaluated in
 *     fp32 and rounded once to T (SURVEY.md Appendix A.1), division is IEEE, rounding is
 *     half-to-even.
 */
#ifndef LLMC_B200_H_
#define LLMC_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LLMC_B200_ABI_VERSION 1

/* dtypes */
enum { LLMC_F32 = 0, LLMC_F16 = 1, LLMC_BF16 = 2 };

/* error codes */
enum {
  LLMC_OK = 0,
  LLMC_EINVAL = -1,      /* bad argument (shape / enum / null pointer)            */
  LLMC_EUNSUPPORTED = -2, /* valid request this build has no kernel for            */
  LLMC_ECUDA = -3,       /* a CUDA runtime / driver call failed (see last_error)  */
  LLMC_EALIGN = -4       /* pointer or leading dimension not suitably aligned     */
};

/* output selector of the quantize kernels */
enum {
  LLMC_OUT_NONE = 0,      /* qparams only                                                      */
  LLMC_OUT_QDQ = 1,       /* fake-quant: dequantised values, dtype = out_dtype                 */
  LLMC_OUT_CODES_I8 = 2,  /* integer codes as int8  (8-bit symmetric; quant.py:890-897)        */
  LLMC_OUT_CODES_U8 = 3,  /* integer codes as uint8 (8-bit asymmetric)                         */
  LLMC_OUT_CODES_I32 = 4, /* one code per int32 (every other bit-width; quant.py:895-896)      */
  LLMC_OUT_PACK_VLLM = 5  /* (code + 2^(bit-1)) packed 32/bit per int32 along the input
                             dimension, element i in bits [bit*i, bit*i+bit), zero padded
                             (VllmRealQuantLinear.pack, module_utils.py:836-862)               */
};
/* OR-ed into out_mode of llmc_quant_static: `round_zp: False` (quant.py:702-707, HQQ's real-valued
 * zero-points): q = clamp(round(x / max(s, 1e-9) + z), qmin, qmax) — the zero-point is added BEFORE
 * the rounding. */
#define LLMC_OUT_FLAG_ZP_INSIDE 0x100

int llmc_b200_abi_version(void);
const char* llmc_b200_error_string(int code);
/* thread-local detail of the most recent failure on the calling thread ("" if none) */
const char* llmc_b200_last_error(void);
/* number of CUDA kernels this library has launched in this process (monotonic) */
long long llmc_b200_launch_count(void);

/* ------------------------------------------------------------------------------------
 * K1+K2  llmc_quant_dynamic — replaces IntegerQuantizer.get_tensor_qparams (quant.py:690-697
 *   = reshape_tensor :612-642 -> get_minmax_range :132-143 -> get_qparams :545-559) followed by
 *   quant :699-708 / dequant :710-712, i.e. fake_quant_weight_dynamic :833-869 (out_mode QDQ),
 *   real_quant_weight_dynamic :916-953 (CODES_*), and VllmRealQuantLinear.pack (PACK_VLLM).
 *
 *   w        [rows, cols] dtype `dtype`, row stride `ld` elements (ld >= cols)
 *   group    elements per quantisation group along a row: group_size (per_group),
 *            cols (per_channel / per_token); cols % group == 0
 *   bit      2..8 ; sym != 0: qmin=-2^(bit-1), qmax=2^(bit-1)-1, zero = 0
 *                    sym == 0: qmin=0, qmax=2^bit-1, zero = clamp(qmin - round(min/scale))
 *   qmin,qmax  override the range when qmin < qmax is given with use_range != 0 (int_range)
 *   col_scale  optional [cols] dtype `dtype`: quantise rT(w * col_scale[c]) instead of w — AWQ's
 *            fake_quantize_weight (awq.py:39-46, 147-164) without touching the weights
 *   scales   [rows * cols/group] dtype `dtype`  (index r*ng + j == the reference's [R*ng,1])
 *   zeros    same shape/dtype, written only when sym == 0 (may be NULL when sym != 0)
 *   out      per out_mode (QDQ: [rows, cols] out_dtype, row stride ld_out;
 *            CODES_*: [rows, cols] dense; PACK_VLLM: [rows, ceil(cols*bit/32)] int32 dense)
 *   All arithmetic is `dtype`-faithful.
 * ------------------------------------------------------------------------------------ */
int llmc_quant_dynamic(const void* w, int64_t rows, int64_t cols, int64_t ld, int dtype,
                       int64_t group, int bit, int sym, int use_range, int qmin, int qmax,
                       const void* col_scale, void* scales, void* zeros, int out_mode, void* out,
                       int64_t ld_out, int out_dtype, void* stream);

/* ------------------------------------------------------------------------------------
 * K2  llmc_quant_static — replaces fake_quant_weight_static (quant.py:785-831),
 *   real_quant_weight_static (:871-914) and GPTQ.w_qdq / w_q (gptq.py:411-452) incl. the
 *   act-order gather `W[:, perm] -> qdq -> [:, invperm]`.
 *
 *   element (r, c) uses qparams[r * q_row_stride + g(c)], g(c) = gmap ? gmap[c] : c / group
 *   (q_row_stride = groups per row; 0 with group = cols selects per_tensor qparams).
 *   (for gptq.py:427-450 pass gmap[c] = invperm[c] / group)
 *   w dtype `w_dtype`; scales/zeros dtype `q_dtype`; arithmetic is faithful to
 *   promote(w_dtype, q_dtype) exactly like torch type promotion (round_dtype = -1), or to
 *   round_dtype = w_dtype with fp32 qparams: torch's CPU path for a 0-dim (per_tensor) scale,
 *   which keeps the scalar in fp32 and rounds every result to the tensor dtype
 *   (ATen BinaryOpsKernel.cpp, scalar-operand branch of div/mul).  zeros may be NULL (= 0).
 *   qmin/qmax: the clamp range.  out as in llmc_quant_dynamic (QDQ written as out_dtype).
 * ------------------------------------------------------------------------------------ */
int llmc_quant_static(const void* w, int64_t rows, int64_t cols, int64_t ld, int w_dtype,
                      const void* scales, const void* zeros, int q_dtype, int round_dtype,
                      int64_t q_row_stride, int64_t group, const int32_t* gmap, int bit,
                      int qmin, int qmax, int out_mode, void* out, int64_t ld_out,
                      int out_dtype, void* stream);

/* ------------------------------------------------------------------------------------
 * llmc_pack_vllm_codes — VllmRealQuantLinear.pack (module_utils.py:836-862) on codes that
 *   are already quantised: codes [rows, cols] int8 (code_bytes 1) or int32 (code_bytes 4)
 *   -> out [rows, ceil(cols / (32/bit))] int32.
 * ------------------------------------------------------------------------------------ */
int llmc_pack_vllm_codes(const void* codes, int code_bytes, int64_t rows, int64_t cols,
                         int bit, int32_t* out, void* stream);

/* ------------------------------------------------------------------------------------
 * llmc_minmax_tensor — per_tensor range (quant.py:133-135): min and max over the whole
 *   tensor written to mm[0], mm[1] (dtype `dtype`).  Two-stage device reduction,
 *   `workspace` >= 2 * 1024 floats.
 * ------------------------------------------------------------------------------------ */
int llmc_minmax_tensor(const void* w, int64_t n, int dtype, void* mm, float* workspace,
                       void* stream);

/* ------------------------------------------------------------------------------------
 * Range search / observers (csrc/range.cu)
 *   llmc_mse_range — `calib_algo: mse`, BaseQuantizer.get_mse_range (quant.py:145-203) on the
 *     reshaped tensor [rows = groups, cols = group elements] (any dtype, evaluated in fp32 like
 *     `tensor.float()`): for i in 0..steps-1 (steps = int(maxshrink * mse_grid), p = 1 - i/grid)
 *     the range (p*min, p*max) is tried with get_qparams (:545-559) + quant_dequant (:699-717) and
 *     the one with the smallest sum |q - x|^norm (norm = 2.4) per row is kept; min_out / max_out
 *     [rows] fp32.  The reference's aliasing of the running range (:165, an improvement shrinks
 *     the base of all later levels) is reproduced.
 *   llmc_histc — torch.histc(x.float(), bins, min=lo, max=hi) for the static histogram observer
 *     (get_static_hist_range, quant.py:462-522): hist [bins] fp32 counts.
 * ------------------------------------------------------------------------------------ */
int llmc_mse_range(const void* w, int64_t rows, int64_t cols, int dtype, int sym, int qmin,
                   int qmax, int steps, float grid, float norm, float* min_out, float* max_out,
                   void* stream);
int llmc_histc(const void* x, int64_t n, int dtype, int bins, float lo, float hi, float* hist,
               void* stream);

/* ------------------------------------------------------------------------------------
 * K2-awq  llmc_pack_awq — replaces AutoawqRealQuantLinear.gemm_pack (module_utils.py:1004-1065).
 *   w       [R, C] fp16/bf16/fp32 (the module weight)
 *   scales  [R, ng] dtype `dtype`, zeros [R, ng] int32 (as returned by real_quant_weight_*)
 *   intweight(r,c) = round((w + rT(z*s)) / s) computed in `dtype` exactly like :1022-1029
 *   (scales are first cast to fp16, :1008), NOT clamped;
 *   qweight [C, R/8] int32: nibble i of word (c, r8) = intweight(r8*8 + order[i], c),
 *   order = {0,2,4,6,1,3,5,7}; qzeros [ng, R/8] packed the same way; scales_out [ng, R] fp16.
 *   Requires bit == 4, R % 32 == 0.
 * ------------------------------------------------------------------------------------ */
int llmc_pack_awq(const void* w, int64_t R, int64_t C, int dtype, const void* scales,
                  int s_dtype, const int32_t* zeros, int64_t group, int32_t* qweight,
                  int32_t* qzeros, void* scales_out_f16, void* stream);

/* ------------------------------------------------------------------------------------
 * K3  llmc_syrk_accum — replaces GPTQ.add_batch's Hessian update (gptq.py:283-290):
 *       H <- H * n/(n+b) + (2/(n+b)) * X^T X          (fp32 H, bf16/fp16 X)
 *   x   [T, C] row-major activations (tokens x in_features), dtype bf16 or fp16
 *   H   [C, C] fp32, full symmetric matrix on return (upper computed on tcgen05 tensor
 *       cores with fp32 TMEM accumulation, mirrored into the lower triangle)
 *   n   samples accumulated so far, b = samples in this call (inp.shape[0], :258)
 *   workspace: split-K partials, >= llmc_syrk_workspace_bytes(T, C) bytes
 * ------------------------------------------------------------------------------------ */
int64_t llmc_syrk_workspace_bytes(int64_t T, int64_t C);
int llmc_syrk_accum(const void* x, int64_t T, int64_t C, int dtype, float* H, double n,
                    double b, void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * Multi-GPU helpers (csrc/comm.cu) — the reference all-reduces the FULL Hessian after every
 *   hooked batch (gptq.py:292-295); H is symmetric, so only its upper triangle needs to cross
 *   NVLink, once per distinct input:
 *   llmc_tri_pack    packed[i*C - i(i-1)/2 + (j-i)] = H[i][j], j >= i   (llmc_tri_elems(C) floats)
 *   llmc_tri_unpack  H[i][j] = H[j][i] = packed[...] * scale            (scale = 1/world: the mean)
 * ------------------------------------------------------------------------------------ */
int64_t llmc_tri_elems(int64_t C);
int llmc_tri_pack(const float* H, int64_t C, float* packed, void* stream);
int llmc_tri_unpack(const float* packed, int64_t C, float scale, float* H, void* stream);

/* ------------------------------------------------------------------------------------
 * G4 helpers  llmc_gptq_prepare — replaces process_hessian_and_weights (gptq.py:128-171)
 *   up to (not including) the Cholesky triple: dead-column fix, act-order gather of W and H,
 *   damping.  perm NULL = identity.
 *     Hp[i,j] = H[perm[i], perm[j]] (+ percdamp*mean(diag) on the diagonal; dead -> 1)
 *     Wp[r,j] = dead[perm[j]] ? 0 : float(W[r, perm[j]])
 *   diag_mean_out: device float[1] scratch.
 *   Hp == NULL skips the Hessian part, W == NULL the weight part: linears that share one input
 *   (q/k/v, gate/up) need Hp once and one Wp each — written into row slices of ONE buffer, they
 *   are then swept by a single llmc_gptq_colblock call (rows are independent given Hinv).
 * ------------------------------------------------------------------------------------ */
int llmc_gptq_prepare(const float* H, int64_t C, const int64_t* perm, float percdamp,
                      float* Hp, const void* W, int64_t R, int w_dtype, float* Wp,
                      float* diag_scratch, void* stream);

/* ------------------------------------------------------------------------------------
 * K4  llmc_chol_inv_upper — replaces the Cholesky triple (gptq.py:172-174):
 *       U = cholesky( cholesky_inverse( cholesky(H) ), upper )
 *   computed as U = R^-1 where H = R R^T, R upper triangular (one reverse-ordered
 *   factorisation + one triangular inverse instead of potrf + potri + potrf; DESIGN.md).
 *   A  [C, C] fp32 in: SPD H (full); out: U in the upper triangle, zeros below.
 *   info: device int[1]: 0 if H is positive-definite, else k = the order of the first leading minor
 *         of the index-REVERSED matrix J H J that is not positive (the factorisation runs bottom-up).
 *   C must be a multiple of 8.  The inverse chain runs on a library-owned side stream (one per
 *   device) that forks from and joins back into `stream`: on return everything is ordered on
 *   `stream`, nothing has synchronised with the host.  One host thread per device.
 * ------------------------------------------------------------------------------------ */
int64_t llmc_chol_workspace_bytes(int64_t C);
int llmc_chol_inv_upper(float* A, int64_t C, void* workspace, int64_t workspace_bytes,
                        int* info, void* stream);

/* ------------------------------------------------------------------------------------
 * fp32-accurate tensor-core GEMM building block ("3xTF32", csrc/tf32.cu) used by K4 and K5:
 *   llmc_split_tf32:  hi = tf32(x), lo = tf32(x - hi)            (x, hi, lo: [rows, cols], ld)
 *   llmc_gemm_f32x3:  C[M,N] = (mode 1) or C -= (mode 0)  A * B  with
 *       A(i,k) = a[i*lda + k] (a_mn = 0, K-major)  or  a[k*lda + i] (a_mn = 1, MN-major)
 *       B(j,k) = b[j*ldb + k] (b_mn = 0)           or  b[k*ldb + j] (b_mn = 1)
 *     evaluated as A_hi*B_hi + A_lo*B_hi + A_hi*B_lo on tcgen05 kind::tf32 with fp32 TMEM
 *     accumulation; lower_only != 0 restricts the update to tiles touching col <= row.
 *   These replace the fp32 cuBLAS SGEMMs of gptq.py:244 and the potrf/potri updates of :172-174.
 * ------------------------------------------------------------------------------------ */
int llmc_split_tf32(const float* x, int64_t rows, int64_t cols, int64_t ld, float* hi,
                    float* lo, void* stream);
int llmc_gemm_f32x3(const float* a_hi, const float* a_lo, int a_mn, int64_t lda,
                    const float* b_hi, const float* b_lo, int b_mn, int64_t ldb, float* c,
                    int64_t ldc, int64_t M, int64_t N, int64_t K, int mode, int lower_only,
                    void* stream);

/* ------------------------------------------------------------------------------------
 * K5  llmc_gptq_colblock — replaces GPTQ.weight_transform (gptq.py:198-244) incl.
 *   search_column_qparams (:358-366).
 *   W      [R, C] fp32, permuted weights; overwritten (scratch)
 *   Hinv   [C, C] fp32 upper factor from llmc_chol_inv_upper
 *   tmp    [R, C] fp32 out: compensated, un-rounded weights (gptq.py:237)
 *   losses [R] fp32 out: per-row sum of (w-q)^2/(2 d^2)  (sum over rows == Losses.sum(), :184)
 *   dynamic groups (static_groups == 0): qparams searched on the compensated columns
 *     [idx, idx+group) when idx % group == 0; written to scales/zeros [R, ng] fp32 in
 *     PERMUTED column order (update_model_qparams, :397-409)
 *   static groups: scales/zeros [R, ng] are inputs, dtype q_dtype; column idx uses group
 *     gmap[idx] (= perm[idx] / group, :225-227) or idx / group when gmap is NULL
 *   group == C means per-channel (qparams always static inputs, search_layer_qparams :368-377).
 *   blocksize must be 128 and group % 128 == 0 or 128 % group == 0.
 *   out_perm [C] int64 or NULL: tmp column i is written to column out_perm[i] (pass the act-order
 *     perm to get tmp[:, invperm] of gptq.py:186-188 without a second pass).
 *   The trailing update W[:, i2:] -= Err1 @ Hinv[i1:i2, i2:] (:244) is applied lazily per 512
 *   columns (same terms, fp32 summation order differs); workspace >= llmc_gptq_workspace_bytes.
 * ------------------------------------------------------------------------------------ */
int64_t llmc_gptq_workspace_bytes(int64_t R, int64_t C);
int llmc_gptq_colblock(float* W, const float* Hinv, int64_t R, int64_t C, int64_t group,
                       int bit, int sym, int static_groups, const int32_t* gmap,
                       void* scales, void* zeros, int q_dtype, float* tmp,
                       const int64_t* out_perm, float* losses, void* workspace,
                       int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * K5s llmc_spqr_colblock — SpQR's column sweep (llmc/compression/quantization/spqr.py:172-268,
 *   326-351), the sibling of llmc_gptq_colblock: same Hessian / Cholesky inputs, same block /
 *   super-panel schedule and trailing updates; the in-block step is SpQR's — per group of `group`
 *   columns (16 | 32 | 64 | 128) the leave-one-out outlier search on the current weights
 *   (:174-192, 232-241), group statistics with outliers replaced by the group mean, scale and zero
 *   pushed through the second-level quantizers (s_* / z_*: special.scale / special.zero,
 *   :326-351); per column quantise -> err, unstructured outlier mask err^2 > threshold (:255-259;
 *   outliers keep their weight), rank-1 update.
 *   W [R,C] fp32 permuted weights (consumed), Hinv [C,C] upper factor (llmc_chol_inv_upper).
 *   bit/sym/round_zp: the weight quantizer (symmetric weights are refused by the reference
 *     itself, spqr.py:334; here sym must be 0).
 *   threshold: DEVICE fp32 scalar = relative_threshold * mean(var(W, 0) / diag(Hinv)^2)
 *     (:194-195), +inf disables both outlier mechanisms; simplified_outliers: skip the
 *     leave-one-out search only.
 *   Outputs: scales / zeros [R, C/group] fp32 (second-level quantised, permuted group order),
 *     tmp [R,C] fp32 and mask [R,C] uint8 scattered through out_perm (tmp[:, invperm],
 *     mask[:, invperm], :163-165), losses [R] = sum of err^2 per row.
 *   Workspace as llmc_gptq_colblock (llmc_gptq_workspace_bytes).
 *   The per-row arithmetic is csrc/spqr_row.cuh, which the CPU tests build for the host and
 *   compare bit for bit with the oracle.
 * ------------------------------------------------------------------------------------ */
int llmc_spqr_colblock(float* W, const float* Hinv, int64_t R, int64_t C, int64_t group,
                       int bit, int sym, int round_zp, int s_bit, int s_sym, int s_round_zp,
                       int z_bit, int z_sym, int z_round_zp, const float* threshold,
                       int simplified_outliers, float* scales, float* zeros, float* tmp,
                       uint8_t* mask, const int64_t* out_perm, float* losses, void* workspace,
                       int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * K6  llmc_gemm_bf16 — Y[M,N] = X[M,K] · W[N,K]^T (+ bias[N]); X, W, Y bf16 or fp16,
 *   fp32 accumulation in TMEM (tcgen05.mma kind::f16), TMA-fed.  This is F.linear of
 *   FakeQuantLinear / EffcientFakeQuantLinear.forward (module_utils.py:643, 719).
 * ------------------------------------------------------------------------------------ */
int llmc_gemm_bf16(const void* x, const void* w, const void* bias, void* y, int64_t M,
                   int64_t N, int64_t K, int dtype, void* stream);

/* ------------------------------------------------------------------------------------
 * K6  llmc_gemm_w4a16 — fake-quant forward on PACKED weights:
 *   Y[M,N] = X[M,K] · dequant(Wq)[N,K]^T (+ bias), dequant(Wq)[n,k] =
 *   rT((code - zero) * scale) rounded to `dtype` exactly like the materialised weight of
 *   FakeQuantLinear (module_utils.py:626-643); group-wise dequant runs inside the tcgen05
 *   operand pipeline.
 *   wq      [N, K/8] int32, LLMC_OUT_PACK_VLLM layout of UNSIGNED codes (code+2^(bit-1) for
 *           symmetric, code for asymmetric)
 *   scales  [N, K/group], zeros [N, K/group] (integer valued; for symmetric pass NULL ->
 *           zero = 2^(bit-1)), both of type `qparam_dtype`:
 *             LLMC_F32  (GPTQ dynamic groups): fp32 arithmetic, one rounding to `dtype`;
 *           A NEGATIVE `group` (-group_size) says that scales / zeros are stored TRANSPOSED,
 *           [K/group, N]: the 32 rows of a dequant warp then read one coalesced segment per group
 *           instead of 32 strided sectors (what EffcientFakeQuantLinear hands over).
 *             == dtype  (RTN / AWQ / exported checkpoints): the same value computed with packed
 *                       half2 / bf16x2 arithmetic — (q - z) is exact and the product of two
 *                       `dtype` numbers rounds once either way — at 2.4 instead of 4.2
 *                       instructions per weight.
 * ------------------------------------------------------------------------------------ */
/* ------------------------------------------------------------------------------------
 * K8 / K9  AWQ pieces (csrc/awq.cu)
 *   llmc_absmean_cols  get_act_scale (awq.py:74-85): out[c] = mean_t |x[t,c]|  (fp32 accumulate,
 *                      rounded to dtype); workspace >= min(256, T/64) * C floats
 *   llmc_div_cols      scaling_input (base_blockwise_quantization.py:876-889): out = x / s[c]
 *   llmc_mse           calculate_loss (awq.py:134-145): out[0] = mean(((a - b) in dtype).float()^2);
 *                      workspace >= 1024 floats; result stays on the device (no host sync)
 *   llmc_awq_clip      AutoClipper.auto_clip_layer (auto_clip.py:83-191), clip_version v1, w_only:
 *                      w [R,C], x [ns,C] = the sampled tokens, 10 shrink levels (max_shrink 0.5,
 *                      n_grid 20); best_max / best_min [R, ng] dtype; workspace >= R*ng*10 floats.
 * ------------------------------------------------------------------------------------ */
int llmc_absmean_cols(const void* x, int64_t T, int64_t C, int dtype, void* out,
                      float* workspace, int64_t workspace_floats, void* stream);
int llmc_div_cols(const void* x, const void* s, int64_t T, int64_t C, int dtype, void* out,
                  void* stream);
int llmc_mse(const void* a, const void* b, int64_t n, int dtype, float* out, float* workspace,
             void* stream);
int llmc_awq_clip(const void* w, int64_t R, int64_t C, const void* x, int64_t ns, int dtype,
                  int64_t group, int bit, int sym, int clip_sym, void* best_max, void* best_min,
                  float* workspace, int64_t workspace_floats, void* stream);

/* ------------------------------------------------------------------------------------
 * llmc_fp8_quant — FloatQuantizer with use_qtorch (quant.py:963-1229), e4m3 (e5m2 != 0: e5m2).
 *   PARITY UNPINNED: qtorch.float_quantize is third-party and absent; restated as IEEE RNE onto
 *   the fp8 grid with saturation to the finite max (csrc/fp8.cu header).
 *   dynamic != 0: per (row, group) scale = rT(max(absmax, 1e-5) / finfo.max) written to `scales`
 *                 (dtype), then out_mode 1: QDQ (dtype) | 2: fp8 bytes | 0: scales only.
 *   dynamic == 0: `scales` is an input: [rows * q_row_stride] dtype, or ONE per-tensor scale
 *                 (q_row_stride 0), fp32 when scale_f32 != 0 (torch's CPU scalar-operand path).
 * ------------------------------------------------------------------------------------ */
int llmc_fp8_quant(const void* w, int64_t rows, int64_t cols, int dtype, int64_t group, int e5m2,
                   int dynamic, void* scales, int q_row_stride, int scale_f32, int out_mode,
                   void* out, void* stream);

/* ------------------------------------------------------------------------------------
 * Q10  128 x 128 block FP8 (DeepSeek-V3 / R1 checkpoints), csrc/fp8.cu — PARITY UNPINNED like
 *   llmc_fp8_quant (qtorch):
 *   llmc_fp8_block_quant    weight_cast_to_fp8 (quant.py:32-43) = FloatQuantizer(e4m3, per_block)
 *       .real_quant_weight_dynamic: per [block x block] tile scale = max(absmax, 1e-5) / finfo.max
 *       (fp32, written to scales [ceil(M/block), ceil(N/block)]), q = fp8(x.float() / scale);
 *       out_mode 0 scales only | 1 QDQ (`dtype`) | 2 fp8 bytes.
 *   llmc_fp8_block_dequant  weight_cast_to_bf16 (quant.py:18-29): bf16(fp8.float() * scale_inv).
 *   The forward on these checkpoints is the block-scaled pair below (llmc_fp8_act_quant +
 *   llmc_fp8_gemm); LlmcFp8Linear keeps the dequantise-once branch as its default.
 * ------------------------------------------------------------------------------------ */
int llmc_fp8_block_quant(const void* w, int64_t M, int64_t N, int dtype, int block, int e5m2,
                         float* scales, int out_mode, void* out, void* stream);
int llmc_fp8_block_dequant(const void* w_fp8, int64_t M, int64_t N, int block, int e5m2,
                           const float* scale_inv, void* out_bf16, void* stream);

/* ------------------------------------------------------------------------------------
 * K7-fp8  block-scaled FP8 forward (csrc/gemm_fp8.cu) — the reference's Triton pair
 *   act_quant / fp8_gemm (kernel.py:31-53, 141-242) behind block_wise_fp8_forward_func.
 *   llmc_fp8_act_quant  x [M, K] (dtype fp32 / fp16 / bf16, contiguous), K % 128 == 0:
 *       per 1 x 128 block s = absmax / 448, y = e4m3(x / s), both divisions `div.full.f32` and
 *       the conversion `cvt.rn.satfinite.e4m3x2.f32` as in the reference's compiled kernel.
 *       y [M, K] e4m3 bytes, s [M, K/128] fp32.  An all-zero block gives s = 0 and NaN codes.
 *   llmc_fp8_gemm  C[M, N] = sum_kb (A_kb . B_kb^T) * a_s[m, kb] * b_s[n / 128, kb]
 *       A [M, K] and B [N, K] e4m3 (K-major), a_s [M, K/128], b_s [ceil(N/128), K/128] fp32,
 *       K % 128 == 0 (weight blocks are 128 wide whatever block size the activations used).
 *       fp32 accumulation, per K-block promotion acc = fma(dot * a_s, b_s, acc), one rounding to
 *       out_dtype (fp32 / fp16 / bf16).  bias (fp32 or bf16, may be NULL) requires a bf16
 *       output and is added as `y += bias` after that rounding: bf16(float(y) + float(bias)).
 * ------------------------------------------------------------------------------------ */
int llmc_fp8_act_quant(const void* x, int64_t M, int64_t K, int dtype, void* y, float* s,
                       void* stream);
int llmc_fp8_gemm(const void* a, const float* a_s, const void* b, const float* b_s,
                  const void* bias, int bias_dtype, void* c, int out_dtype, int64_t M, int64_t N,
                  int64_t K, void* stream);

/* ------------------------------------------------------------------------------------
 * Block-forward glue (csrc/block_ops.cu) for F2 block_forward
 * (base_blockwise_quantization.py:367-390): one pass each instead of the HF modules' eager chains.
 *   llmc_rmsnorm   y = weight * (x.float() * rsqrt(mean(x^2) + eps)).to(dtype)     x,y [rows, cols]
 *   llmc_rope      x[B,S,H,D] <- x*cos + rotate_half(x)*sin  (in place; cos/sin [S, D], dtype)
 *   llmc_silu_mul  y = silu(gate) * up                                             n elements
 *   llmc_add       y = a + b
 * ------------------------------------------------------------------------------------ */
int llmc_rmsnorm(const void* x, const void* weight, void* y, int64_t rows, int64_t cols, float eps,
                 int dtype, void* stream);
int llmc_rope(void* x, const void* cosv, const void* sinv, int64_t B, int64_t S, int64_t H,
              int64_t D, int dtype, void* stream);
int llmc_silu_mul(const void* gate, const void* up, void* y, int64_t n, int dtype, void* stream);
int llmc_add(const void* a, const void* b, void* y, int64_t n, int dtype, void* stream);

int llmc_gemm_w4a16(const void* x, const int32_t* wq, const void* scales, const void* zeros,
                    int qparam_dtype, const void* bias, void* y, int64_t M, int64_t N, int64_t K,
                    int64_t group, int dtype, void* stream);
/* llmc_gemm_w8a16 — the same fused forward for INT8 weights (W8A16: rtn_w8a16.yml and the
 *   per-channel W8 configs): wq [N, K/4] int32 = 4 UNSIGNED codes per word along K (code + 128
 *   for symmetric; zeros NULL -> 128), group = K for per-channel.  Dequant in fp32
 *   ((q - z) * s, one rounding to `dtype`), bit-identical to the materialised weight. */
int llmc_gemm_w8a16(const void* x, const int32_t* wq, const void* scales, const void* zeros,
                    int qparam_dtype, const void* bias, void* y, int64_t M, int64_t N, int64_t K,
                    int64_t group, int dtype, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LLMC_B200_H_ */
