"""ORACLE (test infrastructure only) — the block-scaled FP8 forward of the reference
(llmc/compression/quantization/kernel.py:31-53, 141-242): act_quant and fp8_gemm restated in
torch on the CPU, plus an fp64 evaluation of the GEMM with an error bound."""
import torch



def act_quant(x, block_size=128):
    """kernel.py:31-53 restated with IEEE division: per 1 x block_size block of the last dimension,
    s = absmax / 448 and y = e4m3(x / s) (round to nearest even, saturating like
    cvt.rn.satfinite).  Caveat: the reference's compiled kernel divides with `div.full.f32`, an
    approximate division (up to 2 ulp) that a CPU cannot reproduce, so scales may differ from it by
    a couple of ulp and codes by one e4m3 step near rounding ties.  An all-zero block gives
    s = 0 and NaN codes, as there."""
    K = x.shape[-1]
    t = x.float().reshape(-1, K // block_size, block_size)
    s = t.abs().amax(dim=-1) / 448.0
    y = (t / s.unsqueeze(-1)).clamp(-448.0, 448.0).to(torch.float8_e4m3fn)
    return y.reshape(x.shape), s.reshape(*x.shape[:-1], K // block_size)


def _block_dots(a, b, K):
    """fp64 per-128-K-block products [kb, M, N]: exact, since each e4m3 x e4m3 product has at most
    8 significant bits and 128 of them span fewer than 53 bits."""
    A = a.reshape(-1, K).float().double().reshape(-1, K // 128, 128)
    B = b.reshape(-1, K).float().double().reshape(-1, K // 128, 128)
    return torch.einsum('mkc,nkc->kmn', A, B)


def _scales(a_s, b_s, M, N, K):
    sa = a_s.reshape(M, K // 128).double()
    sb = b_s.reshape(-1, K // 128).double()[torch.arange(N) // 128]      # n // 128 (kernel.py:196)
    return sa, sb


def fp8_gemm(a, a_s, b, b_s):
    """kernel.py:141-242 in fp32: per K-block dot (correctly rounded to fp32), then
    acc = fma(fp32(dot * a_s), b_s, acc) in the order of the reference's tcgen05 code.  Returns fp32
    [..., N]; the tensor core's own summation order inside a block may differ in the last bits."""
    K = a.shape[-1]
    M, N = a.numel() // K, b.shape[0]
    dots = _block_dots(a, b, K).float()
    sa, sb = _scales(a_s, b_s, M, N, K)
    acc = torch.zeros(M, N, dtype=torch.float32)
    for kb in range(K // 128):
        t = (dots[kb] * sa[:, kb].float()[:, None])
        acc = (t.double() * sb[:, kb][None, :] + acc.double()).float()
    return acc.reshape(*a.shape[:-1], N)


def fp8_gemm_exact(a, a_s, b, b_s):
    """The same sum in fp64 (exact products, one fp64 rounding per K-block) and a bound on what any
    fp32 per-K-block promotion may deviate from it: (K/128 + 3) ulp-units of fp32 applied to
    sum_kb |a_s b_s| sum_k |a_k b_k|.  Returns (exact fp64 [M, N], bound fp64 [M, N])."""
    K = a.shape[-1]
    M, N = a.numel() // K, b.shape[0]
    dots = _block_dots(a, b, K)
    sa, sb = _scales(a_s, b_s, M, N, K)
    A = a.reshape(-1, K).float().double().abs().reshape(-1, K // 128, 128)
    B = b.reshape(-1, K).float().double().abs().reshape(-1, K // 128, 128)
    mags = torch.einsum('mkc,nkc->kmn', A, B)
    w = sa.t()[:, :, None] * sb.t()[:, None, :]
    exact = (dots * w).sum(0)
    bound = (K // 128 + 3) * 2.0 ** -23 * (mags * w.abs()).sum(0)
    return exact, bound
