"""Block-scaled FP8 kernels — mirror of llmc/compression/quantization/kernel.py:31-53, 217-242.

`act_quant` and `fp8_gemm` keep the reference's shapes, dtypes and asserts; both run in
libllmc_b200.so (csrc/gemm_fp8.cu) on tcgen05 instead of Triton.
"""
import torch

from ._lib import F32, call, dtype_enum, ptr, require_cuda, stream_ptr
from .prof import TIMER


def act_quant(x, block_size=128):
    """kernel.py:31-53: per 1 x block_size block of the last dimension, s = absmax / 448 and
    y = e4m3(x / s).  Returns (y float8_e4m3fn shaped like x, s fp32 [..., K / block_size])."""
    assert x.is_contiguous(), 'Input tensor must be contiguous'
    assert (
        x.size(-1) % block_size == 0
    ), f'Last dimension size must be divisible by block_size (block_size={block_size})'
    if block_size != 128:
        # fp8_gemm indexes the weight scales as n // 128 (kernel.py:196), so the pair only
        # composes for 128-wide blocks.
        raise NotImplementedError(f'act_quant: block_size={block_size}; only 128 is supported')
    require_cuda(x)
    y = torch.empty_like(x, dtype=torch.float8_e4m3fn)
    s = x.new_empty(*x.size()[:-1], x.size(-1) // block_size, dtype=torch.float32)
    K = x.size(-1)
    M = x.numel() // K
    with TIMER.span('fp8_act_quant', flops=0.0,
                    nbytes=float(M * K * (x.element_size() + 1) + M * (K // 128) * 4)):
        call('llmc_fp8_act_quant', ptr(x), M, K, dtype_enum(x.dtype), ptr(y), ptr(s),
             stream_ptr(x.device))
    return y, s


def fp8_gemm_out(a, a_s, b, b_s, out_dtype, bias=None):
    """C = sum_kb (A_kb . B_kb^T) * a_s[m, kb] * b_s[n // 128, kb], rounded once to out_dtype.
    bias (fp32 or bf16) needs out_dtype bf16 and is added after that rounding, as `y += bias`."""
    assert a.is_contiguous() and b.is_contiguous(), 'Input tensors must be contiguous'
    assert (
        a_s.is_contiguous() and b_s.is_contiguous()
    ), 'Scaling factor tensors must be contiguous'
    require_cuda(a, a_s, b, b_s, bias)
    K = a.size(-1)
    M = a.numel() // K
    N = b.size(0)
    if a.dtype != torch.float8_e4m3fn or b.dtype != torch.float8_e4m3fn:
        raise TypeError(f'fp8_gemm: operands must be float8_e4m3fn (got {a.dtype}, {b.dtype})')
    if a_s.dtype != torch.float32 or b_s.dtype != torch.float32:
        raise TypeError('fp8_gemm: scales must be float32')
    if b.size(-1) != K or a_s.numel() != M * (K // 128) or b_s.numel() < -(-N // 128) * (K // 128):
        raise ValueError(f'fp8_gemm: shape mismatch a {tuple(a.shape)} a_s {tuple(a_s.shape)} '
                         f'b {tuple(b.shape)} b_s {tuple(b_s.shape)}')
    c = a.new_empty(*a.size()[:-1], N, dtype=out_dtype)
    bias_dt = F32
    if bias is not None:
        bias = bias.contiguous()
        bias_dt = dtype_enum(bias.dtype)
    with TIMER.span('fp8_gemm', flops=2.0 * M * N * K,
                    nbytes=float(M * K + N * K + c.element_size() * M * N + 4 * (M + N // 128 + 1) * (K // 128))):
        call('llmc_fp8_gemm', ptr(a), ptr(a_s), ptr(b), ptr(b_s), ptr(bias), bias_dt, ptr(c),
             dtype_enum(out_dtype), M, N, K, stream_ptr(a.device))
    return c


def fp8_gemm(a, a_s, b, b_s):
    """kernel.py:217-242: returns torch.get_default_dtype()."""
    return fp8_gemm_out(a, a_s, b, b_s, torch.get_default_dtype())

