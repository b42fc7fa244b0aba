"""Quantised linear modules — mirror of llmc/compression/quantization/module_utils.py.

FakeQuantLinear (:586-678), EffcientFakeQuantLinear (:681-759), OriginFloatLinear (:396-457),
VllmRealQuantLinear (:762-876) + aliases (:879-933), AutoawqRealQuantLinear (:936-1065) +
MlcllmRealQuantLinear (:1068-1084), and the type maps (:1087-1138).  Same `.new(...)`
factories, buffer names and `buf_*` hand-off; the forward GEMM and the packers run in
libllmc_b200.so.

128 x 128 block-FP8 weights (DeepSeek-V3 / R1 checkpoints) have two forwards, which are two of
the reference's semantics rather than two implementations of one result:
  * dequantise-once (the reference on pre-Hopper GPUs, module_utils.py:163-167): the weight is
    cast to bf16 once and every later forward is a bf16 GEMM on it;
  * block-scaled (the reference on Hopper and newer, :40-45, 151-161): block_wise_fp8_forward_func
    quantises the activations per 1 x 128 block and runs the FP8 GEMM with per-block scale
    promotion (csrc/gemm_fp8.cu), keeping the weight in fp8.
OriginFloatLinear, FakeQuantLinear and EffcientFakeQuantLinear built from an fp8 module always take
the block-scaled forward, as the reference does.  LlmcFp8Linear takes it when
USE_FP8GEMM_TRITON_KERNEL is true (the reference's switch, named after its Triton kernels; here it
selects the CUDA pair), initialised from the environment variable LLMC_B200_FP8_GEMM ('1' = on)
and off by default, so LlmcFp8Linear keeps dequantising once unless asked.
"""
import os
from functools import partial

import torch
import torch.nn as nn

from ._lib import call, dtype_enum, ptr, require_cuda, stream_ptr
from .kernel import act_quant, fp8_gemm, fp8_gemm_out
from .prof import TIMER

USE_FP8GEMM_TRITON_KERNEL = os.environ.get('LLMC_B200_FP8_GEMM', '0') == '1'


def block_wise_fp8_forward_func(x, w, w_scale, block_size, bias):
    """module_utils.py:40-45: act_quant -> fp8_gemm -> .to(bf16) -> `y += bias`.  When
    fp8_gemm's default-dtype result reaches bf16 in one rounding (default dtype fp32 or bf16), the
    bf16 cast and the bias add run in the GEMM's epilogue, with the same two roundings."""
    x, scale = act_quant(x, block_size)
    if torch.get_default_dtype() in (torch.float32, torch.bfloat16) and (
            bias is None or bias.dtype in (torch.float32, torch.bfloat16)):
        return fp8_gemm_out(x, scale, w, w_scale, torch.bfloat16, bias)
    y = fp8_gemm(x, scale, w, w_scale).to(torch.bfloat16)
    if bias is not None:
        y += bias
    return y


def _fp8_source(dst, ori_module):
    """The reference's fp8 branch of the wrappers' __init__ (e.g. module_utils.py:413-418)."""
    dst.fp8_forward = dst.weight.dtype == torch.float8_e4m3fn
    if dst.fp8_forward:
        dst.weight_scale_inv = ori_module.weight_scale_inv
        dst.block_size = ori_module.block_size


def linear_forward(x, weight, bias=None):
    """F.linear on the tcgen05 GEMM (csrc/gemm.cu) — y = x @ weight.T (+ bias)."""
    require_cuda(x, weight)
    if x.dtype != weight.dtype:
        raise TypeError(f'activation dtype {x.dtype} != weight dtype {weight.dtype}')
    K = x.shape[-1]
    N = weight.shape[0]
    x2 = x.reshape(-1, K)
    if not x2.is_contiguous():
        x2 = x2.contiguous()
    w = weight if weight.is_contiguous() else weight.contiguous()
    y = torch.empty((x2.shape[0], N), dtype=x.dtype, device=x.device)
    b = None
    if bias is not None:
        b = bias.to(x.dtype).contiguous()
    M = x2.shape[0]
    with TIMER.span('gemm', flops=2.0 * M * N * K, nbytes=2.0 * (M * K + N * K + M * N)):
        call('llmc_gemm_bf16', ptr(x2), ptr(w), ptr(b), ptr(y), M, N, K, dtype_enum(x.dtype),
             stream_ptr(x.device))
    return y.reshape(*x.shape[:-1], N)


def linear_forward_w4(x, wq, scales, zeros, group, bias=None, bits=4, qparams_t=False):
    """Fake-quant forward on PACKED int4 weights (csrc/gemm_w4.cu): y = x @ dequant(wq).T + bias,
    bit-identical to linear_forward(x, rT((code - zero) * scale)) — the materialised weight of
    FakeQuantLinear (module_utils.py:626-643) — while reading 4.25 instead of 16 bits per weight.

    wq [N, K/8] int32 (unsigned codes, LLMC_OUT_PACK_VLLM layout), scales [N, K/group] in x.dtype
    or fp32, zeros likewise or None (None => 8, the symmetric +2^(bit-1) storage offset)."""
    require_cuda(x, wq, scales)
    K = x.shape[-1]
    N = wq.shape[0]
    assert bits in (4, 8)
    assert wq.dtype == torch.int32 and wq.shape[1] * (32 // bits) == K, (wq.shape, K)
    x2 = x.reshape(-1, K)
    x2 = x2 if x2.is_contiguous() else x2.contiguous()
    # qparams already in the activation dtype (RTN / AWQ / exported checkpoints) take the packed
    # half2 / bf16x2 dequant path; fp32 qparams (GPTQ dynamic groups) the fp32 one — same values
    native = scales.dtype == x.dtype and (zeros is None or zeros.dtype == x.dtype)
    qdt = x.dtype if native else torch.float32
    # qparams_t: scales / zeros already stored [K/group, N] (coalesced loads in the kernel)
    shape = (-1, N) if qparams_t else (N, -1)
    s = scales.reshape(shape).to(qdt).contiguous()
    z = zeros.reshape(shape).to(qdt).contiguous() if zeros is not None else None
    b = bias.to(x.dtype).contiguous() if bias is not None else None
    y = torch.empty((x2.shape[0], N), dtype=x.dtype, device=x.device)
    M = x2.shape[0]
    with TIMER.span(f'gemm_w{bits}a16', flops=2.0 * M * N * K,
                    nbytes=2.0 * M * K + bits / 8.0 * N * K + 8.0 * N * K / group + 2.0 * M * N):
        call(f'llmc_gemm_w{bits}a16', ptr(x2), ptr(wq.contiguous()), ptr(s), ptr(z), dtype_enum(qdt), ptr(b), ptr(y), M, N, K,
             int(-group if qparams_t else group), dtype_enum(x.dtype), stream_ptr(x.device))
    return y.reshape(*x.shape[:-1], N)


def _copy_bufs(dst, ori_module):
    for name, buf in ori_module.named_buffers():
        if name.startswith('buf_'):
            dst.register_buffer(name, buf.data)
    for name, buf in ori_module.named_parameters():
        if name.startswith('buf_'):
            dst.register_buffer(name, buf.data)


def _func_name(any_callable):
    if isinstance(any_callable, partial):
        return any_callable.func.__name__
    return any_callable.__name__


class OriginFloatLinear(nn.Module):
    """module_utils.py:396-457 — plain linear on the (transformed) float weight."""

    def __init__(self, weight, bias, ori_module):
        super().__init__()
        self.register_buffer('weight', weight)
        if bias is not None:
            self.register_buffer('bias', bias)
        else:
            self.bias = None
        _copy_bufs(self, ori_module)
        if getattr(self, 'buf_rotate', False):
            raise NotImplementedError('online rotation (QuaRot) is out of scope (SURVEY §2 #12)')
        self.buf_rotate = False
        _fp8_source(self, ori_module)

    @torch.no_grad()
    def forward(self, x):
        if self.fp8_forward:
            return block_wise_fp8_forward_func(x, self.weight, self.weight_scale_inv, self.block_size,
                                               self.bias)
        return linear_forward(x, self.weight, self.bias)

    @classmethod
    @torch.no_grad()
    def new(cls, module):
        bias = module.bias.data if getattr(module, 'bias', None) is not None else None
        new_module = cls(module.weight.data, bias, module)
        new_module.in_features = module.in_features
        new_module.out_features = module.out_features
        return new_module

    def __repr__(self):
        return (f'OriginFloatLinear(in_features={self.in_features},'
                f'out_features={self.out_features}, bias={self.bias is not None},'
                f'online_rotate={self.buf_rotate},'
                f'fp8_forward={self.fp8_forward})')


class LlmcFp8Linear(nn.Module):
    """module_utils.py:130-191 — holder of a 128x128 block-FP8 checkpoint weight (`weight` fp8 +
    `weight_scale_inv` fp32 [ceil(out/bs), ceil(in/bs)]).  Forward: with USE_FP8GEMM_TRITON_KERNEL
    the block-scaled FP8 GEMM on the fp8 weight (:153-161); otherwise the reference's other branch
    (:162-167), dequantise ONCE to bf16 (llmc_fp8_block_dequant) and run the tcgen05 GEMM."""

    def __init__(self, in_features, out_features, bias, block_size):
        super().__init__()
        self.block_size, self.in_features, self.out_features = block_size, in_features, out_features
        if bias is not None:
            self.bias = nn.Parameter(torch.empty(out_features))
        else:
            self.register_parameter('bias', None)
        self.weight = nn.Parameter(torch.empty(out_features, in_features, dtype=torch.float8_e4m3fn),
                                   requires_grad=False)
        so, si = -(-out_features // block_size), -(-in_features // block_size)
        self.weight_scale_inv = nn.Parameter(torch.empty(so, si, dtype=torch.float32), requires_grad=False)

    @torch.no_grad()
    def forward(self, x):
        if self.weight.data.dtype == torch.float8_e4m3fn:
            if USE_FP8GEMM_TRITON_KERNEL:
                return block_wise_fp8_forward_func(x, self.weight, self.weight_scale_inv,
                                                   self.block_size, self.bias)
            from .quant_float import weight_cast_to_bf16
            self.weight.data = weight_cast_to_bf16(self.weight.data, self.weight_scale_inv.data,
                                                   self.block_size)
        return linear_forward(x, self.weight.data, self.bias)

    @classmethod
    @torch.no_grad()
    def new(cls, module, block_size):
        return cls(module.in_features, module.out_features, module.bias, block_size)

    def __repr__(self):
        return (f'LlmcFp8Linear(in_features={self.in_features}, out_features={self.out_features}, '
                f'bias={self.bias is not None}, weight_shape={self.weight.shape}, '
                f'weight_dtype={self.weight.dtype}, block_size={self.block_size}, '
                f'use_fp8gemm_triton_kernel={USE_FP8GEMM_TRITON_KERNEL})')


class FakeQuantLinear(nn.Module):
    """module_utils.py:586-678 — calibration-time wrapper; w_qdq is evaluated lazily on the
    first forward and cached in the non-persistent `tmp_weight` buffer (:626-629)."""

    def __init__(self, weight, bias, ori_module, w_qdq, a_qdq):
        super().__init__()
        self.register_buffer('weight', weight)
        if bias is not None:
            self.register_buffer('bias', bias)
        else:
            self.bias = None
        self.a_qdq = a_qdq
        self.w_qdq = w_qdq
        _copy_bufs(self, ori_module)
        if getattr(self, 'buf_rotate', False):
            raise NotImplementedError('online rotation (QuaRot) is out of scope (SURVEY §2 #12)')
        self.buf_rotate = False
        _fp8_source(self, ori_module)
        self.dynamic_quant_weight = False
        self.dynamic_quant_tmp_weight = False

    def forward(self, x):
        if self.a_qdq is not None:
            x = self.a_qdq(x, self)
        if not hasattr(self, 'tmp_weight'):
            self.register_buffer('tmp_weight', self.w_qdq(self), persistent=False)
            self.tmp_bias = self.bias
        elif self.dynamic_quant_weight:
            self.tmp_weight = self.w_qdq(self)
            self.tmp_bias = self.bias
        elif self.dynamic_quant_tmp_weight:
            self.tmp_weight = self.w_qdq(self)
        if self.fp8_forward:
            # the reference evaluates (and caches) w_qdq above, then runs on the fp8 weight (:638-641)
            return block_wise_fp8_forward_func(x, self.weight, self.weight_scale_inv, self.block_size,
                                               self.bias)
        return linear_forward(x, self.tmp_weight, self.tmp_bias)

    @classmethod
    @torch.no_grad()
    def new(cls, module, w_qdq, a_qdq):
        bias = module.bias.data if getattr(module, 'bias', None) is not None else None
        new_module = cls(module.weight.data, bias, ori_module=module, w_qdq=w_qdq, a_qdq=a_qdq)
        new_module.in_features = module.in_features
        new_module.out_features = module.out_features
        new_module.w_qdq_name = _func_name(w_qdq)
        new_module.a_qdq_name = _func_name(a_qdq) if a_qdq is not None else 'None'
        return new_module

    def __repr__(self):
        return (f'FakeQuantLinear(in_features={self.in_features},'
                f'out_features={self.out_features}, bias={self.bias is not None},'
                f'weight_quant={self.w_qdq_name},'
                f'act_quant={self.a_qdq_name},'
                f'online_rotate={self.buf_rotate})')


def pack_unsigned_codes(codes, bits, signed):
    """[N, K] integer codes -> [N, K*bits/32] int32 of UNSIGNED codes, little-end first along K
    (the weight layout of llmc_gemm_w4a16 / llmc_gemm_w8a16).  llmc_pack_vllm_codes adds the
    +2^(bits-1) storage offset of module_utils.py:842-844, so asymmetric (already unsigned) codes are
    shifted down first."""
    require_cuda(codes)
    c = codes.to(torch.int32)
    if not signed:
        c = c - (1 << (bits - 1))
    c = c.contiguous()
    rows, cols = c.shape
    pf = 32 // bits
    out = torch.empty((rows, cols // pf), dtype=torch.int32, device=c.device)
    call('llmc_pack_vllm_codes', ptr(c), 4, rows, cols, int(bits), ptr(out), stream_ptr(c.device))
    return out


class EffcientFakeQuantLinear(nn.Module):
    """module_utils.py:681-759 — eval-time wrapper: w_qdq applied once in `new`.

    B200 extension (K6): when the weight quantizer is a plain INT4 / INT8 group or channel
    quantizer, `new` keeps the PACKED codes + group qparams instead of the dequantised weight and
    the forward runs the fused dequant -> tcgen05 GEMM (csrc/gemm_w4.cu) — bit-identical to F.linear
    on the materialised weight (tests/test_gpu_gemm_w4.py), at 4.25 / 8.25 instead of 16 bits per
    weight in HBM.  `.weight` then dequantises on demand.  LLMC_B200_FUSED_DEQUANT=0 disables it."""

    def __init__(self, weight, bias, ori_module, a_qdq, packed=None):
        super().__init__()
        if packed is None:
            self.register_buffer('weight', weight)
        else:
            self.register_buffer('qweight', packed['qweight'])
            self.register_buffer('qscales', packed['scales'])
            if packed['zeros'] is not None:
                self.register_buffer('qzeros', packed['zeros'])
            else:
                self.qzeros = None
            self.q_bits, self.q_group, self.q_dtype = packed['bits'], packed['group'], packed['dtype']
            # [K/group, N] copies for the GEMM (coalesced qparam loads); tiny next to the codes
            self.register_buffer('qscales_t', packed['scales'].t().contiguous(), persistent=False)
            self.register_buffer('qzeros_t', packed['zeros'].t().contiguous()
                                 if packed['zeros'] is not None else None, persistent=False)
        self.packed = packed is not None
        if bias is not None:
            self.register_buffer('bias', bias)
        else:
            self.bias = None
        self.a_qdq = a_qdq
        _copy_bufs(self, ori_module)
        if getattr(self, 'buf_rotate', False):
            raise NotImplementedError('online rotation (QuaRot) is out of scope (SURVEY §2 #12)')
        self.buf_rotate = False
        if packed is None:
            _fp8_source(self, ori_module)
        else:
            self.fp8_forward = False

    def __getattr__(self, name):
        if name == 'weight' and self.__dict__.get('packed', False):
            return self.dequantized_weight()
        return super().__getattr__(name)

    @torch.no_grad()
    def dequantized_weight(self):
        """rT((code - zero) * scale): the tensor the reference holds in `.weight` (elementwise, exact)."""
        bits, pf = self.q_bits, 32 // self.q_bits
        sh = torch.arange(pf, device=self.qweight.device, dtype=torch.int32) * bits
        codes = ((self.qweight.unsqueeze(-1) >> sh) & ((1 << bits) - 1)).reshape(self.qweight.shape[0], -1)
        N, K = codes.shape
        z = self.qzeros if self.qzeros is not None else float(1 << (bits - 1))
        s = self.qscales
        c = codes.reshape(N, -1, self.q_group).to(s.dtype)
        zz = z.reshape(N, -1, 1) if torch.is_tensor(z) else z
        return ((c - zz) * s.reshape(N, -1, 1)).reshape(N, K).to(self.q_dtype)

    @torch.no_grad()
    def forward(self, x):
        if self.a_qdq is not None:
            x = self.a_qdq(x, self)
        if self.fp8_forward:
            return block_wise_fp8_forward_func(x, self.weight, self.weight_scale_inv, self.block_size,
                                               self.bias)
        if self.packed:
            return linear_forward_w4(x, self.qweight, self.qscales_t, self.qzeros_t, self.q_group, self.bias,
                                     bits=self.q_bits, qparams_t=True)
        return linear_forward(x, self.weight, self.bias)

    @classmethod
    @torch.no_grad()
    def new(cls, module, w_qdq, a_qdq, debug_print={}):
        packer = getattr(w_qdq, 'packed', None)
        packed = None
        fp8 = module.weight.dtype == torch.float8_e4m3fn     # fp8 checkpoints: never packed
        if packer is not None and not fp8 and os.environ.get('LLMC_B200_FUSED_DEQUANT', '1') != '0':
            packed = packer(module)
        weight = w_qdq(module) if packed is None else None
        bias = module.bias.data if getattr(module, 'bias', None) is not None else None
        new_module = cls(weight, bias, ori_module=module, a_qdq=a_qdq, packed=packed)
        new_module.in_features = module.in_features
        new_module.out_features = module.out_features
        new_module.w_qdq_name = _func_name(w_qdq)
        new_module.a_qdq_name = _func_name(a_qdq) if a_qdq is not None else 'None'
        new_module.debug_print = debug_print
        return new_module

    def __repr__(self):
        return (f'EffcientFakeQuantLinear(in_features={self.in_features},'
                f'out_features={self.out_features}, bias={self.bias is not None},'
                f'weight_quant={self.w_qdq_name},'
                f'act_quant={self.a_qdq_name},'
                f'online_rotate={self.buf_rotate},'
                f'fp8_forward={self.fp8_forward})')


def _cfg_get(cfg, key, default=None):
    if isinstance(cfg, dict):
        return cfg.get(key, default)
    return getattr(cfg, key, default)


class VllmRealQuantLinear(nn.Module):
    """module_utils.py:762-876 — compressed-tensors layout: `weight_packed` / `weight`,
    `weight_scale` (fp16 when packed) or `weight_scale_inv`, `input_scale`."""

    def __init__(self, weight, bias, scales, input_scale, need_pack, scales_name):
        super().__init__()
        self.register_buffer('weight_packed' if need_pack else 'weight', weight)
        if bias is not None:
            self.register_buffer('bias', bias)
        else:
            self.bias = None
        self.register_buffer(scales_name, scales)
        self.register_buffer('input_scale', input_scale)

    @torch.no_grad()
    def forward(self, x):
        raise NotImplementedError

    @classmethod
    @torch.no_grad()
    def new(cls, module, w_q, quant_config):
        weight, scales = cls.quant_pack(module, w_q, quant_config)
        input_scale = getattr(module, 'buf_act_scales_0', None)
        act = _cfg_get(quant_config, 'act')
        if (act is not None and _cfg_get(act, 'static', False)
                and _cfg_get(quant_config, 'quant_type', 'int-quant') == 'int-quant'):
            input_scale = input_scale.unsqueeze(0)
        bias = module.bias.data if module.bias is not None else None
        wcfg = _cfg_get(quant_config, 'weight')
        need_pack = _cfg_get(wcfg, 'need_pack', False)
        scales_name = ('weight_scale_inv' if _cfg_get(wcfg, 'granularity') == 'per_block'
                       else 'weight_scale')
        new_module = cls(weight, bias, scales, input_scale, need_pack, scales_name)
        new_module.in_features = module.in_features
        new_module.out_features = module.out_features
        new_module.weight_shape, new_module.weight_dtype = weight.shape, weight.dtype
        new_module.scales_shape, new_module.scales_dtype = scales.shape, scales.dtype
        new_module.zeros_shape = new_module.zeros_dtype = None
        return new_module

    @classmethod
    @torch.no_grad()
    def quant_pack(cls, module, w_q, quant_config):
        weight, scales, zeros = w_q(module)
        if _cfg_get(_cfg_get(quant_config, 'weight'), 'need_pack', False):
            weight, scales = cls.pack(weight, scales, quant_config)
        return weight, scales

    @classmethod
    @torch.no_grad()
    def pack(cls, weight, scales, quant_config):
        """module_utils.py:836-862 on the device (the reference goes GPU->numpy->GPU)."""
        require_cuda(weight)
        num_bits = _cfg_get(_cfg_get(quant_config, 'weight'), 'bit')
        codes = weight.contiguous()
        if codes.dtype == torch.uint8:
            codes = codes.view(torch.int8)
        assert codes.dtype in (torch.int8, torch.int32), codes.dtype
        rows, cols = codes.shape
        pf = 32 // num_bits
        out = torch.empty((rows, (cols + pf - 1) // pf), dtype=torch.int32, device=codes.device)
        call('llmc_pack_vllm_codes', ptr(codes), codes.element_size(), rows, cols, int(num_bits),
             ptr(out), stream_ptr(codes.device))
        return out, scales.to(torch.float16)

    def __repr__(self):
        return ('VllmRealQuantLinear(' + f'in_features={self.in_features}, '
                + f'out_features={self.out_features}, ' + f'bias={self.bias is not None}, '
                + f'weight_shape={self.weight_shape}, ' + f'weight_dtype={self.weight_dtype}, '
                + f'scales_shape={self.scales_shape}, ' + f'scales_dtype={self.scales_dtype}, '
                + f'zeros_shape={self.zeros_shape}, ' + f'zeros_dtype={self.zeros_dtype})')


class LightllmRealQuantLinear(VllmRealQuantLinear):
    pass


class SglRealQuantLinear(VllmRealQuantLinear):
    pass


class Lightx2vRealQuantLinear(VllmRealQuantLinear):
    pass


class AutoawqRealQuantLinear(nn.Module):
    """module_utils.py:936-1065 — AutoAWQ GEMM layout: qweight [C, R/8], qzeros [ng, R/8],
    scales [ng, R] fp16."""

    def __init__(self, weight, bias, scales, zeros):
        super().__init__()
        self.register_buffer('qweight', weight)
        if bias is not None:
            self.register_buffer('bias', bias)
        else:
            self.bias = None
        self.register_buffer('scales', scales)
        if zeros is not None:
            self.register_buffer('qzeros', zeros)
        else:
            self.qzeros = None

    @torch.no_grad()
    def forward(self, x):
        raise NotImplementedError

    @classmethod
    @torch.no_grad()
    def new(cls, module, w_q, quant_config):
        weight, scales, zeros = cls.quant_pack(module, w_q, quant_config)
        bias = module.bias.data if module.bias is not None else None
        new_module = cls(weight, bias, scales, zeros)
        new_module.in_features = module.in_features
        new_module.out_features = module.out_features
        new_module.weight_shape, new_module.weight_dtype = weight.shape, weight.dtype
        new_module.scales_shape, new_module.scales_dtype = scales.shape, scales.dtype
        new_module.zeros_shape = zeros.shape if zeros is not None else None
        new_module.zeros_dtype = zeros.dtype if zeros is not None else None
        return new_module

    @classmethod
    @torch.no_grad()
    def quant_pack(cls, module, w_q, quant_config):
        _, scales, zeros = w_q(module)
        pack_version = _cfg_get(_cfg_get(quant_config, 'weight'), 'pack_version')
        if pack_version != 'gemm_pack':
            raise NotImplementedError(f'Not support {pack_version}.')
        return cls.gemm_pack(module, module.weight.data, scales, zeros, quant_config)

    @classmethod
    @torch.no_grad()
    def gemm_pack(cls, module, weight, scales, zeros, quant_config):
        """module_utils.py:1004-1065 as one tiled kernel (csrc/pack_awq.cu)."""
        assert scales is not None and zeros is not None
        wcfg = _cfg_get(quant_config, 'weight')
        bit, group_size = _cfg_get(wcfg, 'bit'), _cfg_get(wcfg, 'group_size')
        if bit != 4:
            raise NotImplementedError('Only 4-bit are supported for now.')
        require_cuda(weight, scales, zeros)
        w = weight.contiguous()
        R, C = w.shape
        ng = C // group_size
        s = scales.contiguous()
        z = zeros.to(torch.int32).contiguous()
        qweight = torch.empty((C, R // 32 * bit), dtype=torch.int32, device=w.device)
        qzeros = torch.empty((ng, R // 32 * bit), dtype=torch.int32, device=w.device)
        scales_out = torch.empty((ng, R), dtype=torch.float16, device=w.device)
        call('llmc_pack_awq', ptr(w), R, C, dtype_enum(w.dtype), ptr(s), dtype_enum(s.dtype),
             ptr(z), int(group_size), ptr(qweight), ptr(qzeros), ptr(scales_out),
             stream_ptr(w.device))
        return qweight, scales_out, qzeros

    def __repr__(self):
        return (f'{type(self).__name__}(' + f'in_features={self.in_features}, '
                + f'out_features={self.out_features}, ' + f'bias={self.bias is not None}, '
                + f'weight_shape={self.weight_shape}, ' + f'weight_dtype={self.weight_dtype}, '
                + f'scales_shape={self.scales_shape}, ' + f'scales_dtype={self.scales_dtype}, '
                + f'zeros_shape={self.zeros_shape}, ' + f'zeros_dtype={self.zeros_dtype})')


class MlcllmRealQuantLinear(AutoawqRealQuantLinear):
    pass


_TRANSFORMERS_LINEAR_TYPES_ = [nn.Linear]

_LLMC_LINEAR_TYPES_ = [
    LlmcFp8Linear, OriginFloatLinear, FakeQuantLinear, EffcientFakeQuantLinear, VllmRealQuantLinear,
    SglRealQuantLinear, AutoawqRealQuantLinear, MlcllmRealQuantLinear, LightllmRealQuantLinear,
    Lightx2vRealQuantLinear,
]

_REALQUANT_LINEAR_MAP_ = {
    'vllm_quant': VllmRealQuantLinear,
    'lightllm_quant': LightllmRealQuantLinear,
    'sgl_quant': SglRealQuantLinear,
    'autoawq_quant': AutoawqRealQuantLinear,
    'mlcllm_quant': MlcllmRealQuantLinear,
    'lightx2v_quant': Lightx2vRealQuantLinear,
}
