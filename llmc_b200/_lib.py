"""ctypes binding of libllmc_b200.so (C ABI declared in include/llmc_b200.h).

There is deliberately NO CPU / eager fallback: if the CUDA library is missing or a kernel
reports an error the call raises.  (The oracle under oracle/ is test infrastructure and is
never imported from here.)
"""
import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libllmc_b200.so')

F32, F16, BF16 = 0, 1, 2
OUT_NONE, OUT_QDQ, OUT_CODES_I8, OUT_CODES_U8, OUT_CODES_I32, OUT_PACK_VLLM = range(6)

_DTYPE = {torch.float32: F32, torch.float16: F16, torch.bfloat16: BF16}

c_i64, c_int, c_vp, c_dbl, c_f32 = (ctypes.c_int64, ctypes.c_int, ctypes.c_void_p,
                                    ctypes.c_double, ctypes.c_float)

# name -> (restype, argtypes); mirrors include/llmc_b200.h one to one.
SIGNATURES = {
    'llmc_b200_abi_version': (c_int, []),
    'llmc_b200_error_string': (ctypes.c_char_p, [c_int]),
    'llmc_b200_last_error': (ctypes.c_char_p, []),
    'llmc_b200_launch_count': (ctypes.c_longlong, []),
    'llmc_quant_dynamic': (c_int, [c_vp, c_i64, c_i64, c_i64, c_int, c_i64, c_int, c_int, c_int,
                                   c_int, c_int, c_vp, c_vp, c_vp, c_int, c_vp, c_i64, c_int, c_vp]),
    'llmc_absmean_cols': (c_int, [c_vp, c_i64, c_i64, c_int, c_vp, c_vp, c_i64, c_vp]),
    'llmc_div_cols': (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_vp, c_vp]),
    'llmc_mse': (c_int, [c_vp, c_vp, c_i64, c_int, c_vp, c_vp, c_vp]),
    'llmc_awq_clip': (c_int, [c_vp, c_i64, c_i64, c_vp, c_i64, c_int, c_i64, c_int, c_int, c_int,
                              c_vp, c_vp, c_vp, c_i64, c_vp]),
    'llmc_quant_static': (c_int, [c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_vp, c_int, c_int, c_i64,
                                  c_i64, c_vp, c_int, c_int, c_int, c_int, c_vp, c_i64, c_int,
                                  c_vp]),
    'llmc_pack_vllm_codes': (c_int, [c_vp, c_int, c_i64, c_i64, c_int, c_vp, c_vp]),
    'llmc_minmax_tensor': (c_int, [c_vp, c_i64, c_int, c_vp, c_vp, c_vp]),
    'llmc_mse_range': (c_int, [c_vp, c_i64, c_i64, c_int, c_int, c_int, c_int, c_int, c_f32, c_f32, c_vp,
                               c_vp, c_vp]),
    'llmc_histc': (c_int, [c_vp, c_i64, c_int, c_int, c_f32, c_f32, c_vp, c_vp]),
    'llmc_pack_awq': (c_int, [c_vp, c_i64, c_i64, c_int, c_vp, c_int, c_vp, c_i64, c_vp, c_vp,
                              c_vp, c_vp]),
    'llmc_tri_elems': (c_i64, [c_i64]),
    'llmc_tri_pack': (c_int, [c_vp, c_i64, c_vp, c_vp]),
    'llmc_tri_unpack': (c_int, [c_vp, c_i64, c_f32, c_vp, c_vp]),
    'llmc_syrk_workspace_bytes': (c_i64, [c_i64, c_i64]),
    'llmc_syrk_accum': (c_int, [c_vp, c_i64, c_i64, c_int, c_vp, c_dbl, c_dbl, c_vp, c_i64,
                                c_vp]),
    'llmc_gptq_prepare': (c_int, [c_vp, c_i64, c_vp, c_f32, c_vp, c_vp, c_i64, c_int, c_vp,
                                  c_vp, c_vp]),
    'llmc_chol_workspace_bytes': (c_i64, [c_i64]),
    'llmc_chol_inv_upper': (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp]),
    'llmc_split_tf32': (c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp]),
    'llmc_gemm_f32x3': (c_int, [c_vp, c_vp, c_int, c_i64, c_vp, c_vp, c_int, c_i64, c_vp, c_i64,
                                c_i64, c_i64, c_i64, c_int, c_int, c_vp]),
    'llmc_gptq_workspace_bytes': (c_i64, [c_i64, c_i64]),
    'llmc_gptq_colblock': (c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_int, c_int, c_int, c_vp,
                                   c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    'llmc_spqr_colblock': (c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_int, c_int, c_int, c_int, c_int,
                                   c_int, c_int, c_int, c_int, c_vp, c_int, c_vp, c_vp, c_vp, c_vp,
                                   c_vp, c_vp, c_vp, c_i64, c_vp]),
    'llmc_gemm_bf16': (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_int, c_vp]),
    'llmc_rmsnorm': (c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, c_f32, c_int, c_vp]),
    'llmc_rope': (c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_int, c_vp]),
    'llmc_silu_mul': (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_vp]),
    'llmc_add': (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_vp]),
    'llmc_fp8_quant': (c_int, [c_vp, c_i64, c_i64, c_int, c_i64, c_int, c_int, c_vp, c_int, c_int, c_int,
                               c_vp, c_vp]),
    'llmc_fp8_block_quant': (c_int, [c_vp, c_i64, c_i64, c_int, c_int, c_int, c_vp, c_int, c_vp, c_vp]),
    'llmc_fp8_block_dequant': (c_int, [c_vp, c_i64, c_i64, c_int, c_int, c_vp, c_vp, c_vp]),
    'llmc_fp8_act_quant': (c_int, [c_vp, c_i64, c_i64, c_int, c_vp, c_vp, c_vp]),
    'llmc_fp8_gemm': (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_int, c_i64, c_i64, c_i64,
                              c_vp]),
    'llmc_gemm_w4a16': (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64,
                                c_int, c_vp]),
    'llmc_gemm_w8a16': (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64,
                                c_int, c_vp]),
}

_lock = threading.Lock()
_lib = None


class LlmcB200Error(RuntimeError):
    pass


def load():
    """Load (once) and return the ctypes handle.  Raises if the library is missing."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise LlmcB200Error(
                f'{LIB_PATH} not found: build it with `python -m llmc_b200.build` '
                '(or __graft_entry__.build()).  llmc_b200 has no CPU fallback.')
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            try:
                fn = getattr(lib, name)
            except AttributeError:
                continue  # tests/test_abi.py reports missing symbols explicitly
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def dtype_enum(dt):
    try:
        return _DTYPE[dt]
    except KeyError:
        raise LlmcB200Error(f'unsupported dtype {dt}') from None


def ptr(t):
    if t is None:
        return None
    return ctypes.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise LlmcB200Error(
                'llmc_b200 kernels run on CUDA tensors only (got a %s tensor); there is no CPU '
                'fallback in the product path' % t.device.type)


def check(rc, what):
    if rc != 0:
        lib = load()
        raise LlmcB200Error('%s failed: %s (%s)' % (
            what, lib.llmc_b200_error_string(rc).decode(), lib.llmc_b200_last_error().decode()))


def call(name, *args):
    lib = load()
    rc = getattr(lib, name)(*args)
    check(rc, name)
