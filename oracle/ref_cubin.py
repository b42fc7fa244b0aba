"""Launch the reference's compiled Triton kernels (oracle/_ref/, written by build_ref_triton.py)
through the CUDA driver API with ctypes: cuModuleLoadData, cuFuncSetAttribute for dynamic shared
memory above 48 KB, cuLaunchKernel on torch's current stream.  Needs neither Triton nor the
reference checkout; refuses a kernel or shape that was not compiled.  Test infrastructure only.
"""
import ctypes
import json
import os

import torch

REF_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), '_ref')
MANIFEST = os.path.join(REF_DIR, 'manifest.json')
CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES = 8

_cuda = None
_manifest = None
_funcs = {}


def available():
    return os.path.exists(MANIFEST)


def manifest():
    global _manifest
    if _manifest is None:
        if not available():
            raise FileNotFoundError(f'{MANIFEST} missing: run oracle/build_ref_triton.py')
        with open(MANIFEST) as fh:
            _manifest = json.load(fh)['kernels']
    return _manifest


def _driver():
    global _cuda
    if _cuda is None:
        _cuda = ctypes.CDLL('libcuda.so.1')
    return _cuda


def _ck(rc, what):
    if rc != 0:
        s = ctypes.c_char_p()
        _driver().cuGetErrorString(rc, ctypes.byref(s))
        raise RuntimeError(f'{what} failed: CUresult {rc} ({s.value.decode() if s.value else "?"})')


def _function(name):
    dev = torch.cuda.current_device()
    key = (name, dev)
    if key in _funcs:
        return _funcs[key]
    ent = manifest()[name]
    torch.cuda.init()
    torch.empty(1, device='cuda')            # makes torch's primary context current
    cu = _driver()
    with open(os.path.join(REF_DIR, ent['file']), 'rb') as fh:
        image = fh.read()
    mod = ctypes.c_void_p()
    _ck(cu.cuModuleLoadData(ctypes.byref(mod), ctypes.c_char_p(image)), f'cuModuleLoadData({name})')
    fn = ctypes.c_void_p()
    _ck(cu.cuModuleGetFunction(ctypes.byref(fn), mod, ent['function'].encode()), 'cuModuleGetFunction')
    if ent['shared'] > 48 * 1024:
        _ck(cu.cuFuncSetAttribute(fn, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES,
                                  ctypes.c_int(ent['shared'])), 'cuFuncSetAttribute')
    _funcs[key] = (fn, ent, image)
    return _funcs[key]


def _launch(name, grid, args):
    """args: torch tensors (pointers), python ints (i32) in .entry order, then the scratch pointers."""
    fn, ent, _ = _function(name)
    if ent['global_scratch_size'] or ent['profile_scratch_size']:
        raise RuntimeError(f'{name}: kernels with scratch memory are not supported by this loader')
    holders = []
    for a in args:
        if a is None:
            holders.append(ctypes.c_void_p(0))
        elif torch.is_tensor(a):
            holders.append(ctypes.c_void_p(a.data_ptr()))
        else:
            holders.append(ctypes.c_int32(a))
    holders += [ctypes.c_void_p(0), ctypes.c_void_p(0)]    # global / profile scratch (size 0)
    if len(holders) != len(ent['params']):
        raise RuntimeError(f'{name}: {len(holders)} arguments for {len(ent["params"])} .entry params')
    params = (ctypes.c_void_p * len(holders))(*[ctypes.cast(ctypes.byref(h), ctypes.c_void_p) for h in holders])
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _ck(_driver().cuLaunchKernel(fn, grid[0], grid[1], grid[2], 32 * ent['num_warps'], 1, 1,
                                 ent['shared'], stream, params, None), f'cuLaunchKernel({name})')


def act_quant(x):
    """kernel.py:31-53 with the reference's compiled act_quant_kernel (block 128)."""
    dt = {torch.bfloat16: 'bf16', torch.float16: 'fp16', torch.float32: 'fp32'}[x.dtype]
    assert x.is_contiguous() and x.size(-1) % 128 == 0
    y = torch.empty_like(x, dtype=torch.float8_e4m3fn)
    s = x.new_empty(*x.size()[:-1], x.size(-1) // 128, dtype=torch.float32)
    _launch(f'act_quant_{dt}', (x.numel() // 128, 1, 1), [x, y, s])
    return y, s


def gemm_configs(N, K):
    """The compiled configurations for (N, K): [(name, BLOCK_M, BLOCK_N, num_stages, mma)]."""
    out = [(k, v['BLOCK_M'], v['BLOCK_N'], v['num_stages'], v['mma'])
           for k, v in manifest().items() if v.get('N') == N and v.get('K') == K]
    if not out:
        raise KeyError(f'no reference fp8_gemm cubin for N={N} K={K}: add it to build_ref_triton.SHAPES')
    return sorted(out, key=lambda c: c[1:4])


def fp8_gemm(a, a_s, b, b_s, name):
    """kernel.py:217-242 with one compiled configuration `name` (fp32 output)."""
    assert a.is_contiguous() and b.is_contiguous() and a_s.is_contiguous() and b_s.is_contiguous()
    K = a.size(-1)
    M = a.numel() // K
    N = b.size(0)
    ent = manifest()[name]
    if (ent['N'], ent['K']) != (N, K):
        raise KeyError(f'{name} was compiled for N={ent["N"]} K={ent["K"]}, not N={N} K={K}')
    c = a.new_empty(*a.size()[:-1], N, dtype=torch.float32)
    grid = (-(-M // ent['BLOCK_M']), -(-N // ent['BLOCK_N']), 1)
    _launch(name, grid, [a, b, c, a_s, b_s, M])
    return c
