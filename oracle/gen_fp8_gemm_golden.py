"""Write tests/golden/fp8_gemm_kat.pt: the reference's fp8_gemm_kernel (llmc/compression/quantization/
kernel.py:141-214) run under Triton's CPU interpreter with two explicit configurations, on fp8
operands and fp32 scales made by torch.  Build machine only (needs the llmc checkout and Triton):

    python oracle/gen_fp8_gemm_golden.py [/path/to/llmc-checkout]

Only the GEMM is taken from the interpreter: its float -> e4m3 conversion does not round to
nearest even, so the fp8 inputs come from torch.  The file holds the seeds, the operands' bytes,
the scales and both outputs."""
import os
import sys

os.environ['TRITON_INTERPRET'] = '1'

import torch  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, 'tests', 'golden', 'fp8_gemm_kat.pt')
SHAPES = [(1, 576, 256), (77, 200, 384), (33, 256, 128)]     # (M, N, K)
CONFIGS = [(16, 32), (64, 128)]                                             # (BLOCK_M, BLOCK_N)


def operands(M, N, K, seed):
    g = torch.Generator().manual_seed(seed)
    a = (torch.randn(M, K, generator=g) * 40).clamp(-448, 448).to(torch.float8_e4m3fn)
    b = (torch.randn(N, K, generator=g) * 40).clamp(-448, 448).to(torch.float8_e4m3fn)
    a_s = torch.rand(M, K // 128, generator=g) * 0.01 + 1e-3
    b_s = torch.rand(-(-N // 128), K // 128, generator=g) * 0.01 + 1e-3
    return a, a_s, b, b_s


def main(ref_root):
    import importlib.util
    spec = importlib.util.spec_from_file_location(
        '_llmc_ref_kernel', os.path.join(ref_root, 'llmc/compression/quantization/kernel.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    kern = mod.fp8_gemm_kernel.fn
    cases = []
    for i, (M, N, K) in enumerate(SHAPES):
        seed = 100 + i
        a, a_s, b, b_s = operands(M, N, K, seed)
        outs = {}
        for bm, bn in CONFIGS:
            c = torch.empty(M, N, dtype=torch.float32)
            grid = (-(-M // bm), -(-N // bn))
            kern[grid](a, b, c, a_s, b_s, M, N, K, BLOCK_SIZE_M=bm, BLOCK_SIZE_N=bn, BLOCK_SIZE_K=128)
            outs[f'm{bm}n{bn}'] = c
        cases.append({'M': M, 'N': N, 'K': K, 'seed': seed, 'a': a.view(torch.uint8),
                      'b': b.view(torch.uint8), 'a_s': a_s, 'b_s': b_s, 'c': outs})
    torch.save({'source': 'kernel.py fp8_gemm_kernel under TRITON_INTERPRET=1', 'cases': cases}, OUT)
    print(OUT, os.path.getsize(OUT))


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else os.environ.get('LLMC_REFERENCE', '/root/reference'))
