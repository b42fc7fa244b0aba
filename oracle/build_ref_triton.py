"""Compile the reference's own Triton kernels (llmc/compression/quantization/kernel.py) for sm_100a
into oracle/_ref/, so that the GPU tests and scripts/bench_fp8_gemm.py can launch them as the
parity oracle and the performance bar without Triton on the GPU machine (oracle/ref_cubin.py).

  * act_quant_kernel for bf16, fp16 and fp32 inputs (BLOCK_SIZE 128);
  * fp8_gemm_kernel with fp32 output for every (N, K) in SHAPES, in all 36 configurations of the
    reference's autotuner (BLOCK_M x BLOCK_N x num_stages, BLOCK_K 128, 8 warps), since which one
    the autotuner picks on a B200 is a matter of timing.

The reference functions are loaded read-only from an llmc checkout (LLMC_REFERENCE, default
REF below); nothing from it is written into the repository.  Each cubin comes with its PTX and an
entry in manifest.json: name, file, num_warps, shared bytes, scratch sizes, the grid rule, the
.entry parameter list parsed from the PTX, and which MMA instruction family the PTX uses.

If the checkout or Triton is missing this prints a note and leaves existing artefacts alone;
it never raises (build() calls it).
"""
import hashlib
import json
import os
import re
import sys
from concurrent.futures import ProcessPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, '_ref')
REF = os.environ.get('LLMC_REFERENCE', '/root/reference')
KERNEL_PY = 'llmc/compression/quantization/kernel.py'

# (N, K) of the tests (DeepSeek-like layers, a ragged N, the tiny Llama of llmc_b200/synth.py) and
# of scripts/bench_fp8_gemm.py (DeepSeek-V3 layers at hidden size 7168)
TEST_SHAPES = [(576, 7168), (1536, 7168), (200, 384), (256, 256), (128, 256), (512, 256),
               (256, 512)]
BENCH_SHAPES = [(1536, 7168), (576, 7168), (24576, 1536), (7168, 16384), (18432, 7168),
                (7168, 18432), (2048, 7168)]
SHAPES = sorted(set(TEST_SHAPES + BENCH_SHAPES))
CONFIGS = [(bm, bn, st) for bm in (16, 32, 64) for bn in (32, 64, 128) for st in (3, 4, 5, 6)]
ACT_DTYPES = {'bf16': '*bf16', 'fp16': '*fp16', 'fp32': '*fp32'}


def gemm_name(N, K, bm, bn, st):
    return f'fp8_gemm_N{N}_K{K}_m{bm}n{bn}s{st}'


def _load_reference(path):
    import importlib.util
    spec = importlib.util.spec_from_file_location('_llmc_ref_kernel', path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _entry_params(ptx):
    m = re.search(r'\.entry\s+\w+\s*\((.*?)\)', ptx, re.S)
    return [' '.join(p.split()) for p in m.group(1).split(',')] if m else []


def _mma_kind(ptx):
    if 'tcgen05.mma' in ptx:
        return 'tcgen05'
    if 'mma.sync' in ptx:
        return 'mma.sync'
    return 'none'


def _compile(job):
    kind, args, ref_path = job
    import triton
    from triton.backends.compiler import GPUTarget
    from triton.compiler import ASTSource
    mod = _load_reference(ref_path)
    target = GPUTarget('cuda', 100, 32)
    if kind == 'act':
        dt, = args
        src = ASTSource(fn=mod.act_quant_kernel,
                        signature={'x_ptr': ACT_DTYPES[dt], 'y_ptr': '*fp8e4nv', 's_ptr': '*fp32',
                                   'BLOCK_SIZE': 'constexpr'},
                        constexprs={'BLOCK_SIZE': 128})
        k = triton.compile(src, target=target)
        name, grid = f'act_quant_{dt}', 'cdiv(numel, 128), 1, 1'
        extra = {'dtype': dt}
    else:
        N, K, bm, bn, st = args
        src = ASTSource(fn=mod.fp8_gemm_kernel.fn,
                        signature={'a_ptr': '*fp8e4nv', 'b_ptr': '*fp8e4nv', 'c_ptr': '*fp32',
                                   'a_s_ptr': '*fp32', 'b_s_ptr': '*fp32', 'M': 'i32',
                                   'N': 'constexpr', 'K': 'constexpr', 'BLOCK_SIZE_M': 'constexpr',
                                   'BLOCK_SIZE_N': 'constexpr', 'BLOCK_SIZE_K': 'constexpr'},
                        constexprs={'N': N, 'K': K, 'BLOCK_SIZE_M': bm, 'BLOCK_SIZE_N': bn,
                                    'BLOCK_SIZE_K': 128})
        k = triton.compile(src, target=target, options={'num_warps': 8, 'num_stages': st})
        name, grid = gemm_name(N, K, bm, bn, st), f'cdiv(M, {bm}), cdiv(N, {bn}), 1'
        extra = {'N': N, 'K': K, 'BLOCK_M': bm, 'BLOCK_N': bn, 'num_stages': st}
    ptx = k.asm['ptx']
    with open(os.path.join(OUT, name + '.cubin'), 'wb') as fh:
        fh.write(k.asm['cubin'])
    with open(os.path.join(OUT, name + '.ptx'), 'w') as fh:
        fh.write(ptx)
    md = k.metadata
    entry = {'name': name, 'file': name + '.cubin', 'function': md.name, 'num_warps': md.num_warps,
             'shared': md.shared, 'global_scratch_size': getattr(md, 'global_scratch_size', 0),
             'profile_scratch_size': getattr(md, 'profile_scratch_size', 0), 'grid': grid,
             'params': _entry_params(ptx), 'mma': _mma_kind(ptx)}
    entry.update(extra)
    return entry


def _key(ref_path, triton_version):
    h = hashlib.sha256()
    with open(ref_path, 'rb') as fh:
        h.update(fh.read())
    h.update(triton_version.encode())
    h.update(repr((SHAPES, CONFIGS, sorted(ACT_DTYPES))).encode())
    return h.hexdigest()


def build(ref_root=REF, jobs=None, quiet=False):
    """Returns the manifest path, or None when the reference or Triton is unavailable."""
    def note(msg):
        if not quiet:
            print(f'oracle/build_ref_triton: {msg}', file=sys.stderr)
    ref_path = os.path.join(ref_root, KERNEL_PY)
    if not os.path.isfile(ref_path):
        note(f'{ref_path} not found; reference cubins not (re)built')
        return None
    try:
        import triton
    except Exception as e:  # noqa: BLE001
        note(f'triton unavailable ({e}); reference cubins not (re)built')
        return None
    manifest = os.path.join(OUT, 'manifest.json')
    key = _key(ref_path, triton.__version__)
    if os.path.exists(manifest):
        try:
            with open(manifest) as fh:
                if json.load(fh).get('key') == key:
                    return manifest
        except Exception:  # noqa: BLE001
            pass
    os.makedirs(OUT, exist_ok=True)
    work = [('act', (dt,), ref_path) for dt in ACT_DTYPES]
    work += [('gemm', (N, K) + cfg, ref_path) for N, K in SHAPES for cfg in CONFIGS]
    try:
        with ProcessPoolExecutor(max_workers=jobs or os.cpu_count()) as ex:
            entries = list(ex.map(_compile, work, chunksize=4))
    except Exception as e:  # noqa: BLE001
        note(f'compiling the reference kernels failed ({type(e).__name__}: {e}); left as is')
        return None
    doc = {'key': key, 'triton': triton.__version__, 'target': 'cuda:100 (sm_100a)',
           'source': KERNEL_PY, 'kernels': {e['name']: e for e in entries}}
    with open(manifest + '.tmp', 'w') as fh:
        json.dump(doc, fh, indent=1)
    os.replace(manifest + '.tmp', manifest)
    note(f'{len(entries)} reference kernels compiled into {OUT}')
    return manifest


if __name__ == '__main__':
    print(build(sys.argv[1] if len(sys.argv) > 1 else REF))
