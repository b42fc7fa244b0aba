"""Build libllmc_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

The library has NO torch / Python dependency: plain `nvcc -shared`, static cudart, the driver
API (cuTensorMapEncodeTiled) resolved at run time through cudaGetDriverEntryPoint so that
the .so also loads on a CPU-only box (tests/test_abi.py checks the exported symbols there).
"""
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB_NAME = 'libllmc_b200.so'
LIB_PATH = os.path.join(HERE, LIB_NAME)

NVCC_FLAGS = [
    '-gencode', 'arch=compute_100a,code=sm_100a',
    '-O3', '-std=c++20', '-lineinfo',
    '-Xcompiler', '-fPIC',
    '--expt-relaxed-constexpr',
    '-cudart', 'static',
]


def _nvcc():
    for cand in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError('nvcc not found; cannot build libllmc_b200.so')


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith('.cu'))


def _digest():
    h = hashlib.sha256()
    inc = os.path.join(HERE, '..', 'include', 'llmc_b200.h')
    files = sources() + sorted(
        os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith('.cuh')) + [inc]
    for f in files:
        with open(f, 'rb') as fh:
            h.update(fh.read())
    h.update(' '.join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile every .cu under csrc/ into objects (parallel) and link the shared library."""
    stamp = LIB_PATH + '.stamp'
    digest = _digest()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp):
        with open(stamp) as fh:
            if fh.read().strip() == digest:
                return LIB_PATH
    nvcc = _nvcc()
    objdir = os.path.join(HERE, 'build')
    os.makedirs(objdir, exist_ok=True)
    procs = []
    objs = []
    for src in sources():
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + '.o')
        objs.append(obj)
        cmd = [nvcc] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-c', src, '-o', obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        txt = out.decode(errors='replace')
        if p.returncode != 0:
            failed = True
            sys.stderr.write(f'--- nvcc failed on {src}\n{txt}\n')
        elif verbose or 'warning' in txt:
            sys.stderr.write(txt)
    if failed:
        raise RuntimeError('nvcc compilation failed')
    cmd = [nvcc, '-shared', '-cudart', 'static', '-gencode', 'arch=compute_100a,code=sm_100a',
           '-o', LIB_PATH] + objs + ['-ldl']
    subprocess.check_call(cmd)
    with open(stamp, 'w') as fh:
        fh.write(digest)
    return LIB_PATH


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
