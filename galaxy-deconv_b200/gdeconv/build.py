"""Build libgdeconv.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo snapshot)."""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(PKG, 'csrc')
LIB = os.path.join(PKG, 'gdeconv', 'libgdeconv.so')
STAMP = LIB + '.srchash'
SOURCES = ['api.cu', 'fft_kernels.cu', 'subnet.cu', 'conv_simt.cu', 'conv_umma.cu', 'conv_rb.cu', 'conv_l1chain.cu', 'conv_l2chain.cu', 'xdense.cu', 'synth.cu', 'shape.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17', '--use_fast_math=false',
              '-Xcompiler', '-fPIC', '-Xcompiler', '-fvisibility=hidden', '--expt-relaxed-constexpr']


def _nvcc():
    for c in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError('nvcc not found')


def source_hash():
    h = hashlib.sha256()
    files = sorted(f for f in os.listdir(CSRC) if f.endswith(('.cu', '.cuh')))
    files.append(os.path.join('..', '..', 'include', 'gdeconv.h'))
    for f in files:
        with open(os.path.join(CSRC, f), 'rb') as fh:
            h.update(f.encode()); h.update(fh.read())
    h.update(' '.join(NVCC_FLAGS).encode())
    return h.hexdigest()


def is_current():
    try:
        return os.path.exists(LIB) and open(STAMP).read().strip() == source_hash()
    except OSError:
        return False


def build(force=False, verbose=False):
    """Compile every .cu to an object (in parallel) and link the shared library."""
    if not force and is_current():
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(PKG, 'build')
    os.makedirs(objdir, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if f != '--use_fast_math=false']
    procs = []
    for s in SOURCES:
        obj = os.path.join(objdir, s.replace('.cu', '.o'))
        cmd = [nvcc, *flags, '-Xptxas', '-v', '-c', os.path.join(CSRC, s), '-o', obj]
        procs.append((s, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs, log = [], []
    for s, obj, p in procs:
        out, _ = p.communicate()
        log.append(f'--- {s}\n{out}')
        if p.returncode != 0:
            raise RuntimeError(f'nvcc failed on {s}:\n{out}')
        objs.append(obj)
    cmd = [nvcc, '-shared', '-gencode', 'arch=compute_100a,code=sm_100a', *objs, '-o', LIB]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError('link failed:\n' + r.stdout)
    with open(os.path.join(objdir, 'ptxas.log'), 'w') as fh:
        fh.write('\n'.join(log))
    with open(STAMP, 'w') as fh:
        fh.write(source_hash())
    if verbose:
        print('\n'.join(log))
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
