"""Build ``libvittles_b200.so`` (sm_100a only) with nvcc, in-tree.

    python -m vittles_b200.build [--force]

Objects are compiled in parallel and linked into
``vittles_b200/lib/libvittles_b200.so``.  The library links the static CUDA
runtime, exports only the ``extern "C"`` functions of
``include/vittles_b200.h`` and has no dependency on torch.
"""
import concurrent.futures
import hashlib
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, 'csrc')
LIBDIR = os.path.join(PKG, 'lib')
LIB = os.path.join(LIBDIR, 'libvittles_b200.so')
OBJDIR = os.path.join(PKG, 'build')
SOURCES = ['common.cu', 'dgemm.cu', 'glm.cu', 'chol.cu', 'synth.cu', 'blockchol.cu', 'tgemm.cu', 'ogemm.cu', 'grouploo.cu', 'abi.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC'] + os.environ.get('VT_NVCC_EXTRA', '').split()


def _nvcc():
    return shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'


def _digest(paths):
    h = hashlib.sha256()
    for p in sorted(paths):
        with open(p, 'rb') as f:
            h.update(p.encode())
            h.update(f.read())
    h.update(' '.join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _all_inputs():
    files = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cu', '.cuh', '.h'))]
    files.append(os.path.join(os.path.dirname(PKG), 'include', 'vittles_b200.h'))
    return files


def is_current():
    stamp = os.path.join(LIBDIR, 'build.sha256')
    if not (os.path.exists(LIB) and os.path.exists(stamp)):
        return False
    with open(stamp) as f:
        return f.read().strip() == _digest(_all_inputs())


def build(force=False, verbose=True):
    if not force and is_current():
        if verbose:
            print('[vittles_b200.build] up to date:', LIB)
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    os.makedirs(OBJDIR, exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(OBJDIR, src.replace('.cu', '.o'))
        cmd = [nvcc] + NVCC_FLAGS + ['-c', os.path.join(CSRC, src), '-o', obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError('nvcc failed for {}:\n{}\n{}'.format(src, r.stdout, r.stderr))
        return obj

    srcs = _sources()
    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        objs = list(ex.map(compile_one, srcs))
    cmd = [nvcc, '-shared', '-gencode', 'arch=compute_100a,code=sm_100a', '-o', LIB] + objs
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError('link failed:\n{}\n{}'.format(r.stdout, r.stderr))
    with open(os.path.join(LIBDIR, 'build.sha256'), 'w') as f:
        f.write(_digest(_all_inputs()))
    if verbose:
        print('[vittles_b200.build] built', LIB)
    return LIB


if __name__ == '__main__':
    build(force='--force' in sys.argv)
