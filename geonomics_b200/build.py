"""In-tree build of libgnxb200.so with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
SOURCES = ['gnx_api.cu']
DEPS = ['gnx_api.cu', 'gnx_kernels.cuh', 'gnx_scan.cuh', 'gnx_common.cuh', 'gnx_strip.cuh', 'gnx_genome_init.cuh', 'gnx_simplify.cuh', '../../include/gnx_b200.h']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
              '-Xcompiler', '-fPIC', '-shared']


def library_path():
    return os.path.join(HERE, 'libgnxb200.so')


def _stale(out):
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def build_library(force=False, verbose=False):
    out = library_path()
    if not force and not _stale(out):
        return out
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    cmd = [nvcc] + NVCC_FLAGS + [os.path.join(CSRC, s) for s in SOURCES] + ['-o', out]
    if verbose:
        cmd.insert(1, '-Xptxas')
        cmd.insert(2, '-v')
        print(' '.join(cmd))
    subprocess.run(cmd, check=True, cwd=CSRC)
    return out
