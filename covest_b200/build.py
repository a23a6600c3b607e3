"""Builds libcovest_b200.so (hand-written CUDA for sm_100a + the C ABI) in-tree with nvcc.

    python -m covest_b200.build            # -> covest_b200/lib/libcovest_b200.so

nvcc cross-compiles without a GPU.  The built library is git-ignored but travels with the tree.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB_DIR = os.path.join(HERE, 'lib')
LIB_PATH = os.path.join(LIB_DIR, 'libcovest_b200.so')
SOURCES = ['kernels.cu', 'factored.cu', 'faithful.cu', 'topk.cu', 'profile.cu', 'kmers.cu', 'capi.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC', '-Xcompiler', '-fvisibility=hidden', '-Xcompiler', '-ffp-contract=off',
              '--fmad=false']


def find_nvcc():
    for cand in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError('nvcc not found (set NVCC=/path/to/nvcc)')


def _deps():
    out = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cu', '.h'))]
    out.append(os.path.join(os.path.dirname(HERE), 'include', 'covest_b200.h'))
    return out


def is_stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(d) > t for d in _deps())


def build_library(force=False, verbose=False):
    """Compile the library if it is missing or older than its sources; returns its path."""
    if not force and not is_stale():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    nvcc = find_nvcc()
    cmd = [nvcc] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-shared'] + \
        [os.path.join(CSRC, s) for s in SOURCES] + ['-o', LIB_PATH]
    if verbose:
        print(' '.join(cmd), file=sys.stderr)
    subprocess.check_call(cmd)
    return LIB_PATH


if __name__ == '__main__':
    print(build_library(force='--force' in sys.argv, verbose='-v' in sys.argv))
