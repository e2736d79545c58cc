"""In-tree build of libdctp.so (hand-written CUDA for sm_100a behind the C ABI in include/dctp.h).

nvcc cross-compiles without a GPU.  The .so lands next to this file so it travels with the
repo snapshot; it is git-ignored.  There is no other backend and no CPU fallback.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
CSRC = os.path.join(HERE, 'csrc')
LIB_PATH = os.path.join(HERE, 'libdctp.so')
SOURCES = [os.path.join(CSRC, 'dctp.cu')]
HEADERS = [os.path.join(CSRC, f) for f in ('umma.cuh', 'score_common.cuh', 'score_umma.cuh', 'score_tmem.cuh', 'score_stack.cuh', 'score_kron.cuh', 'score_large.cuh', 'score_simt.cuh', 'topk.cuh', 'gather.cuh', 'score_alt.cuh', 'widen.cuh')] + \
          [os.path.join(REPO, 'include', 'dctp.h')]
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-shared', '-Xcompiler', '-fPIC', '-Xptxas', '-v']


def find_nvcc():
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    return 'nvcc'


def is_stale():
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(p) > built for p in SOURCES + HEADERS)


def build_library(force=False, verbose=False):
    """Compile libdctp.so if missing or older than its sources.  Returns the path."""
    if not force and not is_stale():
        return LIB_PATH
    cmd = [find_nvcc()] + NVCC_FLAGS + ['-I', os.path.join(REPO, 'include'), '-o', LIB_PATH] + SOURCES
    proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or proc.returncode != 0:
        sys.stderr.write(proc.stdout)
    if proc.returncode != 0:
        raise RuntimeError('nvcc failed (%d): %s' % (proc.returncode, ' '.join(cmd)))
    return LIB_PATH


if __name__ == '__main__':
    print(build_library(force='--force' in sys.argv, verbose=True))
