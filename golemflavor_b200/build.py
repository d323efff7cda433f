"""In-tree build of ``libgolemflavor_b200.so`` with nvcc for sm_100a.

``python -m golemflavor_b200.build [--force]``.  The library lands in ``golemflavor_b200/lib/`` (git-ignored,
but it travels with the working tree to the GPU box).
"""

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB_DIR = os.path.join(HERE, 'lib')
LIB_PATH = os.path.join(LIB_DIR, 'libgolemflavor_b200.so')
SOURCES = ['gf_api.cu', 'gf_lnprob.cu', 'gf_scan.cu', 'gf_ensemble.cu', 'gf_profile.cu']
HEADERS = ['gf_common.cuh', 'gf_model.cuh', 'gf_physics.cuh', 'gf_scan_dev.cuh', 'gf_ensemble_dev.cuh', 'gf_profile_dev.cuh', 'gf_ndtri_table.h', os.path.join('..', '..', 'include', 'golemflavor_b200.h')]
NVCC_FLAGS = ['-O3', '-std=c++17', '--threads', '4', '-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo',
              '-Xcompiler', '-fPIC', '-shared', '-Xlinker', '-soname=libgolemflavor_b200.so']


def nvcc_path():
    for cand in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError('nvcc not found (set NVCC=/path/to/nvcc)')


TORCH_OPS_SRC = os.path.join(CSRC, 'gf_torch_ops.cpp')
TORCH_OPS_PATH = os.path.join(LIB_DIR, 'libgolemflavor_b200_torch.so')


def build_torch_ops(force=False, verbose=False):
    """Compile the `torch.ops.golemflavor.*` registration (gf_torch_ops.cpp) with g++ against the torch headers of the
    running interpreter, linked to the C-ABI library next to it (rpath $ORIGIN).  In-tree, no JIT cache."""
    deps = [TORCH_OPS_SRC, os.path.join(CSRC, '..', '..', 'include', 'golemflavor_b200.h')]
    if not force and os.path.exists(TORCH_OPS_PATH) and all(os.path.getmtime(d) <= os.path.getmtime(TORCH_OPS_PATH) for d in deps):
        return TORCH_OPS_PATH
    build_library()
    import torch
    tdir = os.path.dirname(torch.__file__)
    cuda_inc = os.path.join(os.path.dirname(os.path.dirname(nvcc_path())), 'include')
    cmd = ['g++', '-O2', '-std=c++17', '-fPIC', '-shared', '-D_GLIBCXX_USE_CXX11_ABI=%d' % int(torch._C._GLIBCXX_USE_CXX11_ABI),
           '-I' + os.path.join(tdir, 'include'), '-I' + os.path.join(tdir, 'include', 'torch', 'csrc', 'api', 'include'), '-I' + cuda_inc,
           TORCH_OPS_SRC, '-o', TORCH_OPS_PATH, '-L' + LIB_DIR, '-lgolemflavor_b200', '-L' + os.path.join(tdir, 'lib'),
           '-ltorch', '-ltorch_cpu', '-ltorch_cuda', '-lc10', '-lc10_cuda', '-Wl,-rpath,$ORIGIN', '-Wl,-rpath,' + os.path.join(tdir, 'lib')]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout)
    if res.returncode != 0:
        raise RuntimeError('g++ failed ({0}): {1}'.format(res.returncode, ' '.join(cmd)))
    return TORCH_OPS_PATH


def is_stale():
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > built for d in deps)


def build_library(force=False, verbose=False):
    """Compile the three translation units into one shared library.  Returns its path."""
    if not force and not is_stale():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    cmd = [nvcc_path()] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + \
        ['-o', LIB_PATH] + [os.path.join(CSRC, f) for f in SOURCES]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout)
    if res.returncode != 0:
        raise RuntimeError('nvcc failed ({0}): {1}'.format(res.returncode, ' '.join(cmd)))
    return LIB_PATH


if __name__ == '__main__':
    print(build_library(force='--force' in sys.argv, verbose='-v' in sys.argv))
    print(build_torch_ops(force='--force' in sys.argv, verbose='-v' in sys.argv))
