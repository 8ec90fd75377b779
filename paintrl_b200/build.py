"""Build the in-tree CUDA library `paintrl_b200/libpaintrl_b200.so` for sm_100a.

    python -m paintrl_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  `-fmad=false` is part of the arithmetic contract (every FP64
product and sum is rounded separately, FMA only where written explicitly); `-lineinfo` keeps the
ncu source page mapped to the .cuh files; the CUDA runtime is linked statically so the library
has no dependency on torch's or the system's libcudart.
"""
import os
import subprocess
import sys

_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_DIR, 'csrc')
SOURCES = [os.path.join(CSRC, 'paintrl_capi.cu')]
HEADERS = [os.path.join(CSRC, 'paintrl_device.cuh'), os.path.join(CSRC, 'paintrl_kernels.cuh'), os.path.join(CSRC, 'paintrl_raster.cuh'), os.path.join(CSRC, 'paintrl_param.cuh'), os.path.join(CSRC, 'paintrl_policy.cuh'),
           os.path.join(CSRC, 'paintrl_learn.cuh'),
           os.path.join(os.path.dirname(_DIR), 'include', 'paintrl.h')]
LIB = os.path.join(_DIR, 'libpaintrl_b200.so')

NVCC_FLAGS = ['-O3', '-std=c++17', '-gencode', 'arch=compute_100a,code=sm_100a', '-fmad=false',
              '-lineinfo', '-cudart', 'static', '-Xcompiler', '-fPIC', '-Xcompiler', '-ffp-contract=off',
              '-shared']


def nvcc_path():
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if cand and (os.path.isfile(cand) or cand == 'nvcc'):
            return cand
    return 'nvcc'


def up_to_date():
    if not os.path.isfile(LIB):
        return False
    t = os.path.getmtime(LIB)
    return all(os.path.getmtime(p) <= t for p in SOURCES + HEADERS + [os.path.abspath(__file__)])


def build(force=False, verbose=False):
    if not force and up_to_date():
        return LIB
    extra = ['-DPAINTRL_PROFILE'] if os.environ.get('PAINTRL_PROFILE') else []   # phase timing build (profiles/)
    extra += ['-DPAINTRL_TRACE'] if os.environ.get('PAINTRL_TRACE') else []     # per-warp timeline build (profiles/timeline.py)
    extra += os.environ.get('PAINTRL_NVCC_EXTRA', '').split()                    # experiments, e.g. -DPAINTRL_PAINT_OCC=32
    cmd = [nvcc_path()] + NVCC_FLAGS + extra + (['-Xptxas', '-v'] if verbose else []) + SOURCES + ['-o', LIB]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout)
    if res.returncode != 0:
        raise RuntimeError('nvcc failed (%d): %s' % (res.returncode, ' '.join(cmd)))
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='--verbose' in sys.argv))
