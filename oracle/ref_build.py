"""Build oracle/_ref/: the REFERENCE's own implementation where it compiles from a few of its source files.
TEST INFRASTRUCTURE (see oracle/__init__.py).

Only the stacked pointnet2 CUDA kernels qualify (stand-alone .cu files: no torch, no THC): they are compiled from the
reference's sources where they lie — nothing is copied — together with oracle/csrc/pointnet2_ref_shim.cu (C-linkage doors)
into oracle/_ref/libpointnet2_stack_ref.so (git-ignored).  `python -m oracle.make_golden roi_pool` runs it on a GPU and
stores its outputs in tests/golden/roi_pool.npz, the checker of tests/test_gpu_roi_pool.py.  The sparse-conv arithmetic
itself (spconv/cumm) is not buildable this way, see DESIGN.md §2.

    python -m oracle.ref_build
"""
from __future__ import annotations

import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
REF_SRC = '/root/reference/pcdet/ops/pointnet2/pointnet2_stack/src'
OUT_DIR = os.path.join(HERE, '_ref')
LIB = os.path.join(OUT_DIR, 'libpointnet2_stack_ref.so')
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')


def available() -> bool:
    return os.path.exists(LIB)


def build(force: bool = False):
    """-> path of the library, or None when /root/reference is absent (GPU box: uses the prebuilt file if it travelled)."""
    if not os.path.isdir(REF_SRC):
        return LIB if available() else None
    srcs = [os.path.join(HERE, 'csrc', 'pointnet2_ref_shim.cu'), os.path.join(REF_SRC, 'voxel_query_gpu.cu'),
            os.path.join(REF_SRC, 'group_points_gpu.cu')]
    if available() and not force and all(os.path.getmtime(LIB) >= os.path.getmtime(s) for s in srcs):
        return LIB
    os.makedirs(OUT_DIR, exist_ok=True)
    cmd = [NVCC, '-O3', '-std=c++17', '-gencode', 'arch=compute_100a,code=sm_100a', '-shared', '-Xcompiler', '-fPIC',
           '-I', os.path.join(HERE, 'csrc', 'ref_shim_include'), '-I', REF_SRC, '-o', LIB] + srcs
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError('building the reference pointnet2 kernels failed:\n%s\n%s' % (r.stdout, r.stderr))
    return LIB


if __name__ == '__main__':
    print(build(force=True))
