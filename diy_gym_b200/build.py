"""Builds libdiygym_b200.so (CUDA kernels + C ABI) for sm_100a with nvcc.  Run: python -m diy_gym_b200.build

dg_kernels.cu is compiled once per team size (-DDG_STEP_T=<T>: only dg_step_kernel<T> and its host wrappers) and once
for everything else (-DDG_SPLIT_BUILD), in parallel, and the objects are linked into one shared library."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.environ.get('DG_LIB') or os.path.join(HERE, 'libdiygym_b200.so')   # DG_LIB: load an alternative build (experiments)
OBJ_DIR = os.path.join(HERE, '_obj')
SOURCE = 'dg_kernels.cu'
TEAMS = [1, 2, 4, 8, 16, 32]
DEPS = ['dg_kernels.cu', 'dg_env.cuh', 'dg_ray.cuh', 'dg_dyn.cuh', 'dg_ik.cuh', 'dg_math.cuh', 'dg_scene.h', 'scene_sections.h', os.path.join('..', '..', 'include', 'diygym_b200.h')]
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17', '-Xcompiler', '-fPIC']


def stale():
    if not os.path.isfile(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def build_library(force=False, verbose=False, extra_flags=()):
    if not force and not stale():
        return LIB
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    os.makedirs(OBJ_DIR, exist_ok=True)
    tag = os.path.splitext(os.path.basename(LIB))[0]
    flags = NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + list(extra_flags)
    jobs = [(['-DDG_SPLIT_BUILD'], os.path.join(OBJ_DIR, '%s_abi.o' % tag))]
    jobs += [(['-DDG_STEP_T=%d' % t], os.path.join(OBJ_DIR, '%s_step_t%d.o' % (tag, t))) for t in TEAMS]

    def compile_one(job):
        defs, obj = job
        subprocess.check_call([nvcc] + flags + defs + ['-c', '-o', obj, os.path.join(CSRC, SOURCE)])
        return obj

    with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as pool:
        objs = list(pool.map(compile_one, jobs))
    subprocess.check_call([nvcc, '-shared', '-o', LIB] + objs)
    return LIB


if __name__ == '__main__':
    build_library(force='--force' in sys.argv, verbose='-v' in sys.argv)
    print(LIB)
