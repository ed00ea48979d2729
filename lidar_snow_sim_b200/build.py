"""
Build the engine's shared library IN-TREE with nvcc for sm_100a (cross-compiles without a GPU):

    python -m lidar_snow_sim_b200.build [--force]

Output: lidar_snow_sim_b200/liblss_b200.so (git-ignored, travels to the GPU box with the snapshot).
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'liblss_b200.so')
SOURCES = ['api.cu', 'tables.cu', 'snowfall.cu', 'solve.cu', 'prepass.cu', 'wet_ground.cu', 'sampler.cu', 'sampler_gpu.cu', 'host_pipeline.cu', 'fog.cu', 'voxelize.cu', 'lisa.cu', 'gather.cu', 'dror.cu']
# -fmad=false: float32/float64 expressions are evaluated as written (mul, then add), like NumPy on the reference host;
# where a fused multiply-add is wanted the source says fma() / __fma_rn() explicitly.
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17', '-fmad=false',
              '-Xcompiler', '-fPIC', '-Xcompiler', '-fvisibility=hidden', '-Xcompiler', '-ffp-contract=off', '--shared', '-cudart', 'static']


def find_nvcc():
    for cand in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError('nvcc not found')


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if not f.startswith('_')] + [__file__] + [os.path.join(HERE, '..', 'include', 'lidar_snow_sim.h')]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, extra=()):
    """Compile every translation unit (in parallel, objects under csrc/_obj/) and link the shared library."""
    env_extra = os.environ.get('LSS_NVCC_FLAGS', '').split()       # tuning experiments: e.g. -DLSS_SOLVE_CTAS=5
    if env_extra:
        extra, force = list(extra) + env_extra, True
    if not force and not needs_build():
        return LIB
    from concurrent.futures import ThreadPoolExecutor
    nvcc = find_nvcc()
    objdir = os.path.join(CSRC, '_obj')
    os.makedirs(objdir, exist_ok=True)
    compile_flags = [f for f in NVCC_FLAGS if f not in ('--shared',)]
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cuh', '.h'))]
    headers.append(os.path.join(HERE, '..', 'include', 'lidar_snow_sim.h'))
    newest_header = max(os.path.getmtime(h) for h in headers)

    def compile_one(src):
        obj = os.path.join(objdir, src.replace('.cu', '.o'))
        path = os.path.join(CSRC, src)
        if (not force and not extra and os.path.exists(obj) and
                os.path.getmtime(obj) > max(os.path.getmtime(path), newest_header, os.path.getmtime(__file__))):
            return obj
        cmd = [nvcc] + compile_flags + list(extra) + ['-c', '-o', obj, path]
        if verbose:
            print(' '.join(cmd))
        subprocess.check_call(cmd)
        return obj

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 4)) as pool:
        objs = list(pool.map(compile_one, SOURCES))
    cmd = [nvcc] + NVCC_FLAGS + ['-o', LIB] + objs
    if verbose:
        print(' '.join(cmd))
    subprocess.check_call(cmd)
    return LIB


if __name__ == '__main__':
    build(force='--force' in sys.argv, verbose=True, extra=['-Xptxas', '-v'] if '-v' in sys.argv else [])
    print(LIB)
