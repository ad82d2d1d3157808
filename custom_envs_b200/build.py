"""In-tree build of libb200env.so for sm_100a (nvcc cross-compiles without a GPU)."""
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(_HERE)
SOURCES = [os.path.join(_HERE, 'csrc', 'b200env.cu'), os.path.join(_HERE, 'csrc', 'b200tc.cu'),
           os.path.join(_HERE, 'csrc', 'b200data.cu'), os.path.join(_HERE, 'csrc', 'b200policy.cu'),
           os.path.join(_HERE, 'csrc', 'b200tiny.cu'), os.path.join(_HERE, 'csrc', 'b200thin.cu')]
HEADERS = [os.path.join(ROOT, 'include', 'b200env.h'), os.path.join(ROOT, 'include', 'b200data.h'),
           os.path.join(ROOT, 'include', 'b200policy.h'),
           os.path.join(_HERE, 'csrc', 'b200env_shared.cuh'), os.path.join(_HERE, 'csrc', 'b200adam.cuh'), os.path.join(_HERE, 'csrc', 'b200tc.h'),
           os.path.join(_HERE, 'csrc', 'b200env_internal.h'), os.path.join(_HERE, 'csrc', 'b200tiny.h'), os.path.join(_HERE, 'csrc', 'b200thin.h')]
OBJ_DIR = os.path.join(_HERE, 'csrc', '_obj')
OUTPUT = os.path.join(_HERE, 'libb200env.so')
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
              '-Xcompiler', '-fPIC', '-I', os.path.join(ROOT, 'include')]


def build_library(force=False, verbose=False):
    """Compile csrc/*.cu -> objects -> custom_envs_b200/libb200env.so; only stale objects are
    recompiled (the env kernels take minutes, the data front-end seconds)."""
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    os.makedirs(OBJ_DIR, exist_ok=True)
    header_time = max(os.path.getmtime(p) for p in HEADERS)
    objects, relink = [], force or not os.path.exists(OUTPUT)
    jobs = []
    for source in SOURCES:
        obj = os.path.join(OBJ_DIR, os.path.splitext(os.path.basename(source))[0] + '.o')
        objects.append(obj)
        newest = max(os.path.getmtime(source), header_time)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < newest:
            cmd = [nvcc] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-c', '-o', obj, source]
            jobs.append((cmd, subprocess.Popen(cmd)))           # translation units compile side by side
            relink = True
    for cmd, proc in jobs:
        if proc.wait() != 0:
            raise subprocess.CalledProcessError(proc.returncode, cmd)
    if relink or os.path.getmtime(OUTPUT) < max(os.path.getmtime(o) for o in objects):
        subprocess.run([nvcc, '-gencode', 'arch=compute_100a,code=sm_100a', '-shared', '-o', OUTPUT] + objects,
                       check=True)
    return OUTPUT
