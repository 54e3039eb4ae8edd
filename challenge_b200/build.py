"""In-tree build of libiris.so (nvcc, sm_100a only).  No GPU is needed to build.

``python -m challenge_b200.build`` or ``__graft_entry__.build()``.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
OBJ = os.path.join(HERE, 'build')
LIB = os.path.join(HERE, 'libiris.so')
SOURCES = ['iris_abi.cu', 'k_fused.cu', 'k_post.cu', 'k_bank.cu', 'k_labels.cu', 'k_metrics.cu',
           'k_ops.cu', 'k_eval.cu', 'k_spec.cu', 'k_resample.cu', 'iris_ops_abi.cu', 'iris_step.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
              '--expt-relaxed-constexpr', '-Xcompiler', '-fPIC']


def _nvcc():
    for cand in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError('nvcc not found; libiris.so cannot be built')


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, lib=None, obj_dir=None):
    """``lib`` / ``obj_dir``: build elsewhere than in-tree (e.g. another revision, loaded with IRIS_LIB)."""
    nvcc = _nvcc()
    global OBJ, LIB
    if lib:
        LIB = lib
    if obj_dir:
        OBJ = obj_dir
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cuh', '.h'))]
    headers.append(os.path.join(HERE, '..', 'include', 'iris.h'))
    objs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        if not os.path.exists(s):
            raise RuntimeError('listed CUDA source %s is missing' % s)
        o = os.path.join(OBJ, src.replace('.cu', '.o'))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            cmd = [nvcc] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-c', s, '-o', o]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if verbose or r.returncode:
                sys.stderr.write(r.stdout + r.stderr)
            if r.returncode:
                raise RuntimeError('nvcc failed on %s' % src)
    if force or _stale(LIB, objs):
        cmd = [nvcc, '-shared', '-o', LIB] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a', '-ldl']
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError('link of libiris.so failed')
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
