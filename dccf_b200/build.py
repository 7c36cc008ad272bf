"""Build the C-ABI library `dccf_b200/libdccf_b200.so` from `dccf_b200/csrc/*.cu` with nvcc for sm_100a.

In-tree build (the .so travels to the GPU box with the repo snapshot; it is git-ignored).  nvcc
cross-compiles without a GPU.  Usage: `python -m dccf_b200.build [--force] [--verbose]`.
"""
import concurrent.futures
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
INCLUDE = os.path.join(os.path.dirname(HERE), 'include')
OBJ_DIR = os.path.join(HERE, 'build')
LIB_PATH = os.path.join(HERE, 'libdccf_b200.so')

NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC', '-Xptxas', '-v']


def _nvcc():
    for cand in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError('nvcc not found: the DCCF B200 kernels cannot be built')


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith('.cu'))


def _digest():
    h = hashlib.sha256()
    deps = sources() + sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith('.cuh'))
    deps += [os.path.join(INCLUDE, 'dccf_b200.h')]
    for path in deps:
        h.update(path.encode())
        with open(path, 'rb') as f:
            h.update(f.read())
    h.update(' '.join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile every .cu and link the shared library; returns its path.  Skips when up to date."""
    stamp = os.path.join(OBJ_DIR, 'stamp')
    digest = _digest()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp) and open(stamp).read() == digest:
        return LIB_PATH
    nvcc = _nvcc()
    os.makedirs(OBJ_DIR, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(OBJ_DIR, os.path.basename(src)[:-3] + '.o')
        cmd = [nvcc] + NVCC_FLAGS + ['-I', INCLUDE, '-c', src, '-o', obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError('nvcc failed for %s:\n%s\n%s' % (src, r.stdout, r.stderr))
        return obj, r.stderr

    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        results = list(ex.map(compile_one, sources()))
    objs = [o for o, _ in results]
    log = '\n'.join(l for _, l in results)
    with open(os.path.join(OBJ_DIR, 'ptxas.log'), 'w') as f:
        f.write(log)
    if verbose:
        print(log)
    cmd = [nvcc, '-shared', '-o', LIB_PATH] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a']
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError('link failed:\n%s\n%s' % (r.stdout, r.stderr))
    with open(stamp, 'w') as f:
        f.write(digest)
    return LIB_PATH


if __name__ == '__main__':
    path = build(force='--force' in sys.argv, verbose='--verbose' in sys.argv)
    print(path)
