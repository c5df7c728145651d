"""Builds libttl_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m tracktolearn_b200.build [--force]
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, 'csrc')
LIB_DIR = os.path.join(HERE, 'lib')
LIB_PATH = os.path.join(LIB_DIR, 'libttl_b200.so')
SOURCES = ['ttl_env.cu', 'ttl_actor.cu', 'ttl_oracle_net.cu', 'ttl_tractogram.cu', 'ttl_sh.cu', 'ttl_prof.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
              '-Xcompiler', '-fPIC']


def _nvcc():
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError('nvcc not found')


def _digest():
    h = hashlib.sha256()
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))]
    files.append(os.path.join(ROOT, 'include', 'ttl_b200.h'))
    for f in files:
        with open(f, 'rb') as fh:
            h.update(fh.read())
    h.update(' '.join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    os.makedirs(LIB_DIR, exist_ok=True)
    stamp = os.path.join(LIB_DIR, 'libttl_b200.sha256')
    digest = _digest()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp):
        with open(stamp) as f:
            if f.read().strip() == digest:
                return LIB_PATH
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(LIB_DIR, src.replace('.cu', '.o'))
        cmd = [_nvcc()] + NVCC_FLAGS + ['-I', os.path.join(ROOT, 'include'), '-I', CSRC, '-c',
                                       os.path.join(CSRC, src), '-o', obj]
        if verbose:
            cmd.insert(1, '-Xptxas')
            cmd.insert(2, '-v')
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(obj)
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out.decode())
        if p.returncode:
            raise RuntimeError('nvcc failed: ' + ' '.join(cmd))
    link = [_nvcc(), '-shared', '-gencode', 'arch=compute_100a,code=sm_100a', '-o', LIB_PATH] + objs
    subprocess.check_call(link)
    with open(stamp, 'w') as f:
        f.write(digest)
    return LIB_PATH


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
