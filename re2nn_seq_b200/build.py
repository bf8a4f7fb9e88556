"""In-tree build of libre2nn_b200.so (sm_100a only).  Used by __graft_entry__.build()."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libre2nn_b200.so')
SOURCES = ['recurrence.cu', 'crf.cu', 'onehot.cu', 'backward.cu', 'maxprod.cu', 'fst.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '--use_fast_math=false', '-Xcompiler', '-fPIC', '-Xptxas', '-v', '--split-compile', '0']


def _source_hash():
    """Content hash of every CUDA source + the public header (mtimes do not survive a snapshot copy)."""
    import hashlib
    h = hashlib.sha256()
    files = [os.path.join(HERE, '..', 'include', 're2nn_b200.h')]
    for root, _, names in os.walk(CSRC):
        files += [os.path.join(root, f) for f in names if f.endswith(('.cu', '.cuh', '.h'))]
    for f in sorted(files):
        h.update(os.path.basename(f).encode())
        h.update(open(f, 'rb').read())
    h.update(' '.join(NVCC_FLAGS + SOURCES).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    stamp = LIB + '.hash'
    digest = _source_hash()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read().strip() == digest:
        return LIB
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    flags = [f for f in NVCC_FLAGS if not f.startswith('--use_fast_math')]
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(CSRC, src[:-3] + '.o')
        objs.append(obj)
        cmd = [nvcc] + flags + ['-c', os.path.join(CSRC, src), '-o', obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            sys.stderr.write(out)
            raise RuntimeError('nvcc failed on %s' % src)
        if verbose:
            sys.stderr.write(out)
    cmd = [nvcc, '-shared', '-o', LIB] + objs + ['-lcudart_static', '-ldl', '-lrt', '-lpthread']
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError('link failed')
    with open(stamp, 'w') as f:
        f.write(digest)
    return LIB


TORCH_LIB = os.path.join(HERE, 'libre2nn_torch.so')


def build_torch_ops(force=False, verbose=False):
    """TORCH_LIBRARY(re2nn, ...) registration (csrc/torch_ops.cpp) -> libre2nn_torch.so next to libre2nn_b200.so."""
    import hashlib
    import torch
    from torch.utils import cpp_extension as ce
    src = os.path.join(CSRC, 'torch_ops.cpp')
    hdr = os.path.join(HERE, '..', 'include', 're2nn_b200.h')
    digest = hashlib.sha256(open(src, 'rb').read() + open(hdr, 'rb').read() + torch.__version__.encode()).hexdigest()
    stamp = TORCH_LIB + '.hash'
    if not force and os.path.exists(TORCH_LIB) and os.path.exists(stamp) and open(stamp).read().strip() == digest:
        return TORCH_LIB
    tlib = os.path.join(os.path.dirname(torch.__file__), 'lib')
    cuda_home = os.environ.get('CUDA_HOME', '/usr/local/cuda')
    cmd = [os.environ.get('CXX', 'g++'), '-O2', '-std=c++17', '-fPIC', '-shared', src, '-o', TORCH_LIB,
           '-D_GLIBCXX_USE_CXX11_ABI=%d' % int(torch._C._GLIBCXX_USE_CXX11_ABI)]
    for inc in ce.include_paths() + [os.path.join(cuda_home, 'include')]:
        cmd += ['-isystem', inc]
    cmd += ['-L' + tlib, '-L' + HERE, '-L' + os.path.join(cuda_home, 'lib64'), '-lc10', '-lc10_cuda', '-ltorch_cpu', '-ltorch_cuda',
            '-ltorch', '-lre2nn_b200', '-lcudart', '-Wl,-rpath,$ORIGIN', '-Wl,-rpath,' + tlib, '-Wl,--no-as-needed']
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError('torch_ops build failed')
    if verbose:
        sys.stderr.write(r.stdout)
    with open(stamp, 'w') as f:
        f.write(digest)
    return TORCH_LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
    print(build_torch_ops(force='--force' in sys.argv, verbose='-v' in sys.argv))
