"""Builds liboflib_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m oflibnumpy_b200.build [--force] [--verbose]

The .so has no Python / torch dependency: cudart is linked statically, symbols are the extern "C" entry points
declared in include/oflib_b200.h.
"""
import hashlib
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, 'csrc')
LIBDIR = os.path.join(PKG, 'lib')
LIBNAME = 'liboflib_b200.so'
SOURCES = ['runtime.cu', 'staging.cu', 'warp_t.cu', 'warp_t_ws.cu', 'combine3.cu', 'combine3_ws.cu', 'fieldgen.cu', 'elementwise.cu', 'forward_s.cu', 'combine12.cu', 'visualise.cu', 'track.cu', 'fit_matrix.cu', 'accumulate.cu', 'evaluate.cu']
NVCC_FLAGS = (['-DOFK_FWD_INSTR'] if os.environ.get('OFK_FWD_INSTR') else []) + ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17', '--use_fast_math=false',
              '-Xcompiler', '-fPIC', '-Xcompiler', '-fvisibility=hidden', '-fmad=true']


def lib_path():
    return os.path.join(LIBDIR, LIBNAME)


def _nvcc():
    for cand in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def _digest():
    h = hashlib.sha256()
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))]
    files.append(os.path.join(os.path.dirname(PKG), 'include', 'oflib_b200.h'))
    files.append(os.path.abspath(__file__))
    for f in files:
        with open(f, 'rb') as fh:
            h.update(fh.read())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile every .cu for sm_100a and link the shared library; skipped when sources are unchanged."""
    os.makedirs(LIBDIR, exist_ok=True)
    stamp = os.path.join(LIBDIR, 'build.sha256')
    dig = _digest()
    if not force and os.path.exists(lib_path()) and os.path.exists(stamp) and open(stamp).read().strip() == dig:
        return lib_path()
    nvcc = _nvcc()
    flags = [f for f in NVCC_FLAGS if f != '--use_fast_math=false']
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(LIBDIR, src.replace('.cu', '.o'))
        cmd = [nvcc] + flags + (['-Xptxas', '-v'] if verbose else []) + ['-c', os.path.join(CSRC, src), '-o', obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            failed = True
            sys.stderr.write("nvcc failed on %s\n" % src)
    if failed:
        raise RuntimeError("oflib_b200 build failed")
    cmd = [nvcc, '-shared', '-gencode', 'arch=compute_100a,code=sm_100a', '-o', lib_path()] + objs
    subprocess.check_call(cmd)
    with open(stamp, 'w') as fh:
        fh.write(dig)
    return lib_path()


if __name__ == '__main__':
    p = build(force='--force' in sys.argv, verbose='--verbose' in sys.argv)
    print(p)
