"""CPU-only checks of the drop-in boundary: the C-ABI library builds, loads, and exports every symbol that
include/oflib_b200.h declares; the ctypes table matches the header; calls fail loudly without a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, 'include', 'oflib_b200.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(of[kh]_\w+)\s*\(', src)))


@pytest.fixture(scope='module')
def lib_path():
    from oflibnumpy_b200 import build
    return build.build()


def test_header_declares_the_hot_path():
    names = header_functions()
    for must in ('ofk_warp_t', 'ofk_combine3', 'ofk_forward_s', 'ofk_from_matrix', 'ofk_valid_geom_t',
                 'ofk_nonzero_flags', 'ofk_addsub', 'ofk_pad', 'ofh_warp_t', 'ofh_combine3', 'ofk_last_error'):
        assert must in names


def test_library_exports_every_declared_symbol(lib_path):
    lib = ctypes.CDLL(lib_path)
    missing = [n for n in header_functions() if not hasattr(lib, n)]
    assert not missing, "declared in the header but not exported: {}".format(missing)


def test_ctypes_table_matches_header(lib_path):
    from oflibnumpy_b200 import _lib
    assert _lib.symbols() == header_functions()
    lib = _lib.load()
    assert lib.ofk_version() == 100


def test_argument_errors_do_not_need_a_gpu(lib_path):
    from oflibnumpy_b200 import _lib
    with pytest.raises(_lib.OflibCudaError, match="flow is NULL"):
        _lib.call('ofk_warp_t', None, 0, 0, 0, None, -1.0, None, None, None, None, 0, 1, 4, 4, 4, 4, 0, 0, 1, None)
    with pytest.raises(_lib.OflibCudaError, match="ref must be"):
        _lib.call('ofk_combine3', 16, None, 16, None, ord('x'), 0.0, 16, 16, None, 1, 4, 4, None)
    # host-buffer entry points: checked before the ring or a device is touched
    with pytest.raises(_lib.OflibCudaError, match="ofh_warp_t: bad arguments"):
        _lib.call('ofh_warp_t', 16, 0, 1, 0, None, -1.0, None, None, 16, None, 0, 1, 4, 4, 0)
    with pytest.raises(_lib.OflibCudaError, match="ofh_combine3: bad arguments"):
        _lib.call('ofh_combine3', 16, None, None, None, ord('t'), 0.0, 16, 16, None, 1, 4, 4, 0)
    with pytest.raises(_lib.OflibCudaError, match="ofh_apply_combine3: ref must be"):
        _lib.call('ofh_apply_combine3', 16, 0, 1, 0, 0, 16, None, 16, None, ord('x'), 0.0, 16, None, 16, 16, None, 1,
                  4, 4, 0)


def test_no_cpu_fallback_without_gpu(lib_path):
    import oflibnumpy_b200 as of
    if of.device.device_count() > 0:
        pytest.skip("a GPU is visible")
    with pytest.raises(of.OflibCudaError):
        of.Flow(np.zeros((4, 4, 2), np.float32))
    with pytest.raises(of.OflibCudaError):
        of.apply_flow(np.ones((4, 4, 2), np.float32), np.zeros((4, 4), np.uint8), 't')


def test_product_does_not_import_oracle():
    """The package must never route through the CPU oracle."""
    pkg = os.path.join(ROOT, 'oflibnumpy_b200')
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle\b', text, flags=re.M), f
                assert 'flowref' not in text and 'remap_q32' not in text, f


def test_oracle_stays_inside_tests_smoke_and_bench_cpu_legs():
    """Nothing under tools/ or examples/ touches the oracle; bench.py imports it only inside its CPU-baseline /
    reference-arm functions; taking workload parameters from tests/golden_inputs.py does not import it either."""
    import subprocess
    import sys
    for sub in ('tools', 'examples'):
        for dirpath, _, files in os.walk(os.path.join(ROOT, sub)):
            for f in files:
                if f.endswith(('.py', '.sh', '.c', '.cu')):
                    text = open(os.path.join(dirpath, f)).read()
                    assert not re.search(r'^\s*(from|import)\s+oracle\b', text, flags=re.M), f
                    assert 'flowref' not in text, f
    bench = open(os.path.join(ROOT, 'bench.py')).read()
    for m in re.finditer(r'^(\s*)(from|import)\s+oracle\b', bench, flags=re.M):
        assert len(m.group(1)) > 0, "bench.py must import the oracle inside its CPU legs only"
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import golden_inputs as gi\n"
            "gi.cfg4_transforms(3)\n"
            "assert not any(m.startswith('oracle') for m in sys.modules), 'oracle imported'\n"
            "print('ok')\n") % (ROOT, os.path.join(ROOT, 'tests'))
    res = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0 and 'ok' in res.stdout, res.stdout + res.stderr


def _build_c_example():
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, 'examples', 'abi_example')
    cmd = ['gcc', '-O2', '-std=c99', '-Wall', '-I' + os.path.join(root, 'include'), os.path.join(root, 'examples', 'abi_example.c'),
           '-L' + os.path.join(root, 'oflibnumpy_b200', 'lib'), '-loflib_b200',
           '-Wl,-rpath,' + os.path.join(root, 'oflibnumpy_b200', 'lib'), '-lm', '-o', exe]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    return exe


def test_header_is_plain_c_and_links():
    """include/oflib_b200.h compiles as C99 and examples/abi_example.c links against the library without Python."""
    _build_c_example()


@pytest.mark.gpu
def test_c_example_runs():
    """The plain-C host program (host-buffer entry points, TMA kernels) checks its own invariants on the GPU."""
    import subprocess
    res = subprocess.run([_build_c_example()], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout + res.stderr
    assert 'abi example ok' in res.stdout
