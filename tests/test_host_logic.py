"""CPU-only tests of the host-side logic of the package (validators, dtype promotion table, sharding, slicing)."""
import os

import numpy as np
import pytest

from oflibnumpy_b200 import _lib, _ops
from oflibnumpy_b200.batch import shard_range
from oflibnumpy_b200.flow import _as_window
from oflibnumpy_b200.ops import matrix_from_transforms, matrix_from_transform, threshold_vectors
from oflibnumpy_b200.validation import get_valid_ref, get_valid_padding, validate_shape, validate_flow_array, \
    validate_transform_list
from oracle import flowref as R


def test_get_valid_ref():
    assert get_valid_ref(None) == 't' and get_valid_ref('s') == 's' and get_valid_ref('t') == 't'
    with pytest.raises(TypeError):
        get_valid_ref(0)
    with pytest.raises(ValueError):
        get_valid_ref('test')


def test_get_valid_padding():
    assert get_valid_padding([1, 2, 3, 4]) == [1, 2, 3, 4]
    with pytest.raises(TypeError):
        get_valid_padding(100)
    with pytest.raises(ValueError):
        get_valid_padding([10, 20, 30, 40, 50])
    with pytest.raises(ValueError):
        get_valid_padding([10., 20, 30, 40])
    with pytest.raises(ValueError):
        get_valid_padding([-10, 10, 10, 10])


def test_validate_shape_and_flow_array():
    validate_shape([10, 20])
    with pytest.raises(TypeError):
        validate_shape('test')
    with pytest.raises(ValueError):
        validate_shape([10, 10, 10])
    with pytest.raises(ValueError):
        validate_shape([-1, 10])
    with pytest.raises(ValueError):
        validate_shape([10., 10])
    f = np.zeros((10, 10, 2))
    assert validate_flow_array(f).dtype == np.float32
    with pytest.raises(TypeError):
        validate_flow_array('test')
    with pytest.raises(ValueError):
        validate_flow_array(np.zeros((10, 10)))
    with pytest.raises(ValueError):
        validate_flow_array(np.zeros((10, 10, 3)))
    for bad in (np.nan, np.inf, -np.inf):
        g = f.copy()
        g[0, 0, 0] = bad
        with pytest.raises(ValueError):
            validate_flow_array(g)


def test_validate_transform_list():
    validate_transform_list([['translation', 1, 2], ['rotation', 1, 2, 3.5], ['scaling', 0, 0, 2]])
    with pytest.raises(TypeError):
        validate_transform_list('test')
    with pytest.raises(TypeError):
        validate_transform_list(['test'])
    with pytest.raises(ValueError):
        validate_transform_list([['translation']])
    with pytest.raises(ValueError):
        validate_transform_list([['test', 1, 2]])
    with pytest.raises(ValueError):
        validate_transform_list([['translation', 1]])
    with pytest.raises(ValueError):
        validate_transform_list([['rotation', 1, 2]])
    with pytest.raises(ValueError):
        validate_transform_list([['scaling', 1, 2, 'x']])


def test_matrices_match_oracle_and_reference_known_answers():
    # known answers "calculated manually" in the reference's tests (tests/test_utils.py:92-171)
    np.testing.assert_allclose(matrix_from_transform('rotation', [0, 0, 90]), [[0, 1, 0], [-1, 0, 0], [0, 0, 1]],
                               atol=1e-12)
    np.testing.assert_allclose(matrix_from_transform('scaling', [0, 0, 2]), np.diag([2, 2, 1]), atol=0)
    np.testing.assert_allclose(matrix_from_transform('translation', [10, 20]), [[1, 0, 10], [0, 1, 20], [0, 0, 1]])
    tl = [['translation', -100, -100], ['rotation', 0, 0, 30], ['translation', 100, 100], ['scaling', 3, 7, 0.8]]
    np.testing.assert_array_equal(matrix_from_transforms(tl), R.matrix_from_transforms(tl))


def test_promotion_table():
    assert _ops.promoted_rule(np.uint8, False) == (_lib.ARITH_RINT, _lib.RULE_GT_HALF)     # uint8 || int8 -> int16
    assert _ops.promoted_rule(np.uint8, True) == (_lib.ARITH_NATIVE, _lib.RULE_GE_HALF)    # uint8 || bool -> uint8
    assert _ops.promoted_rule(np.int16, False)[1] == _lib.RULE_GT_HALF
    assert _ops.promoted_rule(np.float32, True) == (_lib.ARITH_NATIVE, _lib.RULE_STRICT)
    assert _ops.promoted_rule(np.float64, False) == (_lib.ARITH_NATIVE, _lib.RULE_STRICT)
    with pytest.raises(TypeError):
        _ops.promoted_rule(np.uint16, False)
    with pytest.raises(TypeError):
        _ops.promoted_rule(np.int32, True)
    # the table is numpy's promotion
    for dt, mask_dt in ((np.uint8, np.int8), (np.uint8, np.bool_), (np.int16, np.int8), (np.uint16, np.bool_)):
        cat = np.concatenate((np.zeros((1, 1, 1), dt), np.zeros((1, 1, 1), mask_dt)), -1).dtype
        arith, _ = _ops.promoted_rule(dt, mask_dt == np.bool_)
        assert (cat == np.int16) == (arith == _lib.ARITH_RINT or dt == np.int16)


def test_shard_range_covers_batch():
    for n in (0, 1, 7, 64, 255, 256):
        for world in (1, 2, 3, 4, 8):
            spans = [shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1


def test_window_detection():
    assert _as_window((slice(2, 5), slice(1, 4)), (10, 10)) == (2, 1, 3, 3)
    assert _as_window(slice(3, None), (10, 8)) == (3, 0, 7, 8)
    assert _as_window((slice(0, 10, 2), slice(None)), (10, 10)) is None
    assert _as_window(3, (10, 10)) is None
    assert _as_window((slice(5, 5),), (10, 10)) is None


def test_threshold_vectors_reference_golden():
    """tests/test_utils.py:322-335 of the reference."""
    vecs = np.zeros((10, 1, 2))
    vecs[0, 0, 0] = -1e-5
    vecs[1, 0, 0] = 1e-4
    vecs[2, 0, 0] = -1e-3
    vecs[3, 0, 0] = 1
    th = threshold_vectors(vecs, threshold=1e-3)
    np.testing.assert_array_equal(th[:4, 0, 0], [0, 0, -1e-3, 1])
    th = threshold_vectors(vecs, threshold=1e-4)
    np.testing.assert_array_equal(th[:4, 0, 0], [0, 1e-4, -1e-3, 1])
    th = threshold_vectors(vecs, threshold=1e-5)
    np.testing.assert_array_equal(th[:4, 0, 0], [-1e-5, 1e-4, -1e-3, 1])


def test_host_view_tracks_in_place_edits():
    """Flow.vecs / Flow.mask hand out read-only views that report the in-place edits numpy can make from Python (item
    assignment, ufuncs with out= / augmented assignment) and make every other writer fail loudly."""
    from oflibnumpy_b200.flow import _tracked_view
    d = [False]
    a = _tracked_view(np.arange(12, dtype=np.float32).reshape(3, 4), d)
    assert isinstance(a, np.ndarray) and not a.flags.writeable
    b = a * 2
    assert type(b) is np.ndarray and b.flags.writeable and not d[0]
    assert float(a.sum()) == 66.0 and not d[0]
    a[0, 0] = 5
    assert d[0] and a[0, 0] == 5 and not a.flags.writeable
    d[0] = False
    a[a > 6] = 0                                      # the reference's documented idiom (docs/usage.rst:316)
    assert d[0]
    d[0] = False
    a += 1
    assert d[0] and a[0, 0] == 6
    d[0] = False
    v = a[1:, :2]                                     # views share buffer and tracking
    v[...] = 9
    assert d[0] and a[1, 0] == 9
    d[0] = False
    np.multiply(a, 2, out=a)
    assert d[0]
    d[0] = False
    for writer in (lambda: a.fill(0), lambda: np.copyto(a, 1), lambda: a.sort()):
        with pytest.raises(ValueError):
            writer()
    assert not d[0]
    m = _tracked_view(np.ones((3, 4), bool), d)
    m[:, 2:] = False                                  # tests/test_flow_class.py:580 of the reference
    assert d[0] and not m[:, 2:].any()
    c = a.copy()
    c[0, 0] = -1                                      # copies are ordinary arrays
    assert a[0, 0] != -1


def test_dataset_loaders_match_reference():
    """Host file readers (oflibnumpy_b200/io.py) against outputs of the reference's loaders on the committed sample
    files (tests/golden/files, written and read back by oracle/gen_golden.py with the unmodified reference)."""
    from conftest import load_golden
    from oflibnumpy_b200 import io
    g = load_golden('datasets')
    files = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'files')
    np.testing.assert_array_equal(io.load_kitti(os.path.join(files, 'kitti_sample.png')), g['out_load_kitti'])
    np.testing.assert_array_equal(io.load_sintel(os.path.join(files, 'sintel_sample.flo')), g['out_load_sintel'])
    np.testing.assert_array_equal(io.load_sintel_mask(os.path.join(files, 'sintel_invalid.png')),
                                  g['out_load_sintel_mask'])
    raw = io.read_kitti_raw(os.path.join(files, 'kitti_sample.png'))
    assert raw.dtype == np.uint16 and raw.shape == g['out_load_kitti'].shape
    with pytest.raises(ValueError):
        io.load_kitti(os.path.join(files, 'does_not_exist.png'))
    with pytest.raises(ValueError):
        io.load_sintel(os.path.join(files, 'kitti_sample.png'))


def test_host_side_presentation_api_is_present():
    """matrix / visualise_arrows / show* and their ndarray wrappers exist with the reference's signatures (they delegate
    to the reference package on a host copy: SURVEY section 2 rows 19-21, not on the hot path)."""
    import inspect
    import oflibnumpy_b200 as of
    sigs = {'matrix': ['self', 'dof', 'method', 'masked'],
            'visualise_arrows': ['self', 'grid_dist', 'img', 'scaling', 'show_mask', 'show_mask_borders', 'colour',
                                 'thickness'],
            'show': ['self', 'wait', 'show_mask', 'show_mask_borders'],
            'show_arrows': ['self', 'wait', 'grid_dist', 'img', 'scaling', 'show_mask', 'show_mask_borders', 'colour']}
    for name, args in sigs.items():
        assert list(inspect.signature(getattr(of.Flow, name)).parameters) == args, name
    for name in ('visualise_flow', 'get_flow_matrix', 'visualise_flow_arrows', 'show_flow', 'show_flow_arrows',
                 'visualise_definition'):
        assert callable(getattr(of, name)), name
