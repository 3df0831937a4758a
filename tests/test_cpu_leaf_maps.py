"""CPU: the declarative leaf maps (octreelib_b200/leaf_maps.py) as plain callables - bit-equal to the functions the
reference fixture tests/golden/map_leaf_points_edge4.npz was recorded with - their argument checks, and the numpy
behaviour the GPU kernels rest on (csrc/leaf_maps.cuh)."""
import numpy as np
import pytest

from octreelib_b200 import leaf_maps
from octreelib_b200.leaf_maps import Centroid, FirstPoints, Shrink


def golden_shrink(cloud, factor=0.5):  # tests/golden/make_map_leaf_points.py
    c = cloud.mean(axis=0)
    return c + factor * (cloud - c)


def golden_centroid(cloud):
    return cloud.mean(axis=0, keepdims=True)


def _clouds():
    rng = np.random.default_rng(5)
    for n in (1, 2, 3, 7, 100, 4097):
        for offset in (0.0, 1e3, -1e5, 1e5):
            for scale in (1e-3, 1.0, 50.0):
                yield rng.normal(size=(n, 3)) * scale + offset


def _bits_equal(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and (a.view(np.uint64) == b.view(np.uint64)).all()


def test_objects_equal_the_golden_functions_bit_for_bit():
    for cloud in _clouds():
        assert _bits_equal(Centroid()(cloud), golden_centroid(cloud))
        for f in (0.5, 0.0, 1.0, 0.25, 1.0 - 2.0 ** -52):
            assert _bits_equal(Shrink(f)(cloud), golden_shrink(cloud, f))
        for k in (0, 1, 3, 10 ** 9):
            assert _bits_equal(FirstPoints(k)(cloud), cloud[:k])


def test_argument_validation():
    for bad in (float("nan"), float("inf"), -float("inf"), "0.5", None, True):
        with pytest.raises(ValueError):
            Shrink(bad)
    assert Shrink(1).factor == 1.0 and Shrink(np.float32(0.5)).factor == 0.5
    with pytest.raises(ValueError):
        FirstPoints(-1)
    for bad in (True, False, 1.0, 2.5, "3", None):
        with pytest.raises(TypeError):
            FirstPoints(bad)
    assert FirstPoints(np.int64(4)).k == 4 and FirstPoints(0).k == 0


def test_native_arguments():
    from octreelib_b200 import _native as N

    assert (Centroid().op, Shrink(0.5).op, FirstPoints(2).op) == (N.OL_MAP_CENTROID, N.OL_MAP_SHRINK, N.OL_MAP_FIRST)
    assert Shrink(-2.0).param == -2.0 and FirstPoints(7).param == 7.0 and FirstPoints(1 << 70).param == float(1 << 53)
    assert {"Centroid", "Shrink", "FirstPoints"} <= set(leaf_maps.__all__)


def test_the_host_dispatch_keeps_other_callables_and_subclasses_on_the_host_path():
    from octreelib_b200._host import ForestHost

    class MyCentroid(Centroid):
        def __call__(self, cloud):
            return cloud[:1]

    assert set(ForestHost._DEVICE_LEAF_MAPS) == {Centroid, Shrink, FirstPoints}
    assert type(MyCentroid()) not in ForestHost._DEVICE_LEAF_MAPS


def _sequential_mean(a):
    s = np.zeros(3)
    for row in a:
        s = s + row
    return s / np.float64(len(a))


@pytest.mark.parametrize("n", list(range(1, 301)) + [4097, 100001])
def test_numpy_mean_along_axis_0_is_a_sequential_row_sum(n):
    """PREMISE of csrc/leaf_maps.cuh (leaf_mean_kernel): for a C-contiguous (n, 3) float64 array, numpy's
    mean(axis=0) is the sum of the rows in order, starting from +0.0, divided once by float64(n) - no pairwise summation
    along axis 0.  If this test fails, the installed numpy changed that, and the GPU Centroid / Shrink no longer equal the
    host path bit for bit: the kernel's summation order has to follow numpy's new one."""
    rng = np.random.default_rng(n)
    for offset in (0.0, 1e5, -3.7e4):
        a = np.ascontiguousarray(rng.normal(size=(n, 3)) * 10.0 ** rng.uniform(-3, 3) + offset)
        assert _bits_equal(a.mean(axis=0), _sequential_mean(a)), (n, offset)
        assert _bits_equal(a.mean(axis=0, keepdims=True)[0], _sequential_mean(a))
