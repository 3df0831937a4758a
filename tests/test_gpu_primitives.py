"""GPU: device primitives against numpy (stable sort order, scans), through the C ABI."""
import numpy as np
import pytest

from gpu_util import exclusive_scan, sort_pairs

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n", [0, 1, 2, 31, 33, 4095, 4096, 4097, 100_003, 1_500_000])
def test_exclusive_scan(n):
    rng = np.random.default_rng(n)
    a = rng.integers(0, 9, size=n).astype(np.uint32)
    out, total = exclusive_scan(a)
    want = np.concatenate([[0], np.cumsum(a.astype(np.uint64))[:-1]]) if n else np.empty(0)
    assert total == int(a.sum())
    assert (out == want.astype(np.uint32)).all()


@pytest.mark.parametrize("n", [0, 1, 7, 4096, 4097, 70_001, 1_200_000])
@pytest.mark.parametrize("bits", [(0, 64), (0, 19), (5, 37), (0, 3), (32, 45)])
def test_sort_pairs_u64_is_stable_lsd(n, bits):
    rng = np.random.default_rng(n + bits[1])
    keys = rng.integers(0, 1 << 63, size=n, dtype=np.uint64) ^ (rng.integers(0, 2, size=n, dtype=np.uint64) << np.uint64(63))
    if n > 10:
        keys[::3] = keys[0]  # many duplicates -> stability matters
    vals = np.arange(n, dtype=np.uint32)
    gk, gv = sort_pairs(keys, vals, *bits)
    mask = np.uint64(((1 << (bits[1] - bits[0])) - 1) << bits[0]) if bits[1] - bits[0] < 64 else np.uint64(2**64 - 1)
    order = np.argsort(keys & mask, kind="stable")
    assert (gv == vals[order]).all()
    assert (gk == keys[order]).all()


@pytest.mark.parametrize("n", [5, 4097, 300_000])
def test_sort_pairs_u32(n):
    rng = np.random.default_rng(n)
    keys = rng.integers(0, 1 << 32, size=n, dtype=np.uint64).astype(np.uint32)
    keys[::2] &= np.uint32(0xFF)  # skewed digits
    vals = rng.permutation(n).astype(np.uint32)
    gk, gv = sort_pairs(keys, vals, 0, 32)
    order = np.argsort(keys, kind="stable")
    assert (gk == keys[order]).all() and (gv == vals[order]).all()


def test_sort_all_equal_and_presorted():
    n = 50_000
    keys = np.full(n, 12345, dtype=np.uint64)
    vals = np.arange(n, dtype=np.uint32)
    gk, gv = sort_pairs(keys, vals, 0, 20)
    assert (gv == vals).all()
    keys = np.arange(n, dtype=np.uint64)
    gk, gv = sort_pairs(keys, vals[::-1].copy(), 0, 17)
    assert (gk == keys).all() and (gv == vals[::-1]).all()


def _coherent_keys(n, dtype, begin, end, seed):
    """keys as a LiDAR map gives them to the grid sort: 97 ascending runs over the whole key range [begin, end), each
    with local noise and repeats; the bits outside the range are random"""
    rng = np.random.default_rng(seed)
    width, runs = end - begin, 97
    i = np.arange(n, dtype=np.uint64)
    run_len = (n + runs - 1) // runs
    step = np.uint64(max((1 << width) // run_len, 1))
    key = (i % np.uint64(run_len)) * step + rng.integers(0, 8 * int(step), size=n, dtype=np.uint64)
    key += (i // np.uint64(run_len)) * np.uint64(0x9E3779B97F4A7C15)  # each run starts elsewhere (wraps mod 2^64)
    rep = np.arange(3, n, 5)
    key[rep] = key[rep - 1]  # repeated keys: stability matters
    if width < 64:
        key &= np.uint64((1 << width) - 1)
    total = 8 * np.dtype(dtype).itemsize
    outside = rng.integers(0, 1 << 64, size=n, dtype=np.uint64) & np.uint64(((1 << total) - 1) ^ (((1 << width) - 1) << begin))
    return ((key << np.uint64(begin)) | outside).astype(dtype)


@pytest.mark.parametrize("dtype,bits", [(np.uint32, (7, 29)), (np.uint32, (0, 23)), (np.uint32, (0, 32)),
                                        (np.uint64, (0, 33)), (np.uint64, (0, 64))])
def test_onesweep_sort_at_the_grid_key_widths(dtype, bits):
    """The grid sort runs on bits [fw, fw + key_bits): over 2^24 coherent keys the decoupled look-back spans > 4000 tiles."""
    n = (1 << 24) + 5
    keys = _coherent_keys(n, dtype, *bits, seed=bits[1])
    vals = np.arange(n, dtype=np.uint32)
    field = (keys.astype(np.uint64) >> np.uint64(bits[0]))
    if bits[1] - bits[0] < 64:
        field &= np.uint64((1 << (bits[1] - bits[0])) - 1)
    order = np.argsort(field, kind="stable")
    gk, gv = sort_pairs(keys, vals, *bits)
    assert (gv == vals[order]).all(), "values out of stable order"
    assert (gk == keys[order]).all(), "keys out of order"


@pytest.mark.parametrize("n", [4097, 250_000])
def test_legacy_sort_path_agrees_with_onesweep(n):
    """radix_sort_pairs uses onesweep below 2^30 pairs and the three-kernel LSD sort above it; the
    legacy path is kept honest by forcing it here."""
    from octreelib_b200 import _native as N
    rng = np.random.default_rng(n)
    keys = rng.integers(0, 1 << 40, size=n, dtype=np.uint64)
    keys[::5] = keys[1]
    vals = np.arange(n, dtype=np.uint32)
    a = sort_pairs(keys, vals, 0, 40)
    N.lib().ol_debug_force_legacy_sort(1)
    try:
        b = sort_pairs(keys, vals, 0, 40)
    finally:
        N.lib().ol_debug_force_legacy_sort(0)
    assert (a[0] == b[0]).all() and (a[1] == b[1]).all()
    order = np.argsort(keys, kind="stable")
    assert (a[1] == vals[order]).all()
