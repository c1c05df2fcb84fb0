"""CPU tests of the segmented sort's boundary: argument errors and their codes, the workspace size, and the loud
failure without a GPU (there is no CPU fallback)."""
import ctypes

import numpy as np
import pytest

import simd_radix_sort_b200 as S


def _has_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def _offsets(*v):
    return np.array(v, dtype=np.int64)


def test_argument_errors():
    L = S.lib()
    k = np.arange(10, dtype=np.uint32)
    o = _offsets(0, 5, 10)
    # unknown key type
    assert L.b200sort_sort_segmented_soa(k.ctypes.data, 42, 10, 2, o.ctypes.data, 1, 0, None, None, None, None, 0) == -1
    # negative or too many segments
    assert L.b200sort_sort_segmented_soa(k.ctypes.data, 4, 10, -1, o.ctypes.data, 1, 0, None, None, None, None, 0) == -1
    assert L.b200sort_sort_segmented_soa(k.ctypes.data, 4, 10, 2**31, o.ctypes.data, 1, 0, None, None, None, None, 0) == -1
    assert b"segments" in L.b200sort_last_error()
    # NULL offsets
    assert L.b200sort_sort_segmented_soa(k.ctypes.data, 4, 10, 2, None, 1, 0, None, None, None, None, 0) == -1
    assert b"offsets" in L.b200sort_last_error()
    # payload element size 65
    sizes = (ctypes.c_uint32 * 1)(65)
    ptrs = (ctypes.c_void_p * 1)(k.ctypes.data)
    assert L.b200sort_sort_segmented_soa(k.ctypes.data, 4, 10, 2, o.ctypes.data, 1, 1, ptrs, sizes, None, None, 0) == -2
    # AoS record size 24 (not a power of two)
    assert L.b200sort_sort_segmented_aos(k.ctypes.data, 6, 24, 1, 1, _offsets(0, 1).ctypes.data, 1, None, None, 0) == -3
    # no segments: nothing to do
    assert L.b200sort_sort_segmented_soa(k.ctypes.data, 4, 10, 0, o.ctypes.data, 1, 0, None, None, None, None, 0) == 0
    assert k.tolist() == list(range(10))
    # the Python layer: offsets must be int64 with at least one value
    with pytest.raises(TypeError):
        S.sort_segmented(o.astype(np.int32), k)
    with pytest.raises(ValueError):
        S.sort_segmented(np.zeros(0, np.int64), k)
    with pytest.raises(ValueError):
        S.sort_rows(k)


def test_workspace_bytes_grows_with_num_and_covers_the_composite_sort():
    for dt, pays, rb in ((np.uint32, [4], 0), (np.float32, [8, 1], 0), (np.uint64, [8], 0), (np.int16, [], 16)):
        sizes = [S.segmented_workspace_bytes(dt, n, 1000, pays, rb) for n in (10**4, 10**5, 10**6, 10**7)]
        assert all(a < b for a, b in zip(sizes, sizes[1:])), (dt, sizes)
        n = 10**6
        w = S.segmented_workspace_bytes(dt, n, 1000, pays, rb)
        if np.dtype(dt).itemsize <= 4:
            # the composite keys plus a whole-array sort of (composite key, payloads or records)
            whole = S.workspace_bytes(np.uint64, n, pays) if rb == 0 else S.workspace_bytes(np.uint64, n, [rb])
            assert w >= 8 * n + whole
        else:
            assert w >= S.workspace_bytes(dt, n, pays, rb)
        assert w % 256 == 0
    assert S.segmented_workspace_bytes(np.uint32, 0, 0) > 0
    assert S.lib().b200sort_segmented_workspace_bytes(42, 10, 1, 0, None, 0) == 0


@pytest.mark.skipif(_has_cuda(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback():
    k = np.array([3, 1, 2, 9, 8], dtype=np.int32)
    with pytest.raises(S.B200SortError) as ei:
        S.sort_segmented(_offsets(0, 3, 5), k)
    assert ei.value.code == -5 and "no CPU fallback" in str(ei.value)
    assert k.tolist() == [3, 1, 2, 9, 8]
    with pytest.raises(S.B200SortError) as ei:
        S.sort_rows(k[:4].reshape(2, 2))
    assert ei.value.code == -5
