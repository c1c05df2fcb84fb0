"""CPU tests of the top-k selection's boundary: argument errors and their codes (checked before any device work), the
Python layer's ValueErrors, the workspace size, and the loud failure without a GPU (there is no CPU fallback)."""
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


def _soa(keys, key_type, n_rows, row_len, k, out_keys, out_index, n_payloads=0, payloads=None, sizes=None, out_payloads=None):
    return S.lib().b200sort_topk_soa(keys, key_type, n_rows, row_len, k, 1, n_payloads, payloads, sizes, out_keys, out_index,
                                     out_payloads, None, None, 0)


def test_argument_errors():
    L = S.lib()
    k = np.arange(1000, dtype=np.float32)
    ok, oi = np.zeros(40, np.float32), np.zeros(40, np.int64)
    K, OK, OI = k.ctypes.data, ok.ctypes.data, oi.ctypes.data
    assert _soa(K, 42, 4, 250, 10, OK, OI) == -1  # unknown key type
    assert b"key type" in L.b200sort_last_error()
    for n_rows, row_len, kk in ((-1, 250, 10), (4, -1, 10), (4, 250, -1)):
        assert _soa(K, 8, n_rows, row_len, kk, OK, OI) == -1
    assert _soa(K, 8, 4, 250, 251, OK, OI) == -1  # k > row_len
    assert b"exceeds" in L.b200sort_last_error()
    assert _soa(K, 8, 2**31, 1, 1, OK, OI) == -1  # too many rows
    assert _soa(K, 8, 2**31 - 1, 2**40, 1, OK, OI) == -1  # n_rows * row_len overflows
    assert b"overflows" in L.b200sort_last_error()
    # NULL input, key output or index when k > 0
    assert _soa(None, 8, 4, 250, 10, OK, OI) == -1
    assert _soa(K, 8, 4, 250, 10, None, OI) == -1
    assert _soa(K, 8, 4, 250, 10, OK, None) == -1
    assert b"out_index" in L.b200sort_last_error()
    # an output overlapping an input
    assert _soa(K, 8, 4, 250, 10, K + 400, OI) == -1
    assert _soa(K, 8, 4, 250, 10, OK, K) == -1
    assert b"overlaps" in L.b200sort_last_error()
    # payload shapes: element size 65, 64 streams
    p = np.zeros(1000, np.uint8)
    ptrs, outs = (ctypes.c_void_p * 64)(*([p.ctypes.data] * 64)), (ctypes.c_void_p * 64)()
    assert _soa(K, 8, 4, 250, 10, OK, OI, 1, ptrs, (ctypes.c_uint32 * 1)(65), outs) == -2
    assert _soa(K, 8, 4, 250, 10, OK, OI, 64, ptrs, (ctypes.c_uint32 * 64)(*([1] * 64)), outs) == -2
    # a NULL output payload
    assert _soa(K, 8, 4, 250, 10, OK, OI, 1, ptrs, (ctypes.c_uint32 * 1)(1), None) == -1
    # two outputs overlapping each other: the key output inside out_index, an output payload inside the key output
    assert _soa(K, 8, 4, 250, 10, OI + 8, OI) == -1
    assert b"two outputs overlap" in L.b200sort_last_error()
    assert _soa(K, 8, 4, 250, 10, OK, OI, 1, ptrs, (ctypes.c_uint32 * 1)(1), (ctypes.c_void_p * 1)(OK + 4)) == -1
    assert b"two outputs overlap" in L.b200sort_last_error()
    # AoS record sizes: 24 (not a power of two), 4 for an 8-byte key
    for rb in (24, 4):
        assert L.b200sort_topk_aos(K, 6, rb, 1, 10, 1, 1, OK, OI, None, None, 0) == -3
    # k == 0 and n_rows == 0 are no-ops, even with NULL arrays
    assert _soa(None, 8, 4, 250, 0, None, None) == 0
    assert _soa(None, 8, 0, 250, 10, None, None) == 0
    assert L.b200sort_topk_aos(None, 6, 16, 0, 10, 1, 1, None, None, None, None, 0) == 0
    assert (ok == 0).all() and (oi == 0).all() and (k == np.arange(1000, dtype=np.float32)).all()


def test_python_value_errors():
    k = np.arange(12, dtype=np.float32)
    with pytest.raises(ValueError):
        S.topk(k, 13)
    with pytest.raises(ValueError):
        S.topk(k, -1)
    with pytest.raises(ValueError):
        S.topk(k.reshape(2, 2, 3), 1)
    with pytest.raises(ValueError):
        S.topk(k.reshape(3, 4), 2, np.zeros((4, 3), np.int64))  # payload leading shape differs
    with pytest.raises(ValueError):
        S.topk_combined(np.zeros((4, 5, 16), np.uint8), np.int64, 6)
    with pytest.raises(ValueError):
        S.topk_combined(np.zeros(16, np.uint8), np.int64, 1)
    with pytest.raises(TypeError):
        S.topk(k.astype(np.float16), 1)


def test_workspace_bytes():
    for dt, pays, rb in ((np.float32, [8], 0), (np.uint64, [8, 4], 0), (np.uint8, [], 0), (np.int16, [], 16)):
        sizes = [S.topk_workspace_bytes(dt, 64, L, 50, pays, rb) for L in (10**3, 10**4, 10**5, 10**6)]
        assert all(a < b for a, b in zip(sizes, sizes[1:])), (dt, sizes)
        for n_rows, row_len, k in ((64, 128256, 50), (1, 2**20, 1000), (3, 100_003, 40_000), (7, 1000, 1000)):
            w = S.topk_workspace_bytes(dt, n_rows, row_len, k, pays, rb)
            assert w % 256 == 0
            assert w >= S.segmented_workspace_bytes(dt, n_rows * k, n_rows, [8])
    assert S.lib().b200sort_topk_workspace_bytes(42, 1, 10, 1, 0, None, 0) == 0
    assert S.topk_workspace_bytes(np.float32, 1, 10, 11) == 0


@pytest.mark.skipif(_has_cuda(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback():
    k = np.array([3, 1, 2, 9, 8, 7], dtype=np.int32)
    with pytest.raises(S.B200SortError) as ei:
        S.topk(k, 2)
    assert ei.value.code == -5 and "no CPU fallback" in str(ei.value)
    with pytest.raises(S.B200SortError) as ei:
        S.topk_combined(np.zeros((4, 8), np.uint8), np.int64, 2)
    assert ei.value.code == -5
    assert k.tolist() == [3, 1, 2, 9, 8, 7]
