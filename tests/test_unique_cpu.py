"""CPU tests of unique's boundary: argument errors and their codes (checked before any device work), the Python layer's
ValueErrors and TypeErrors, the workspace size, and the loud failure without a GPU (there is no CPU fallback)."""
import numpy as np
import pytest

import simd_radix_sort_b200 as S


def _has_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def _u(keys, key_type, num, out_keys, counts=None, inverse=None, n_unique=None, consecutive=0):
    return S.lib().b200sort_unique(keys, key_type, num, consecutive, out_keys, counts, inverse, n_unique, None, None, 0)


def test_argument_errors():
    L = S.lib()
    k = np.arange(1000, dtype=np.float32)
    ok, oc, oi, nu = np.zeros(1000, np.float32), np.zeros(1000, np.int64), np.zeros(1000, np.int64), np.zeros(1, np.int64)
    K, OK, OC, OI, NU = k.ctypes.data, ok.ctypes.data, oc.ctypes.data, oi.ctypes.data, nu.ctypes.data
    for consecutive in (0, 1):
        assert _u(K, 42, 1000, OK, OC, OI, NU, consecutive) == -1  # unknown key type
        assert b"key type" in L.b200sort_last_error()
        assert _u(K, 8, -1, OK, OC, OI, NU, consecutive) == -1
        assert b"negative" in L.b200sort_last_error()
        # NULL keys, out_keys or out_num_unique when num > 0
        assert _u(None, 8, 1000, OK, OC, OI, NU, consecutive) == -1
        assert _u(K, 8, 1000, None, OC, OI, NU, consecutive) == -1
        assert _u(K, 8, 1000, OK, OC, OI, None, consecutive) == -1
        assert b"out_num_unique" in L.b200sort_last_error()
        # misaligned: keys or out_keys to the key type, int64 outputs to 8 bytes
        assert _u(K + 2, 8, 999, OK, OC, OI, NU, consecutive) == -1
        assert _u(K, 8, 1000, OK + 1, OC, OI, NU, consecutive) == -1
        assert b"aligned" in L.b200sort_last_error()
        for bad in ((OC + 4, OI, NU), (OC, OI + 4, NU), (OC, OI, NU + 4)):
            assert _u(K, 8, 999, OK, *bad, consecutive=consecutive) == -1
            assert b"8-byte" in L.b200sort_last_error()
        # an output overlapping the input, or another output
        assert _u(K, 8, 1000, K + 400, OC, OI, NU, consecutive) == -1
        assert _u(K, 8, 1000, OK, K, OI, NU, consecutive) == -1
        assert b"overlaps the input" in L.b200sort_last_error()
        assert _u(K, 8, 1000, OK, OC, OC + 800, NU, consecutive) == -1
        assert _u(K, 8, 1000, OK, OC, OI, OI + 8 * 999, consecutive) == -1
        assert _u(K, 8, 1000, OC + 8, OC, None, NU, consecutive) == -1
        assert b"two outputs overlap" in L.b200sort_last_error()
        # num == 0 without out_num_unique: nothing to write
        assert _u(None, 8, 0, None, consecutive=consecutive) == 0
    assert (ok == 0).all() and (oc == 0).all() and (oi == 0).all() and (nu == 0).all()
    assert (k == np.arange(1000, dtype=np.float32)).all()


def test_python_value_and_type_errors():
    for bad in (np.float16, np.bool_, np.complex64):
        with pytest.raises(TypeError):
            S.unique(np.zeros(4, bad))
        with pytest.raises(TypeError):
            S.unique_consecutive(np.zeros(4, bad))
        with pytest.raises(TypeError):
            S.unique_workspace_bytes(bad, 10)
    with pytest.raises(ValueError):
        S.unique_workspace_bytes(np.int32, -1)


def test_workspace_bytes():
    for dt in (np.uint8, np.int16, np.float32, np.int32, np.uint64, np.float64):
        for consecutive in (False, True):
            for inverse in (False, True):
                sizes = [S.unique_workspace_bytes(dt, n, consecutive, inverse) for n in (0, 1, 4095, 4096, 4097, 10**6, 2**24 + 5)]
                assert all(a <= b for a, b in zip(sizes, sizes[1:])), (dt, consecutive, inverse, sizes)
                assert sizes[-1] > sizes[-2] > sizes[3]
                assert all(s % 256 == 0 and s > 0 for s in sizes)
                n = 2**20 + 3
                w = S.unique_workspace_bytes(dt, n, consecutive, inverse)
                assert w >= (n + 1) * 8  # the run starts
                if not consecutive:  # the sorted copy and the sort of it
                    idx = [4] if inverse else []
                    assert w >= n * np.dtype(dt).itemsize + S.workspace_bytes(dt, n, idx)
            # the inverse costs nothing without the sort
            assert S.unique_workspace_bytes(dt, 10**6, True, True) == S.unique_workspace_bytes(dt, 10**6, True, False)
        assert S.unique_workspace_bytes(dt, 10**6, False, True) > S.unique_workspace_bytes(dt, 10**6, False, False)
        assert S.unique_workspace_bytes(dt, 10**6, False, False) > S.unique_workspace_bytes(dt, 10**6, True, False)
    assert S.lib().b200sort_unique_workspace_bytes(42, 10, 0, 0) == 0
    assert S.lib().b200sort_unique_workspace_bytes(4, -1, 0, 0) == 0


def test_index_width_switch_at_2p32():
    # sorted mode with the inverse sorts (key, position) pairs: u32 positions up to 2^32 records, u64 above
    n = 2**32
    below, above = (S.unique_workspace_bytes(np.uint8, m, False, True) for m in (n, n + 1))
    assert above - below > 4 * n  # 4 more bytes per position, and the sort's shadow copy of them
    for consecutive, inverse in ((True, True), (False, False)):
        a, b = (S.unique_workspace_bytes(np.uint8, m, consecutive, inverse) for m in (n, n + 1))
        assert b - a <= 512


@pytest.mark.skipif(_has_cuda(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback():
    k = np.array([3, 1, 2, 3, 3, 1], dtype=np.int32)
    for fn in (S.unique, S.unique_consecutive):
        with pytest.raises(S.B200SortError) as ei:
            fn(k, return_inverse=True, return_counts=True)
        assert ei.value.code == -5 and "no CPU fallback" in str(ei.value)
    assert k.tolist() == [3, 1, 2, 3, 3, 1]
