"""GPU tests (-m gpu) of the host call path every single-GPU entry point shares.

A public call starts its own profile, so with option "profile" set b200sort_last_profile lists exactly the kernels that
b200sort_last_stats counts for that call: those of the sorts it runs inside and of a hybrid sort's fall-back included,
nothing of an earlier call.  Also the placement errors: host arrays given to a call that takes device arrays only, and a
call that mixes host and device arrays."""

import numpy as np
import pytest

import simd_radix_sort_b200 as S

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _loaded():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    before = S.launch_count()
    yield
    assert S.launch_count() > before, "no kernels of libb200sort.so were launched"


@pytest.fixture
def profiled():
    """option "profile" set for the test, after a profiled sort that leaves entries of its own"""
    with S.options(profile=1):
        k = torch.arange(4096, 0, -1, dtype=torch.int32, device="cuda")
        S.sort(k.numel(), k)
        assert len(S.last_profile()) > 0
        yield


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.cpu().numpy()


def profile_of_call(algo):
    """-> (stats, profile kinds) of the last call, after checking that the profile lists every kernel it launched"""
    st = S.last_stats()
    kinds = [kind for kind, _ in S.last_profile()]
    assert st["algo"] == algo, st
    assert len(kinds) == st["kernel_launches"], (kinds, st)
    return st, kinds


def test_lsd_sort(profiled):
    rng = np.random.default_rng(1)
    keys = rng.integers(-2**31, 2**31, 1 << 20, dtype=np.int32)
    k, p = dev(keys), dev(np.arange(keys.size, dtype=np.int64))
    S.sort(keys.size, k, p)
    st, kinds = profile_of_call(1)
    assert st["kernel_launches"] > 0 and "sweep" in kinds
    assert host(k).tobytes() == np.sort(keys).tobytes()


def test_hybrid_sort(profiled):
    rng = np.random.default_rng(2)
    keys = rng.integers(0, 2**64, 300_000, dtype=np.uint64)
    k = dev(keys)
    with S.options(algo=2):
        S.sort(keys.size, k)
    st, _ = profile_of_call(2)
    assert st["fell_back"] == 0 and st["kernel_launches"] > 0
    assert host(k).tobytes() == np.sort(keys).tobytes()


def test_hybrid_fall_back(profiled):
    # top digits a function of a group of 1000 records, low word random: long buckets of distinct keys
    n = 300_000
    rng = np.random.default_rng(3)
    g = np.arange(n) // 1000
    f = rng.integers(0, 2**32, g.max() + 1, dtype=np.uint64)
    keys = (f[g] << np.uint64(32)) | rng.integers(0, 2**32, n, dtype=np.uint64)
    k = dev(keys)
    with S.options(algo=2):
        S.sort(n, k)
    st, kinds = profile_of_call(2)
    assert st["fell_back"] == 1
    assert kinds.count("scan") >= 2, kinds  # the hybrid attempt's plan and the digit-by-digit sort's
    assert host(k).tobytes() == np.sort(keys).tobytes()


@pytest.mark.parametrize("dtype", [np.uint32, np.uint64])
def test_segmented_long_segments(profiled, dtype):
    # segments longer than CAP (16384 records for 4-byte keys, 8192 for 8-byte keys) take whole-array sorts: one of
    # (segment, key) pairs over all segments for 4-byte keys, one per long segment beside the short-segment kernels for
    # 8-byte keys
    rng = np.random.default_rng(4)
    offsets = np.array([0, 100, 20_000, 20_050, 45_000, 60_000], np.int64)
    keys = rng.integers(0, np.iinfo(dtype).max, 60_000, dtype=dtype)
    k = dev(keys)
    S.sort_segmented(dev(offsets), k)
    st, kinds = profile_of_call(3)
    assert "sweep" in kinds and ("segment" in kinds) == (dtype == np.uint64), kinds
    got = host(k)
    for a, b in zip(offsets[:-1], offsets[1:]):
        assert got[a:b].tobytes() == np.sort(keys[a:b]).tobytes()


def test_topk(profiled):
    rng = np.random.default_rng(5)
    keys = rng.standard_normal((64, 5000)).astype(np.float32)
    values, index = S.topk(dev(keys), 100)
    st, kinds = profile_of_call(4)
    assert "select" in kinds and "segment" in kinds
    assert host(values).tobytes() == (-np.sort(-keys, axis=1)[:, :100]).tobytes()
    assert np.array_equal(np.take_along_axis(keys, host(index), axis=1), host(values))


@pytest.mark.parametrize("fn", [S.unique, S.unique_consecutive])
def test_unique(profiled, fn):
    rng = np.random.default_rng(6)
    keys = rng.integers(0, 1000, 100_000, dtype=np.int32)
    values, inverse, counts = fn(dev(keys), return_inverse=True, return_counts=True)
    st, kinds = profile_of_call(5)
    assert "unique" in kinds and st["num"] == keys.size
    assert np.array_equal(host(values)[host(inverse)], keys) and int(host(counts).sum()) == keys.size


def test_unique_of_nothing(profiled):
    values, inverse, counts = S.unique(torch.empty(0, dtype=torch.int32, device="cuda"), return_inverse=True, return_counts=True)
    assert values.numel() == 0 and inverse.numel() == 0 and counts.numel() == 0
    st, kinds = profile_of_call(5)
    assert st["num"] == 0 and kinds == []


def test_placement_errors():
    k0 = np.arange(1000, dtype=np.float32)
    # host arrays given to top-k or unique: -7
    for call in (lambda x: S.topk(x, 10), lambda x: S.unique(x, return_counts=True)):
        for keys in (k0.copy(), torch.from_numpy(k0.copy())):
            with pytest.raises(S.B200SortError) as ei:
                call(keys)
            assert ei.value.code == -7
    # host and device arrays in one call: -1, and nothing moves
    kd = dev(k0[::-1])
    hp = np.arange(1000, dtype=np.int64)
    with pytest.raises(S.B200SortError) as ei:
        S.sort(1000, kd, hp)
    assert ei.value.code == -1 and "all in host memory or all in device memory" in str(ei.value)
    with pytest.raises(S.B200SortError) as ei:
        S.sort_segmented(np.array([0, 500, 1000], np.int64), kd)
    assert ei.value.code == -1 and "offsets" in str(ei.value)
    assert host(kd).tobytes() == k0[::-1].tobytes() and (hp == np.arange(1000)).all()
