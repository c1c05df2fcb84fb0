"""GPU tests (-m gpu) of the state the library keeps between calls: the per-device workspace and host-staging
caches (and b200sort_release_cache), and the per-thread, per-device events and streams.  Host-array calls all
stage through the cached staging buffer: below 2^20 records, or for AoS and key-only arrays, as a whole; SoA
arrays with payloads from 2^20 records through the pipelined path."""
import threading

import numpy as np
import pytest

import oracle_lib as O
import simd_radix_sort_b200 as S

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

PIPELINED_N = (1 << 20) + 1


@pytest.fixture(scope="module", autouse=True)
def _loaded():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    assert S.lib_path().exists(), "libb200sort.so must be built (no fallback)"
    before = S.launch_count()
    yield
    assert S.launch_count() > before, "no kernels of libb200sort.so were launched"


def _host_soa(keys, up=True):
    """sorts host copies of keys + an index payload; checks both against the oracle"""
    k, idx = keys.copy(), np.arange(len(keys), dtype=np.uint64)
    S.sort(len(k), k, idx, up=up)
    assert k.tobytes() == O.total_order_sorted_keys(keys, up).tobytes()
    assert keys[idx].tobytes() == k.tobytes() and np.array_equal(np.sort(idx), np.arange(len(keys), dtype=np.uint64))


def _host_keys_only(keys, up=True):
    k = keys.copy()
    S.sort(len(k), k, up=up)
    assert k.tobytes() == O.total_order_sorted_keys(keys, up).tobytes()


def _host_aos(keys, record_bytes=16, up=True):
    """records whose payload bytes derive from the key: the sorted records are the records of the sorted keys"""
    rec = O.make_records(keys, record_bytes)
    S.sort_combined(len(keys), rec, keys.dtype, up=up)
    assert rec.tobytes() == O.make_records(O.total_order_sorted_keys(keys, up), record_bytes).tobytes()


def _both_staging_paths(seed):
    _host_aos(O.make_keys("Uniform", np.int64, 300_000, seed=seed))
    _host_keys_only(O.make_keys("Gaussian", np.float32, 500_000, seed=seed + 1), up=False)
    _host_soa(O.make_keys("Uniform", np.uint64, 200_000, seed=seed + 2))  # below 2^20: staged as a whole
    _host_soa(O.make_keys("Uniform", np.uint32, PIPELINED_N, seed=seed + 3))  # pipelined
    _host_aos(O.make_keys("Uniform", np.uint16, PIPELINED_N, seed=seed + 4), record_bytes=4)  # AoS: staged as a whole


def test_host_staging_paths_back_to_back_and_after_release():
    _both_staging_paths(seed=1)
    S.lib().b200sort_release_cache()
    _both_staging_paths(seed=11)
    S.lib().b200sort_release_cache()
    _host_soa(O.make_keys("Uniform", np.uint32, PIPELINED_N, seed=21))  # pipelined first after a release
    _host_aos(O.make_keys("Uniform", np.int64, 1000, seed=22))


def test_two_threads_host_and_device_arrays():
    """two host threads, each sorting its own host and device arrays with the library's caches (workspace=None)"""
    errors = []

    def work(t):
        try:
            for i in range(20):
                seed = 1000 * t + i
                _host_soa(O.make_keys("Uniform", np.int64, 100_000 + 17 * t, seed=seed))
                keys = O.make_keys("Uniform", np.uint32, 300_000 + 5 * t, seed=seed)
                k = torch.from_numpy(keys).cuda()
                p = torch.arange(len(keys), dtype=torch.int32, device="cuda")
                S.sort(len(keys), k, p)
                torch.cuda.current_stream().synchronize()
                hk, hp = k.cpu().numpy(), p.cpu().numpy()
                assert hk.tobytes() == O.total_order_sorted_keys(keys).tobytes(), (t, i)
                assert keys[hp].tobytes() == hk.tobytes(), (t, i)
        except Exception as ex:  # (re-raised by the main thread)
            errors.append(ex)

    threads = [threading.Thread(target=work, args=(t,)) for t in range(2)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    if errors:
        raise errors[0]


def test_one_thread_alternates_devices_with_host_arrays():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    for i in range(6):
        with torch.cuda.device(i % 2):
            _host_soa(O.make_keys("Uniform", np.uint64, PIPELINED_N, seed=40 + i))  # pipelined: per-device streams
            _host_keys_only(O.make_keys("Uniform", np.int32, 70_000, seed=50 + i))
