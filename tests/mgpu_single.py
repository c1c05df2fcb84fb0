"""Development vehicle: the multi-GPU entry points with a ONE-rank communicator on one GPU (NCCL allows a world of
one): exercises splitters, counting, the peer-store partition kernel (into this rank's own landing arrays), the
chunked / overlapped exchange with its arrival flags and the forced-plan local sort -- everything except real
peer traffic.  Also run by tests/test_gpu_mgpu.py on single-GPU boxes.   python tests/mgpu_single.py"""
import ctypes
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import oracle_lib as O  # noqa: E402
import simd_radix_sort_b200 as S  # noqa: E402


def main():
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    L = S.lib()
    buf = (ctypes.c_ubyte * 128)()
    assert L.b200sort_mgpu_unique_id(buf) == 0, L.b200sort_last_error()
    comm = ctypes.c_void_p()
    assert L.b200sort_mgpu_comm_create(ctypes.byref(comm), 1, 0, buf) == 0, L.b200sort_last_error()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def run(keys, up, tag, want_overlap=None, offset=0):
        """offset: keys and payloads are views that start `offset` elements into their allocations"""
        n = len(keys)
        cap = n + 4096
        kbuf = torch.zeros(cap + offset, dtype=torch.from_numpy(keys[:1]).dtype, device=dev)
        pbuf = torch.zeros(cap + offset, dtype=torch.uint64, device=dev)
        k, p = kbuf[offset:], pbuf[offset:]
        k[:n].copy_(torch.from_numpy(keys))
        p[:n].copy_(torch.from_numpy(np.arange(n, dtype=np.uint64)))
        ptrs = (ctypes.c_void_p * 1)(p.data_ptr())
        sizes = (ctypes.c_uint32 * 1)(8)
        got = ctypes.c_int64(0)
        rc = L.b200sort_mgpu_sort_soa(comm, k.data_ptr(), S.KEY_TYPES[keys.dtype.name], n, cap, int(up), 1, ptrs, sizes, ctypes.byref(got), st)
        assert rc == 0, (tag, L.b200sort_last_error())
        torch.cuda.synchronize()
        assert got.value == n, tag
        hk, hp = k[:n].cpu().numpy(), p[:n].cpu().numpy().astype(np.int64)
        assert hk.tobytes() == O.total_order_sorted_keys(keys, up).tobytes(), tag + ": key sequence"
        assert keys[hp].tobytes() == hk.tobytes() and np.array_equal(np.sort(hp), np.arange(n)), tag + ": payloads"
        if want_overlap is not None:
            assert L.b200sort_mgpu_used_overlap(comm) == want_overlap, (tag, "overlap path", L.b200sort_mgpu_used_overlap(comm))
        print("ok", tag, flush=True)

    n = (1 << 20) + 4099
    rng = np.random.default_rng(1)
    run(O.make_keys("Uniform", np.uint64, n, 1), True, "plain u64")
    run(O.make_keys("Gaussian", np.float32, n, 2), False, "plain f32 desc")
    # keys and payloads at 8 mod 16: the count and partition kernels take their paths for keys that are not dense and
    # 16-byte aligned
    run(O.make_keys("Uniform", np.uint64, n, 30), True, "u64 at offset 1", offset=1)
    with S.options(host_plan_min_log2=0):
        run(O.make_keys("Uniform", np.uint64, n, 3), True, "landing u64", 0)
        with S.options(mgpu_chunk_min_log2=12, mgpu_overlap=2):   # 2: also with a world of one (this vehicle)
            for chunks, persist in ((4, 0), (1, 3), (3, 4), (8, 2)):
                with S.options(mgpu_chunks=chunks, mgpu_persist_x2=persist):
                    run(O.make_keys("Uniform", np.uint64, n, 4 + chunks), True, f"overlap u64 chunks={chunks}", 1)
                    run(O.make_keys("Uniform", np.int64, n, 14 + chunks), False, f"overlap i64 desc chunks={chunks}", 1)
        run(np.zeros(n, np.int64), True, "zero")
        run(O.make_keys("Gaussian", np.int64, n, 31), False, "i64 desc at offset 1", offset=1)
        run(rng.integers(-8, 8, size=n, dtype=np.int64), False, "few unique")
    assert L.b200sort_mgpu_comm_destroy(comm) == 0
    print("MGPU_SINGLE_OK", flush=True)


if __name__ == "__main__":
    main()
