"""Worker of tests/test_gpu_mgpu.py: one process per GPU (torchrun), sorts sharded records with
b200sort_mgpu_sort_soa and checks the distributed result against numpy on rank 0."""
import ctypes
import os
import sys
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import oracle_lib as O  # noqa: E402
import simd_radix_sort_b200 as S  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    L = S.lib()
    uid = [None]
    if rank == 0:
        buf = (ctypes.c_ubyte * 128)()
        assert L.b200sort_mgpu_unique_id(buf) == 0, L.b200sort_last_error()
        uid[0] = bytes(buf)
    dist.broadcast_object_list(uid, src=0)
    comm = ctypes.c_void_p()
    assert L.b200sort_mgpu_comm_create(ctypes.byref(comm), world, rank, (ctypes.c_ubyte * 128).from_buffer_copy(uid[0])) == 0, \
        L.b200sort_last_error()

    cases = [(np.uint64, "Uniform", True, 1_000_003), (np.float32, "Gaussian", False, 400_000), (np.int16, "Uniform", True, 250_000),
             (np.int64, "Gaussian", True, 300_000), (np.float64, "Uniform", False, 2_000_000)]
    L.b200sort_mgpu_used_p2p.argtypes = [ctypes.c_void_p]
    # records scattered straight into peer memory (twice: with the large-sort flow forced, whose local sort
    # reads the landing arrays in its first pass) / exchanged with ncclSend+ncclRecv
    for p2p, big_flow in ((1, 1), (1, 0), (0, 0)):
        with S.options(mgpu_p2p=p2p, host_plan_min_log2=0 if big_flow else 24, algo=2 if big_flow else 0):
            for ci, (dt, distname, up, n_base) in enumerate(cases):
                n_local = n_base + 1000 * rank
                keys = O.make_keys(distname, dt, n_local, seed=100 * ci + rank)
                pay = (np.arange(n_local, dtype=np.uint64) + (rank << 40))
                pay2 = (np.arange(n_local) % 65521).astype(np.uint16)  # a second, narrow payload stream
                cap = int((n_base + 1000 * world) * 1.5) + 4096      # the same on every rank (peer path needs equal layouts)
                k = torch.zeros(cap, dtype=torch.from_numpy(keys[:1]).dtype, device=dev)
                p = torch.zeros(cap, dtype=torch.uint64, device=dev)
                p2 = torch.zeros(cap, dtype=torch.uint16, device=dev)
                k[:n_local].copy_(torch.from_numpy(keys))
                p[:n_local].copy_(torch.from_numpy(pay))
                p2[:n_local].copy_(torch.from_numpy(pay2))
                ptrs = (ctypes.c_void_p * 2)(p.data_ptr(), p2.data_ptr())
                sizes = (ctypes.c_uint32 * 2)(8, 2)
                got = ctypes.c_int64(0)
                for rep in range(2):  # twice: the second call reuses the mapped peer workspaces
                    if rep:
                        k[:n_local].copy_(torch.from_numpy(keys))
                        p[:n_local].copy_(torch.from_numpy(pay))
                        p2[:n_local].copy_(torch.from_numpy(pay2))
                    rc = L.b200sort_mgpu_sort_soa(comm, k.data_ptr(), S.KEY_TYPES[np.dtype(dt).name], n_local, cap, int(up), 2, ptrs, sizes,
                                                  ctypes.byref(got), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
                    assert rc == 0, L.b200sort_last_error()
                    torch.cuda.synchronize()
                assert L.b200sort_mgpu_used_p2p(comm) == p2p, f"case {ci}: path taken {L.b200sort_mgpu_used_p2p(comm)}, wanted {p2p}"
                m = got.value
                out_k, out_p, out_p2 = k[:m].cpu().numpy(), p[:m].cpu().numpy(), p2[:m].cpu().numpy()
                gathered = [None] * world
                dist.all_gather_object(gathered, (keys, pay, out_k, out_p, out_p2))
                if rank == 0:
                    all_in_k = np.concatenate([g[0] for g in gathered])
                    all_out_k = np.concatenate([g[2] for g in gathered])
                    all_out_p = np.concatenate([g[3] for g in gathered])
                    all_out_p2 = np.concatenate([g[4] for g in gathered])
                    want = O.total_order_sorted_keys(all_in_k, up)
                    assert all_out_k.tobytes() == want.tobytes(), f"case {ci} p2p={p2p} big={big_flow}: distributed key sequence differs"
                    # payload followed its key: payload encodes (source rank, source index)
                    src_rank, src_idx = all_out_p >> np.uint64(40), all_out_p & np.uint64((1 << 40) - 1)
                    offs = np.cumsum([0] + [len(g[0]) for g in gathered])[:-1]
                    pos = offs[src_rank.astype(np.int64)] + src_idx.astype(np.int64)
                    assert all_in_k[pos].tobytes() == all_out_k.tobytes(), f"case {ci} p2p={p2p} big={big_flow}: payload did not follow its key"
                    assert np.array_equal(np.sort(pos), np.arange(len(all_in_k))), f"case {ci} p2p={p2p} big={big_flow}: not a permutation"
                    assert np.array_equal(all_out_p2, (src_idx % np.uint64(65521)).astype(np.uint16)), f"case {ci} p2p={p2p} big={big_flow}: second payload"
                    sizes_out = [len(g[2]) for g in gathered]
                    assert max(sizes_out) <= 1.3 * (sum(sizes_out) / world) + 70000, f"case {ci}: unbalanced {sizes_out}"

    def check_global(tag, keys, out_k, out_src, up, cap):
        gathered = [None] * world
        dist.all_gather_object(gathered, (keys, out_k, out_src))
        if rank == 0:
            all_in = np.concatenate([g[0] for g in gathered])
            all_out = np.concatenate([g[1] for g in gathered])
            src = np.concatenate([g[2] for g in gathered])
            assert all_out.tobytes() == O.total_order_sorted_keys(all_in, up).tobytes(), f"{tag}: distributed key sequence differs"
            src_rank, src_idx = src >> np.uint64(40), src & np.uint64((1 << 40) - 1)
            offs = np.cumsum([0] + [len(g[0]) for g in gathered])[:-1]
            pos = offs[src_rank.astype(np.int64)] + src_idx.astype(np.int64)
            assert all_in[pos].tobytes() == all_out.tobytes(), f"{tag}: payload did not follow its key"
            assert np.array_equal(np.sort(pos), np.arange(len(all_in))), f"{tag}: not a permutation"
            assert max(len(g[1]) for g in gathered) <= cap, f"{tag}: a rank is over capacity"

    # ---- skewed keys (SURVEY 8e(3)): never ENOMEM at capacity 1.125 * N / G; heavy key values are split --------
    rngs = np.random.default_rng(1000 + rank)
    table = np.random.default_rng(7).integers(-2**63, 2**63 - 1, size=1 << 12, dtype=np.int64)
    n_local = 300_000
    skew = {
        "zero": np.zeros(n_local, np.int64),
        "zero_one": rngs.integers(0, 2, size=n_local).astype(np.uint64),
        "few_unique16": rngs.integers(-8, 8, size=n_local, dtype=np.int64),
        "zipf": table[np.minimum(rngs.zipf(1.3, size=n_local), 1 << 12) - 1],
        "gauss_f32": rngs.normal(0, 1, size=n_local).astype(np.float32),
        "heavy_value_45pct": np.where(rngs.random(n_local) < 0.45, np.uint64(77), rngs.integers(0, 2**64, size=n_local, dtype=np.uint64)),
        "sorted_u16": np.sort(rngs.integers(0, 2**16, size=n_local, dtype=np.uint16)),
    }
    cap = int(1.125 * n_local) + 64
    for big_flow in (0, 1):
        with S.options(host_plan_min_log2=0 if big_flow else 24):
            for name, keys in skew.items():
                for up in (True, False):
                    keys = np.ascontiguousarray(keys)
                    k = torch.zeros(cap, dtype=torch.from_numpy(keys[:1]).dtype, device=dev)
                    p = torch.zeros(cap, dtype=torch.uint64, device=dev)
                    k[:n_local].copy_(torch.from_numpy(keys))
                    p[:n_local].copy_(torch.from_numpy(np.arange(n_local, dtype=np.uint64) + (rank << 40)))
                    ptrs = (ctypes.c_void_p * 1)(p.data_ptr())
                    sizes = (ctypes.c_uint32 * 1)(8)
                    got = ctypes.c_int64(0)
                    rc = L.b200sort_mgpu_sort_soa(comm, k.data_ptr(), S.KEY_TYPES[keys.dtype.name], n_local, cap, int(up), 1, ptrs, sizes,
                                                  ctypes.byref(got), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
                    assert rc == 0, (name, up, L.b200sort_last_error())
                    torch.cuda.synchronize()
                    check_global(f"skew {name} up={up} big={big_flow}", keys, k[:got.value].cpu().numpy(), p[:got.value].cpu().numpy(), up, cap)

    # ---- combined records: b200sort_mgpu_sort_aos (DataElement<int64, uint64>) ------------------------------------
    for up in (True, False):
        keys = O.make_keys("Gaussian", np.int64, n_local, seed=33 + rank)
        rec = np.empty((n_local, 2), np.int64)
        rec[:, 0] = keys
        rec[:, 1] = (np.arange(n_local, dtype=np.uint64) + (rank << 40)).view(np.int64)
        r = torch.zeros((cap, 2), dtype=torch.int64, device=dev)
        r[:n_local].copy_(torch.from_numpy(rec))
        got = ctypes.c_int64(0)
        rc = L.b200sort_mgpu_sort_aos(comm, r.data_ptr(), S.KEY_TYPES["int64"], 16, n_local, cap, int(up), ctypes.byref(got),
                                      ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0, L.b200sort_last_error()
        torch.cuda.synchronize()
        out = r[:got.value].cpu().numpy()
        check_global(f"aos up={up}", keys, np.ascontiguousarray(out[:, 0]), np.ascontiguousarray(out[:, 1]).view(np.uint64), up, cap)

    # ---- overlapped exchange: chunked partition kernels, arrival flags, first pass of the receivers chunk by chunk ----
    # landing arrays at test size; the overlapped exchange is off by default (DESIGN.md section 5)
    with S.options(host_plan_min_log2=0, mgpu_chunk_min_log2=12, mgpu_overlap=1):
        L.b200sort_mgpu_used_overlap.argtypes = [ctypes.c_void_p]
        for n_chunks, persist in ((4, 0), (3, 3), (8, 4), (1, 0)):
            with S.options(mgpu_chunks=n_chunks, mgpu_persist_x2=persist):   # 0: one partition kernel per chunk; else looping CTAs, persist/2 per SM
                for dt, up in ((np.uint64, True), (np.int64, False), (np.uint64, False)):
                    n_loc = (1 << 19) + 4099 + 77 * rank
                    keys = O.make_keys("Uniform", dt, n_loc, seed=500 + rank + n_chunks)
                    capo = int(1.125 * ((1 << 19) + 4099 + 77 * world)) + 4096
                    k = torch.zeros(capo, dtype=torch.from_numpy(keys[:1]).dtype, device=dev)
                    p = torch.zeros(capo, dtype=torch.uint64, device=dev)
                    for rep in range(2):
                        k[:n_loc].copy_(torch.from_numpy(keys))
                        p[:n_loc].copy_(torch.from_numpy(np.arange(n_loc, dtype=np.uint64) + (rank << 40)))
                        ptrs = (ctypes.c_void_p * 1)(p.data_ptr())
                        sizes = (ctypes.c_uint32 * 1)(8)
                        got = ctypes.c_int64(0)
                        rc = L.b200sort_mgpu_sort_soa(comm, k.data_ptr(), S.KEY_TYPES[np.dtype(dt).name], n_loc, capo, int(up), 1, ptrs, sizes,
                                                      ctypes.byref(got), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
                        assert rc == 0, L.b200sort_last_error()
                        torch.cuda.synchronize()
                    assert L.b200sort_mgpu_used_overlap(comm) == 1, "the overlapped exchange was not taken"
                    check_global(f"overlap chunks={n_chunks} {np.dtype(dt).name} up={up}", keys, k[:got.value].cpu().numpy(),
                                 p[:got.value].cpu().numpy(), up, capo)
    dist.barrier()
    assert L.b200sort_mgpu_comm_destroy(comm) == 0
    dist.destroy_process_group()
    print(f"MGPU_GPU_OK {rank}", flush=True)


if __name__ == "__main__":
    main()
