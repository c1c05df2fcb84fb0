"""GPU tests (-m gpu) of the top-k selection (topk, topk_combined; b200sort_topk_soa / _aos).

Bar: the keys of every row equal, byte for byte, the first k keys of a stable numpy argsort of the order-mapped row
(oracle_lib.order_key); the indices of a row are distinct positions inside it and keys[index] equals the output keys;
every payload output (or AoS record) is the input's element at that index; the inputs are unchanged."""
import ctypes

import numpy as np
import pytest

import oracle_lib as O
import simd_radix_sort_b200 as S

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ALL_DTYPES = [np.dtype(d) for d in O.KEY_DTYPES]


@pytest.fixture(scope="module", autouse=True)
def _loaded():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    before = S.launch_count()
    yield
    assert S.launch_count() > before, "no kernels of libb200sort.so were launched"


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.cpu().numpy()


def keys_of(dt, n, rng):
    """random keys with duplicates; floats with +-0, +-inf and +-NaN among them"""
    dt = np.dtype(dt)
    if dt.kind == "f":
        k = rng.standard_normal(n).astype(dt)
        sp = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, -np.nan], dtype=dt)
        m = rng.random(n) < 0.05
        k[m] = sp[rng.integers(0, len(sp), int(m.sum()))]
        return k
    info = np.iinfo(dt)
    return rng.integers(int(info.min), int(info.max), size=n, dtype=dt, endpoint=True)


def sorted_order(keys2d, largest):
    """positions of every row in the output order (stable argsort of the order-mapped keys)"""
    return np.argsort(O.order_key(keys2d, up=not largest), axis=1, kind="stable")


def check(keys2d, k, largest, vals, idx, pays_in=(), pays_out=(), order=None):
    B, L = keys2d.shape
    vals, idx = vals.reshape(B, k), idx.reshape(B, k)
    if order is None:
        order = sorted_order(keys2d, largest)
    exp = np.take_along_axis(keys2d, order[:, :k], 1)
    assert vals.tobytes() == exp.tobytes(), "keys differ from the stable top-k of the order-mapped keys"
    assert idx.dtype == np.int64
    if k:
        assert idx.min() >= 0 and idx.max() < L
        s = np.sort(idx, axis=1)
        assert (s[:, 1:] != s[:, :-1]).all(), "indices of a row repeat"
    assert np.take_along_axis(keys2d, idx, 1).tobytes() == vals.tobytes(), "keys[index] differs from the output keys"
    for p_in, p_out in zip(pays_in, pays_out):
        tail = p_in.shape[2:]
        want = np.take_along_axis(p_in, idx.reshape((B, k) + (1,) * len(tail)), 1)
        assert p_out.reshape((B, k) + tail).tobytes() == want.tobytes(), "a payload does not follow the index"


def run(keys, k, largest, pays=(), order=None):
    """topk of the numpy keys (1-D or 2-D) and payloads on the device; checked; -> (values, indices, payload outputs)"""
    kd, pd = dev(keys), [dev(p) for p in pays]
    vals, idx, *po = S.topk(kd, k, *pd, largest=largest)
    assert tuple(vals.shape) == keys.shape[:-1] + (k,) and tuple(idx.shape) == tuple(vals.shape)
    torch.cuda.synchronize()
    assert host(kd).tobytes() == keys.tobytes(), "the keys changed"
    for p, d in zip(pays, pd):
        assert host(d).tobytes() == p.tobytes(), "a payload changed"
    k2 = keys.reshape(-1, keys.shape[-1])
    p2 = [p.reshape(k2.shape + p.shape[keys.ndim:]) for p in pays]
    check(k2, k, largest, host(vals), host(idx), p2, [host(o) for o in po], order)
    return host(vals), host(idx), [host(o) for o in po]


def k_values(n):
    return sorted({k for k in (1, 2, 17, n // 2, n - 1, n) if 0 < k <= n})


@pytest.mark.parametrize("dt", ALL_DTYPES, ids=lambda d: d.name)
def test_every_key_type_whole_arrays(dt):
    rng = np.random.default_rng(1)
    for n in (1, 2, 255, 256, 257, 4097, 2**20 + 3):
        keys = keys_of(dt, n, rng)
        for largest in (True, False):
            order = sorted_order(keys.reshape(1, n), largest)
            for k in k_values(n):
                run(keys, k, largest, order=order)


@pytest.mark.parametrize("dt", ALL_DTYPES, ids=lambda d: d.name)
def test_every_key_type_rows(dt):
    rng = np.random.default_rng(2)
    for B, L in ((7, 1000), (3, 2**17 + 1), (64, 128256)):
        keys = keys_of(dt, B * L, rng).reshape(B, L)
        for largest in (True, False):
            order = sorted_order(keys, largest)
            for k in k_values(L):
                run(keys, k, largest, order=order)


@pytest.mark.parametrize("k", [1, 50, 1024])
def test_matches_torch_topk_on_sampling_rows(k):
    g = torch.Generator(device="cuda").manual_seed(3)
    x = torch.randn(64, 128256, device="cuda", generator=g)
    vals, idx = S.topk(x, k)
    ref = torch.topk(x, k)
    assert torch.equal(vals, ref.values)
    assert torch.equal(torch.gather(x, 1, idx), vals)
    vals, idx = S.topk(x, k, largest=False)
    assert torch.equal(vals, torch.topk(x, k, largest=False).values)
    assert torch.equal(torch.gather(x, 1, idx), vals)


def test_ties_and_the_reread_path():
    rng = np.random.default_rng(4)
    n = 300_001
    for dt in (np.uint32, np.float32, np.int64):
        for largest in (True, False):
            equal = np.full(n, 7, dtype=dt)  # every digit's bucket holds the whole row
            for k in (1, 1000, n // 2, n):
                run(equal, k, largest)
            two = np.where(rng.random(n) < 0.5, 3, 9).astype(dt)
            for k in (1, n // 3, n // 2, n - 1):
                run(two, k, largest)
    # the k-th place inside a run of 10^6 equal keys
    m = 3 * 10**6
    keys = rng.integers(0, 2**32, m, dtype=np.uint64).astype(np.uint32)
    run_pos = rng.permutation(m)[:10**6]
    keys[run_pos] = 2**31
    above = int((keys > 2**31).sum())
    for k in (above + 1, above + 500_000, above + 10**6):
        run(keys, k, True)
    # a constant top byte (u32) and constant top 7 bytes (u64): the first bucket exceeds the candidate buffer, so
    # later passes re-read the row
    u32 = (0xAB000000 | rng.integers(0, 2**24, 2**20 + 5)).astype(np.uint32)
    u64 = (np.uint64(0x0123456789ABCD00) | rng.integers(0, 256, 2**20 + 5).astype(np.uint64)).astype(np.uint64)
    for keys in (u32, u64):
        for largest in (True, False):
            for k in (1, 100, 70_000, len(keys) // 2):
                run(keys, k, largest)


def test_payload_shapes_and_offset_views():
    rng = np.random.default_rng(5)
    B, L, k = 5, 3001, 77
    keys = keys_of(np.float32, B * L, rng).reshape(B, L)
    run(keys, k, True)
    sizes = (1, 2, 3, 8, 12, 16, 64)
    pays = [rng.integers(0, 256, (B, L, s), dtype=np.uint8) for s in sizes]
    pays.append(rng.integers(0, 2**60, (B, L), dtype=np.int64))
    run(keys, k, True, pays)
    run(keys, k, False, pays[:1])
    # 63 streams
    pays63 = [rng.integers(0, 256, (B, L, 1 + i % 9), dtype=np.uint8) for i in range(63)]
    run(keys, k, False, pays63)
    # keys and payloads as views one element into larger buffers (not 16-byte aligned)
    kbuf, pbuf8 = dev(np.zeros(B * L + 1, np.float32)), dev(np.zeros(B * L + 1, np.int64))
    pbuf12 = dev(np.zeros((B * L + 1, 3), np.int32))
    kbuf[1:] = dev(keys.reshape(-1))
    p8, p12 = rng.integers(0, 2**60, B * L, dtype=np.int64), rng.integers(0, 2**31, (B * L, 3), dtype=np.int32)
    pbuf8[1:], pbuf12[1:] = dev(p8), dev(p12)
    kv, p8v, p12v = kbuf[1:].view(B, L), pbuf8[1:].view(B, L), pbuf12[1:].view(B, L, 3)
    vals, idx, o8, o12 = S.topk(kv, k, p8v, p12v)
    check(keys, k, True, host(vals), host(idx), [p8.reshape(B, L), p12.reshape(B, L, 3)], [host(o8), host(o12)])


def test_records_of_every_power_of_two_size():
    rng = np.random.default_rng(6)
    B, L, k = 3, 20_000, 333
    for dt in ALL_DTYPES:
        keys = keys_of(dt, B * L, rng)
        for rb in (1, 2, 4, 8, 16, 32, 64):
            if rb < dt.itemsize:
                continue
            rec = O.make_records(keys, rb).reshape(B, L, rb)
            for largest in (True, False):
                rd = dev(rec)
                out, idx = S.topk_combined(rd, dt, k, largest=largest)
                assert host(rd).tobytes() == rec.tobytes()
                out, idx = host(out), host(idx)
                vals = np.ascontiguousarray(out[:, :, :dt.itemsize]).view(dt).reshape(B, k)
                check(keys.reshape(B, L), k, largest, vals, idx, [rec], [out])


def test_every_branch_of_the_ordering_step():
    rng = np.random.default_rng(7)
    # k = 20000 > 8192 on 8-byte keys: one whole-array sort per row; k = 40000 > 16384 on f32: the composite-key sort
    for dt, k in ((np.uint64, 20_000), (np.float64, 20_000), (np.float32, 40_000), (np.int16, 40_000)):
        keys = keys_of(dt, 3 * 100_003, rng).reshape(3, 100_003)
        idx_pay = np.arange(keys.size, dtype=np.int64).reshape(keys.shape)
        for largest in (True, False):
            run(keys, k, largest, [idx_pay])


def test_positions_above_2p32():
    n = 2**32 + 2**20
    g = torch.Generator(device="cuda").manual_seed(8)
    x = torch.randint(0, 255, (n,), device="cuda", dtype=torch.uint8, generator=g)
    planted = torch.tensor([2**32, 2**32 + 1, 2**32 + 12345, n - 1], device="cuda")
    x[planted] = 255
    vals, idx = S.topk(x, 4)
    assert sorted(host(idx).tolist()) == sorted(host(planted).tolist())
    assert (host(vals) == 255).all()
    vals, idx = S.topk(x, 6)
    assert set(host(planted).tolist()) <= set(host(idx).tolist()) and (host(vals)[4:] == 254).all()
    assert torch.equal(x[idx], vals)
    del x


def test_caller_workspace_side_stream_stats_and_profile():
    rng = np.random.default_rng(9)
    B, L, k = 16, 50_000, 300
    keys = keys_of(np.float32, B * L, rng).reshape(B, L)
    pay = rng.integers(0, 2**60, (B, L), dtype=np.int64)
    kd, pd = dev(keys), dev(pay)
    nbytes = S.topk_workspace_bytes(np.float32, B, L, k, [8])
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    vals, idx, po = S.topk(kd, k, pd, workspace=ws)
    check(keys, k, True, host(vals), host(idx), [pay], [host(po)])
    st = S.last_stats()
    assert st["algo"] == 4 and st["num"] == B * L and st["key_bytes"] == 4 and st["record_bytes"] == 12
    assert st["kernel_launches"] > 0 and st["passes_planned"] == 0 and st["hist_sweeps"] == 0
    # a side stream, two calls back to back; the outputs are allocated on that stream
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    a = S.topk(kd, k, pd, largest=True, stream=s.cuda_stream)
    b = S.topk(kd, k, pd, largest=False, stream=s.cuda_stream)
    s.synchronize()
    check(keys, k, True, host(a[0]), host(a[1]), [pay], [host(a[2])])
    check(keys, k, False, host(b[0]), host(b[1]), [pay], [host(b[2])])
    with S.options(profile=1):
        S.topk(kd, k)
        kinds = [kind for kind, _ in S.last_profile()]
    assert "select" in kinds and "segment" in kinds
    assert S.last_stats()["algo"] == 4


def test_errors_leave_the_outputs_untouched():
    L = S.lib()
    k0 = np.arange(1000, dtype=np.float32)
    # host arrays (numpy, CPU tensors): -7
    for keys in (k0, torch.from_numpy(k0)):
        with pytest.raises(S.B200SortError) as ei:
            S.topk(keys, 10)
        assert ei.value.code == -7
    kd = dev(k0.reshape(4, 250))
    out = torch.full((4, 10), -1.0, device="cuda")
    idx = torch.full((4, 10), -1, dtype=torch.int64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    # an output inside the input
    assert L.b200sort_topk_soa(kd.data_ptr(), 8, 4, 250, 10, 1, 0, None, None, kd.data_ptr() + 400, idx.data_ptr(), None, stream,
                               None, 0) == -1
    # k > row_len
    assert L.b200sort_topk_soa(kd.data_ptr(), 8, 4, 250, 251, 1, 0, None, None, out.data_ptr(), idx.data_ptr(), None, stream,
                               None, 0) == -1
    # a host output with device inputs
    hout = np.full((4, 10), -1.0, np.float32)
    assert L.b200sort_topk_soa(kd.data_ptr(), 8, 4, 250, 10, 1, 0, None, None, hout.ctypes.data, idx.data_ptr(), None, stream,
                               None, 0) == -7
    # a caller workspace that is too small
    ws = torch.empty(1024, dtype=torch.uint8, device="cuda")
    assert L.b200sort_topk_soa(kd.data_ptr(), 8, 4, 250, 10, 1, 0, None, None, out.data_ptr(), idx.data_ptr(), None, stream,
                               ctypes.c_void_p(ws.data_ptr()), 1024) == -4
    torch.cuda.synchronize()
    assert (host(out) == -1.0).all() and (host(idx) == -1).all() and (hout == -1.0).all()
    assert host(kd).tobytes() == k0.tobytes()
