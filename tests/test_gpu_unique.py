"""GPU tests (-m gpu) of unique and unique_consecutive (b200sort_unique).

Bar: against a numpy reference built on bit patterns (oracle_lib.order_key: equality of keys is equality of bits, the
order of the distinct keys is the library's total order), every call's values are equal byte for byte, its counts and
its inverse exactly, and U.  Through the C ABI: the input is unchanged, output entries >= U keep a sentinel, and guard
bytes around every output are unchanged."""

import numpy as np
import pytest

import oracle_lib as O
import simd_radix_sort_b200 as S

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ALL_DTYPES = [np.dtype(d) for d in O.KEY_DTYPES]
TILE = 4096  # keys per tile of the run-compaction kernel (UNQ_TILE)
SMALL_SIZES = (0, 1, 2, TILE - 1, TILE, TILE + 1, 3 * TILE + 5, 2**20 + 3)
OPTIONS = [(False, False), (False, True), (True, False), (True, True)]  # (return_inverse, return_counts)


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


def bits(keys):
    return keys.view(f"uint{keys.dtype.itemsize * 8}")


def reference(keys, consecutive):
    """-> (values, inverse, counts) of the flattened numpy keys, on bit patterns"""
    keys = keys.reshape(-1)
    n = len(keys)
    if consecutive:
        b = bits(keys)
        head = np.ones(n, bool)
        head[1:] = b[1:] != b[:-1]
        starts = np.flatnonzero(head)
        return keys[head], (np.cumsum(head) - 1).astype(np.int64), np.diff(np.append(starts, n)).astype(np.int64)
    _, first, inverse, counts = np.unique(O.order_key(keys), return_index=True, return_inverse=True, return_counts=True)
    return keys[first], inverse.reshape(-1).astype(np.int64), counts.astype(np.int64)


def run(keys, consecutive, ref=None, options=OPTIONS, kd=None):
    """unique of the numpy keys on the device with every option set, each checked against the reference"""
    ref = reference(keys, consecutive) if ref is None else ref
    kd = dev(keys) if kd is None else kd
    fn = S.unique_consecutive if consecutive else S.unique
    for inv, cnt in options:
        out = fn(kd, return_inverse=inv, return_counts=cnt)
        out = out if isinstance(out, tuple) else (out,)
        assert len(out) == 1 + inv + cnt
        assert host(out[0]).tobytes() == ref[0].tobytes(), f"values differ ({keys.dtype}, n={keys.size}, consecutive={consecutive})"
        if inv:
            assert out[1].dtype == torch.int64 and tuple(out[1].shape) == keys.shape
            assert np.array_equal(host(out[1]).reshape(-1), ref[1]), "inverse differs"
        if cnt:
            assert out[-1].dtype == torch.int64
            assert np.array_equal(host(out[-1]), ref[2]), "counts differ"
    assert host(kd).tobytes() == keys.tobytes(), "the input changed"


def random_keys(dt, n, rng):
    if dt.kind == "f":
        return rng.standard_normal(n).astype(dt)
    info = np.iinfo(dt)
    return rng.integers(int(info.min), int(info.max), size=n, dtype=dt, endpoint=True)


def distributions(dt, n, rng):
    """named key arrays of type dt and length n"""
    out = {"random": random_keys(dt, n, rng), "equal": np.full(n, 7, dt)}
    if n <= 2 ** (8 * dt.itemsize):
        out["distinct"] = rng.permutation(n).astype(np.uint64).astype(dt) if dt.kind != "f" else \
            (rng.permutation(n) - n // 2).astype(dt)
    pick = lambda vals: np.asarray(vals, dtype=dt)[rng.integers(0, len(vals), n)]
    out["two"] = pick([3, 9])
    out["sixteen"] = pick(np.arange(16) * 5 - 20 if dt.kind != "u" else np.arange(16) * 5)
    out["zipf"] = np.minimum(rng.zipf(1.3, n), 100).astype(dt)
    # runs longer than several tiles, in random value order; runs that start exactly at tile (and half-tile) boundaries
    lens = rng.integers(3 * TILE, 5 * TILE, max(1, n // (3 * TILE)))
    out["long_runs"] = np.resize(np.repeat(np.asarray(rng.integers(0, 100, len(lens)), dtype=dt), lens), n)
    out["tile_runs"] = ((np.arange(n) // TILE) % 100).astype(dt)
    out["half_tile_runs"] = ((np.arange(n) // (TILE // 2)) % 7).astype(dt)
    return out


def float_specials(dt, n, rng):
    u = f"uint{dt.itemsize * 8}"
    if dt == np.float32:
        nans = np.array([0x7FC00000, 0x7FC00001, 0x7F800001, 0xFFC00000, 0xFFC12345], np.uint32).view(np.float32)
        denorm = np.array([1, 2, 0x007FFFFF, 0x80000001], np.uint32).view(np.float32)
    else:
        nans = np.array([0x7FF8000000000000, 0x7FF8000000000001, 0x7FF0000000000001, 0xFFF8000000000000],
                        np.uint64).view(np.float64)
        denorm = np.array([1, 2, 0x000FFFFFFFFFFFFF, 0x8000000000000001], np.uint64).view(np.float64)
    sp = np.concatenate([np.array([0.0, -0.0, np.inf, -np.inf, 1.0, -1.0], dt), nans.astype(dt, copy=False),
                         denorm.astype(dt, copy=False)])
    assert sp.dtype == dt and len(np.unique(bits(sp))) == len(sp)
    return sp[rng.integers(0, len(sp), n)].view(u).view(dt)


@pytest.mark.parametrize("dt", ALL_DTYPES, ids=lambda d: d.name)
@pytest.mark.parametrize("consecutive", [False, True], ids=["sorted", "consecutive"])
def test_every_key_type_size_and_distribution(dt, consecutive):
    rng = np.random.default_rng(1)
    for n in SMALL_SIZES:
        for name, keys in distributions(dt, n, rng).items():
            ref = reference(keys, consecutive)
            if name == "distinct" and not consecutive:
                assert len(ref[0]) == n
            if name == "equal" and n:
                assert len(ref[0]) == 1
            run(keys, consecutive, ref)
        if dt.kind == "f":
            run(float_specials(dt, n, rng), consecutive)


@pytest.mark.parametrize("dt", [np.dtype(np.float32), np.dtype(np.int32), np.dtype(np.uint32)], ids=lambda d: d.name)
def test_large_4_byte_keys(dt):
    # 2^24 + 5 records: the sort reads its plan back and takes the 8192-key wide tiles
    rng = np.random.default_rng(2)
    n = 2**24 + 5
    for keys in (random_keys(dt, n, rng), (rng.integers(0, 1000, n)).astype(dt)):
        for consecutive in (False, True):
            run(keys, consecutive)


@pytest.mark.parametrize("dt", [np.dtype(np.uint64), np.dtype(np.int64), np.dtype(np.float64)], ids=lambda d: d.name)
def test_large_8_byte_keys(dt):
    # 2^22 + 3 records of 8-byte keys: the hybrid sort; 2^24 + 5: with its plan read back
    rng = np.random.default_rng(3)
    for n in (2**22 + 3, 2**24 + 5):
        keys = random_keys(dt, n, rng)
        keys[rng.integers(0, n, n // 3)] = keys[: n // 3]  # duplicates
        run(keys, False)
    run(float_specials(np.dtype(np.float64), 2**22 + 3, rng) if dt.kind == "f" else np.full(2**22 + 3, 5, dt), False)


@pytest.mark.parametrize("dt", [torch.uint8, torch.int8, torch.int16, torch.int32, torch.int64, torch.float32, torch.float64],
                         ids=str)
def test_matches_torch(dt):
    g = torch.Generator(device="cuda").manual_seed(4)
    for n in (1, 5000, 2**20 + 3):
        for hi in (3, 1000):
            x = torch.randint(0 if dt == torch.uint8 else -hi, hi, (n,), generator=g, device="cuda").to(dt)
            if dt.is_floating_point:
                x = x + 0.5  # (no +-0, no NaN: torch's equality and the library's agree)
            x2 = x.view(-1, 1) if n % 2 else x.view(2, -1)  # (the input is flattened; the inverse keeps its shape)
            for fn, ref in ((S.unique, lambda t, **kw: torch.unique(t, sorted=True, **kw)), (S.unique_consecutive, torch.unique_consecutive)):
                for inv in (False, True):
                    for cnt in (False, True):
                        got, want = fn(x2, return_inverse=inv, return_counts=cnt), ref(x2, return_inverse=inv, return_counts=cnt)
                        got = got if isinstance(got, tuple) else (got,)
                        want = want if isinstance(want, tuple) else (want,)
                        assert len(got) == len(want)
                        for a, b in zip(got, want):
                            assert a.shape == b.shape and a.dtype == b.dtype and torch.equal(a, b)


def _abi(x, key_type, num, consecutive, outs, stream=None, ws=None, ws_bytes=0):
    keys_ptr = x.data_ptr() if x is not None else None
    return S.lib().b200sort_unique(keys_ptr, key_type, num, consecutive, *outs, stream or torch.cuda.current_stream().cuda_stream,
                                   ws, ws_bytes)


class Guarded:
    """device outputs of num entries between guard bytes, filled with a sentinel"""
    G = 256

    def __init__(self, num, key_bytes, counts=True, inverse=True):
        self.num, self.kb = num, key_bytes
        self.bufs = {"keys": self._buf(num * key_bytes, key_bytes), "n_unique": self._buf(8, 8)}
        if counts:
            self.bufs["counts"] = self._buf(num * 8, 8)
        if inverse:
            self.bufs["inverse"] = self._buf(num * 8, 8)

    def _buf(self, nbytes, align):
        b = torch.full((nbytes + 2 * self.G + align,), 0xAB, dtype=torch.uint8, device="cuda")
        # (offset by `align` bytes: only as aligned as the type demands)
        return b, self.G + (align if align < 16 else 0)

    def ptr(self, name):
        if name not in self.bufs:
            return None
        b, off = self.bufs[name]
        return b.data_ptr() + off

    def outs(self):
        return [self.ptr(n) for n in ("keys", "counts", "inverse", "n_unique")]

    def region(self, name, nbytes):
        b, off = self.bufs[name]
        return host(b[off:off + nbytes])

    def check(self, ref, dt):
        """outputs equal the reference; entries >= U and guard bytes untouched"""
        for name, (b, off) in self.bufs.items():
            h = host(b)
            n_bytes = {"keys": self.num * self.kb, "n_unique": 8}.get(name, self.num * 8)
            assert (h[:off] == 0xAB).all() and (h[off + n_bytes:] == 0xAB).all(), f"guard bytes of {name} changed"
        U = len(ref[0])
        assert int(self.region("n_unique", 8).view(np.int64)[0]) == U
        k = self.region("keys", self.num * self.kb)
        assert k[:U * self.kb].tobytes() == ref[0].tobytes() and (k[U * self.kb:] == 0xAB).all()
        if "counts" in self.bufs:
            c = self.region("counts", self.num * 8)
            assert np.array_equal(c[:U * 8].view(np.int64), ref[2]) and (c[U * 8:] == 0xAB).all()
        if "inverse" in self.bufs:
            assert np.array_equal(self.region("inverse", self.num * 8).view(np.int64), ref[1])

    def untouched(self):
        return all((host(b) == 0xAB).all() for b, _ in self.bufs.values())


def test_memory_safety_through_the_c_abi():
    rng = np.random.default_rng(5)
    for dt in ALL_DTYPES:
        code = O.key_code(dt)
        for n in (1, TILE + 1, 3 * TILE + 5):
            keys = random_keys(dt, n, rng)
            keys[rng.integers(0, n, n // 2)] = keys[rng.integers(0, n, n // 2)]
            keys[n // 3: n // 3 + 50] = keys[n // 3]
            for consecutive in (0, 1):
                ref = reference(keys, consecutive)
                for counts, inverse in ((True, True), (False, False), (True, False)):
                    g = Guarded(n, dt.itemsize, counts, inverse)
                    kd = dev(keys)
                    assert _abi(kd, code, n, consecutive, g.outs()) == 0
                    torch.cuda.synchronize()
                    g.check(ref, dt)
                    assert host(kd).tobytes() == keys.tobytes()
            # consecutive mode: an input at element offset 1 (aligned only to its type)
            buf = dev(np.concatenate([keys[:1], keys]))
            view = buf[1:]
            ref = reference(keys, True)
            g = Guarded(n, dt.itemsize)
            assert _abi(view, code, n, 1, g.outs()) == 0
            torch.cuda.synchronize()
            g.check(ref, dt)
            run(keys, True, ref, kd=view)
            run(keys, False, kd=view)


def test_workspace():
    rng = np.random.default_rng(6)
    L = S.lib()
    n = 3 * TILE + 5
    keys = rng.integers(0, 500, n).astype(np.int32)
    kd = dev(keys)
    for consecutive in (0, 1):
        ref = reference(keys, consecutive)
        nbytes = S.unique_workspace_bytes(np.int32, n, bool(consecutive), True)
        # exactly the stated size
        ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        g = Guarded(n, 4)
        assert _abi(kd, 5, n, consecutive, g.outs(), ws=ws.data_ptr(), ws_bytes=nbytes) == 0
        torch.cuda.synchronize()
        g.check(ref, np.int32)
        # filled with garbage
        ws.random_(0, 256)
        g = Guarded(n, 4)
        assert _abi(kd, 5, n, consecutive, g.outs(), ws=ws.data_ptr(), ws_bytes=nbytes) == 0
        torch.cuda.synchronize()
        g.check(ref, np.int32)
        # 128 bytes past a 256-byte boundary: EINVAL; one byte short: ENOMEM; outputs untouched
        big = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
        g = Guarded(n, 4)
        assert _abi(kd, 5, n, consecutive, g.outs(), ws=big.data_ptr() + 128, ws_bytes=nbytes) == -1
        assert b"256-byte" in L.b200sort_last_error()
        assert _abi(kd, 5, n, consecutive, g.outs(), ws=ws.data_ptr(), ws_bytes=nbytes - 1) == -4
        torch.cuda.synchronize()
        assert g.untouched()
        # through Python
        run(keys, bool(consecutive), ref)
        out = (S.unique_consecutive if consecutive else S.unique)(kd, return_inverse=True, return_counts=True, workspace=ws)
        assert host(out[0]).tobytes() == ref[0].tobytes() and np.array_equal(host(out[1]), ref[1])
    # the cached workspace, reused across shapes (growing and shrinking)
    for n in (2**20 + 3, 17, 3 * TILE + 5, 2**21):
        keys = rng.integers(-50, 50, n).astype(np.int64)
        run(keys, False)
        run(keys, True)


def test_side_stream_stats_profile_and_empty():
    rng = np.random.default_rng(7)
    n = 2**20 + 3
    keys = rng.integers(0, 10_000, n).astype(np.float32)
    kd = dev(keys)
    refs = [reference(keys, c) for c in (False, True)]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    a = S.unique(kd, return_inverse=True, return_counts=True, stream=s.cuda_stream)
    b = S.unique_consecutive(kd, return_inverse=True, return_counts=True, stream=s.cuda_stream)
    s.synchronize()
    for got, ref in zip((a, b), refs):
        assert host(got[0]).tobytes() == ref[0].tobytes()
        assert np.array_equal(host(got[1]), ref[1]) and np.array_equal(host(got[2]), ref[2])
    for fn, sort_kinds in ((S.unique, True), (S.unique_consecutive, False)):
        fn(kd, return_counts=True)
        st = S.last_stats()
        assert st["algo"] == 5 and st["num"] == n and st["key_bytes"] == 4 and st["record_bytes"] == 4
        assert st["kernel_launches"] >= 2 and st["passes_planned"] == 0
        with S.options(profile=1):
            fn(kd, return_inverse=True, return_counts=True)
            kinds = [k for k, _ in S.last_profile()]
        assert "unique" in kinds
        assert ("sweep" in kinds and "hist" in kinds) == sort_kinds
        if not sort_kinds:
            assert set(kinds) == {"unique"}
    # num = 0: U = 0 is written, nothing else
    for consecutive in (0, 1):
        g = Guarded(0, 4)
        assert _abi(kd, 8, 0, consecutive, g.outs()) == 0
        torch.cuda.synchronize()
        assert int(g.region("n_unique", 8).view(np.int64)[0]) == 0
        assert S.last_stats()["algo"] == 5 and S.last_stats()["num"] == 0
        for fn in (S.unique, S.unique_consecutive):
            v, i, c = fn(torch.empty(0, dtype=torch.int32, device="cuda"), return_inverse=True, return_counts=True)
            assert v.numel() == 0 and i.numel() == 0 and c.numel() == 0


def test_host_arrays_are_refused():
    k0 = np.array([3, 1, 3, 3], np.int32)
    for keys in (k0, torch.from_numpy(k0)):
        for fn in (S.unique, S.unique_consecutive):
            with pytest.raises(S.B200SortError) as ei:
                fn(keys, return_counts=True)
            assert ei.value.code == -7
    # a host output with a device input
    kd = dev(k0)
    g = Guarded(4, 4)
    hout = np.full(4, -1, np.int64)
    outs = g.outs()
    outs[2] = hout.ctypes.data
    assert _abi(kd, 5, 4, 0, outs) == -7
    torch.cuda.synchronize()
    assert g.untouched() and (hout == -1).all()


def test_positions_above_2p32():
    n = 2**32 + 2**20
    ws = S.unique_workspace_bytes(np.uint8, n, False, True)
    need = ws + n * (1 + 1 + 8 + 8) + (8 << 30)
    S.lib().b200sort_release_cache()  # (what earlier tests left cached counts as free memory here)
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"needs {need / 2**30:.0f} GiB of device memory, {free / 2**30:.0f} GiB free")
    g = torch.Generator(device="cuda").manual_seed(8)
    x = torch.randint(0, 200, (n,), device="cuda", dtype=torch.uint8, generator=g)
    planted = torch.tensor([2**32, 2**32 + 1, 2**32 + 12345, n - 1], device="cuda")
    x[planted] = 250
    values, inverse, counts = S.unique(x, return_inverse=True, return_counts=True)
    chunk = 2**28
    hist = torch.zeros(256, dtype=torch.int64, device="cuda")
    for c in range(0, n, chunk):
        hist += torch.bincount(x[c:c + chunk].to(torch.int32), minlength=256)
    present = torch.nonzero(hist).flatten()
    assert torch.equal(values.to(torch.int64), present)
    assert torch.equal(counts, hist[present]) and int(hist[250]) == 4
    lut = torch.full((256,), -1, dtype=torch.int64, device="cuda")
    lut[present] = torch.arange(len(present), device="cuda")
    for c in range(0, n, chunk):
        assert torch.equal(inverse[c:c + chunk], lut[x[c:c + chunk].to(torch.int64)])
    st = S.last_stats()
    assert st["algo"] == 5 and st["num"] == n
