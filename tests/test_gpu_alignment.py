"""GPU tests (-m gpu) of arrays that are aligned to their element type but not to 16 bytes, through every sort flow.

A caller gets such arrays without doing anything unusual: `x[1:]`, `narrow()`, a byte view of a record buffer, or a
segment of a segmented sort.  The library picks kernel branches from the addresses: vector or one-key-per-load key
tiles in the probe and histogram sweeps, the chunk width each stream moves in (which also decides whether 4-byte
keys may take the 8192-key wide tiles), TMA key tiles, the L2 column prefetch and the paired 16-byte stores only
when both sides of the ping-pong are aligned, and the scalar branch of the copy-back.

Every case places each array at a chosen address mod 16 inside a buffer with guard bytes on both sides, and checks:
- the key bytes equal numpy's total-order sort (oracle_lib.total_order_sorted_keys) exactly;
- the index payload is a permutation and keys[idx] is the sorted key sequence;
- every other payload equals its input row at that index;
- the guard bytes before and after every array are unchanged;
- through S.last_stats(), that the flow the case targets really ran."""
import ctypes

import numpy as np
import pytest

import oracle_lib as O
import simd_radix_sort_b200 as S

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ALL_DTYPES = [np.dtype(d) for d in O.KEY_DTYPES]
GUARD = 64  # bytes before and after every array
EINVAL = -1
# (keys misaligned, payloads misaligned)
VARIANTS = {"keys": (True, False), "payloads": (False, True), "both": (True, True)}
# the address mod 16 of a misaligned array, by element width: aligned to the element, not to 16 bytes
MISALIGN = {1: 1, 2: 6, 4: 4, 8: 8, 12: 12, 16: 8}


@pytest.fixture(scope="module", autouse=True)
def _loaded():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    before = S.launch_count()
    yield
    assert S.launch_count() > before, "no kernels of libb200sort.so were launched"


class Placed:
    """A copy of a numpy array at an address that is `mis` mod 16, in a device (or host) byte buffer with GUARD random
    bytes on either side.  `view` is what the sort gets: a torch tensor (or numpy array) of the array's dtype and
    shape; `result()` reads the array back and checks the guard bytes."""

    def __init__(self, a, mis, rng, on_device=True):
        a = np.ascontiguousarray(a)
        self.dtype, self.shape, nb = a.dtype, a.shape, a.nbytes
        size = nb + 2 * GUARD + 16
        if on_device:
            self.buf = torch.empty(size, dtype=torch.uint8, device="cuda")
            base = self.buf.data_ptr()
        else:
            self.buf = np.empty(size, np.uint8)
            base = self.buf.ctypes.data
        self.off = GUARD + (mis - base - GUARD) % 16
        self.nb = nb
        self.init = rng.integers(0, 256, size, dtype=np.uint8)
        self.init[self.off:self.off + nb] = a.reshape(-1).view(np.uint8)
        if on_device:
            self.buf.copy_(torch.from_numpy(self.init))
            self.view = self.buf[self.off:self.off + nb].view(getattr(torch, a.dtype.name)).view(a.shape)
        else:
            self.buf[:] = self.init
            self.view = self.buf[self.off:self.off + nb].view(a.dtype).reshape(a.shape)
        assert (self.addr() - mis) % 16 == 0

    def addr(self):
        return self.view.data_ptr() if isinstance(self.view, torch.Tensor) else self.view.ctypes.data

    def result(self):
        got = self.buf.cpu().numpy() if isinstance(self.buf, torch.Tensor) else self.buf
        assert got[:self.off].tobytes() == self.init[:self.off].tobytes(), "guard bytes before the array changed"
        assert got[self.off + self.nb:].tobytes() == self.init[self.off + self.nb:].tobytes(), "guard bytes after the array changed"
        return got[self.off:self.off + self.nb].copy().view(self.dtype).reshape(self.shape)


def keys_of(dt, n, rng, dups=True):
    """random bit patterns of every kind (NaNs of many payloads for floats), plus three each of +-0, +-inf and NaN,
    and (dups) one value 64 times.  (Without dups for the flows asserted to end without the full segment finish: a
    run of equal keys among other keys that share its leading bits is longer than the last pass orders.)"""
    dt = np.dtype(dt)
    k = rng.integers(0, 256, n * dt.itemsize, dtype=np.uint8).view(dt)
    if dt.kind == "f":
        sp = np.array([0.0, -0.0, np.inf, -np.inf, np.nan], dtype=dt)
        k[rng.integers(0, n, 3 * len(sp))] = np.repeat(sp, 3)
    if dups:
        k[rng.integers(0, n, 64)] = k[0]
    return k


def payload_of_width(w, n, rng):
    if w in (1, 2, 4, 8):
        return rng.integers(0, 2**(8 * w), n, dtype=f"u{w}")
    return rng.integers(0, 256, (n, w), dtype=np.uint8)


def width_of(a):
    return a.dtype.itemsize * (a.shape[1] if a.ndim > 1 else 1)


def sort_placed(keys, pays, key_mis, pay_mis, up, rng, on_device=True):
    """sorts `keys` (first payload: the index) placed at key_mis / pay_mis[i] mod 16; checks the result, returns the
    statistics"""
    n = len(keys)
    pk = Placed(keys, key_mis, rng, on_device)
    pp = [Placed(p, m, rng, on_device) for p, m in zip(pays, pay_mis)]
    S.sort(n, pk.view, *[p.view for p in pp], up=up)
    if on_device:
        torch.cuda.synchronize()
    st = S.last_stats()
    out_k = pk.result()
    out_p = [p.result() for p in pp]
    want = O.total_order_sorted_keys(keys, up)
    assert out_k.tobytes() == want.tobytes(), (keys.dtype, n, up, key_mis, pay_mis)
    idx = out_p[0].astype(np.int64)
    assert idx.min() >= 0 and idx.max() < n and np.all(np.bincount(idx, minlength=n) == 1), "index payload is not a permutation"
    assert keys[idx].tobytes() == out_k.tobytes()
    for i, (pi, po) in enumerate(zip(pays[1:], out_p[1:])):
        assert np.array_equal(po, pi[idx]), (f"payload {i + 1} ({width_of(pi)} bytes)", key_mis, pay_mis)
    assert st["num"] == n and st["key_bytes"] == keys.dtype.itemsize
    return st


def variant_addresses(variant, keys, pays):
    """(key address mod 16, [payload addresses mod 16]) of one alignment variant"""
    mk, mp = VARIANTS[variant]
    return MISALIGN[keys.dtype.itemsize] if mk else 0, [MISALIGN[width_of(p)] if mp else 0 for p in pays]


PAYLOAD_WIDTHS = (1, 2, 4, 8, 12, 16)


@pytest.mark.parametrize("dt", ALL_DTYPES, ids=lambda d: d.name)
def test_lsd_path(dt):
    """the digit-by-digit path at 300,001 records; 1-byte keys end after one pass in the shadow arrays, so the copy-back
    moves every stream (the scalar branch for the misaligned ones)"""
    n = 300_001
    rng = np.random.default_rng(dt.num)
    keys = keys_of(dt, n, rng)
    for variant in VARIANTS:
        for up in (True, False):
            idx = np.arange(n, dtype=np.uint32 if up else np.uint64)
            pays = [idx] + [payload_of_width(w, n, rng) for w in PAYLOAD_WIDTHS]
            km, pm = variant_addresses(variant, keys, pays)
            st = sort_placed(keys, pays, km, pm, up, rng)
            assert st["algo"] == 1, st


def test_wide_tiles_for_4_byte_keys():
    """4-byte keys at 2^24 + 4097 with default options: 8192-key wide tiles are chosen for 4-byte keys when every
    stream moves in chunks of <= 4 bytes, from 2^24 records; the plan is read back.  The 8-byte payload lies at 4 mod
    16 in every variant, so it moves in 4-byte chunks: that is what makes the sort eligible for the wide tiles."""
    n = (1 << 24) + 4097
    assert S.get_option("wide_tiles") == 1 and S.get_option("tile_cfg") == -1 and S.get_option("max_chunk") >= 8
    assert n >= 1 << S.get_option("host_plan_min_log2")
    rng = np.random.default_rng(24)
    keys = keys_of(np.float32, n, rng)
    for variant, up in zip(VARIANTS, (True, False, True)):
        pays = [np.arange(n, dtype=np.uint32), rng.integers(0, 256, (n, 8), dtype=np.uint8)]
        km, pm = variant_addresses(variant, keys, pays)
        pm[1] = 4
        st = sort_placed(keys, pays, km, pm, up, rng)
        assert st["algo"] == 1 and st["record_bytes"] == 16 and st["passes_planned"] <= 4, st


@pytest.mark.parametrize("host_plan", [False, True], ids=["2p22", "2p24_host_plan"])
def test_hybrid_path_8_byte_keys(host_plan):
    """8-byte keys with default options on the MSB hybrid path: at 2^22 + 4099 the full segment finish orders the final
    segments; at 2^24 + 4099 the plan is read back, the last pass orders the tile-local segments and the junction
    kernel the tile-straddling ones, with no full segment finish"""
    n = (1 << 24) + 4099 if host_plan else (1 << 22) + 4099
    assert (n >= 1 << S.get_option("host_plan_min_log2")) == host_plan and S.get_option("algo") == 0
    rng = np.random.default_rng(22 + host_plan)
    widths = (12, 2) if host_plan else PAYLOAD_WIDTHS  # (2^24 records: fewer payload bytes)
    for variant, (dt, up) in zip(VARIANTS, ((np.float64, True), (np.int64, False), (np.uint64, True))):
        keys = keys_of(dt, n, rng, dups=not host_plan)
        idx = np.arange(n, dtype=np.uint32 if up else np.uint64)
        pays = [idx] + [payload_of_width(w, n, rng) for w in widths]
        km, pm = variant_addresses(variant, keys, pays)
        st = sort_placed(keys, pays, km, pm, up, rng)
        assert st["algo"] == 2 and st["fell_back"] == 0 and st["cut_digit"] >= 2, st
        assert st["segfix_passes"] == (0 if host_plan else 1), st


@pytest.mark.parametrize("dt", [np.int64, np.float64], ids=lambda d: np.dtype(d).name)
def test_records_at_8_mod_16(dt):
    """AoS records of 8, 16, 32 and 64 bytes taken from a flat byte buffer at byte 8, so that records of 16 bytes or
    more sit at 8 mod 16, on the hybrid path (2^22 + 4099 records), with and without the plan read back"""
    n = (1 << 22) + 4099
    rng = np.random.default_rng(np.dtype(dt).num + 8)
    keys = keys_of(dt, n, rng, dups=False)
    for rb, host_plan, up in ((8, False, True), (16, True, False), (32, False, False), (64, True, True)):
        rec = rng.integers(0, 256, (n, rb), dtype=np.uint8)
        rec[:, :8] = keys.view(np.uint8).reshape(n, 8)
        if rb > 8:
            rec[:, 8:16] = np.arange(n, dtype=np.uint64).view(np.uint8).reshape(n, 8)
        r = Placed(rec, 8, rng)
        with S.options(host_plan_min_log2=0 if host_plan else 24):
            S.sort_combined(n, r.view, dt, up=up)
        torch.cuda.synchronize()
        st = S.last_stats()
        assert st["algo"] == 2 and st["record_bytes"] == rb and st["fell_back"] == 0, (rb, st)
        assert st["segfix_passes"] == (0 if host_plan else 1), (rb, st)
        out = r.result()
        got_k = np.ascontiguousarray(out[:, :8]).view(dt).reshape(-1)
        assert got_k.tobytes() == O.total_order_sorted_keys(keys, up).tobytes(), (rb, up)
        if rb > 8:
            idx = np.ascontiguousarray(out[:, 8:16]).view(np.uint64).reshape(-1).astype(np.int64)
            assert np.all(np.bincount(idx, minlength=n) == 1), rb
            assert np.array_equal(out, rec[idx]), rb  # whole records travelled


def test_host_arrays_at_an_odd_element_offset():
    """host numpy arrays at element offset 1 (>= 2^20 records with payloads): the pipelined staging sorts the keys with
    a 4-byte index while the payloads upload, then gathers the payloads"""
    n = (1 << 20) + 12345
    rng = np.random.default_rng(20)
    for dt, up in ((np.float32, False), (np.uint64, True), (np.int16, True)):
        keys = keys_of(dt, n, rng)
        for variant in VARIANTS:
            pays = [np.arange(n, dtype=np.uint64)] + [payload_of_width(w, n, rng) for w in (2, 12, 1)]
            km, pm = variant_addresses(variant, keys, pays)
            st = sort_placed(keys, pays, km, pm, up, rng, on_device=False)
            assert st["record_bytes"] == np.dtype(dt).itemsize + 4, st  # (keys + index: the pipelined path)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


@pytest.mark.parametrize("dt,byte_off", [(np.uint32, 2), (np.int64, 4), (np.float64, 2), (np.int16, 1)],
                         ids=["u32_at_2", "i64_at_4", "f64_at_2", "i16_at_1"])
def test_key_array_misaligned_to_its_type_is_rejected(dt, byte_off):
    """keys at an address that is not a multiple of their own size: B200SORT_EINVAL, and nothing moved, through
    b200sort_sort_soa, b200sort_sort_aos and b200sort_sort_segmented_soa"""
    dt = np.dtype(dt)
    kb = dt.itemsize
    n = 300_001
    rng = np.random.default_rng(kb + byte_off)
    L = S.lib()
    k = Placed(rng.integers(0, 256, n * 16 + 16, dtype=np.uint8), 0, rng)  # (room for n // 4 records of 16 bytes too)
    p = Placed(np.arange(n, dtype=np.uint64), 8, rng)
    offsets = Placed(np.array([0, 5, n // 2, n], np.int64), 0, rng)
    key_addr = ctypes.c_void_p(k.addr() + byte_off)
    ptrs = (ctypes.c_void_p * 1)(p.addr())
    sizes = (ctypes.c_uint32 * 1)(8)
    code = S.KEY_TYPES[dt.name]
    rc = L.b200sort_sort_soa(key_addr, code, n, 1, 1, ptrs, sizes, _stream(), None, 0)
    assert rc == EINVAL, (rc, L.b200sort_last_error())
    rc = L.b200sort_sort_aos(key_addr, code, 16, n // 4, 1, _stream(), None, 0)
    assert rc == EINVAL, (rc, L.b200sort_last_error())
    rc = L.b200sort_sort_segmented_soa(key_addr, code, n, 3, ctypes.c_void_p(offsets.addr()), 1, 1, ptrs, sizes, _stream(), None, 0)
    assert rc == EINVAL, (rc, L.b200sort_last_error())
    torch.cuda.synchronize()
    for a in (k, p, offsets):
        assert a.result().tobytes() == a.init[a.off:a.off + a.nb].tobytes()
