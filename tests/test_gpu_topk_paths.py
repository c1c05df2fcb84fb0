"""GPU tests (-m gpu) of every path of the top-k radix select, against tests/topk_model.py.

Rows of one call take different paths at once (read the candidate buffer, re-read the row, finish, done), many short
rows share the pass kernel's persistent CTAs and the decision kernel's grid-stride loop, candidate buckets sit exactly
at the buffer size or one above it, and outputs sit at addresses aligned only to their type.  Outputs are checked as
in test_gpu_topk.py.  Calls with a caller workspace are also checked white-box: after the call, the workspace holds
every row's TopkRow, which must equal the model's (all but item_base, which depends on the order of atomics), the
control block's work items of passes 1 … KB, which must equal the model's sum over the rows (this is where a pass
that re-read a row its buffer would have served shows), and the histograms, which must be all zero."""
import ctypes

import numpy as np
import pytest

import oracle_lib as O
import simd_radix_sort_b200 as S
import topk_model as M
from test_gpu_topk import check, dev, host, sorted_order

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ALL_DTYPES = [np.dtype(d) for d in O.KEY_DTYPES]


@pytest.fixture(scope="module", autouse=True)
def _loaded():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    before = S.launch_count()
    yield
    assert S.launch_count() > before, "no kernels of libb200sort.so were launched"


def check_state(ws, keys2d, k, largest, sel=None):
    """the selection state left in the caller workspace `ws` equals the model's"""
    B, L = keys2d.shape
    kb = keys2d.dtype.itemsize
    sel = M.select_keys(keys2d, k, largest) if sel is None else sel
    _, hist_off, ctrl_off = M.layout(B)
    head = host(ws[:ctrl_off + M.CTRL_BYTES])
    rows = head[:B * M.ROW_DTYPE.itemsize].view(M.ROW_DTYPE)
    for f in M.STATE_FIELDS:
        bad = np.nonzero(rows[f] != sel.state[f])[0]
        assert len(bad) == 0, (f"TopkRow.{f} of row {bad[0]} (of {len(bad)}) is {rows[f][bad[0]]}, the model's "
                               f"{sel.state[f][bad[0]]} (depth {sel.depth[bad[0]]}, {L} records, k {k})")
    items = head[ctrl_off:ctrl_off + M.CTRL_BYTES].view(np.uint64)
    want = np.zeros(M.MAX_PASSES, np.int64)
    want[:kb + 1] = sel.items.sum(axis=0)
    assert items.tolist() == want.tolist(), "work items per pass differ from the model's (a pass read more than it needed)"
    assert not head[hist_off:hist_off + B * M.RADIX * 8].any(), "a row's histogram is not zero after the call"


def run_ws(keys2d, k, largest, fill=None, order=None, sel=None, records=0):
    """topk (records > 0: topk_combined of records of that many bytes) with a caller workspace (filled with `fill`);
    outputs and the state checked"""
    B, L = keys2d.shape
    dt = keys2d.dtype
    nbytes = S.topk_workspace_bytes(dt, B, L, k, [], records)
    ws = (torch.empty if fill is None else lambda n, **kw: torch.full((n,), fill, **kw))(nbytes, dtype=torch.uint8, device="cuda")
    if records:
        rec = O.make_records(keys2d.reshape(-1), records).reshape(B, L, records)
        rd = dev(rec)
        out, idx = S.topk_combined(rd, dt, k, largest=largest, workspace=ws)
        out, idx = host(out), host(idx)
        assert host(rd).tobytes() == rec.tobytes()
        vals = np.ascontiguousarray(out[:, :, :dt.itemsize]).view(dt).reshape(B, k)
        check(keys2d, k, largest, vals, idx, [rec], [out], order)
    else:
        kd = dev(keys2d)
        vals, idx = S.topk(kd, k, largest=largest, workspace=ws)
        assert host(kd).tobytes() == keys2d.tobytes()
        check(keys2d, k, largest, host(vals), host(idx), order=order)
    check_state(ws, keys2d, k, largest, sel)


def mixed_k(L):
    return sorted({1, 33, L // 3, L - 1})


@pytest.mark.parametrize("L", [1000, 3 * 8192 + 5])
@pytest.mark.parametrize("dt", ALL_DTYPES, ids=lambda d: d.name)
def test_mixed_rows(dt, L):
    # row r from generator r % G: adjacent work items belong to rows in different modes; the odd row length makes
    # rows alternate between the vector and the scalar read path
    rng = np.random.default_rng(21)
    for largest in (True, False):
        for k in mixed_k(L):
            G = len(M.generators(dt, L, k))
            keys = M.mixed_rows(dt, 2 * G + 1, L, k, largest, rng)
            run_ws(keys, k, largest)


@pytest.mark.parametrize("dt", [np.dtype(d) for d in (np.uint8, np.int32, np.uint64, np.float64)], ids=lambda d: d.name)
def test_mixed_rows_records(dt):
    # 16-byte records: the strided read path
    rng = np.random.default_rng(22)
    for L in (1000, 3 * 8192 + 5):
        for largest, k in ((True, 33), (False, L // 3)):
            keys = M.mixed_rows(dt, len(M.generators(dt, L, k)) + 3, L, k, largest, rng)
            run_ws(keys, k, largest, records=16)


SHORT_SHAPES = [(5000, 1), (5000, 2), (4000, 15), (4000, 16), (4000, 17), (3000, 33), (20000, 100), (1300, 8192), (1300, 8193)]


@pytest.mark.parametrize("B,L", SHORT_SHAPES, ids=lambda x: str(x))
def test_many_short_rows(B, L):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert B > 8 * sms, "the decision kernel's grid must stride over the rows"
    rng = np.random.default_rng(23)
    for dt in (np.dtype(np.uint8), np.dtype(np.int16), np.dtype(np.float32), np.dtype(np.float64)):
        ks = sorted({1, 2, 32, 33, L // 2, L - 1, L} & set(range(1, L + 1)))
        for i, k in enumerate(ks):
            largest = (i + L) % 2 == 0
            # 64 or so distinct rows, row r from generator r % G; the others repeat them, and so do the model's
            # state and the reference order
            G = len(M.generators(dt, L, k))
            n = G * -(-64 // G)
            rep = np.arange(B) % n
            distinct = M.mixed_rows(dt, n, L, k, largest, rng)
            keys = distinct[rep]
            s = M.select_keys(distinct, k, largest)
            sel = M.Selection(s.kb, L, k, s.cap, s.state[rep], s.items[rep], s.depth[rep], s.reads[rep], ())
            run_ws(keys, k, largest, order=sorted_order(distinct, largest)[rep], sel=sel)


def test_a_million_rows_of_eight():
    # 2^20 segments of k = 3 through the ordering step's warp path (outputs only)
    rng = np.random.default_rng(24)
    keys = rng.integers(0, 2**32, (2**20, 8), dtype=np.uint64).astype(np.uint32)
    keys[::3, 5] = keys[::3, 2]  # ties
    for largest in (True, False):
        vals, idx = S.topk(dev(keys), 3, largest=largest)
        check(keys, 3, largest, host(vals), host(idx))


def test_workspace_hygiene():
    rng = np.random.default_rng(25)
    # a caller workspace full of garbage: the state regions are zeroed, the rest written before it is read
    for dt, L, k in ((np.dtype(np.float32), 1000, 33), (np.dtype(np.uint64), 3 * 8192 + 5, 1000), (np.dtype(np.int8), 20_000, 17)):
        for largest in (True, False):
            keys = M.mixed_rows(dt, 2 * len(M.generators(dt, L, k)), L, k, largest, rng)
            run_ws(keys, k, largest, fill=0xA5)
    # the cached workspace: a large call, then smaller ones of other shapes and key types
    for dt, B, L, k in ((np.float64, 64, 128256, 1000), (np.uint8, 7, 1000, 600), (np.int32, 3000, 33, 5)):
        keys = (rng.standard_normal((B, L)) * 100).astype(dt) if dt == np.float64 else \
            rng.integers(np.iinfo(dt).min, np.iinfo(dt).max, (B, L), dtype=dt, endpoint=True)
        for largest in (True, False):
            vals, idx = S.topk(dev(keys), k, largest=largest)
            check(keys, k, largest, host(vals), host(idx))


class Placed:
    """a device buffer of random guard bytes with an array of `nbytes` bytes at 256-byte boundary + `mod`"""
    def __init__(self, nbytes, mod, rng):
        self.init = rng.integers(0, 256, nbytes + 1024, dtype=np.uint8)
        self.buf = dev(self.init)
        self.off = 512 - self.buf.data_ptr() % 256 + mod
        self.nbytes = nbytes

    @property
    def ptr(self):
        return self.buf.data_ptr() + self.off

    def get(self):
        """-> the array's bytes; the guard bytes around it must be unchanged"""
        b = host(self.buf)
        o, e = self.off, self.off + self.nbytes
        assert b[:o].tobytes() == self.init[:o].tobytes() and b[e:].tobytes() == self.init[e:].tobytes(), \
            "a byte outside the output changed"
        return b[o:e].copy()


@pytest.mark.parametrize("dt", [np.dtype(d) for d in (np.uint8, np.int16, np.float32, np.uint64)], ids=lambda d: d.name)
def test_unaligned_outputs(dt):
    """through the C ABI: out_keys at key width mod 16, out_index at 8 mod 16, payload outputs of 1, 2 and 12 bytes at
    element offset 1 and of 16 bytes at 8 mod 16; k = 2 (warp segments), 33 (one CTA per segment) and above the
    segmented sort's CAP (long segments), so every branch of the ordering step writes a misaligned out_keys"""
    rng = np.random.default_rng(26)
    L = 40_000 if dt.itemsize < 8 else 20_000
    B = 3
    cap = 16384 if dt.itemsize <= 4 else 8192
    kb = dt.itemsize
    keys = M.mixed_rows(dt, B, L, 33, True, rng)
    kd = dev(keys)
    sizes = (1, 2, 12, 16)
    pays = [rng.integers(0, 256, (B, L, s), dtype=np.uint8) for s in sizes]
    pd = [dev(p) for p in pays]
    lib = S.lib()
    stream = torch.cuda.current_stream().cuda_stream
    for k in (2, 33, cap + 17):
        for largest in (True, False):
            ok = Placed(B * k * kb, kb % 16, rng)
            oi = Placed(B * k * 8, 8, rng)
            op = [Placed(B * k * s, s if s < 16 else 8, rng) for s in sizes]
            ptrs = (ctypes.c_void_p * 4)(*[p.data_ptr() for p in pd])
            esz = (ctypes.c_uint32 * 4)(*sizes)
            outs = (ctypes.c_void_p * 4)(*[o.ptr for o in op])
            rc = lib.b200sort_topk_soa(kd.data_ptr(), O.key_code(dt), B, L, k, int(largest), 4, ptrs, esz, ok.ptr, oi.ptr, outs,
                                       stream, None, 0)
            assert rc == 0, lib.b200sort_last_error()
            torch.cuda.synchronize()
            vals = ok.get().view(dt).reshape(B, k)
            idx = oi.get().view(np.int64).reshape(B, k)
            check(keys, k, largest, vals, idx, pays, [o.get().reshape(B, k, s) for o, s in zip(op, sizes)])
            # AoS 16-byte records at 8 mod 16
            rec = O.make_records(keys.reshape(-1), 16).reshape(B, L, 16)
            rd = dev(rec)
            orec, oi2 = Placed(B * k * 16, 8, rng), Placed(B * k * 8, 8, rng)
            rc = lib.b200sort_topk_aos(rd.data_ptr(), O.key_code(dt), 16, B, L, k, int(largest), orec.ptr, oi2.ptr, stream, None, 0)
            assert rc == 0, lib.b200sort_last_error()
            torch.cuda.synchronize()
            out = orec.get().reshape(B, k, 16)
            vals = np.ascontiguousarray(out[:, :, :kb]).view(dt).reshape(B, k)
            check(keys, k, largest, vals, oi2.get().view(np.int64).reshape(B, k), [rec], [out])
