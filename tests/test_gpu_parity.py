"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI (simd_radix_sort_b200 -> ctypes ->
libb200sort.so), against the golden vectors produced by the compiled reference, against the oracle on
seeded inputs, and through size-independent properties at larger sizes.

Bar: bit-exact key sequence; payloads exact where determined by the key, else the same
(key, payload) multiset per equal-key run (the reference is not stable)."""
import hashlib
import json

import numpy as np
import pytest

import oracle_lib as O
import simd_radix_sort_b200 as S

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ALL_DTYPES = [np.dtype(d) for d in O.KEY_DTYPES]


def dev(a: np.ndarray):
    return torch.from_numpy(a).cuda()


def host(t) -> np.ndarray:
    return t.cpu().numpy()


def gpu_sort_soa(keys: np.ndarray, payloads, up=True, on_device=True):
    """returns (sorted keys, [payloads]) as numpy; on_device=False exercises the host-staging path"""
    if on_device:
        k = dev(keys)
        ps = [dev(p) for p in payloads]
        S.sort(len(keys), k, *ps, up=up)
        torch.cuda.synchronize()
        return host(k), [host(p) for p in ps]
    k = keys.copy()
    ps = [p.copy() for p in payloads]
    S.sort(len(k), k, *ps, up=up)
    return k, ps


@pytest.fixture(scope="module", autouse=True)
def _loaded():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    assert S.lib_path().exists(), "libb200sort.so must be built (no fallback)"
    before = S.launch_count()
    yield
    assert S.launch_count() > before, "no kernels of libb200sort.so were launched"


def test_golden_soa_all_types(golden_dir):
    z = np.load(golden_dir / "soa_keys.npz")
    n_cases = 0
    for name in z.files:
        if not name.startswith("in|"):
            continue
        _, dt, up, dist, n = name.split("|")
        keys = z[name]
        want = z["out|" + name[3:]]
        idx = np.arange(len(keys), dtype=np.uint32)
        got, (perm,) = gpu_sort_soa(keys, [idx], bool(int(up)))
        if np.dtype(dt).kind == "f" and int(n) <= 16:
            # reference quirk (SURVEY 8a): <= 16 elements are insertion-sorted with IEEE compare; inputs
            # hold no -0.0 there, so the byte patterns agree anyway
            pass
        assert got.tobytes() == want.tobytes(), name
        assert np.array_equal(np.sort(perm), idx), name
        assert keys[perm].tobytes() == got.tobytes(), name
        n_cases += 1
    assert n_cases >= 10 * 2 * 6 * 7


def test_golden_aos_all_record_sizes(golden_dir):
    z = np.load(golden_dir / "aos_records.npz")
    n_cases = 0
    for name in z.files:
        if not name.startswith("inkeys|"):
            continue
        _, dt, rb, up, dist, n = name.split("|")
        rec = O.make_records(z[name], int(rb))
        want = O.make_records(z["outkeys|" + name[7:]], int(rb))
        r = dev(rec)
        S.sort_combined(len(rec), r, np.dtype(dt), up=bool(int(up)))
        assert host(r).tobytes() == want.tobytes(), name
        n_cases += 1
    assert n_cases > 100


def test_config1_u32_u32_1m_matches_reference_hashes(golden_dir):
    gold = json.loads((golden_dir / "golden_c1.json").read_text())
    for n_str, g in gold.items():
        k, p = O.c1_input(int(n_str), 42)
        gk, (gp,) = gpu_sort_soa(k, [p], True)
        assert gk[:3].tolist() == g["sorted_head"] and int(gk[-1]) == g["sorted_tail"]
        assert hashlib.sha256(gk.tobytes()).hexdigest() == g["sha256_sorted_keys"]
        assert hashlib.sha256(gp.tobytes()).hexdigest() == g["sha256_sorted_payloads"]
        assert O.check_payloads(gk, [gp])


@pytest.mark.parametrize("dt", ALL_DTYPES, ids=lambda d: d.name)
def test_against_oracle_port_shapes_and_distributions(dt):
    """the (type x shape x distribution x direction) matrix of src/test.cpp:100-179 at n = 1..3000"""
    shapes = [[], [np.uint8], [np.uint16], [np.uint32], [np.uint64], [np.uint64, np.uint8], [np.uint64, np.uint64],
              [np.uint64] * 3, [np.uint32, np.float64, np.uint16], [np.uint8] * 7]
    for up in (True, False):
        for dist in O.DISTRIBUTIONS:
            for n in (1, 10, 100, 3000):
                keys = O.make_keys(dist, dt, n, seed=n + 11)
                if dt.kind == "f" and n <= 16:
                    keys = np.where(keys == 0, dt.type(0), keys)
                shape = shapes[(n + len(dist)) % len(shapes)]
                pay = [(np.arange(n) * 7 + j).astype(s) for j, s in enumerate(shape)]
                k_o, p_o = keys.copy(), [p.copy() for p in pay]
                O.port_sort_soa(k_o, p_o, up)
                k_g, p_g = gpu_sort_soa(keys, pay, up)
                assert k_g.tobytes() == k_o.tobytes(), (dist, n, up)
                assert O.runs_multiset_equal(k_o, p_o, p_g), (dist, n, up)


def test_63_payload_streams_and_wide_payloads():
    # src/test.cpp:124-137: 63 x uint8 payload streams
    n = 5000
    keys = O.make_keys("Uniform", np.uint16, n, seed=1)
    pay = [((np.arange(n) + j) % 251).astype(np.uint8) for j in range(63)]
    k_o, p_o = keys.copy(), [p.copy() for p in pay]
    O.port_sort_soa(k_o, p_o, True)
    k_g, p_g = gpu_sort_soa(keys, pay, True)
    assert k_g.tobytes() == k_o.tobytes() and O.runs_multiset_equal(k_o, p_o, p_g)
    # 16/32/64-byte payload elements (multi-register payload vectors in the reference, src/simd.hpp:47-74)
    for width in (16, 32, 64):
        keys = O.make_keys("Gaussian", np.int32, n, seed=width)
        rows = np.random.default_rng(width).integers(0, 255, size=(n, width), dtype=np.uint8)
        k, p = dev(keys), dev(rows)
        S.sort(n, k, p, up=False)
        kg, pg = host(k), host(p)
        order = np.argsort(O.order_key(keys, False), kind="stable")
        assert kg.tobytes() == keys[order].tobytes()
        assert O.runs_multiset_equal(kg, [np.ascontiguousarray(pg)], [np.ascontiguousarray(rows[order])])


def test_float_specials_order():
    for dt in (np.float32, np.float64):
        a = np.array([0.0, -0.0, np.inf, -np.inf, 1.0, -1.0, 5e-324, -5e-324, 3.5, -3.5] * 5, dtype=dt)
        for up in (True, False):
            k_o = a.copy()
            O.port_sort_soa(k_o, [], up)
            k_g, _ = gpu_sort_soa(a, [], up)
            assert k_g.tobytes() == k_o.tobytes()


def test_host_pointer_staging_path():
    for dt, n in ((np.uint32, 100_000), (np.float64, 33_333)):
        keys = O.make_keys("Uniform", dt, n, seed=9)
        idx = np.arange(n, dtype=np.uint64)
        k, (p,) = gpu_sort_soa(keys, [idx], True, on_device=False)
        assert k.tobytes() == O.total_order_sorted_keys(keys, True).tobytes()
        assert keys[p].tobytes() == k.tobytes() and np.array_equal(np.sort(p), idx)


def test_empty_and_one_record():
    """(arrays that are not 16-byte aligned: tests/test_gpu_alignment.py)"""
    for n in (0, 1):
        k = dev(np.arange(5, dtype=np.int64))
        S.sort(n, k)
        assert host(k).tolist() == [0, 1, 2, 3, 4]


@pytest.mark.parametrize("case", ["u64_u64", "f32_3streams_desc", "aos_i64_f64_fewunique", "u32_u32", "i64_zipf"])
def test_large_properties(case):
    """larger sizes: sortedness, permutation (payload = index), key multiset via checksums; oracle = numpy"""
    n = 1 << 22
    rng = np.random.default_rng(123)
    if case == "u64_u64":
        keys = rng.integers(0, 2**64, size=n, dtype=np.uint64)
        k, (p,) = gpu_sort_soa(keys, [np.arange(n, dtype=np.uint64)], True)
        assert k.tobytes() == np.sort(keys).tobytes() and keys[p].tobytes() == k.tobytes()
        assert np.array_equal(np.sort(p), np.arange(n, dtype=np.uint64))
    elif case == "u32_u32":
        keys = rng.integers(0, 2**32, size=n, dtype=np.uint32)
        k, (p,) = gpu_sort_soa(keys, [np.arange(n, dtype=np.uint32)], True)
        assert k.tobytes() == np.sort(keys).tobytes() and keys[p].tobytes() == k.tobytes()
    elif case == "f32_3streams_desc":  # BASELINE.json config 3 shape
        keys = rng.uniform(-1, 1, size=n).astype(np.float32)
        keys[:8 * 100_003:100_003] = [0.0, -0.0, np.inf, -np.inf, 1e-45, -1e-45, 3.4e38, -3.4e38]  # SURVEY 8d edge set
        i32 = np.arange(n, dtype=np.int32)
        f64 = np.arange(n, dtype=np.float64)
        u16 = (np.arange(n) % 65536).astype(np.uint16)
        k, (a, b, c) = gpu_sort_soa(keys, [i32, f64, u16], False)
        assert k.tobytes() == O.total_order_sorted_keys(keys, False).tobytes()
        assert keys[a].tobytes() == k.tobytes() and np.array_equal(b, a.astype(np.float64))
        assert np.array_equal(c, (a % 65536).astype(np.uint16))
    elif case == "aos_i64_f64_fewunique":  # BASELINE.json config 4 shape: DataElement<int64,double>
        keys = rng.integers(-8, 8, size=n, dtype=np.int64)
        rec = np.zeros((n, 16), np.uint8)
        rec[:, :8] = keys.view(np.uint8).reshape(n, 8)
        rec[:, 8:] = np.arange(n, dtype=np.float64).view(np.uint8).reshape(n, 8)
        r = dev(rec)
        S.sort_combined(n, r, np.int64, up=True)
        out = host(r)
        ok = np.ascontiguousarray(out[:, :8]).reshape(-1).view(np.int64)
        op = np.ascontiguousarray(out[:, 8:]).reshape(-1).view(np.float64).astype(np.int64)
        assert ok.tobytes() == np.sort(keys).tobytes()
        assert np.array_equal(keys[op], ok) and np.array_equal(np.sort(op), np.arange(n))
    else:
        ranks = np.minimum((rng.pareto(1.0, size=n)).astype(np.int64), (1 << 20) - 1)
        table = rng.integers(-2**63, 2**63 - 1, size=1 << 20, dtype=np.int64)
        keys = table[ranks]
        k, (p,) = gpu_sort_soa(keys, [np.arange(n, dtype=np.uint32)], True)
        assert k.tobytes() == np.sort(keys).tobytes() and keys[p].tobytes() == k.tobytes()


def test_tile_geometries_agree():
    """both tile geometries of the scatter kernel"""
    n = 300_000
    keys = O.make_keys("Uniform", np.uint64, n, seed=77)
    want = np.sort(keys)
    for cfg in range(2):
        with S.options(tile_cfg=cfg):
            k, (p,) = gpu_sort_soa(keys, [np.arange(n, dtype=np.uint32)], True)
            assert k.tobytes() == want.tobytes(), cfg
            assert keys[p].tobytes() == k.tobytes(), cfg


def test_wide_tiles_for_4_byte_keys():
    """8192-key tiles (tile geometry 2): chosen automatically for 4-byte keys with <= 4-byte chunks from 2^24 records
    (test_gpu_large covers that size), forced here at sizes with full, partial and single tiles"""
    with S.options(tile_cfg=2):
        for n in (5, 8191, 8193, 300_000, (1 << 22) + 4099):
            for dt, up in ((np.uint32, True), (np.float32, False), (np.int32, False)):
                keys = O.make_keys("Uniform" if n % 2 else "Gaussian", dt, n, seed=n % 97)
                a, b = np.arange(n, dtype=np.uint32), (np.arange(n) % 251).astype(np.uint8)
                for big in (24, 0):
                    with S.options(host_plan_min_log2=big):
                        k, (pa, pb) = gpu_sort_soa(keys, [a, b], up)
                        assert k.tobytes() == O.total_order_sorted_keys(keys, up).tobytes(), (n, dt, up, big)
                        assert keys[pa].tobytes() == k.tobytes() and np.array_equal(np.sort(pa), a), (n, dt, up, big)
                        assert np.array_equal(pb, (pa % 251).astype(np.uint8)), (n, dt, up, big)


@pytest.mark.parametrize("max_chunk", [1, 2, 4, 8])
def test_max_chunk_below_the_key_width(max_chunk):
    """option max_chunk narrower than the key: payloads move in chunks that narrow, keys and whole records never in
    chunks narrower than the key (large-sort flow, whose lean kernels read the key from the record's first chunk)"""
    n = (1 << 20) + 77
    rng = np.random.default_rng(max_chunk)
    with S.options(host_plan_min_log2=0, max_chunk=max_chunk):
        keys = rng.integers(0, 2**64, size=n, dtype=np.uint64)
        keys[::13] = keys[7]  # duplicates of one value
        idx = np.arange(n, dtype=np.uint64)
        k, (p,) = gpu_sort_soa(keys, [idx], True)
        assert k.tobytes() == O.total_order_sorted_keys(keys, True).tobytes()
        assert np.array_equal(np.sort(p), idx) and keys[p.astype(np.int64)].tobytes() == k.tobytes()
        rk = rng.integers(-2**63, 2**63 - 1, size=n, dtype=np.int64)
        rec = np.zeros((n, 16), np.uint8)
        rec[:, :8] = rk.view(np.uint8).reshape(n, 8)
        rec[:, 8:] = np.arange(n, dtype=np.int64).view(np.uint8).reshape(n, 8)
        r = dev(rec)
        S.sort_combined(n, r, np.int64, up=True)
        out = host(r)
        ok = np.ascontiguousarray(out[:, :8]).reshape(-1).view(np.int64)
        op = np.ascontiguousarray(out[:, 8:]).reshape(-1).view(np.int64)
        assert ok.tobytes() == O.total_order_sorted_keys(rk, True).tobytes()
        assert np.array_equal(np.sort(op), np.arange(n)) and np.array_equal(rk[op], ok)


@pytest.mark.parametrize("first_atomic", [0, 1])
def test_unstable_first_pass_ranking(first_atomic):
    """large-sort flow: the first executed pass may rank with one shared-memory atomic per key (unstable);
    every later pass stays stable -- same result either way, payloads follow their keys"""
    n = (1 << 20) + 4099
    rng = np.random.default_rng(5 + first_atomic)
    with S.options(host_plan_min_log2=0, first_atomic=first_atomic, algo=2):
        for dt in (np.uint64, np.int64, np.float64):
            keys = O.make_keys("Uniform", dt, n, seed=21)
            keys[::11] = keys[5]  # duplicates of one value
            for up in (True, False):
                idx = np.arange(n, dtype=np.uint64)
                k, (p,) = gpu_sort_soa(keys, [idx], up)
                assert k.tobytes() == O.total_order_sorted_keys(keys, up).tobytes(), (dt, up)
                assert np.array_equal(np.sort(p), idx) and keys[p.astype(np.int64)].tobytes() == k.tobytes(), (dt, up)


@pytest.mark.parametrize("up", [True, False])
def test_last_pass_window_at_tile_edges_with_32_bit_cut(up):
    """ADVICE r1 (high): with the cut at bit 32 the swept bits are the raw high word; a key whose high word is 1
    sits in the first (ascending) / last (descending) slot of its tile, where the window of the tile-local
    ordering looks one slot outside the tile.  Slots outside the tile must never pair with a key."""
    n = (1 << 20) + 4099
    rng = np.random.default_rng(32)
    with S.options(algo=2, host_plan_min_log2=0, margin_bits=11):  # log2(n) + 11 = 31.01 -> four swept digits, cut at bit 32
        hi = rng.integers(0, 2**32, size=n, dtype=np.uint64)
        # plenty of keys with raw high word 1 (and 0, 2: neighbours), in runs so that they also meet in one tile
        hi[rng.integers(0, n, size=n // 8)] = 1
        hi[rng.integers(0, n, size=n // 16)] = 0
        hi[rng.integers(0, n, size=n // 16)] = 2
        lo = rng.integers(0, 2**32, size=n, dtype=np.uint64)
        keys = (hi << np.uint64(32)) | lo
        idx = np.arange(n, dtype=np.uint32)
        for dt in (np.uint64, np.int64):
            kk = np.ascontiguousarray(keys.view(dt))
            k, (p,) = gpu_sort_soa(kk, [idx], up)
            st = S.last_stats()
            assert st["algo"] == 2
            assert k.tobytes() == O.total_order_sorted_keys(kk, up).tobytes(), (dt, up)
            assert np.array_equal(np.sort(p), idx) and kk[p].tobytes() == k.tobytes(), (dt, up)
        # sparse version: exactly the edge keys, unique low words (cut digit 4 is checked)
        keys2 = (rng.integers(0, 2**32, size=n, dtype=np.uint64) << np.uint64(32)) | lo
        keys2[:4096] = (np.uint64(1) << np.uint64(32)) | np.arange(4096, dtype=np.uint64)[::-1]
        k, (p,) = gpu_sort_soa(keys2, [idx], up)
        assert S.last_stats()["cut_digit"] == 4, S.last_stats()
        assert k.tobytes() == O.total_order_sorted_keys(keys2, up).tobytes()
        assert kk is not None and keys2[p].tobytes() == k.tobytes()


def test_caller_workspace_and_stats():
    n = 200_000
    keys = O.make_keys("Uniform", np.int64, n, seed=5)
    ws = torch.empty(S.workspace_bytes(np.int64, n, [8]) + 512, dtype=torch.uint8, device="cuda")
    off = (-ws.data_ptr()) % 256
    k, p = dev(keys), dev(np.arange(n, dtype=np.int64))
    S.sort(n, k, p, up=False, workspace=ws[off:])
    assert host(k).tobytes() == np.sort(keys)[::-1].tobytes()
    st = S.last_stats()
    assert st["num"] == n and st["record_bytes"] == 16 and st["kernel_launches"] > 0
    small = torch.empty(1024, dtype=torch.uint8, device="cuda")
    with pytest.raises(S.B200SortError) as ei:
        S.sort(n, k, p, workspace=small)
    assert ei.value.code == -4
    # big enough, but 128 bytes past a 256-byte boundary: rejected, nothing moves
    k0, p0 = host(k), host(p)
    with pytest.raises(S.B200SortError) as ei:
        S.sort(n, k, p, workspace=ws[off + 128:])
    assert ei.value.code == -1
    assert host(k).tobytes() == k0.tobytes() and host(p).tobytes() == p0.tobytes()


# ------------------------------------------------------------------------------------------------
# MSB hybrid path (8-byte keys): top-digit sweeps + in-shared-memory segment finish
# ------------------------------------------------------------------------------------------------
def _hybrid_cases(n, rng):
    u = rng.integers(0, 2**64, size=n, dtype=np.uint64)
    yield "uniform_u64", u, np.uint64
    yield "uniform_i64", u.view(np.int64).copy(), np.int64
    yield "f64_uniform", rng.uniform(-1, 1, size=n), np.float64
    yield "f64_gauss", rng.normal(0, 1, size=n), np.float64
    yield "i64_gauss100", np.round(rng.normal(0, 100, size=n)).astype(np.int64), np.int64
    yield "few_unique", rng.integers(-8, 8, size=n, dtype=np.int64), np.int64
    yield "zero", np.zeros(n, np.int64), np.int64
    yield "zero_one", rng.integers(0, 2, size=n).astype(np.uint64), np.uint64
    table = rng.integers(-2**63, 2**63 - 1, size=1 << 12, dtype=np.int64)
    yield "dups_of_4096_values", table[rng.integers(0, 1 << 12, size=n)], np.int64
    yield "sorted", np.sort(u), np.uint64
    yield "small_range_u64", rng.integers(0, 1 << 20, size=n, dtype=np.uint64), np.uint64
    # top digits look high-entropy but are a function of a group id: medium (100) and long (1000) buckets
    # with distinct keys -> rank loop, resp. the fall-back to the digit-by-digit path
    for glen, tag in ((100, "medium_segments"), (1000, "long_segments_fallback")):
        g = np.arange(n) // glen
        f = rng.integers(0, 2**32, size=g.max() + 1, dtype=np.uint64)
        yield tag, (f[g] << np.uint64(32)) | rng.integers(0, 2**32, size=n, dtype=np.uint64), np.uint64


@pytest.mark.parametrize("n", [1, 17, 2049, 300_000, (1 << 20) + 77])
def test_hybrid_msb_path_matches_total_order(n):
    rng = np.random.default_rng(n)
    with S.options(algo=2):
        for name, keys, dt in _hybrid_cases(n, rng):
            keys = np.ascontiguousarray(keys.astype(dt))
            for up in (True, False):
                idx = np.arange(n, dtype=np.uint32)
                k, (p,) = gpu_sort_soa(keys, [idx], up)
                want = O.total_order_sorted_keys(keys, up)
                assert k.tobytes() == want.tobytes(), (name, n, up)
                assert np.array_equal(np.sort(p), idx) and keys[p].tobytes() == k.tobytes(), (name, n, up)
            if name == "long_segments_fallback" and n >= 300_000:
                assert S.last_stats()["fell_back"] == 1
            if name == "uniform_u64" and n >= 300_000:
                st = S.last_stats()
                assert st["algo"] == 2 and st["fell_back"] == 0 and st["cut_digit"] >= 2 and st["segfix_passes"] == 1


def test_hybrid_aos_and_multi_stream():
    n = 500_000
    rng = np.random.default_rng(5)
    with S.options(algo=2):
        keys = rng.integers(-2**63, 2**63 - 1, size=n, dtype=np.int64)
        keys[::7] = keys[3]  # duplicates
        rec = np.zeros((n, 32), np.uint8)
        rec[:, :8] = keys.view(np.uint8).reshape(n, 8)
        rec[:, 8:16] = np.arange(n, dtype=np.int64).view(np.uint8).reshape(n, 8)
        r = dev(rec)
        S.sort_combined(n, r, np.int64, up=False)
        out = host(r)
        ok = np.ascontiguousarray(out[:, :8]).reshape(-1).view(np.int64)
        op = np.ascontiguousarray(out[:, 8:16]).reshape(-1).view(np.int64)
        assert ok.tobytes() == np.sort(keys)[::-1].tobytes()
        assert np.array_equal(keys[op], ok) and np.array_equal(np.sort(op), np.arange(n))
        # SoA with three payload streams incl. a 2-byte one (ANYCHUNK instantiations)
        fk = rng.uniform(-1, 1, size=n)
        a, b, c = np.arange(n, dtype=np.int32), np.arange(n, dtype=np.float64), (np.arange(n) % 65536).astype(np.uint16)
        k, (pa, pb_, pc) = gpu_sort_soa(fk, [a, b, c], True)
        assert k.tobytes() == np.sort(fk).tobytes() and fk[pa].tobytes() == k.tobytes()
        assert np.array_equal(pb_, pa.astype(np.float64)) and np.array_equal(pc, (pa % 65536).astype(np.uint16))


# ------------------------------------------------------------------------------------------------
# Large-sort flow (host reads the plan back; the last pass orders tile-local segments, junction_fix_kernel
# the tile-straddling ones): forced at test sizes with host_plan_min_log2 = 0
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,margin", [(300_000, 2), ((1 << 20) + 77, 2), ((1 << 20) + 77, -2), ((1 << 20) + 77, -5)])
def test_hybrid_host_plan_tile_local_ordering_and_junctions(n, margin):
    rng = np.random.default_rng(n + margin)
    with S.options(algo=2, host_plan_min_log2=0, margin_bits=margin):
        for name, keys, dt in _hybrid_cases(n, rng):
            keys = np.ascontiguousarray(keys.astype(dt))
            for up in (True, False):
                idx = np.arange(n, dtype=np.uint32)
                k, (p,) = gpu_sort_soa(keys, [idx], up)
                want = O.total_order_sorted_keys(keys, up)
                assert k.tobytes() == want.tobytes(), (name, n, up)
                assert np.array_equal(np.sort(p), idx) and keys[p].tobytes() == k.tobytes(), (name, n, up)
            if name == "uniform_u64" and margin == 2:
                st = S.last_stats()  # no full segment finish: the last pass and the junction kernel did it
                assert st["algo"] == 2 and st["fell_back"] == 0 and st["cut_digit"] >= 2 and st["segfix_passes"] == 0


def test_hybrid_host_plan_aos_and_multi_stream():
    n = (1 << 19) + 4099
    rng = np.random.default_rng(77)
    with S.options(algo=2, host_plan_min_log2=0, margin_bits=-2):  # about four keys per final segment: plenty of runs and junctions
        for rec_bytes in (16, 32, 64):
            keys = rng.integers(-2**63, 2**63 - 1, size=n, dtype=np.int64)
            keys[::5] = keys[1::5][: len(keys[::5])]  # duplicates
            rec = np.zeros((n, rec_bytes), np.uint8)
            rec[:, :8] = keys.view(np.uint8).reshape(n, 8)
            rec[:, 8:16] = np.arange(n, dtype=np.int64).view(np.uint8).reshape(n, 8)
            if rec_bytes > 16:
                rec[:, 16:] = (np.arange(n)[:, None] * 7 + np.arange(rec_bytes - 16)[None, :]).astype(np.uint8)
            for up in (True, False):
                r = dev(rec)
                S.sort_combined(n, r, np.int64, up=up)
                out = host(r)
                ok = np.ascontiguousarray(out[:, :8]).reshape(-1).view(np.int64)
                op = np.ascontiguousarray(out[:, 8:16]).reshape(-1).view(np.int64)
                assert ok.tobytes() == O.total_order_sorted_keys(keys, up).tobytes(), (rec_bytes, up)
                assert np.array_equal(np.sort(op), np.arange(n)) and np.array_equal(keys[op], ok)
                assert np.array_equal(out, rec[op]), (rec_bytes, up)  # whole records travelled
        fk = rng.uniform(-1, 1, size=n)
        a, b, c = np.arange(n, dtype=np.int32), np.arange(n, dtype=np.float64), (np.arange(n) % 65536).astype(np.uint16)
        for up in (True, False):
            k, (pa, pb_, pc) = gpu_sort_soa(fk, [a, b, c], up)
            assert k.tobytes() == O.total_order_sorted_keys(fk, up).tobytes() and fk[pa].tobytes() == k.tobytes()
            assert np.array_equal(pb_, pa.astype(np.float64)) and np.array_equal(pc, (pa % 65536).astype(np.uint16))


@pytest.mark.parametrize("host_plan", [0, 24])
def test_hybrid_left_shift_plan_for_common_leading_bits(host_plan):
    """keys that agree on a few leading bits (a shard of a multi-GPU sort): the plan shifts them out and
    needs one pass less; same result either way"""
    n = 3 << 18
    rng = np.random.default_rng(9)
    body = rng.integers(0, 2**58, size=n, dtype=np.uint64)
    passes = {}
    with S.options(algo=2, host_plan_min_log2=host_plan, margin_bits=-1):
        for name, keys in (("u64_top6", body | np.uint64(0b101011 << 58)),
                           ("i64_neg", (body | np.uint64(0b111111 << 58)).view(np.int64)),
                           ("f64", (body >> np.uint64(2) | np.uint64(0x3FF << 52)).view(np.float64))):
            keys = np.ascontiguousarray(keys)
            for allow in (1, 0):
                with S.options(allow_lshift=allow):
                    for up in (True, False):
                        idx = np.arange(n, dtype=np.uint32)
                        k, (p,) = gpu_sort_soa(keys, [idx], up)
                        assert k.tobytes() == O.total_order_sorted_keys(keys, up).tobytes(), (name, allow, up)
                        assert np.array_equal(np.sort(p), idx) and keys[p].tobytes() == k.tobytes(), (name, allow, up)
                    passes[(name, allow)] = S.last_stats()["passes_planned"]
        assert passes[("u64_top6", 1)] < passes[("u64_top6", 0)], passes


@pytest.mark.parametrize("pinned", [False, True])
def test_host_arrays_pipelined_staging(pinned):
    """host SoA arrays, >= 2^20 records: keys are sorted with an index while the payloads upload, payloads are
    permuted afterwards (pageable and pinned host memory take different issue orders)"""
    n = (1 << 20) + 12345
    rng = np.random.default_rng(31)
    for dt, up in ((np.uint64, True), (np.float32, False), (np.int16, True)):
        keys = O.make_keys("Uniform", dt, n, seed=3)
        pays = [np.arange(n, dtype=np.uint64), (np.arange(n) % 65521).astype(np.uint16),
                rng.integers(0, 255, size=(n, 12), dtype=np.uint8)]  # 8-, 2- and 12-byte payload elements
        if pinned:
            tk = torch.from_numpy(keys.copy()).pin_memory()
            tp = [torch.from_numpy(p.copy()).pin_memory() for p in pays]
            k, ps = tk.numpy(), [t.numpy() for t in tp]
        else:
            k, ps = keys.copy(), [p.copy() for p in pays]
        before = S.launch_count()
        L = S.lib()
        import ctypes
        ptrs = (ctypes.c_void_p * 3)(*[p.ctypes.data for p in ps])
        sizes = (ctypes.c_uint32 * 3)(8, 2, 12)
        rc = L.b200sort_sort_soa(ctypes.c_void_p(k.ctypes.data), S.KEY_TYPES[np.dtype(dt).name], n, int(up), 3, ptrs, sizes, None, None, 0)
        assert rc == 0, L.b200sort_last_error()
        assert S.launch_count() > before
        want = O.total_order_sorted_keys(keys, up)
        assert k.tobytes() == want.tobytes(), (dt, up, pinned)
        src = ps[0].astype(np.int64)
        assert np.array_equal(np.sort(src), np.arange(n)) and keys[src].tobytes() == k.tobytes()
        assert np.array_equal(ps[1], (src % 65521).astype(np.uint16))
        assert np.array_equal(ps[2], pays[2][src])


# ------------------------------------------------------------------------------------------------
# SURVEY 8(f) rank 3: the advanced overload sort<Up, BitSorter, CmpSorterNoSort>(thresh, ...) -- buckets of at most
# `thresh` elements stay unordered (src/radix_sort.hpp:279, src/cmp_sorters.hpp:66-78).  On the GPU: the digit
# sweeps run, the segment finish does not (a key-only check replaces it).
# ------------------------------------------------------------------------------------------------
def _within_thresh_of_sorted(out_o, sorted_o, thresh):
    """every element is less than `thresh` places away from a position where the full sort could have put it"""
    n = len(out_o)
    lo = sorted_o[np.maximum(np.arange(n) - (thresh - 1), 0)]
    hi = sorted_o[np.minimum(np.arange(n) + (thresh - 1), n - 1)]
    return bool(np.all((out_o >= lo) & (out_o <= hi)))


@pytest.mark.parametrize("thresh", [16, 64, 4])
def test_cmp_sorter_none_partial_sort_contract(thresh):
    n = (1 << 20) + 333
    rng = np.random.default_rng(thresh)
    CMP_NONE = 1
    with S.options(algo=2,            # (the MSB hybrid path is the default from 2^22 records)
                   host_plan_min_log2=0,
                   margin_bits=-2):   # about four keys per final segment: plenty of unordered small buckets
        for dt, up in ((np.uint64, True), (np.int64, False), (np.float64, True)):
            keys = O.make_keys("Uniform", dt, n, seed=9 + thresh)
            idx = np.arange(n, dtype=np.uint32)
            k, p = dev(keys), dev(idx)
            before = S.launch_count()
            S.sort(n, k, p, up=up, cmp_sort_threshold=thresh, cmp_sorter=CMP_NONE)
            torch.cuda.synchronize()
            st = S.last_stats()
            hk, hp = host(k), host(p)
            assert np.array_equal(np.sort(hp), idx) and keys[hp].tobytes() == hk.tobytes()      # a permutation, payloads follow
            so = O.order_key(O.total_order_sorted_keys(keys, up), up)
            assert _within_thresh_of_sorted(O.order_key(hk, up), so, max(thresh, 1)), (dt, up, thresh)
            if thresh >= 8:
                # the early-out really happened: no segment finish, and the result is NOT the full sort
                assert st["algo"] == 2 and st["segfix_passes"] == 0 and st["cut_digit"] >= 2, st
                assert hk.tobytes() != O.total_order_sorted_keys(keys, up).tobytes()
            else:
                assert hk.tobytes() == O.total_order_sorted_keys(keys, up).tobytes()              # small thresholds: full sort
        # a segment longer than the threshold (1000 distinct keys sharing all swept bits) must still be sorted
        g = np.arange(n) // 1000
        f = rng.integers(0, 2**32, size=g.max() + 1, dtype=np.uint64)
        keys = (f[g] << np.uint64(32)) | rng.integers(0, 2**32, size=n, dtype=np.uint64)
        k = dev(keys)
        S.sort(n, k, up=True, cmp_sort_threshold=max(thresh, 8), cmp_sorter=CMP_NONE)
        torch.cuda.synchronize()
        hk = host(k)
        so = np.sort(keys)
        assert np.array_equal(np.sort(hk), so) and _within_thresh_of_sorted(hk, so, max(thresh, 8))
        # AoS entry point
        rec = O.make_records(O.make_keys("Uniform", np.int64, n, seed=3), 16)
        r = dev(rec)
        L = S.lib()
        import ctypes
        rc = L.b200sort_sort_aos_ex(ctypes.c_void_p(r.data_ptr()), S.KEY_TYPES["int64"], 16, n, 1, 32, CMP_NONE,
                                    ctypes.c_void_p(torch.cuda.current_stream().cuda_stream), None, 0)
        assert rc == 0, L.b200sort_last_error()
        torch.cuda.synchronize()
        out = host(r)
        ok = np.ascontiguousarray(out[:, :8]).reshape(-1).view(np.int64)
        assert _within_thresh_of_sorted(O.order_key(ok, True), O.order_key(np.sort(ok), True), 32)
        assert out.tobytes() == O.make_records(ok, 16).tobytes()   # records stayed whole
