"""GPU tests (-m gpu) of the segmented sort (sort_segmented, sort_segmented_combined, sort_rows): every segment
sorted on its own, through every branch (tiny and medium segments in shared memory; keys of <= 4 bytes with a
segment longer than CAP as one composite-key sort; 8-byte keys with one whole-array sort per long segment).

Bar: inside every segment the key sequence is np.sort of the order-mapped keys byte for byte; the (key, payload)
multiset of every equal-key run of every segment is unchanged (so payloads match exactly on unique keys); the
bytes outside [offsets[0], offsets[-1]) are unchanged."""
import numpy as np
import pytest

import oracle_lib as O
import simd_radix_sort_b200 as S

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ALL_DTYPES = [np.dtype(d) for d in O.KEY_DTYPES]
CAP = {1: 16384, 2: 16384, 4: 16384, 8: 8192}  # longest segment sorted in shared memory, per key width


@pytest.fixture(scope="module", autouse=True)
def _loaded():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    before = S.launch_count()
    yield
    assert S.launch_count() > before, "no kernels of libb200sort.so were launched"


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def keys_of(dt, n, rng, specials=True):
    dt = np.dtype(dt)
    if dt.kind == "f":
        k = rng.standard_normal(n).astype(dt)
        if specials:
            sp = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, -np.nan], dtype=dt)
            m = rng.random(n) < 0.05
            k[m] = sp[rng.integers(0, len(sp), int(m.sum()))]
        return k
    info = np.iinfo(dt)
    hi = min(int(info.max), 1000) if rng.random() < 0.3 else int(info.max)  # some duplicate-heavy inputs
    return rng.integers(max(int(info.min), -hi - 1), hi, size=n, dtype=dt, endpoint=True)


def full_range_keys(dt, n, rng):
    """random bit patterns (for floats with +-0, +-inf and NaN among them): a long segment of these keys has digits
    below the hybrid path's cut, so its sort runs the segment finish"""
    k = rng.integers(0, 2**64, n, dtype=np.uint64).view(dt)
    if k.dtype.kind == "f":
        k[rng.integers(0, n, 15)] = np.repeat(np.array([0.0, -0.0, np.inf, -np.inf, np.nan]), 3)
    return k


def offsets_of(lengths, first=0):
    return np.concatenate([[first], first + np.cumsum(lengths)]).astype(np.int64)


def expected(keys, offsets, up):
    """(perm, runs): the permutation of the covered range that sorts every segment by the total order, ties by
    position, and the (segment, ordered key) rows of the result, whose equal runs the multiset check compares"""
    lo, hi = int(offsets[0]), int(offsets[-1])
    seg = np.repeat(np.arange(len(offsets) - 1), np.diff(offsets))
    kk = keys[lo:hi]
    ok = O.order_key(kk, up).astype(np.uint64)
    perm = np.lexsort((ok, seg))
    runs = np.ascontiguousarray(np.stack([seg.astype(np.uint64), ok[perm]], axis=1))
    return perm, runs


def check(keys_in, keys_out, pays_in, pays_out, offsets, up):
    lo, hi = int(offsets[0]), int(offsets[-1])
    perm, runs = expected(keys_in, offsets, up)
    assert keys_out[:lo].tobytes() == keys_in[:lo].tobytes() and keys_out[hi:].tobytes() == keys_in[hi:].tobytes()
    assert keys_out[lo:hi].tobytes() == keys_in[lo:hi][perm].tobytes()
    for pi, po in zip(pays_in, pays_out):
        assert po[:lo].tobytes() == pi[:lo].tobytes() and po[hi:].tobytes() == pi[hi:].tobytes()
    if pays_in:
        assert O.runs_multiset_equal(runs, [p[lo:hi] for p in pays_out], [p[lo:hi][perm] for p in pays_in])


def check_with_index(keys_in, keys_out, pays_in, pays_out, offsets, up):
    """check() for calls too large for the lexsort of expected().  pays_in[0] is the index np.arange(n), and pays_out[0]
    must be a permutation of the covered range that keeps every record in its segment, with keys_out == keys_in[idx]
    and the ordered keys non-decreasing inside every segment.  Equal ordered keys have equal bytes, so that is
    expected()'s key sequence byte for byte.  Every other payload must equal its input at that index."""
    lo, hi = int(offsets[0]), int(offsets[-1])
    for a, b in [(keys_in, keys_out)] + list(zip(pays_in, pays_out)):
        assert b[:lo].tobytes() == a[:lo].tobytes() and b[hi:].tobytes() == a[hi:].tobytes()
    seg = np.repeat(np.arange(len(offsets) - 1), np.diff(offsets))
    idx = pays_out[0][lo:hi].astype(np.int64)
    assert idx.min() >= lo and idx.max() < hi and np.all(np.bincount(idx - lo, minlength=hi - lo) == 1), "not a permutation"
    assert np.array_equal(seg[idx - lo], seg), "a record left its segment"
    assert keys_out[lo:hi].tobytes() == keys_in[idx].tobytes()
    ok = O.order_key(keys_out[lo:hi], up)
    assert np.all((ok[1:] >= ok[:-1]) | (seg[1:] != seg[:-1])), "a segment is not sorted"
    for pi, po in zip(pays_in[1:], pays_out[1:]):
        assert np.array_equal(po[lo:hi], pi[idx])


def odd_starts(lens, first, which):
    """lengthens the segment before each of `which` by one where needed, so that those segments start at odd records"""
    for j in sorted(which):
        if (first + int(lens[:j].sum())) % 2 == 0:
            lens[j - 1] += 1
    return offsets_of(lens, first)


def run_soa(keys, pays, offsets, up=True, on_device=True, **kw):
    if on_device:
        k, ps, o = dev(keys), [dev(p) for p in pays], dev(offsets)
        S.sort_segmented(o, k, *ps, up=up, **kw)
        torch.cuda.synchronize()
        return k.cpu().numpy(), [p.cpu().numpy() for p in ps]
    k, ps = keys.copy(), [p.copy() for p in pays]
    S.sort_segmented(offsets.copy(), k, *ps, up=up, **kw)
    return k, ps


def sort_and_check(keys, pays, offsets, up=True, on_device=True):
    k, ps = run_soa(keys, pays, offsets, up, on_device)
    check(keys, k, pays, ps, offsets, up)
    if len(keys) <= 1:  # (nothing to sort: a no-op that leaves the statistics alone)
        return None
    st = S.last_stats()
    assert st["algo"] == 3 and st["num"] == len(keys) and st["key_bytes"] == keys.dtype.itemsize
    assert st["kernel_launches"] >= 1
    return st


def mixed_lengths(rng, n_seg, longest=3000):
    lens = rng.integers(0, 40, n_seg)
    big = rng.random(n_seg) < 0.3
    lens[big] = rng.integers(33, longest, int(big.sum()))
    return lens


@pytest.mark.parametrize("dt", ALL_DTYPES, ids=lambda d: d.name)
def test_every_key_type_both_directions(dt):
    rng = np.random.default_rng(dt.num)
    for up in (True, False):
        lens = mixed_lengths(rng, 400)
        offsets = offsets_of(lens, first=3)
        n = int(offsets[-1]) + 5
        keys = keys_of(dt, n, rng)
        idx = np.arange(n, dtype=np.uint32)
        sort_and_check(keys, [idx], offsets, up)


@pytest.mark.parametrize("k", range(16))
def test_lengths_around_powers_of_two(k):
    """every power-of-two bin bound, each length in a call of its own (one segment above CAP would send a call
    with keys of <= 4 bytes down the composite branch)"""
    rng = np.random.default_rng(100 + k)
    for length in sorted({max(2**k - 1, 0), 2**k, 2**k + 1}):
        n_seg = max(3, (1 << 17) // max(length, 1))
        for dt in (np.uint32, np.uint64, ALL_DTYPES[k % len(ALL_DTYPES)]):
            dt = np.dtype(dt)
            lens = np.full(n_seg, length)
            lens[::7] = 0  # empty segments in between
            offsets = offsets_of(lens)
            keys = keys_of(dt, int(offsets[-1]), rng)
            pay = rng.integers(0, 2**63, len(keys), dtype=np.uint64)
            sort_and_check(keys, [pay], offsets, up=bool(length & 1))


def test_payload_shapes_and_unaligned_views():
    rng = np.random.default_rng(7)
    lens = mixed_lengths(rng, 300, longest=2500)
    offsets = offsets_of(lens)
    n = int(offsets[-1])
    for dt in (np.uint16, np.float32, np.int64):
        keys = keys_of(dt, n, rng)
        for shape in ([], [1], [2, 8, 16], [64], [1, 16, 64]):
            pays = [rng.integers(0, 256, (n, w), dtype=np.uint8) if w > 8 else rng.integers(0, 2**(8 * w), n, dtype=f"u{w}")
                    for w in shape]
            sort_and_check(keys, pays, offsets, up=len(shape) % 2 == 0)
    # 63 payload streams
    keys = keys_of(np.uint32, n, rng)
    pays = [((np.arange(n) + j) % 251).astype(np.uint8) for j in range(63)]
    sort_and_check(keys, pays, offsets)
    # unaligned views: keys[1:] and payloads[1:] of device arrays
    for dt in (np.uint32, np.uint64):
        keys = keys_of(dt, n + 1, rng)
        pay = np.arange(n + 1, dtype=np.uint64)
        kd, pd, od = dev(keys), dev(pay), dev(offsets)
        S.sort_segmented(od, kd[1:], pd[1:])
        torch.cuda.synchronize()
        got_k, got_p = kd.cpu().numpy(), pd.cpu().numpy()
        assert got_k[0] == keys[0] and got_p[0] == pay[0]
        check(keys[1:], got_k[1:], [pay[1:]], [got_p[1:]], offsets, True)


def test_records_of_every_power_of_two_size():
    rng = np.random.default_rng(9)
    lens = mixed_lengths(rng, 200, longest=2000)
    lens[5] = 20000  # one segment above CAP: composite branch for keys of <= 4 bytes, a whole-array sort for 8 bytes
    offsets = offsets_of(lens, first=2)
    n = int(offsets[-1]) + 3
    for dt in (np.uint8, np.int16, np.float32, np.float64):
        dt = np.dtype(dt)
        rb = dt.itemsize
        while rb <= 64:
            for offs in (offsets, offsets_of(np.minimum(lens, 3000), first=2)):
                keys = keys_of(dt, n, rng)
                rec = O.make_records(keys, rb)
                rec[:, dt.itemsize:] = rng.integers(0, 256, (n, rb - dt.itemsize), dtype=np.uint8)
                r = dev(rec)
                S.sort_segmented_combined(dev(offs), r, dt, up=rb != 8)
                got = r.cpu().numpy()
                gk = np.ascontiguousarray(got[:, :dt.itemsize]).reshape(-1).view(dt)
                check(keys, gk, [rec[:, dt.itemsize:].copy()] if rb > dt.itemsize else [],
                      [np.ascontiguousarray(got[:, dt.itemsize:])] if rb > dt.itemsize else [], offs, rb != 8)
            rb *= 2


@pytest.mark.parametrize("dt", [np.uint8, np.int16, np.uint32, np.float32], ids=lambda d: np.dtype(d).name)
def test_composite_branch(dt):
    dt = np.dtype(dt)
    rng = np.random.default_rng(dt.num + 50)
    lens = mixed_lengths(rng, 500)
    lens[[3, 77, 400]] = [CAP[dt.itemsize] + 1, 40000, 70000]
    offsets = offsets_of(lens, first=11)
    n = int(offsets[-1]) + 7
    keys = keys_of(dt, n, rng)
    for up in (True, False):
        sort_and_check(keys, [np.arange(n, dtype=np.int64), rng.integers(0, 256, (n, 3), dtype=np.uint8)], offsets, up)
        sort_and_check(keys, [], offsets, up)


def test_composite_branch_above_2p24():
    """u16 keys: 2^20 short segments and one long one, a span above 2^24 records from an odd offsets[0] (so the payload
    streams of the composite sort start at odd records); the segment index fills 20 bits of the composite key"""
    rng = np.random.default_rng(56)
    lens = rng.integers(0, 24, 1 << 20)
    lens[1000] = 5_000_000
    offsets = offsets_of(lens, first=7)
    assert offsets[-1] - offsets[0] >= 1 << 24
    n = int(offsets[-1]) + 5
    keys = keys_of(np.uint16, n, rng)
    pays = [np.arange(n, dtype=np.uint64), rng.integers(0, 256, (n, 12), dtype=np.uint8)]
    for up in (True, False):
        with S.options(profile=1):
            k, ps = run_soa(keys, pays, offsets, up)
        assert S.last_stats()["algo"] == 3
        check_with_index(keys, k, pays, ps, offsets, up)
        kinds = [kd for kd, _ in S.last_profile()]
        # the composite sort read its plan back: the smaller flow always launches one full segment finish; this one
        # launches none (nothing left below the cut) or the junction kernel and the gated finish
        assert "sweep" in kinds and kinds.count("segfix") in (0, 2), kinds


def test_sort_rows_matches_torch_sort_on_sampling_shape():
    """f32 rows are one composite-key sort of all rows: (64, 128256) below 2^24 records, whose sort launches one full
    segment finish, and (136, 128256) and (68, 250001) above, where that sort reads its plan back and launches none
    (nothing left below the cut) or two (the junction kernel and the gated finish).  f64 rows of odd length are one
    whole-array sort per row, every other row at 8 mod 16."""
    g = torch.Generator(device="cuda").manual_seed(3)
    for B, L, dt, n_segfix in ((64, 128256, torch.float32, (1,)), (136, 128256, torch.float32, (0, 2)), (68, 250001, torch.float32, (0, 2)),
                               (68, 250001, torch.float64, (0,))):
        logits = torch.randn(B, L, device="cuda", generator=g, dtype=dt)
        logits[:, :17] = logits[:, 17:34]  # duplicates inside every row
        for up in (False, True):
            want_v, _ = torch.sort(logits, dim=-1, descending=not up)
            idx = torch.arange(L, device="cuda", dtype=torch.int64).repeat(B, 1).contiguous()
            k = logits.clone()
            with S.options(profile=1):
                S.sort_rows(k, idx, up=up)
            torch.cuda.synchronize()
            assert torch.equal(k, want_v), (B, L, dt, up)
            assert torch.equal(torch.gather(logits, 1, idx), k), (B, L, dt, up)
            assert torch.equal(idx.sort(dim=-1).values, torch.arange(L, device="cuda").repeat(B, 1)), (B, L, dt, up)
            kinds = [kd for kd, _ in S.last_profile()]
            assert "sweep" in kinds and kinds.count("segfix") in n_segfix, (B, L, dt, kinds)
            del want_v, idx, k
    # the same through numpy host arrays, ascending
    logits = torch.randn(64, 128256, device="cuda", generator=g)
    idx = torch.arange(128256, dtype=torch.int64).repeat(4, 1).numpy()
    kh = logits[:4].cpu().numpy().copy()
    S.sort_rows(kh, idx)
    assert np.array_equal(kh, torch.sort(logits[:4], dim=-1).values.cpu().numpy())
    assert np.array_equal(np.take_along_axis(logits[:4].cpu().numpy(), idx, 1), kh)


@pytest.mark.parametrize("dt", [np.uint64, np.int64, np.float64], ids=lambda d: np.dtype(d).name)
def test_wide_keys_with_long_segments(dt):
    dt = np.dtype(dt)
    rng = np.random.default_rng(dt.num + 70)
    lens = mixed_lengths(rng, 600)
    lens[[10, 300, 599]] = [CAP[8] + 1, 50000, 120000]
    offsets = offsets_of(lens)
    keys = keys_of(dt, int(offsets[-1]), rng)
    for up in (True, False):
        sort_and_check(keys, [np.arange(len(keys), dtype=np.uint32), rng.integers(0, 2**60, len(keys), dtype=np.uint64)], offsets, up)


@pytest.mark.parametrize("dt", [np.int64, np.float64], ids=lambda d: np.dtype(d).name)
def test_wide_keys_with_hybrid_long_segments(dt):
    """8-byte keys: long segments of 2^22 + 5 and 2^24 + 3 records starting at odd records (8 mod 16), among short and
    CAP + 1 segments.  Their whole-array sorts take the hybrid path, the longer one reading its plan back: one
    "segfix" entry for the first, two (the junction kernel and the gated full segment finish) for the second."""
    dt = np.dtype(dt)
    rng = np.random.default_rng(dt.num + 90)
    lens = mixed_lengths(rng, 600)
    lens[[10, 200, 400, 599]] = [CAP[8] + 1, (1 << 22) + 5, (1 << 24) + 3, CAP[8] + 1]
    offsets = odd_starts(lens, 3, [200, 400])
    n = int(offsets[-1]) + 2
    keys = full_range_keys(dt, n, rng)
    pays = [np.arange(n, dtype=np.uint64), rng.integers(0, 2**16, n, dtype=np.uint16)]
    for up in (True, False):
        with S.options(profile=1):
            k, ps = run_soa(keys, pays, offsets, up)
        assert S.last_stats()["algo"] == 3
        check_with_index(keys, k, pays, ps, offsets, up)
        kinds = [kd for kd, _ in S.last_profile()]
        assert "sweep" in kinds and "segment" in kinds and kinds.count("segfix") == 3, kinds


def test_combined_records_with_a_hybrid_long_segment():
    """16-byte i64 records with one segment of 2^22 + 1 records at an odd start: its whole-array sort of records takes
    the hybrid path"""
    rng = np.random.default_rng(91)
    lens = mixed_lengths(rng, 300)
    lens[100] = (1 << 22) + 1
    offsets = odd_starts(lens, 1, [100])
    n = int(offsets[-1]) + 1
    keys = full_range_keys(np.int64, n, rng)
    rec = np.empty((n, 16), np.uint8)
    rec[:, :8] = keys.view(np.uint8).reshape(n, 8)
    rec[:, 8:] = np.arange(n, dtype=np.uint64).view(np.uint8).reshape(n, 8)
    r = dev(rec)
    with S.options(profile=1):
        S.sort_segmented_combined(dev(offsets), r, np.int64, up=False)
    got = r.cpu().numpy()
    assert S.last_stats()["algo"] == 3
    kinds = [kd for kd, _ in S.last_profile()]
    assert "sweep" in kinds and "segment" in kinds and kinds.count("segfix") == 1, kinds
    idx = np.ascontiguousarray(got[:, 8:]).view(np.uint64).reshape(-1)
    check_with_index(keys, np.ascontiguousarray(got[:, :8]).view(np.int64).reshape(-1), [np.arange(n, dtype=np.uint64), rec], [idx, got],
                     offsets, False)


def test_one_segment_equals_sort():
    rng = np.random.default_rng(12)
    for dt in (np.uint32, np.float64, np.int8):
        keys = keys_of(dt, 300_001, rng)
        a = dev(keys)
        b = dev(keys)
        S.sort(len(keys), a)
        S.sort_segmented(dev(np.array([0, len(keys)], np.int64)), b)
        torch.cuda.synchronize()
        assert a.cpu().numpy().tobytes() == b.cpu().numpy().tobytes()  # (bit patterns: the keys include NaNs)


@pytest.mark.parametrize("on_device", [True, False], ids=["device", "host"])
def test_invalid_offsets_move_nothing(on_device):
    rng = np.random.default_rng(13)
    n = 5000
    keys = keys_of(np.uint32, n, rng)
    pay = np.arange(n, dtype=np.uint32)
    good = offsets_of(np.full(100, 50))
    for bad in (good[::-1].copy(), np.concatenate([[-1], good[1:]]), np.concatenate([good[:-1], [n + 1]]),
                np.array([0, 40, 30, 100], np.int64)):
        with pytest.raises(S.B200SortError) as ei:
            run_soa(keys, [pay], bad.astype(np.int64), on_device=on_device)
        assert ei.value.code == -1
        if on_device:
            k, o, p = dev(keys), dev(bad.astype(np.int64)), dev(pay)
            with pytest.raises(S.B200SortError):
                S.sort_segmented(o, k, p)
            torch.cuda.synchronize()
            assert np.array_equal(k.cpu().numpy(), keys) and np.array_equal(p.cpu().numpy(), pay)
        else:
            k, p = keys.copy(), pay.copy()
            with pytest.raises(S.B200SortError):
                S.sort_segmented(bad.astype(np.int64), k, p)
            assert np.array_equal(k, keys) and np.array_equal(p, pay)


def test_host_arrays():
    rng = np.random.default_rng(14)
    for dt, longest in ((np.int32, 3000), (np.float64, 20000), (np.uint16, 30000)):
        lens = mixed_lengths(rng, 200, longest)
        offsets = offsets_of(lens, first=1)
        keys = keys_of(dt, int(offsets[-1]) + 1, rng)
        sort_and_check(keys, [np.arange(len(keys), dtype=np.uint64)], offsets, on_device=False)
    rec = O.make_records(keys_of(np.int64, 10000, rng), 16)
    offsets = offsets_of(np.full(100, 100))
    r = rec.copy()
    S.sort_segmented_combined(offsets, r, np.int64)
    kk = np.ascontiguousarray(r[:, :8]).reshape(-1).view(np.int64)
    check(np.ascontiguousarray(rec[:, :8]).reshape(-1).view(np.int64), kk, [rec[:, 8:].copy()], [np.ascontiguousarray(r[:, 8:])], offsets, True)


@pytest.mark.parametrize("dt", [np.uint32, np.uint64], ids=lambda d: np.dtype(d).name)
def test_caller_workspace(dt):
    rng = np.random.default_rng(15)
    lens = mixed_lengths(rng, 300)
    lens[7] = 20000
    offsets = offsets_of(lens)
    n = int(offsets[-1])
    keys = keys_of(dt, n, rng)
    pay = np.arange(n, dtype=np.uint32)
    need = S.segmented_workspace_bytes(dt, n, len(lens), [4])
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    k, ps = run_soa(keys, [pay], offsets, workspace=ws)
    check(keys, k, [pay], ps, offsets, True)
    short = ws[: need - 256]
    with pytest.raises(S.B200SortError) as ei:
        run_soa(keys, [pay], offsets, workspace=short)
    assert ei.value.code == -4
    # big enough, but 128 bytes past a 256-byte boundary: rejected, nothing moves
    big = torch.empty(need + 512, dtype=torch.uint8, device="cuda")
    off = (-big.data_ptr()) % 256 + 128
    k, p, o = dev(keys), dev(pay), dev(offsets)
    with pytest.raises(S.B200SortError) as ei:
        S.sort_segmented(o, k, p, workspace=big[off:])
    assert ei.value.code == -1
    assert k.cpu().numpy().tobytes() == keys.tobytes() and p.cpu().numpy().tobytes() == pay.tobytes()


def test_back_to_back_on_a_non_default_stream():
    rng = np.random.default_rng(16)
    s = torch.cuda.Stream()
    lens = mixed_lengths(rng, 1000)
    offsets = offsets_of(lens)
    n = int(offsets[-1])
    k1, k2 = keys_of(np.float32, n, rng), keys_of(np.uint64, n, rng)
    with torch.cuda.stream(s):
        a, b, o = dev(k1), dev(k2), dev(offsets)
        p = torch.arange(n, device="cuda", dtype=torch.int64)
        S.sort_segmented(o, a, p)
        S.sort_segmented(o, b, p, up=False)
    s.synchronize()
    ga, gp = a.cpu().numpy(), p.cpu().numpy()
    perm, _ = expected(k1, offsets, True)
    assert ga.tobytes() == k1[perm].tobytes()
    assert b.cpu().numpy().tobytes() == k2[expected(k2, offsets, False)[0]].tobytes()
    assert np.array_equal(np.sort(gp), np.arange(n))


def test_profile_records_the_segment_kernels():
    rng = np.random.default_rng(17)
    offsets = offsets_of(mixed_lengths(rng, 500))
    keys = keys_of(np.uint32, int(offsets[-1]), rng)
    with S.options(profile=1):
        run_soa(keys, [], offsets)
    kinds = [k for k, _ in S.last_profile()]
    assert "segment" in kinds


@pytest.mark.parametrize("on_device", [True, False], ids=["device", "host"])
def test_overlapping_offsets_are_rejected_before_anything_moves(on_device):
    """offsets that go back and forth: every other segment is valid on its own, and together they hold far more
    records than the array (more entries than the bin lists, and the long-segment list, have room for)"""
    rng = np.random.default_rng(18)
    for dt, length in ((np.uint32, 100), (np.uint64, 100), (np.uint64, 20000), (np.float32, 20000)):
        keys = keys_of(dt, length, rng)
        pay = np.arange(length, dtype=np.uint32)
        offsets = np.tile(np.array([0, length], np.int64), 500_001)[: 1_000_001]
        if on_device:
            k, p = dev(keys), dev(pay)
            with pytest.raises(S.B200SortError) as ei:
                S.sort_segmented(dev(offsets), k, p)
            torch.cuda.synchronize()
            k, p = k.cpu().numpy(), p.cpu().numpy()
        else:
            k, p = keys.copy(), pay.copy()
            with pytest.raises(S.B200SortError) as ei:
                S.sort_segmented(offsets, k, p)
        assert ei.value.code == -1, (dt, length)
        assert k.tobytes() == keys.tobytes() and np.array_equal(p, pay)
    # the library still works afterwards
    sort_and_check(keys_of(np.uint32, 5000, rng), [np.arange(5000, dtype=np.uint32)], offsets_of(np.full(50, 100)), on_device=on_device)


@pytest.mark.parametrize("on_device", [True, False], ids=["device", "host"])
def test_offsets_are_checked_when_nothing_can_move(on_device):
    for num in (0, 1):
        keys = np.arange(num, dtype=np.uint32)
        put = dev if on_device else (lambda a: a)
        S.sort_segmented(put(np.array([0, num, num], np.int64)), put(keys.copy()))  # valid: nothing to do
        for bad in ([0, 5], [0, num, 0, num] if num else [0, 2, 0], [-1, 0]):
            with pytest.raises(S.B200SortError) as ei:
                S.sort_segmented(put(np.array(bad, np.int64)), put(keys.copy()))
            assert ei.value.code == -1, (num, bad)


@pytest.mark.parametrize("dt", [np.uint32, np.uint64], ids=lambda d: np.dtype(d).name)
def test_profile_of_a_call_with_long_segments(dt):
    """a long segment runs whole-array sorts inside the call: its profile keeps the segment kernels' entries too"""
    rng = np.random.default_rng(19)
    lens = mixed_lengths(rng, 300)
    lens[4] = 40000
    offsets = offsets_of(lens)
    keys = keys_of(dt, int(offsets[-1]), rng)
    with S.options(profile=1):
        run_soa(keys, [np.arange(len(keys), dtype=np.uint32)], offsets)
    kinds = [k for k, _ in S.last_profile()]
    assert "other" in kinds and "sweep" in kinds, kinds  # classify (+ pack / unpack), the whole-array passes
    if np.dtype(dt).itemsize == 8:
        assert "segment" in kinds, kinds  # the short segments
