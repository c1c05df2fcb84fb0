"""GPU tests (-m gpu) of the pass plan: key sets shaped to reach each branch of scan_kernel's plan, for keys of 1, 2, 4
and 8 bytes, with the plan made on the device and read back on the host, checked against numpy and against the
exact plan model of tests/plan_model.py.

A wrong plan does not fault: it skips a digit some keys differ in, subtracts something other than the smallest key, or
sweeps too few digits, and the array comes out wrongly ordered for key sets of one shape only.  Each case here checks:
- the key bytes equal numpy's total-order sort exactly;
- the index payload is a permutation and keys[idx] is the sorted key sequence;
- every other payload (2- and 12-byte rows) equals its input row at idx; AoS records travel whole;
- with the plan read back (host_plan_min_log2=0): passes_planned, hist_sweeps and kernel_launches equal the model, which
  proves the branch the case aims at was taken; with the plan on the device: every pass and hist_kernel launched.

Then keys the probe's sparse sample cannot see (section "sampled probe"), and every documented single-GPU option
value against the same inputs (section "options")."""
import numpy as np
import pytest

import oracle_lib as O
import simd_radix_sort_b200 as S
from plan_model import from_order, lsd_plan

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ALL_DTYPES = [np.dtype(d) for d in O.KEY_DTYPES]
FLOWS = {"device_plan": 24, "host_plan": 0}  # host_plan_min_log2


@pytest.fixture(scope="module", autouse=True)
def _loaded():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    before = S.launch_count()
    yield
    assert S.launch_count() > before, "no kernels of libb200sort.so were launched"


def udtype(kb):
    return np.dtype(f"uint{8 * kb}")


def rand_bits(rng, kb, n):
    return rng.integers(0, 256, n * kb, dtype=np.uint8).view(udtype(kb))


def sorted_keys(keys, up):
    """numpy's total-order sort of `keys` (the order of oracle_lib.order_key)"""
    return from_order(np.sort(O.order_key(keys, up)), keys.dtype, up)


def to_dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def check_soa(keys, pays, out_k, out_p, want):
    """key bytes exact, index a permutation that reproduces them, every other payload row follows its key"""
    n = len(keys)
    assert out_k.tobytes() == want.tobytes(), "keys are not in numpy's order"
    idx = out_p[0].astype(np.int64)
    assert len(idx) == n and np.all(np.bincount(idx, minlength=n) == 1), "index payload is not a permutation"
    assert keys[idx].tobytes() == out_k.tobytes(), "index payload does not follow the keys"
    for i, (p, po) in enumerate(zip(pays[1:], out_p[1:])):
        assert np.array_equal(po, p[idx]), f"payload {i + 1} does not follow the keys"


def sort_soa(keys, pays, up, **opts):
    """sorts device copies of keys + payloads under `opts`; -> (keys, payloads, stats)"""
    k = to_dev(keys)
    ps = [to_dev(p) for p in pays]
    with S.options(**opts):
        S.sort(len(keys), k, *ps, up=up)
    torch.cuda.synchronize()
    st = S.last_stats()
    return k.cpu().numpy(), [p.cpu().numpy() for p in ps], st


def records_of(keys, rng, rb=16):
    """AoS records of rb bytes: the key at offset 0, a u32 index at offset 8, random bytes elsewhere"""
    n, kb = len(keys), keys.dtype.itemsize
    rec = rng.integers(0, 256, (n, rb), dtype=np.uint8)
    rec[:, :kb] = keys.view(np.uint8).reshape(n, kb)
    rec[:, 8:12] = np.arange(n, dtype=np.uint32).view(np.uint8).reshape(n, 4)
    return rec


def sort_and_check_aos(keys, rec, up, want, **opts):
    n, kb = len(keys), keys.dtype.itemsize
    r = to_dev(rec)
    with S.options(**opts):
        S.sort_combined(n, r, keys.dtype, up=up)
    torch.cuda.synchronize()
    st = S.last_stats()
    out = r.cpu().numpy()
    assert np.ascontiguousarray(out[:, :kb]).tobytes() == want.tobytes(), "AoS keys are not in numpy's order"
    idx = np.ascontiguousarray(out[:, 8:12]).view(np.uint32).reshape(-1).astype(np.int64)
    assert np.all(np.bincount(idx, minlength=n) == 1), "AoS index is not a permutation"
    assert np.array_equal(out, rec[idx]), "AoS records did not travel whole"
    assert st["record_bytes"] == rec.shape[1]
    return st


def check_plan_stats(st, plan, flow):
    assert st["algo"] == 1, st
    want = plan.host_flow_stats if flow == "host_plan" else plan.device_flow_stats
    got = {k: st[k] for k in want}
    assert got == want, (flow, plan, st)


# ---------------------------------------------------------------------------------------------------------------------
# structured keys: each generator aims at one branch of the plan.  Keys are built as order-mapped values (ascending
# order) of the key width and mapped back to raw keys, so that one generator makes the same plan shape for every type
# of that width; both directions sort the same raw keys.
# ---------------------------------------------------------------------------------------------------------------------
def structured_cases(dt, n, rng):
    """-> {name: (raw keys, predicate the plan must satisfy)}: the predicate proves the generator reaches its branch"""
    kb = dt.itemsize
    W = 8 * kb
    M = (1 << W) - 1
    ud = udtype(kb)

    def U(v):
        return np.asarray(v, dtype=np.uint64).astype(ud) if kb < 8 else np.asarray(v, dtype=np.uint64)

    def spread(base, lo, hi):  # base + uniform integers in [lo, hi]
        return U(np.uint64(base) + rng.integers(lo, hi, n, endpoint=True).astype(np.uint64))

    cases = {}
    cases["full_width"] = (rand_bits(rng, kb, n), lambda p: p.passes == kb and not p.reduce and p.hist_done)
    if kb >= 2:
        low = 0xFF if kb == 2 else 0xFFFF
        cases["const_low"] = ((rand_bits(rng, kb, n) & U(M ^ low)) | U(0x5AA5 & low),
                              lambda p: p.skip[0] and not p.hist_done and p.passes == (1 if kb == 2 else kb - 2))
        top = 0xA7 if kb < 8 else 0xA7B3C1
        tb = 8 if kb < 8 else 24
        cases["const_high"] = ((rand_bits(rng, kb, n) & U(M >> tb)) | U(top << (W - tb)),
                               lambda p: p.passes == kb - tb // 8 and not p.reduce and p.hist_done)
    if kb >= 4:
        mid = kb // 2 - 1  # byte 1 of 4, byte 3 of 8: the passes after it read the other side of the ping-pong
        cases["const_mid"] = ((rand_bits(rng, kb, n) & U(M ^ (0xFF << (8 * mid)))) | U(0x3C << (8 * mid)),
                              lambda p: p.skip[mid] and p.passes == kb - 1 and p.hist_done)
    d = min(1, kb - 1)  # exactly one varying digit: an odd pass count, the result is copied back
    cst = 0xA55AA55AA55AA55A & M & ~(0xFF << (8 * d))
    cases["one_digit"] = (U(cst) | (rand_bits(rng, 1, n).astype(ud) << ud.type(8 * d)),
                          lambda p: p.passes == 1 and not p.reduce)
    cases["all_zero"] = (np.zeros(n, ud), lambda p: p.passes == 0)
    cases["all_equal"] = (np.full(n, 0x5A3C5A3C5A3C5A3C & M, ud), lambda p: p.passes == 0)
    # a narrow range across a digit boundary: every digit up to the boundary varies, the range spans fewer
    if kb == 1:
        cases["narrow_boundary"] = (spread(0x80, -20, 20), lambda p: p.passes == 1)
    elif kb == 2:
        cases["narrow_boundary"] = (spread(0x4000, -100, 100), lambda p: p.reduce and p.passes == 1 and p.planned == 2)
    else:
        cases["narrow_boundary"] = (spread(0x1234567890AB0000 & M, -300, 300),
                                    lambda p: p.reduce and p.passes == 2 and p.planned == 3)
    # a narrow range across the sign (signed: -s..s; float: denormals of both signs and +-0)
    s = {1: 20, 2: 100}.get(kb, 300)
    u = spread(1 << (W - 1), -s, s)
    u[:2] = U([(1 << (W - 1)) - 1, 1 << (W - 1)])  # (float: -0 and +0; signed: -1 and 0)
    cases["narrow_sign"] = (u, lambda p: p.varying == M and (kb == 1 or (p.reduce and p.passes == (1 if kb == 2 else 2))))
    # a narrow range of negative values (floats: around -1.25; unsigned: near the top)
    if dt.kind == "f":
        base = int(O.order_key(np.array([-1.25], dt))[0])
    elif dt.kind == "i":
        base = int(O.order_key(np.array([-100 if kb == 1 else -1000], dt))[0])
    else:
        base = M - 1000 if kb > 1 else 200
    cases["narrow_negative"] = (spread(base, 0, 40 if kb == 1 else 600), lambda p: p.passes <= 2)
    vals = rand_bits(rng, kb, 5)
    cases["heavy_duplicates"] = (vals[rng.integers(0, 5, n)], lambda p: True)
    # one key differs: the top digit varies only in the key at one index
    tail = n % 4096
    for name, pos in (("one_differs_at_last", n - 1), ("one_differs_at_1", 1),
                      ("one_differs_in_last_tile", n - tail + tail // 2 if tail > 2 else n // 2 + 1)):
        if kb == 1:
            u = np.full(n, 0x41, ud)
            u[pos] = 0x3E
        else:
            u = U(0x1111111111111111 & M & ~0xFF) | rand_bits(rng, 1, n).astype(ud)
            u[pos] ^= U(0x40 << (W - 8))
        cases[name] = (u, lambda p: p.passes == (1 if kb == 1 else 2) and not p.reduce)
    return {name: (from_order(u, dt, True), pred) for name, (u, pred) in cases.items()}


SIZES = {"one_partial_tile": 3001, "2p20_plus_4099": (1 << 20) + 4099, "40x8192": 40 * 8192}


@pytest.mark.parametrize("size", list(SIZES), ids=list(SIZES))
@pytest.mark.parametrize("dt", ALL_DTYPES, ids=lambda d: d.name)
def test_structured_keys(dt, size):
    """every generator of its width x both directions x both flows, SoA with an index, 2- and 12-byte rows (1- and
    2-byte chunks: the ANYCHUNK scatter; more than one column: nstage=2), plus one AoS case"""
    n = SIZES[size]
    rng = np.random.default_rng(1000 * dt.num + n % 997)
    pays2 = rng.integers(0, 256, (n, 2), dtype=np.uint8)
    pays12 = rng.integers(0, 256, (n, 12), dtype=np.uint8)
    for name, (keys, pred) in structured_cases(dt, n, rng).items():
        for up in (True, False):
            plan = lsd_plan(keys, up)
            assert pred(plan), (name, up, plan)  # the generator reaches the branch it is named for
            want = sorted_keys(keys, up)
            pays = [np.arange(n, dtype=np.uint32 if up else np.uint64), pays2, pays12]
            for flow, hp in FLOWS.items():
                out_k, out_p, st = sort_soa(keys, pays, up, algo=1, host_plan_min_log2=hp)
                check_soa(keys, pays, out_k, out_p, want)
                check_plan_stats(st, plan, flow)
    keys = structured_cases(dt, n, rng)["narrow_sign"][0]
    rec = records_of(keys, rng)
    for up in (True, False):
        plan = lsd_plan(keys, up)
        for flow, hp in FLOWS.items():
            st = sort_and_check_aos(keys, rec, up, sorted_keys(keys, up), algo=1, host_plan_min_log2=hp)
            check_plan_stats(st, plan, flow)


# ---------------------------------------------------------------------------------------------------------------------
# sampled probe: from n / (keys per probe tile) >= 8192 tiles (2^26 keys of <= 4 bytes, 2^25 dense 8-byte keys) the
# probe's histograms and its min/max come from one key per thread of every probe_sample-th tile.  In a full, dense,
# 16-byte aligned tile thread t's sampled key is base + t * 16/kb (probe_kernel: u[0] of KeyTile::load's vector
# branch); in the partial last tile it is base + t, t < 256.  Keys at odd indices outside the first 256 of the last tile
# are therefore never sampled.  Skipping must still use the exact OR/AND of every key, and Plan::sub the exact minimum
# from minmax_kernel.
# ---------------------------------------------------------------------------------------------------------------------
N_SPARSE = (1 << 26) + 4099
N_SPARSE_8 = (1 << 25) + 4099


def hidden_case(dt, n, case, rng):
    """-> (raw keys, mask of the keys the probe may sample).  The visible keys' smallest and largest values sit at
    index 0 and 16/kb, the first two sampled keys of tile 0, which is sampled whatever probe_sample is: so the sampled
    range is exactly the visible keys' range."""
    kb = dt.itemsize
    W = 8 * kb
    ud = udtype(kb)
    tile = 8192 if kb < 8 else 4096  # keys per probe tile
    full = n - n % tile
    hidden_full = 2 * rng.integers(64, full // 2, 5) + 1  # odd indices in full tiles
    # an odd index of the partial last tile past its first 256 keys (8-byte keys at 2^25 + 4099: the last tile holds 3
    # keys, so its keys may be sampled; only the case that does not depend on it uses it)
    hidden_last = np.array([full + 1001 if n - full > 1001 else n - 1])
    visible = np.ones(n, bool)
    if case == "digit_only_in_hidden":
        # the visible keys vary in their low digit(s) only; the hidden ones also in the top digit
        low = (1 << (24 if kb == 8 else 8)) - 1 if kb > 1 else 0
        c = (0x2222222222222222 & ((1 << W) - 1)) & ~low if kb > 1 else 0x40
        u = (np.uint64(c) | rng.integers(0, low, n, endpoint=True).astype(np.uint64)).astype(ud)
        lo, hi = c, c | low
        where = np.concatenate([hidden_full, hidden_last]) if n - full > 1001 else hidden_full
        if kb == 1:
            u[where] = 0x41
            u[where[::2]] = 0x3F
        else:
            u[where] ^= ud.type(0x41 << (W - 8))
    else:
        base = {1: 0x40, 2: 0x40F0, 4: 0x7FFFFED4 if dt.kind == "i" else 0x1234FF00, 8: (1 << 56) - 30000}[kb]
        if case == "far_outside_the_sample" and kb == 8:
            base = 0x5500000000000000
        span = {1: 20, 2: 100, 4: 600, 8: 60000}[kb]
        u = (np.uint64(base) + rng.integers(0, span, n, endpoint=True).astype(np.uint64)).astype(ud)
        lo, hi = base, base + span
        if case == "one_below_min_in_full_tile":
            where, value = hidden_full[:1], base - 1
        elif case == "one_below_min_in_last_tile":
            where, value = hidden_last, base - 1
        else:
            where, value = hidden_full[:1], base + (1 << (W - 2 if kb < 8 else 60))
        u[where] = ud.type(value)
    visible[where] = False
    u[0], u[16 // kb] = ud.type(lo), ud.type(hi)
    return from_order(u, dt, True), visible


HIDDEN_CASES = ["digit_only_in_hidden", "one_below_min_in_full_tile", "one_below_min_in_last_tile",
                "far_outside_the_sample"]


def check_sorted_big(keys, out):
    """1- and 2-byte keys: a counting oracle (np.bincount of the ordered keys); wider keys: numpy's sort"""
    kb = keys.dtype.itemsize
    if kb <= 2:
        got = O.order_key(out)
        assert np.all(got[1:] >= got[:-1]), "not ordered"
        cnt = np.bincount(O.order_key(keys), minlength=1 << (8 * kb))
        assert np.array_equal(np.bincount(got, minlength=1 << (8 * kb)), cnt), "not a permutation of the keys"
    else:
        assert out.tobytes() == sorted_keys(keys, True).tobytes(), "keys are not in numpy's order"


@pytest.mark.parametrize("case", HIDDEN_CASES)
@pytest.mark.parametrize("dt", [np.uint8, np.int16, np.int32, np.float32], ids=lambda d: np.dtype(d).name)
def test_keys_the_sample_cannot_see(dt, case):
    """default options at 2^26 + 4099 records: the sort is exact although the probe's sample misses the keys that make
    the difference; passes_planned follows the exact keys, hist_sweeps shows whether minmax_kernel ran"""
    dt = np.dtype(dt)
    n = N_SPARSE
    rng = np.random.default_rng(26 + dt.num)
    keys, visible = hidden_case(dt, n, case, rng)
    plan = lsd_plan(keys, True, sampled=O.order_key(keys[visible]))
    k = to_dev(keys)
    S.sort(n, k)
    torch.cuda.synchronize()
    st = S.last_stats()
    check_sorted_big(keys, k.cpu().numpy())
    assert st["algo"] == 1 and plan.host_flow_stats == {f: st[f] for f in plan.host_flow_stats}, (plan, st)
    if case != "digit_only_in_hidden" and dt.itemsize > 1:
        assert st["hist_sweeps"] >= 2  # the exact min/max sweep ran
    if case.startswith("one_below_min") and dt.itemsize > 1:
        assert plan.reduce and plan.mn == int(O.order_key(keys).min())


@pytest.mark.parametrize("sample", [1, 7, 1 << 30])
def test_u8_hidden_keys_at_other_sampling_rates(sample):
    n = N_SPARSE
    for case in HIDDEN_CASES:
        rng = np.random.default_rng(sample + len(case))
        keys, visible = hidden_case(np.dtype(np.uint8), n, case, rng)
        plan = lsd_plan(keys, True, sampled=O.order_key(keys[visible]))
        k = to_dev(keys)
        with S.options(probe_sample=sample):
            S.sort(n, k)
        torch.cuda.synchronize()
        st = S.last_stats()
        check_sorted_big(keys, k.cpu().numpy())
        assert plan.host_flow_stats == {f: st[f] for f in plan.host_flow_stats}, (case, plan, st)


@pytest.mark.parametrize("case", HIDDEN_CASES)
def test_i64_hybrid_keys_the_sample_cannot_see(case):
    """i64 at 2^25 + 4099 on the MSB hybrid path (plan read back, sparse sampling).  These key sets make no cut (the
    sampled entropies add up to less than log2 n + 2), so the plan's passes are the LSD model's; the probe's guessed
    digit (4) is skipped, so hist_kernel always runs"""
    dt = np.dtype(np.int64)
    n = N_SPARSE_8
    rng = np.random.default_rng(25 + len(case))
    keys, visible = hidden_case(dt, n, case, rng)
    plan = lsd_plan(keys, True, sampled=O.order_key(keys[visible]))
    k = to_dev(keys)
    S.sort(n, k)
    torch.cuda.synchronize()
    st = S.last_stats()
    check_sorted_big(keys, k.cpu().numpy())
    assert st["algo"] == 2 and st["cut_digit"] == 0 and st["fell_back"] == 0, st
    assert st["passes_planned"] == plan.passes and st["hist_sweeps"] == 2 + int(plan.want_minmax), (plan, st)
    if case != "digit_only_in_hidden":
        assert plan.want_minmax
    if case.startswith("one_below_min"):
        assert plan.reduce and plan.passes == 2


# ---------------------------------------------------------------------------------------------------------------------
# options: every documented single-GPU option value gives the same bytes, and the plan the model predicts
# ---------------------------------------------------------------------------------------------------------------------
OPTION_VALUES = [{}, {"allow_skip": 0}, {"allow_reduce": 0}, {"allow_lshift": 0}, {"probe_guess": 0},
                 {"hist_match": 1}, {"bytewise": 0}, {"first_atomic": 0}, {"tma_keys": 0}, {"prefetch_cols": 0},
                 {"nstage": 1}, {"nstage": 2}, {"tile_cfg": 0}, {"tile_cfg": 1}, {"tile_cfg": 2}, {"wide_tiles": 0},
                 {"spin_ns": 200}, {"fix_in_pass": 0}, {"junction_table": 0}]
PLAN_OPTIONS = ("allow_skip", "allow_reduce", "probe_guess")
N_OPT = (1 << 18) + 4099


def option_inputs():
    rng = np.random.default_rng(18)
    n = N_OPT
    f = rng.integers(0, 256, 4 * n, dtype=np.uint8).view(np.float32)
    f[rng.integers(0, n, 40)] = np.repeat(np.array([0.0, -0.0, np.inf, -np.inf, np.nan, -np.nan, 1e-40, -1e-40],
                                                   np.float32), 5)
    nan_payload = np.array([0x7FC00001, 0xFFC12345, 0x7F800001], np.uint32).view(np.float32)
    f[rng.integers(0, n, 3)] = nan_payload
    return {
        "i32_range_reduced": (rng.integers(-5000, 5000, n, endpoint=True).astype(np.int32),
                              [np.arange(n, dtype=np.uint32), rng.integers(0, 256, (n, 2), dtype=np.uint8),
                               rng.integers(0, 256, (n, 12), dtype=np.uint8)]),
        "f32_specials": (f, [np.arange(n, dtype=np.uint32)]),
        "u64_8_byte_payload": (rand_bits(rng, 8, n), [np.arange(n, dtype=np.uint64)]),
        "u16_const_low_byte": ((rand_bits(rng, 2, n) & np.uint16(0xFF00)) | np.uint16(0x33), [np.arange(n, dtype=np.uint32)]),
    }


@pytest.mark.parametrize("opt", OPTION_VALUES, ids=lambda o: "default" if not o else "_".join(f"{k}={v}" for k, v in o.items()))
def test_every_option_value(opt):
    """fixed inputs under each non-default option value, with the plan on the device and read back: keys in numpy's
    order, payloads following, and the plan of the model (whose rules allow_skip, allow_reduce and probe_guess change)"""
    plan_opts = {k: v for k, v in opt.items() if k in PLAN_OPTIONS}
    rng = np.random.default_rng(7)
    for name, (keys, pays) in option_inputs().items():
        for up in (True, False):
            plan = lsd_plan(keys, up, **plan_opts)
            want = sorted_keys(keys, up)
            for flow, hp in FLOWS.items():
                out_k, out_p, st = sort_soa(keys, pays, up, algo=1, host_plan_min_log2=hp, **opt)
                check_soa(keys, pays, out_k, out_p, want)
                check_plan_stats(st, plan, flow)
    # 16-byte AoS records
    keys = rng.integers(-(1 << 40), 1 << 40, N_OPT).astype(np.int64)
    rec = records_of(keys, rng)
    for flow, hp in FLOWS.items():
        plan = lsd_plan(keys, False, **plan_opts)
        st = sort_and_check_aos(keys, rec, False, sorted_keys(keys, False), algo=1, host_plan_min_log2=hp, **opt)
        check_plan_stats(st, plan, flow)
    # i64 on the hybrid path with the plan read back: the last pass orders the tile-local segments and the junction
    # kernel the others, unless fix_in_pass=0 (or the smaller tile, which has no such pass) asks for the full finish
    n = (1 << 22) + 4099
    keys = rand_bits(rng, 8, n).view(np.int64)
    pays = [np.arange(n, dtype=np.uint64)]
    out_k, out_p, st = sort_soa(keys, pays, True, host_plan_min_log2=0, **opt)
    check_soa(keys, pays, out_k, out_p, sorted_keys(keys, True))
    assert st["algo"] == 2 and st["fell_back"] == 0 and st["cut_digit"] >= 2, st
    full_finish = opt.get("fix_in_pass") == 0 or opt.get("tile_cfg") == 1
    assert st["segfix_passes"] == (1 if full_finish else 0), (opt, st)


@pytest.mark.parametrize("host_pipeline", [0, 1])
def test_host_pipeline(host_pipeline):
    """host arrays of >= 2^20 records with payloads: the pipelined staging sorts the keys with a 4-byte index while the
    payloads upload (record_bytes = key + 4); without it the whole records are staged and sorted"""
    n = (1 << 20) + 4099
    rng = np.random.default_rng(20 + host_pipeline)
    keys = rng.integers(-5000, 5000, n, endpoint=True).astype(np.int32)
    pays = [np.arange(n, dtype=np.uint32), rng.integers(0, 256, (n, 2), dtype=np.uint8),
            rng.integers(0, 256, (n, 12), dtype=np.uint8)]
    for up in (True, False):
        k, ps = keys.copy(), [p.copy() for p in pays]
        with S.options(host_pipeline=host_pipeline):
            S.sort(n, k, *ps, up=up)
        st = S.last_stats()
        check_soa(keys, pays, k, ps, sorted_keys(keys, up))
        assert st["record_bytes"] == (4 + 4 if host_pipeline else 4 + 4 + 2 + 12), st
