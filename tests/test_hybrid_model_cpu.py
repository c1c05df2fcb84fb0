"""CPU tests of tests/hybrid_model.py, the exact model of the 8-byte-key hybrid path and its finishes: the plan's
rules on hand-worked key sets, each finish on hand-worked arrays, the emulated finishes against a brute-force
statement of what they must achieve (tiny tiles and caps, so that every branch runs at a few hundred keys), and every
generator of the GPU tests reaching the branch it is named for."""
import numpy as np
import pytest

import hybrid_model as H
import oracle_lib as O

U = np.uint64
DTYPES = [np.dtype(d) for d in (np.uint64, np.int64, np.float64)]


def pk(top, mid, low, wbit=24):
    """plan keys top | mid | low with the swept bits at wbit and above (top = digit 7)"""
    return ((np.asarray(top, np.uint64) << U(56)) | (np.asarray(mid, np.uint64) << U(wbit))
            | np.asarray(low, np.uint64)).astype(np.uint64)


def run_fix(w, tile, fix_cap=H.FIX_CAP, jf_cap=H.JF_CAP, table=True, wbit=24):
    res, G, fpf, fpl = H.fix_pass(w, np.arange(len(w)), 7, wbit, w, wbit, tile, fix_cap)
    if not res.fix_flag:
        H.junction_fix(res, G, fpf, fpl, wbit, table, jf_cap)
    return res


# ---------------------------------------------------------------------------------------------------------------------
# the plan
# ---------------------------------------------------------------------------------------------------------------------
def test_plan_cut_and_the_two_sweeps_rule():
    rng = np.random.default_rng(1)
    n = 1 << 16
    u = rng.integers(0, 2**64, n, dtype=np.uint64)
    p = H.hybrid_plan(u, margin_bits=2)  # need 18: 8 + 8 + 8 reaches it at digit 5
    assert (p.cut_digit, p.n_exec, p.final_sel, p.first_exec_p1, p.lshift, p.sub) == (5, 3, 1, 6, 0, 0)
    assert p.hist_done  # the host's guess: 8 - ceil(18 / 8) = 5
    assert H.hybrid_plan(u, margin_bits=-10).cut_digit == 7  # need 6: the top digit alone
    # only digits 7, 6 and 0 vary: the cut at digit 1 would save one sweep (digit 0) -- no cut
    v = (u & U(0xFFFF0000000000FF)) | U(0x0000123456789A00)
    p = H.hybrid_plan(v, margin_bits=6)  # need 22: 8 + 8, then digits 5..1 are skipped, digit 0 reaches it
    assert p.cut_digit == 0 and p.n_exec == 3
    with pytest.raises(H.Ambiguous):
        H.hybrid_plan(u, margin_bits=8)  # need 24 against 3 x (8 - 0.0056): too close to say


def test_plan_left_shift_and_range_reduction():
    rng = np.random.default_rng(2)
    n = 1 << 16
    b = H.KeyBuilder(n, 4, rng, lshift=3)
    p = H.hybrid_plan(b.u(), margin_bits=int(round(30.5 - 16)))
    assert (p.lshift, p.cut_digit, p.cut_bit, p.n_exec, p.hist_done) == (3, 4, 29, 4, False)
    assert H.hybrid_plan(b.u(), margin_bits=14, allow_lshift=0).cut_digit == 3  # unshifted: 5 + 8 + 8 + 8 + 8
    # a range of 2^20 across bit 32 spans 3 digit positions, fewer than the 5 the plan sweeps: subtract the minimum
    u = U(0x6A5F0000FFFF8000) + rng.integers(0, 1 << 20, n, dtype=np.uint64)
    p = H.hybrid_plan(u)
    assert (p.cut_digit, p.sub, p.skip, p.want_minmax) == (0, int(u.min()), (False,) * 3 + (True,) * 5, True)


# ---------------------------------------------------------------------------------------------------------------------
# the finishes, worked by hand
# ---------------------------------------------------------------------------------------------------------------------
def test_last_pass_orders_nine_and_checks_ten():
    tile = 32
    top = np.arange(32) % 16 + 100
    mid = np.arange(32) * 10
    low = np.zeros(32, np.int64)
    # nine keys of one prefix in tile 0 (bucket 5), reversed: ordered by the last pass
    top[:9], mid[:9], low[:9] = 5, 1, np.arange(9)[::-1]
    res = run_fix(pk(top, mid, low), tile)
    assert not res.fix_flag and res.fix_runs[(9, "ordered")] == 1 and res.fix_moved_runs[9] == 1
    assert np.array_equal(res.w[:9] & U(0xFF), np.arange(9))
    # ten: too long to be ordered in the pass; reversed raises the flag, in order does not
    top[:10], mid[:10], low[:10] = 5, 1, np.arange(10)[::-1]
    res = run_fix(pk(top, mid, low), tile)
    assert res.fix_flag and res.fix_runs[(10, "long_inverted")] == 1
    low[:10] = np.arange(10)
    res = run_fix(pk(top, mid, low), tile)
    assert not res.fix_flag and res.fix_runs[(10, "long_in_order")] == 1


@pytest.mark.parametrize("kl,kr,how,kind,flag", [
    (1, 1, "inverted", ("swap", 2), False), (16, 16, "interleaved", ("rank", 32), False),
    (16, 17, "inverted", ("long_inverted", 0), True), (16, 17, "in_order", ("long_in_order", 0), False)])
def test_junction_segments(kl, kr, how, kind, flag):
    """a segment of kl keys at the end of tile 0 and kr at the start of tile 1 (each part ascending)"""
    tile = 64
    v = np.arange(kl + kr)
    left, right = {"inverted": (v[kr:], v[:kr]), "in_order": (v[:kl], v[kl:]),
                   "interleaved": H._interleave(v, [kl, kr])}[how]
    top = np.arange(128) % 200 + 20
    mid = np.arange(128) * 4
    low = np.zeros(128, np.int64)
    top[tile - kl:tile + kr], mid[tile - kl:tile + kr] = 3, mid[tile - kl]
    mid[tile + kr:] = np.maximum(mid[tile + kr:], mid[tile - kl])
    low[tile - kl:tile + kr] = np.r_[left, right]
    res = run_fix(pk(top, mid, low), tile)
    assert not res.fix_flag and res.junctions[kind] == 1 and res.junction_flag == flag
    if not flag:
        assert np.all(res.w[1:] >= res.w[:-1])


def test_three_tile_segment_and_empty_next_tile():
    """tile 1 holds one key of the segment (tiles 0, 1, 2) or none of its bucket (tiles 0, 2): the first junction's
    thread orders the whole segment, found through the fingerprints or, over the empty tile, the key compare"""
    tile = 16
    for k_mid in (1, 0):
        top = (np.arange(64) * 7) % 200 + 20
        mid = np.arange(64) * 4
        low = np.arange(64) * 0
        seg = [13, 14, 15] + ([16 + 5] if k_mid else []) + [32, 33]
        top[16:32] = 210 + np.arange(16) % 8  # tile 1: other buckets, one mid (the segment's)
        mid[13:34] = 100
        mid[34:] = np.maximum(mid[34:], 101)
        low[16:32] = np.arange(16)
        top[seg] = 3
        low[seg] = [2, 5, 7] + ([1] if k_mid else []) + [0, 6]
        for table in (True, False):
            res = run_fix(pk(top, mid, low), tile, table=table)
            L = len(seg)
            assert not res.fix_flag and not res.junction_flag
            assert res.junctions[("rank", L)] == 1 and res.tiles_spanned[2 + k_mid] == 1
            assert res.junctions[("owned_by_earlier", L)] == k_mid
            assert res.direct_compares == ((0 if k_mid else 1) if table else 1 + k_mid)
            assert np.all(res.w[1:] >= res.w[:-1])


def test_fingerprint_collision_is_not_a_segment():
    """prefixes whose 32-bit fingerprints (hi ^ lo of the masked key, cut at bit 16) agree meet at a junction: the key
    compare tells them apart"""
    wbit = 16
    tile = 8
    w = np.array([(7 << 56) | (i << 24) | (0x77 << 16) | 9 for i in range(16)], np.uint64)
    a = (7 << 56) | (0x10 << 48) | (0x21 << 16) | 5   # digit 6 = 0x10, digit 2 = 0x21
    b = (7 << 56) | (0x11 << 48) | (0x20 << 16) | 3   # both xor-ed with 1: the same fingerprint
    w[7], w[8] = a, b
    w[9:] = np.maximum(w[9:], np.uint64(b) + np.arange(1, 8, dtype=np.uint64))
    w[:7] = (np.arange(7, dtype=np.uint64) + 1) << U(56)  # other buckets
    res = run_fix(w, tile, wbit=wbit)
    assert res.collisions == 1 and not res.junctions and not res.junction_flag


def test_segment_finish_chunks_and_halo():
    """chunks of 256 positions, 32 keys of halo: a segment across a chunk edge and one reaching 31 keys into the
    next chunk are ordered by the chunk holding their head; 33 distinct keys fall back, 33 equal ones do not"""
    n = 700
    top = np.zeros(n, np.int64)
    mid = np.arange(n) * 3
    low = np.arange(n) * 0

    def finish(w, sel=0):
        res = H.Finish(w.copy(), np.arange(n))
        return H.segfix(res.w, res.ids, 24, sel, res)

    for a, L in ((250, 10), (255, 32), (0, 7), (n - 7, 7)):
        m, lo = mid.copy(), low.copy()
        m[a:a + L] = m[a]
        lo[a:a + L] = np.arange(L)[::-1]
        res = finish(pk(top, m, lo))
        assert not res.fall_back and res.segfix_segments[("short", L)] == 1
        assert res.segfix_moved == 2 * (L // 2) and np.all(res.w[1:] >= res.w[:-1])
        assert res.segfix_chunk_crossers == int(a // 256 != (a + L - 1) // 256)
        assert finish(pk(top, m, lo), sel=1).segfix_moved == n  # from the shadow: every record moves
    for lows, fb in ((np.arange(33)[::-1], True), (np.full(33, 4), False)):
        m, lo = mid.copy(), low.copy()
        m[300:333], lo[300:333] = m[300], lows
        assert finish(pk(top, m, lo)).fall_back == fb


# ---------------------------------------------------------------------------------------------------------------------
# the emulation against brute force, with tiny tiles and caps
# ---------------------------------------------------------------------------------------------------------------------
def random_last_pass_input(rng, n, n_prefixes):
    """plan keys ordered by mid (the lower swept digits), few prefixes so that runs and segments of every length
    occur, random low parts (sometimes equal)"""
    mid = np.sort(rng.integers(0, n_prefixes, n))
    top = rng.integers(0, 4, n)
    low = rng.integers(0, 6 if rng.random() < 0.3 else 1000, n)
    return pk(top, mid, low)


@pytest.mark.parametrize("seed", range(200))
def test_fix_and_junctions_against_brute_force(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(40, 400))
    tile = int(rng.choice([8, 16, 32]))
    fix_cap, jf_cap = int(rng.integers(1, 5)), int(rng.integers(3, 12))
    w = random_last_pass_input(rng, n, int(rng.integers(n // 6 + 1, n)))
    res = run_fix(w, tile, fix_cap, jf_cap, table=bool(rng.integers(0, 2)))
    # brute force: runs of a tile = its keys of one prefix; segments = all keys of one prefix
    pre = w >> U(24)
    tiles = np.arange(n) // tile
    fix_flag = junction_flag = False
    after = w.copy()
    for t in range(tiles.max() + 1):
        for p in np.unique(pre[tiles == t]):
            i = np.flatnonzero((tiles == t) & (pre == p))
            if len(i) > fix_cap + 1:
                fix_flag |= bool(np.any(w[i][1:] < w[i][:-1]))
            else:
                after[i] = np.sort(w[i])
    for p in np.unique(pre):
        s = after[pre == p]
        if len(s) > jf_cap:
            junction_flag |= bool(np.any(s[1:] < s[:-1]))
    assert res.fix_flag == fix_flag
    if not fix_flag:
        assert res.junction_flag == junction_flag
        if not junction_flag:  # the design's invariant: no flag -> in order
            assert np.array_equal(res.w, np.sort(w))
    assert np.array_equal(w[res.ids], res.w)


@pytest.mark.parametrize("seed", range(100))
def test_segment_finish_against_brute_force(seed):
    rng = np.random.default_rng(1000 + seed)
    n = int(rng.integers(30, 500))
    maxseg = int(rng.choice([4, 8, 32]))
    chunk = maxseg * int(rng.integers(1, 5))
    w = random_last_pass_input(rng, n, int(rng.integers(n // (2 * maxseg) + 1, n)))
    w = w[np.argsort(w >> U(24), kind="stable")]
    sel = int(rng.integers(0, 2))
    res = H.segfix(w.copy(), np.arange(n), 24, sel, H.Finish(w.copy(), np.arange(n)), chunk, maxseg, maxseg)
    pre = w >> U(24)
    want = w.copy()
    fall_back = False
    for p in np.unique(pre):
        i = np.flatnonzero(pre == p)
        if len(i) <= maxseg:
            want[i] = np.sort(w[i])
        else:
            fall_back |= bool(np.any(w[i] != w[i[0]]))
    assert res.fall_back == fall_back and np.array_equal(res.w, want) and np.array_equal(w[res.ids], res.w)
    assert res.segfix_moved == (n if sel else int(np.sum((want != w) | (res.ids != np.arange(n)))))


# ---------------------------------------------------------------------------------------------------------------------
# every generator reaches its branch, for every key type and direction, in the device flow and the FIX flow; the
# emulated output is the total-order sort
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("gen", list(H.GENERATORS))
def test_generator_reaches_its_branch(gen):
    for dt in DTYPES:
        for up in (True, False):
            case = H.GENERATORS[gen](dt, up, np.random.default_rng(len(gen) * 7 + dt.num))
            want = O.total_order_sorted_keys(case.keys, up)
            for flow in H.FLOWS:
                pred = H.predict(case.keys, up, flow, margin_bits=case.margin_bits, first_atomic=0)
                assert case.expect(pred), (gen, dt, up, flow, pred.plan, pred.stats)
                assert case.keys[pred.finish.ids].tobytes() == want.tobytes(), (gen, dt, up, flow)
                assert not pred.tie_dependent


def test_generators_fail_when_the_caps_differ():
    """the cap generators pin the caps: with FIX_CAP + 1, JF_CAP - 1 or SF_MAXSEG - 1 in the model they miss their
    branch"""
    dt = np.dtype(np.uint64)
    for gen, cap in (("run9_reversed", dict(fix_cap=H.FIX_CAP - 1)), ("run10_reversed", dict(fix_cap=H.FIX_CAP + 1)),
                     ("junction32", dict(jf_cap=H.JF_CAP - 1)), ("junction33_inverted", dict(jf_cap=H.JF_CAP + 1))):
        case = H.GENERATORS[gen](dt, True, np.random.default_rng(len(gen) * 7 + dt.num))
        assert not case.expect(H.predict(case.keys, True, "host", margin_bits=case.margin_bits, first_atomic=0, **cap))
    for gen, cap in (("segfix32", H.SF_MAXSEG - 1), ("segfix33_distinct", H.SF_MAXSEG + 1)):
        case = H.GENERATORS[gen](dt, True, np.random.default_rng(len(gen) * 7 + dt.num))
        assert not case.expect(H.predict(case.keys, True, "device", margin_bits=case.margin_bits, sf_maxseg=cap,
                                         word=cap))
