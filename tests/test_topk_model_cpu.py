"""CPU tests of tests/topk_model.py: the order map the model uses is the library's, hand-worked selections, the model
against brute force on random rows, and every row generator reaching its branch for every key type it applies to."""
import numpy as np
import pytest

import oracle_lib as O
import topk_model as M

ALL_DTYPES = [np.dtype(d) for d in O.KEY_DTYPES]


def _make_key_order(dt, ascending):
    """make_key_order (b200sort.cu) for a numpy dtype: -> (xor_const, neg_xor)"""
    kb = dt.itemsize
    mask, sign = (1 << 8 * kb) - 1, 1 << (8 * kb - 1)
    xor_const = sign if dt.kind in "if" else 0
    neg_xor = mask ^ sign if dt.kind == "f" else 0
    if not ascending:
        xor_const ^= mask
    return xor_const, neg_xor


def _to_ordered(raw: int, kb: int, ko) -> int:
    """to_ordered<KB, false> (kernels.cuh) of one raw key"""
    neg = ((1 << 8 * kb) - 1) if (raw >> (8 * kb - 1)) & 1 else 0
    return raw ^ ko[0] ^ (neg & ko[1])


@pytest.mark.parametrize("dt", ALL_DTYPES, ids=lambda d: d.name)
def test_order_key_is_the_kernels_map(dt):
    rng = np.random.default_rng(11)
    kb = dt.itemsize
    udt = np.dtype(f"u{kb}")
    raw = rng.integers(0, (1 << 8 * kb) - 1, 2000, dtype=np.uint64, endpoint=True).astype(udt)
    edges = [0, 1, (1 << 8 * kb) - 1, 1 << (8 * kb - 1), (1 << (8 * kb - 1)) - 1, (1 << (8 * kb - 1)) + 1]
    raw = np.concatenate([raw, np.array(edges, np.uint64).astype(udt)])
    if dt.kind == "f":
        raw = np.concatenate([raw, M.float_specials(dt).view(udt)])
    keys = raw.view(dt)
    for largest in (True, False):
        ko = _make_key_order(dt, not largest)
        want = np.array([_to_ordered(int(r), kb, ko) for r in raw], np.uint64).astype(udt)
        got = O.order_key(keys, up=not largest)
        assert got.dtype == udt and got.tobytes() == want.tobytes()
        assert M._raw(got, dt, largest).tobytes() == keys.tobytes(), "from_order is not the inverse of order_key"


def _state(s, row=0):
    return {f: int(s.state[f][row]) for f in M.STATE_FIELDS}


def test_hand_worked_selections():
    # u32, all equal, L = 1000, k = 3: every bucket holds 1000 > cap = 63 records, so passes 1-4 re-read the row and
    # pass 4 finishes it (after the last decision, so its mode stays LAST)
    s = M.select_keys(np.full(1000, 7, np.uint32), 3, True)
    assert s.cap == 63 and s.depth[0] == 3 and s.items[0].tolist() == [0, 1, 1, 1, 1] and s.reads[0] == 5
    assert _state(s) == dict(T=~np.uint32(7) & 0xFFFFFFFF, k_left=3, cand=1000, src_n=1000, out_ctr=0, tie_ctr=1000,
                             wr_ctr=0, mode=M.LAST, in_buf=0, write_buf=0, pad_=0)
    # k = L: the first bucket holds every record still to select -- finished at decision 0 and DONE at decision 1
    s = M.select_keys(np.full(1000, 7, np.uint32), 1000, False)
    assert s.depth[0] == 0 and s.items[0].tolist() == [0, 1, 0, 0, 0] and s.reads[0] == 2
    assert _state(s) == dict(T=0, k_left=1000, cand=1000, src_n=0, out_ctr=0, tie_ctr=1000, wr_ctr=0, mode=M.DONE, in_buf=0,
                             write_buf=0, pad_=0)
    # u16 keys 0x0100 + i for i < 200 and one 0x0500, smallest 3: bucket 1 of digit 0 holds 200 records (> cap = 13),
    # bucket 2 of digit 1 is the third -- finished at the last decision, pass 2 re-reads the row
    keys = np.concatenate([0x0100 + np.arange(200), [0x0500]]).astype(np.uint16)
    s = M.select_keys(keys, 3, False)
    assert s.cap == 13 and s.depth[0] == 1 and s.reads[0] == 3 and s.items[0].tolist() == [0, 1, 1]
    assert _state(s) == dict(T=0x0102, k_left=1, cand=1, src_n=200, out_ctr=2, tie_ctr=1, wr_ctr=0, mode=M.LAST, in_buf=0,
                             write_buf=0, pad_=0)
    # the same keys, largest 3: 0x0500 is alone in its bucket of digit 0 (ordered 0xFA, selected by pass 1); the
    # k_left = 2 others are 0x01C7 and 0x01C6 of the 200 in bucket 0xFE, and digit 1 picks 0x01C6 (ordered 0xFE39)
    s = M.select_keys(keys, 3, True)
    t = s.trace[0]
    assert t["b"][0] == 0xFE and t["below"][0] == 1 and t["kl"][0] == 2 and t["c"][0] == 200 and t["write_buf"][0] == 0
    assert s.state["T"][0] == 0xFFFF - 0x01C6 and s.state["k_left"][0] == 1 and s.state["cand"][0] == 1
    assert s.depth[0] == 1 and s.state["out_ctr"][0] == 2
    # u8: one decision; uniform bytes, L = 4096 (cap 256): pass 1 reads the row and finishes it
    s = M.select_keys(np.arange(4096).astype(np.uint8), 100, False)
    assert s.depth[0] == 0 and s.items[0].tolist() == [0, 1] and s.reads[0] == 2 and _state(s)["mode"] == M.LAST
    assert s.state["T"][0] == 6 and s.state["k_left"][0] == 4 and s.state["cand"][0] == 16
    # u32, L = 300000 (37 chunks, cap 18750), top byte 0, byte 1 0x10 for 10000 records and 0x20 for the rest,
    # smallest 1: passes 1 and 2 read the row, pass 2 buffers the 10000 candidates, pass 3 reads 2 chunks of them
    rng = np.random.default_rng(12)
    L = 300_000
    keys = np.where(np.arange(L) < 10_000, 0x00100000, 0x00200000).astype(np.uint32) | rng.integers(0, 2**16, L, dtype=np.uint32)
    s = M.select_keys(rng.permutation(keys), 1, False)
    assert s.items[0].tolist()[:4] == [0, 37, 37, 2] and s.items[0][4] == 1 and s.reads[0] == 3
    assert s.trace[1]["c"][0] == 10_000 and s.trace[1]["write_buf"][0] == 1 and s.trace[2]["src_n"][0] == 10_000


def test_layout_mirrors_topk_layout():
    assert M.ROW_DTYPE.itemsize == 80 and M.CTRL_BYTES == 128
    assert M.layout(1) == (0, 256, 256 + 2048)
    assert M.layout(5) == (0, 512, 512 + 5 * 2048)
    assert M.layout(3000) == (0, 240128, 240128 + 3000 * 2048)


@pytest.mark.parametrize("dt", ALL_DTYPES, ids=lambda d: d.name)
def test_model_against_brute_force(dt):
    rng = np.random.default_rng(13)
    kb = dt.itemsize
    for L in (1, 2, 17, 300, 5000):
        for k in sorted({1, 2, L // 3, L - 1, L} & set(range(1, L + 1))):
            for largest in (True, False):
                # few distinct values, then full-width ones: ties and deep decisions, then early finishes
                pool = rng.integers(0, (1 << 8 * kb) - 1, 1 + int(rng.integers(1, 9)), dtype=np.uint64, endpoint=True)
                rows = [pool[rng.integers(0, len(pool), L)], rng.integers(0, (1 << 8 * kb) - 1, L, dtype=np.uint64, endpoint=True)]
                u = np.stack(rows)
                s = M.select(u, k, kb)
                for r in range(len(rows)):
                    d = int(s.depth[r])
                    shift = np.uint64(8 * (kb - 1 - d))
                    pre, T = u[r] >> shift, np.uint64(s.state["T"][r])
                    kth = np.sort(u[r])[k - 1]
                    assert 0 <= d < kb
                    assert (kth >> shift) == T, "the k-th smallest key does not have the prefix T"
                    assert (pre < T).sum() == k - s.state["k_left"][r] == s.state["out_ctr"][r]
                    assert (pre == T).sum() == s.state["cand"][r] == s.state["tie_ctr"][r]
                    assert 1 <= s.state["k_left"][r] <= s.state["cand"][r]
                    # finished at d: its bucket is taken whole, or d is the last digit; never earlier
                    assert s.state["k_left"][r] == s.state["cand"][r] or d == kb - 1
                    for e in range(d):
                        sh = np.uint64(8 * (kb - 1 - e))
                        assert ((u[r] >> sh) <= (kth >> sh)).sum() > k, f"row {r} should have finished at {e}"
                    assert s.state["mode"][r] == (M.LAST if d == kb - 1 else M.DONE)
                    assert s.reads[r] == 1 + sum(1 for t in s.trace[:d + 1] if t["in_buf"][r] == 0)


@pytest.mark.parametrize("dt", ALL_DTYPES, ids=lambda d: d.name)
def test_every_generator_reaches_its_branch(dt):
    rng = np.random.default_rng(14)
    kb = dt.itemsize
    seen = set()
    for L in (1, 2, 16, 17, 33, 100, 1000, 3 * 8192 + 5):
        for k in sorted({1, 2, 33, L // 3, L - 1, L} & set(range(1, L + 1))):
            for largest in (True, False):
                for g in M.generators(dt, L, k):
                    keys = g(dt, L, k, largest, rng)  # (asserts its branch)
                    assert keys.dtype == dt and keys.shape == (L,)
                    seen.add(g.__name__)
    want = {"gen_uniform", "gen_equal", "gen_two_values", "gen_run"} | {f"gen_const_top{j}" for j in range(1, kb)}
    want |= {f"gen_early{d}" for d in range(kb)}
    want |= {f"gen_cap{o}_d{D}" for D in (0, 1) if D < kb - 1 for o in ("", "_over")}
    if dt.kind == "f":
        want.add("gen_specials")
    assert seen == want


def test_a_wrong_cap_breaks_the_cap_generators(monkeypatch):
    # the cap-boundary rows are built from the documented buffer size; a model whose cap rule differs misses them: a
    # larger cap buffers the "cap + 1" buckets, a smaller one re-reads the rows of the exactly full ones
    rng = np.random.default_rng(15)
    for div, broken in ((8, "gen_cap_over"), (32, "gen_cap_d")):
        monkeypatch.setattr(M, "TOPK_CAP_DIV", div)
        for g in M.GENERATORS:
            if g.__name__.startswith(broken) and g.applies(np.uint32, 1000, 33):
                with pytest.raises(AssertionError, match="does not reach its branch"):
                    g(np.uint32, 1000, 33, True, rng)


def test_mixed_rows_cycle_the_generators():
    rng = np.random.default_rng(16)
    gens = M.generators(np.float64, 1000, 33)
    keys = M.mixed_rows(np.float64, 3 * len(gens) + 2, 1000, 33, True, rng)
    s = M.select_keys(keys, 33, True)
    # the rows take different paths in the same pass: several depths, and both buffer and row reads at one decision
    assert len(set(s.depth.tolist())) >= 5
    assert {0, 1} <= set(s.trace[2]["in_buf"].tolist())
