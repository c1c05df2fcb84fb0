"""An exact numpy model of the top-k radix select (TEST INFRASTRUCTURE ONLY), and named row generators that each
reach one branch of it.

The selection keeps one state record per row (TopkRow), and the decision kernel moves every row through its own
sequence of modes: which row reads its candidate buffer, which re-reads the row, which is finishing and which is done
all differ from row to row in the same pass.  A wrong branch still selects plausible records, so the tests compare
the state the device leaves in the workspace, row by row, with `select`, which restates the decision rule.  Every
rule cites the line it restates (simd-radix-sort_b200/csrc):

- topk_host.cuh:51: rows, histograms and the control block are zeroed; topk.cuh:86 (topk_init_kernel): k_left = k.
- topk.cuh:41: cap = ceil(row_len / TOPK_CAP_DIV) candidate-buffer entries per row.
- topk.cuh:152-165 (`kind` of topk_pass_kernel): pass p >= 1 keeps as candidates the records whose top p digits equal
  T, and counts their digit p; pass 0 counts digit 0 of every record.  A finishing (LAST) pass counts nothing.
- topk.cuh:291-340 (topk_decide_kernel), decision d after pass d, for every row:
  - :294 a DONE row is skipped; :295-298 a LAST row (finished by pass d) becomes DONE;
  - :300-314 the bucket b of digit d is the first where the inclusive count reaches k_left;
  - :319 kl = k_left - (records below b), c = hist[b], src_n = the previous cand;
  - :318 in_buf = the previous write_buf (pass d wrote the buffer pass d + 1 reads);
  - :320 the next mode is LAST when c == kl or d == KB - 1;
  - :321 T = (T << 8) | b;  :326 write_buf = (next mode ACTIVE and c <= cap);  :328-329 wr_ctr = tie_ctr = 0;
  - :330-332 items[d + 1] += ceil((in_buf ? src_n : row_len) / TOPK_CHUNK).
- topk.cuh:187-188 (`reserve`): out_ctr counts every record emitted below T; the finishing pass counts the records
  equal to T in tie_ctr (so tie_ctr = cand), and a non-finishing pass counts its buffered candidates in wr_ctr.
- topk_host.cuh:66-71: key-width + 1 passes and key-width decisions; pass p >= 1 reads the row unless in_buf.
- topk_host.cuh:14-31 (topk_layout): rows at offset 0, then the histograms, then TopkCtrl, each at a 256-byte boundary.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

import oracle_lib as O
from plan_model import from_order  # the inverse of oracle_lib.order_key

TOPK_CHUNK = 8192   # topk.cuh:36
TOPK_CAP_DIV = 16   # topk.cuh:37
RADIX = 256
MAX_PASSES = 16     # kernels.cuh:20
ACTIVE, LAST, DONE = 0, 1, 2  # topk.cuh:39

# TopkRow (topk.cuh:44-57; its size is a static_assert there)
ROW_DTYPE = np.dtype([("T", "<u8"), ("k_left", "<u8"), ("cand", "<u8"), ("src_n", "<u8"), ("out_ctr", "<u8"),
                      ("tie_ctr", "<u8"), ("wr_ctr", "<u8"), ("item_base", "<u8"), ("mode", "<u4"), ("in_buf", "<u4"),
                      ("write_buf", "<u4"), ("pad_", "<u4")])
assert ROW_DTYPE.itemsize == 80
CTRL_BYTES = 8 * MAX_PASSES  # TopkCtrl (topk.cuh:59-61)
# the fields of TopkRow the model gives: item_base depends on the order of the decisions' atomics
STATE_FIELDS = ("T", "k_left", "cand", "src_n", "out_ctr", "tie_ctr", "wr_ctr", "mode", "in_buf", "write_buf", "pad_")


def topk_cap(row_len: int) -> int:
    return -(-row_len // TOPK_CAP_DIV)


def _align256(x: int) -> int:
    return (x + 255) // 256 * 256


def layout(n_rows: int) -> tuple:
    """-> (rows, hist, ctrl) byte offsets of the first three regions of the workspace (topk_host.cuh:19-26)"""
    hist_off = _align256(ROW_DTYPE.itemsize * n_rows)
    return 0, hist_off, hist_off + _align256(RADIX * 8 * n_rows)


@dataclass(frozen=True)
class Selection:
    """The selection of B rows of one call.  Per-row arrays of length B, except `items` (B, KB + 1) and `trace`."""
    kb: int
    row_len: int
    k: int
    cap: int
    state: np.ndarray    # ROW_DTYPE (B,): the TopkRow each row ends with (item_base 0)
    items: np.ndarray    # (B, KB + 1): work items each row adds to pass p (p >= 1)
    depth: np.ndarray    # the decision after which the row's pass finishes it
    reads: np.ndarray    # full reads of the row: pass 0 and every pass p >= 1 without in_buf
    trace: tuple         # per decision d: dict of (B,) arrays b, below, kl, c, mode, in_buf, src_n, write_buf
                         # (-1 for rows the decision does not decide)


def select(u: np.ndarray, k: int, kb: int) -> Selection:
    """The selection of the k smallest of every row of ordered keys `u` ((B, L) or (L,), unsigned, KB bytes each:
    oracle_lib.order_key(keys, up=not largest))."""
    u = np.asarray(u).astype(np.uint64)
    u = u.reshape(1, -1) if u.ndim == 1 else u
    B, L = u.shape
    if not 1 <= k <= L:
        raise ValueError("k must be in [1, row_len]")
    cap = topk_cap(L)
    T = np.zeros(B, np.uint64)
    k_left = np.full(B, k, np.int64)
    cand, src_n = np.zeros(B, np.int64), np.zeros(B, np.int64)
    in_buf, write_buf = np.zeros(B, bool), np.zeros(B, bool)
    mode = np.full(B, ACTIVE, np.uint32)
    items = np.zeros((B, kb + 1), np.int64)
    depth, reads = np.full(B, -1, np.int64), np.ones(B, np.int64)
    trace = []
    for d in range(kb):
        mode[mode == LAST] = DONE
        act = np.nonzero(mode == ACTIVE)[0]
        if len(act) == 0:
            break
        ua = u[act]
        if d == 0:
            sel = np.ones(ua.shape, bool)
        else:
            sel = (ua >> np.uint64(8 * (kb - d))) == T[act][:, None]
        digit = ((ua >> np.uint64(8 * (kb - 1 - d))) & np.uint64(0xFF)).astype(np.int64)
        ri = np.nonzero(sel)[0]
        hist = np.bincount(ri * RADIX + digit[sel], minlength=len(act) * RADIX).reshape(len(act), RADIX)
        incl = np.cumsum(hist, axis=1)
        b = np.argmax(incl >= k_left[act][:, None], axis=1)
        ar = np.arange(len(act))
        c = hist[ar, b]
        below = incl[ar, b] - c
        kl = k_left[act] - below
        nxt = np.where((c == kl) | (d == kb - 1), LAST, ACTIVE).astype(np.uint32)
        in_buf[act] = write_buf[act]
        src_n[act] = cand[act]
        T[act] = (T[act] << np.uint64(8)) | b.astype(np.uint64)
        write_buf[act] = (nxt == ACTIVE) & (c <= cap)
        k_left[act], cand[act], mode[act] = kl, c, nxt
        n = np.where(in_buf[act], src_n[act], L)
        items[act, d + 1] = (n + TOPK_CHUNK - 1) // TOPK_CHUNK
        reads[act] += ~in_buf[act]
        depth[act[nxt == LAST]] = d
        rec = {}
        for name, v in (("b", b), ("below", below), ("kl", kl), ("c", c), ("mode", nxt), ("in_buf", in_buf[act]),
                        ("src_n", src_n[act]), ("write_buf", write_buf[act])):
            rec[name] = np.full(B, -1, np.int64)
            rec[name][act] = v
        trace.append(rec)
    st = np.zeros(B, ROW_DTYPE)
    st["T"], st["k_left"], st["cand"], st["src_n"] = T, k_left, cand, src_n
    st["out_ctr"], st["tie_ctr"] = k - k_left, cand
    st["mode"], st["in_buf"] = mode, in_buf
    return Selection(kb, L, k, cap, st, items, depth, reads, tuple(trace))


def select_keys(keys: np.ndarray, k: int, largest: bool) -> Selection:
    """`select` of raw keys (1-D or (B, L)) of one of the ten key types"""
    return select(O.order_key(np.ascontiguousarray(keys), up=not largest), k, keys.dtype.itemsize)


# ---------------------------------------------------------------------------------------------------------------
# Row generators.  Each takes (dtype, row_len, k, largest, rng), writes the row in ordered-key space, asserts through
# `select` that the row reaches the branch it is named for, and returns raw keys.  `applies(dtype, row_len, k)` tells
# whether the branch exists for those shapes.
# ---------------------------------------------------------------------------------------------------------------
def _rand(rng, lo: int, hi: int, n: int) -> np.ndarray:
    """n uniform integers in [lo, hi] as uint64"""
    return rng.integers(lo, hi, size=n, dtype=np.uint64, endpoint=True)


def _raw(u: np.ndarray, dtype, largest: bool) -> np.ndarray:
    dt = np.dtype(dtype)
    return from_order(np.asarray(u, np.uint64).astype(f"u{dt.itemsize}"), dt, up=not largest)


def _doc_cap(row_len: int) -> int:
    # the candidate buffer's documented size, ceil(row_len / 16) entries (DESIGN.md §4).  Deliberately not the
    # model's TOPK_CAP_DIV: the cap-boundary rows are built from the documented size and must reach the branch the
    # model's rule gives for them.
    return (row_len + 15) // 16


def _finish(u, dtype, k, largest, check, what):
    keys = _raw(u, dtype, largest)
    s = select_keys(keys, k, largest)
    assert check(s), f"{what} ({np.dtype(dtype).name}, row_len {len(u)}, k {k}) does not reach its branch"
    return keys


def gen_uniform(dtype, L, k, largest, rng):
    """uniform keys: pass 0 and pass 1 read the row, later passes read the candidate buffer (2 reads once L >= 1000)"""
    kb = np.dtype(dtype).itemsize
    u = _rand(rng, 0, (1 << 8 * kb) - 1, L)
    return _finish(u, dtype, k, largest, lambda s: L < 1000 or s.reads[0] == 2, "uniform")


def gen_equal(dtype, L, k, largest, rng):
    """all keys equal: every bucket holds the whole row; it finishes at the last digit (at digit 0 when k = L)"""
    kb = np.dtype(dtype).itemsize
    u = np.full(L, _rand(rng, 0, (1 << 8 * kb) - 1, 1)[0], np.uint64)
    return _finish(u, dtype, k, largest,
                   lambda s: s.state["cand"][0] == L and s.depth[0] == (0 if k == L else kb - 1), "all equal")


def gen_two_values(dtype, L, k, largest, rng):
    """two distinct values, k < L: the threshold's bucket ends up holding exactly the records of the k-th one's value"""
    kb = np.dtype(dtype).itemsize
    a, b = 0, 0
    while a == b:
        a, b = (int(x) for x in _rand(rng, 0, (1 << 8 * kb) - 1, 2))
    u = np.where(rng.random(L) < 0.5, np.uint64(a), np.uint64(b))
    u[:2] = a, b
    rng.shuffle(u)
    kth = np.sort(u)[k - 1]
    return _finish(u, dtype, k, largest, lambda s: s.state["cand"][0] == (u == kth).sum(), "two values")


def gen_const_top(j: int):
    """the top j bytes constant, digit j spread evenly, lower bytes uniform: passes 1 … j + 1 re-read the row (the
    top j buckets hold the whole row), later passes read the buffer: j + 2 reads of the row"""
    def gen(dtype, L, k, largest, rng):
        kb = np.dtype(dtype).itemsize
        low = 8 * (kb - 1 - j)
        top = _rand(rng, 0, (1 << 8 * j) - 1, 1)[0]
        dig = rng.permutation(np.arange(L, dtype=np.uint64) % np.uint64(RADIX))
        u = (top << np.uint64(8 * (kb - j))) | (dig << np.uint64(low)) | _rand(rng, 0, (1 << low) - 1, L)
        return _finish(u, dtype, k, largest, lambda s: s.reads[0] == j + 2, f"constant top {j} bytes")
    gen.applies = lambda dtype, L, k: j < np.dtype(dtype).itemsize and k < L
    gen.__name__ = f"gen_const_top{j}"
    return gen


def gen_early(dd: int):
    """the row finishes at decision dd because its bucket holds exactly the records still to select (cand == kl):
    the k-th and (k+1)-th records share their top dd digits and differ in digit dd; some records lie below or above
    that prefix"""
    def gen(dtype, L, k, largest, rng):
        kb = np.dtype(dtype).itemsize
        low = 8 * (kb - 1 - dd)
        qmax = (1 << 8 * dd) - 1
        q = int(_rand(rng, 0, qmax, 1)[0])
        x = int(rng.integers(0, 255))  # digit dd: [0, x] below the threshold's bucket boundary, [x + 1, 255] above

        def key(prefix, digit):
            n = len(digit)
            return ((np.asarray(prefix, np.uint64) << np.uint64(8 * (kb - dd))) | (digit.astype(np.uint64) << np.uint64(low))
                    | _rand(rng, 0, (1 << low) - 1, n))

        n_lo_out = int(rng.integers(0, k)) if q > 0 else 0
        n_hi_out = int(rng.integers(0, L - k)) if q < qmax else 0
        n_lo, n_hi = k - n_lo_out, L - k - n_hi_out
        parts = [key(q, rng.integers(0, x, n_lo, endpoint=True)), key(q, rng.integers(x + 1, 255, n_hi, endpoint=True))]
        if n_lo_out:
            parts.append(key(_rand(rng, 0, q - 1, n_lo_out), rng.integers(0, 255, n_lo_out, endpoint=True)))
        if n_hi_out:
            parts.append(key(_rand(rng, q + 1, qmax, n_hi_out), rng.integers(0, 255, n_hi_out, endpoint=True)))
        u = rng.permutation(np.concatenate(parts))
        return _finish(u, dtype, k, largest,
                       lambda s: s.depth[0] == dd and s.state["k_left"][0] == s.state["cand"][0], f"early finish at {dd}")
    gen.applies = lambda dtype, L, k: dd < np.dtype(dtype).itemsize and k < L
    gen.__name__ = f"gen_early{dd}"
    return gen


def _cap_kl_range(L: int, k: int, size: int) -> tuple:
    """the k_left values at which the k-th record falls inside a bucket of `size` records with kl < c, with the
    rest of the row split below and above it"""
    return max(1, k - (L - size)), min(size - 1, k)


def gen_cap(D: int, over: bool):
    """the k-th record's bucket at digit D holds exactly the documented buffer size (`over`: one more) with kl < c:
    pass D + 1 fills its candidate buffer to the last entry (`over`: the row is re-read by pass D + 2).  At D = 1
    every record shares digit 0, so pass 2 writes buffer 0 and pass 3 reads it with src_n = the buffer size."""
    def gen(dtype, L, k, largest, rng):
        kb = np.dtype(dtype).itemsize
        size = _doc_cap(L) + int(over)
        lo, hi = _cap_kl_range(L, k, size)
        kl = int(rng.integers(lo, hi, endpoint=True))
        below, above = k - kl, L - size - (k - kl)
        x = int(rng.integers(1, 254, endpoint=True))
        dig = np.concatenate([rng.integers(0, x - 1, below, endpoint=True), np.full(size, x),
                              rng.integers(x + 1, 255, above, endpoint=True)]).astype(np.uint64)
        low = 8 * (kb - 1 - D)
        u = (dig << np.uint64(low)) | _rand(rng, 0, (1 << low) - 1, L)
        if D == 1:
            u |= _rand(rng, 0, 255, 1)[0] << np.uint64(8 * (kb - 1))
        u = rng.permutation(u)

        def check(s):
            t = s.trace[D]
            return (t["c"][0] == size and t["kl"][0] < size and t["mode"][0] == ACTIVE and t["write_buf"][0] == (not over)
                    and (D == 0 or s.trace[0]["c"][0] == L))
        return _finish(u, dtype, k, largest, check, f"bucket of {'cap + 1' if over else 'cap'} at digit {D}")

    def applies(dtype, L, k):
        size = _doc_cap(L) + int(over)
        lo, hi = _cap_kl_range(L, k, size)
        return D < np.dtype(dtype).itemsize - 1 and 2 <= size <= L and lo <= hi and (D == 0 or k < L)
    gen.applies = applies
    gen.__name__ = f"gen_cap{'_over' if over else ''}_d{D}"
    return gen


def gen_run(dtype, L, k, largest, rng):
    """the k-th place inside a run of equal keys with records below and above it: k_left < cand at the last digit"""
    kb = np.dtype(dtype).itemsize
    top = (1 << 8 * kb) - 1
    R = int(rng.integers(max(2, L // 4), L, endpoint=True))
    lo, hi = max(0, k - R + 1), min(k - 1, L - R)
    if lo > hi:
        R, lo, hi = L, 0, 0
    n_below = int(rng.integers(lo, hi, endpoint=True))
    n_above = L - R - n_below
    v = int(_rand(rng, 1 if n_below else 0, top - 1 if n_above else top, 1)[0])
    # half of the others anywhere below / above the run, half within 4096 of it (sharing its top digits)
    below = np.where(rng.random(n_below) < 0.5, _rand(rng, 0, v - 1, n_below), _rand(rng, max(0, v - 4096), v - 1, n_below))
    above = np.where(rng.random(n_above) < 0.5, _rand(rng, v + 1, top, n_above),
                     _rand(rng, v + 1, min(top, v + 4096), n_above))
    u = rng.permutation(np.concatenate([below, np.full(R, v, np.uint64), above]).astype(np.uint64))
    return _finish(u, dtype, k, largest, lambda s: s.depth[0] == kb - 1 and s.state["k_left"][0] < s.state["cand"][0]
                   and s.state["cand"][0] == R, "k-th place inside a run")


def float_specials(dtype) -> np.ndarray:
    """raw bit patterns (as the float dtype) of ±0, ±inf, NaNs of both signs with distinct payloads (quiet and
    signalling), the smallest and largest denormals of both signs, and the smallest normals"""
    dt = np.dtype(dtype)
    if dt == np.float32:
        bits = [0x00000000, 0x80000000, 0x7F800000, 0xFF800000, 0x7FC00000, 0x7FC00001, 0x7F800001, 0x7F800002,
                0x7FFFFFFF, 0xFFC00000, 0xFFC00001, 0xFF800001, 0xFFFFFFFF, 0x00000001, 0x00000002, 0x007FFFFF,
                0x80000001, 0x80000002, 0x807FFFFF, 0x00800000, 0x80800000]
        return np.array(bits, np.uint32).view(np.float32)
    bits = [0x0000000000000000, 0x8000000000000000, 0x7FF0000000000000, 0xFFF0000000000000, 0x7FF8000000000000,
            0x7FF8000000000001, 0x7FF0000000000001, 0x7FF0000000000002, 0x7FFFFFFFFFFFFFFF, 0xFFF8000000000000,
            0xFFF8000000000001, 0xFFF0000000000001, 0xFFFFFFFFFFFFFFFF, 0x0000000000000001, 0x0000000000000002,
            0x000FFFFFFFFFFFFF, 0x8000000000000001, 0x8000000000000002, 0x800FFFFFFFFFFFFF, 0x0010000000000000,
            0x8010000000000000]
    return np.array(bits, np.uint64).view(np.float64)


def gen_specials(dtype, L, k, largest, rng):
    """a row of float specials only, each present once the row is long enough: the k-th place falls among ±0, NaN
    patterns of both signs, ±inf and denormals (some of which differ only in the lowest digit)"""
    sp = float_specials(dtype)
    raw = sp[rng.integers(0, len(sp), L)]
    raw[:min(L, len(sp))] = sp[:min(L, len(sp))]
    raw = rng.permutation(raw)
    u = O.order_key(raw, up=not largest)
    kth = np.sort(u)[k - 1]
    spu = O.order_key(sp, up=not largest)
    return _finish(u, dtype, k, largest, lambda s: (spu == kth).any(), "float specials")


gen_uniform.applies = lambda dtype, L, k: True
gen_equal.applies = lambda dtype, L, k: True
gen_two_values.applies = lambda dtype, L, k: k < L
gen_run.applies = lambda dtype, L, k: L >= 2 and k < L
gen_specials.applies = lambda dtype, L, k: np.dtype(dtype).kind == "f"

GENERATORS = ([gen_uniform, gen_equal, gen_two_values] + [gen_const_top(j) for j in range(1, 8)]
              + [gen_early(d) for d in range(8)] + [gen_cap(D, over) for D in (0, 1) for over in (False, True)]
              + [gen_run, gen_specials])


def generators(dtype, L: int, k: int) -> list:
    """the generators whose branch exists for rows of `dtype`, row_len L and this k"""
    return [g for g in GENERATORS if g.applies(dtype, L, k)]


def mixed_rows(dtype, B: int, L: int, k: int, largest: bool, rng) -> np.ndarray:
    """(B, L) keys whose row r comes from generator r % G of the G that apply"""
    gens = generators(dtype, L, k)
    return np.stack([gens[r % len(gens)](dtype, L, k, largest, rng) for r in range(B)])
