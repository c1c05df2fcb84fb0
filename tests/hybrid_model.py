"""An exact numpy model of the MSB hybrid path of 8-byte keys and of its four finishes (TEST INFRASTRUCTURE ONLY),
and named key-set generators that each reach one branch of it.

The hybrid path sweeps only the top digits.  What is left -- runs of keys that agree on every swept bit ("segments")
-- is ordered by the last pass (runs a tile holds), the junction kernel (segments across a tile boundary), the
segment finish or the fall-back to the digit-by-digit path.  Which one runs is decided by two device flags.  A wrong
finish does not fault: it leaves a few records out of order for one key shape, or runs a full extra pass.  So the
tests compare the statistics of every sort with `predict`, which restates the rules, and the CPU tests check that the
emulated finishes order exactly what the design says they order.  Where each rule comes from
(simd-radix-sort_b200/csrc):

- kernels.cuh, probe_kernel: below the sparse-sampling size (b200sort.cu, DevSort::make_plan: n / hist_tile_keys
  >= 8192) every key feeds the digit histograms, so `entropies` are those of all order-mapped keys.
- kernels.cuh, scan_kernel (hybrid branch):
  - entropy of position p = log2 m - sum(c log2 c) / m, computed in float32 with log2f: `Ambiguous` is raised when a
    sum it compares lies within AMBIGUITY_BITS of its threshold;
  - `choose_cut`: from the top position down add the entropies of positions not skipped; the cut is the first p at
    which the sum reaches need = log2 n + margin_bits; a cut that saves fewer than two sweeps is no cut;
  - the left-shift variant: l = clz(varying) & 7 (8-byte keys, allow_lshift); shifted entropies spread each
    position's entropy evenly over its varying bits; taken iff cut2 != 0 and it sweeps fewer positions;
  - range reduction (allow_reduce, mn != 0, digits of the exact range < planned) clears the cut and the shift;
  - hist_done: the probe's guessed digit (b200sort.cu, make_plan: cut = 8 - ceil(need / 8) if >= 2, else 0) is the
    first executed one, and neither a subtraction nor a shift is planned.
- b200sort.cu, DevSort::run_passes: use_fix = plan read back, cut != 0, not partial, SoA keys or a key chunk >= 8,
  tile_cfg == kDefaultTileCfg, fix_in_pass.  Tile sizes: sweep_select.cuh, kTileCfgs (cfg 0: 256 x 16 = 4096 keys,
  cfg 1: 256 x 8 = 2048 keys and no FIX pass).  launch_sweep: the FIX pass is always stable; with the plan read back
  and first_atomic the first executed pass ranks unstably unless its digit is skewed (entropy < 5).
- kernels.cuh, onesweep_kernel<..., FIX>: a tile is staged in stable bucket order; runs of keys that agree on the
  swept bits (>= cut_bit = 8 cut - lshift of the raw key) of at most FIX_CAP + 1 keys are put in full-key order; a
  longer run raises flags[1] if one of its adjacent pairs is inverted.  jtable: 32-bit fingerprints (hi ^ lo of the
  masked raw key) of the first and last key of every (tile, bucket) part.
- hybrid.cuh, junction_fix_kernel: thread (t, d) with g = look-back prefix of tile t, g_end of the last tile, g_prev
  of tile t - 1 (-1 for t = 0) works iff g < g_end, g > 0, g != g_prev; candidate by fingerprints when the next tile
  has keys in the bucket (g_next != g) and the table is on, else by a key compare at g - 1, g; the segment around g
  is extended at most JF_CAP + 1 keys either way; len > JF_CAP raises flags[1] iff the keys at g - 1, g are
  inverted; lo < g_prev leaves it to the earlier junction's thread; else swap (len 2) or stable rank order.
- hybrid.cuh, segfix_kernel: chunks of SF_CHUNK positions with SF_HALO keys either side; heads where the swept bits
  change; the start / end of a position's segment are searched in its 32-position word and the one before / after;
  a segment is long if either is not found or it has more than SF_MAXSEG keys; the chunk holding the head orders a
  short one; a long one must be one repeated key (else flags[0]: fall-back).  It returns at once when cut == 0.
  flags[2] counts the queued moves: every position when the data lies in the shadow (final_sel 1), else the
  displaced members of short segments.
- b200sort.cu, DevSort::finish / statistics / fall_back: the launches of each flow; segfix_passes; algorithmic_bytes =
  hist_sweeps n K + (passes_planned + segfix_passes) 2 n R; the fall-back adds the LSD sort's own statistics.
"""
from __future__ import annotations

import math
from collections import Counter
from dataclasses import dataclass, field

import numpy as np

import oracle_lib as O
from plan_model import digits_of_range, from_order, lsd_plan

KB = 8
RADIX = 256
FIX_CAP = 8          # kernels.cuh: longest run - 1 the last pass orders
JF_CAP = 32          # hybrid.cuh: longest segment the junction kernel orders
SF_MAXSEG = 32       # hybrid.cuh: longest segment the segment finish orders (= SF_HALO)
SF_CHUNK = 256       # hybrid.cuh: positions of one warp
WORD = 32            # hybrid.cuh: head flags are ballot words of 32 positions
TILE_OF_CFG = {0: 4096, 1: 2048}  # sweep_select.cuh, kTileCfgs (threads x ipt)
DEFAULT_TILE_CFG = 0
AMBIGUITY_BITS = 0.25
M64 = (1 << 64) - 1


class Ambiguous(ValueError):
    """a sum the float32 plan compares lies too close to its threshold for the model to say which way it goes"""


def _u(x) -> np.uint64:
    return np.uint64(x)


def entropies(w: np.ndarray) -> list:
    """entropy (bits) of each digit position of the keys w (float64)"""
    n = len(w)
    out = []
    for p in range(KB):
        c = np.bincount(((w >> _u(8 * p)) & _u(255)).astype(np.int64), minlength=RADIX).astype(np.float64)
        c = c[c > 0]
        out.append(max(math.log2(n) - float(np.sum(c * np.log2(c))) / n, 0.0))
    return out


def _choose_cut(ent, skip, need, gaps):
    skip = list(skip)
    c, acc = 0, 0.0
    for p in range(KB - 1, -1, -1):
        if not skip[p]:
            acc += ent[p]
        gaps.append(acc - need)
        if acc >= need:
            c = p
            break
    if sum(1 for p in range(c) if not skip[p]) < 2:
        c = 0
    for p in range(c):
        skip[p] = True
    return c, skip, KB - sum(skip)


@dataclass(frozen=True)
class HybridPlan:
    n: int
    varying: int
    entropies: tuple
    cut_digit: int
    lshift: int
    sub: int
    skip: tuple
    n_exec: int
    final_sel: int       # side holding the result after the last executed pass (0 = the caller's arrays)
    first_exec_p1: int
    top_p1: int          # digit position + 1 of the last executed pass (0: none)
    skewed: tuple
    hist_done: bool
    want_minmax: bool    # host-plan flow: minmax_kernel and a second scan run

    @property
    def cut_bit(self) -> int:
        """lowest swept bit of the unshifted order-mapped key"""
        return 8 * self.cut_digit - self.lshift

    def plan_keys(self, u: np.ndarray) -> np.ndarray:
        """the keys every kernel of the sort compares: (order-mapped key - sub) << lshift"""
        return (u - _u(self.sub)) << _u(self.lshift)


def hybrid_plan(keys: np.ndarray, up: bool = True, *, margin_bits: int = 2, allow_skip: int = 1, allow_reduce: int = 1,
                allow_lshift: int = 1, probe_guess: int = 1) -> HybridPlan:
    """The plan scan_kernel makes for 8-byte `keys` on the hybrid path (probe without sparse sampling)."""
    u = O.order_key(np.ascontiguousarray(keys).reshape(-1), up)
    n = len(u)
    if keys.dtype.itemsize != KB or n == 0:
        raise ValueError("the hybrid path sorts 8-byte keys")
    if n // 4096 >= 8192:
        raise ValueError("the probe samples sparsely at this size: not modelled")
    varying = int(np.bitwise_or.reduce(u)) & int(np.bitwise_or.reduce(~u))
    skip = [bool(allow_skip) and ((varying >> (8 * p)) & 0xFF) == 0 for p in range(KB)]
    n_const = sum(skip)
    ent = entropies(u)
    need = math.log2(n) + margin_bits
    gaps = []
    cut, skip1, n1 = _choose_cut(ent, skip, need, gaps)
    lshift, ent_used = 0, ent
    l = (64 - varying.bit_length()) & 7 if (allow_lshift and varying != 0) else 0
    if l:
        v2 = (varying << l) & M64
        ent2, skip2 = [], []
        for p in range(KB):
            vb = (varying >> (8 * p)) & 0xFF
            vb_lo = (varying >> (8 * (p - 1))) & 0xFF if p > 0 else 0
            n_all, n_take = bin(vb).count("1"), bin(vb & (0xFF >> l)).count("1")
            m_all, m_take = bin(vb_lo).count("1"), bin(vb_lo & ~(0xFF >> l) & 0xFF).count("1")
            e = 0.0
            if n_all:
                e += ent[p] * n_take / n_all
            if m_all:
                e += ent[p - 1] * m_take / m_all
            ent2.append(e)
            skip2.append(bool(allow_skip) and ((v2 >> (8 * p)) & 0xFF) == 0)
        cut2, skip2, n2 = _choose_cut(ent2, skip2, need, gaps)
        if cut2 != 0 and n2 < n1:
            lshift, cut, skip1, ent_used = l, cut2, skip2, ent2
    if any(abs(g) < AMBIGUITY_BITS for g in gaps):
        raise Ambiguous(f"entropy sums {gaps} against need {need}")
    mn, mx = int(u.min()), int(u.max())
    planned = (1 if cut else 0) + KB - sum(skip1)
    reduce = bool(allow_reduce) and mn != 0 and digits_of_range(mn, mx) < planned
    sub = 0
    skewed = [e < 5.0 for e in ent_used]
    if reduce:
        rb = digits_of_range(mn, mx)
        sub, cut, lshift = mn, 0, 0
        skip1 = [p >= rb for p in range(KB)]
        skewed = [True] * KB
    # (the host-plan flow sees the exact range only after minmax_kernel, which it runs iff the probe's range -- here
    #  the exact one -- says that range reduction may pay: exactly when it does; the second scan makes the plan above)
    want_minmax = reduce
    execd = [p for p in range(KB) if not skip1[p]]
    guess = 8 - math.ceil(need / 8.0)
    guess_p1 = (guess if guess >= 2 else 0) + 1 if probe_guess else 0
    first_p1 = execd[0] + 1 if execd else 0
    hist_done = guess_p1 != 0 and first_p1 == guess_p1 and sub == 0 and lshift == 0
    return HybridPlan(n, varying, tuple(ent_used), cut, lshift, sub, tuple(skip1), len(execd), len(execd) & 1, first_p1,
                      execd[-1] + 1 if execd else 0, tuple(skewed), hist_done, want_minmax)


# ---------------------------------------------------------------------------------------------------------------------
# the finishes, on the plan keys w (and the raw keys for the fingerprints); every function returns what it did
# ---------------------------------------------------------------------------------------------------------------------
def _runs(prefix: np.ndarray, breaks: np.ndarray = None):
    """(start, length) of the maximal runs of equal prefixes; `breaks`: positions where a run must also start"""
    n = len(prefix)
    head = np.ones(n, bool)
    head[1:] = prefix[1:] != prefix[:-1]
    if breaks is not None:
        head |= breaks
    starts = np.flatnonzero(head)
    return starts, np.diff(np.append(starts, n))


@dataclass
class Finish:
    """what the finishes did to one sort: the output, the flags, and which branch every run / junction / segment took"""
    w: np.ndarray                  # plan keys, in output order
    ids: np.ndarray                # input position of each output record
    fix_flag: bool = False         # flags[1] raised by the last pass
    junction_flag: bool = False    # flags[1] raised by the junction kernel
    fall_back: bool = False        # flags[0] raised by the segment finish
    segfix_ran: bool = False
    segfix_moved: int = 0
    fix_runs: Counter = field(default_factory=Counter)    # (length, "ordered" | "long_in_order" | "long_inverted")
    fix_moved_runs: Counter = field(default_factory=Counter)  # lengths of ordered runs in which a key moved
    # (kind, length) of every segment a junction thread found: swap / rank (ordered it), in_order (nothing to move),
    # owned_by_earlier (left to an earlier junction), long_in_order / long_inverted (length 0: too long; flag if inverted)
    junctions: Counter = field(default_factory=Counter)
    direct_compares: int = 0       # candidates found by the key compare (next tile without keys in the bucket)
    collisions: int = 0            # equal fingerprints, different segments
    tiles_spanned: Counter = field(default_factory=Counter)  # junction segments ordered, by tiles they span
    segfix_segments: Counter = field(default_factory=Counter)  # ("short" | "long_equal" | "long_distinct", length)
    segfix_chunk_crossers: int = 0  # short segments with keys in two chunks
    slot0_hw1_short: int = 0       # tiles whose slot 0 is a key with raw high word 1 in a run of <= FIX_CAP + 1 keys


def fix_pass(x: np.ndarray, ids: np.ndarray, top: int, wbit: int, raw: np.ndarray, raw_bit: int, tile: int,
             fix_cap: int = FIX_CAP):
    """The last pass with the FIX ordering, on its input x (plan keys, swept bits >= wbit; the raw keys' swept bits
    are those >= raw_bit) -> (Finish, look-back prefixes G[t][d], fingerprints of the first / last key of every
    (tile, bucket) part).  The kernel's 32-bit compare (raw_bit >= 32) is the same decision on the raw high word."""
    n = len(x)
    n_tiles = -(-n // tile)
    ti = np.arange(n) // tile
    dig = ((x >> _u(8 * top)) & _u(255)).astype(np.int64)
    order = np.lexsort((np.arange(n), dig, ti))  # staged: by tile, then bucket, stable
    xs, ids_s, raws, tis, ds = x[order], ids[order], raw[order], ti[order], dig[order]
    pref = xs >> _u(wbit)
    starts, lens = _runs(pref, np.r_[True, tis[1:] != tis[:-1]])
    res = Finish(xs, ids_s)
    run_of = np.repeat(np.arange(len(starts)), lens)
    short = np.repeat(lens <= fix_cap + 1, lens)
    inv = np.zeros(n, bool)
    inv[1:] = (run_of[1:] == run_of[:-1]) & (xs[1:] < xs[:-1])
    inv_run = np.zeros(len(starts), bool)
    np.logical_or.at(inv_run, run_of[inv], True)
    for s, ln, iv in zip(starts, lens, inv_run):
        if ln >= 2:
            res.fix_runs[(int(ln), "ordered" if ln <= fix_cap + 1 else ("long_inverted" if iv else "long_in_order"))] += 1
            if ln <= fix_cap + 1 and iv:
                res.fix_moved_runs[int(ln)] += 1
    res.fix_flag = bool(np.any(inv_run & (lens > fix_cap + 1)))
    # slot 0 of a tile holding a key whose raw high word is 1 (the 32-bit compare's out-of-tile placeholder), in a short run
    if raw_bit >= 32:
        first = np.flatnonzero(np.r_[True, tis[1:] != tis[:-1]])
        hw1 = (raws[first] >> _u(32)) == 1
        res.slot0_hw1_short = int(np.sum(hw1 & short[first]))
    within = np.lexsort((np.arange(n), np.where(short, xs, _u(0)), run_of))
    xs, ids_s, raws, ds, tis = xs[within], ids_s[within], raws[within], ds[within], tis[within]
    # the tile's parts of every bucket, at their global places: a stable sort of the staged tiles by bucket
    glob = np.argsort(ds, kind="stable")
    cnt = np.zeros((n_tiles, RADIX), np.int64)
    np.add.at(cnt, (tis, ds), 1)
    bstart = np.concatenate([[0], np.cumsum(cnt.sum(0))[:-1]])
    G = bstart[None, :] + np.cumsum(cnt, 0)
    m = (raws >> _u(raw_bit)) << _u(raw_bit)
    fp = ((m >> _u(32)) ^ (m & _u(0xFFFFFFFF))).astype(np.uint64)
    fp_first = np.zeros((n_tiles, RADIX), np.uint64)
    fp_last = np.zeros((n_tiles, RADIX), np.uint64)
    part_head = np.r_[True, (tis[1:] != tis[:-1]) | (ds[1:] != ds[:-1])]
    part_tail = np.r_[part_head[1:], True]
    fp_first[tis[part_head], ds[part_head]] = fp[part_head]
    fp_last[tis[part_tail], ds[part_tail]] = fp[part_tail]
    res.w, res.ids = xs[glob], ids_s[glob]
    return res, G, fp_first, fp_last


def junction_fix(res: Finish, G: np.ndarray, fp_first, fp_last, wbit: int, use_table: bool = True,
                 jf_cap: int = JF_CAP) -> Finish:
    """junction_fix_kernel on the output of the last pass (res.w / res.ids, in place); swept bits >= wbit"""
    w, ids = res.w, res.ids
    n = len(w)
    n_tiles = G.shape[0]
    pre = w >> _u(wbit)
    part_start = np.vstack([np.r_[0, G[-1][:-1]], G[:-1]])  # (bucket d starts where bucket d - 1 ends)
    for t in range(n_tiles - 1):
        g_row, g_end = G[t], G[n_tiles - 1]
        g_prev_row = G[t - 1] if t > 0 else np.full(RADIX, -1)
        work = np.flatnonzero((g_row < g_end) & (g_row > 0) & (g_row != g_prev_row))
        for d in work:
            g, g_prev, g_next = int(g_row[d]), int(g_prev_row[d]), int(G[t + 1][d])
            if use_table and g_next != g:
                cand = fp_last[t][d] == fp_first[t + 1][d]
            else:
                cand = pre[g - 1] == pre[g]
                res.direct_compares += int(cand)
            if not cand:
                continue
            if pre[g - 1] != pre[g]:
                res.collisions += 1
                continue
            lo, hi = g - 1, g + 1
            while lo > 0 and g - lo <= jf_cap and pre[lo - 1] == pre[g]:
                lo -= 1
            while hi < n and hi - g <= jf_cap and pre[hi] == pre[g]:
                hi += 1
            ln = hi - lo
            if ln > jf_cap:
                inverted = bool(w[g] < w[g - 1])
                res.junctions[("long_inverted" if inverted else "long_in_order", 0)] += 1
                res.junction_flag |= inverted
                continue
            if lo < g_prev:
                res.junctions[("owned_by_earlier", ln)] += 1
                continue
            o = np.argsort(w[lo:hi], kind="stable")
            moved = bool(np.any(o != np.arange(ln)))
            res.junctions[("swap" if ln == 2 else "rank", ln) if moved else ("in_order", ln)] += 1
            # tiles whose (non-empty) part of the bucket holds keys of [lo, hi)
            ps, pe = part_start[:, d], G[:, d]
            res.tiles_spanned[int(np.sum((pe > ps) & (ps < hi) & (pe > lo)))] += 1
            w[lo:hi], ids[lo:hi] = w[lo:hi][o], ids[lo:hi][o]
    return res


def segfix(w: np.ndarray, ids: np.ndarray, wbit: int, sel: int, res: Finish, chunk: int = SF_CHUNK,
           maxseg: int = SF_MAXSEG, word: int = WORD) -> Finish:
    """segfix_kernel: every chunk classifies its own positions with the kernel's windowed start / end search (halo =
    maxseg keys either side), then the short segments are put in stable full-key order"""
    n = len(w)
    halo = maxseg
    W = chunk + 2 * halo
    pre = w >> _u(wbit)
    cls = np.zeros(n, np.int8)   # 0: one-key segment, 1: long, 2: member of a short segment
    for s0 in range(0, n, chunk):
        e0 = min(s0 + chunk, n)
        w0, w1 = max(s0 - halo, 0), min(e0 + halo, n)
        wn = w1 - w0
        h = np.zeros(W + 2 * word, bool)   # head flags of the window (+ the word after it)
        pw = pre[w0:w1]
        h[1:wn] = pw[1:] != pw[:-1]
        h[0] = w0 == 0                     # unknown unless the array starts here
        h[wn] = w1 == n                    # the array end closes the last segment
        pos = np.arange(s0 - w0, e0 - w0)  # the chunk's own positions
        j = pos // word
        heads = np.r_[-W, np.flatnonzero(h), 3 * W]  # (sentinels: no head found)
        k = np.searchsorted(heads, pos, side="right")
        st = np.where(heads[k - 1] >= (j - 1) * word, heads[k - 1], -1)    # in this word or the one before
        en = np.where(heads[k] <= (j + 2) * word - 1, heads[k], -1)        # in this word or the one after
        one = h[pos] & h[pos + 1]
        long_ = ~one & ((st < 0) | (en < 0) | (en - st > maxseg))
        keys = w[w0:w1]
        if np.any(long_ & (pos > 0) & ~h[pos] & (keys[pos] != keys[pos - 1])):
            res.fall_back = True
        cls[w0 + pos] = np.where(one, 0, np.where(long_, 1, 2))
    head = np.r_[True, pre[1:] != pre[:-1]]
    seg = np.cumsum(head) - 1
    short = cls == 2
    order = np.lexsort((np.arange(n), np.where(short, w, _u(0)), seg))
    displaced = order != np.arange(n)
    res.segfix_moved = n if sel != 0 else int(np.sum(displaced & short))
    starts, lens = _runs(pre)
    for s, ln in zip(starts, lens):
        if ln > maxseg:
            res.segfix_segments[("long_equal" if np.all(w[s:s + ln] == w[s]) else "long_distinct", int(ln))] += 1
        elif ln >= 2:
            res.segfix_segments[("short", int(ln))] += 1
            res.segfix_chunk_crossers += int(s // chunk != (s + ln - 1) // chunk)
    res.segfix_ran = True
    res.w, res.ids = w[order], ids[order]
    return res


# ---------------------------------------------------------------------------------------------------------------------
# one sort: plan, passes, finishes, statistics
# ---------------------------------------------------------------------------------------------------------------------
FLOWS = ("device", "host")  # host_plan_min_log2 above / at most log2 n: the plan is made on the device / read back


@dataclass
class Prediction:
    plan: HybridPlan
    flow: str
    use_fix: bool
    tie_dependent: bool     # the first executed pass ranks unstably: the order of ties in the last pass is not known
    finish: Finish          # the emulation (for the stable tie order when tie_dependent)
    stats: dict             # what last_stats() reports; a value of None is timing-dependent
    flags_tie_free: bool    # the flags (and so segfix_passes / fell_back) are the same for every tie order

    @property
    def flag(self) -> bool:
        return self.finish.fix_flag or self.finish.junction_flag


def predict(keys: np.ndarray, up: bool, flow: str, *, record_bytes: int = 8, margin_bits: int = 2,
            first_atomic: int = 1, fix_in_pass: int = 1, junction_table: int = 1, tile_cfg: int = DEFAULT_TILE_CFG,
            allow_skip: int = 1, allow_reduce: int = 1, allow_lshift: int = 1, probe_guess: int = 1,
            tile: int = None, fix_cap: int = FIX_CAP, jf_cap: int = JF_CAP, sf_chunk: int = SF_CHUNK,
            sf_maxseg: int = SF_MAXSEG, word: int = WORD) -> Prediction:
    """What a hybrid sort (algo = 2) of 8-byte SoA keys or records (key chunk >= 8 bytes) does in `flow`; `tile` and
    the caps default to the library's."""
    keys = np.ascontiguousarray(keys).reshape(-1)
    n = len(keys)
    opts = dict(allow_skip=allow_skip, allow_reduce=allow_reduce, probe_guess=probe_guess)
    plan = hybrid_plan(keys, up, margin_bits=margin_bits, allow_lshift=allow_lshift, **opts)
    u = O.order_key(keys, up)
    raw = keys.view(np.uint64)
    w = plan.plan_keys(u)
    cut = plan.cut_digit
    host = flow == "host"
    use_fix = host and cut != 0 and tile_cfg == DEFAULT_TILE_CFG and fix_in_pass != 0
    tile = tile or TILE_OF_CFG[tile_cfg]
    execd = [p for p in range(KB) if not plan.skip[p]]
    # a stable first pass unless the plan is read back, first_atomic is on and the first digit is not skewed (the
    # FIX pass, which may be the only one, is always stable)
    tie_dependent = (host and first_atomic != 0 and bool(execd) and not plan.skewed[execd[0]]
                     and not (use_fix and len(execd) == 1))
    if tie_dependent and abs(plan.entropies[execd[0]] - 5.0) < AMBIGUITY_BITS:
        raise Ambiguous("skew of the first executed digit")
    ids = np.arange(n)
    top = execd[-1] if execd else 0
    wbit = 8 * cut
    if use_fix:
        # the last pass's input: the keys stably sorted by the swept digits below its own
        below = np.zeros(n, np.uint64)
        for p in execd[:-1]:
            below |= w & _u(0xFF << (8 * p))
        xo = np.argsort(below, kind="stable")
        res, G, fpf, fpl = fix_pass(w[xo], ids[xo], top, wbit, raw[xo], plan.cut_bit, tile, fix_cap)
        if not res.fix_flag:
            junction_fix(res, G, fpf, fpl, wbit, junction_table != 0, jf_cap)
        if res.fix_flag or res.junction_flag:
            segfix(res.w, res.ids, wbit, plan.final_sel, res, sf_chunk, sf_maxseg, word)
    else:
        swept = np.zeros(n, np.uint64)
        for p in execd:
            swept |= w & _u(0xFF << (8 * p))
        o = np.argsort(swept, kind="stable")
        res = Finish(w[o], ids[o])
        if cut != 0:
            segfix(res.w, res.ids, wbit, plan.final_sel, res, sf_chunk, sf_maxseg, word)
    fell = res.fall_back
    # statistics (b200sort.cu: DevSort::make_plan, finish, statistics, fall_back)
    if host:
        hist_sweeps = 1 + int(plan.want_minmax) + (0 if plan.hist_done else 1)
        launches = 2 + 2 * int(plan.want_minmax) + (0 if plan.hist_done else 1) + plan.n_exec
        if use_fix:
            launches += 2 + (1 if plan.final_sel == 1 else 0)  # junction kernel, gated finish, gated copy-back
        else:
            launches += 2 if cut != 0 else 1                  # (finish,) copy-back
    else:
        hist_sweeps, launches = 2, 3 + KB + 2  # probe, scan, hist_kernel, every pass, finish, copy-back
    segfix_passes = int(res.segfix_ran)
    if use_fix:
        moved = 0 if not res.segfix_ran else (n if plan.final_sel == 1 else None)  # (s_given_up: which tiles gave up)
    else:
        moved = res.segfix_moved if cut != 0 else 0
        if tie_dependent and cut != 0 and plan.final_sel == 0:
            moved = None
    rb = record_bytes
    stats = {"algo": 2, "cut_digit": cut, "passes_planned": plan.n_exec, "hist_sweeps": hist_sweeps,
             "kernel_launches": launches, "segfix_passes": segfix_passes, "fell_back": int(fell), "segfix_moved": moved,
             "algorithmic_bytes": hist_sweeps * n * KB + (plan.n_exec + segfix_passes) * 2 * n * rb}
    if fell:
        lp = lsd_plan(keys, up, **opts)
        ls = lp.host_flow_stats if host else lp.device_flow_stats
        for f in ("passes_planned", "hist_sweeps", "kernel_launches"):
            stats[f] += ls[f]
        stats["algorithmic_bytes"] += ls["hist_sweeps"] * n * KB + ls["passes_planned"] * 2 * n * rb
        o = np.argsort(res.w, kind="stable")  # the digit-by-digit sort of the array as the hybrid left it
        res.w, res.ids = res.w[o], res.ids[o]
    # every tie order gives the same flags when no segment longer than FIX_CAP + 1 holds two different keys
    sw = np.sort(w)
    starts, lens = _runs(sw >> _u(wbit)) if cut else (np.zeros(0, int), np.zeros(0, int))
    flags_tie_free = not tie_dependent or all(sw[s] == sw[s + ln - 1] for s, ln in zip(starts, lens) if ln > fix_cap + 1)
    return Prediction(plan, flow, use_fix, tie_dependent, res, stats, flags_tie_free)


# ---------------------------------------------------------------------------------------------------------------------
# generators.  Keys are built as order-mapped values u = top | mid | low for the direction of the sort and mapped back
# (plan_model.from_order), so one generator makes the same shape for u64, i64 and f64 in both directions:
#   top: the digit the last pass sweeps (bits 56 - l .. 63 - l under a left shift by l);
#   mid: the swept bits below it, non-decreasing over the array -- so the caller's array IS the last pass's input
#        (it is already ordered by the lower swept digits), and the tile that holds a key is known;
#   low: the bits below the cut (the full-key order inside a segment).
# With sort_prefix the array is ordered by top | mid as well: the segment finish's input is then the array itself.
# Random top and mid bits give each swept digit about 8 bits of entropy, so need = log2 n + margin with
# margin = 8 (8 - cut) - 4 - log2 n puts the cut at `cut`, 4 bits away from either neighbour.
# ---------------------------------------------------------------------------------------------------------------------
def _interleave(v, sizes):
    """the ascending values v dealt round-robin to parts of these sizes, the last part first: every part ascending,
    and the first value of each part below the last value of the part before it (an inverted junction)"""
    parts = [[] for _ in sizes]
    order = [i for i in reversed(range(len(sizes)))]
    k = 0
    for x in v:
        while len(parts[order[k % len(order)]]) >= sizes[order[k % len(order)]]:
            k += 1
        parts[order[k % len(order)]].append(x)
        k += 1
    return [np.array(p, dtype=np.uint64) for p in parts]


class KeyBuilder:
    def __init__(self, n, cut, rng, lshift=0, sort_prefix=False, tile=TILE_OF_CFG[0]):
        self.n, self.cut, self.l, self.rng, self.tile, self.sort_prefix = n, cut, lshift, rng, tile, sort_prefix
        self.cb = 8 * cut - lshift          # lowest swept bit of u
        self.mb = 56 - 8 * cut              # bits of mid
        self.top = rng.integers(0, 256, n).astype(np.uint64)
        self.mid = np.sort(rng.integers(0, 1 << self.mb, n, dtype=np.uint64))
        self.low = rng.integers(0, 1 << self.cb, n, dtype=np.uint64)
        if sort_prefix:
            o = np.lexsort((self.mid, self.top))
            self.top, self.mid = self.top[o], self.mid[o]
        self.margin = int(round(8 * (8 - cut) - 4 - math.log2(n)))

    def distinct_lows(self, k):
        """k distinct low parts, ascending"""
        while True:
            v = np.unique(self.rng.integers(0, 1 << self.cb, k, dtype=np.uint64))
            if len(v) == k:
                return v

    def segment(self, a, lows, top=None):
        """positions a .. a + len(lows) - 1 become one segment (one prefix) with these low parts"""
        k = len(lows)
        self.top[a:a + k] = self.top[a] if top is None else top
        self.mid[a:a + k] = self.mid[a]
        if not self.sort_prefix:
            self.mid[a + k:] = np.maximum(self.mid[a + k:], self.mid[a])
        self.low[a:a + k] = lows
        return self

    def across(self, J, kl, kr, how="interleaved", top=None):
        """a segment of kl keys ending at position J - 1 and kr keys starting at J, each part ascending; `how`:
        interleaved (the junction has to merge them), in_order (left part below right part), inverted (above)"""
        v = self.distinct_lows(kl + kr)
        if how == "interleaved":
            left, right = _interleave(v, [kl, kr])
        elif how == "in_order":
            left, right = v[:kl], v[kl:]
        else:
            left, right = v[kr:], v[:kr]
        return self.segment(J - kl, np.r_[left, right], top)

    def spanning(self, t, kl, k_mid, kr, how="interleaved"):
        """a segment of kl keys at the end of tile t, k_mid keys inside tile t + 1 and kr keys at the start of tile
        t + 2.  Every key of tile t + 1 then has the segment's mid: its other keys take other top digits, in
        ascending order per digit (long runs, in order)"""
        T = self.tile
        a, b = (t + 1) * T, (t + 2) * T
        topP = int(self.top[a - kl])
        mid = self.mid[a - kl]
        self.mid[a - kl:b + kr] = mid
        self.mid[b + kr:] = np.maximum(self.mid[b + kr:], mid)
        others = self.rng.permutation(np.arange(T) % 255).astype(np.uint64)  # at most 17 keys per digit
        self.top[a:b] = np.where(others >= topP, others + 1, others)
        self.low[a:b] = np.sort(self.rng.integers(0, 1 << self.cb, T, dtype=np.uint64))
        v = self.distinct_lows(kl + k_mid + kr)
        if how == "interleaved":
            left, midp, right = _interleave(v, [kl, k_mid, kr])
        elif how == "in_order":
            left, midp, right = v[:kl], v[kl:kl + k_mid], v[kl + k_mid:]
        else:  # inverted at the second junction
            left, midp, right = v[:kl], v[kl + kr:], v[kl:kl + kr]
        self.top[a - kl:a] = topP
        self.low[a - kl:a] = left
        if k_mid:
            pos = a + (T - k_mid) // 2 + np.arange(k_mid)
            self.top[pos] = topP
            self.low[pos] = midp
        self.top[b:b + kr] = topP
        self.low[b:b + kr] = right
        return self

    def u(self):
        l = self.l
        u = (self.top << _u(56 - l)) | (self.mid << _u(self.cb)) | self.low
        if l:
            u |= _u((0b101 & ((1 << l) - 1)) << (64 - l))
        return u

    def keys(self, dt, up):
        return from_order(self.u(), dt, up)


@dataclass(frozen=True)
class Case:
    keys: np.ndarray
    margin_bits: int
    expect: object   # expect(Prediction) -> bool: the branch the generator is named for was reached


N_DEFAULT = (1 << 17) + 300   # 33 tiles of 4096, the last one holding 300 keys; not a multiple of 256 either


def _flowed(device, host):
    """the branch in the device flow / in the flow with the FIX pass"""
    return lambda p: (host(p) if p.use_fix else device(p)) and p.stats["cut_digit"] == p.plan.cut_digit


def _no_flag(p):
    return not p.flag and not p.finish.fall_back


def g_uniform(dt, up, rng, n=N_DEFAULT):
    b = KeyBuilder(n, 5, rng)  # 24 swept bits: random runs of two or three keys in one tile
    return Case(b.keys(dt, up), b.margin, _flowed(
        lambda p: p.finish.segfix_segments[("short", 2)] > 0 and not p.finish.fall_back,
        lambda p: _no_flag(p) and p.finish.fix_runs[(2, "ordered")] > 0 and p.stats["segfix_passes"] == 0))


def _run(k, how, name):
    def gen(dt, up, rng, n=N_DEFAULT):
        b = KeyBuilder(n, 3, rng)
        v = b.distinct_lows(k)
        lows = {"reversed": v[::-1], "in_order": v, "equal": np.full(k, v[0])}[how]
        b.segment(5 * b.tile + 100, lows)
        ordered = k <= FIX_CAP + 1
        kind = "ordered" if ordered else ("long_inverted" if how == "reversed" else "long_in_order")
        host = (lambda p: p.finish.fix_runs[(k, kind)] == 1 and p.flag == (kind == "long_inverted")
                and (not ordered or p.finish.fix_moved_runs[k] == 1))
        dev_kind = ("short", k) if k <= SF_MAXSEG else (("long_equal" if how == "equal" else "long_distinct"), k)
        return Case(b.keys(dt, up), b.margin, _flowed(lambda p: p.finish.segfix_segments[dev_kind] == 1
                                                      and not p.finish.fall_back, host))
    gen.__name__ = name
    return gen


def g_junction2(dt, up, rng, n=N_DEFAULT):
    b = KeyBuilder(n, 3, rng).across(7 * 4096, 1, 1, "inverted")
    return Case(b.keys(dt, up), b.margin, _flowed(lambda p: not p.finish.fall_back,
                                                  lambda p: _no_flag(p) and p.finish.junctions[("swap", 2)] == 1))


def g_junction3to31(dt, up, rng, n=N_DEFAULT):
    b = KeyBuilder(n, 3, rng)
    for i, L in enumerate(range(3, 32)):
        b.across((i + 2) * b.tile, L // 2, L - L // 2)
    return Case(b.keys(dt, up), b.margin, _flowed(
        lambda p: not p.finish.fall_back,
        lambda p: _no_flag(p) and all(p.finish.junctions[("rank", L)] == 1 for L in range(3, 32))))


def g_junction32(dt, up, rng, n=N_DEFAULT):
    b = KeyBuilder(n, 3, rng).across(9 * 4096, 16, 16)
    return Case(b.keys(dt, up), b.margin, _flowed(lambda p: not p.finish.fall_back,
                                                  lambda p: _no_flag(p) and p.finish.junctions[("rank", 32)] == 1))


def _junction33(how):
    def gen(dt, up, rng, n=N_DEFAULT):
        b = KeyBuilder(n, 3, rng).across(9 * 4096, 16, 17, how)
        inv = how == "inverted"
        return Case(b.keys(dt, up), b.margin, _flowed(
            lambda p: p.finish.fall_back,  # 33 distinct keys: too long for the segment finish
            lambda p: p.finish.junctions[("long_inverted" if inv else "long_in_order", 0)] == 1 and p.flag == inv
            and not p.finish.fix_flag))
    gen.__name__ = f"g_junction33_{how}"
    return gen


def g_three_tiles_one_middle(dt, up, rng, n=N_DEFAULT):
    """six segments over three tiles each (one key in the middle one): the earliest junction's thread orders them"""
    b = KeyBuilder(n, 3, rng)
    for t in range(1, 25, 4):
        b.spanning(t, 5, 1, 6)
    return Case(b.keys(dt, up), b.margin, _flowed(
        lambda p: not p.finish.fall_back,
        lambda p: _no_flag(p) and p.finish.tiles_spanned[3] == 6 and p.finish.junctions[("owned_by_earlier", 12)] == 6))


def _three_tiles_whole_middle(how):
    def gen(dt, up, rng, n=N_DEFAULT):
        b = KeyBuilder(n, 3, rng).spanning(3, 4, 4096, 5, how)
        inv = how == "inverted"
        return Case(b.keys(dt, up), b.margin, _flowed(
            lambda p: p.finish.fall_back,
            lambda p: p.finish.junctions[("long_inverted", 0)] == int(inv) and p.flag == inv and not p.finish.fix_flag
            and p.finish.fix_runs[(4096, "long_in_order")] == 1))
    gen.__name__ = f"g_three_tiles_whole_middle_{how}"
    return gen


def g_empty_next_tile(dt, up, rng, n=N_DEFAULT):
    """a segment at the end of tile t and the start of tile t + 2, tile t + 1 without keys in its bucket: found by
    the key compare, not by the fingerprints"""
    b = KeyBuilder(n, 3, rng)
    for t in (2, 10, 20):
        b.spanning(t, 6, 0, 7)
    return Case(b.keys(dt, up), b.margin, _flowed(
        lambda p: not p.finish.fall_back,
        lambda p: _no_flag(p) and p.finish.direct_compares == 3 and p.finish.junctions[("rank", 13)] == 3))


def g_fingerprint_collision(dt, up, rng, n=N_DEFAULT):
    """cut at digit 2: prefixes A (digit 6 = x, digit 2 = y) and B (x ^ z, y ^ z) have equal fingerprints (hi ^ lo
    of the masked key); A is the last key of tile 8's part of a bucket, B the first of tile 9's"""
    b = KeyBuilder(n, 2, rng)
    for J in (9 * b.tile, 17 * b.tile):
        mA = int(b.mid[J - 1])
        x = mA >> 32
        if x == 0xFF:
            mA &= ~(1 << 32)
            x = 0xFE
        z = (~x & (x + 1)) & 0xFF  # lowest zero bit of x: x ^ z > x
        mB = ((x ^ z) << 32) | (mA & 0xFFFFFF00 & 0xFFFFFFFF) | ((mA & 0xFF) ^ z)
        b.mid[J - 1], b.mid[J] = mA, mB
        b.mid[J + 1:] = np.maximum(b.mid[J + 1:], np.uint64(mB) + np.arange(1, n - J, dtype=np.uint64))
        b.top[J] = b.top[J - 1]
    return Case(b.keys(dt, up), b.margin, _flowed(lambda p: not p.finish.fall_back,
                                                  lambda p: _no_flag(p) and p.finish.collisions == 2))


def _device_segments(name, parts, fall_back):
    """segments at given positions of the segment finish's input (the array ordered by its prefix)"""
    def gen(dt, up, rng, n=N_DEFAULT):
        b = KeyBuilder(n, 3, rng, sort_prefix=True)
        for a, k, how in parts(n):
            v = b.distinct_lows(k)
            b.segment(a, {"reversed": v[::-1], "equal": np.full(k, v[0])}[how])
        crossers = sum(1 for a, k, how in parts(n) if k <= SF_MAXSEG and a // SF_CHUNK != (a + k - 1) // SF_CHUNK)
        return Case(b.keys(dt, up), b.margin, _flowed(
            lambda p: p.finish.fall_back == fall_back and p.finish.segfix_chunk_crossers == crossers,
            lambda p: p.finish.fall_back == (fall_back and p.flag)))
    gen.__name__ = name
    return gen


def g_cut4_high_word_1(dt, up, rng, n=(1 << 19) + 300):
    """cut at bit 32 (the last pass compares raw high words): a block of eight tiles whose keys all have the mid of a
    raw high word of 1, one key per tile with exactly that high word and the smallest top digit -- slot 0 of the
    tile, a run of one key next to the out-of-tile placeholder"""
    b = KeyBuilder(n, 4, rng)
    u1 = int(O.order_key(np.array([(1 << 32) | 5], np.uint64).view(dt), up)[0])
    t1, m1 = u1 >> 56, (u1 >> 32) & 0xFFFFFF
    T = b.tile
    a = min(-(-int(np.searchsorted(b.mid, np.uint64(m1))) // T) * T, (n // T - 7) * T) if m1 else 0
    blk = slice(a, a + 6 * T)  # six whole tiles
    before = b.mid.copy()
    b.mid[:a] = np.minimum(b.mid[:a], m1 - 1)
    b.mid[a + 6 * T:] = np.maximum(b.mid[a + 6 * T:], m1 + 1)
    forced = b.mid != before  # (keys pushed to one mid beside the block: in ascending order, so no run is inverted)
    b.low[forced] = np.sort(b.low[forced])
    b.mid[blk] = m1
    if t1 < 255:
        b.top[blk] = rng.integers(t1 + 1, 256, 6 * T).astype(np.uint64)
        b.top[a + 77:a + 6 * T:T] = t1
    b.low[blk] = np.sort(rng.integers(0, 1 << 32, 6 * T, dtype=np.uint64))
    return Case(b.keys(dt, up), b.margin, _flowed(  # (device flow: the block's long segments fall back)
        lambda p: p.finish.fall_back,
        lambda p: _no_flag(p) and p.plan.cut_bit == 32 and (t1 == 255 or p.finish.slot0_hw1_short == 6)))


def _cut_at(cut, lshift=0):
    """cut at `cut` (after a left shift by lshift): a reversed run of 9 keys, a reversed pair and a junction segment
    of 12 keys"""
    def gen(dt, up, rng, n=N_DEFAULT):
        b = KeyBuilder(n, cut, rng, lshift)
        if lshift:
            b.margin = int(round(30.5 - math.log2(n)))  # unshifted sums 5, 13, 21, 29, 37; shifted 8, 16, 24, 32
        b.segment(3 * b.tile + 500, b.distinct_lows(9)[::-1])
        b.segment(4 * b.tile + 900, b.distinct_lows(2)[::-1])
        b.across(11 * b.tile, 5, 7)
        return Case(b.keys(dt, up), b.margin, _flowed(
            lambda p: not p.finish.fall_back and p.plan.lshift == lshift,
            lambda p: _no_flag(p) and p.plan.lshift == lshift and p.finish.fix_moved_runs[9] == 1
            and p.finish.fix_moved_runs[2] >= 1 and p.finish.junctions[("rank", 12)] == 1))
    gen.__name__ = f"g_cut{cut}" + (f"_lshift{lshift}" if lshift else "")
    return gen


def g_negative_run(dt, up, rng, n=N_DEFAULT):
    """segments of negative i64 / f64 keys (the in-run order of the raw keys is flipped for negative floats and for a
    descending sort): a reversed run of 9 and of 2, and junction segments of 2 and 5"""
    b = KeyBuilder(n, 3, rng)
    neg_top = 0x21 if up else 0xDE  # order-mapped top bit 0 (ascending) / 1 (descending): a negative raw key
    b.segment(6 * b.tile + 1000, b.distinct_lows(9)[::-1], neg_top)
    b.segment(6 * b.tile + 2000, b.distinct_lows(2)[::-1], neg_top)
    b.across(13 * b.tile, 1, 1, "inverted", neg_top)
    b.across(15 * b.tile, 2, 3, "interleaved", neg_top)
    return Case(b.keys(dt, up), b.margin, _flowed(
        lambda p: not p.finish.fall_back,
        lambda p: _no_flag(p) and p.finish.fix_moved_runs[9] == 1 and p.finish.fix_moved_runs[2] >= 1
        and p.finish.junctions[("swap", 2)] == 1 and p.finish.junctions[("rank", 5)] == 1))


def g_small_range(dt, up, rng, n=N_DEFAULT):
    """keys of a 20-bit range across bit 32: range reduction, no cut -- the segment finish has nothing to do"""
    u = np.uint64(0x6A5F0000FFFF8000) + rng.integers(0, 1 << 20, n, dtype=np.uint64)
    return Case(from_order(u, dt, up), 2, lambda p: p.plan.cut_digit == 0 and p.plan.sub != 0
                and p.stats["segfix_passes"] == 0 and p.stats["segfix_moved"] == 0)


def g_small_values(dt, up, rng, n=N_DEFAULT):
    """order-mapped keys below 2^20 (test_gpu_parity's small_range_u64): the top digits are skipped, no cut"""
    u = rng.integers(0, 1 << 20, n, dtype=np.uint64)
    return Case(from_order(u, dt, up), 2, lambda p: p.plan.cut_digit == 0 and p.plan.sub == 0
                and p.stats["segfix_passes"] == 0 and p.stats["segfix_moved"] == 0)


GENERATORS = {g.__name__[2:]: g for g in [
    g_uniform,
    _run(9, "reversed", "g_run9_reversed"), _run(10, "reversed", "g_run10_reversed"),
    _run(10, "in_order", "g_run10_in_order"), _run(40, "equal", "g_run40_equal"),
    g_junction2, g_junction3to31, g_junction32, _junction33("inverted"), _junction33("in_order"),
    g_three_tiles_one_middle, _three_tiles_whole_middle("in_order"), _three_tiles_whole_middle("inverted"),
    g_empty_next_tile, g_fingerprint_collision,
    _device_segments("g_segfix32", lambda n: [(20000 + 40, 32, "reversed")], False),
    _device_segments("g_segfix33_distinct", lambda n: [(20000 + 40, 33, "reversed")], True),
    _device_segments("g_segfix33_equal", lambda n: [(20000 + 40, 33, "equal")], False),
    _device_segments("g_chunk_edges", lambda n: [(0, 7, "reversed"), (256 * 30 - 5, 10, "reversed"),
                                                 (256 * 50 - 1, 32, "reversed"), (256 * 70 - 31, 32, "reversed"),
                                                 (n - 7, 7, "reversed")], False),
    g_cut4_high_word_1, _cut_at(2), _cut_at(3), _cut_at(4), _cut_at(5), _cut_at(4, 3),
    g_negative_run, g_small_range, g_small_values,
]}
