"""An exact numpy model of the pass plan of a digit-by-digit (LSD) sort (TEST INFRASTRUCTURE ONLY).

The plan decides, before any record moves, which digit positions a sort sweeps, whether it subtracts the smallest
key first (range reduction), whether the probe's guessed histogram stands in for hist_kernel, and -- when the plan is
read back on the host -- whether the exact min/max sweep and a second planning step run.  A wrong decision does not
fault: it orders the array wrongly, and only for key sets of a particular shape.  For the digit-by-digit path the plan
follows exactly from the order-mapped keys and the options, so `lsd_plan` restates it and the tests compare it with
`last_stats()`.

Where each rule comes from (simd-radix-sort_b200/csrc):
- kernels.cuh, probe_kernel: OR / OR-of-complements of EVERY ordered key, masked to the key width (`KEYMASK`), and
  the min / max of the sampled keys only (`smax_key`, `snmin_key`) unless `with_minmax`.
- kernels.cuh, scan_kernel:
  - `varying = or_bits & nand_bits`; digit position p is skipped iff `allow_skip` and its 8 bits of `varying` are 0;
  - `planned` = positions not skipped (+ 1 for a hybrid cut, 0 here: the LSD path has no cut);
  - `digits_of_range(mn, mx)` = 0 if mx == mn else floor(log2(mx - mn)) // 8 + 1;
  - without the exact min/max: `want_minmax = allow_reduce && mn != 0 && mx >= mn && digits_of_range < planned` on
    the SAMPLED range;
  - with it: range reduction iff `allow_reduce && mn != 0 && rb < planned`, and then `sub = mn` and position p is
    skipped iff `p >= rb`;
  - `hist_done = guess_p1 != 0 && first_exec_p1 == guess_p1 && sub == 0 && lshift == guess_lshift`.
- b200sort.cu, DevSort::make_plan: `big = n >= 2^host_plan_min_log2` (the plan is read back); the probe gets the
  exact min/max (`with_minmax`) only when not big; the LSD guess is digit 0 (`guess_p1 = probe_guess ? 1 : 0`); in the
  big flow minmax_kernel and a second scan run iff `want_minmax`, and hist_kernel is launched unless `hist_done`.
  The small flow launches everything: probe, scan, hist_kernel and one scatter pass per digit position.
- b200sort.cu, DevSort::statistics: `passes_planned = n_exec` when the plan is on the host, else the key width;
  `hist_sweeps` counts probe + minmax + hist_kernel launches.
- b200sort.cu, DevSort::finish: the LSD path always launches copyback_kernel (it returns at once when the result
  already lies in the caller's arrays); DevSort::run counts every launch into `kernel_launches`.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

import oracle_lib as O


def digits_of_range(mn: int, mx: int) -> int:
    """digit positions (of 8 bits) that the range [mn, mx] spans (scan_kernel's digits_of_range)"""
    return 0 if mx == mn else ((mx - mn).bit_length() - 1) // 8 + 1


@dataclass(frozen=True)
class LsdPlan:
    kb: int
    varying: int         # bits on which the ordered keys differ
    planned: int         # digit positions swept before range reduction is considered
    mn: int              # exact smallest / largest ordered key
    mx: int
    rb: int              # digit positions the exact range spans
    reduce: bool         # range reduction (Plan::sub = mn)
    passes: int          # digit passes executed (Plan::n_exec)
    skip: tuple          # per digit position: skipped
    hist_done: bool      # the probe's exact histogram of digit 0 is the first pass's: no hist_kernel
    want_minmax: bool    # host-plan flow: minmax_kernel and a second scan run
    hist_sweeps: int     # host-plan flow: probe + minmax + hist_kernel
    kernel_launches: int  # host-plan flow: probe, scan, (minmax, scan), (hist), passes, copy-back

    # what last_stats() reports for the flow that makes the plan on the device (every kernel is launched)
    @property
    def device_flow_stats(self) -> dict:
        return {"passes_planned": self.kb, "hist_sweeps": 2, "kernel_launches": 4 + self.kb}

    @property
    def host_flow_stats(self) -> dict:
        return {"passes_planned": self.passes, "hist_sweeps": self.hist_sweeps, "kernel_launches": self.kernel_launches}


def lsd_plan(keys: np.ndarray, up: bool = True, *, allow_skip: int = 1, allow_reduce: int = 1, probe_guess: int = 1,
             sampled=None) -> LsdPlan:
    """The plan the digit-by-digit sort of `keys` makes.

    `sampled`: the order-mapped keys the probe samples when it samples sparsely (n / hist tile keys >= 8192), or None
    when it sees every key.  Only `want_minmax` (and with it `hist_sweeps` and `kernel_launches` of the host-plan flow)
    depends on the sample; the passes never do."""
    kb = keys.dtype.itemsize
    mask = (1 << (8 * kb)) - 1
    u = O.order_key(np.ascontiguousarray(keys).reshape(-1), up)
    if len(u) == 0:
        raise ValueError("no keys")
    or_bits = int(np.bitwise_or.reduce(u))
    nand_bits = int(np.bitwise_or.reduce(~u)) & mask
    varying = or_bits & nand_bits
    skip = [bool(allow_skip) and ((varying >> (8 * p)) & 0xFF) == 0 for p in range(kb)]
    planned = kb - sum(skip)
    mn, mx = int(u.min()), int(u.max())
    rb = digits_of_range(mn, mx)
    reduce = bool(allow_reduce) and mn != 0 and rb < planned
    if reduce:
        skip = [p >= rb for p in range(kb)]
    passes = kb - sum(skip)
    hist_done = bool(probe_guess) and not reduce and not skip[0]
    s = u if sampled is None else np.asarray(sampled, dtype=u.dtype)
    smn, smx = int(s.min()), int(s.max())
    if smn < mn or smx > mx:
        raise ValueError("the sampled keys are not inside the range of the keys")
    # (a sample inside [mn, mx] spans at most rb digits and has smn >= mn: `reduce` implies `want_minmax`, so the
    # host-plan flow, which only learns the exact range by the min/max sweep, makes the same plan as the device flow)
    want_minmax = bool(allow_reduce) and smn != 0 and smx >= smn and digits_of_range(smn, smx) < planned
    hist_sweeps = 1 + int(want_minmax) + (0 if hist_done else 1)
    kernel_launches = 2 + 2 * int(want_minmax) + (0 if hist_done else 1) + passes + 1
    return LsdPlan(kb, varying, planned, mn, mx, rb, reduce, passes, tuple(skip), hist_done, want_minmax, hist_sweeps,
                   kernel_launches)


def from_order(u: np.ndarray, dtype, up: bool = True) -> np.ndarray:
    """The keys of `dtype` whose order-mapped values (oracle_lib.order_key) are `u`: the inverse of order_key."""
    dt = np.dtype(dtype)
    bits = dt.itemsize * 8
    udt = np.dtype(f"uint{bits}")
    u = np.asarray(u).astype(udt, copy=True)
    if not up:
        u = ~u
    sign = udt.type(1 << (bits - 1))
    if dt.kind == "i":
        u ^= sign
    elif dt.kind == "f":
        u = np.where((u & sign) != 0, u ^ sign, ~u).astype(udt)
    return u.view(dt)
