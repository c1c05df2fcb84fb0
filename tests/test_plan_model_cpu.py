"""CPU tests of tests/plan_model.py against plans worked out by hand from scan_kernel's rules."""
import numpy as np
import pytest

import oracle_lib as O
from plan_model import digits_of_range, from_order, lsd_plan


def test_digits_of_range():
    assert digits_of_range(5, 5) == 0
    assert digits_of_range(0, 1) == 1
    assert digits_of_range(0, 255) == 1
    assert digits_of_range(0, 256) == 2
    assert digits_of_range(0xFF80, 0x10080) == 2      # 0x100: 9 bits
    assert digits_of_range(0, (1 << 64) - 1) == 8


@pytest.mark.parametrize("dt", O.KEY_DTYPES, ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("up", [True, False])
def test_from_order_inverts_order_key(dt, up):
    rng = np.random.default_rng(1)
    k = rng.integers(0, 256, 4096 * np.dtype(dt).itemsize, dtype=np.uint8).view(dt)
    u = O.order_key(k, up)
    assert from_order(u, dt, up).tobytes() == k.tobytes()


def test_i32_small_range_crossing_the_sign():
    """i32 in [-100, 100]: ordered 0x7fffff9c .. 0x80000064, so every digit position varies; the range (200) spans
    one digit: reduce to one pass, which the probe's guessed histogram (unreduced digit 0) cannot stand in for"""
    k = np.arange(-100, 101, dtype=np.int32)
    for up in (True, False):
        p = lsd_plan(k, up)
        assert p.varying == 0xFFFFFFFF and p.planned == 4
        assert p.rb == 1 and p.reduce and p.passes == 1 and p.skip == (False, True, True, True)
        assert p.mn == (0x7FFFFF9C if up else 0x7FFFFF9B)
        assert not p.hist_done and p.want_minmax
        assert p.host_flow_stats == {"passes_planned": 1, "hist_sweeps": 3, "kernel_launches": 7}
        assert p.device_flow_stats == {"passes_planned": 4, "hist_sweeps": 2, "kernel_launches": 8}


def test_u32_multiples_of_256_below_2_16():
    """u32 multiples of 256 below 2^16: only digit 1 varies (one pass); mn == 0 rules out the reduction; the guess
    (digit 0) missed, so hist_kernel counts digit 1"""
    k = np.arange(0, 1 << 16, 256, dtype=np.uint32)
    p = lsd_plan(k)
    assert p.varying == 0xFF00 and p.planned == 1 and p.mn == 0 and not p.reduce
    assert p.passes == 1 and p.skip == (True, False, True, True)
    assert not p.hist_done and not p.want_minmax
    assert p.host_flow_stats == {"passes_planned": 1, "hist_sweeps": 2, "kernel_launches": 5}
    # descending: ordered keys 0xffffffff - 256 i, so mn != 0, but the range spans 2 digits, more than the 1 planned
    d = lsd_plan(k, up=False)
    assert d.planned == 1 and d.rb == 2 and not d.reduce and d.passes == 1 and not d.hist_done


def test_one_u8_value_repeated():
    """one u8 value: nothing varies, nothing is swept; hist_kernel is still launched (and returns at once)"""
    k = np.full(1000, 7, np.uint8)
    p = lsd_plan(k)
    assert p.varying == 0 and p.planned == 0 and p.rb == 0 and not p.reduce and p.passes == 0
    assert not p.hist_done and not p.want_minmax
    assert p.host_flow_stats == {"passes_planned": 0, "hist_sweeps": 2, "kernel_launches": 4}
    # without skipping: the all-equal non-zero keys are reduced to range 0, which also sweeps nothing
    q = lsd_plan(k, allow_skip=0)
    assert q.planned == 1 and q.reduce and q.passes == 0 and q.want_minmax
    assert q.host_flow_stats == {"passes_planned": 0, "hist_sweeps": 3, "kernel_launches": 6}
    # all zero (ordered): mn == 0, no reduction; every pass runs without skipping
    z = lsd_plan(np.zeros(10, np.uint16), allow_skip=0)
    assert z.planned == 2 and not z.reduce and z.passes == 2 and z.hist_done


@pytest.mark.parametrize("dt", [np.uint8, np.uint16, np.uint32, np.uint64])
def test_unsigned_keys_from_zero(dt):
    """unsigned keys in [0, 300]: mn == 0, so no reduction; the digit positions above 300 are skipped"""
    k = np.arange(0, 301, dtype=np.uint64).astype(dt)
    kb = np.dtype(dt).itemsize
    p = lsd_plan(k)
    assert p.mn == 0 and not p.reduce and not p.want_minmax
    assert p.passes == min(kb, 2) and p.hist_done
    assert p.host_flow_stats["kernel_launches"] == 3 + p.passes
    r = lsd_plan(k, allow_reduce=0)
    assert r.passes == p.passes
    s = lsd_plan(k, allow_skip=0)
    assert s.passes == kb and s.planned == kb and not s.reduce


def test_f32_denormals_around_zero():
    """f32 in [-1e-40, 1e-40] with +-0: ordered keys from just below 0x7fffffff (-0) to just above 0x80000000 (+0) --
    the range crosses the sign, so every digit varies, yet it spans 3 digits only"""
    k = np.array([-1e-40, -1e-41, -0.0, 0.0, 1e-41, 1e-40], np.float32)
    for up in (True, False):
        p = lsd_plan(k, up)
        assert p.varying == 0xFFFFFFFF and p.planned == 4
        assert p.rb == 3 and p.reduce and p.passes == 3 and p.skip == (False, False, False, True)
        assert not p.hist_done and p.want_minmax
        assert p.host_flow_stats == {"passes_planned": 3, "hist_sweeps": 3, "kernel_launches": 9}


def test_options_change_the_plan():
    k = np.arange(-100, 101, dtype=np.int32)
    assert lsd_plan(k, allow_reduce=0).passes == 4
    assert lsd_plan(k, allow_reduce=0).hist_done
    assert not lsd_plan(k, allow_reduce=0, probe_guess=0).hist_done
    assert lsd_plan(k, allow_reduce=0, probe_guess=0).host_flow_stats["hist_sweeps"] == 2
    assert lsd_plan(k, allow_skip=0).passes == 1  # (every digit varies anyway)


def test_sampled_range_only_decides_the_minmax_sweep():
    """sparse sampling: the sample's range decides whether the exact min/max sweep runs; the passes come from the
    exact keys"""
    u = np.array([0x12340000 + i for i in range(300)] + [0x1233FFFF], np.uint32)
    p = lsd_plan(u, sampled=u[:300])
    assert p.want_minmax and p.reduce and p.passes == 2 and p.hist_sweeps == 3
    # one key far outside a narrow sample: the min/max sweep runs, but the exact range rules the reduction out
    v = np.concatenate([u[:300], np.array([0x92340000], np.uint32)])
    q = lsd_plan(v, sampled=v[:300])
    assert q.want_minmax and not q.reduce and q.passes == 3 and q.hist_done
    assert q.host_flow_stats == {"passes_planned": 3, "hist_sweeps": 2, "kernel_launches": 8}
    # a sample at ordered 0: the min/max sweep is not worth it
    w = np.concatenate([np.zeros(4, np.uint32), u])
    assert not lsd_plan(w, sampled=w[:4]).want_minmax
    with pytest.raises(ValueError):
        lsd_plan(u[:300], sampled=v[300:])  # (a sample is a subset of the keys)
