"""CPU-side tests of the drop-in boundary: the C-ABI library builds/loads, exports every symbol that
include/b200sort.h declares, validates its arguments like the reference's static_asserts do, and fails
loudly (no CPU fallback) when no CUDA device is present.  No compute happens here."""
import ctypes
import json
import re
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import simd_radix_sort_b200 as S

ROOT = Path(__file__).resolve().parent.parent


def _has_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_library_exports_every_declared_symbol():
    header = (ROOT / "include" / "b200sort.h").read_text()
    declared = set(re.findall(r"\b(b200sort_[a-z0-9_]+)\s*\(", header))
    assert {"b200sort_sort_soa", "b200sort_sort_aos", "b200sort_workspace_bytes", "b200sort_last_error"} <= declared
    out = subprocess.run(["nm", "-D", "--defined-only", str(S.lib_path())], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (b200sort_[a-z0-9_]+)", out))
    assert declared <= exported, declared - exported
    L = S.lib()
    for name in declared:
        assert getattr(L, name) is not None
    assert S.version() == 100


def test_workspace_bytes_covers_shadow_streams():
    n = 1_000_000
    w = S.workspace_bytes(np.uint64, n, [8])
    assert w >= 2 * 8 * n and w < 2 * 8 * n + (64 << 20)
    w = S.workspace_bytes(np.int64, n, record_bytes=16)
    assert w >= 16 * n
    assert S.workspace_bytes(np.float32, 0, [4, 8, 2]) > 0


def test_argument_errors_match_reference_rules():
    L = S.lib()
    k = np.arange(10, dtype=np.uint32)
    # unknown key type
    assert L.b200sort_sort_soa(k.ctypes.data, 42, 10, 1, 0, None, None, None, None, 0) == -1
    # negative num
    assert L.b200sort_sort_soa(k.ctypes.data, 4, -1, 1, 0, None, None, None, None, 0) == -1
    # record size must be a power of two >= sizeof(key) (src/radix_sort.hpp:318-319)
    assert L.b200sort_sort_aos(k.ctypes.data, 6, 24, 1, 1, None, None, 0) == -3
    assert L.b200sort_sort_aos(k.ctypes.data, 6, 4, 1, 1, None, None, 0) == -3
    assert b"power of two" in L.b200sort_last_error()
    # payload element sizes 1..64
    sizes = (ctypes.c_uint32 * 1)(65)
    ptrs = (ctypes.c_void_p * 1)(k.ctypes.data)
    assert L.b200sort_sort_soa(k.ctypes.data, 4, 10, 1, 1, ptrs, sizes, None, None, 0) == -2
    assert L.b200sort_set_option(b"no_such_option", 1) == -1
    assert L.b200sort_set_option(b"algo", 0) == 0


@pytest.mark.skipif(_has_cuda(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback():
    k = np.array([3, 1, 2], dtype=np.int32)
    with pytest.raises(S.B200SortError) as ei:
        S.sort(3, k)
    assert ei.value.code == -5 and "no CPU fallback" in str(ei.value)
    assert k.tolist() == [3, 1, 2]  # untouched


def test_product_never_imports_the_oracle():
    pkg = ROOT / "simd-radix-sort_b200"
    for f in list(pkg.rglob("*.py")) + list(pkg.rglob("*.cu")) + list(pkg.rglob("*.cuh")) + list((ROOT / "include").rglob("*")):
        if f.is_file():
            txt = f.read_text(errors="ignore")
            assert "oracle" not in txt.lower() or f.name == "sortbench.cu", f


def test_splitters_balance_and_cover():
    L = S.lib()
    rng = np.random.default_rng(0)
    for bits, world in ((8, 2), (16, 8), (16, 3), (4, 4)):
        hist = rng.integers(0, 1000, size=1 << bits).astype(np.uint64)
        bounds = np.zeros(world + 1, np.uint32)
        rc = L.b200sort_mgpu_splitters(hist.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)), bits, world,
                                       bounds.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)))
        assert rc == 0
        assert bounds[0] == 0 and bounds[-1] == (1 << bits) and np.all(np.diff(bounds.astype(np.int64)) >= 0)
        loads = np.array([hist[bounds[r]:bounds[r + 1]].sum() for r in range(world)], dtype=np.float64)
        ideal = hist.sum() / world
        # each boundary may sit up to 1/64 of a share off its target in favour of an aligned bin index
        assert np.all(np.abs(loads - ideal) <= ideal / 32 + hist.max() + 1), (loads, ideal)
    # skew: one bin holds everything -> one rank gets it all, the others nothing, still a cover
    hist = np.zeros(256, np.uint64)
    hist[17] = 1000
    bounds = np.zeros(5, np.uint32)
    assert L.b200sort_mgpu_splitters(hist.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)), 8, 4,
                                     bounds.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32))) == 0
    loads = [int(hist[bounds[r]:bounds[r + 1]].sum()) for r in range(4)]
    assert sum(loads) == 1000 and max(loads) == 1000


def test_splitters_prefer_aligned_boundaries():
    """near-uniform histograms and a power-of-two world: every boundary lands on a multiple of 2^bits / world,
    so each shard's keys share their leading log2(world) bits (what the local sort's left-shifted plan needs)"""
    L = S.lib()
    rng = np.random.default_rng(5)
    bits = 16
    for world in (2, 4, 8):
        hist = rng.poisson(250.0, size=1 << bits).astype(np.uint64)  # a 2^24-key sample of uniform keys
        bounds = np.zeros(world + 1, np.uint32)
        assert L.b200sort_mgpu_splitters(hist.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)), bits, world,
                                         bounds.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32))) == 0
        step = (1 << bits) // world
        assert bounds.tolist() == [r * step for r in range(world + 1)], bounds
    # a skewed histogram must not be forced onto aligned boundaries at the price of balance
    hist = np.ones(1 << bits, np.uint64)
    hist[: 1 << 12] = 1000
    bounds = np.zeros(5, np.uint32)
    assert L.b200sort_mgpu_splitters(hist.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)), bits, 4,
                                     bounds.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32))) == 0
    loads = np.array([hist[bounds[r]:bounds[r + 1]].sum() for r in range(4)], dtype=np.float64)
    assert np.all(np.abs(loads - hist.sum() / 4) <= hist.sum() / 4 / 32 + 1001), loads


def test_range_bins_make_narrow_key_ranges_splittable():
    """the splitter histogram covers the sampled key range, not the key space: N(0, 1000) int64 keys (two
    distinct top-16-bit values!) still split evenly over 8 ranks; full-width keys keep bin = top 16 bits"""
    L = S.lib()
    u64p, u32p = ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint32)
    L.b200sort_mgpu_range_bins.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_int, ctypes.c_int, u64p, ctypes.POINTER(ctypes.c_int)]
    import oracle_lib as O
    rng = np.random.default_rng(11)
    bits, nb = 16, 1 << 16
    for name, keys in (("gauss_i64", np.round(rng.normal(0, 1000, 400_000)).astype(np.int64)),
                       ("uniform_u64", rng.integers(0, 2**64, 400_000, dtype=np.uint64)),
                       ("small_u32", rng.integers(0, 5000, 400_000, dtype=np.uint32)),
                       ("f64_unit", rng.uniform(-1, 1, 400_000))):
        u = O.order_key(keys, True).astype(np.uint64)
        sample = u[::7]
        lo, shift = ctypes.c_uint64(0), ctypes.c_int(0)
        assert L.b200sort_mgpu_range_bins(int(sample.min()), int(sample.max()), keys.dtype.itemsize, bits, ctypes.byref(lo), ctypes.byref(shift)) == 0
        lo, shift = np.uint64(lo.value), np.uint64(shift.value)
        # range_bin() of csrc/kernels.cuh, restated
        b = np.where(u <= lo, np.uint64(0), np.minimum((u - lo) >> shift, np.uint64(nb - 1))).astype(np.int64)
        assert np.all(np.diff(b[np.argsort(u, kind="stable")]) >= 0), name  # monotonic in the key
        if name == "uniform_u64":
            assert lo == 0 and shift == 48
        hist = np.bincount(b, minlength=nb).astype(np.uint64)
        world = 8
        bounds = np.zeros(world + 1, np.uint32)
        assert L.b200sort_mgpu_splitters(hist.ctypes.data_as(u64p), bits, world, bounds.ctypes.data_as(u32p)) == 0
        loads = np.array([hist[bounds[r]:bounds[r + 1]].sum() for r in range(world)], dtype=np.float64)
        ideal = len(keys) / world
        assert loads.max() <= ideal * (1 + 1 / 32) + hist.max() + 1, (name, loads)
        if name != "small_u32":
            assert loads.max() <= 1.2 * ideal, (name, loads)  # what the default capacity (1.125x + slack) tolerates


def _documented_options() -> dict:
    """{name: bracketed default} of the option list in INTEGRATION.md section 6"""
    doc = (ROOT / "INTEGRATION.md").read_text()
    sec = doc[doc.index("## 6. Options"):].split("\n## ")[0]
    return {name: int(v) for name, v in re.findall(r"`(\w+)` \[(-?\d+)", sec)}


def test_documented_option_defaults_in_a_fresh_process():
    documented = _documented_options()
    code = ("import json, simd_radix_sort_b200 as S; "
            f"print(json.dumps({{n: S.get_option(n) for n in {sorted(documented)!r}}}))")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, check=True).stdout
    assert json.loads(out) == documented


def test_option_table_matches_the_documented_names():
    src = (ROOT / "simd-radix-sort_b200" / "csrc" / "b200sort.cu").read_text()
    table = re.findall(r'\{"(\w+)", &Options::(\w+)\}', src)
    assert all(name == member for name, member in table), table
    names = [name for name, _ in table]
    assert len(names) == len(set(names))
    assert set(names) == set(_documented_options())


def test_max_chunk_takes_powers_of_two_up_to_16():
    L = S.lib()
    before = S.get_option("max_chunk")
    for v in (0, 3, 12, 32):
        assert L.b200sort_set_option(b"max_chunk", v) == -1, v
        assert S.get_option("max_chunk") == before
    for v in (1, 2, 4, 8, 16):
        with S.options(max_chunk=v):
            assert S.get_option("max_chunk") == v
    assert S.get_option("max_chunk") == before


def test_options_restores_the_earlier_values_when_the_body_raises():
    before = {"algo": S.get_option("algo"), "margin_bits": S.get_option("margin_bits")}
    with pytest.raises(ZeroDivisionError):
        with S.options(algo=2, margin_bits=-3):
            assert S.get_option("algo") == 2 and S.get_option("margin_bits") == -3
            1 / 0
    assert {n: S.get_option(n) for n in before} == before
    # a name the library does not know raises, and what was already set is restored
    with pytest.raises(S.B200SortError):
        with S.options(algo=1, no_such_option=1):
            pass
    assert S.get_option("algo") == before["algo"]
