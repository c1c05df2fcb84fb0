"""GPU tests (-m gpu) of the finishes of the 8-byte-key hybrid path against the exact model of tests/hybrid_model.py.

The hybrid path sweeps only the top digits; the last pass, the junction kernel, the segment finish or the fall-back
orders what is left, and two device flags choose between them.  A wrong finish does not fault: it leaves a few records
out of order for one key shape, or silently runs a full extra pass.  Every generator of hybrid_model.GENERATORS puts
runs and segments exactly at the caps (9 / 10 keys in one tile, 32 / 33 across a junction or in the segment finish),
across three tiles, next to a tile without keys in the bucket, on a fingerprint collision, across the segment finish's
256-position chunks and at the array's ends.  Each case checks:
- the key bytes equal numpy's total-order sort;
- the index payload is a permutation that reproduces the keys (and, where every pass is stable, is the stable order);
- last_stats() equals the model: cut_digit, passes_planned, hist_sweeps, kernel_launches, segfix_passes, fell_back,
  algorithmic_bytes and, where it is deterministic, segfix_moved.
Three flows: the plan made on the device (host_plan_min_log2 = 24), read back with a stable first pass (= 0,
first_atomic = 0: every prediction exact) and read back with default options (the first pass ranks unstably: only what
no tie order changes is compared)."""
import numpy as np
import pytest

import hybrid_model as H
import oracle_lib as O
import simd_radix_sort_b200 as S

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DTYPES = [np.dtype(d) for d in (np.uint64, np.int64, np.float64)]
FLOWS = {"device_plan": ("device", dict(host_plan_min_log2=24, first_atomic=0)),
         "host_plan_stable": ("host", dict(host_plan_min_log2=0, first_atomic=0)),
         "host_plan_default": ("host", dict(host_plan_min_log2=0))}
MODEL_OPTIONS = ("first_atomic", "fix_in_pass", "junction_table", "tile_cfg")


@pytest.fixture(scope="module", autouse=True)
def _loaded():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    before = S.launch_count()
    yield
    assert S.launch_count() > before, "no kernels of libb200sort.so were launched"


def to_dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def expected(pred):
    """the statistics the model can vouch for: all of them unless the first pass was unstable and a tie order could
    change a flag; segfix_moved where it is not timing-dependent"""
    st = {k: v for k, v in pred.stats.items() if v is not None}
    if pred.tie_dependent and not pred.flags_tie_free:
        st = {k: st[k] for k in ("algo", "cut_digit")}
    return st


def predict(keys, up, flow, margin, opts, record_bytes):
    model_opts = {k: v for k, v in opts.items() if k in MODEL_OPTIONS}
    return H.predict(keys, up, flow, margin_bits=margin, record_bytes=record_bytes, **model_opts)


def sort_soa(keys, pays, up, opts):
    k, ps = to_dev(keys), [to_dev(p) for p in pays]
    with S.options(algo=2, **opts):
        S.sort(len(keys), k, *ps, up=up)
    torch.cuda.synchronize()
    return k.cpu().numpy(), [p.cpu().numpy() for p in ps], S.last_stats()


def check_case(keys, up, margin, flow_name, pays=None, extra=None):
    """one sort of keys + payloads (default: a u32 index) in one flow against numpy and the model"""
    flow, opts = FLOWS[flow_name]
    opts = {**opts, "margin_bits": margin, **(extra or {})}
    n = len(keys)
    pays = pays if pays is not None else [np.arange(n, dtype=np.uint32)]
    rb = 8 + sum(p.dtype.itemsize * (p.shape[1] if p.ndim > 1 else 1) for p in pays)
    pred = predict(keys, up, flow, margin, opts, rb)
    out_k, out_p, st = sort_soa(keys, pays, up, opts)
    want = O.total_order_sorted_keys(keys, up)
    assert out_k.tobytes() == want.tobytes(), "keys are not in numpy's order"
    idx = out_p[0].astype(np.int64)
    assert np.all(np.bincount(idx, minlength=n) == 1), "index payload is not a permutation"
    assert keys[idx].tobytes() == out_k.tobytes(), "index payload does not follow the keys"
    if not pred.tie_dependent:
        assert np.array_equal(idx, np.argsort(O.order_key(keys, up), kind="stable")), "not the stable order"
    for i, (p, po) in enumerate(zip(pays[1:], out_p[1:])):
        assert np.array_equal(po, p[idx]), f"payload {i + 1} does not follow the keys"
    want_st = expected(pred)
    got = {f: st[f] for f in want_st}
    assert got == want_st, (flow_name, pred.plan, got, want_st)
    return pred


@pytest.mark.parametrize("flow_name", list(FLOWS))
@pytest.mark.parametrize("gen", list(H.GENERATORS))
def test_generators(gen, flow_name):
    """every generator x u64 / i64 / f64 x both directions, with a u32 index"""
    for dt in DTYPES:
        for up in (True, False):
            rng = np.random.default_rng(len(gen) * 7 + dt.num)
            case = H.GENERATORS[gen](dt, up, rng)
            pred = check_case(case.keys, up, case.margin_bits, flow_name)
            if flow_name != "host_plan_default":
                assert case.expect(pred), (gen, dt, up, flow_name)  # the branch the generator is named for


@pytest.mark.parametrize("n", [(1 << 16) + 77, (1 << 20) + 333])
@pytest.mark.parametrize("gen", ["uniform", "negative_run"])
def test_other_sizes(gen, n):
    for dt in DTYPES:
        for up in (True, False):
            case = H.GENERATORS[gen](dt, up, np.random.default_rng(n % 1000 + dt.num), n)
            for flow_name in FLOWS:
                check_case(case.keys, up, case.margin_bits, flow_name)


@pytest.mark.parametrize("spanning", [False, True])
def test_default_options_at_the_hybrid_size(spanning):
    """2^22 + 4099 records with every option at its default: the hybrid path is chosen by itself, plan on the device.
    Top digits of 7 varying bits put the entropy sums (7, 15, 23, 31) clear of log2 n + 2 = 24: the cut is at digit 4"""
    n = (1 << 22) + 4099
    dt = np.dtype(np.int64)
    b = H.KeyBuilder(n, 4, np.random.default_rng(22))
    b.top &= np.uint64(0xBF)  # (bit 6 constant, the leading bit varying: no left shift)
    if spanning:
        for t in range(10, 1000, 97):
            b.spanning(t, 7, 1, 8)
    keys = b.keys(dt, True)
    pred = H.predict(keys, True, "device", record_bytes=16)
    assert pred.plan.cut_digit == 4
    k, p = to_dev(keys), to_dev(np.arange(n, dtype=np.uint64))
    with S.options():
        S.sort(n, k, p)
    torch.cuda.synchronize()
    st = S.last_stats()
    out_k, idx = k.cpu().numpy(), p.cpu().numpy().astype(np.int64)
    assert out_k.tobytes() == O.total_order_sorted_keys(keys, True).tobytes()
    assert np.array_equal(idx, np.argsort(O.order_key(keys), kind="stable"))
    want = expected(pred)
    assert {f: st[f] for f in want} == want, (pred.plan, st)


# ---------------------------------------------------------------------------------------------------------------------
# the payload shapes that take different move code in the finishes, and the options that change the finish, on
# generators that raise the flags (the last pass's, the junction kernel's, the segment finish's) or need a merge
# ---------------------------------------------------------------------------------------------------------------------
FLAGGED = ["run10_reversed", "junction33_inverted", "three_tiles_one_middle", "junction3to31", "segfix32",
           "segfix33_distinct", "three_tiles_whole_middle_inverted"]


@pytest.mark.parametrize("flow_name", ["device_plan", "host_plan_stable"])
@pytest.mark.parametrize("shape", ["u8_u16", "row16"])
def test_payload_shapes(shape, flow_name):
    """SoA payloads of 1 and 2 bytes (segfix_kernel<8, true>, the byte-wise junction moves) and of 16 bytes (the
    uint4 junction moves, the cb == 16 path of the segment finish)"""
    for gen in FLAGGED:
        for dt, up in ((np.dtype(np.uint64), True), (np.dtype(np.float64), False)):
            case = H.GENERATORS[gen](dt, up, np.random.default_rng(len(gen)))
            n = len(case.keys)
            rng = np.random.default_rng(n)
            extra = ([rng.integers(0, 256, n, dtype=np.uint8), rng.integers(0, 1 << 16, n, dtype=np.uint16)]
                     if shape == "u8_u16" else [rng.integers(0, 256, (n, 16), dtype=np.uint8)])
            check_case(case.keys, up, case.margin_bits, flow_name, [np.arange(n, dtype=np.uint32)] + extra)


@pytest.mark.parametrize("flow_name", ["device_plan", "host_plan_stable"])
@pytest.mark.parametrize("rb", [16, 32, 64])
def test_records(rb, flow_name):
    """AoS records (key at offset 0, u32 index at offset 8, random bytes elsewhere) travel whole"""
    for gen in FLAGGED:
        dt, up = np.dtype(np.int64), rb != 32
        case = H.GENERATORS[gen](dt, up, np.random.default_rng(rb))
        keys, n = case.keys, len(case.keys)
        rec = np.random.default_rng(n).integers(0, 256, (n, rb), dtype=np.uint8)
        rec[:, :8] = keys.view(np.uint8).reshape(n, 8)
        rec[:, 8:12] = np.arange(n, dtype=np.uint32).view(np.uint8).reshape(n, 4)
        flow, opts = FLOWS[flow_name]
        pred = predict(keys, up, flow, case.margin_bits, opts, rb)
        r = to_dev(rec)
        with S.options(algo=2, margin_bits=case.margin_bits, **opts):
            S.sort_combined(n, r, dt, up=up)
        torch.cuda.synchronize()
        st = S.last_stats()
        out = r.cpu().numpy()
        assert np.ascontiguousarray(out[:, :8]).tobytes() == O.total_order_sorted_keys(keys, up).tobytes(), gen
        idx = np.ascontiguousarray(out[:, 8:12]).view(np.uint32).reshape(-1).astype(np.int64)
        assert np.array_equal(idx, np.argsort(O.order_key(keys, up), kind="stable")), gen
        assert np.array_equal(out, rec[idx]), f"{gen}: records did not travel whole"
        want = expected(pred)
        assert {f: st[f] for f in want} == want, (gen, pred.plan, st, want)


@pytest.mark.parametrize("option", [{"fix_in_pass": 0}, {"junction_table": 0}, {"tile_cfg": 1}])
def test_finish_options(option):
    """without the FIX pass (the full segment finish runs), junctions found by key compares only, 2048-key tiles"""
    for gen in FLAGGED + ["junction2", "empty_next_tile", "fingerprint_collision", "cut4_high_word_1"]:
        for dt, up in ((np.dtype(np.int64), True), (np.dtype(np.float64), False)):
            case = H.GENERATORS[gen](dt, up, np.random.default_rng(len(gen) + 3))
            for flow_name in ("device_plan", "host_plan_stable"):
                check_case(case.keys, up, case.margin_bits, flow_name, extra=option)


def test_no_cut_reports_no_segment_finish():
    """a plan without a cut (range reduction, or only low digits varying) in the flow that plans on the device: the
    finish is launched and returns at once -- it is not counted as a pass, and moves nothing"""
    for gen in ("small_range", "small_values"):
        case = H.GENERATORS[gen](np.dtype(np.uint64), True, np.random.default_rng(5))
        n = len(case.keys)
        _, _, st = sort_soa(case.keys, [np.arange(n, dtype=np.uint32)], True, dict(host_plan_min_log2=24))
        assert st["cut_digit"] == 0 and st["segfix_passes"] == 0 and st["segfix_moved"] == 0, st
        assert st["algorithmic_bytes"] == st["hist_sweeps"] * n * 8 + st["passes_planned"] * 2 * n * 12, st
