#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 sort (BASELINE.json metric: Gpairs/s, key+payload sorted).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config c2|c3|c4] [--dump-outputs DIR]

A "step" is one complete sort of one batch of synthetic records.
  N = 1 : --config c2 (default) = BASELINE.json configs[1]: uint64 key + uint64 payload, 1e9 uniform records, ascending
          --config c3 = configs[2]: float key + (int32, double, uint16) payload streams, 5e8 records, descending
          --config c4 = configs[3]: combined DataElement<int64,double> records, 2e9 records, Zipf-skewed keys
                        (--dist few_unique: 16 distinct keys -8..7)
  N > 1 : configs[4] (weak scaling): every rank holds 1e9 records of the c2 shape; one step = sampled top
          histogram -> NCCL all-reduce -> splitters -> exact destination counts -> NCCL all-gather -> ONE scatter
          pass that writes every record straight into its destination GPU's memory over NVLink -> local sort.
`value` is device-resident throughput (records of all ranks / max-over-ranks CUDA-event time of the
sort itself; the untimed copy that restores the unsorted input between steps is outside the events).
`e2e` is the same sort through the public API with HOST (pinned) buffers, H2D + D2H inside the timing.
`--impl reference` times the reference's own CPU implementation (oracle/_ref, else the oracle port) on a
bounded sample of the SAME generator (records mix64(seed + i), tests/oracle_lib.py) and reports the time
of the records it actually sorted.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

METRIC = "Gpairs/s (key+payload) sorted"
SEED = 12345

# records per GPU, record bytes, key bytes, description (BASELINE.json configs)
CONFIGS = {
    "c2": dict(n=1_000_000_000, rec=16, kb=8, dtype="u64", up=True,
               workload="uint64 key + uint64 payload, 1e9 uniform-random records on 1 B200, ascending (BASELINE.json configs[1])"),
    "c3": dict(n=500_000_000, rec=18, kb=4, dtype="f32", up=False,
               workload="float key + 3 separate payload streams (int32, double, uint16), 5e8 records uniform in (-1,1) "
                        "+ the +-0/+-inf/denormal/FLT_MAX edge set, descending (BASELINE.json configs[2])"),
    "c4": dict(n=2_000_000_000, rec=16, kb=8, dtype="i64", up=True,
               workload="combined DataElement<int64,double> AoS records, 2e9 records, Zipf-skewed keys over 2^20 values "
                        "(BASELINE.json configs[3])"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--dist", default=None, choices=[None, "zipf", "few_unique"], help="c4 key distribution (default zipf)")
    ap.add_argument("--records", dest="n", type=int, default=0, help="records per GPU (development override)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--cpu-sample", type=int, default=0, help="records of the CPU baseline sample (default: per config)")
    ap.add_argument("--opt", action="append", default=[], help="library option name=value (development / ablations)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed sample of the arrays the last step sorted as DIR/<name>.npy")
    return ap.parse_args()


# ---------------------------------------------------------------------------------------------------
# synthetic records: ONE generator for both arms.  Record i of rank r derives from x = mix64(SEED + r*n + i)
# (counter-based; numpy on the host, torch on the device produce identical bits).
# ---------------------------------------------------------------------------------------------------
EDGE_F32 = [0.0, -0.0, float("inf"), float("-inf"), 1e-45, -1e-45, 3.4028234663852886e38, -3.4028234663852886e38]


def host_records(cfg: str, dist, start: int, count: int):
    """numpy arrays of records [start, start+count) of the workload: (keys, [payloads]) or an (n,16) uint8 AoS"""
    import oracle_lib as O
    x = O.mix64_numpy(start, count, SEED)
    idx = np.arange(start, start + count, dtype=np.int64)
    if cfg == "c2":
        return x, [idx.astype(np.uint64)]
    if cfg == "c3":
        u = (x >> np.uint64(11)).astype(np.float64) * (2.0 ** -53) * 2.0 - 1.0
        keys = u.astype(np.float32)
        for j, v in enumerate(EDGE_F32):
            pos = j * 1_000_003 - start
            if 0 <= pos < count:
                keys[pos] = np.float32(v)
        return keys, [idx.astype(np.int32), idx.astype(np.float64), (idx % 65536).astype(np.uint16)]
    keys = c4_keys_numpy(x, dist)
    rec = np.empty((count, 2), np.int64)
    rec[:, 0] = keys
    rec[:, 1] = idx.astype(np.float64).view(np.int64)
    return rec.view(np.uint8).reshape(count, 16), None


def c4_keys_numpy(x, dist):
    import oracle_lib as O
    if dist == "few_unique":
        return (x % np.uint64(16)).astype(np.int64) - 8
    u = (x >> np.uint64(11)).astype(np.float64) * (2.0 ** -53)
    rank = np.exp2(20.0 * u * u).astype(np.uint64)          # heavy head, long tail over 2^20 ranks
    with np.errstate(over="ignore"):
        h = rank * np.uint64(0x1234567) + np.uint64(99)
    # value of a rank = mix64(h): evaluated through the same generator (seed 0, counter h)
    return _mix64_values(h).view(np.int64)


def _mix64_values(h):
    import oracle_lib as O
    with np.errstate(over="ignore"):
        x = h + np.uint64(O._M1)
        x = (x ^ (x >> np.uint64(30))) * np.uint64(O._M2)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(O._M3)
        return x ^ (x >> np.uint64(31))


def device_records(cfg: str, dist, start: int, n: int, dev):
    """the same records on the device (torch), generated in chunks"""
    import torch
    import oracle_lib as O

    def s64(v):
        v &= (1 << 64) - 1
        return v - (1 << 64) if v >= (1 << 63) else v

    def lsr(t, s):
        return (t >> s) & ((1 << (64 - s)) - 1)

    def mixv(h):
        x = h + s64(O._M1)
        x = (x ^ lsr(x, 30)) * s64(O._M2)
        x = (x ^ lsr(x, 27)) * s64(O._M3)
        return x ^ lsr(x, 31)

    step = 1 << 26
    if cfg == "c2":
        keys = torch.empty(n, dtype=torch.int64, device=dev)
        for s in range(0, n, step):
            c = min(step, n - s)
            keys[s:s + c] = O.mix64_torch(start + s, c, SEED, dev)
        pay = torch.arange(start, start + n, dtype=torch.int64, device=dev)
        return [keys.view(torch.uint64), pay.view(torch.uint64)]
    if cfg == "c3":
        keys = torch.empty(n, dtype=torch.float32, device=dev)
        for s in range(0, n, step):
            c = min(step, n - s)
            x = O.mix64_torch(start + s, c, SEED, dev)
            keys[s:s + c] = (lsr(x, 11).to(torch.float64) * (2.0 ** -53) * 2.0 - 1.0).to(torch.float32)
        for j, v in enumerate(EDGE_F32):
            pos = j * 1_000_003 - start
            if 0 <= pos < n:
                keys[pos] = v
        idx = torch.arange(start, start + n, dtype=torch.int64, device=dev)
        u16 = idx & 0xFFFF  # the uint16 payload stream, held as the int16 with the same bits (torch's uint16 is barebones)
        return [keys, idx.to(torch.int32), idx.to(torch.float64), torch.where(u16 >= 32768, u16 - 65536, u16).to(torch.int16)]
    rec = torch.empty((n, 2), dtype=torch.int64, device=dev)
    for s in range(0, n, step):
        c = min(step, n - s)
        x = O.mix64_torch(start + s, c, SEED, dev)
        if dist == "few_unique":
            k = (x & 15) - 8
        else:
            u = lsr(x, 11).to(torch.float64) * (2.0 ** -53)
            rank = torch.exp2(20.0 * u * u).to(torch.int64)
            k = mixv(rank * 0x1234567 + 99)
        rec[s:s + c, 0] = k
        rec[s:s + c, 1] = torch.arange(start + s, start + s + c, dtype=torch.int64, device=dev).to(torch.float64).view(torch.int64)
        del x, k
    return [rec]


# ---------------------------------------------------------------------------------------------------
# CPU baseline (the only place bench.py touches oracle/)
# ---------------------------------------------------------------------------------------------------
DEFAULT_CPU_SAMPLE = {"c2": 1 << 27, "c3": 1 << 27, "c4": 1 << 26}


def cpu_sort_sample(cfg: str, dist, sample_n: int):
    """Sorts the first sample_n records of the workload on the host with the reference's own implementation
    (oracle/_ref: radixSort.hpp compiled as is, single-threaded like the reference) or, where that
    cannot run, the oracle port.  Returns (seconds, kind, sample description, cores, records sorted)."""
    import oracle_lib as O

    kind = "reference" if O.ref_available() else "port"
    if kind == "port":
        sample_n = min(sample_n, 1 << 23)
    keys, pays = host_records(cfg, dist, 0, sample_n)
    up = CONFIGS[cfg]["up"]
    if cfg == "c4":
        fn = O.ref_sort_aos if kind == "reference" else O.port_sort_aos
        t0 = time.perf_counter()
        fn(keys, np.int64, up)
        dt = time.perf_counter() - t0
        k = np.ascontiguousarray(keys.view(np.int64).reshape(-1, 2)[:, 0])
        assert bool(np.all(k[:-1] <= k[1:]))
    else:
        fn = O.ref_sort_soa if kind == "reference" else O.port_sort_soa
        t0 = time.perf_counter()
        fn(keys, pays, up)
        dt = time.perf_counter() - t0
        ok = O.order_key(keys[:: max(1, sample_n // (1 << 20))], up)
        assert bool(np.all(ok[:-1] <= ok[1:]))
    return dt, kind, (f"the first {sample_n} records of the workload (same counter-based generator as the GPU arm), "
                      f"1 thread (the reference is single-threaded)"), 1, sample_n


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = args.config if args.gpus == 1 else "c2"
    sample_n = args.cpu_sample or DEFAULT_CPU_SAMPLE[cfg]
    vals, secs = [], []
    kind, sample, used_n = "reference", "", sample_n
    for i in range(args.warmup + args.steps):
        dt, kind, sample, cores, used_n = cpu_sort_sample(cfg, args.dist, sample_n)
        if i >= args.warmup:
            vals.append(used_n / dt * 1e-9)
            secs.append(dt)
        if dt > 40:  # keep the whole run within minutes on a slow host
            sample_n = max(sample_n // 2, 1 << 20)
    v = statistics.mean(vals)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "Gpairs/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * statistics.mean(secs), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": CONFIGS[cfg]["dtype"], "data": "synthetic",
        "config": {"workload": CONFIGS[cfg]["workload"] + "; each step sorts a bounded sample of it on the host",
                   "records_per_step": used_n, "ms_per_step_is_for": "the records_per_step actually sorted (no extrapolation)"},
        "cpu_baseline": {"value": v, "unit": "Gpairs/s", "cores": 1, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": "Gpairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# --dump-outputs: what the timed path returned, so that two builds can be compared output for output
# ---------------------------------------------------------------------------------------------------
DUMP_SAMPLE = 1 << 20  # records per dump: at most 5 float64 columns of them, 40 MB


def dump_outputs(out_dir: str, cfg: str, work, m: int, world: int, rank: int):
    """Writes records at fixed positions of the sorted output work[*][:m] as float32 / float64 .npy files.

    The positions are one seeded random record per stratum of m / DUMP_SAMPLE records (every record when m is
    smaller) and are written too, as positions.npy.  Values are exact: 32-bit and narrower integers become
    float64, and every 64-bit integer column is split into the unsigned 32-bit halves <name>_hi / <name>_lo of its
    bit pattern.  The sort is not stable, so payloads of equal keys may legitimately come in another order."""
    import torch
    s = min(m, DUMP_SAMPLE // world)
    if s == m:
        pos = np.arange(m, dtype=np.int64)
    else:
        lo = np.arange(s, dtype=np.int64) * m // s
        hi = np.arange(1, s + 1, dtype=np.int64) * m // s
        pos = lo + (np.random.default_rng(SEED).random(s) * (hi - lo)).astype(np.int64)
    idx = torch.from_numpy(pos).to(work[0].device)

    def take(t):
        t = t[:m]
        return (t.view(torch.int64) if t.dtype == torch.uint64 else t)[idx].cpu().numpy()

    if cfg == "c2":
        cols = {"keys": take(work[0]), "payload": take(work[1])}
    elif cfg == "c3":
        cols = {"keys": take(work[0]), "payload_i32": take(work[1]), "payload_f64": take(work[2]),
                "payload_u16": take(work[3]).view(np.uint16)}
    else:
        cols = {"keys": take(work[0][:, 0]), "payload_f64": take(work[0][:, 1]).view(np.float64)}
    cols["positions"] = pos
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    prefix = f"rank{rank}_" if world > 1 else ""
    for name, a in cols.items():
        if a.dtype.kind in "iu" and a.dtype.itemsize == 8 and name != "positions":
            u = a.view(np.uint64)
            np.save(out / f"{prefix}{name}_hi.npy", (u >> np.uint64(32)).astype(np.float64))
            np.save(out / f"{prefix}{name}_lo.npy", (u & np.uint64(0xFFFFFFFF)).astype(np.float64))
        else:
            np.save(out / f"{prefix}{name}.npy", a if a.dtype.kind == "f" else a.astype(np.float64))


# ---------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.gpu_index)], stdout=self.tmp, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self, t_begin=None, t_end=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.tmp.flush()
        rows = [r.strip().split(", ") for r in Path(self.tmp.name).read_text().splitlines() if r.strip()]
        os.unlink(self.tmp.name)
        import datetime
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                if t_begin is not None:
                    ts = datetime.datetime.strptime(r[0].strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    if ts < t_begin - 0.05 or ts > t_end + 0.05:
                        continue
                sm.append(float(r[2])); mx.append(float(r[3]))
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for name, val in zip(names, r[6:10]):
                    if val.strip().lower() == "active":
                        reasons.add(name)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
def measured_peak_gbs():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic_per_launch(kernel: str):
    """dram read+write bytes per launch of the dominant kernel from the committed ncu capture, scaled to
    this run's launch size; None if no capture is committed."""
    p = ROOT / "profiles" / "dominant_kernel_traffic.json"
    if not p.exists():
        return None
    try:
        j = json.loads(p.read_text())
        return j.get(kernel)
    except Exception:
        return None


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import oracle_lib as O  # generator only (mix64); nothing under oracle/ is loaded on this arm before cpu_baseline
    import simd_radix_sort_b200 as S

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    multi = world > 1
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the sort has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    comm = None
    if multi:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        uid = [None]
        if rank == 0:
            buf = (ctypes.c_ubyte * 128)()
            rc = S.lib().b200sort_mgpu_unique_id(buf)
            if rc:
                raise S.B200SortError(rc, S.lib().b200sort_last_error().decode())
            uid[0] = bytes(buf)
        dist.broadcast_object_list(uid, src=0)
        comm = ctypes.c_void_p()
        idbuf = (ctypes.c_ubyte * 128).from_buffer_copy(uid[0])
        rc = S.lib().b200sort_mgpu_comm_create(ctypes.byref(comm), world, rank, idbuf)
        if rc:
            raise S.B200SortError(rc, S.lib().b200sort_last_error().decode())

    for o in args.opt:
        name, val = o.split("=")
        S.set_option(name, int(val))
    cfg = "c2" if multi else args.config
    C = CONFIGS[cfg]
    n = args.n or C["n"]
    rec_bytes, up = C["rec"], C["up"]
    cap = n if not multi else int(n * 1.125) + 4096
    src = device_records(cfg, args.dist, rank * n, n, dev)     # pristine input (never sorted)
    work = [torch.empty((cap,) + t.shape[1:], dtype=t.dtype, device=dev) for t in src]

    def key_bits(t):  # int64 view of the key column (c3: the float bits widened)
        if cfg == "c3":
            return t.view(torch.int32).to(torch.int64)
        if cfg == "c4":
            return t[:, 0]
        return t.view(torch.int64)

    key_sum = int(key_bits(src[0]).sum().item())  # wraps mod 2^64: a permutation-invariant checksum

    def restore():
        for w, t in zip(work, src):
            w[:n].copy_(t)

    out_n = [n]

    def do_sort():
        if not multi:
            if cfg == "c4":
                S.sort_combined(n, work[0].view(torch.uint8).reshape(-1, 16), np.int64, up=up)
            else:
                S.sort(n, *work, up=up)
        else:
            ptrs = (ctypes.c_void_p * 1)(work[1].data_ptr())
            sizes = (ctypes.c_uint32 * 1)(8)
            got = ctypes.c_int64(0)
            rc = S.lib().b200sort_mgpu_sort_soa(comm, work[0].data_ptr(), S.KEY_TYPES["uint64"], n, cap, 1, 1, ptrs, sizes,
                                                ctypes.byref(got), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
            if rc:
                raise S.B200SortError(rc, S.lib().b200sort_last_error().decode())
            out_n[0] = got.value

    def barrier():
        if multi:
            dist.barrier()
        torch.cuda.synchronize()

    def ordered(kb64):
        """int64 whose signed ascending order is the order the sort must produce"""
        if cfg == "c2":
            return kb64 ^ (-(2**63))                      # unsigned ascending
        if cfg == "c4":
            return kb64                                   # signed ascending
        neg = kb64 & 0x80000000                           # c3: float bits, descending
        u = torch.where(neg != 0, (~kb64) & 0xFFFFFFFF, kb64 ^ 0x80000000)
        return -u

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()  # nvidia-smi needs a moment to start; only samples inside the timed region are kept
    # ---- warm-up (also the correctness gate: a fast wrong sort is not a result) ----
    for w in range(args.warmup):
        restore()
        do_sort()
    torch.cuda.synchronize()
    m = out_n[0]
    ks = key_bits(work[0][:m])
    okeys = ordered(ks)
    assert bool((okeys[1:] >= okeys[:-1]).all().item()), "result is not sorted"
    my_sum = int(ks.sum().item())
    if not multi:
        assert my_sum == key_sum, "key multiset changed"
        probe = torch.randint(0, n, (1 << 20,), device=dev)
        if cfg == "c4":
            srcidx = work[0][:n, 1].view(torch.float64)[probe].to(torch.int64)
        elif cfg == "c3":
            srcidx = work[1][:n][probe].to(torch.int64)
            assert bool((work[2][:n][probe] == srcidx.to(torch.float64)).all().item()), "f64 payload stream lost its key"
            assert bool(((work[3][:n][probe].to(torch.int64) & 0xFFFF) == srcidx % 65536).all().item()), "u16 payload stream lost its key"
        else:
            srcidx = work[1][:n].view(torch.int64)[probe]
        assert bool((key_bits(src[0])[srcidx] == ks[probe]).all().item()), "payload did not follow its key"
    else:
        tot = torch.tensor([m, my_sum, key_sum], dtype=torch.int64, device=dev)  # (sums wrap mod 2^64 like the inputs')
        dist.all_reduce(tot)
        assert int(tot[0].item()) == n * world, "records were lost in the exchange"
        assert int(tot[1].item()) == int(tot[2].item()), "key multiset changed in the exchange"
        # payloads (global index): every sampled payload still points at its key
        probe = torch.randint(0, max(m, 1), (1 << 18,), device=dev)
        gidx = work[1][:m].view(torch.int64)[probe]
        regen = torch.stack([O.mix64_torch(int(i), 1, SEED, dev)[0] for i in gidx[:64].tolist()]) if m > 0 else ks[:0]
        assert bool((regen == ks[probe[:64]]).all().item()), "payload did not follow its key through the exchange"
        # rank boundaries: my last key <= next rank's first key
        edge = torch.stack([okeys[0], okeys[-1]]) if m > 0 else torch.zeros(2, dtype=torch.int64, device=dev)
        edges = [torch.zeros_like(edge) for _ in range(world)]
        dist.all_gather(edges, edge)
        for r in range(world - 1):
            assert int(edges[r][1].item()) <= int(edges[r + 1][0].item()), "rank ranges overlap"
    del okeys, ks

    # ---- timed steps ----
    S.set_option("profile", 1)
    step_ms = []
    prof = []
    launches0 = S.launch_count()
    barrier()
    t_begin = time.time()
    for k in range(args.steps):
        restore()
        if multi:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        do_sort()
        e1.record()
        e1.synchronize()
        step_ms.append(e0.elapsed_time(e1))
        prof.append(S.last_profile())
    barrier()
    t_end = time.time()
    clocks = sampler.stop(t_begin, t_end) if rank == 0 else None
    launches = S.launch_count() - launches0
    S.set_option("profile", 0)
    stats = S.last_stats()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, cfg, work, out_n[0], world, rank)

    total_ms = sum(step_ms)
    if multi:
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = (n * world) / (ms_per_step * 1e-3) * 1e-9

    # ---- end-to-end through the public API with host buffers ----
    e2e = None
    h2d = d2h = n * rec_bytes
    try:
        if args.e2e_steps <= 0:
            raise RuntimeError("skipped (--e2e-steps 0)")
        host = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in src]
        e2e_ms = []
        for k in range(args.e2e_steps + 1):  # the first one is a warm-up (staging buffers get allocated): not timed
            for h, t in zip(host, src):
                h.copy_(t)
            torch.cuda.synchronize()
            if multi:
                dist.barrier()
            t0 = time.perf_counter()
            if not multi:
                # host pointers: H2D, sort, D2H inside the call
                if cfg == "c4":
                    S.sort_combined(n, host[0].view(torch.uint8).reshape(-1, 16).numpy(), np.int64, up=up)
                else:
                    S.sort(n, *[h.numpy() if h.dtype != torch.uint64 else h.view(torch.int64).numpy().view(np.uint64) for h in host], up=up)
            else:
                for w, h in zip(work, host):
                    w[:n].copy_(h, non_blocking=True)
                do_sort()
                m = out_n[0]
                for w, h in zip(work, host):
                    h[:min(m, n)].copy_(w[:min(m, n)], non_blocking=True)
                torch.cuda.synchronize()
            if k > 0:
                e2e_ms.append((time.perf_counter() - t0) * 1e3)
        e2e_t = statistics.mean(e2e_ms)
        if multi:
            t = torch.tensor([e2e_t], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_t = float(t.item())
        if not multi:
            hk = key_bits(host[0][::4097].to(dev))
            ho = ordered(hk)
            assert bool((ho[1:] >= ho[:-1]).all().item()), "host result not sorted"
        e2e = {"value": (n * world) / (e2e_t * 1e-3) * 1e-9, "unit": "Gpairs/s", "h2d_bytes_per_step": h2d * world,
               "d2h_bytes_per_step": d2h * world, "ms_per_step": e2e_t, "steps": args.e2e_steps, "warmup": 1}
        del host
    except Exception as ex:  # e.g. the box cannot pin that much memory
        e2e = {"value": None, "unit": "Gpairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "error": str(ex)[:200]}

    if rank != 0:
        if multi:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (the digit scatter pass) ----
    peak, peak_src = measured_peak_gbs()
    # scatter launches of skipped digit positions return at once; only executed passes count
    sweep_all = [ms for step in prof for kind, ms in step if kind == "sweep"]
    n_exec = max(int(stats["passes_planned"]), 1)
    sweep_ms = sorted(sweep_all, reverse=True)[: n_exec * args.steps] if stats["algo"] == 2 else [x for x in sweep_all if x > 0.02]
    per_kind = {}
    for step in prof:
        for kind, ms in step:
            per_kind[kind] = per_kind.get(kind, 0.0) + ms / args.steps
    n_sweep_launch = stats["num"]  # records one scatter launch moves (the local sort's size on this rank)
    alg_bytes = 2 * n_sweep_launch * rec_bytes
    avg_sweep = statistics.mean(sweep_ms) if sweep_ms else None
    achieved = alg_bytes / (avg_sweep * 1e-3) * 1e-9 if avg_sweep else None
    traffic = ncu_traffic_per_launch("onesweep_kernel") if cfg == "c2" else None
    roofline = {"bound": "hbm", "kernel": "onesweep_kernel (digit scatter pass)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak if achieved else None, "peak_source": peak_src,
                "traffic": traffic * (n_sweep_launch / 67108864) if traffic else None,
                "traffic_source": ("EXTRAPOLATED: ncu --set full dram__bytes_read+write of one launch at 2^26 records "
                                   "(profiles/dominant_kernel_traffic.json) scaled linearly to this launch size") if traffic else None,
                "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": avg_sweep,
                "sweep_launches_per_step": len(sweep_ms) / args.steps,
                "ms_per_step_by_kernel": per_kind,
                "whole_sort": {"algorithmic_bytes": stats["algorithmic_bytes"],
                               "achieved_gbs": stats["algorithmic_bytes"] / (ms_per_step * 1e-3) * 1e-9 if not multi else None,
                               "floor_2NR_gbs": 2 * n * world * rec_bytes / (ms_per_step * 1e-3) * 1e-9}}

    # ---- CPU baseline beside it (bounded sample, rank 0, N=1 only) ----
    cpu = None
    if not multi and args.cpu_sample >= 0:
        dt, kind, sample, cores, used_n = cpu_sort_sample(cfg, args.dist, args.cpu_sample or DEFAULT_CPU_SAMPLE[cfg])
        cpu = {"value": used_n / dt * 1e-9, "unit": "Gpairs/s", "cores": cores, "kind": kind, "sample": sample}

    exchange = None
    if multi:
        S.lib().b200sort_mgpu_used_p2p.argtypes = [ctypes.c_void_p]
        exchange = ("scatter pass writes straight into peer memory (cudaIpc-mapped workspaces)"
                    if S.lib().b200sort_mgpu_used_p2p(comm) else "local scatter pass + ncclSend/ncclRecv")
    workload = C["workload"] if not multi else (
        f"uint64 key + uint64 payload, {world}e9 records sharded over {world} B200, exchanged over NVLink "
        "(BASELINE.json configs[4], 1e9 per GPU)")
    if cfg == "c4" and args.dist == "few_unique":
        workload = workload.replace("Zipf-skewed keys over 2^20 values", "few-unique keys (16 values -8..7)")
    line = {
        "metric": METRIC, "value": value, "unit": "Gpairs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": C["dtype"],
        "data": "synthetic",
        "config": {"workload": workload, "name": "c5" if multi else cfg,
                   "records_per_gpu": n, "record_bytes": rec_bytes, "ascending": up,
                   "l2": f"inputs ({n * rec_bytes / 1e9:.0f} GB per GPU) are larger than L2; no flush needed",
                   "algo": {1: "LSD one-sweep", 2: "hybrid MSB"}.get(stats["algo"], "?"),
                   "scatter_passes": stats["passes_planned"], "hist_sweeps": stats["hist_sweeps"],
                   "generator": "record i = f(mix64(12345 + i)) on both arms (tests/oracle_lib.py)",
                   **({"exchange": exchange} if multi else {})},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
    }
    print(json.dumps(line), flush=True)
    if multi:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
