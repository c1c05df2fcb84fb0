#!/usr/bin/env python
"""Measures the top-k selection on one GPU; prints one JSON line per workload.

    python tests/bench_topk.py [--iters 10] [--warmup 2] [--only a,b,c,d,e,f]

Workloads (N keys of K bytes in all; largest unless said otherwise):
  a  64 x 128256 f32, k = 50 (the top-k sampling shape), against torch.topk and against S.sort_rows + slice
  b  the same with k = 1024
  c  one row of 2^30 f32, k = 1000, against torch.topk
  d  one row of 2^28 u64 keys + u64 payload, k = 2^16, against S.sort + slice
  e  4096 x 32768 f32, k = 32
  f  one row of 2^28 u32 keys with a constant top byte, k = 1000 (candidates never fit the buffer: the re-read path)
Times come from CUDA events around each call alone.  Between timed calls a 512 MB buffer is overwritten (outside the
events), so every call reads its keys from HBM, not from the 126 MB L2; the sort baselines also get their unsorted
input restored there.  `keys_read_share` is N K bytes over the call time, as a share of bench.measured_peak_gbs():
the share of peak bandwidth one read of the keys would take.  `ok` comes from the checks of tests/test_gpu_topk.py:
the keys equal the reference's (torch.topk, or the sorted array's first k), the indices of a row are distinct,
keys[index] equals the keys, and the payload output is the payload at the index."""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402  (measured_peak_gbs)
import simd_radix_sort_b200 as S  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # (the power limit is part of the number; say why it is missing)
        out = f"unknown ({e})"
    return name, out


_scrub = None


def scrub():
    """overwrite 512 MB, which evicts the previous call's data from L2"""
    global _scrub
    if _scrub is None:
        _scrub = torch.empty(1 << 27, dtype=torch.float32, device="cuda")
    _scrub.fill_(1.0)


def timed(fn, iters, warmup, restore=lambda: None):
    for _ in range(warmup):
        restore()
        fn()
    ms = 0.0
    for _ in range(iters):
        restore()
        scrub()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms += e0.elapsed_time(e1)
    return ms / iters


def check(keys, vals, idx, expected_vals, pay=None, pay_out=None):
    """keys (B, L), outputs (B, k): values as expected (bit for bit), distinct indices, keys[index] = values, payload[index]"""
    if not torch.equal(vals.view(-1).view(torch.uint8), expected_vals.reshape(-1).contiguous().view(torch.uint8)):
        return False
    s = torch.sort(idx, dim=1).values
    if s.shape[1] > 1 and not bool((s[:, 1:] != s[:, :-1]).all()):
        return False
    if bool((idx < 0).any()) or bool((idx >= keys.shape[1]).any()):
        return False
    if not torch.equal(torch.gather(keys, 1, idx).view(torch.uint8), vals.view(torch.uint8)):
        return False
    return pay is None or torch.equal(torch.gather(pay, 1, idx), pay_out)


def report(name, ms, n, key_bytes, ok, extra):
    peak, src = bench.measured_peak_gbs()
    gbs = n * key_bytes / (ms * 1e-3) / 1e9
    gpu, power = card()
    line = dict(workload=name, ms_per_call=round(ms, 4), keys=n, bytes_NK=n * key_bytes, keys_read_gbs=round(gbs, 1),
                keys_read_share=round(gbs / peak, 4), hbm_peak_gbs=peak, hbm_peak_source=src, gpu=gpu, power_limit=power, ok=bool(ok))
    line.update(extra)
    print(json.dumps(line), flush=True)


def float_rows(name, B, L, k, args, sort_baseline):
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(B, L, device="cuda", generator=g)
    ms = timed(lambda: S.topk(x, k), args.iters, args.warmup)
    vals, idx = S.topk(x, k)
    ok = check(x, vals, idx, torch.topk(x, k).values)
    extra = dict(k=k, torch_topk_ms=round(timed(lambda: torch.topk(x, k), args.iters, args.warmup), 4))
    if sort_baseline:
        y, i = x.clone(), torch.empty(B, L, dtype=torch.int64, device="cuda")
        i0 = torch.arange(L, device="cuda").repeat(B, 1)

        def restore():
            y.copy_(x)
            i.copy_(i0)

        def sort_slice():
            S.sort_rows(y, i, up=False)
            return y[:, :k].clone(), i[:, :k].clone()

        extra["sort_rows_slice_ms"] = round(timed(sort_slice, args.iters, args.warmup, restore), 4)
    report(name, ms, B * L, 4, ok, extra)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--only", default="a,b,c,d,e,f")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_topk.py measures on a GPU; there is nothing to measure without one"
    torch.cuda.set_device(0)
    which = set(args.only.split(","))
    if "a" in which:
        float_rows("a: 64 x 128256 f32, k = 50", 64, 128256, 50, args, True)
    if "b" in which:
        float_rows("b: 64 x 128256 f32, k = 1024", 64, 128256, 1024, args, True)
    if "c" in which:
        float_rows("c: 2^30 f32, k = 1000", 1, 1 << 30, 1000, args, False)
    if "d" in which:
        n, k = 1 << 28, 1 << 16
        g = torch.Generator(device="cuda").manual_seed(2)
        k0 = torch.randint(-2**63, 2**63 - 1, (n,), device="cuda", generator=g, dtype=torch.int64)
        keys, p0 = k0.view(torch.uint64), torch.arange(n, device="cuda", dtype=torch.int64)
        ms = timed(lambda: S.topk(keys, k, p0), args.iters, args.warmup)
        vals, idx, po = S.topk(keys, k, p0)
        y, p = k0.clone(), p0.clone()

        def restore():
            y.copy_(k0)
            p.copy_(p0)

        def sort_slice():
            S.sort(n, y.view(torch.uint64), p, up=False)
            return y[:k].clone(), p[:k].clone()

        sort_ms = timed(sort_slice, max(1, args.iters // 2), 1, restore)
        restore()
        ev, _ = sort_slice()
        ok = check(k0.view(1, n), vals.view(torch.int64).view(1, k), idx.view(1, k), ev, p0.view(1, n), po.view(1, k))
        report("d: 2^28 u64 + u64 payload, k = 2^16", ms, n, 8, ok, dict(k=k, sort_slice_ms=round(sort_ms, 4)))
        del k0, y, p, p0
    if "e" in which:
        float_rows("e: 4096 x 32768 f32, k = 32", 4096, 32768, 32, args, False)
    if "f" in which:
        n, k = 1 << 28, 1000
        g = torch.Generator(device="cuda").manual_seed(3)
        x = torch.randint(0, 2**24, (n,), device="cuda", generator=g, dtype=torch.int32) | 0x2B000000  # (as int32: the same order)
        keys = x.view(torch.uint32)
        ms = timed(lambda: S.topk(keys, k), args.iters, args.warmup)
        vals, idx = S.topk(keys, k)
        ok = check(x.view(1, n), vals.view(torch.int32).view(1, k), idx.view(1, k), torch.topk(x, k).values)
        report("f: 2^28 u32 with a constant top byte, k = 1000", ms, n, 4, ok,
               dict(k=k, torch_topk_ms=round(timed(lambda: torch.topk(x, k), args.iters, args.warmup), 4)))


if __name__ == "__main__":
    main()
