#!/usr/bin/env python
"""Measures the segmented sort on one GPU; prints one JSON line per workload.

    python tests/bench_segmented.py [--iters 10] [--warmup 2] [--only a,b,c,d,e]

Workloads (records are key + payload, R bytes each):
  a  2^17 rows x 1024 u32 keys + u32 payload (sort_rows), against torch.sort(dim=-1) + the same payload gather
  b  2^27 u64 keys + u64 payload in segments of random length 1..4000
  c  64 x 128256 f32 logits + int64 index (the top-p sampling shape), against torch.sort(dim=-1)
  d  u64 keys + u64 payload: 16 segments of 2^24 records plus 10^5 short ones (one whole-array sort per long one)
  e  the baseline the segmented call replaces: one b200sort_sort_soa call per segment, on a subsample of a and b
Times come from CUDA events around the sort call alone; the unsorted input is restored between calls, outside
the events.  `hbm_share` is 2 N R bytes over the call time, as a share of bench.measured_peak_gbs().  Every
result is checked: keys equal the input keys gathered by the payload (a global index), every payload stays in
its own segment, and keys are in order inside every segment."""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
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


def ordered(k: torch.Tensor, up=True) -> torch.Tensor:
    """int64 tensor whose order is the library's total order of the keys (float, signed or unsigned bit patterns)"""
    if k.dtype == torch.float32:
        u = k.view(torch.int32).to(torch.int64) & 0xFFFFFFFF
        u = torch.where(u >= 0x80000000, 0xFFFFFFFF - u, u + 0x80000000)
    elif k.dtype == torch.int64:  # (holds the u64 bit patterns: flipping the sign bit orders them as unsigned)
        u = k ^ torch.iinfo(torch.int64).min
    else:  # u32 held in int64
        u = k
    return u if up else -u - 1


def check(keys_in, keys_out, idx_out, seg_of, up=True):
    """keys_out = keys_in[idx_out]; every index stays in its segment; keys in order inside every segment"""
    if not torch.equal(keys_in[idx_out], keys_out):
        return False
    pos = torch.arange(len(keys_out), device=keys_out.device)
    if not torch.equal(seg_of[idx_out], seg_of[pos]):
        return False
    o = ordered(keys_out, up)
    same = seg_of[1:] == seg_of[:-1]
    return bool(((o[1:] >= o[:-1]) | ~same).all())


def timed(fn, restore, iters, warmup):
    for _ in range(warmup):
        restore()
        fn()
    ms = 0.0
    for _ in range(iters):  # (restore() rewrites the input, which also evicts it from L2 for inputs above 126 MB)
        restore()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms += e0.elapsed_time(e1)
    return ms / iters


def report(name, ms, n, rec_bytes, ok, extra=None):
    peak, src = bench.measured_peak_gbs()
    gbs = 2 * n * rec_bytes / (ms * 1e-3) / 1e9
    gpu, power = card()
    line = dict(workload=name, ms_per_call=round(ms, 4), records_per_s=n / (ms * 1e-3), bytes_2NR=2 * n * rec_bytes,
                achieved_gbs=round(gbs, 1), hbm_share=round(gbs / peak, 4), hbm_peak_gbs=peak, hbm_peak_source=src,
                gpu=gpu, power_limit=power, ok=bool(ok))
    if extra:
        line.update(extra)
    print(json.dumps(line), flush=True)


def segments(lengths, dev):
    offsets = torch.zeros(len(lengths) + 1, dtype=torch.int64, device=dev)
    offsets[1:] = torch.cumsum(torch.as_tensor(lengths, dtype=torch.int64, device=dev), 0)
    seg_of = torch.repeat_interleave(torch.arange(len(lengths), device=dev), torch.as_tensor(lengths, device=dev))
    return offsets, seg_of


def rows(B, L, dtype, idx_dtype, up, args, name, dev, baseline):
    g = torch.Generator(device=dev).manual_seed(1)
    if dtype == torch.float32:
        k0 = torch.randn(B, L, device=dev, generator=g)
    else:  # (u32 keys below 2^31: torch.sort of the same bits as int32 gives the same order)
        k0 = torch.randint(0, 2**31, (B, L), device=dev, generator=g, dtype=torch.int32)
    i0 = torch.arange(L, device=dev, dtype=idx_dtype).repeat(B, 1).contiguous()
    k, i = k0.clone(), i0.clone()

    def restore():
        k.copy_(k0)
        i.copy_(i0)

    kv = k if dtype == torch.float32 else k.view(torch.uint32)
    ms = timed(lambda: S.sort_rows(kv, i, up=up), restore, args.iters, args.warmup)
    ok = torch.equal(k, torch.sort(k0, dim=-1, descending=not up).values) and torch.equal(torch.gather(k0, 1, i.to(torch.int64)), k)
    rec = k0.element_size() + i0.element_size()
    extra = {}
    if baseline:
        def torch_sort():
            v, p = torch.sort(k0, dim=-1, descending=not up)
            torch.gather(i0, 1, p)

        extra["torch_sort_ms"] = round(timed(torch_sort, lambda: None, args.iters, args.warmup), 4)
    report(name, ms, B * L, rec, ok, extra)


def soa_segments(lengths, name, args, dev):
    offsets, seg_of = segments(lengths, dev)
    n = int(offsets[-1])
    g = torch.Generator(device=dev).manual_seed(2)
    k0 = torch.randint(-2**63, 2**63 - 1, (n,), device=dev, generator=g, dtype=torch.int64)
    i0 = torch.arange(n, device=dev, dtype=torch.int64)
    k, i = k0.clone(), i0.clone()

    def restore():
        k.copy_(k0)
        i.copy_(i0)

    def call():  # (int64 tensors holding u64 bit patterns: sorted as uint64 through the C ABI)
        ptrs = (S._api.ctypes.c_void_p * 1)(i.data_ptr())
        sizes = (S._api.ctypes.c_uint32 * 1)(8)
        rc = S.lib().b200sort_sort_segmented_soa(k.data_ptr(), S.KEY_TYPES["uint64"], n, len(lengths), offsets.data_ptr(), 1, 1, ptrs,
                                                 sizes, torch.cuda.current_stream().cuda_stream, None, 0)
        S._api._check(rc)

    ms = timed(call, restore, args.iters, args.warmup)
    report(name, ms, n, 16, check(k0, k, i, seg_of), dict(segments=len(lengths)))
    return offsets, k0


def per_call(name, offsets, k0, i0, n_sub, args):
    """one b200sort_sort_soa call per segment, over the first n_sub segments"""
    offs = offsets[: n_sub + 1].cpu().tolist()
    k, i = k0.clone(), i0.clone()

    def restore():
        k.copy_(k0)
        i.copy_(i0)

    def calls():
        for s, e in zip(offs[:-1], offs[1:]):
            S.sort(e - s, k[s:e], i[s:e])

    ms = timed(calls, restore, max(1, args.iters // 5), 1)
    n = offs[-1] - offs[0]
    report(name, ms, n, k0.element_size() + i0.element_size(), True, dict(segments=n_sub, ms_per_segment=round(ms / n_sub, 5)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--only", default="a,b,c,d,e")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_segmented.py measures on a GPU; there is nothing to measure without one"
    dev = torch.device("cuda:0")
    which = set(args.only.split(","))
    rng = np.random.default_rng(5)
    if "a" in which:
        rows(1 << 17, 1024, torch.int32, torch.int32, True, args, "a: 2^17 x 1024 u32 + u32 (sort_rows)", dev, True)
    if "b" in which or "e" in which:
        lens_b = rng.integers(1, 4001, (1 << 27) // 2000 + 10_000)
        ends = np.cumsum(lens_b)
        cut = int(np.searchsorted(ends, 1 << 27))  # the segment that reaches 2^27 records is cut there
        lens_b = lens_b[: cut + 1]
        lens_b[-1] -= int(ends[cut]) - (1 << 27)
        offsets_b, k0_b = soa_segments(lens_b.tolist(), "b: 2^27 u64 + u64, segments of 1..4000", args, dev) if "b" in which else (None, None)
    if "c" in which:
        rows(64, 128256, torch.float32, torch.int64, False, args, "c: 64 x 128256 f32 + int64 index (sort_rows, descending)", dev, True)
    if "d" in which:
        small = rng.integers(2, 200, 100_000).tolist()
        lens_d = [1 << 24] * 16 + small
        rng.shuffle(lens_d)
        soa_segments(lens_d, "d: u64 + u64, 16 x 2^24 + 10^5 short segments", args, dev)
    if "e" in which:
        B, L = 1000, 1024
        g = torch.Generator(device=dev).manual_seed(1)
        k0 = torch.randint(0, 2**31, (B * L,), device=dev, generator=g, dtype=torch.int64).to(torch.int32)
        i0 = torch.arange(B * L, device=dev, dtype=torch.int32)
        per_call("e: per-call sort, 1000 rows of workload a", torch.arange(B + 1, device=dev) * L, k0, i0, B, args)
        if offsets_b is None:
            offsets_b, _ = segments(lens_b.tolist(), dev)
        n_sub = 1000
        n = int(offsets_b[n_sub])
        k0 = torch.randint(-2**63, 2**63 - 1, (n,), device=dev, generator=g, dtype=torch.int64)
        per_call("e: per-call sort, 1000 segments of workload b", offsets_b, k0, torch.arange(n, device=dev, dtype=torch.int64), n_sub, args)


if __name__ == "__main__":
    main()
