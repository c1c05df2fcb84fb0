#!/usr/bin/env python
"""Measures unique and unique_consecutive on one GPU against torch.unique and torch.unique_consecutive; prints one JSON
line per workload.

    python tests/bench_unique.py [--iters 5] [--warmup 1] [--sizes 20,24,28] [--dtypes int32,int64,float32]

Workloads: 2^s keys for every s of --sizes, of every dtype of --dtypes, uniform (random bits; randn for float32) or
few-unique (1000 values), without and with the inverse (counts always).  Before timing, the outputs of both library
calls are checked for exact equality with torch's (`ok`).  Times come from CUDA events around each call alone, and
include reading U back (one host wait, in torch as here).  Between timed calls a 512 MB buffer is overwritten
(outside the events), so every call reads its keys from HBM, not from the 126 MB L2.

`scan_*` is the run-compaction kernel alone, from the library's profile (option "profile"), against the bytes the cost
model of DESIGN.md §4 gives it: it reads N K (plus N I of positions after the sort, I = 4 up to 2^32 keys), writes
U (K + 8) (the entries and the run starts) and, with the inverse, N 8.  `scan_share` is that rate over
bench.measured_peak_gbs()."""
from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import bench  # noqa: E402  (measured_peak_gbs)
import simd_radix_sort_b200 as S  # noqa: E402
from bench_topk import card, timed  # noqa: E402


def keys_of(dtype, n, dist, g):
    if dist == "few":
        return torch.randint(0, 1000, (n,), device="cuda", generator=g).to(dtype)
    if dtype.is_floating_point:
        return torch.randn(n, device="cuda", generator=g, dtype=dtype)
    info = torch.iinfo(dtype)
    return torch.randint(info.min, info.max, (n,), device="cuda", generator=g, dtype=dtype)


def agree(got, want):
    got, want = (got if isinstance(got, tuple) else (got,)), (want if isinstance(want, tuple) else (want,))
    return len(got) == len(want) and all(a.shape == b.shape and torch.equal(a, b) for a, b in zip(got, want))


def scan_ms(fn, x, inverse):
    """the run-compaction kernel's time: with counts asked for, the last two profile entries of kind "unique" are the
    scan and the counts kernel"""
    with S.options(profile=1):
        fn(x, return_inverse=inverse, return_counts=True)
        entries = [ms for kind, ms in S.last_profile() if kind == "unique"]
    return entries[-2]


def workload(dtype, log2n, dist, inverse, args, g):
    n = 1 << log2n
    x = keys_of(dtype, n, dist, g)
    kb = x.element_size()
    mine = {"sorted": S.unique, "consecutive": S.unique_consecutive}
    theirs = {"sorted": lambda t, **kw: torch.unique(t, sorted=True, **kw), "consecutive": torch.unique_consecutive}
    line = dict(workload=f"2^{log2n} {str(dtype).replace('torch.', '')} {dist}{' +inverse' if inverse else ''}", keys=n,
                key_bytes=kb)
    ok = True
    peak, src = bench.measured_peak_gbs()
    for mode in ("sorted", "consecutive"):
        kw = dict(return_inverse=inverse, return_counts=True)
        out = mine[mode](x, **kw)
        ok = ok and agree(out, theirs[mode](x, **kw))
        U = out[0].numel()
        line[f"{mode}_unique"] = U
        line[f"{mode}_ms"] = round(timed(lambda: mine[mode](x, **kw), args.iters, args.warmup), 4)
        line[f"{mode}_torch_ms"] = round(timed(lambda: theirs[mode](x, **kw), args.iters, args.warmup), 4)
        idx_bytes = (4 if n <= 2**32 else 8) if (mode == "sorted" and inverse) else 0
        model = n * (kb + idx_bytes) + U * (kb + 8) + (n * 8 if inverse else 0)
        t = scan_ms(mine[mode], x, inverse)
        line[f"{mode}_scan_ms"] = round(t, 4)
        line[f"{mode}_scan_model_bytes"] = model
        line[f"{mode}_scan_gbs"] = round(model / (t * 1e-3) / 1e9, 1)
        line[f"{mode}_scan_share"] = round(model / (t * 1e-3) / 1e9 / peak, 4)
    gpu, power = card()
    line.update(hbm_peak_gbs=peak, hbm_peak_source=src, gpu=gpu, power_limit=power, ok=bool(ok))
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--sizes", default="20,24,28")
    ap.add_argument("--dtypes", default="int32,int64,float32")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_unique.py measures on a GPU; there is nothing to measure without one"
    torch.cuda.set_device(0)
    g = torch.Generator(device="cuda").manual_seed(1)
    for log2n in (int(s) for s in args.sizes.split(",")):
        for dtype in (getattr(torch, d) for d in args.dtypes.split(",")):
            for dist in ("uniform", "few"):
                for inverse in (False, True):
                    workload(dtype, log2n, dist, inverse, args, g)


if __name__ == "__main__":
    main()
