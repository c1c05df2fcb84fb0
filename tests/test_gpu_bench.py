"""bench.py on the device: --dump-outputs writes exact float samples of what the timed sort returned (-m gpu)."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402

pytestmark = pytest.mark.gpu


def test_bench_dump_outputs_are_the_sorted_records(tmp_path):
    n = 1 << 22
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--records", str(n), "--steps", "3", "--warmup", "1",
                        "--e2e-steps", "0", "--cpu-sample", "-1", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["gpu_launches"] > 0
    got = {p.stem: np.load(p) for p in tmp_path.glob("*.npy")}
    assert sorted(got) == ["keys_hi", "keys_lo", "payload_hi", "payload_lo", "positions"]
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    assert all(a.dtype == np.float64 for a in got.values())

    def u64(name):
        return (got[name + "_hi"].astype(np.uint64) << np.uint64(32)) | got[name + "_lo"].astype(np.uint64)

    pos = got["positions"].astype(np.int64)
    assert len(pos) == bench.DUMP_SAMPLE
    keys, _ = bench.host_records("c2", None, 0, n)
    k = u64("keys")
    assert np.array_equal(k, np.sort(keys)[pos])
    assert np.array_equal(keys[u64("payload").astype(np.int64)], k)  # every payload followed its key
