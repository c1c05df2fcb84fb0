"""CPU checks of bench.py's plumbing: both arms must draw the SAME records (one counter-based generator, numpy on the
host, torch on the device), and the reference arm must run and print its JSON line without a GPU."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402

torch = pytest.importorskip("torch")


@pytest.mark.parametrize("cfg,dist", [("c2", None), ("c3", None), ("c4", None), ("c4", "few_unique")])
def test_host_and_device_generators_agree(cfg, dist):
    start, n = 999_900, 200_000  # (spans two of c3's injected edge values, at 1_000_003 and 2_000_006 -> only the first)
    h = bench.host_records(cfg, dist, start, n)
    d = bench.device_records(cfg, dist, start, n, "cpu")
    if cfg == "c4":
        assert np.array_equal(h[0].view(np.int64).reshape(-1, 2), d[0].numpy())
        return
    host_arrays = [h[0]] + h[1]
    assert len(host_arrays) == len(d)
    for a, b in zip(host_arrays, d):
        bb = b.view(torch.int64).numpy().view(np.uint64) if b.dtype == torch.uint64 else b.numpy()
        assert a.tobytes() == bb.tobytes(), (cfg, a.dtype)
    if cfg == "c3":
        assert np.isposinf(h[0][2 * 1_000_003 - start]) if 2 * 1_000_003 - start < n else True
        assert h[0][1_000_003 - start].tobytes() == np.float32(-0.0).tobytes()  # the edge set is really in there


def test_mix64_numpy_matches_torch():
    import oracle_lib as O
    a = O.mix64_numpy(123, 10_000, 77)
    b = O.mix64_torch(123, 10_000, 77, "cpu").numpy().view(np.uint64)
    assert np.array_equal(a, b)
    assert len(np.unique(a)) == len(a)


@pytest.mark.parametrize("cfg", ["c2", "c3", "c4"])
def test_reference_arm_prints_its_json_line(cfg):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--config", cfg, "--cpu-sample", str(1 << 16)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "Gpairs/s" and line["value"] > 0
    assert line["config"]["records_per_step"] == 1 << 16
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] == 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["gpu_launches"] == 0
    # ms_per_step is the time of the records actually sorted
    assert abs(line["ms_per_step"] * 1e-3 * line["value"] * 1e9 - (1 << 16)) < 1


@pytest.mark.parametrize("cfg", ["c2", "c3", "c4"])
def test_dump_outputs_are_exact_float_samples(cfg, tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 1000)
    work = bench.device_records(cfg, None, 0, 5000, "cpu")
    for m, want in ((5000, 1000), (700, 700)):  # a sample of a larger output, all of a smaller one
        out = tmp_path / str(m)
        bench.dump_outputs(str(out), cfg, work, m, 1, 0)
        got = {p.stem: np.load(p) for p in out.glob("*.npy")}
        assert all(a.dtype in (np.float32, np.float64) for a in got.values())
        pos = got["positions"].astype(np.int64)
        assert len(pos) == want and np.all(np.diff(pos) > 0) and pos[0] >= 0 and pos[-1] < m

        def u64(name):
            return (got[name + "_hi"].astype(np.uint64) << np.uint64(32)) | got[name + "_lo"].astype(np.uint64)

        if cfg == "c2":
            assert np.array_equal(u64("keys"), work[0].view(torch.int64).numpy().view(np.uint64)[pos])
            assert np.array_equal(u64("payload"), work[1].view(torch.int64).numpy().view(np.uint64)[pos])
        elif cfg == "c3":
            assert got["keys"].tobytes() == work[0].numpy()[pos].tobytes()
            assert np.array_equal(got["payload_i32"], work[1].numpy()[pos])
            assert np.array_equal(got["payload_f64"], work[2].numpy()[pos])
            assert np.array_equal(got["payload_u16"], work[3].numpy().view(np.uint16)[pos])
        else:
            rec = work[0].numpy()
            assert np.array_equal(u64("keys").view(np.int64), rec[pos, 0])
            assert np.array_equal(got["payload_f64"], rec[pos, 1].view(np.float64))
    # the positions are a fixed function of (m, sample size)
    bench.dump_outputs(str(tmp_path / "again"), cfg, work, 5000, 1, 0)
    assert np.array_equal(np.load(tmp_path / "again" / "positions.npy"), np.load(tmp_path / "5000" / "positions.npy"))


def test_reference_arm_other_ranks_exit_quietly():
    import os
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""
