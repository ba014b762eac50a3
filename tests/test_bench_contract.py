"""bench.py's JSON contract, checked on the arm that runs without a GPU (`--impl reference`), and its
--dump-outputs files."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1",
                          "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "Mpix/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["vs_baseline"] is None and "workload" in d["config"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_reference_arm_on_other_ranks_is_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_lays_scans_end_to_end(tmp_path, monkeypatch):
    """The dump holds each frame's valid scan bytes in frame order (never the unused tail of a frame's
    buffer), whole when they fit and as the seeded sample when they do not."""
    import torch
    import bench
    rng = np.random.default_rng(3)
    lens = np.array([5, 0, 300, 17, 1])
    scan = torch.from_numpy(rng.integers(0, 256, (len(lens), 320), dtype=np.uint8))
    ovf = torch.tensor([0, 0, 1, 0, 0], dtype=torch.int32)
    valid = np.concatenate([scan[k, :n].numpy() for k, n in enumerate(lens)])
    for limit in (bench.DUMP_SAMPLE_BYTES, 64):
        monkeypatch.setattr(bench, "DUMP_SAMPLE_BYTES", limit)
        out = tmp_path / str(limit)
        bench.dump_outputs(str(out), torch, scan, torch.from_numpy(lens), ovf)
        got = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
        assert set(got) == {"scan_lengths", "scan_overflow", "scan_bytes_sample"}
        assert got["scan_lengths"].dtype == np.float64 and got["scan_lengths"].tolist() == lens.tolist()
        assert got["scan_overflow"].dtype == np.float64 and got["scan_overflow"].tolist() == [0, 0, 1, 0, 0]
        pos = bench.dump_sample_positions(int(lens.sum()))
        assert len(pos) == min(limit, lens.sum()) and (np.diff(pos) > 0).all() and pos[-1] < lens.sum()
        assert got["scan_bytes_sample"].dtype == np.float32
        assert np.array_equal(got["scan_bytes_sample"], valid[pos].astype(np.float32))
    assert np.array_equal(bench.dump_sample_positions(10 ** 8), bench.dump_sample_positions(10 ** 8))


def test_dump_outputs_is_refused_for_the_cpu_arm(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=120)
    assert out.returncode != 0 and "--dump-outputs" in out.stderr


@pytest.mark.gpu
def test_dump_outputs_are_the_encoded_scans_and_repeat(po, lib, tmp_path):
    """Two runs with the same arguments dump the same arrays, and they are the scans the CPU oracle
    encodes from bench.py's frames; --steps is the number of timed steps the JSON line reports."""
    import bench
    runs = []
    for r in range(2):
        d = tmp_path / f"run{r}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3",
                              "--warmup", "1", "--frames", "2", "--e2e-frames", "1", "--e2e-steps", "1",
                              "--configs", "none", "--no-cpu", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == 3
        assert sum(os.path.getsize(d / f) for f in os.listdir(d)) <= 64 << 20
        runs.append({f[:-4]: np.load(d / f) for f in os.listdir(d)})
    assert runs[0].keys() == runs[1].keys()
    for k in runs[0]:
        assert runs[0][k].dtype in (np.float32, np.float64)
        assert np.array_equal(runs[0][k], runs[1][k]), k
    frames = bench.make_frames(2)
    scans = [bench.scan_of(po.jpeg_encode(f, bench.W, bench.H, po.RGB, bench.QUALITY, po.S420)) for f in frames]
    assert runs[0]["scan_lengths"].tolist() == [len(s) for s in scans]
    assert runs[0]["scan_overflow"].tolist() == [0, 0]
    valid = np.frombuffer(b"".join(scans), np.uint8)
    assert np.array_equal(runs[0]["scan_bytes_sample"], valid[bench.dump_sample_positions(valid.size)].astype(np.float32))
