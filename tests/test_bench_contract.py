"""bench.py contract checks: the reference arm's JSON line, the no-fallback rule, and --dump-outputs (its writer without a
GPU, the whole timed path on one)."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from multimodal_autonomous_driving_perception_and_planning_b200 import _native

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_module():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "1080p lane-detect frames/s" and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_product_sources_never_touch_the_oracle_or_the_reference_tree():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may use oracle/; nothing may read /root/reference
    at run time (docstrings citing reference lines are fine)."""
    pkg = os.path.join(ROOT, "multimodal_autonomous_driving_perception_and_planning_b200")
    for base, _, files in os.walk(pkg):
        for fn in files:
            if not fn.endswith((".py", ".cu", ".cuh", ".h")):
                continue
            src = open(os.path.join(base, fn), encoding="utf-8").read()
            assert "import oracle" not in src and "from oracle" not in src, fn
            for line in src.splitlines():
                code = line.split("#", 1)[0].split("//", 1)[0]
                assert "open('/root/reference" not in code and 'open("/root/reference' not in code, (fn, line)


def _load_dump(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_writes_every_record_field_as_float64(tmp_path):
    bench = _bench_module()
    recs = np.zeros(300, _native.RECORD_DTYPE)
    recs["n_segments"] = np.arange(300)
    recs["offset"] = np.linspace(-5, 5, 300)
    recs["side"]["points"][:, 1, :, 0] = np.arange(50)
    fit, valid = np.full((2, 2, 3), 0.5), np.ones((2, 2), np.uint8)
    bench.dump_outputs(str(tmp_path / "all"), recs, fit, valid)
    got = _load_dump(tmp_path / "all")
    want = {"side_" + k for k in _native.SIDE_DTYPE.names} | (set(_native.RECORD_DTYPE.names) - {"side"})
    assert set(got) == want | {"frame_index", "state_fit", "state_valid"}
    assert all(a.dtype == np.float64 for a in got.values())
    assert np.array_equal(got["frame_index"], np.arange(300)) and np.array_equal(got["n_segments"], np.arange(300))
    assert np.array_equal(got["offset"], recs["offset"]) and got["side_points"].shape == (300, 2, 50, 2)
    assert np.array_equal(got["side_points"][:, 1, :, 0], np.tile(np.arange(50), (300, 1)))
    assert np.array_equal(got["state_fit"], fit) and np.array_equal(got["state_valid"], valid)
    # over the size limit: the same seeded sample of frames every time, within the limit
    limit = 200_000
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), recs, fit, valid, limit=limit)
        assert sum(f.stat().st_size for f in (tmp_path / d).iterdir()) <= limit
    a, b = _load_dump(tmp_path / "a"), _load_dump(tmp_path / "b")
    idx = a["frame_index"].astype(np.int64)
    assert 0 < len(idx) < 300 and np.all(np.diff(idx) > 0)
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert np.array_equal(a["n_segments"], idx) and np.array_equal(a["offset"], recs["offset"][idx])


def test_bench_refuses_zero_steps_and_dumps_of_the_reference_arm():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                             timeout=120)
        assert out.returncode == 2 and "error" in out.stderr, extra


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step_and_repeat_exactly(tmp_path):
    """Two runs with the same arguments dump the same arrays, and they are the records (and smoothing state) that the
    public API returns for the same frames after the same number of batches: 3 warm-up + --steps timed ones."""
    import torch
    from multimodal_autonomous_driving_perception_and_planning_b200 import LaneDetector, SyntheticDataGenerator
    steps, frames = 2, 8
    dumps = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                              "--frames", str(frames), "--distinct", str(frames), "--skip-cpu", "--skip-e2e",
                              "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-2000:]
        line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
        assert json.loads(line)["steps"] == steps
        dumps.append(_load_dump(tmp_path / run))
    a, b = dumps
    assert set(a) == set(b) and all(np.array_equal(a[k], b[k]) for k in a)
    assert all(v.dtype == np.float64 for v in a.values())
    assert np.array_equal(a["frame_index"], np.arange(frames))
    dev = SyntheticDataGenerator(1920, 1080).generate_batch_device(frames, start_frame=0, device=0)
    det = LaneDetector(device=0, max_batch=frames)
    for _ in range(3 + steps):
        det.detect_batch(dev)
    torch.cuda.synchronize()
    recs = det.last_records
    for k in _native.SIDE_DTYPE.names:
        assert np.array_equal(a["side_" + k], recs["side"][k].astype(np.float64)), k
    for k in set(_native.RECORD_DTYPE.names) - {"side"}:
        assert np.array_equal(a[k], recs[k].astype(np.float64)), k
    assert a["side_valid"].any()
    for s, fit in enumerate((det.prev_left_fit, det.prev_right_fit)):
        assert a["state_valid"][0, s] == (fit is not None)
        assert fit is None or np.array_equal(a["state_fit"][0, s], fit)
    det.close()
