"""bench.py's JSON-line contract, checked on the CPU through the reference arm (the GPU arm prints the same keys plus the
roofline / launch counters; it is exercised on the GPU box)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args, timeout=900):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT)


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout  # exactly one line on stdout, whatever libraries print
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                "data", "config", "e2e", "cpu_baseline"):
        assert key in d, key
    assert d["metric"] == "pairwise_registrations_per_sec" and d["unit"] == "pairs/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["vs_baseline"] is None and "workload" in d["config"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]


def test_gpu_arm_fails_loudly_without_a_device():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode != 0 and not r.stdout.strip()  # no CPU fallback, no number


def test_dump_outputs_keeps_a_fixed_ordered_sample_within_the_budget(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    big = np.arange(100_000 * 4, dtype=np.float32).reshape(-1, 4)  # 1.6 MB
    small = np.eye(4)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"big": big, "small": small}, budget=1 << 20)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 1 << 20  # files, headers included
    a = np.load(tmp_path / "a" / "big.npy")
    assert np.array_equal(a, np.load(tmp_path / "b" / "big.npy"))  # the same sample every run
    assert a.dtype == np.float32 and a.shape[1] == 4 and len(a) > 0.95 * (1 << 19) / 16  # close to half the budget
    assert (np.diff(a[:, 0]) > 0).all() and (a[:, 0] % 4 == 0).all() and (a[:, 1:] == a[:, :1] + [1, 2, 3]).all()  # whole rows, in order
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), small)  # within its share: saved whole


def test_reference_arm_dumps_what_its_timed_step_computed(tmp_path, oracle, tiny_maps):
    import oracle_py
    r = _bench("--impl", "reference", "--workload", "tiny", "--steps", "2", "--warmup", "0", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    assert os.listdir(tmp_path) == ["transforms.npy"]
    got = np.load(tmp_path / "transforms.npy")
    want = oracle.estimate_maps_transforms(tiny_maps[0], oracle_py.default_params(descriptor_type=2))["transforms"]
    assert got.dtype == np.float32 and got.shape == (2, 4, 4) and np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_steps_below_one_are_refused():
    r = _bench("--impl", "reference", "--workload", "tiny", "--steps", "0")
    assert r.returncode != 0 and not r.stdout.strip()


@pytest.mark.gpu
def test_gpu_arm_times_the_steps_asked_for_and_dumps_what_a_caller_receives(tmp_path, ctx, mm, tiny_maps):
    lines = {}
    for steps in (1, 2):
        r = _bench("--workload", "tiny", "--steps", str(steps), "--warmup", "0", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / str(steps)))
        assert r.returncode == 0, r.stderr[-2000:]
        lines[steps] = json.loads(r.stdout)
        assert os.listdir(tmp_path / str(steps)) == ["transforms.npy"]
    assert lines[2]["steps"] == 2 and lines[2]["gpu_launches"] == 2 * lines[1]["gpu_launches"] > 0  # launches of the timed window
    want = ctx.estimate_maps_transforms(tiny_maps[0], mm.default_params(descriptor_type="FPFH"))
    for steps in (1, 2):
        got = np.load(tmp_path / str(steps) / "transforms.npy")
        assert got.dtype == np.float32 and got.shape == (2, 4, 4) and np.array_equal(got.view(np.uint32), want.view(np.uint32))
