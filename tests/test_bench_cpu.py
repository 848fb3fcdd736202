"""bench.py's reference arm (`--impl reference`): the CPU port of the reference's path, timed on the
host cores.  Contract checks that need no GPU: the JSON line's keys, all host threads in use even
when the launcher exports OMP_NUM_THREADS=1 (torchrun does), ranks other than 0 stay silent."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra):
    env = dict(os.environ)
    env.update(env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                           "--steps", "1", "--warmup", "0"], env=env, capture_output=True, text=True, timeout=600)


def test_reference_arm_line_and_threads():
    res = _run({"OMP_NUM_THREADS": "1"})
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "rays/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("geodesic rays/sec") and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["value"] > 0 and abs(d["e2e"]["value"] - d["value"]) < 1e-6 * d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and "sample" in cb
    assert cb["cores"] == len(os.sched_getaffinity(0))
    assert d["gpu_launches"] == 0 and "workload" in d["config"]


def test_reference_arm_other_ranks_are_silent():
    res = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_dump_frame_sample(tmp_path):
    """--dump-outputs on a 4K uint8 frame: float32 pixels at float64 indices, the same pixels every call,
    at most 64 MB in all."""
    import numpy as np
    import torch
    import bench
    frame = torch.from_numpy(np.random.default_rng(1).integers(0, 256, (2160, 3840, 3), dtype=np.uint8))
    dumps = []
    for d in ("a", "b"):
        bench.dump_frame(frame, str(tmp_path / d))
        assert sum(os.path.getsize(tmp_path / d / f) for f in os.listdir(tmp_path / d)) <= 64e6
        dumps.append((np.load(tmp_path / d / "frame.npy"), np.load(tmp_path / d / "frame_pixel_index.npy")))
    (pix, idx), (pix_b, idx_b) = dumps
    assert pix.dtype == np.float32 and idx.dtype == np.float64 and pix.shape == (bench.DUMP_PIXELS, 3)
    assert np.array_equal(pix, pix_b) and np.array_equal(idx, idx_b)
    assert (np.diff(idx) > 0).all() and idx[0] >= 0 and idx[-1] < 2160 * 3840
    assert np.array_equal(pix, frame.numpy().reshape(-1, 3)[idx.astype(np.int64)])


def test_steps_must_be_positive():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True,
                         text=True, timeout=600)
    assert res.returncode == 2 and "--steps" in res.stderr
