"""CPU: the reference arm of bench.py prints one JSON line with the contract's keys.
GPU: --dump-outputs writes the records of the last timed step, the same ones from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json(built):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c2",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["unit"] == "Mrays/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and "workload" in line["config"]


def test_reference_arm_other_ranks_exit_quietly(built):
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=60, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_reference_arm_refuses_dump_outputs(tmp_path):
    """The CPU reference returns no GPU records: --dump-outputs with --impl reference is an error, not an empty directory."""
    d = tmp_path / "dump"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(d)],
                         capture_output=True, text=True, timeout=60)
    assert out.returncode == 2 and "--dump-outputs" in out.stderr and not d.exists()


@pytest.mark.gpu
def test_dump_outputs_repeat_and_match_the_oracle(built, port, tmp_path):
    """The C2 wavefront (cast, trace, spawn, trace) with --dump-outputs, twice: the same files with the same bytes, at most
    64 MB, float32 / float64 only; the hits written are the oracle's hits for the rays written beside them."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tracer_b200 import harness as H, layout as L
    dumps = []
    for k in range(2):
        d = tmp_path / f"run{k}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c2", "--steps", "3", "--warmup", "1",
                              "--no-cpu-baseline", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-4000:]
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["steps"] == 3 and line["e2e"]["steps"] == 3
        files = sorted(d.iterdir())
        assert sum(f.stat().st_size for f in files) <= 64 << 20
        dumps.append({f.stem: np.load(f) for f in files})
    a, b = dumps
    assert a.keys() == b.keys() and all(a[k].tobytes() == b[k].tobytes() for k in a), "two runs wrote different outputs"
    assert {v.dtype for v in a.values()} <= {np.dtype(np.float32), np.dtype(np.float64)}
    idx = a["ray_index"]
    n_primary = 1920 * 1080
    assert np.all(np.diff(idx) > 0) and idx[0] >= 0 and (idx < n_primary).any() and (idx >= n_primary).any()
    rays = np.zeros(idx.size, dtype=L.ray_dtype)
    hits = np.zeros(idx.size, dtype=L.hit_dtype)
    for dt, rec, name in ((L.ray_dtype, rays, "ray"), (L.hit_dtype, hits, "hit")):
        for f in dt.names:
            rec[f] = a[f"{name}_{f}"]
    sub = np.arange(0, idx.size, 7)
    want = port.trace(H.scene_c2(), rays[sub], nthreads=8)["hits"]
    for f in L.hit_dtype.names:                                  # C2 is triangles only: every field bit-exact
        assert np.array_equal(hits[f][sub].view(np.uint32), want[f].view(np.uint32)), f


@pytest.mark.gpu
def test_dump_outputs_whole_batch_of_a_plain_trace(built, port, tmp_path):
    """C1 (one trq_trace over 921,600 camera rays, small enough to be written whole): every ray's record, in batch order,
    ids and t bit for bit the oracle's."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tracer_b200 import harness as H, layout as L
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1", "--steps", "1", "--warmup", "1",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-4000:]
    a = {f.stem: np.load(f) for f in tmp_path.iterdir()}
    assert sorted(a) == sorted(["ray_index"] + [f"hit_{f}" for f in L.hit_dtype.names])
    rays = H.camera_rays((13, 2, 3), (0, 0, 0), np.float32(20 * np.pi / 180), 1280, 720)
    assert np.array_equal(a["ray_index"], np.arange(rays.size, dtype=np.float64))
    sub = np.arange(0, rays.size, 11)
    want = port.trace(H.scene_c1(), rays[sub], nthreads=8)["hits"]
    for f in ("flags", "pType", "pIndex", "leafNode", "material"):
        assert np.array_equal(a[f"hit_{f}"][sub], want[f].astype(np.float64)), f
    assert np.array_equal(a["hit_t"][sub].view(np.uint32), want["t"].view(np.uint32))
