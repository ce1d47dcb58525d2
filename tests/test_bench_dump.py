"""bench.py --dump-outputs: the last timed step's position and velocity blocks, sampled to the rows bench.dump_rows
picks, float64 and under 64 MB, equal to what the scalar oracle computes for those cells.  --steps sets the number
of timed steps of both arms."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, *args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3",
                        "--dump-outputs", str(out_dir), *args], capture_output=True, text=True, cwd=ROOT, timeout=1200)
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads([ln for ln in r.stdout.splitlines() if ln.strip()][-1])
    assert out["steps"] == 2
    return out


def _check_against_oracle(out_dir, oracle, pos_tol, vel_tol):
    sys.path.insert(0, ROOT)
    import bench

    tles, jd, fr, _ = bench.workload("config2")
    rows = bench.dump_rows(len(tles), len(jd))
    assert 0 < len(rows) < len(tles)
    assert sorted(os.listdir(out_dir)) == ["pos.npy", "vel.npy"]
    assert sum(os.path.getsize(os.path.join(out_dir, f)) for f in os.listdir(out_dir)) <= 64_000_000
    pos = np.load(os.path.join(out_dir, "pos.npy"))
    vel = np.load(os.path.join(out_dir, "vel.npy"))
    for a in (pos, vel):
        assert a.dtype == np.float64 and a.shape == (len(rows), len(jd), 3) and np.isfinite(a).all()
    # every dumped row at every 16th epoch, the whole catalog through the oracle so its reference epoch is the bench's
    po, vo, err, _ = oracle.constellation_propagate(tles, jd[::16].copy(), fr[::16].copy(), threads=0)
    assert not err[rows].any()
    assert np.max(np.abs(pos[:, ::16] - po[rows])) < pos_tol
    assert np.max(np.abs(vel[:, ::16] - vo[rows])) < vel_tol


def test_reference_arm_dumps_its_last_step(tmp_path, oracle):
    # the CPU SIMD port is held to the scalar path at src/Sgp4Batch.zig:180-189's 1e-3 km / 1e-6 km/s
    out = _bench(tmp_path, "--impl", "reference")
    assert out["impl"] == "reference"
    _check_against_oracle(tmp_path, oracle, 1e-3, 1e-6)


@pytest.mark.gpu
def test_gpu_arm_dumps_its_last_step(tmp_path, oracle):
    out = _bench(tmp_path, "--no-subrecords", "--no-cpu-baseline")
    assert out["gpu_launches"] == 2
    _check_against_oracle(tmp_path, oracle, 1e-6, 1e-9)
