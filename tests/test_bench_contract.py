"""bench.py against the benchmark contract: the JSON line of the reference arm (runs without a GPU) and the arrays --dump-outputs
writes (GPU)."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    pytest.importorskip("cv2")
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=REPO)
    assert out.returncode == 0, out.stderr[-2000:]
    assert len(out.stdout.strip().splitlines()) == 1, "stdout must hold the JSON line and nothing else"
    line = json.loads(out.stdout.strip())
    assert line["impl"] == "reference" and line["unit"] == "frames/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["steps"] == 1 and line["vs_baseline"] is None and line["data"] == "synthetic"
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    """--dump-outputs writes the last timed step's results: the same arrays whatever --steps (the inputs are seeded), the same
    results the line's output_checksum covers, and --steps sets the work of the timed loop."""
    small = ["--warmup", "1", "--frame-sets", "2", "--no-e2e", "--no-geometry", "--no-extra", "--cpu-sample", "0"]
    lines = {}
    for steps in (2, 3):
        out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--steps", str(steps), *small,
                              "--dump-outputs", str(tmp_path / str(steps))], capture_output=True, text=True, timeout=900, cwd=REPO)
        assert out.returncode == 0, out.stderr[-2000:]
        lines[steps] = json.loads(out.stdout.strip())
        assert lines[steps]["steps"] == steps
    assert lines[3]["gpu_launches"] * 2 == lines[2]["gpu_launches"] * 3
    names = sorted(os.listdir(tmp_path / "2"))
    assert names == sorted(os.listdir(tmp_path / "3"))
    for name in names:
        a, b = np.load(tmp_path / "2" / name), np.load(tmp_path / "3" / name)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), name
    z = {n[:-4]: np.load(tmp_path / "2" / n) for n in names}
    assert z["det_count"].shape == (2, 16) and z["det_count"].sum() > 0 and z["corr_n_obj"].sum() > 0
    assert np.array_equal(z["frame_sets"], [0, 1])
    nv, no = z["corr_n_valid"].astype(np.int32), z["corr_n_obj"].astype(np.int32)
    h = hashlib.sha1()
    h.update(nv.tobytes()); h.update(no.tobytes())
    for s in range(len(nv)):
        h.update(z["corr_img"][s, :nv[s]].astype(np.int32).tobytes())
        h.update(z["corr_obj"][s, :no[s]].tobytes())
    assert h.hexdigest()[:16] == lines[2]["output_checksum"]["sha1_16"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, cwd=REPO, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
