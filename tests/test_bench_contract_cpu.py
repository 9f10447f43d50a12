"""bench.py's reference arm (CPU only) prints one JSON line with the contract's keys; runs on a small read set."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DUMPED = ("target_ids", "segments_per_target", "segment_lengths", "sample_target_ids", "sample_bases")


def test_reference_arm_json_line(tmp_path):
    dumps = []
    for run in range(2):
        dumps.append(tmp_path / f"out{run}")
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                              "--reads", "300", "--read-len", "6000", "--dump-outputs", str(dumps[-1])],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["metric"] == "corrected_bases_per_sec" and d["unit"] == "bases/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # --dump-outputs: the corrected reads of the last timed step, float arrays, identical from run to run
    a, b = ({n: np.load(p / f"{n}.npy") for n in DUMPED} for p in dumps)
    for n in DUMPED:
        assert a[n].dtype in (np.float32, np.float64) and np.array_equal(a[n], b[n]), n
    assert len(a["target_ids"]) == len(a["segments_per_target"]) > 0
    assert a["segments_per_target"].sum() == len(a["segment_lengths"])
    assert set(a["sample_target_ids"]) <= set(a["target_ids"]) and len(a["sample_target_ids"]) > 0
    assert len(a["sample_bases"]) > 0 and set(np.unique(a["sample_bases"])) <= set(map(float, b"ACGT"))
    per_target = dict(zip(a["target_ids"], np.split(a["segment_lengths"], np.cumsum(a["segments_per_target"])[:-1].astype(int))))
    assert len(a["sample_bases"]) == sum(per_target[t].sum() for t in a["sample_target_ids"])
    assert d["value"] * d["ms_per_step"] / 1e3 == pytest.approx(a["segment_lengths"].sum())  # bases of the one timed step


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
