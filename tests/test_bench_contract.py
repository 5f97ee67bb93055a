"""bench.py's reference arm (the CPU oracle port timed on the host cores) runs without a GPU: check the JSON contract
and --dump-outputs.  On the GPU: the GPU arm's dumped outputs are the oracle arm's."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--cpu-sample-scenes", "2",
                          "--steps", "1", "--warmup", "3"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "pair_associations_per_sec"
    assert line["unit"] == "pair-associations/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["ms_per_step"] > 0
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "scenes" in cb["sample"]
    e2e = line["e2e"]
    assert e2e["value"] == line["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    assert line["config"]["workload"].startswith("cfg5")


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def _bench(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def _load(d):
    return {p.name[:-4]: np.load(p) for p in sorted(d.iterdir())}


def test_reference_arm_dumps_the_last_timed_frame(tmp_path):
    line = _bench("--impl", "reference", "--cpu-sample-scenes", "2", "--steps", "2", "--warmup", "3",
                  "--dump-outputs", str(tmp_path))
    assert line["steps"] == 2
    d = _load(tmp_path)
    assert sorted(d) == ["epochs", "ids", "lengths", "voting_types"]
    assert d["ids"].dtype == np.float64 and d["epochs"].dtype == np.float64 and d["voting_types"].dtype == np.float32
    assert len({len(a) for a in d.values()}) == 1 and len(d["ids"]) > 0
    assert np.all(d["epochs"] == 3 + 2)          # every detection of the last frame carries that frame's epoch
    bad = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert bad.returncode != 0 and "--steps" in bad.stderr


def test_dump_outputs_samples_rows_above_the_limit(tmp_path, monkeypatch):
    import bench

    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 20_000)
    ids = np.arange(5000, dtype=np.uint64) * 3
    boxes = np.arange(5000 * 6, dtype=np.float32).reshape(5000, 6)
    bench.dump_outputs(str(tmp_path), {"ids": ids, "boxes": boxes})
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 20_000
    d = _load(tmp_path)
    rows = d["rows"].astype(np.int64)
    assert len(rows) > 100 and np.all(np.diff(rows) > 0)
    assert np.array_equal(d["ids"], ids[rows].astype(np.float64)) and np.array_equal(d["boxes"], boxes[rows])


@pytest.mark.gpu
def test_gpu_arm_dumps_the_oracle_answer(tmp_path):
    """The GPU arm's last timed frame, dumped, is the oracle's on the same seeded frames (4 scenes of cfg5)."""
    common = ("--steps", "2", "--warmup", "3")
    line = _bench("--scenes", "4", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "gpu"), *common)
    assert line["steps"] == 2
    _bench("--impl", "reference", "--cpu-sample-scenes", "4", "--dump-outputs", str(tmp_path / "ref"), *common)
    g, r = _load(tmp_path / "gpu"), _load(tmp_path / "ref")
    assert sorted(g) == ["epochs", "ids", "lengths", "observed_boxes", "predicted_boxes", "voting_types"]
    for k in r:
        assert g[k].dtype == r[k].dtype and np.array_equal(g[k], r[k]), k
    assert np.all(g["epochs"] == 3 + 2)
    n = len(g["ids"])
    assert g["predicted_boxes"].shape == g["observed_boxes"].shape == (n, 6)
    assert g["predicted_boxes"].dtype == np.float32 and np.all(np.isfinite(g["observed_boxes"][:, [0, 1, 3, 4]]))
