"""CPU checks of bench.py's reference arm (the unmodified reference copied to baseline/_ref, driven through
oracle/ref_runner.py -- the one place besides tests/ and smoke() that may execute oracle/), of its argument checks and output
dump, and of the result writers: the JSON line bench.py prints, no GPU needed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(bench.ref_dir() is None, reason="the unmodified reference is not part of the repository; "
                                                     "baseline/setup_ref.py copies it to baseline/_ref where it is installed")
def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1", "--steps", "1",
                          "--warmup", "0", "--ref-poses", "200"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "sweeps/s" and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] == 1
    assert d["extrapolated"] is True and d["cpu_baseline"]["extrapolated"] is True and "EXTRAPOLATED" in d["cpu_baseline"]["sample"]
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


def test_result_writers_round_trip(tmp_path):
    from icm_slam_b200.offline import save_result, load_result
    rng = np.random.default_rng(7)
    res = dict(x=rng.normal(size=(3, 50)), mapa=rng.normal(size=(2, 7)), cambios=rng.random((4, 3)), mapa_inicial=rng.normal(size=(2, 9)),
               x_inicial=rng.normal(size=(3, 50)), labels=np.arange(20, dtype=np.int32))
    for ext in ("mat", "npz"):
        back = load_result(save_result(str(tmp_path / ("r." + ext)), res))
        for k in ("x", "mapa", "cambios", "mapa_inicial", "x_inicial"):
            assert np.array_equal(np.asarray(back[k]), res[k]), (ext, k)
        assert np.array_equal(np.asarray(back["labels"]).ravel(), res["labels"])


def test_steps_below_one_is_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120,
                         cwd=ROOT)
    assert out.returncode == 2 and "--steps" in out.stderr


def test_dump_outputs_writes_float64_and_a_seeded_sample(tmp_path):
    rng = np.random.default_rng(3)
    poses = rng.normal(size=(3, 1000))
    labels = rng.integers(-1, 1 << 20, size=bench.DUMP_COLUMNS + 17).astype(np.int32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), poses=poses, associations=labels)
    assert sorted(os.listdir(tmp_path / "a")) == ["associations.npy", "associations_index.npy", "poses.npy"]
    p = np.load(tmp_path / "a" / "poses.npy")
    assert p.dtype == np.float64 and np.array_equal(p, poses)
    idx = np.load(tmp_path / "a" / "associations_index.npy")
    c = np.load(tmp_path / "a" / "associations.npy")
    assert idx.dtype == c.dtype == np.float64 and c.shape == idx.shape == (bench.DUMP_COLUMNS,)
    assert np.all(np.diff(idx) > 0) and np.array_equal(c, labels[idx.astype(np.int64)])
    for f in os.listdir(tmp_path / "a"):
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
    # the largest single-GPU workload (c4: 1M poses, ~100k landmarks, ~25M labels) stays under 64 MB
    assert (3 * 1_000_000 + 2 * 2 * 316 * 316 + 2 * bench.DUMP_COLUMNS) * 8 < 64 << 20
