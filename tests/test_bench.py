"""bench.py: argument checks, the --dump-outputs files, and (on the GPU) that the dumps are the timed results and
that --steps sets the number of timed steps, device-resident and end to end."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")
TINY = ["--gpus", "1", "--warmup", "1", "--images", "6", "--proposals", "300", "--chunk", "4",
        "--no-extras", "--no-cpu-baseline"]


def _bench(*args):
    p = subprocess.run([sys.executable, BENCH, *args], capture_output=True, text=True, timeout=900)
    return p.returncode, p.stdout, p.stderr


@pytest.mark.parametrize("args", [["--steps", "0"],
                                  ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_rejects_bad_arguments(args):
    rc, _, err = _bench(*args)
    assert rc == 2 and "error" in err, err


def test_dump_outputs_writes_float64_rows_and_samples_above_the_limit(tmp_path, monkeypatch):
    import bench
    rows = torch.arange(600 * 6, dtype=torch.float64).reshape(600, 6)
    bench.dump_outputs(str(tmp_path / "all"), {"detections": rows})
    got = np.load(tmp_path / "all" / "detections.npy")
    assert got.dtype == np.float64 and np.array_equal(got, rows.numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096 + 100 * 6 * 8)
    bench.dump_outputs(str(tmp_path / "a"), {"detections": rows})
    bench.dump_outputs(str(tmp_path / "b"), {"detections": rows})
    a, b = np.load(tmp_path / "a" / "detections.npy"), np.load(tmp_path / "b" / "detections.npy")
    assert a.shape == (100, 6) and np.array_equal(a, b)                 # fixed, seeded sample
    ids = a[:, 0].astype(np.int64) // 6
    assert (np.diff(ids) > 0).all() and np.array_equal(a, rows.numpy()[ids])   # whole rows, original order


def test_dump_outputs_shares_the_limit_and_takes_only_floats(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 200_000)
    arrays = {"rows": np.ones((4000, 10)), "masks": np.ones((40, 30, 40), np.float32)}   # 320 kB + 192 kB
    bench.dump_outputs(str(tmp_path), arrays)
    got = {k: np.load(tmp_path / f"{k}.npy") for k in arrays}
    assert sum((tmp_path / f"{k}.npy").stat().st_size for k in arrays) <= 200_000
    assert got["rows"].dtype == np.float64 and got["masks"].dtype == np.float32
    assert 0 < len(got["rows"]) < 4000 and 0 < len(got["masks"]) < 40
    small = {"rows": np.ones((10, 10)), "masks": np.ones((20, 30, 40), np.float32)}      # under the limit: kept whole
    bench.dump_outputs(str(tmp_path / "small"), small)
    assert all(np.array_equal(np.load(tmp_path / "small" / f"{k}.npy"), v) for k, v in small.items())
    with pytest.raises(TypeError):
        bench.dump_outputs(str(tmp_path / "u8"), {"masks": np.ones((2, 2), np.uint8)})


@pytest.mark.gpu
def test_dump_is_the_timed_result_and_steps_set_the_timed_steps(tmp_path):
    lines, dumps = {}, {}
    for steps in (1, 2):
        out = tmp_path / f"steps{steps}"
        rc, stdout, err = _bench(*TINY, "--steps", str(steps), "--dump-outputs", str(out))
        assert rc == 0, err[-3000:]
        lines[steps] = json.loads(stdout.strip().splitlines()[-1])
        dumps[steps] = np.load(out / "detections.npy")
    for steps, line in lines.items():
        d = dumps[steps]
        assert line["steps"] == steps and d.dtype == np.float64 and d.shape == (line["detections"], 6)
        assert hashlib.sha256(d.tobytes()).hexdigest() == line["detections_sha256"]
        assert line["e2e"]["steps"] == steps and line["e2e"]["rle_complete"]
    assert lines[1]["detections"] > 0
    assert np.array_equal(dumps[1], dumps[2])                           # same inputs, same result
    assert lines[2]["gpu_launches"] == 2 * lines[1]["gpu_launches"]     # launches counted over the timed steps only


@pytest.mark.gpu
def test_antialias_dump_is_the_last_step_and_repeats(tmp_path):
    dumps, names = {}, ("discovery", "annotations", "masks", "mask_index")
    for steps in (1, 2):
        out = tmp_path / f"steps{steps}"
        rc, stdout, err = _bench("--config", "antialias", "--images", "2", "--proposals", "300", "--warmup", "1",
                                 "--steps", str(steps), "--dump-outputs", str(out))
        assert rc == 0, err[-3000:]
        line = json.loads(stdout.strip().splitlines()[-1])
        d = dumps[steps] = {k: np.load(out / f"{k}.npy") for k in names}
        assert line["steps"] == steps and d["annotations"].shape == (line["annotations"], 10) and line["annotations"] > 0
        assert d["discovery"].shape[1] == 5 and set(np.unique(d["discovery"][:, 0])) <= {0.0, 1.0}
        k = min(line["annotations"], 16)
        assert d["masks"].shape == (k, 480, 640) and d["masks"].dtype == np.float32
        assert set(np.unique(d["masks"])) <= {0.0, 1.0} and d["mask_index"].shape == (k,)
        assert (np.diff(d["mask_index"]) > 0).all() and d["mask_index"][-1] < line["annotations"]
    for k in names:
        assert np.array_equal(dumps[1][k], dumps[2][k]), k                 # same inputs, same result
