"""CPU test of bench.py's reference arm (the CPU oracle port): one JSON line with the contract's keys.  The GPU arm is
exercised on the GPU box; this guards the part of the contract that must also work without a GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ, YB_CPU_THREADS=str(min(8, os.cpu_count() or 1)), YB_CPU_IMAGES="2", CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "images/sec" and d["unit"] == "images/s"
    assert d["higher_is_better"] is True and d["value"] > 0
    for k in ("n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["product_modules_loaded"] == []          # the reference arm never touches the product package / its .so
    assert d["steps"] == 1 and len(cb["candidates"]) >= 1 and "images_per_s" in cb["candidates"][-1]
    assert all(len(c["pass_seconds_slowest_worker"]) == 1 for c in cb["candidates"] if "images_per_s" in c)


def test_bench_params_follow_the_products_conv_table():
    sys.path.insert(0, ROOT)
    import bench
    from yolov3_tensorflow_b200.model import yolov3
    ps = bench.make_bench_params()
    table = yolov3.conv_table(80)
    assert len(ps) == len(table) == 75
    for p, (cin, cout, k, s, bn) in zip(ps, table):
        assert p["w"].shape == (k, k, cin, cout) and (("gamma" in p) == bool(bn))
    assert np.all(ps[58]["b"].reshape(3, -1)[:, 4] == -2.0)
    # the GPU arm builds the same parameters from the product's table (it never imports oracle/): identical arrays
    ps2 = bench.make_bench_params(specs=table)
    for p, q in zip(ps, ps2):
        assert p.keys() == q.keys() and all(np.array_equal(p[k], q[k]) for k in p)


def _load_dump(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_writes_each_images_detections(tmp_path):
    import torch
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(1)
    n, cap = 3, 50
    out = (torch.from_numpy(rng.random((n, cap, 4), dtype=np.float32)),
           torch.from_numpy(rng.random((n, cap), dtype=np.float32)),
           torch.from_numpy(rng.integers(0, 80, (n, cap)).astype(np.int32)),
           torch.from_numpy(rng.integers(0, 10647, (n, cap)).astype(np.int32)),
           torch.tensor([50, 0, 20], dtype=torch.int32))
    assert bench.dump_outputs(str(tmp_path / "all"), out) == ["boxes", "counts", "indices", "labels", "scores"]
    got = _load_dump(tmp_path / "all")
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    rows = np.concatenate([np.arange(50), 2 * cap + np.arange(20)])      # image 0: all 50 slots, image 2: the first 20
    assert np.array_equal(got["counts"], [50, 0, 20])
    for name, t in zip(("boxes", "scores", "labels", "indices"), out):
        assert np.array_equal(got[name], t.numpy().reshape(n * cap, -1)[rows].reshape(got[name].shape)), name
    # above the byte limit: a seeded sample of the same rows, in order, identical from call to call
    for d in ("s1", "s2"):
        assert bench.dump_outputs(str(tmp_path / d), out, limit=1000) == ["boxes", "counts", "indices", "labels", "rows",
                                                                         "scores"]
    s1, s2 = _load_dump(tmp_path / "s1"), _load_dump(tmp_path / "s2")
    assert sum(a.nbytes for a in s1.values()) <= 1000
    sel = s1["rows"].astype(np.int64)
    assert len(sel) > 0 and np.all(np.diff(sel) > 0) and sel[-1] < 70
    for name in ("boxes", "scores", "labels", "indices"):
        assert np.array_equal(s1[name], got[name][sel]), name
    assert all(np.array_equal(s1[k], s2[k]) for k in s1)


@pytest.mark.gpu
def test_gpu_arm_follows_steps_and_dumps_the_last_step(tmp_path):
    """The GPU arm at a small shape, twice with different --steps: every timed loop reports the requested count, and
    the dumped detections are the same arrays (the inputs do not depend on the step count) and match the step's
    detection count."""
    dumps = []
    for steps in (2, 3):
        d = tmp_path / f"steps{steps}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                            "--batch", "4", "--size", "128", "--train-batch", "2", "--train-size", "128", "--no-train608",
                            "--no-cpu-baseline", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([l for l in r.stdout.strip().splitlines() if l.startswith("{")][-1])
        assert line["steps"] == steps and line["train"]["steps"] == steps
        got = _load_dump(d)
        assert sorted(got) == ["boxes", "counts", "indices", "labels", "scores"]
        assert all(a.dtype in (np.float32, np.float64) for a in got.values())
        assert got["counts"].shape == (4,) and got["boxes"].shape == (line["detections_per_step"], 4)
        assert got["counts"].sum() == line["detections_per_step"] > 0
        dumps.append(got)
    assert all(np.array_equal(dumps[0][k], dumps[1][k]) for k in dumps[0])
