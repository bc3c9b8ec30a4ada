"""Checks of bench.py.  CPU: the reference arm (`bench.py --impl reference`) prints one JSON line with the keys every bench
line carries, a non-zero rank under a multi-rank launch prints nothing and exits 0, the b200 arm refuses to run without a
CUDA device instead of falling back to the CPU path, and --dump-outputs keeps to its size budget.  GPU: the arrays
--dump-outputs writes are what the library returns for the same seeded inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None, timeout=600):
    e = dict(os.environ)
    e.pop("RANK", None); e.pop("WORLD_SIZE", None); e.pop("LOCAL_RANK", None)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, env=e,
                          timeout=timeout, cwd=ROOT)


def test_reference_arm_line():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--ref-chunks", "2", "--n-target", "700", "--no-one-core"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1                                   # ONE JSON line on stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "ncuts_chunks_per_sec" and d["unit"] == "chunks/s"
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1 and d["higher_is_better"] is True
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and d["dtype"] == "f64"
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert abs(d["value"] - 2 / (d["ms_per_step"] / 1e3)) <= 1e-6 * d["value"]          # chunks of a step / its time
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]


def test_reference_arm_other_ranks_stay_silent():
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1", "--ref-chunks", "1", "--n-target", "700"],
             env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29999"}, timeout=120)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip() == ""


def test_b200_arm_needs_a_device():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a CUDA device is present")
    r = _run(["--steps", "1", "--warmup", "1", "--batch", "1", "--n-target", "600", "--cpu-chunks", "0"], timeout=300)
    assert r.returncode != 0                                 # no silent CPU path
    assert r.stdout.strip() == ""


def test_bad_arguments_are_refused():
    r = _run(["--steps", "0"], timeout=120)
    assert r.returncode != 0 and "--steps" in r.stderr and r.stdout.strip() == ""
    r = _run(["--impl", "reference", "--dump-outputs", "unused"], timeout=120)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr and r.stdout.strip() == ""


def test_dump_outputs_types_and_budget(tmp_path, monkeypatch):
    import bench
    rng = np.random.default_rng(3)
    labels = rng.integers(0, 500, size=300_000).astype(np.int32)
    arrays = {"labels": labels, "num_segments": np.array([7, 9], np.int32), "score": np.float64(0.25)}
    bench.dump_outputs(str(tmp_path / "whole"), arrays)
    got = {f[:-4]: np.load(tmp_path / "whole" / f) for f in os.listdir(tmp_path / "whole")}
    assert sorted(got) == ["labels", "num_segments", "score"]
    assert got["labels"].dtype == np.float32 and np.array_equal(got["labels"], labels)
    assert got["score"].dtype == np.float64 and got["score"] == 0.25
    # over the budget: the large array is sampled, the same elements every time, small ones stay whole
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["labels.npy", "labels_index.npy", "num_segments.npy", "score.npy"]
    assert sum(np.load(tmp_path / "a" / f).nbytes for f in files) <= 1 << 20
    a = {f: np.load(tmp_path / "a" / f) for f in files}
    assert all(np.array_equal(a[f], np.load(tmp_path / "b" / f)) for f in files)
    idx = a["labels_index.npy"]
    assert idx.dtype == np.float64 and len(idx) > 50_000 and np.all(np.diff(idx) > 0)
    assert np.array_equal(a["labels.npy"], labels[idx.astype(np.int64)])
    assert np.array_equal(a["num_segments.npy"], [7, 9])


@pytest.mark.gpu
def test_dump_outputs_are_the_library_results(cuda_device, tmp_path):
    """Batch and map workload at a small size: the dumped labels (and map metrics) equal one library call on the same
    seeded chunks."""
    import bench
    from autoinst_b200 import api
    from autoinst_b200.synthetic import CONFIGS, make_map
    cfg = CONFIGS["tarl_spatial"]
    kw = dict(alpha=cfg["alpha"], theta=cfg["theta"], T=cfg["T"], device=cuda_device)
    common = ["--steps", "2", "--warmup", "1", "--cpu-chunks", "0", "--roof-steps", "0", "--no-python-surface"]

    r = _run(common + ["--batch", "3", "--n-target", "1500", "--seed", "50", "--dump-outputs", str(tmp_path / "batch")])
    assert r.returncode == 0, r.stderr[-2000:]
    chunks = bench.make_batch(3, 1500, 50, "tarl_spatial")
    res = api.segment_chunks([c.points for c in chunks], [c.tarl for c in chunks], **kw)
    lab = np.load(tmp_path / "batch" / "labels.npy")
    assert lab.dtype == np.float32 and np.array_equal(lab, np.concatenate(res.labels))
    assert np.array_equal(np.load(tmp_path / "batch" / "num_segments.npy"), res.num_segments)

    r = _run(common + ["--workload", "map", "--map-chunks", "3", "--map-lo", "1500", "--map-hi", "2500", "--seed", "9",
                       "--dump-outputs", str(tmp_path / "map")])
    assert r.returncode == 0, r.stderr[-2000:]
    chunks = make_map(3, (1500, 2500), features="tarl", seed=9)
    res = api.segment_chunks([c.points for c in chunks], [c.tarl for c in chunks], **kw)
    flat = np.concatenate(res.labels)
    assert np.array_equal(np.load(tmp_path / "map" / "labels.npy"), flat)
    metrics = api.MapPost(chunks, device=cuda_device, min_points=20).merge_and_score(flat)
    for k, v in metrics.items():
        assert abs(np.load(tmp_path / "map" / f"metrics_{k}.npy") - v) <= 1e-12, k
