"""bench.py's command-line contract: the reference arm prints one JSON line with the agreed keys, the product
arm refuses to run without CUDA (no CPU fallback), and --dump-outputs writes the timed step's result (checked
against the oracle on a GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(*args, env=None):
    e = dict(os.environ)
    e.pop("RANK", None); e.pop("WORLD_SIZE", None); e.pop("LOCAL_RANK", None)
    if env:
        e.update(env)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          timeout=600, cwd=ROOT, env=e)


def test_reference_arm_json_line():
    r = run("--impl", "reference", "--queries", "2", "--steps", "1", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout  # exactly one line on stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["unit"] == "UIDs/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["steps"] == 1 and d["warmup"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    assert cb["cores"] == min(2, os.cpu_count())  # the threads that are actually busy: one per query
    e2e = d["e2e"]
    assert e2e["value"] == d["value"] and e2e["unit"] == d["unit"]
    assert e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_reference_arm_same_config_at_n_gpus():
    """At N GPUs the reference arm runs the whole job's N x Q queries on rank 0 and reports the GPU arm's config."""
    r = run("--impl", "reference", "--gpus", "2", "--queries", "2", "--steps", "1", "--warmup", "1",
            env={"RANK": "0", "LOCAL_RANK": "0", "WORLD_SIZE": "2"})
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip())
    assert d["n_gpus"] == 2 and d["config"]["queries_per_gpu"] == 2
    assert "2 GPU(s)" in d["config"]["parallelism"]
    assert d["cpu_baseline"]["cores"] == min(4, os.cpu_count())
    assert "4 queries (2 x 2)" in d["cpu_baseline"]["sample"]


def test_reference_arm_other_ranks_exit_quietly():
    r = run("--impl", "reference", "--gpus", "2", "--queries", "2", "--steps", "1", "--warmup", "0",
            env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_files_and_budget(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench

    offsets = np.array([0, 3, 5], np.uint64)
    uids = np.array([1, 7, 9, 2, (1 << 53) - 1], np.uint64)
    bench.dump_outputs(str(tmp_path / "a"), offsets, uids, 0, 1)
    assert sorted(os.listdir(tmp_path / "a")) == ["offsets.npy", "uids.npy"]
    got = np.load(tmp_path / "a" / "uids.npy")
    assert got.dtype == np.float64 and np.array_equal(got.astype(np.uint64), uids)
    assert np.array_equal(np.load(tmp_path / "a" / "offsets.npy"), offsets.astype(np.float64))

    # over budget: a seeded sample of positions, the same from run to run, within the byte budget
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 2 * (8 * 3 + 16 * 100))
    big = np.arange(10_000, dtype=np.uint64) * 3
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), offsets, big, 1, 2)
    names = ["offsets_rank1.npy", "uids_index_rank1.npy", "uids_rank1.npy"]
    assert sorted(os.listdir(tmp_path / "b")) == names
    assert sum(os.path.getsize(tmp_path / "b" / n) - 128 for n in names) <= bench.DUMP_MAX_BYTES // 2
    idx = np.load(tmp_path / "b" / "uids_index_rank1.npy").astype(np.int64)
    assert idx.size == 100 and np.all(np.diff(idx) > 0)
    assert np.array_equal(np.load(tmp_path / "b" / "uids_rank1.npy"), big[idx].astype(np.float64))
    for n in names:
        assert np.array_equal(np.load(tmp_path / "b" / n), np.load(tmp_path / "c" / n))

    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "d"), offsets, np.array([1 << 53], np.uint64), 0, 1)


def test_steps_must_be_positive():
    r = run("--steps", "0")
    assert r.returncode != 0 and "--steps" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_is_the_timed_result(tmp_path, orc):
    """The dumped arrays are the last timed step's per-query results, equal to the oracle on the seeded inputs."""
    r = run("--steps", "3", "--warmup", "0", "--queries", "2", "--no-e2e", "--no-ops", "--no-dense",
            "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["steps"] == 3 and d["bit_exact"] is True
    sys.path.insert(0, ROOT)
    import bench

    off = np.load(tmp_path / "offsets.npy").astype(np.int64)
    uids = np.load(tmp_path / "uids.npy").astype(np.uint64)
    assert off.size == 3 and off[-1] == uids.size == d["out_uids_per_step"]
    for i, q in enumerate(bench.make_queries(2, 0)):
        assert np.array_equal(uids[off[i]:off[i + 1]], orc.intersect_sorted(q))


def test_product_arm_needs_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = run("--steps", "1", "--warmup", "0", "--queries", "1")
    assert r.returncode != 0
    assert "CUDA" in (r.stderr + r.stdout)
