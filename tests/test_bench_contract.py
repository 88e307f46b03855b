"""bench.py's output contract on CPU: the reference arm (no GPU needed) prints exactly one JSON line with the
keys the driver reads, for every workload; the b200 arm refuses to run without a CUDA device."""
import json
import os
import subprocess
import sys

import pytest

import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e", "gpu_launches"}


def _run(args, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          timeout=timeout, cwd=ROOT)


@pytest.mark.parametrize("workload,extra", [(None, ["--scale", "0.01"]), ("contig5m", []),
                                            ("train500m", ["--scale", "0.001"]), ("reads100", ["--scale", "0.01"]),
                                            ("reads400", ["--scale", "0.05"]),
                                            ("simplescore", ["--scale", "0.004"])])
def test_reference_arm_prints_one_json_line(workload, extra):
    wl = ["--workload", workload] if workload else []  # no --workload: the default (reads100)
    r = _run(["--impl", "reference", *wl, "--steps", "1", "--warmup", "0", *extra])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert REQUIRED <= set(d), REQUIRED - set(d)
    assert d["impl"] == "reference" and d["value"] > 0 and d["gpu_launches"] == 0
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    if workload is None:
        assert d["config"]["workload"].startswith("reads100")
    assert isinstance(d["config"].get("workload"), str) and "model" not in {k for k in d["config"] if k == "model_family"}


def test_b200_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = _run(["--steps", "1", "--warmup", "1"])
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    return b


def test_dump_of_scoring_outputs_is_exact_seeded_and_bounded(tmp_path, monkeypatch):
    """--dump-outputs: ORF table and start lists written as float64 tables that restate every field exactly; the whole
    output when it fits the budget, else the same seeded sample of ORFs with their complete start lists on every run."""
    import numpy as np
    b = _bench_module()
    rng = np.random.default_rng(1)
    n_seqs, n_orfs = 50, 400
    ooff = np.concatenate([[0], np.sort(rng.integers(0, n_orfs, n_seqs - 1)), [n_orfs]]).astype(np.int64)
    soff = np.concatenate([[0], np.cumsum(rng.integers(0, 9, n_orfs))]).astype(np.int64)
    orfs = np.zeros(n_orfs, O.ORF_DTYPE)
    for f in O.ORF_DTYPE.names:
        orfs[f] = rng.integers(-5, 1 << 20, n_orfs)
    starts = np.zeros(int(soff[-1]), O.START_DTYPE)
    for f in ("j", "pos", "which", "truncated", "first", "n_err"):
        starts[f] = rng.integers(-3, 1 << 20, len(starts))
    starts["score"] = rng.normal(size=len(starts))
    starts["err_pos"] = rng.integers(0, 400, (len(starts), 2))
    starts["err_type"] = rng.integers(0, 4, (len(starts), 2))

    full = b.scoring_outputs(orfs, ooff, starts, soff)
    assert full["counts"].tolist() == [n_seqs, n_orfs, len(starts)] and len(full["orfs"]) == n_orfs
    assert (full["starts"][:, 3].view(np.uint64) == starts["score"].view(np.uint64)).all()
    assert full["starts"][:, 8:10].tolist() == starts["err_pos"].tolist()
    assert full["orfs"][:, 1].tolist() == np.repeat(np.arange(n_seqs), np.diff(ooff)).tolist()

    monkeypatch.setattr(b, "DUMP_BYTES", 8 * (3 + n_seqs + n_orfs) + 8 * (6 * 60 + 12 * 300))
    part = b.scoring_outputs(orfs, ooff, starts, soff)
    again = b.scoring_outputs(orfs.copy(), ooff.copy(), starts.copy(), soff.copy())
    assert 0 < len(part["orfs"]) < n_orfs and all((part[k] == again[k]).all() for k in part)
    assert sum(a.nbytes for a in part.values()) <= b.DUMP_BYTES
    for row in part["orfs"]:
        i = int(row[0])
        mine = part["starts"][part["starts"][:, 0] == i]
        assert mine[:, 1].tolist() == starts["j"][soff[i]:soff[i + 1]].tolist()
        assert row[2:].tolist() == [orfs[f][i] for f in O.ORF_DTYPE.names]
    b.dump_outputs(str(tmp_path / "d"), part)
    assert (np.load(tmp_path / "d" / "starts.npy") == part["starts"]).all()
    assert {np.load(p).dtype for p in (tmp_path / "d").iterdir()} == {np.dtype(np.float64)}


def test_reads100_job_order_balances_clusters_over_ranks():
    """The batches a rank is dealt (b = rank + world * i) must have the same mean cluster index -- i.e. the same mean GC
    content, which sets the ORF density and so the cost of a step -- at every world size, and every cluster appears twice
    in the job list (BASELINE configs[4]: 16 clusters x 625 000 reads = two batches each)."""
    b = _bench_module()
    n_batches = b.READS100_CLUSTERS * (b.READS100_PER_CLUSTER // b.READS100_BATCH)
    clusters = [b.reads100_cluster_of_batch(i) for i in range(n_batches)]
    assert sorted(clusters) == sorted(list(range(b.READS100_CLUSTERS)) * 2)
    for world in (1, 2, 4, 8):
        for rank in range(world):
            mine = [b.reads100_cluster_of_batch((rank + world * i) % n_batches) for i in range(b.MAX_RESIDENT_BATCHES)]
            assert sum(mine) * 2 == (b.READS100_CLUSTERS - 1) * len(mine), (world, rank, mine)
