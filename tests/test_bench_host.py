"""CPU checks of bench.py's host-side logic (no GPU, no timing): the training-sample layout both arms share, the
k-means seeding rule, the reference arm's host-built index on a tiny workload, the --dump-outputs writer and the
argument checks, and that the committed scan-traffic stamp belongs to the committed kernel sources (otherwise the
bench line would carry no `roofline.traffic`)."""
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import oracle as O  # noqa: E402
from fabstir_vectordb_b200 import synth  # noqa: E402


def test_training_sample_is_blocks_of_64_rows():
    rows = bench.train_sample_rows(1_000_000, 65536)
    assert rows.shape == (65536,)
    stride = 1_000_000 // 65536
    assert rows[:64].tolist() == list(range(64))
    assert rows[64] == 64 * stride and rows[65] == 64 * stride + 1
    assert rows.max() < 1_000_000 and len(set(rows.tolist())) == 65536


def test_kmeans_seeds_come_from_distinct_mixture_components():
    nlist, n_train, n_total = 1024, 65536, 1_000_000
    seeds = bench.train_sample_rows(n_total, n_train)[bench.init_rows_of_sample(nlist, n_train)]
    comps = seeds % np.uint64(bench.n_comp_for(nlist))
    assert len(set(comps.tolist())) == nlist          # the clumped seeding of early round 1 gave nlist / 16


def test_nprobe_and_workload_names():
    assert bench.nprobe_for(1) == 32 and bench.nprobe_for(8) == 32
    assert "nlist=8192" in bench.workload_name(8) and "8000000x384" in bench.workload_name(8)


def test_reference_arm_host_index_small(monkeypatch):
    """host_index (numpy generator + the oracle's k-means and assignment, no product library) on a tiny workload:
    the lists partition the rows, every row sits in the list of its nearest centroid, and a search finds a
    database row from a slightly perturbed copy of it."""
    monkeypatch.setattr(bench, "TRAIN_ITERS", 4)
    n_total, nlist = 4096, 16
    n_comp = bench.n_comp_for(nlist)
    ivf, x = bench.host_index(n_total, nlist, n_comp, lambda m: None)
    assert x.shape == (n_total, bench.DIM)
    assert np.array_equal(x[:8], synth.rows(0, 8, bench.DIM, n_comp, bench.SIGMA, bench.SEED))
    assert sum(ivf.list_len(l) for l in range(nlist)) == n_total
    assert np.array_equal(ivf.assign, O.assign(x, ivf.centroids))
    q = bench.host_queries(8, n_total, n_comp, 0)
    ids, dist, cnt = O.hybrid_batch_search(ivf, None, None, q, 5, nlist, tiers=2)
    base = synth.query_base_rows(0, 8, n_total, bench.SEED_Q)
    assert (cnt == 5).all() and ids[:, 0].tolist() == base.tolist()


def test_dump_outputs_writes_float_arrays(tmp_path):
    """--dump-outputs: ids / distances / counts of a step as .npy in float64 / float32; the id of an empty slot
    (0xFFFFFFFF) survives exactly."""
    import torch
    ids = torch.tensor([[3, 7], [999_999, -1]], dtype=torch.int32)
    dist = torch.tensor([[0.5, 1.25], [0.75, float("inf")]], dtype=torch.float32)
    cnt = torch.tensor([2, 1], dtype=torch.int32)
    out = tmp_path / "out"
    bench.dump_outputs(str(out), ids, dist, cnt)
    assert sorted(os.listdir(out)) == ["counts.npy", "distances.npy", "ids.npy"]
    got = {n: np.load(out / f"{n}.npy") for n in ("ids", "distances", "counts")}
    assert got["ids"].dtype == np.float64 and got["ids"].tolist() == [[3, 7], [999_999, 0xFFFFFFFF]]
    assert got["distances"].dtype == np.float32 and np.array_equal(got["distances"], dist.numpy())
    assert got["counts"].dtype == np.float64 and got["counts"].tolist() == [2, 1]


def test_bench_arguments_are_checked_before_any_work(monkeypatch):
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"],
                 ["--config", "cfg3", "--dump-outputs", "x"]):
        monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
        with pytest.raises(SystemExit) as e:
            bench.main()
        assert e.value.code == 2


def test_committed_scan_traffic_stamp_matches_the_kernel_sources():
    with open(os.path.join(ROOT, "profiles", "scan_traffic.json")) as fh:
        tj = json.load(fh)
    assert tj["source_digest"] == bench.scan_source_digest(), \
        "the scan kernels changed after the ncu capture: re-capture (scripts/gpu_evidence.sh + summarize_ncu.py --traffic)"
    assert 1.0e9 < tj["dram_bytes_per_launch"] < 2.0e9
