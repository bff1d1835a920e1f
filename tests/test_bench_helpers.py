"""Host-side helpers of bench.py (no GPU): deterministic data generation, recall metric, peak lookup."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_gen_unit_rows_deterministic_and_unit_norm():
    import torch

    import bench
    gen = lambda seed, dist, chunk=128: bench.gen_unit_rows_device(torch, seed, 300, 64, dist, chunk=chunk, device="cpu").numpy()
    a, b = gen(123, "latent"), gen(123, "latent")
    assert np.array_equal(a, b) and a.dtype == np.float32 and a.shape == (300, 64)
    np.testing.assert_allclose(np.linalg.norm(a, axis=1), 1.0, rtol=1e-5)
    assert not np.array_equal(a, gen(124, "latent"))
    iid = gen(123, "iid")
    # the latent model has neighbourhood structure: pairwise similarities spread far wider than for i.i.d. rows
    assert (a @ a.T)[np.triu_indices(300, 1)].std() > 1.4 * (iid @ iid.T)[np.triu_indices(300, 1)].std()


def test_recall_at_k_matches_accuracy_metrics_semantics():
    import bench
    # jvector-examples/.../util/AccuracyMetrics.java:38-50: |top-k found ∩ top-k truth| / (queries * k)
    found = np.array([[1, 2, 3, -1], [9, 8, 7, 6]])
    truth = np.array([[3, 2, 5, 6], [6, 7, 8, 9]])
    assert bench.recall_at_k(found, truth, 4) == (2 + 4) / 8.0
    assert bench.recall_at_k(found, truth, 2) == (1 + 0) / 4.0


def test_dump_outputs_dtypes_and_seeded_row_sample(tmp_path, monkeypatch):
    import bench
    nodes = np.arange(1000 * 10, dtype=np.int32).reshape(1000, 10)
    scores = np.linspace(0, 1, 10000, dtype=np.float32).reshape(1000, 10)
    bench.dump_outputs(str(tmp_path / "all"), {"c2_nodes": nodes, "c2_scores": scores})
    assert np.load(tmp_path / "all" / "c2_nodes.npy").dtype == np.float64
    assert np.array_equal(np.load(tmp_path / "all" / "c2_nodes.npy"), nodes) and np.array_equal(np.load(tmp_path / "all" / "c2_scores.npy"), scores)
    # over the cap: the same seeded rows of every array, within the cap, and the same rows run after run
    monkeypatch.setattr(bench, "DUMP_BYTES", 8192)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"c2_nodes": nodes, "c2_scores": scores})
    n, s = np.load(tmp_path / "a" / "c2_nodes.npy"), np.load(tmp_path / "a" / "c2_scores.npy")
    assert n.dtype == np.float64 and s.dtype == np.float32 and 0 < len(n) == len(s) and n.nbytes + s.nbytes <= 8192
    rows = (n[:, 0] // 10).astype(np.int64)
    assert np.array_equal(nodes[rows], n) and np.array_equal(scores[rows], s)
    assert np.array_equal(np.load(tmp_path / "b" / "c2_nodes.npy"), n)


def test_measured_peaks_and_traffic_table():
    import bench
    peak, src = bench.measured_peaks()
    assert peak > 1000
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        assert peak == float(json.load(open(p))["hbm_gbs"]) and src.startswith("measured")
    assert bench.NCU_TRAFFIC[("c2", 1_000_000, 10_000, 100)] > 9e10
