"""The stored bench lines (profiles/r0N_bench_*.json, written by bench.py on the GPU box) carry every key of the bench
contract; a guard against a bench.py edit that silently drops one.  Round 1 lines: config C2 as a batch, one sequence
per GPU (weak scaling).  Round 2 lines: config C5, the same 4096 pairs split over the GPUs (strong scaling), with the
other configurations as named sub-results."""
import glob
import json
import os
import re
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
        "vs_baseline", "dtype", "data", "config"]


def lines():
    out = []
    for f in sorted(glob.glob(os.path.join(ROOT, "profiles", "r0[12]_bench_*.json"))):
        for ln in open(f):
            if ln.startswith("{"):
                out.append((os.path.basename(f), json.loads(ln)))
    return out


@pytest.mark.parametrize("name,d", lines())
def test_bench_line_has_the_contract_keys(name, d):
    for k in BASE:
        assert k in d, (name, k)
    assert d["metric"] == "ICP scan-pairs/s" and d["unit"] == "pairs/s" and d["higher_is_better"] is True
    assert d["dtype"] == "f64" and d["data"] == "synthetic" and "workload" in d["config"] and d["vs_baseline"] is None
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"])
    assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"]) if d.get("cpu_baseline") else True
    if d.get("impl") == "reference":
        assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
        assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["kind"] in ("port", "reference")
        return
    assert d["value"] > 0 and d["e2e"]["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0
    assert d["gpu_launches"] > 0
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    if name.startswith("r01"):
        pairs = int(re.search(r"C2: (\d+)-pair", d["config"]["workload"]).group(1))   # per GPU (weak scaling)
        assert abs(d["value"] - d["n_gpus"] * pairs / (d["ms_per_step"] * 1e-3)) / d["value"] < 1e-6  # whole-job aggregate
    else:
        pairs = int(re.search(r"C5: batched ICP of (\d+) independent", d["config"]["workload"]).group(1))
        assert d["scaling"] == "strong" and d["workload_stats"]["pairs"] == pairs
        assert abs(d["value"] - pairs / (d["ms_per_step"] * 1e-3)) / d["value"] < 1e-6   # the job is always the same pairs
        assert d["workload_stats"]["status_ok_frac"] == 1.0
        assert 0 < d["e2e"]["h2d_ceiling"]["e2e_frac_of_ceiling"] <= 1.05
        c4 = d["c4_loop_closure"]
        assert c4["n_gpus"] == d["n_gpus"] and c4["ms_per_detect"] > 0 and c4["top10_that_are_true_revisits"] >= 3
        if d["n_gpus"] == 1:
            assert d["c2_streaming"]["ms_per_frame_mean"] > 0 and d["c2_batch"]["pairs_per_s"] > 0
            assert d["c3_knn_normals"]["knn_plus_normals_queries_per_s"] > 0
            assert d["roofline"]["issue"] is None or 0 < d["roofline"]["issue"]["frac"] < 1
    if d["n_gpus"] == 1:
        r = d["roofline"]
        assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["bound"] in ("hbm", "tensor")
        assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
        assert d["cpu_baseline"]["cores"] >= 1


def test_dump_outputs_files(tmp_path, monkeypatch):
    """bench.py --dump-outputs: one float64 .npy per result field, only values the caller received (finite: nothing from
    past a pair's history length), rows of all files aligned, and above the size cap the same seeded sample of pairs on
    every run, the cap shared by the ranks of the job."""
    import numpy as np
    import slam_b200
    monkeypatch.syspath_prepend(ROOT)
    import bench

    def batch(n, seed):
        rng = np.random.default_rng(seed)
        r = np.zeros(n, dtype=slam_b200.ICP_DTYPE)
        r["transformation"] = rng.normal(size=(n, 16))
        r["final_error"] = rng.uniform(size=n)
        r["converged"] = rng.integers(0, 2, n)
        r["status"] = rng.integers(0, 7, n)
        r["history_len"] = rng.integers(1, 10, n)
        r["num_iterations"] = r["history_len"] + 100
        h = rng.uniform(size=r["error_history"].shape)
        h[np.arange(h.shape[1]) >= r["history_len"][:, None]] = np.nan     # slots past the history must not be written
        r["error_history"] = h
        return slam_b200.ICPResultBatch(r)

    recs = [batch(5, 0), batch(3, 1)]
    ids = np.arange(8) * 64 + 5
    fields = ("pair_id", "transformation", "final_error", "num_iterations", "converged", "status", "history_len",
              "error_history")

    def load(d):
        return {f: np.load(tmp_path / d / (f + ".npy")) for f in fields}

    def rows_match(got, want_ids):
        """every row k of every file is the result of pair got["pair_id"][k]"""
        want = {int(i): r for i, r in zip(ids, (x for b in recs for x in b))}
        hist = np.split(got["error_history"], np.cumsum(got["history_len"].astype(np.int64))[:-1])
        assert np.array_equal(got["pair_id"], want_ids) and len(hist) == len(want_ids)
        for k, i in enumerate(want_ids):
            w = want[int(i)]
            assert np.array_equal(got["transformation"][k], w.transformation) and got["final_error"][k] == w.final_error
            assert (got["num_iterations"][k], got["converged"][k], got["status"][k]) == (w.num_iterations, w.converged,
                                                                                         w.status)
            assert got["history_len"][k] == len(w.error_history) and np.array_equal(hist[k], w.error_history)

    bench.dump_outputs(str(tmp_path / "all"), ids, recs)
    assert sorted(os.listdir(tmp_path / "all")) == sorted(f + ".npy" for f in fields)
    got = load("all")
    for f, a in got.items():
        assert a.dtype == np.float64 and np.all(np.isfinite(a)), f
    rows_match(got, ids)

    monkeypatch.setattr(bench, "DUMP_BYTES", 3 * 151 * 8)      # room for three of the eight pairs
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), ids, recs)
    s1 = load("s1")
    assert len(s1["pair_id"]) == 3 and np.array_equal(s1["pair_id"], load("s2")["pair_id"])
    assert sum(a.nbytes for a in s1.values()) <= bench.DUMP_BYTES
    rows_match(s1, s1["pair_id"])

    monkeypatch.setattr(bench, "DUMP_BYTES", 4 * 151 * 8)      # two ranks: two pairs each
    for r in (0, 1):
        bench.dump_outputs(str(tmp_path / "ranks"), ids, recs, rank=r, world=2)
    assert sorted(os.listdir(tmp_path / "ranks")) == sorted(f + s + ".npy" for f in fields for s in ("_rank0", "_rank1"))
    assert sum(np.load(tmp_path / "ranks" / f).nbytes for f in os.listdir(tmp_path / "ranks")) <= bench.DUMP_BYTES
