#!/usr/bin/env python
"""Loop-closure detection over a whole recorded sequence: per-frame sb_loop_detect against one sb_loop_detect_batch.

The database is config C4's (bench.py:sub_c4): 4000 keyframes on the 1.2 km C2 loop (3.3 laps: true revisits),
64-beam scans voxel-downsampled at 0.5 m.  The queries are the node's schedule (slam_node.cpp:159:
frame % 10 == 0 && frame > 50): entries 60, 70, ..., 3990.  Two detector configs: the node's (slam_node.cpp:77-81:
gap 50, threshold 0.2, fitness 0.3, 3 candidates) and C4's stress setting (threshold 1e300, 10 candidates).

Per config, timed with host clocks around synchronised work after a warm-up:
  (a) one sb_loop_detect per query on a detector grown entry by entry (only the detect calls are timed);
  (b) one sb_loop_detect_batch over all queries (database bulk-loaded with sb_loop_add_frames);
  (c) sb_loop_candidates_batch alone: the many-query search + selection.
(a) and (b) must accept the same loops.  Prints one JSON line.

    python scripts/loop_sequence_bench.py [--n-db 4000] [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import SENSOR, VOXEL, make_poses, make_world  # noqa: E402  (also puts python/ and tests/ on sys.path)

# fp64 DMUL + DADD per (query, entry) pair of the many-query search: sum_ab only, 1200 cells x 60 shifts
OPS_PER_PAIR = 2 * 1200 * 60
# the one-query search (k_sc_distance) also forms sum_aa and sum_bb per pair and shift
OPS_PER_PAIR_SINGLE = 3 * 2 * 1200 * 60
# data-sheet fp64 rate of one HGX B200 GPU (37 TFLOP/s with an FMA counted as two): DMUL / DADD per second
DATASHEET_FP64_OPS = 37e12 / 2

CONFIGS = {
    "node": dict(frame_gap=50, sc_distance_threshold=0.2, icp_fitness_threshold=0.3, max_candidates=3),
    "c4_stress": dict(frame_gap=50, sc_distance_threshold=1e300, icp_fitness_threshold=0.3, max_candidates=10),
}


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    first = out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else ""
    parts = [p.strip() for p in first.split(",")] if first else []
    return dict(zip(["gpu_name", "power_limit", "max_sm_clock"], parts)) if len(parts) == 3 else {"gpu": "unknown"}


def build_clouds(eng, syn, torch, n_db):
    """Voxel-downsampled C4 keyframes (bench.py:sub_c4), as one host CSR array."""
    world = make_world(syn)
    poses = make_poses(syn, n_db + 1)
    rays = SENSOR["beams"] * SENSOR["azimuth_steps"]
    chunk = 250
    d_raw = torch.empty(chunk * rays * 3, dtype=torch.float64, device="cuda")
    parts, offs = [], [np.zeros(1, dtype=np.int64)]
    for c0 in range(0, n_db, chunk):
        c1 = min(n_db, c0 + chunk)
        off = eng.synth_scans_dev(SENSOR, world, poses[c0:c1], 7000 + c0, d_raw.data_ptr())
        h = d_raw[:int(off[-1]) * 3].cpu().numpy().reshape(-1, 3)
        ds, doff = eng.voxel_downsample_batch(h, off, VOXEL)
        parts.append(ds)
        offs.append(doff[1:] + offs[-1][-1])
    del d_raw
    return np.vstack(parts), np.concatenate(offs)


def keyed(loops):
    return [(r["query_frame"], r["match_frame"], r["icp_fitness"]) for r in loops]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-db", type=int, default=4000)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    import oracle_lib
    import slam_b200
    if not torch.cuda.is_available():
        raise SystemExit("loop_sequence_bench.py measures the GPU: no CUDA device")
    eng = slam_b200.Engine(0)
    syn = oracle_lib.Synth()
    n_db = args.n_db
    xyz, off = build_clouds(eng, syn, torch, n_db)
    frames = np.arange(n_db)
    queries = [f for f in range(n_db) if f % 10 == 0 and f > 50]
    causal_pairs = int(sum(queries))   # query q sees the entries 0..q-1
    out = dict(workload=f"{n_db} C4 keyframes (64-beam, voxel {VOXEL}), {len(queries)} queries on the node's schedule "
                        "(entries 60, 70, ...)", n_db=n_db, n_queries=len(queries), causal_pairs=causal_pairs)
    out.update(gpu_info())
    for name, cfg in CONFIGS.items():
        # (a) per-frame: grow entry by entry, time only the detect calls
        seq = slam_b200.LoopClosureDetector(eng, **cfg)
        seq.reserve(n_db + 1, int(off[-1]) + 1)
        a_loops, t_a = [], 0.0
        for f in range(n_db):
            seq.addFrame(xyz[off[f]:off[f + 1]], int(frames[f]))
            if f in (queries[0], queries[1]):   # warm-up of the detect path
                seq.detect()
            if f % 10 == 0 and f > 50:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                a_loops.append(seq.detect())
                t_a += time.perf_counter() - t0
        seq.close()
        # (b) one batch call on a bulk-loaded detector
        bat = slam_b200.LoopClosureDetector(eng, **cfg)
        bat.reserve(n_db + 1, int(off[-1]) + 1)
        t0 = time.perf_counter()
        bat.addFrames(xyz, off, frames)
        t_add = time.perf_counter() - t0
        bat.detect_batch(queries[:20])   # warm-up
        t_b = []
        for _ in range(args.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            b_loops = bat.detect_batch(queries)
            t_b.append(time.perf_counter() - t0)
        assert [keyed(x) for x in a_loops] == [keyed(x) for x in b_loops], f"{name}: (a) and (b) disagree"
        # (c) the search alone, and the one-query search on the full database for comparison
        bat.candidates_batch(queries)
        t_c = []
        for _ in range(args.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            bat.candidates_batch(queries)
            t_c.append(time.perf_counter() - t0)
        bat.candidates_local(capacity=16)
        t0 = time.perf_counter()
        for _ in range(10):
            bat.candidates_local(capacity=16)
        t_single = (time.perf_counter() - t0) / 10
        bat.close()
        tb, tc = min(t_b), min(t_c)
        ops = causal_pairs * OPS_PER_PAIR + (queries[-1] + 1) * 60 * 2400
        out[name] = dict(
            config=cfg,
            a_ms_total=t_a * 1e3, a_ms_per_query=t_a * 1e3 / len(queries),
            b_ms_total=tb * 1e3, b_ms_per_query=tb * 1e3 / len(queries), speedup_b_over_a=t_a / tb,
            add_frames_ms=t_add * 1e3,
            c_ms=tc * 1e3, c_pairs_per_s=causal_pairs / tc,
            single_query_pairs_per_s=(n_db - 1) / t_single, search_rate_ratio=causal_pairs / tc / ((n_db - 1) / t_single),
            c_fp64_ops_per_s=ops / tc, c_fraction_of_datasheet_fp64=ops / tc / DATASHEET_FP64_OPS,
            datasheet_pairs_per_s_bound=DATASHEET_FP64_OPS / OPS_PER_PAIR,
            queries_with_loops=sum(1 for x in b_loops if x), accepted_loops=sum(len(x) for x in b_loops))
    eng.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
