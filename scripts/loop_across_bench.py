#!/usr/bin/env python
"""Loop closures across detectors: sb_loop_detect_across / sb_loop_candidates_across against the workaround they
replace, sb_loop_detect_batch / sb_loop_candidates_batch on a scratch detector that holds copies of the other
detectors' entries followed by the query entries (frame 2^30, frame_gap 1: the same results, bit for bit).

The database is config C4's 4000 keyframes (loop_sequence_bench.py: build_clouds; 3.3 laps of the C2 loop, so the
parts revisit each other) split into 4 detectors of 1000 consecutive keyframes.  Cases, per detector config
(loop_sequence_bench.py: CONFIGS, frame_gap unused here), each with a warm-up, host clocks around synchronised work and
`reps` alternated repetitions (the minimum is reported):
  (a) fleet step: 100 calls, each with one query per detector (entry 10 t of every detector in call t); the
      workaround answers a call with one detect_batch per query detector.  Under the stress config every query walks
      thousands of failing candidates (about 1.7 s per call), so (a) runs its first 10 calls there;
  (b) offline merge: detector 0's node-schedule entries (60, 70, ..., 990) against the other three in one call;
  (c) search and selection alone: candidates_across for (b)'s queries against candidates_batch on (b)'s scratch
      detector, the same number of (query, entry) pairs.
The scratch detectors are built untimed; their build time and the bytes they copy are reported as the workaround's
copy cost.  A torch.profiler pass over (a) gives the kernel time of the squared-sum pre-pass (k_sc_sq_across) against
the search and selection kernels.  Writes profiles/loop_across_bench.json and prints it.

    python scripts/loop_across_bench.py [--reps 3] [--out profiles/loop_across_bench.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from loop_sequence_bench import CONFIGS, OPS_PER_PAIR, build_clouds, gpu_info  # noqa: E402

N_DB, PARTS = 4000, 4
CALLS = dict(node=100, c4_stress=10)
Q_FRAME = 1 << 30


def keyed(loops):
    return [[(r["match_frame"], r["icp_fitness"], r["transform"].tobytes()) for r in q] for q in loops]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "loop_across_bench.json"))
    args = ap.parse_args()
    import torch
    import oracle_lib
    import slam_b200
    if not torch.cuda.is_available():
        raise SystemExit("loop_across_bench.py measures the GPU: no CUDA device")
    eng = slam_b200.Engine(0)
    syn = oracle_lib.Synth()
    t_start = time.perf_counter()
    log = lambda *a: print(f"[{time.perf_counter() - t_start:7.1f} s]", *a, flush=True)
    xyz, off = build_clouds(eng, syn, torch, N_DB)
    log("keyframes built")
    per = N_DB // PARTS
    part = [(xyz[off[p * per]:off[(p + 1) * per]], off[p * per:(p + 1) * per + 1] - off[p * per]) for p in range(PARTS)]
    frames = [np.arange(p * per, (p + 1) * per) for p in range(PARTS)]
    descs = np.stack([eng.sc_compute(xyz[off[f]:off[f + 1]]) for f in range(N_DB)])
    merge = [(0, e) for e in range(per) if e % 10 == 0 and e > 50]
    out = dict(workload=f"{N_DB} C4 keyframes (64-beam, voxel 0.5) in {PARTS} detectors of {per}; (a) {CALLS} calls x "
                        f"{PARTS} queries, (b)/(c) {len(merge)} queries of detector 0 against the other three",
               n_db=N_DB, detectors=PARTS)
    out.update(gpu_info())

    def scratch(cfg, qd, entries):
        """other detectors' clouds and descriptors, then the query entries: (detector, first query, bytes copied)"""
        det = slam_b200.LoopClosureDetector(eng, **dict(cfg, frame_gap=1))
        rows = 0
        for d in range(PARTS):
            if d != qd:
                det.addFrames(part[d][0], part[d][1], frames[d], descs[d * per:(d + 1) * per])
                rows += len(part[d][0])
        first = det.size()
        qi = [qd * per + e for e in entries]
        qx = [xyz[off[f]:off[f + 1]] for f in qi]
        qo = np.zeros(len(qi) + 1, dtype=np.int64)
        qo[1:] = np.cumsum([len(c) for c in qx])
        det.addFrames(np.vstack(qx), qo, [Q_FRAME] * len(qi), descs[qi])
        return det, first, rows * 24 + (PARTS - 1) * per * 9600

    def clock(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0, r

    for name, base in CONFIGS.items():
        cfg = {k: v for k, v in base.items() if k != "frame_gap"}
        calls = CALLS[name]
        fleet = [[(d, (10 * t) % per) for d in range(PARTS)] for t in range(calls)]
        dbs = []
        for d in range(PARTS):
            det = slam_b200.LoopClosureDetector(eng, frame_gap=base["frame_gap"], **cfg)
            det.addFrames(part[d][0], part[d][1], frames[d], descs[d * per:(d + 1) * per])
            dbs.append(det)
        t0 = time.perf_counter()
        fl_scr = [scratch(cfg, d, [(10 * t) % per for t in range(calls)]) for d in range(PARTS)]
        mg_scr = scratch(cfg, 0, [e for _, e in merge])
        t_build = time.perf_counter() - t0
        log(name, "scratch detectors built")
        copy_bytes = sum(s[2] for s in fl_scr) + mg_scr[2]

        def fleet_across():
            return [slam_b200.detect_across(dbs, q) for q in fleet]

        def fleet_scratch():
            return [[fl_scr[d][0].detect_batch([fl_scr[d][1] + t])[0] for d in range(PARTS)] for t in range(calls)]

        def merge_across():
            return slam_b200.detect_across(dbs, merge)

        mq = list(range(mg_scr[1], mg_scr[1] + len(merge)))

        def merge_scratch():
            return mg_scr[0].detect_batch(mq)

        def cand_across():
            return slam_b200.candidates_across(dbs, merge)

        def cand_scratch():
            return mg_scr[0].candidates_batch(mq)

        cases = dict(a=(fleet_across, fleet_scratch), b=(merge_across, merge_scratch), c=(cand_across, cand_scratch))
        times = {k: ([], []) for k in cases}
        res = {}
        for k, (fa, fs) in cases.items():   # warm-up
            fa() if k != "a" else [slam_b200.detect_across(dbs, q) for q in fleet[:3]]
            fs() if k != "a" else [fl_scr[d][0].detect_batch([fl_scr[d][1]]) for d in range(PARTS)]
        for _ in range(args.reps):
            for k, (fa, fs) in cases.items():
                ta, ra = clock(fa)
                ts, rs = clock(fs)
                times[k][0].append(ta)
                times[k][1].append(ts)
                res[k] = (ra, rs)
                log(name, k, f"across {ta * 1e3:.1f} ms, scratch {ts * 1e3:.1f} ms")
        # the same loops, bit for bit
        fa_, fs_ = res["a"]
        assert [keyed(x) for x in fa_] == [keyed(x) for x in fs_], f"{name}: fleet results differ"
        assert keyed(res["b"][0]) == keyed(res["b"][1]), f"{name}: merge results differ"
        (la, ca), (ls, cs) = res["c"]
        assert np.array_equal(ca, cs) and all(np.array_equal(x[0], y[0]) for x, y in zip(la, ls))
        # kernel times of one pass of (a)
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fleet_across()
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.key_averages():
            for kname in ("k_sc_sq_across", "k_sc_distance_across", "k_loop_select_across"):
                if kname in ev.key:
                    kern[kname] = kern.get(kname, 0.0) + ev.device_time_total / 1e3   # ms
        a_ms, as_ms = min(times["a"][0]) * 1e3, min(times["a"][1]) * 1e3
        b_ms, bs_ms = min(times["b"][0]) * 1e3, min(times["b"][1]) * 1e3
        c_s, cs_s = min(times["c"][0]), min(times["c"][1])
        pairs = len(merge) * (PARTS - 1) * per
        ld = PARTS * ((per + 7) // 8 * 8)
        ops = pairs * OPS_PER_PAIR + (ld + len(merge)) * 60 * 2400
        out[name] = dict(
            config=cfg, a_calls=calls,
            a_fleet_ms_per_call=a_ms / calls, a_scratch_ms_per_call=as_ms / calls, a_ratio_across_over_scratch=a_ms / as_ms,
            a_kernel_ms_per_call={k: v / calls for k, v in kern.items()},
            a_sq_share_of_call=kern.get("k_sc_sq_across", 0.0) / a_ms,
            a_accepted=sum(len(x) for call in fa_ for x in call),
            b_merge_ms=b_ms, b_scratch_ms=bs_ms, b_ratio_across_over_scratch=b_ms / bs_ms,
            b_accepted=sum(len(x) for x in res["b"][0]),
            c_pairs=pairs, c_across_ms=c_s * 1e3, c_scratch_ms=cs_s * 1e3,
            c_across_pairs_per_s=pairs / c_s, c_scratch_pairs_per_s=pairs / cs_s, c_rate_ratio=cs_s / c_s,
            c_across_fp64_ops_per_s=ops / c_s,
            scratch_build_s=t_build, scratch_copy_bytes=copy_bytes)
        for s in fl_scr + [mg_scr]:
            s[0].close()
        for d in dbs:
            d.close()
        print(name, json.dumps(out[name]), flush=True)
    eng.close()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
