#!/usr/bin/env python
"""bench.py — headline benchmark: ICP scan-pairs/s on BASELINE.json configs[4] (SURVEY.md 8d, C5): 4096 INDEPENDENT
synthetic scan pairs (64-beam, ~119k points per scan, voxel 0.5 m, normals k = 20, ICP 50 it / 1e-6), pair i in scene
seed 100 + i mod 64 with a relative pose drawn U(0.5, 1.5) m x U(-0.1, 0.1) m x U(-0.02, 0.02) rad from seed 1000 + i.

A step = one pass of the whole front end over ALL pairs: per pair two voxel grids, one index + normals (target), one
index (source), point-to-plane ICP; results on the host.
  value : pairs/s with the raw scans already resident in HBM (sb_register_batch_dev), CUDA-event timed.
  e2e   : the same through sb_register_batch_f32 with HOST (pinned) float32 records: H2D of every scan + D2H of the
          results inside the timed region.
  N > 1 : STRONG scaling — the same 4096 pairs, pair p on rank p % N (python/sharding.py), every rank registers its
          share, one NCCL all-gather of the result records per step; value = 4096 / max-over-ranks time.
Named sub-results (rank 0, N = 1 only unless noted): c2_batch (1000 consecutive frame pairs of one sequence as ONE
batch), c2_streaming (one frame per call, the way slam_node drives the API: ms/frame mean / p50 / p99), c3_knn_normals
(128 beams, voxel 0.2, k = 10), c4_loop_closure (4000-keyframe Scan Context search + ICP verification of the top 10;
at N > 1 the database is sharded over the ranks and the number is ms per detect() across the job).
--impl reference times the CPU oracle (the reference's algorithm restated: its sources build here only over an Eigen
stand-in) on all host cores over a bounded sample of the same pairs, same per-pair work.
--dump-outputs DIR writes the results of the last timed step as DIR/<name>.npy (see dump_outputs).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "lidar-slam-from-scratch_b200", "python"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

SENSOR = dict(beams=64, azimuth_steps=1875, elev_top_deg=2.0, elev_bot_deg=-24.8, max_range=120.0, noise_sigma=0.02,
              sensor_height=1.73)
VOXEL = 0.5
LOOP_LEN_M = 1200.0
RADIUS = LOOP_LEN_M / (2.0 * np.pi)
C5_PAIRS = 4096
C5_SCENES = 64


# ---------------------------------------------------------------------------------------------------------------
# workloads
# ---------------------------------------------------------------------------------------------------------------
def make_world(synth):
    """Box city around a 1.2 km circular loop (SURVEY.md 8d, C2)."""
    half = RADIUS + 100.0
    n_boxes = int(400 * (2 * half) ** 2 / 180.0 ** 2)
    return synth.scene(11, n_boxes=n_boxes, half_extent=half, path_kind=1, radius=RADIUS, corridor_half=6.0)


def make_poses(synth, n_scans, step_m=1.0):
    return np.stack([synth.pose(1, RADIUS, i * step_m) for i in range(n_scans)])


def c5_pair(i):
    """Pair i of config C5: (scene index, index within the scene, target pose, source pose, relative pose)."""
    s, j = i % C5_SCENES, i // C5_SCENES
    rng = np.random.default_rng(1000 + i)
    rel = np.array([rng.uniform(0.5, 1.5), rng.uniform(-0.1, 0.1), rng.uniform(-0.02, 0.02)])
    base = np.array([-40.0 + 1.25 * j, 0.0, 0.0])     # along the scene's free corridor: 64 different places per scene
    return s, j, base, base + rel, rel


def c5_scene(synth, s):
    return synth.scene(100 + s, n_boxes=400)            # SURVEY.md 8d C1/C5 scene recipe, seed 100 + i mod 64


def c5_noise_seed(s):
    return 200000 + 1000 * s                            # scan 2j (target) / 2j + 1 (source) of the scene add their index


def c5_pairs_of_rank(n_pairs, rank, world):
    """Round-robin ownership (sharding.shard_units), listed scene by scene: the order the scans are generated in."""
    import sharding
    ids = sharding.shard_units(n_pairs, rank, world)
    return np.array(sorted(ids, key=lambda i: (i % C5_SCENES, i // C5_SCENES)), dtype=np.int64)


def c5_generate(eng, synth, pair_ids, d_raw_ptr, rays):
    """Raycasts the scans of `pair_ids` (grouped by scene) into device memory: rows of scan 2l (target of local pair l)
    and 2l + 1 (its source).  Returns the CSR offsets of the 2 * len(pair_ids) scans."""
    off = [0]
    l = 0
    while l < len(pair_ids):
        s = int(pair_ids[l]) % C5_SCENES
        m = l
        poses = []
        while m < len(pair_ids) and int(pair_ids[m]) % C5_SCENES == s:
            _, j, tgt, src, _ = c5_pair(int(pair_ids[m]))
            assert j == m - l, "ranks own whole scenes (world divides 64) so that scan seeds do not depend on the sharding"
            poses += [tgt, src]
            m += 1
        o = eng.synth_scans_dev(SENSOR, c5_scene(synth, s), np.array(poses), c5_noise_seed(s), d_raw_ptr + 24 * off[-1])
        off += [off[-1] + int(x) for x in o[1:]]
        l = m
    return np.array(off, dtype=np.int64)


class ClockSampler:
    def __init__(self, device):
        self.device = device
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        # NVML in-process (a sample costs microseconds, so a 0.2 s timed region still gets ~10 of them); nvidia-smi
        # as a subprocess only if the binding is missing
        try:
            import pynvml
            pynvml.nvmlInit()
            try:  # the CUDA ordinal need not be the NVML index (CUDA_VISIBLE_DEVICES): go by PCI address
                import torch
                pr = torch.cuda.get_device_properties(self.device)
                h = pynvml.nvmlDeviceGetHandleByPciBusId(
                    ("%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)).encode())
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.device)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            bits = {"hw_slowdown": pynvml.nvmlClocksThrottleReasonHwSlowdown,
                    "hw_thermal_slowdown": pynvml.nvmlClocksThrottleReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": pynvml.nvmlClocksThrottleReasonSwThermalSlowdown,
                    "sw_power_cap": pynvml.nvmlClocksThrottleReasonSwPowerCap}
            while not self._stop.is_set():
                self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for n, b in bits.items():
                    if r & b:
                        self.reasons.add(n)
                self._stop.wait(0.02)
            return
        except Exception:
            pass
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.check_output(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                               str(self.device)], timeout=5).decode().strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=10)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def workload_config(n_pairs, world=1, note=None):
    c = {"workload": f"C5: batched ICP of {n_pairs} independent synthetic scan pairs (64 beams x 1875 az, ~119k pts/scan; "
                     "pair i: scene seed 100 + i mod 64, relative pose U(0.5,1.5) m x U(-0.1,0.1) m x U(-0.02,0.02) rad, "
                     "seed 1000 + i)",
         "voxel_m": VOXEL, "normals_k": 20, "icp_max_iterations": 50, "icp_tolerance": 1e-6,
         "stages": "per pair: 2 x voxel_downsample + index + normals (target) + index (source) + point-to-plane ICP",
         "parallelism": f"pair p on rank p % {world}; one NCCL all-gather of the result records per step" if world > 1
                        else "1 GPU",
         "l2": "inputs (GBs of raw scans) are larger than the 126 MB L2"}
    if note:
        c["note"] = note
    return c


def cpu_pair_c5(orc, raw_src, raw_tgt):
    """The reference's work for one independent pair on the CPU oracle: voxel_downsample of both scans
    (file_utils.cpp:148-196) + icp_point_to_plane (icp.hpp:157-258) with the reference's doubled NN search."""
    ds, _ = orc.voxel_downsample(raw_src, VOXEL)
    dt, _ = orc.voxel_downsample(raw_tgt, VOXEL)
    return orc.icp_point_to_plane(ds, dt, faithful_cost=1)


def c5_scans_cpu(syn, i, threads=8):
    s, j, tgt, src, _ = c5_pair(i)
    world = c5_scene(syn, s)
    return (syn.scan(SENSOR, world, tgt, c5_noise_seed(s) + 2 * j, threads=threads),
            syn.scan(SENSOR, world, src, c5_noise_seed(s) + 2 * j + 1, threads=threads))


def run_reference(args):
    """--impl reference: CPU oracle on all host cores over a bounded sample of the same pairs."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle_lib
    from concurrent.futures import ThreadPoolExecutor
    orc, syn = oracle_lib.Oracle(), oracle_lib.Synth()
    cores = os.cpu_count() or 1
    n_pairs = max(cores, min(2 * cores, 64))
    scans = [c5_scans_cpu(syn, i, threads=cores) for i in range(n_pairs)]

    def one(i):  # ctypes releases the GIL: real parallelism over independent pairs
        tgt, src = scans[i]
        return cpu_pair_c5(orc, src, tgt)["num_iterations"]

    def step():
        with ThreadPoolExecutor(cores) as ex:
            return list(ex.map(one, range(n_pairs)))

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    value = n_pairs / dt
    sample = f"pairs 0..{n_pairs - 1} of the same {C5_PAIRS} pairs per step, {cores} threads, one pair per task, same per-pair work"
    print(json.dumps({
        "impl": "reference", "metric": "ICP scan-pairs/s", "value": value, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(C5_PAIRS, note=f"bounded sample: {n_pairs} of the {C5_PAIRS} pairs per step"),
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ---------------------------------------------------------------------------------------------------------------
# sub-results
# ---------------------------------------------------------------------------------------------------------------
def sub_c2(eng, slam_b200, syn, torch, frames, want_streaming=True):
    """C2: `frames` consecutive frame pairs of one sequence registered as ONE batch (consecutive pairs share scans: one
    voxel grid, one index and one set of normals per frame), and the same sequence one frame per call."""
    world = make_world(syn)
    poses = make_poses(syn, frames + 1)
    rays = SENSOR["beams"] * SENSOR["azimuth_steps"]
    d_raw = torch.empty((frames + 1) * rays * 3, dtype=torch.float64, device="cuda")
    off = eng.synth_scans_dev(SENSOR, world, poses, 1000, d_raw.data_ptr())
    src = np.arange(1, frames + 1, dtype=np.int32)   # source = current frame (slam_node.cpp:132-138)
    tgt = np.arange(0, frames, dtype=np.int32)       # target = previous frame
    cfg = eng.icp_config()
    for _ in range(3):
        res, sc = eng.register_batch(None, off, src, tgt, voxel=VOXEL, cfg=cfg, want_sc=True, device_ptr=d_raw.data_ptr())
    eng.set_profiling(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stream = torch.cuda.current_stream()
    reps = 3
    e0.record(stream)
    for _ in range(reps):
        res, sc = eng.register_batch(None, off, src, tgt, voxel=VOXEL, cfg=cfg, want_sc=True, device_ptr=d_raw.data_ptr())
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    st = eng.stage_ms()
    eng.set_profiling(False)
    out = {"c2_batch": {"workload": f"{frames} consecutive frame pairs of one sequence as one batch (+ Scan Context of every "
                                    "frame); scans resident in HBM",
                        "pairs_per_s": frames / (ms * 1e-3), "ms_per_batch": ms, "batch_ms_per_pair": ms / frames,
                        "stages_ms_last_batch": {k: round(v, 3) for k, v in st.items()},
                        "icp_iterations_mean": float(res.num_iterations.mean()),
                        "converged_frac": float(res.converged.mean())}}
    if want_streaming:
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        import stream_latency
        n_s = min(frames, 150) + 1
        h_s = d_raw[:int(off[n_s]) * 3].cpu().numpy().reshape(-1, 3)
        scans_s = [np.ascontiguousarray(h_s[off[i]:off[i + 1]]) for i in range(n_s)]
        out["c2_streaming"] = stream_latency.process_frames(eng, slam_b200, scans_s, VOXEL)
    del d_raw
    return out


def sub_c3(eng, syn, torch):
    world = make_world(syn)
    s128 = dict(SENSOR, beams=128, azimuth_steps=2048)
    n3 = 48
    poses = make_poses(syn, n3)
    d3 = torch.empty(n3 * 128 * 2048 * 3, dtype=torch.float64, device="cuda")
    off3 = eng.synth_scans_dev(s128, world, poses, 5000, d3.data_ptr())
    cfg3 = eng.icp_config(max_iterations=0, normals_k=10)   # index + normals only; no ICP iterations
    p3s, p3t = np.arange(1, n3, dtype=np.int32), np.arange(0, n3 - 1, dtype=np.int32)
    for _ in range(3):
        eng.register_batch(None, off3, p3s, p3t, voxel=0.2, cfg=cfg3, device_ptr=d3.data_ptr())
    eng.set_profiling(True)
    eng.register_batch(None, off3, p3s, p3t, voxel=0.2, cfg=cfg3, device_ptr=d3.data_ptr())
    st3, c3 = eng.stage_ms(), eng.last_counts()
    eng.set_profiling(False)
    del d3
    return {"workload": "128 beams x 2048 az, voxel 0.2 m, k = 10, %d indexed clouds of %.0f points" %
                        (n3 - 1, c3["target_rows"] / (n3 - 1)),
            "knn_plus_normals_queries_per_s": c3["target_rows"] / (st3["normals"] * 1e-3),
            "ms": st3["normals"], "index_build_ms": st3["index_build"], "voxel_ms": st3["voxel"],
            "raw_points_per_s_voxel_grid": c3["raw_rows"] / (st3["voxel"] * 1e-3)}


def sub_c4(eng, slam_b200, syn, torch, dist, rank, world_size, n_db=4000, reps=10):
    """C4 (SURVEY.md 8d): Scan Context search over a 4000-keyframe database built from 4000 poses on the C2 loop (3.3
    laps: true revisits) + ICP verification of the top 10.  The database (descriptors AND clouds) is sharded by entry id
    (sb_loop_create(rank, world)); per detect(): local search -> all-gather of the local candidates -> identical merge
    -> each rank verifies the candidates it owns -> all-gather of the results -> acceptance in the reference's order."""
    import sharding
    world = make_world(syn)
    poses = make_poses(syn, n_db + 1)
    rays = SENSOR["beams"] * SENSOR["azimuth_steps"]
    chunk = 250
    d_raw = torch.empty(chunk * rays * 3, dtype=torch.float64, device="cuda")
    det = slam_b200.LoopClosureDetector(eng, frame_gap=50, sc_distance_threshold=1e300, icp_fitness_threshold=0.3,
                                        max_candidates=10, rank=rank, world=world_size)
    det.reserve(n_db // world_size + 2, (n_db // world_size + 2) * 9500)
    t_build = time.perf_counter()
    for c0 in range(0, n_db, chunk):
        c1 = min(n_db, c0 + chunk)
        off = eng.synth_scans_dev(SENSOR, world, poses[c0:c1], 7000 + c0, d_raw.data_ptr())
        h = d_raw[:int(off[-1]) * 3].cpu().numpy().reshape(-1, 3)
        ds, doff = eng.voxel_downsample_batch(h, off, VOXEL)
        for f in range(c0, c1):
            det.addFrame(ds[doff[f - c0]:doff[f - c0 + 1]], f)
    t_build = time.perf_counter() - t_build
    del d_raw

    def detect():
        md, me, acc, _ = sharding.sharded_detect(det, rank, world_size, top_k=10)
        return md, me, acc

    for _ in range(3):
        detect()
    torch.cuda.synchronize()
    if world_size > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        md, me, acc = detect()
    torch.cuda.synchronize()
    if world_size > 1:
        dist.barrier()
    dt = (time.perf_counter() - t0) / reps
    # search alone (device search + candidate copy), for the FLOP rate
    t0 = time.perf_counter()
    for _ in range(reps):
        det.candidates_local(capacity=16)
    dts = (time.perf_counter() - t0) / reps
    det.close()
    q = n_db - 1
    true_revisits = [int(e) for e in me[:10] if abs(((q - int(e)) % int(LOOP_LEN_M))) <= 3 or abs(((q - int(e)) % int(LOOP_LEN_M)) - LOOP_LEN_M) <= 3]
    return {"workload": f"1 query (frame {q}) vs {n_db} keyframes of the C2 loop (20x60 descriptors, 60 column shifts), "
                        "top-10 verified by ICP (30 it), database sharded by entry id over the ranks",
            "n_gpus": world_size, "ms_per_detect": dt * 1e3, "ms_search_local": dts * 1e3,
            "descriptor_pairs_per_s": n_db / dts, "gflops_fp64_search": 2 * 60 * 1200 * n_db / dts / 1e9 / 1.0,
            "top10_entries": [int(e) for e in me[:10]], "top10_sc_distance": [float(d) for d in md[:10]],
            "accepted_entries": acc, "top10_that_are_true_revisits": len(true_revisits),
            "db_build_s": t_build}


def bind_to_gpu_numa_node(torch, device):
    """Runs this process on the CPUs next to its GPU (sysfs local_cpulist of the GPU's PCI function) so that the pinned
    staging buffers allocated afterwards and the threads that fill them sit on that NUMA node.  Returns what it did."""
    try:
        pr = torch.cuda.get_device_properties(device)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        base = "/sys/bus/pci/devices/" + bdf
        node = int(open(base + "/numa_node").read().strip())
        cpus = set()
        for part in open(base + "/local_cpulist").read().strip().split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"pci": bdf, "numa_node": node, "cpus": len(cpus)}
    except Exception as ex:
        return {"error": repr(ex)}


DUMP_BYTES = 60_000_000   # the files' payload of the whole job: under 64 MB with their headers


def dump_outputs(out_dir, ids, recs, rank=0, world=1):
    """--dump-outputs: what sb_register_batch_dev returned for this rank's pairs in the last timed step, one float64 .npy
    per result field, rows in generation order (`pair_id` names the pair of each row).  error_history holds the pairs'
    histories one after the other, history_len[i] values for pair i, so every value written is one the caller received.
    The inputs are seeded, so two builds run with the same arguments can be compared file by file.  4096 pairs take
    under 1 MB.  With N ranks each writes its own files (suffix _rank<r>) within DUMP_BYTES / N; above that, a fixed,
    seeded sample of its pairs."""
    rec = np.concatenate([r.rec for r in recs])
    row_bytes = 8 * (1 + 16 + 5 + rec["error_history"].shape[1])   # a pair's fields with a full-length history
    keep = np.arange(len(rec))
    cap = DUMP_BYTES // world
    if len(rec) * row_bytes > cap:
        keep = np.sort(np.random.default_rng(rank).choice(len(rec), cap // row_bytes, replace=False))
    rec, hl = rec[keep], rec["history_len"][keep]
    out = {"pair_id": np.asarray(ids)[keep], "transformation": rec["transformation"].reshape(-1, 4, 4),
           "final_error": rec["final_error"], "num_iterations": rec["num_iterations"], "converged": rec["converged"],
           "status": rec["status"], "history_len": hl,
           "error_history": rec["error_history"][np.arange(rec["error_history"].shape[1]) < hl[:, None]]}
    os.makedirs(out_dir, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), np.asarray(v, dtype=np.float64))


# ---------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs", type=int, default=C5_PAIRS, help="independent pairs per step (4096 = config C5)")
    ap.add_argument("--pairs-per-call", type=int, default=4096, help="pairs handed to one sb_register_batch call")
    ap.add_argument("--frames", type=int, default=1000, help="frame pairs of the C2 sub-result")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="skip the C2 / C3 / C4 sub-results")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the results of the GPU path (--impl ours)")
    sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree, which may be read-only
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import oracle_lib
    import sharding
    import slam_b200

    rank = int(os.environ.get("RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(torch, local_rank)   # before any pinned allocation: staging memory next to the GPU
    if world_size > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    assert C5_SCENES % world_size == 0, "ranks own whole scenes: the number of GPUs must divide 64"
    stream = torch.cuda.Stream()
    NP = args.pairs
    with torch.cuda.stream(stream):
        eng = slam_b200.Engine(local_rank, stream=stream.cuda_stream)
        syn = oracle_lib.Synth()
        rays = SENSOR["beams"] * SENSOR["azimuth_steps"]
        ids = c5_pairs_of_rank(NP, rank, world_size)          # this rank's pairs, in generation order
        n_loc = len(ids)
        d_raw = torch.empty(2 * n_loc * rays * 3, dtype=torch.float64, device="cuda")
        off = c5_generate(eng, syn, ids, d_raw.data_ptr(), rays)   # input generation (untimed)
        n_raw = int(off[-1])
        cfg = eng.icp_config()
        # calls of at most --pairs-per-call pairs: scans [2 c0, 2 c1) of the rank
        calls = [(c0, min(n_loc, c0 + args.pairs_per_call)) for c0 in range(0, n_loc, args.pairs_per_call)]

        def call_args(c0, c1):
            o = off[2 * c0:2 * c1 + 1] - off[2 * c0]
            k = np.arange(c1 - c0, dtype=np.int32)
            return o, 2 * k + 1, 2 * k                        # source = scan 2l + 1, target = scan 2l

        def step_dev():
            recs = []
            for c0, c1 in calls:
                o, ps, pt = call_args(c0, c1)
                res = eng.register_batch(None, o, ps, pt, voxel=VOXEL, cfg=cfg, device_ptr=d_raw.data_ptr() + 24 * int(off[2 * c0]))
                recs.append(res)
            return recs

        # exchange buffers of the sharded path: one 21-double record per pair (pair id + sharding.RECORD), all-gathered
        W = sharding.RECORD + 1
        g_host = torch.empty((n_loc, W), dtype=torch.float64, pin_memory=True)
        g_dev = torch.empty((n_loc, W), dtype=torch.float64, device="cuda")
        g_all = torch.empty((world_size * n_loc, W), dtype=torch.float64, device="cuda") if world_size > 1 else None
        g_work = [None]

        def records(recs):
            r = np.concatenate([x.records20() for x in recs])
            return np.concatenate([ids[:, None].astype(np.float64), r], axis=1)

        def gather(recs):
            """NCCL all-gather of the result records: the only exchange of the sharded path (SURVEY.md 8e).  It is queued
            behind the step on the engine's stream and overlaps the next step; the closing barrier + synchronize waits for
            the last one, so every step's records have arrived inside the timed region."""
            if world_size == 1:
                return None
            if g_work[0] is not None:
                g_work[0].wait()   # stream-level wait: the previous gather must have read g_dev before it is rewritten
            g_host.numpy()[...] = records(recs)
            g_dev.copy_(g_host, non_blocking=True)
            g_work[0] = dist.all_gather_into_tensor(g_all, g_dev, async_op=True)
            return g_all

        def barrier():
            if world_size > 1:
                dist.barrier()
            torch.cuda.synchronize()

        # ---- warm-up
        for _ in range(max(args.warmup, 3)):
            recs = step_dev()
            gather(recs)
        # ---- timed: device-resident inputs
        eng.set_profiling(True)
        sampler = ClockSampler(local_rank)
        barrier()
        if rank == 0:  # one sampler per node: nvidia-smi from every rank perturbs the run it is meant to watch
            sampler.start()
        l0 = eng.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stage_acc, counts_acc = {}, {}
        gathered = None
        e0.record(stream)
        for _ in range(args.steps):
            recs = []
            for c0, c1 in calls:
                o, ps, pt = call_args(c0, c1)
                recs.append(eng.register_batch(None, o, ps, pt, voxel=VOXEL, cfg=cfg,
                                               device_ptr=d_raw.data_ptr() + 24 * int(off[2 * c0])))
                for k, v in eng.stage_ms().items():
                    stage_acc[k] = stage_acc.get(k, 0.0) + v
                for k, v in eng.last_counts().items():
                    counts_acc[k] = counts_acc.get(k, 0) + v
            gathered = gather(recs)
        e1.record(stream)
        barrier()
        clocks = sampler.stop()
        launches = eng.launch_count - l0
        ms = e0.elapsed_time(e1) / args.steps
        eng.set_profiling(False)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, ids, recs, rank, world_size)
        mine = records(recs)
        if gathered is not None:  # the exchange really delivered every rank's records: all 4096 pair ids, once each
            allrec = gathered.cpu().numpy()
            assert np.array_equal(allrec[rank * n_loc:(rank + 1) * n_loc], mine)
            assert np.array_equal(np.sort(allrec[:, 0].astype(np.int64)), np.arange(NP))
        else:
            allrec = mine
        t_ms = torch.tensor([ms], device="cuda", dtype=torch.float64)
        if world_size > 1:
            dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        ms_max = float(t_ms.item())
        value = NP / (ms_max * 1e-3)     # strong scaling: the job is always the same NP pairs
        per_rank = None
        if world_size > 1:
            me_t = torch.tensor([ms, sum(stage_acc.values()) / args.steps], device="cuda", dtype=torch.float64)
            allr = [torch.empty_like(me_t) for _ in range(world_size)]
            dist.all_gather(allr, me_t)
            per_rank = {"step_ms": [round(float(a[0]), 2) for a in allr],
                        "device_busy_ms": [round(float(a[1]), 2) for a in allr]}

        # ---- e2e: host (pinned) float32 records — what a PLY / KITTI file holds (file_utils.cpp:91-97) — through
        # sb_register_batch_f32, H2D of every scan and D2H of the results inside the timed region
        e2e = None
        if not args.no_e2e:
            h32 = torch.empty((n_raw, 3), dtype=torch.float32, pin_memory=True)
            step_rows = 32 * 1024 * 1024
            for r0 in range(0, n_raw, step_rows):
                r1 = min(n_raw, r0 + step_rows)
                blk = d_raw[3 * r0:3 * r1]
                b32 = blk.to(torch.float32)
                assert torch.equal(b32.to(torch.float64), blk)  # the scans are float32-born: nothing is lost
                h32[r0:r1].copy_(b32.view(-1, 3))
            torch.cuda.synchronize()
            h_np = h32.numpy()

            def step_host():
                out = []
                for c0, c1 in calls:
                    o, ps, pt = call_args(c0, c1)
                    out.append(eng.register_batch(h_np[int(off[2 * c0]):int(off[2 * c1])], o, ps, pt, voxel=VOXEL, cfg=cfg))
                return out

            # the ceiling of this path: every rank of the job copying its pinned records to its GPU at the same time
            d_sink = torch.empty((min(n_raw, 1 << 28), 3), dtype=torch.float32, device="cuda")
            rows_c = d_sink.shape[0]
            barrier()
            c0_, c1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps_c = 3
            c0_.record(stream)
            for _ in range(reps_c):
                for r0 in range(0, n_raw, rows_c):
                    r1 = min(n_raw, r0 + rows_c)
                    d_sink[:r1 - r0].copy_(h32[r0:r1], non_blocking=True)
            c1_.record(stream)
            barrier()
            t_c = torch.tensor([c0_.elapsed_time(c1_) / reps_c], device="cuda", dtype=torch.float64)
            if world_size > 1:
                dist.all_reduce(t_c, op=dist.ReduceOp.MAX)
            copy_ms = float(t_c.item())
            del d_sink
            for _ in range(2):
                gather(step_host())
            barrier()
            t0 = time.perf_counter()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record(stream)
            for _ in range(args.steps):
                r2 = step_host()
                gather(r2)
            g1.record(stream)
            barrier()
            wall = (time.perf_counter() - t0) / args.steps * 1e3
            ms2 = max(g0.elapsed_time(g1) / args.steps, wall)  # host-side work (staging, result decode) counts
            t2 = torch.tensor([ms2], device="cuda", dtype=torch.float64)
            if world_size > 1:
                dist.all_reduce(t2, op=dist.ReduceOp.MAX)
            assert np.array_equal(records(r2), mine)            # same bits as the device-resident path
            e2e = {"value": NP / (float(t2.item()) * 1e-3), "unit": "pairs/s",
                   "h2d_bytes_per_step": int(n_raw * 12) * world_size if world_size == 1 else None,
                   "d2h_bytes_per_step": int(n_loc * 1184), "ms_per_step": float(t2.item()),
                   "input": "pinned host float32 xyz records (as read from disk), widened on the device"}
            # bytes over all ranks
            hb = torch.tensor([float(n_raw * 12), float(n_loc * 1184)], device="cuda", dtype=torch.float64)
            if world_size > 1:
                dist.all_reduce(hb)
            e2e["h2d_bytes_per_step"], e2e["d2h_bytes_per_step"] = int(hb[0].item()), int(hb[1].item())
            # how close the step is to doing nothing but the copies (all ranks at once, same buffers, same node)
            e2e["h2d_ceiling"] = {"copy_only_ms_per_step": copy_ms, "aggregate_gb_per_s": hb[0].item() / copy_ms / 1e6,
                                  "pairs_per_s_if_copy_bound": NP / (copy_ms * 1e-3),
                                  "e2e_frac_of_ceiling": copy_ms / float(t2.item()), "numa": numa}
            del h32

        # ---- C4 on every rank (sharded database); the other sub-results on rank 0 at N = 1
        subs = {}
        if not args.no_sub:
            try:
                subs["c4_loop_closure"] = sub_c4(eng, slam_b200, syn, torch, dist, rank, world_size)
            except Exception as ex:  # the headline line must still be printed
                subs["c4_loop_closure"] = {"error": repr(ex)}

        if rank != 0:
            if world_size > 1:
                dist.destroy_process_group()
            return

        # ---- roofline of the dominant stage (algorithmic bytes: SURVEY.md 8d / DESIGN.md)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        st = {k: v / args.steps for k, v in stage_acc.items()}
        cn = {k: v / args.steps for k, v in counts_acc.items()}
        N, M, T, Q = cn["raw_rows"], cn["voxel_rows"], cn["target_rows"], cn["nn_queries"]
        n_calls = len(calls)
        alg = {"voxel": 24 * N + 24 * M, "index_build": 52 * T, "normals": 48 * (T / 2),
               "icp_loop": 72 * Q + 232 * n_loc * max(cn["icp_iter_launches"] / n_calls, 1)}
        kern = {"voxel": "k_vox_insert (+ clear/list/sort/finalize/collect/patch)",
                "index_build": "k_morton/k_sort_*/k_gather_leaves",
                "normals": "k_self_knn (+ k_knn_redo + k_normals_from_graph)",
                "icp_loop": "k_icp_match/k_icp_fallback/k_icp_accum/k_icp_solve in the CUDA-graph WHILE loop"}
        traffic = {}
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        except Exception:
            pass
        dom = max(alg, key=lambda k: st.get(k, 0.0))
        dom_ms = st[dom]
        launches_dom = {"normals": 3 * n_calls, "voxel": 7 * n_calls, "index_build": 8 * n_calls}.get(
            dom, int(4 * cn["icp_iter_launches"] + 7 * n_calls))
        achieved = alg[dom] / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
        tr = traffic.get(dom, {})
        sm_mhz = clocks.get("sm_mhz") or peaks.get("sm_max_mhz", 1965.0)
        issue_peak = 148 * 4 * sm_mhz * 1e6           # warp-instructions per second the chip can issue
        roofline = {"bound": "hbm", "kernel": kern[dom], "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak,
                    # DRAM bytes per unit of work of that kernel from the committed ncu capture, scaled to this launch
                    "traffic": (tr["dram_bytes_per_unit"] * tr_units(dom, cn) / max(n_calls, 1) if "dram_bytes_per_unit" in tr else None),
                    "traffic_source": tr.get("source"),
                    "peak_source": peak_src,
                    "algorithmic_bytes_per_step": int(alg[dom]), "launches_per_step": int(launches_dom),
                    "avg_launch_ms": dom_ms / max(launches_dom, 1),
                    "stages_ms": st,
                    "stage_frac_of_peak": {k: (alg[k] / (st[k] * 1e-3) / 1e9 / peak if st.get(k, 0) > 0 else None)
                                           for k in alg},
                    # the path is instruction-issue-bound, not bandwidth-bound (DESIGN.md section 6): the same stage
                    # against the chip's issue rate, warp-instructions per unit from the committed ncu capture
                    "issue": ({"warp_inst_per_unit": tr["warp_inst_per_unit"], "unit": tr.get("unit"),
                               "achieved_warp_inst_per_s": tr["warp_inst_per_unit"] * tr_units(dom, cn) / (dom_ms * 1e-3),
                               "peak_warp_inst_per_s": issue_peak,
                               "frac": tr["warp_inst_per_unit"] * tr_units(dom, cn) / (dom_ms * 1e-3) / issue_peak}
                              if "warp_inst_per_unit" in tr and dom_ms > 0 else None)}

        # ---- cpu_baseline: the oracle, 1 thread (the reference is single-threaded), bounded sample of the same pairs
        orc = oracle_lib.Oracle()
        rec_by_id = {int(r[0]): r[1:] for r in allrec}
        t0 = time.perf_counter()
        tgt0, src0 = c5_scans_cpu(syn, 0)
        cpu_first = cpu_pair_c5(orc, src0, tgt0)
        t1 = time.perf_counter() - t0
        n_cpu = int(max(1, min(8, args.cpu_seconds / max(t1, 1e-3))))
        cpu_scans = [(tgt0, src0)] + [c5_scans_cpu(syn, i) for i in range(1, n_cpu)]
        t0 = time.perf_counter()
        cpu_out = [cpu_pair_c5(orc, s_, t_) for (t_, s_) in cpu_scans]
        cpu_dt = time.perf_counter() - t0
        max_dt, max_rel = 0.0, 0.0
        for i in range(n_cpu):   # parity spot check on the same pairs, and the pose the pair was generated with
            Tg = rec_by_id[i][:16].reshape(4, 4)
            dT = Tg @ np.linalg.inv(cpu_out[i]["transformation"])
            max_dt = max(max_dt, float(np.linalg.norm(dT[:3, 3])))
            rel = c5_pair(i)[4]
            max_rel = max(max_rel, float(np.hypot(Tg[0, 3] - rel[0], Tg[1, 3] - rel[1])))
        cpu_baseline = {"value": n_cpu / cpu_dt, "unit": "pairs/s", "cores": 1, "kind": "port",
                        "sample": f"pairs 0..{n_cpu - 1} of the same {NP} pairs, single thread, reference cost model (NN search "
                                  "twice per iteration); the reference's own sources build only over an Eigen stand-in "
                                  "(oracle/_ref), a checker whose eager loops are not Eigen's speed",
                        "parity_max_translation_diff_m": max_dt, "max_offset_from_generating_pose_m": max_rel}

        # ---- the other configurations BASELINE.json names, as named sub-results
        if not args.no_sub and world_size == 1:
            try:
                subs.update(sub_c2(eng, slam_b200, syn, torch, args.frames))
                subs["c3_knn_normals"] = sub_c3(eng, syn, torch)
            except Exception as ex:
                subs["error"] = repr(ex)

        iters = allrec[:, 1 + 17]
        conv = allrec[:, 1 + 18]
        out = {
            "metric": "ICP scan-pairs/s", "value": value, "unit": "pairs/s", "n_gpus": world_size, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_max, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(NP, world_size),
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "per_rank": per_rank,
            "roofline": roofline, "cpu_baseline": cpu_baseline,
            "workload_stats": {"pairs": NP, "pairs_this_rank": n_loc, "calls_per_step": n_calls,
                               "raw_points_per_scan": N / (2 * n_loc), "voxel_points_per_scan": M / (2 * n_loc),
                               "icp_iterations_mean": float(iters.mean()), "icp_iterations_max": int(iters.max()),
                               "converged_frac": float(conv.mean()), "status_ok_frac": float((allrec[:, 1 + 19] == 0).mean())},
        }
        out.update(subs)
        print(json.dumps(out))
        if world_size > 1:
            dist.destroy_process_group()


def tr_units(stage, cn):
    """Units of work of a stage in this step, as profiles/r02_traffic.json counts them."""
    return {"normals": cn["target_rows"] / 2, "voxel": cn["raw_rows"], "index_build": cn["target_rows"],
            "icp_loop": cn["nn_queries"]}[stage]


if __name__ == "__main__":
    main()
