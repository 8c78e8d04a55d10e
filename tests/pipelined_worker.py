"""Child process of tests/test_scale_parity.py::test_pipelined_sub_batches_in_a_subprocess.

SB_ICP_SUB and SB_CHUNK_MB are read once per process, so the pipelined host path with one ICP sub-batch per chunk is
checked in a process of its own: python pipelined_worker.py <dir>.  <dir> holds the parent's C5 sample (scans32.npy,
offsets.npy) and what sb_register_batch_dev returned for it (bits.npy, sc.npy).  Prints one marker line per check.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "lidar-slam-from-scratch_b200", "python"))
import torch  # noqa: E402

import slam_b200  # noqa: E402
from test_scale_parity import result_bits, same_bits  # noqa: E402

CHAIN = 310          # clouds of the > 256 sub-batch case: one chunk each, 309 of them make a pair ready


def pinned_f32(rows):
    buf = torch.empty(rows.shape, dtype=torch.float32, pin_memory=True).numpy()
    buf[...] = rows
    return buf


def main(d):
    assert os.environ.get("SB_ICP_SUB") == "1" and os.environ.get("SB_CHUNK_MB") == "1"
    eng = slam_b200.Engine(0)
    # 1. the C5 sample through sb_register_batch_f32 from pinned memory, one ICP sub-batch per ready pair
    rows = np.load(os.path.join(d, "scans32.npy"))
    off = np.load(os.path.join(d, "offsets.npy"))
    n = (len(off) - 1) // 2
    k = np.arange(n, dtype=np.int32)
    h = pinned_f32(rows)
    res, sc = eng.register_batch(h, off, 2 * k + 1, 2 * k, voxel=0.5, want_sc=True)
    assert same_bits(result_bits(res), np.load(os.path.join(d, "bits.npy")))
    assert same_bits(sc, np.load(os.path.join(d, "sc.npy")))
    print("SAMPLE_F32_SUB1 identical", n, flush=True)
    del h

    # 2. a chain of CHAIN full scans (copies of the sample's first six), pairs (i + 1 -> i).  Every cloud is larger
    # than SB_CHUNK_MB, so every chunk holds one cloud and every chunk after the first makes one pair ready: more
    # ICP sub-batches than the context has staging slots for (Ctx::ICP_SLOTS = 256)
    sizes = np.diff(off)[:6]
    assert np.all(sizes * 12 > (1 << 20)), sizes
    clouds = [rows[off[c]:off[c + 1]] for c in range(6)]
    chain = np.concatenate([clouds[i % 6] for i in range(CHAIN)])
    coff = np.r_[0, np.cumsum([len(clouds[i % 6]) for i in range(CHAIN)])].astype(np.int64)
    src = np.arange(1, CHAIN, dtype=np.int32)
    tgt = np.arange(0, CHAIN - 1, dtype=np.int32)
    hc = pinned_f32(chain)
    d64 = torch.from_numpy(hc).to("cuda").double()
    torch.cuda.synchronize()
    dev = eng.register_batch(None, coff, src, tgt, voxel=0.5, device_ptr=d64.data_ptr())
    del d64
    got = eng.register_batch(hc, coff, src, tgt, voxel=0.5)
    assert same_bits(result_bits(got), result_bits(dev))
    assert np.all(got.status == 0)
    print("CHAIN_SUBBATCHES", CHAIN - 1, "pairs", len(src), "identical", flush=True)

    # 3. a non-finite row in the last cloud: the error is found in the last chunk, after hundreds of sub-batches were
    # launched.  The call raises; the next call on the same engine returns what a fresh engine returns
    saved = hc[coff[-2]].copy()
    hc[coff[-2]] = np.nan
    try:
        eng.register_batch(hc, coff, src, tgt, voxel=0.5)
        raise AssertionError("a NaN row did not raise")
    except slam_b200.SlamB200Error as e:
        assert e.status == 5, e
    hc[coff[-2]] = saved
    again = eng.register_batch(hc, coff, src, tgt, voxel=0.5)
    fresh_eng = slam_b200.Engine(0)
    fresh = fresh_eng.register_batch(hc, coff, src, tgt, voxel=0.5)
    fresh_eng.close()
    assert same_bits(result_bits(again), result_bits(fresh))
    assert same_bits(result_bits(again), result_bits(dev))
    print("ERROR_THEN_CLEAN identical", flush=True)
    eng.close()
    print("PIPELINED_WORKER_OK", flush=True)


if __name__ == "__main__":
    main(sys.argv[1])
