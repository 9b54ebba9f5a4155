#!/usr/bin/env python
"""Loop detection over a drive's own keyframes: the drive's sequential liorf_sc_detect_loop_closure_id calls against one
liorf_sc_detect_loop_closure_id_batch call.

A looped synthetic drive (bench.Sequence(..., loop=True), KITTI-shaped HDL-64 scans) runs through liorf_process_frame with loop_every = 10;
every loop check is recorded (the database size at the call, loop_id, loop_yaw).  One batch call with the stale-tree schedule of that call
history (liorf_b200.sc_tree_schedule) must reproduce every id and every yaw bit.  A twin context holding the same descriptors then replays
the same calls sequentially (only the detect calls timed, database growth between them untimed) and the two arms alternate, each timed with
the host clock around work that ends in a stream synchronise.  The loops found are verified with one loopClosureICPBatch call (performSCLoopClosure's
form: loopKeyCur = n_db - 1, loop_index = 0, history_search_num = 25, 0.5 m leaf).
usage: python tools/profile_sc_detect_batch.py [out_dir (default: <tmp>/liorf_sc_detect_batch)] [frames] [reps]"""
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.profile_icp_batch import gpu_label  # noqa: E402


def main():
    import bench
    import liorf_b200
    out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(tempfile.gettempdir(), "liorf_sc_detect_batch")
    n_frames = int(sys.argv[2]) if len(sys.argv) > 2 else 1050
    reps = int(sys.argv[3]) if len(sys.argv) > 3 else 5
    os.makedirs(out_dir, exist_ok=True)
    seq = bench.Sequence(n_frames, 0, loop=True)
    pipe = bench.GpuPipeline(seq, 0)
    checks = []                                                # (database size at the call, loop_id, loop_yaw)
    t0 = time.time()
    for s in range(0, n_frames, 100):
        fr = range(s, min(n_frames, s + 100))
        pipe.stage(range(s, min(n_frames, s + 101)))
        for i in fr:
            guess = seq.initial_guess(i, pipe.prev)
            fo = pipe.ctx.processFrameIn(pipe._frame_in(i, "dev"), guess, None)
            pipe.prev = np.array(fo.pose[:], np.float32)
            if fo.loop_checked:
                checks.append((pipe.ctx.scSize(), int(fo.loop_id), np.float32(fo.loop_yaw)))
        for i in fr:
            pipe.dev_raw.pop(i, None); pipe.pin_raw.pop(i, None); seq.raw.pop(i, None)
    ctx = pipe.ctx
    n_kf = ctx.numKeyframes()
    assert ctx.scSize() == n_kf
    n_db = np.array([c[0] for c in checks], np.int32)
    want_id = np.array([c[1] for c in checks], np.int32)
    want_yaw = np.array([c[2] for c in checks], np.float32)
    n_tree = liorf_b200.sc_tree_schedule(n_db)
    print(f"drive: {n_frames} frames, {n_kf} keyframes, {len(checks)} loop checks, {int((want_id >= 0).sum())} loops, {time.time() - t0:.0f} s", flush=True)

    lid, yaw, _, _ = ctx.detectLoopClosureIDBatch(n_db, n_tree)
    assert np.array_equal(lid, want_id), np.nonzero(lid != want_id)
    assert np.array_equal(yaw.view(np.int32), want_yaw.view(np.int32)), np.nonzero(yaw.view(np.int32) != want_yaw.view(np.int32))

    descs = np.stack([ctx.scGet(i)[0].reshape(-1) for i in range(n_kf)])

    def sequential():
        """a fresh twin context whose database grows as the drive grew it; only the detect calls are timed"""
        twin = liorf_b200.Context()
        have, dt, out = 0, 0.0, []
        for n in n_db:
            if n > have:
                twin.scAddDescriptors(descs[have:n]); have = n          # ends in a stream synchronise
            t = time.perf_counter()
            r = twin.detectLoopClosureID()                               # ends in a stream synchronise
            dt += time.perf_counter() - t
            out.append(r[0])
        twin.close()
        return dt, np.array(out, np.int32)

    def batch():
        t = time.perf_counter()
        r = ctx.detectLoopClosureIDBatch(n_db, n_tree)                   # returns after its one stream synchronise
        return time.perf_counter() - t, r[0]

    sequential(); batch()                                        # warm-up of both arms
    ts, tb = [], []
    for _ in range(reps):
        a, ra = sequential(); b, rb = batch()
        assert np.array_equal(ra, want_id) and np.array_equal(rb, want_id)
        ts.append(a); tb.append(b)

    found = lid >= 0
    cur, pre = n_db[found] - 1, lid[found]
    t = time.perf_counter()
    icp = ctx.loopClosureICPBatch(cur, pre, 0, 25, 0.5, 20.0, 100, as_arrays=True)
    t_icp = time.perf_counter() - t
    accepted = int(((icp["ran"] != 0) & (icp["converged"] != 0) & (icp["fitness"] <= 0.3)).sum())

    name, smi = gpu_label()
    res = dict(gpu=name, nvidia_smi=smi, frames=n_frames, keyframes=n_kf, loop_checks=len(checks), loops=int(found.sum()), reps=reps,
               ids_and_yaw_bit_identical=True,
               sequential_ms_median=1e3 * float(np.median(ts)), sequential_ms_min=1e3 * min(ts), sequential_ms_max=1e3 * max(ts),
               batch_ms_median=1e3 * float(np.median(tb)), batch_ms_min=1e3 * min(tb), batch_ms_max=1e3 * max(tb),
               icp_batch_pairs=int(found.sum()), icp_batch_ms=1e3 * t_icp, icp_accepted=accepted)
    print(json.dumps(res), flush=True)
    with open(os.path.join(out_dir, "sc_detect_batch.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(f"{name} | {smi}")
    ctx.close()


if __name__ == "__main__":
    main()
