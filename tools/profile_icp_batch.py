#!/usr/bin/env python
"""Loop-closure verification throughput: B single-pair liorf_loop_closure_icp calls against one liorf_loop_closure_icp_batch call.

A looped synthetic drive (bench.Sequence(..., loop=True), KITTI-shaped HDL-64 scans) runs through liorf_process_frame; the pairs
detectLoopClosureID proposes along the way (performSCLoopClosure's form: loop_index = 0, history_search_num = 25, 0.5 m leaf) are
padded with wrong-place pairs up to B.  For each B the two arms alternate, each timed with the host clock around work that ends in a
stream synchronise, after a warm-up of both; every batch result is compared with the single-pair results bit for bit.
usage: python tools/profile_icp_batch.py [out_dir (default: <tmp>/liorf_icp_batch)] [frames] [reps]"""
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_label():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return name, q


def main():
    import bench
    out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(tempfile.gettempdir(), "liorf_icp_batch")
    n_frames = int(sys.argv[2]) if len(sys.argv) > 2 else 1050
    reps = int(sys.argv[3]) if len(sys.argv) > 3 else 5
    os.makedirs(out_dir, exist_ok=True)
    seq = bench.Sequence(n_frames, 0, loop=True)
    pipe = bench.GpuPipeline(seq, 0)
    proposed = []
    t0 = time.time()
    for s in range(0, n_frames, 100):
        fr = range(s, min(n_frames, s + 100))
        pipe.stage(range(s, min(n_frames, s + 101)))
        for i in fr:
            guess = seq.initial_guess(i, pipe.prev)
            fo = pipe.ctx.processFrameIn(pipe._frame_in(i, "dev"), guess, None)
            pipe.prev = np.array(fo.pose[:], np.float32)
            if fo.loop_checked and fo.loop_id >= 0:
                proposed.append((pipe.ctx.numKeyframes() - 1, int(fo.loop_id)))
        for i in fr:                                           # keep host / device memory of the staged scans bounded
            pipe.dev_raw.pop(i, None); pipe.pin_raw.pop(i, None); seq.raw.pop(i, None)
    ctx = pipe.ctx
    n_kf = ctx.numKeyframes()
    print(f"drive: {n_frames} frames, {n_kf} keyframes, {len(proposed)} proposed loops, {time.time() - t0:.0f} s", flush=True)
    rng = np.random.default_rng(11)
    pairs = list(dict.fromkeys(proposed))
    while len(pairs) < 256:                                    # wrong places: a keyframe against one at least 60 keyframes away
        a = int(rng.integers(0, n_kf)); b = int(rng.integers(0, n_kf))
        if abs(a - b) >= 60:
            pairs.append((a, b))
    hs, leaf, mcd, iters = 25, 0.5, 20.0, 100
    name, smi = gpu_label()
    res = dict(gpu=name, nvidia_smi=smi, frames=n_frames, keyframes=n_kf, proposed_loops=len(proposed), history_search_num=hs, icp_leaf=leaf,
               max_corr_dist=mcd, max_iters=iters, reps=reps, runs=[])

    def single(P):
        t = time.perf_counter()
        r = [ctx.loopClosureICP(c, p, hs, 0, leaf, mcd, iters) for c, p in P]          # each call ends in a stream synchronise
        return time.perf_counter() - t, r

    def batch(P):
        cur = np.array([p[0] for p in P], np.int32); pre = np.array([p[1] for p in P], np.int32)
        t = time.perf_counter()
        r = ctx.loopClosureICPBatch(cur, pre, 0, hs, leaf, mcd, iters)                   # returns after its last stream synchronise
        return time.perf_counter() - t, list(r)

    for B in (1, 8, 64, 256):
        P = pairs[:B]
        single(P); batch(P)                                    # warm-up: module load, buffer growth of both arms
        ts, tb = [], []
        ok = True
        for _ in range(reps):
            a, ra = single(P); b, rb = batch(P)
            ts.append(a); tb.append(b)
            ok = ok and all(bytes(x) == bytes(y) for x, y in zip(ra, rb))
        ran = sum(r.ran for r in rb)
        conv = sum(r.ran and r.converged and r.fitness <= 0.3 for r in rb)
        row = dict(B=B, ran=ran, accepted=conv, bit_identical=bool(ok),
                   single_ms_median=1e3 * float(np.median(ts)), single_ms_min=1e3 * min(ts), single_ms_max=1e3 * max(ts),
                   batch_ms_median=1e3 * float(np.median(tb)), batch_ms_min=1e3 * min(tb), batch_ms_max=1e3 * max(tb),
                   single_pairs_per_s=B / float(np.median(ts)), batch_pairs_per_s=B / float(np.median(tb)),
                   mean_n_source=float(np.mean([r.n_source for r in rb])), mean_n_target=float(np.mean([r.n_target for r in rb])))
        res["runs"].append(row)
        print(json.dumps(row), flush=True)
        with open(os.path.join(out_dir, "icp_batch.json"), "w") as f:          # after every B: a partial run keeps what it measured
            json.dump(res, f, indent=1)
    print(f"{name} | {smi}")
    ctx.close()
    assert all(r["bit_identical"] for r in res["runs"])


if __name__ == "__main__":
    main()
