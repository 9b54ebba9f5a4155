"""Teardown of a context (liorf_destroy): the context's streams drain first, then every member releases what it owns.  A context destroyed
with work still queued on all three of its streams leaves nothing behind that changes a later context's results; borrowers of a ScanContext
database release nothing of the owner's; and create / destroy cycles that touch every lazily acquired resource return the device memory
they took."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N_FRAMES = 8          # four keyframes of ~5 k points: every local map of the drive is above the graph-path threshold


@pytest.fixture(scope="module")
def drive(synth, oracle):
    import bench
    seq = bench.Sequence(N_FRAMES, 0)
    for i in range(N_FRAMES):
        seq.frame(i)
    return bench, seq


def _kitti_solve(case):
    import liorf_b200
    c = liorf_b200.Context()
    for cloud, pose in case["keyframes"]:
        c.addKeyframeCloud(cloud, pose)
    m = c.extractSurroundingKeyFrames(list(range(len(case["keyframes"]))))
    c.setCurrentScan(case["scan"])
    ds, n = c.downsampleCurrentScan(len(case["scan"]))
    pose, tr = c.scan2MapOptimization(case["init"], 30)
    out = dict(m=m, n=n, ds=ds, pose=np.array(pose, np.float32), trace=tr.poses(), iters=tr.iters)
    c.close()
    return out


def _same_batch(a, b):
    return all(np.array_equal(np.nan_to_num(x, nan=-7.0), np.nan_to_num(y, nan=-7.0)) for x, y in zip(a, b))


def test_destroy_with_work_in_flight(drive, kitti_case):
    """look-ahead frame on stream_pre, a graph-path local-map build on stream_map and an asynchronous solve on the main stream, then
    liorf_destroy without liorf_sync; a fresh context then solves the small KITTI case bit-identically to one that ran before"""
    bench, seq = drive
    before = _kitti_solve(kitti_case)
    gpu = bench.GpuPipeline(seq, 0)
    gpu.stage(range(N_FRAMES))
    for i in range(N_FRAMES - 1):
        gpu.step(i, "dev", lookahead=True)                   # the last step leaves frame N_FRAMES - 1's front end queued on stream_pre
    c = gpu.ctx
    assert c.numKeyframes() >= 2
    c.extractSurroundingKeyFrames([0], want_count=False)     # not the resident selection: the map chain is queued on stream_map
    c.scan2MapOptimizationAsync(gpu.prev, 30)
    c.close()
    after = _kitti_solve(kitti_case)
    for k in before:
        assert np.array_equal(before[k], after[k]), k


def test_borrowers_release_nothing_of_the_owner(synth):
    """a borrower is destroyed and the owner still answers bit-identically; a context that borrowed from a borrower reads the owner's
    database, so it keeps answering after the context it borrowed from is gone"""
    import liorf_b200
    K, Q = 3000, 200
    db = synth.sc_descriptors(K, seed=111)
    qd = synth.sc_queries(db, Q, seed=112)[0]
    owner = liorf_b200.Context(); owner.scAddDescriptors(db); owner.scSetSearchPath(2)
    ref = owner.scQueryBatch(qd)
    b1 = liorf_b200.Context(); b1.scBorrowDatabase(owner); b1.scSetSearchPath(2)
    b2 = liorf_b200.Context(); b2.scBorrowDatabase(b1); b2.scSetSearchPath(2)
    assert b2.scSize() == K
    assert _same_batch(b1.scQueryBatch(qd), ref) and _same_batch(b2.scQueryBatch(qd), ref)
    b1.close()
    assert _same_batch(b2.scQueryBatch(qd), ref)
    with pytest.raises(liorf_b200.api.LiorfError):
        b2.scAddDescriptors(db[:1])
    b2.close()
    assert _same_batch(owner.scQueryBatch(qd), ref)
    owner.close()


def test_shard_lanes_torn_down_borrower_first(synth):
    """two ranks on one device mapping each other's windows by pointer, each with a second lane that borrows the rank's database and index:
    the borrowing lanes are destroyed first, and the owners keep answering with the windows they still share"""
    import torch
    import liorf_b200
    from liorf_b200.sc_sharded import PeerShardedSearch
    K, Q, world = 3000, 200, 2
    db = synth.sc_descriptors(K, seed=121)
    bounds = [0, 1400, 3000]
    ref = liorf_b200.Context(); ref.scAddDescriptors(db)
    owners = [liorf_b200.Context() for _ in range(world)]
    for g, c in enumerate(owners):
        c.scAddDescriptors(db[bounds[g]:bounds[g + 1]]); c.scSetSearchPath(2)
    S0 = [PeerShardedSearch(c, g, world, bounds, Q, torch) for g, c in enumerate(owners)]
    for s in S0:
        s.connect_local(S0)
    PeerShardedSearch.sync_keys_local(S0)
    for c in owners:
        c.sync()
    guests = [liorf_b200.Context() for _ in range(world)]
    for g, c in enumerate(guests):
        c.scBorrowDatabase(owners[g]); c.scSetSearchPath(2)
    S1 = [PeerShardedSearch(c, g, world, bounds, Q, torch, k_total_max=0) for g, c in enumerate(guests)]
    for s in S1:
        s.connect_local(S1)
    qs = [synth.sc_queries(db, Q, seed=122 + b)[0] for b in range(2)]
    d_q = [torch.from_numpy(q).to(S0[0].dev) for q in qs]
    expect = [ref.scQueryBatch(q) for q in qs]
    torch.cuda.synchronize()

    def run(lanes):
        res = {}
        for step in (1, 2, 4):                               # one device: every push is queued before the waits that need it
            for lane in lanes:
                for g in range(world):
                    res[(lane, g)] = (S0, S1)[lane][g].query(d_q[lane], phases=step)
        for c in owners + (guests if 1 in lanes else []):
            c.sync()
        torch.cuda.synchronize()
        for lane in lanes:
            for g in range(world):
                loop, sh, dd, cand = [t.cpu().numpy() for t in res[(lane, g)]]
                assert _same_batch((loop, sh, dd, cand), expect[lane]), (lane, g)

    run((0, 1))
    for c in guests:
        c.close()
    run((0,))
    for c in owners:
        c.close()
    ref.close()


def _process_gpu_bytes(pynvml):
    """device memory NVML attributes to this process, over every device (a read-only query)"""
    total, seen = 0, False
    for d in range(pynvml.nvmlDeviceGetCount()):
        for p in pynvml.nvmlDeviceGetComputeRunningProcesses(pynvml.nvmlDeviceGetHandleByIndex(d)):
            if p.pid == os.getpid() and p.usedGpuMemory is not None:
                total += p.usedGpuMemory; seen = True
    return total if seen else None


def test_repeated_create_destroy_cycles(drive, synth, monkeypatch):
    """20 cycles, each creating a context, touching every lazily acquired resource and destroying it; the process's device memory after
    cycle 20 equals that after cycle 2 (regression guard: a leaked buffer, pinned block or window shows up here)"""
    pynvml = pytest.importorskip("pynvml")
    import torch
    from liorf_b200.sc_sharded import PeerShardedSearch
    bench, seq = drive
    monkeypatch.setenv("LIORF_HOST_TIMING", "1")             # read at create: timeline events of liorf_process_frame
    extra = synth.sc_descriptors(200, seed=131)

    def cycle():
        gpu = bench.GpuPipeline(seq, 0)
        c = gpu.ctx
        c.enableTiming(True)                                 # profiler events
        for fn in (c.lib.liorf_debug_voxelgrid_stamps, c.lib.liorf_debug_s2m_clocks, c.lib.liorf_debug_s2m_arrivals):
            assert fn(c.h, 1, None) == 0                      # debug stamp buffers
        gpu.stage(range(N_FRAMES))
        for i in range(N_FRAMES):
            gpu.step(i, "dev", lookahead=True)               # look-ahead front ends, graph-path local maps, keyframes, ScanContext entries
        n_kf = c.numKeyframes()
        assert c.loopClosureICP(n_kf - 1, 0, history_search_num=2).ran == 1
        assert len(c.loopClosureICPBatch([n_kf - 1, n_kf - 2], [0, 0], 0, history_search_num=2)) == 2
        c.scAddDescriptors(extra)
        c.scSetSearchPath(2)                                 # tensor-core search: operand image, centre, overflow counter
        n_db = np.arange(31, c.scSize() + 1)
        c.detectLoopClosureIDBatch(n_db, n_db - 30)
        s = PeerShardedSearch(c, 0, 1, [0, c.scSize()], 64, torch)
        s.connect_local([s])                                 # shard window, counters
        c.sync()
        c.close()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()

    pynvml.nvmlInit()
    try:
        used = {}
        for k in range(1, 21):
            cycle()
            if k in (2, 20):
                used[k] = _process_gpu_bytes(pynvml)
                if used[k] is None:
                    pytest.skip("NVML does not report this process's device memory here")
        assert abs(used[20] - used[2]) <= 2 << 20, used
    finally:
        pynvml.nvmlShutdown()
