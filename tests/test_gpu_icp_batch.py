"""Batched loop-closure verification (liorf_loop_closure_icp_batch): every pair of a batch must equal liorf_loop_closure_icp on the same
pair bit for bit, whatever the batch's size, order or grouping into waves; checked here on a keyframe store built to reach every
branch — true revisits and wrong places, a keyframe 500 m away (no correspondence), clouds below either size guard, a dense keyframe
that needs the in-pair grid-stride loop, and a cloud that trips PCL's int32 VoxelGrid guard."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

N_STREET = 20
KF_REV_A, KF_REV_B, KF_FAR, KF_SMALL, KF_DENSE = 20, 21, 22, 23, 24


def _lattice():
    """160 000 points on 0.5 m voxel centres (80 x 80 x 25): more than 4 x 148 x 256 = 151 552 voxels survive the ICP leaf."""
    g = (np.arange(80, dtype=np.float32) + 0.5) * 0.5 - 20.0
    gz = (np.arange(25, dtype=np.float32) + 0.5) * 0.5 - 2.0
    x, y, z = np.meshgrid(g, g, gz, indexing="ij")
    return np.stack([x.ravel(), y.ravel(), z.ravel(), np.zeros(x.size, np.float32)], 1).astype(np.float32)


@pytest.fixture(scope="module")
def store(synth, oracle):
    kfs = []
    for k in range(N_STREET):
        p = np.array([0, 0, 0, 1.0 * k, 0, 0], np.float64)
        ds, _, _ = oracle.voxel_grid(synth.raw_to_xyzi(synth.scan(synth.HDL64, p, seed=900 + k)), 0.4)
        kfs.append((ds, p.astype(np.float32)))
    for true_x, seed, drift in ((4.0, 990, (0, 0, np.deg2rad(2.0), 4.6, -0.4, 0.0)), (12.0, 991, (0, 0, np.deg2rad(-1.5), 11.5, 0.3, 0.0))):
        ds, _, _ = oracle.voxel_grid(synth.raw_to_xyzi(synth.scan(synth.HDL64, np.array([0, 0, 0, true_x, 0, 0], np.float64), seed=seed)), 0.4)
        kfs.append((ds, np.array(drift, np.float32)))                                   # revisits with odometry drift
    kfs.append((kfs[3][0], np.array([0, 0, 0, 500.0, 0, 0], np.float32)))              # 500 m away: nothing within max_corr_dist
    kfs.append((kfs[5][0][:200].copy(), kfs[5][1]))                                     # below the source guard
    kfs.append((_lattice(), np.array([0, 0, 0, 10.0, 0, 0], np.float32)))               # dense: > 151 552 points after the ICP leaf
    return kfs


def _ctx(kfs):
    import liorf_b200
    c = liorf_b200.Context()
    for cl, p in kfs:
        c.addKeyframeCloud(cl, p)
    return c


def _pairs():
    L = []
    L += [(KF_REV_A, 4, -1), (KF_REV_B, 12, -1), (KF_REV_A, 4, 0), (KF_REV_B, 12, 0), (KF_REV_A, 4, 3), (KF_REV_B, 12, KF_REV_A)]   # true loops
    L += [(KF_REV_A, 15, -1), (KF_REV_B, 2, 0), (9, 17, -1), (3, 11, 7)]                                        # wrong places
    L += [(KF_FAR, 10, -1), (KF_FAR, 10, 0), (KF_FAR, KF_FAR, -1)]                                           # far / no correspondence
    L += [(KF_SMALL, 5, -1), (KF_SMALL, 5, 0), (5, KF_SMALL, -1), (6, KF_SMALL, 0)]                          # guards on either side
    L += [(KF_DENSE, 10, -1), (KF_DENSE, 10, 0)]                                                              # in-pair grid stride
    L += [(0, 1, -1), (1, 0, 0), (KF_DENSE, N_STREET - 1, -1), (N_STREET - 1, KF_DENSE, 0), (2, 24, -1)]     # windows clipped at both ends
    L += [(7, 7, 0), (KF_REV_A, KF_REV_A, -1), (KF_REV_A, 4, -1), (KF_REV_B, 12, -1), (KF_SMALL, 5, -1)]     # cur == pre, duplicates
    L += [(k, (k + 6) % N_STREET, -1 if k % 2 else 0) for k in range(0, N_STREET, 2)]                        # more mixed pairs
    return L


def _batch(c, pairs, hs, iters, **kw):
    cur, pre, li = (np.array([p[i] for p in pairs], np.int32) for i in range(3))
    return list(c.loopClosureICPBatch(cur, pre, li, history_search_num=hs, max_iters=iters, **kw))


@pytest.fixture(scope="module")
def runs(store):
    """every (history_search_num, max_iters) batch of the mixed pair list, with the single-pair call on each pair"""
    c = _ctx(store)
    pairs = _pairs()
    out = {}
    for hs in (0, 2, 25):
        for iters in (3, 100):
            b = _batch(c, pairs, hs, iters)
            s = [c.loopClosureICP(cu, pr, hs, li, max_iters=iters) for cu, pr, li in pairs]
            out[(hs, iters)] = (b, s)
    c.close()
    return pairs, out


def test_batch_is_bit_identical_to_single_pair_calls(runs):
    pairs, out = runs
    states = {}
    guard_src = guard_tgt = 0
    spread = 0
    for (hs, iters), (b, s) in out.items():
        assert len(b) == len(s) == len(pairs)
        for p, (rb, rs) in enumerate(zip(b, s)):
            assert bytes(rb) == bytes(rs), (hs, iters, pairs[p], [(f, getattr(rb, f), getattr(rs, f)) for f, _ in type(rb)._fields_])
        ran = [r for r in b if r.ran]
        for r in b:
            if not r.ran:
                guard_src += r.n_source < 300
                guard_tgt += r.n_source >= 300 and r.n_target < 1000
        for r in ran:
            states.setdefault((iters, r.convergence_state), 0)
            states[(iters, r.convergence_state)] += 1
        if ran:
            its = [r.iterations for r in ran]
            spread = max(spread, max(its) - min(its))
        print(f"hs={hs:2d} max_iters={iters:3d}: ran {len(ran)}/{len(b)}, iterations {sorted(set(r.iterations for r in ran))}, "
              f"states {sorted(set(r.convergence_state for r in ran))}, n_source max {max(r.n_source for r in b)}")
    print("states (max_iters, state) -> count:", states, "| guard failures source/target:", guard_src, guard_tgt, "| iteration spread:", spread)
    assert guard_src > 0 and guard_tgt > 0
    assert any(st == 5 for (_, st) in states)
    assert states.get((3, 1), 0) > 0
    assert any(states.get((100, st), 0) > 0 for st in (2, 3, 4))
    assert spread >= 5
    assert max(r.n_source for (b, _) in out.values() for r in b if r.ran) > 4 * 148 * 256      # the in-pair grid-stride loop ran


def test_batch_results_do_not_depend_on_order_or_waves(store):
    c = _ctx(store)
    pairs = _pairs()
    ref = [bytes(r) for r in _batch(c, pairs, 2, 100)]
    rev = [bytes(r) for r in _batch(c, pairs[::-1], 2, 100)][::-1]
    assert rev == ref
    for w in (1, 3, 7):
        c.debugIcpBatchWave(w)
        assert [bytes(r) for r in _batch(c, pairs, 2, 100)] == ref, w
    c.debugIcpBatchWave(0)
    c.close()


def test_segment_past_the_int32_voxel_guard(store):
    """A cloud spanning 2 km x 2 km x 100 m trips PCL's "leaf size too small" guard at 0.5 m (passes through unfiltered) while the
    clouds next to it in the same VoxelGrid pass are filtered normally."""
    rng = np.random.default_rng(5)
    huge = np.concatenate([rng.uniform(-1000, 1000, (3000, 2)), rng.uniform(0, 100, (3000, 1)), np.zeros((3000, 1))], 1).astype(np.float32)
    kfs = store[:6] + [(huge, np.zeros(6, np.float32))]
    c = _ctx(kfs)
    pairs = [(2, 4, -1), (6, 6, -1), (6, 3, 0), (3, 6, -1), (1, 5, 0)]
    b = _batch(c, pairs, 0, 100)
    for (cu, pr, li), rb in zip(pairs, b):
        rs = c.loopClosureICP(cu, pr, 0, li, max_iters=100)
        assert bytes(rb) == bytes(rs), (cu, pr, li)
    assert b[1].ran == 1 and b[1].n_source == b[1].n_target == len(huge)        # unfiltered
    assert b[0].n_source < len(store[2][0])                                      # filtered
    c.close()


def _rot_err(Ta, Tb):
    """angle of Ta Tb^T from its skew part (well conditioned for small angles, unlike arccos of the trace)"""
    R = Ta[:3, :3].astype(np.float64) @ Tb[:3, :3].astype(np.float64).T
    v = 0.5 * np.array([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]])
    return float(np.arcsin(min(1.0, np.linalg.norm(v))))


def test_batch_matches_oracle(store, oracle):
    import pyicp
    c = _ctx(store)
    pairs = [(KF_REV_A, 4, -1), (KF_REV_B, 12, -1), (KF_REV_A, 4, 0)]
    b = _batch(c, pairs, 2, 100)
    clouds, poses = [k[0] for k in store], [k[1] for k in store]
    for (cu, pr, li), r in zip(pairs, b):
        o_src = pyicp.loop_find_near_keyframes(clouds, poses, cu, 0, li, 0.5, oracle)
        o_tgt = pyicp.loop_find_near_keyframes(clouds, poses, pr, 2, li, 0.5, oracle)
        rs = c.loopClosureICP(cu, pr, 2, li)                       # the same pair alone: its clouds are the batch's (bit-identical results)
        src, tgt = c.icpClouds(rs.n_source, rs.n_target)
        assert bytes(rs) == bytes(r)
        assert r.n_source == len(o_src) and r.n_target == len(o_tgt)
        assert np.array_equal(src, o_src) and np.array_equal(tgt, o_tgt)
        o = pyicp.icp(o_src, o_tgt, 20.0, 100)
        T = np.array(r.transform[:], np.float32).reshape(4, 4)
        assert r.ran == 1 and r.converged == int(o["converged"])
        assert abs(r.iterations - o["iterations"]) <= 1
        assert np.max(np.abs(T[:3, 3] - o["transform"][:3, 3])) < 1e-4 and _rot_err(T, o["transform"]) < 1e-5
        assert abs(r.fitness - o["fitness"]) < 1e-3 * max(o["fitness"], 1e-3)
    c.close()


def test_batch_leaves_the_single_pair_clouds_and_the_pipeline_alone(store):
    c = _ctx(store)
    rs = c.loopClosureICP(KF_REV_A, 4, 2, -1)
    src0, tgt0 = c.icpClouds(rs.n_source, rs.n_target)
    _batch(c, _pairs(), 25, 100)
    src1, tgt1 = c.icpClouds(rs.n_source, rs.n_target)
    assert np.array_equal(src0, src1) and np.array_equal(tgt0, tgt1)
    c.close()

    import bench
    n = 14
    seq = bench.Sequence(n, 0)
    a = bench.GpuPipeline(seq, 0); b = bench.GpuPipeline(seq, 0)
    a.stage(range(n)); b.stage(range(n))
    outs = []
    for pipe, verify in ((a, False), (b, True)):
        fos = []
        for i in range(n):
            guess = seq.initial_guess(i, pipe.prev)
            nxt = pipe._frame_in(i + 1, "dev") if (i + 1) in pipe.dev_raw else None
            fo = pipe.ctx.processFrameIn(pipe._frame_in(i, "dev"), guess, nxt)
            pipe.prev = np.array(fo.pose[:], np.float32)
            fos.append(bytes(fo))
            k = pipe.ctx.numKeyframes()
            if verify and k > 0:
                cur = np.arange(k, dtype=np.int32)
                res = pipe.ctx.loopClosureICPBatch(cur, cur[::-1].copy(), np.zeros(k, np.int32), history_search_num=2)
                assert len(res) == k
        outs.append(fos)
    assert outs[0] == outs[1]
    assert a.ctx.numKeyframes() == b.ctx.numKeyframes() > 2
    for k in range(a.ctx.numKeyframes()):
        ca, pa, ta = a.ctx.getKeyframe(k); cb, pb, tb = b.ctx.getKeyframe(k)
        assert np.array_equal(ca, cb) and np.array_equal(pa, pb) and ta == tb
    a.ctx.close(); b.ctx.close()


def test_batch_arguments(store):
    import ctypes as C
    import liorf_b200
    c = _ctx(store[:4])
    assert len(c.loopClosureICPBatch([], [], [])) == 0
    lib = c.lib
    out = (liorf_b200.api.IcpResult * 3)()
    C.memset(out, 0x5a, C.sizeof(out))
    before = bytes(out)
    cur = (C.c_int * 3)(0, 1, 4); pre = (C.c_int * 3)(1, 2, 0); li = (C.c_int * 3)(-1, 0, 0)
    f = lib.liorf_loop_closure_icp_batch
    args = lambda cu, pr, l, n, hs=2, leaf=0.5, mcd=20.0, it=100, o=out: f(c.h, cu, pr, l, C.c_int(n), C.c_int(hs), C.c_float(leaf), C.c_float(mcd), C.c_int(it), o)
    assert args(cur, pre, li, 3) == -2 and bytes(out) == before                  # key 4 of 4 keyframes, at the end of a valid batch
    li_bad = (C.c_int * 3)(-1, 0, -2)
    cur_ok = (C.c_int * 3)(0, 1, 3)
    assert args(cur_ok, pre, li_bad, 3) == -2 and bytes(out) == before          # loop_index -2
    assert args(None, pre, li, 3) == -2 and args(cur_ok, None, li, 3) == -2 and args(cur_ok, pre, None, 3) == -2
    assert args(cur_ok, pre, li, 3, o=None) == -2
    assert args(cur_ok, pre, li, 3, hs=-1) == -2 and args(cur_ok, pre, li, 3, leaf=0.0) == -2 and args(cur_ok, pre, li, 3, mcd=0.0) == -2
    assert args(cur_ok, pre, li, 3, it=0) == -2 and args(cur_ok, pre, li, -1) == -2
    assert bytes(out) == before
    assert args(None, None, None, 0, o=None) == 0                                 # an empty batch needs no arrays
    assert args(cur_ok, pre, li, 3) == 0 and bytes(out) != before
    c.close()
