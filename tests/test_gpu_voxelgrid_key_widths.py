"""VoxelGrid at every key width, grid width and chunk length its implementations run with, against an exact model of PCL.

pcl_voxel_grid below restates pcl::VoxelGrid<PointXYZI>::applyFilter (PCL 1.10) in numpy: fp32 bounds, PCL's int32 guard on the
d = (int64)(extent * inv) + 1 product (the input is returned unchanged), min_b / div_b, the float index arithmetic, the index in
PCL's wrapping int stored as unsigned int and sorted unsigned, and centroids as sequential fp32 sums in ascending input index (the
canonical rule for PCL's unspecified intra-voxel order).  The guard bounds d while the index uses div_b, which can be one larger per
axis, so a cloud that passes it can have voxel indices past 2^31 and even past 2^32 (wrapped).

Every GPU case compares out, membership and keys bit for bit (uint32 views) on every path that can take the cloud: auto, the
multi-kernel radix path, the one-kernel cooperative path (k_vg_fused) at several grid widths, the one-CTA path (k_vg_small, n <= 3072),
the local map replayed from CUDA graphs, and the segmented path of the batched loop-closure ICP.  The clouds fix the largest voxel index
exactly (two corner points fix div_b) and carry intensities 2^24, 1, -2^24 in the three members of most voxels, so that any other
intra-voxel order changes a centroid bit."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

VGS_CAP = 3072                 # largest cloud of the one-CTA path (csrc/voxelgrid.cuh)
VGF_TILE = 1024                # points per tile of the one-kernel path
INT32_MAX = 2 ** 31 - 1


# ---------------------------------------------------------------------------------------------- the model
def pcl_voxel_grid(pts, leaf, reverse_sums=False):
    """(out, membership, keys) as oracle.voxel_grid returns them (keys None when the guard fires).  reverse_sums=True sums each voxel in
    descending input index instead: only for showing that the clouds below are sensitive to the intra-voxel order."""
    pts = np.ascontiguousarray(pts, np.float32).reshape(-1, 4)
    n = len(pts)
    if n == 0:
        return np.zeros((0, 4), np.float32), np.zeros(0, np.int32), np.zeros(0, np.int32)
    xyz = pts[:, :3]
    mn, mx = xyz.min(0), xyz.max(0)
    inv = np.float32(1.0) / np.float32(leaf)
    d = ((mx - mn) * inv).astype(np.int64) + 1
    if int(d[0]) * int(d[1]) * int(d[2]) > INT32_MAX:                      # "Leaf size is too small for the input dataset"
        return pts.copy(), np.arange(n, dtype=np.int32), None
    min_b = np.floor(mn * inv).astype(np.int64)
    div_b = np.floor(mx * inv).astype(np.int64) - min_b + 1
    ijk = (np.floor(xyz * inv) - min_b.astype(np.float32)).astype(np.int64)    # (int)(floor(p * inv) - (float)min_b), all in fp32
    idx = (ijk[:, 0] + ijk[:, 1] * div_b[0] + ijk[:, 2] * (div_b[0] * div_b[1])) & 0xFFFFFFFF
    idx = idx.astype(np.uint32)                                            # PCL's int, wrapped, stored as unsigned int
    order = np.argsort(idx, kind="stable")                                 # (unsigned index, input index)
    sk = idx[order]
    head = np.r_[True, sk[1:] != sk[:-1]]
    seg = np.cumsum(head) - 1
    nseg = int(seg[-1]) + 1
    starts = np.flatnonzero(head)
    count = np.diff(np.r_[starts, n])
    rank = np.arange(n) - starts[seg]                                      # position inside the voxel, in ascending input index
    if reverse_sums:
        rank = count[seg] - 1 - rank
    membership = np.empty(n, np.int32)
    membership[order] = seg
    acc = np.zeros((nseg, 4), np.float32)
    by_rank = np.argsort(rank, kind="stable")
    bounds = np.searchsorted(rank[by_rank], np.arange(int(count.max()) + 1))
    for k in range(int(count.max())):                                      # the k-th member of every voxel that has one, in fp32
        sel = by_rank[bounds[k]:bounds[k + 1]]
        acc[seg[sel]] += pts[order[sel]]
    out = acc / count.astype(np.float32)[:, None]
    return out, membership, sk[head].view(np.int32)


# ---------------------------------------------------------------------------------------------- the clouds
def make_cloud(n, leaf, lo_cells, hi_cells, seed):
    """n points whose bounds are exactly lo_cells * leaf and hi_cells * leaf (float cell coordinates; both corners are points of the
    cloud, the upper one the largest on every axis) and whose interior comes in triples of one voxel with intensities 2^24, 1, -2^24,
    the three members far apart in input order.  Coordinates are multiples of leaf / 8, so every product with 1 / leaf is exact."""
    lo = np.asarray(lo_cells, np.float64); hi = np.asarray(hi_cells, np.float64)
    rng = np.random.default_rng(seed)
    corners = np.array([[*lo, 7.0], [*hi, -3.0]])
    m = max(0, n - 2)
    q = (m + 2) // 3
    cell_lo = np.floor(lo); cell_hi = np.floor(hi)
    cells = cell_lo + np.floor(rng.random((q, 3)) * (cell_hi - cell_lo + 1))
    copies = []
    for inten in (2.0 ** 24, 1.0, -(2.0 ** 24)):
        p = cells + rng.integers(0, 8, (q, 3)) / 8.0
        p = np.clip(p, lo, hi)                                             # stays inside the bounds the corners fix
        copies.append(np.concatenate([p, np.full((q, 1), inten)], 1))
    body = np.concatenate(copies, 0)[:m]
    pts = np.concatenate([corners[:1], body, corners[1:]], 0)[:n] if n >= 2 else corners[:n]
    return (pts * np.array([leaf, leaf, leaf, 1.0])).astype(np.float32)


def box_cloud(n, div_b, leaf=0.25, origin=(-37, 5, -3), seed=0):
    """div_b exactly as given (corners on voxel faces: d == div_b): largest voxel index div_b product - 1"""
    o = np.asarray(origin, np.float64)
    return make_cloud(n, leaf, o, o + np.asarray(div_b) - 1, seed)


def key_width_cases():
    """largest index 2^k - 1 (div_b product 2^k) and 2^k (product 2^k + 1): 1 -> 2, 2 -> 3, 3 -> 4 passes of the one-kernel path's 8-bit
    digits and every boundary of the one-CTA path's 4-bit digits"""
    exact = {4: (4, 2, 2), 8: (16, 4, 4), 12: (16, 16, 16), 16: (64, 32, 32), 20: (128, 128, 64), 24: (256, 256, 256)}
    plus1 = {4: (17, 1, 1), 8: (257, 1, 1), 12: (241, 17, 1), 16: (65537, 1, 1), 20: (61681, 17, 1), 24: (673, 257, 97)}
    out = []
    for k in sorted(exact):
        out.append((f"max2^{k}-1", exact[k], 2 ** k - 1))
        out.append((f"max2^{k}", plus1[k], 2 ** k))
    return out


KEY_WIDTHS = key_width_cases()

# past 2^31 at leaf 1.0 (extents under one leaf more than d: div_b = d + 1 where the bounds cross a voxel face)
CUBE = dict(leaf=1.0, lo=(0.5, 0.5, 0.5), hi=(1290.25, 1290.25, 1290.25))          # d 1290^3 passes, div_b 1291^3: indices to 2^31 + 4.2 M
SLAB = dict(leaf=1.0, lo=(0.5, 0.5, 0.5), hi=(46340.25, 46341.25, 1.25))           # d 46340 x 46341 x 1 passes, div_b 46341 x 46342 x 2 > 2^32
PASS_MAX = dict(leaf=1.0, lo=(0.0, 0.0, 0.0), hi=(46339.0, 46340.0, 0.0))          # largest d product that passes: 46340 x 46341 x 1
TRIP_MIN = dict(leaf=1.0, lo=(0.0, 0.0, 0.0), hi=(46340.0, 46340.0, 0.0))          # smallest that trips the guard: 46341^2
WIDE = {"cube": CUBE, "slab": SLAB, "pass_max": PASS_MAX, "trip_min": TRIP_MIN}


def wide_cloud(name, n, seed=11, scale=1.0):
    c = WIDE[name]
    pts = make_cloud(n, c["leaf"], c["lo"], c["hi"], seed)
    pts[:, :3] *= np.float32(scale)
    return pts


def _u32(a):
    return np.ascontiguousarray(a).view(np.uint32)


def assert_same(got, want, what):
    g_out, g_mem, g_keys = got
    w_out, w_mem, w_keys = want
    assert g_out.shape == w_out.shape, (what, g_out.shape, w_out.shape)
    assert np.array_equal(_u32(g_mem), _u32(w_mem)), what
    assert np.array_equal(_u32(g_keys), _u32(w_keys)), what
    assert np.array_equal(_u32(g_out), _u32(w_out)), what


# ---------------------------------------------------------------------------------------------- CPU: the model against the oracle
def cpu_cases():
    cases = [(f"key{label}", box_cloud(3000, db, seed=i), 0.25) for i, (label, db, _) in enumerate(KEY_WIDTHS)]
    cases += [(f"{name}-{n}", wide_cloud(name, n), 1.0) for name in WIDE for n in (3000, 20000)]
    cases += [(f"n{n}", box_cloud(n, (200, 200, 20), seed=n), 0.25) for n in (1, 2, 3, 3072, 3073, 148 * 1024 + 1)]
    return cases


@pytest.mark.parametrize("case", cpu_cases(), ids=lambda c: c[0])
def test_model_equals_oracle(oracle, case):
    _, pts, leaf = case
    want = pcl_voxel_grid(pts, leaf)
    got = oracle.voxel_grid(pts, leaf)
    assert np.array_equal(_u32(got[0]), _u32(want[0])) and np.array_equal(got[1], want[1])
    if want[2] is None:
        assert got[2] is None
    else:
        assert np.array_equal(_u32(got[2]), _u32(want[2]))


def test_cases_reach_the_intended_indices():
    """the clouds have the largest voxel index they are named for, and the wide ones land on the intended side of the guard"""
    for i, (label, db, top) in enumerate(KEY_WIDTHS):
        _, _, keys = pcl_voxel_grid(box_cloud(3000, db, seed=i), 0.25)
        assert int(_u32(keys).max()) == top, label
        assert np.all(np.diff(_u32(keys).astype(np.int64)) > 0)
    _, _, keys = pcl_voxel_grid(wide_cloud("cube", 5000), 1.0)
    k = _u32(keys).astype(np.int64)
    assert k.max() == 1291 ** 3 - 1 and (k >= 2 ** 31).sum() >= 1 and (k < 2 ** 31).sum() >= 1
    _, _, keys = pcl_voxel_grid(wide_cloud("slab", 3000), 1.0)
    assert (46341 * 46342 * 2 - 1) - 2 ** 32 in set(_u32(keys).tolist())   # the upper corner's index wrapped past 2^32
    _, _, keys = pcl_voxel_grid(wide_cloud("pass_max", 3000), 1.0)
    assert keys is not None and int(_u32(keys).max()) == 46340 * 46341 - 1
    out, mem, keys = pcl_voxel_grid(wide_cloud("trip_min", 3000), 1.0)
    assert keys is None and len(out) == 3000


@pytest.mark.parametrize("name", ["key" + KEY_WIDTHS[-1][0], "cube", "slab"])
def test_model_is_sensitive_to_intra_voxel_order(name):
    pts = box_cloud(3000, KEY_WIDTHS[-1][1], seed=len(KEY_WIDTHS) - 1) if name.startswith("key") else wide_cloud(name, 3000)
    leaf = 0.25 if name.startswith("key") else 1.0
    fwd, mem, keys = pcl_voxel_grid(pts, leaf)
    rev, mem_r, keys_r = pcl_voxel_grid(pts, leaf, reverse_sums=True)
    assert np.array_equal(mem, mem_r) and np.array_equal(keys, keys_r)
    assert not np.array_equal(_u32(fwd), _u32(rev))


# ---------------------------------------------------------------------------------------------- GPU: every path of liorf_voxel_grid
def _max_coresident(ctx):
    """widest grid the width hook accepts (binary search; the hook refuses what cannot be co-resident)"""
    import liorf_b200
    lo, hi = 1, 1 << 16
    while lo < hi:
        mid = (lo + hi + 1) // 2
        try:
            ctx.debugVoxelGridGrid(mid); lo = mid
        except liorf_b200.api.LiorfError:
            hi = mid - 1
    ctx.debugVoxelGridGrid(0)
    return lo


def check_paths(ctx, pts, leaf, widths, want=None):
    """auto, multi-kernel, one-kernel at each width, one-CTA when n <= 3072 (that is auto's choice there)"""
    if want is None:
        want = pcl_voxel_grid(pts, leaf)
    if want[2] is None:                                                    # the guard: every point its own voxel, key = input index
        want = (want[0], want[1], np.arange(len(pts), dtype=np.int32))
    n = len(pts)
    bad = []                                                               # every path that differs, not only the first

    def one(what):
        try:
            assert_same(ctx.voxelGrid(pts, leaf), want, what)
        except AssertionError:
            bad.append(what)
    try:
        ctx.forceLargeVoxelGrid(False)
        one(("auto (one-CTA)" if n <= VGS_CAP else "auto", n))
        ctx.forceLargeVoxelGrid(True)
        one(("multi", n))
        ctx.forceFusedVoxelGrid(True)
        for g in widths:
            ctx.debugVoxelGridGrid(g)
            one(("fused", g, n))
    finally:
        ctx.forceFusedVoxelGrid(False)
        ctx.debugVoxelGridGrid(0)
    assert not bad, bad


@pytest.fixture(scope="module")
def gctx():
    import liorf_b200
    c = liorf_b200.Context()
    c.max_g = _max_coresident(c)
    yield c
    c.close()


def _widths(c):
    return sorted({1, 2, 3, 16, 148, c.max_g})


@pytest.mark.gpu
def test_width_hook_bounds(gctx):
    import liorf_b200
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert gctx.max_g >= 2 * sms                                           # k_vg_fused is built for two CTAs per SM
    for bad in (-1, gctx.max_g + 1):
        with pytest.raises(liorf_b200.api.LiorfError):
            gctx.debugVoxelGridGrid(bad)
    gctx.debugVoxelGridGrid(gctx.max_g); gctx.debugVoxelGridGrid(0)


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(KEY_WIDTHS)), ids=[k[0] for k in KEY_WIDTHS])
def test_key_widths(gctx, i):
    label, db, _ = KEY_WIDTHS[i]
    check_paths(gctx, box_cloud(3000, db, seed=i), 0.25, _widths(gctx))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3000, 20000])
@pytest.mark.parametrize("name", list(WIDE))
def test_past_2_31(gctx, name, n):
    check_paths(gctx, wide_cloud(name, n), 1.0, _widths(gctx))


def _size_cases():
    cases = []
    for g in ("1", "2", "3", "16", "148", "max"):
        for mult, add in ((1, -1), (1, 0), (1, 1), (3, 1), (4, 0), (4, 1)):
            cases.append((g, mult, add))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("g,mult,add", _size_cases(), ids=lambda v: str(v))
def test_fused_chunk_lengths(gctx, g, mult, add):
    """n = G x 1024 - 1 .. 4 G x 1024 + 1 on G CTAs: partial last tiles, chunks of 1 to 4 tiles and a partial tile inside a multi-tile
    chunk; auto runs the same width and switches to the multi-kernel path past four tiles per CTA"""
    G = gctx.max_g if g == "max" else int(g)
    n = mult * G * VGF_TILE + add
    pts = box_cloud(n, (200, 200, 20), seed=n)
    want = pcl_voxel_grid(pts, 0.25)
    try:
        gctx.debugVoxelGridGrid(G)
        assert_same(gctx.voxelGrid(pts, 0.25), want, ("auto", G, n))
        gctx.forceFusedVoxelGrid(True)
        assert_same(gctx.voxelGrid(pts, 0.25), want, ("fused", G, n))
    finally:
        gctx.forceFusedVoxelGrid(False)
        gctx.debugVoxelGridGrid(0)


@pytest.mark.gpu
def test_fused_more_than_four_tiles_per_cta(gctx):
    n = 6 * 16 * VGF_TILE + 517
    pts = box_cloud(n, (300, 200, 20), seed=3)
    check_paths(gctx, pts, 0.25, [16])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 3072, 3073])
def test_small_fused_boundary(gctx, n):
    check_paths(gctx, box_cloud(n, (200, 200, 20), seed=n), 0.25, [1, 148])


# ---------------------------------------------------------------------------------------------- GPU: the local map under graph replay
def _map_keyframes():
    """keyframe clouds of exact sizes: selections of them reach raw totals on both sides of each 64 k-point graph bucket"""
    sizes = [65535, 1, 2, 65536]
    kfs = []
    for k, n in enumerate(sizes):
        pts = box_cloud(n, (240, 240, 24), leaf=0.25, origin=(-120, -120, -8), seed=100 + k)
        pose = np.array([0.01 * k, -0.02 * k, 0.3 * k, 0.7 * k, -0.4 * k, 0.05 * k], np.float32)
        kfs.append((pts, pose))
    return kfs


MAP_SELECTIONS = {65535: [0], 65536: [0, 1], 65537: [0, 2], 131072: [3, 0, 1], 131073: [0, 3, 2], 131074: [0, 3, 2, 1]}


@pytest.mark.gpu
@pytest.mark.parametrize("grid", [None, "16", "148"])
def test_local_map_graph_replay(oracle, monkeypatch, grid):
    import liorf_b200
    if grid is None:
        monkeypatch.delenv("LIORF_MAP_VG_GRID", raising=False)
    else:
        monkeypatch.setenv("LIORF_MAP_VG_GRID", grid)                      # read when the context is created
    kfs = _map_keyframes()
    c = liorf_b200.Context()
    try:
        for cl, p in kfs:
            c.addKeyframeCloud(cl, p)
        leaf = liorf_b200.api.Params.default().surroundingKeyframeMapLeafSize
        want = {}
        for tot, sel in MAP_SELECTIONS.items():
            raw = np.concatenate([oracle.transform_cloud(kfs[i][0], kfs[i][1]) for i in sel], 0)
            assert len(raw) == tot
            want[tot] = pcl_voxel_grid(raw, leaf)[0]
        seq = [65535, 65537, 131073, 65536, 131072, 131074, 65535, 131073, 65537, 65536, 131074, 131072]
        for tot in seq:                                                    # each bucket captured once, replayed at other device-side counts
            m = c.extractSurroundingKeyFrames(MAP_SELECTIONS[tot])
            got = c.getLocalMap()
            assert m == len(want[tot]) and np.array_equal(_u32(got), _u32(want[tot])), (grid, tot)
    finally:
        c.close()


# ---------------------------------------------------------------------------------------------- GPU: the segmented path of the ICP batch
ICP_LEAF = 0.5


def _icp_keyframes():
    """cube and slab clouds scaled to the ICP leaf (sources of <= 3072 points take the one-CTA path in the single-pair call), an ordinary
    pair, and a slab's pass_max neighbour; every cloud passes the 300 / 1000 point guards after filtering"""
    s = ICP_LEAF
    kfs = [
        wide_cloud("cube", 3072, seed=21, scale=s),      # 0: source, range 1291^3
        wide_cloud("slab", 3072, seed=22, scale=s),      # 1: source, range past 2^32 on its own
        wide_cloud("cube", 6000, seed=23, scale=s),      # 2: target
        wide_cloud("slab", 6000, seed=24, scale=s),      # 3: target
        box_cloud(3072, (80, 80, 16), leaf=s, origin=(-40, -40, -8), seed=25),   # 4: ordinary
        box_cloud(6000, (80, 80, 16), leaf=s, origin=(-40, -40, -8), seed=26),   # 5: ordinary
        wide_cloud("pass_max", 6000, seed=27, scale=s),  # 6: target, range just under 2^31
    ]
    return [(k, np.zeros(6, np.float32)) for k in kfs]


@pytest.mark.gpu
def test_icp_batch_past_2_32(oracle):
    import liorf_b200
    kfs = _icp_keyframes()
    c = liorf_b200.Context()
    try:
        for cl, p in kfs:
            c.addKeyframeCloud(cl, p)
        iters = 5
        single = {}

        def one(cu, pr, li):
            if (cu, pr, li) not in single:
                r = c.loopClosureICP(cu, pr, 0, li, icp_leaf=ICP_LEAF, max_iters=iters)
                src, tgt = c.icpClouds(r.n_source, r.n_target)
                pose = lambda k: kfs[li if li != -1 else k][1]
                w_src = pcl_voxel_grid(oracle.transform_cloud(kfs[cu][0], pose(cu)), ICP_LEAF)[0]
                w_tgt = pcl_voxel_grid(oracle.transform_cloud(kfs[pr][0], pose(pr)), ICP_LEAF)[0]
                assert np.array_equal(_u32(src), _u32(w_src)) and np.array_equal(_u32(tgt), _u32(w_tgt)), (cu, pr, li)
                assert r.ran == 1, (cu, pr, li, r.n_source, r.n_target)
                single[(cu, pr, li)] = bytes(r)
            return single[(cu, pr, li)]

        def batch(pairs):
            cur, pre, li = (np.array([p[i] for p in pairs], np.int32) for i in range(3))
            res = c.loopClosureICPBatch(cur, pre, li, history_search_num=0, icp_leaf=ICP_LEAF, max_iters=iters)
            for p, r in zip(pairs, res):
                assert bytes(r) == one(*p), p

        batch([(0, 2, -1)])                              # one pair: 2 x 1291^3 > 2^32
        batch([(1, 6, -1)])                              # one pair: the slab's wrapped range alone passes 2^32
        batch([(4, 5, -1), (0, 2, -1), (1, 3, 0), (5, 4, -1), (0, 6, -1), (4, 2, -1), (1, 5, -1), (4, 5, 0)])   # halved down to single pairs
        batch([(4, 5, -1), (5, 4, -1), (4, 6, -1)])      # ordinary pairs, one beside a range near 2^31: no split
    finally:
        c.close()
