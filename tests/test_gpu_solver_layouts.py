"""The persistent scan-to-map solver (k_scan2map_persistent, liorf_b200/csrc/scan2map.cuh) at every layout it can choose.

The layout follows from the downsampled scan size n and the number of worker CTAs W = CTAs - 1:
  one round       n <= W * 128              per-query state in registers and shared memory
  global state    n >  W * 128              per-query state in global memory, rounds = ceil(n / (W * 512)); each worker loops over
                                            the rounds and carries its fp64 partial sums across them
The per-function calls launch one CTA per SM, liorf_process_frame SPARE_SMS fewer; liorf_debug_s2m_grid (Context.solverGrid) sets
the width of both, so that small widths reach the multi-round layouts on ordinary scans.  Every solve is compared with the CPU
oracle iteration by iteration (north-star tolerance, 1e-4 m / 1e-5 rad; selected-row counts within 3), and the caches and forced
global state must not change a bit.  The module records the (CTAs, n) of every solve and checks at the end that together they
reached each layout."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

QPB, QPB_GLOBAL = 128, 512          # S2MP_QPB / S2MP_QPB_GLOBAL: queries per worker and round, one-round / global-state layout
SPARE_SMS = 16                      # S2M_SPARE_SMS (capi.cu): the SMs liorf_process_frame's solver leaves to the next frame's front end
POS_TOL, ROT_TOL = 1e-4, 1e-5
RUNS = set()                        # (CTAs, n, forced global state) of every solve of this module


def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def resolve(ctas):
    """'sms' / 'sms-16' / an int -> a CTA count (skips a width the device cannot hold)"""
    v = {"sms": num_sms(), "sms-16": num_sms() - SPARE_SMS}.get(ctas, ctas)
    if v > num_sms():
        pytest.skip(f"{v} CTAs > {num_sms()} SMs")
    return v


def layout(ctas, n, global_state=False):
    """the kernel's own choice: (workers, one-round layout?, rounds)"""
    W = ctas - 1
    one = not global_state and n <= W * QPB
    return W, one, 1 if one else -(-n // (W * QPB_GLOBAL))


def solve(c, ctas, n, init, iters, cache=True, global_state=False):
    """one forced-iteration solve on `ctas` CTAs; returns (final pose, per-iteration poses, selected-row counts, trace)"""
    c.solverGrid(ctas); c.disableSolverCache(not cache); c.solverGlobalState(global_state)
    c.setLMState(0, np.eye(6, dtype=np.float32))
    pose, tr = c.scan2MapOptimization(init, iters, force_all_iters=True)
    c.solverGrid(0); c.disableSolverCache(False); c.solverGlobalState(False)
    RUNS.add((ctas or num_sms(), n, global_state))                  # 0: the per-function default, one CTA per SM
    return pose, tr.poses().copy(), tr.nsels().copy(), tr


def assert_matches_oracle(run, o, iters):
    _, poses, nsel, tr = run
    assert tr.ran == 1 and tr.iters == iters == o["iters"]
    dpos = np.max(np.abs(poses[:, 3:] - o["trace"][:, 3:]), axis=1)
    drot = np.max(np.abs(poses[:, :3] - o["trace"][:, :3]), axis=1)
    assert dpos.max() < POS_TOL and drot.max() < ROT_TOL, (np.argmax(dpos > POS_TOL), dpos, drot)
    assert np.max(np.abs(nsel.astype(int) - o["nsel"].astype(int))) <= 3, (nsel, o["nsel"])


def assert_first_selection_exact(c, run, init, n):
    """Iteration 0 runs at the start pose in every layout, and which rows it selects depends on the query alone: their number equals,
    exactly, the selected flags of the per-function surfOptimization kernel at that pose.  (The oracle's count may differ by a few
    borderline points: its pointSel comes from host trig.)  A query that a round skips or counts twice shows up here."""
    assert run[2][0] == int(c.surfOptimization(init, n)["flag"].sum())


def assert_same_bits(a, b):
    assert np.array_equal(a[2], b[2]), (a[2], b[2])
    assert np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32))
    assert np.array_equal(a[0].view(np.uint32), b[0].view(np.uint32))


def near(pose, truth):
    return np.linalg.norm(pose[3:] - truth[3:]) < 0.05


@pytest.fixture(scope="module")
def kitti(oracle, kitti_case):
    """kitti_case's local map (oracle VoxelGrid, 0.5 m) and the device's downsampled scan"""
    import liorf_b200
    raw = np.concatenate([oracle.transform_cloud(cl, p) for cl, p in kitti_case["keyframes"]])
    o_map, _, _ = oracle.voxel_grid(raw, 0.5)
    c = liorf_b200.Context()
    c.setLocalMap(o_map); c.setCurrentScan(kitti_case["scan"])
    ds, _ = c.downsampleCurrentScan(len(kitti_case["scan"]))
    c.close()
    return dict(map=o_map, ds=ds, init=kitti_case["init"], truth=kitti_case["truth"])


def kitti_ctx(kitti, scan):
    """a context holding the kitti map and `scan` as the current scan; returns (context, device-downsampled scan)"""
    import liorf_b200
    c = liorf_b200.Context()
    c.setLocalMap(kitti["map"]); c.setCurrentScan(scan)
    ds, _ = c.downsampleCurrentScan(len(scan))
    return c, ds


def subset(ds, n):
    """n points of the downsampled scan, evenly spaced through it.  Each is its own voxel's centroid, so downsampling them again keeps
    exactly these n.  (A prefix would be one slab of the voxel-key order, ground points only.)"""
    idx = np.round(np.linspace(0, len(ds) - 1, n)).astype(int)
    assert len(np.unique(idx)) == n
    return ds[idx]


# ---------------------------------------------------------------------------------------------- a. grid sweep
@pytest.fixture(scope="module")
def kitti_oracle(oracle, kitti):
    return oracle.scan2map(kitti["ds"], kitti["map"], kitti["init"], 30, force_all=True)


@pytest.mark.parametrize("ctas", [2, 3, 9, 17, 34, 101, "sms-16", "sms"])
def test_grid_sweep(kitti, kitti_oracle, ctas):
    """The whole kitti_case scan at widths from one worker (15 rounds) to the full device (one round): every iteration against the
    oracle, and the caches off / the global layout forced give the same trace bit for bit."""
    ctas = resolve(ctas)
    c, ds = kitti_ctx(kitti, kitti["ds"])
    n = len(ds)
    base = solve(c, ctas, n, kitti["init"], 30)
    assert_matches_oracle(base, kitti_oracle, 30)
    assert_first_selection_exact(c, base, kitti["init"], n)
    assert near(base[0], kitti["truth"])
    assert_same_bits(solve(c, ctas, n, kitti["init"], 30, cache=False), base)
    if layout(ctas, n)[1]:
        assert_same_bits(solve(c, ctas, n, kitti["init"], 30, global_state=True), base)
    c.close()


# ---------------------------------------------------------------------------------------------- b. exact layout boundaries
EDGES = {"W*128": lambda W: W * QPB, "W*128+1": lambda W: W * QPB + 1, "W*512": lambda W: W * QPB_GLOBAL, "W*512+1": lambda W: W * QPB_GLOBAL + 1}


def run_subset(oracle, kitti, ctas, n):
    """n points of the kitti scan on `ctas` CTAs: oracle check and cache on / off bit identity.  Subsets of a street scan are degenerate
    along the street (the start pose's offset there is unobservable), so the final pose is compared with the oracle's only."""
    c, ds = kitti_ctx(kitti, subset(kitti["ds"], n))
    assert len(ds) == n
    o = oracle.scan2map(ds, kitti["map"], kitti["init"], 30, force_all=True)
    base = solve(c, ctas, n, kitti["init"], 30)
    assert_matches_oracle(base, o, 30)
    assert_first_selection_exact(c, base, kitti["init"], n)
    assert_same_bits(solve(c, ctas, n, kitti["init"], 30, cache=False), base)
    c.close()


@pytest.mark.parametrize("edge", list(EDGES))
@pytest.mark.parametrize("ctas", [2, 9])
def test_layout_boundaries(oracle, kitti, ctas, edge):
    """n exactly on and one past the one-round limit (W * 128) and the one-global-round limit (W * 512)."""
    n = EDGES[edge](ctas - 1)
    W, one, rounds = layout(ctas, n)
    assert (one, rounds) == {"W*128": (True, 1), "W*128+1": (False, 1), "W*512": (False, 1), "W*512+1": (False, 2)}[edge]
    run_subset(oracle, kitti, ctas, n)


@pytest.mark.parametrize("n", [31, 97])
def test_scans_smaller_than_the_grid(oracle, kitti, n):
    """Fewer queries than workers on the full-device grid: most workers are idle and send zero partial sums.  31 is the smallest scan
    the solver runs on (n > 30, :1300); below 50 selected rows the LM step leaves the pose alone (:1178)."""
    ctas = resolve("sms")
    assert n < ctas - 1
    run_subset(oracle, kitti, ctas, n)


# ---------------------------------------------------------------------------------------------- c. multi-round at the default grids
def dense_scene(rng):
    """A 32 m x 32 m hall (floor, four 4 m walls, twelve pillars) as a 0.5 m lattice map and a dense scan of the same surfaces seen from
    `truth`: at a 0.1 m leaf the scan keeps ~165 k points, three global rounds on 147 or 131 workers."""
    rects = [((-16, -16, -1.5), (1, 0, 0), (0, 1, 0), 32, 32)]                    # (origin, u, v, length along u, length along v)
    for o, u in (((-16, -16, -1.5), (1, 0, 0)), ((-16, 16, -1.5), (1, 0, 0)), ((-16, -16, -1.5), (0, 1, 0)), ((16, -16, -1.5), (0, 1, 0))):
        rects.append((o, u, (0, 0, 1), 32, 4))
    for px, py in rng.uniform(-11, 11, size=(12, 2)):
        for o, u in (((px, py, -1.5), (1, 0, 0)), ((px, py + 1.2, -1.5), (1, 0, 0)), ((px, py, -1.5), (0, 1, 0)), ((px + 1.2, py, -1.5), (0, 1, 0))):
            rects.append((o, u, (0, 0, 1), 1.2, 2.5))
        rects.append(((px, py, 1.0), (1, 0, 0), (0, 1, 0), 1.2, 1.2))

    def sample(step=None, density=None):
        out = []
        for o, u, v, lu, lv in rects:
            if step is not None:
                a, b = (g.ravel() for g in np.meshgrid(np.arange(0, lu, step), np.arange(0, lv, step)))
            else:
                a, b = rng.uniform(0, lu, int(density * lu * lv)), rng.uniform(0, lv, int(density * lu * lv))
            out.append(np.asarray(o) + a[:, None] * np.asarray(u) + b[:, None] * np.asarray(v))
        p = np.concatenate(out)
        p[:, 2] += 0.03 * np.sin(0.7 * p[:, 0]) * np.cos(0.5 * p[:, 1])          # gently curved: no surface lies on a voxel boundary
        return p

    mp = sample(step=0.5)
    mp += rng.normal(scale=0.005, size=mp.shape)
    mp = np.concatenate([mp, np.zeros((len(mp), 1))], 1).astype(np.float32)
    world = sample(density=330)
    truth = np.array([0.01, -0.02, 0.03, 0.2, -0.1, 0.05], np.float32)
    from bench import pose_to_T
    Ti = np.linalg.inv(pose_to_T(truth.astype(np.float64)))
    scan = np.concatenate([world @ Ti[:3, :3].T + Ti[:3, 3], np.ones((len(world), 1))], 1).astype(np.float32)
    init = (truth + np.array([0.004, -0.003, 0.01, 0.12, 0.08, -0.03], np.float32)).astype(np.float32)
    return mp, scan, truth, init


DENSE_ITERS = 10                    # the oracle's 5-NN is a brute-force scan of the map: ten forced iterations keep it to seconds


@pytest.fixture(scope="module")
def dense(oracle):
    import liorf_b200
    mp, scan, truth, init = dense_scene(np.random.default_rng(31))
    c = liorf_b200.Context(mappingSurfLeafSize=0.1)
    c.reserve(len(scan), len(mp))
    c.setLocalMap(mp); c.setCurrentScan(scan)
    ds, n = c.downsampleCurrentScan(len(scan))
    o = oracle.scan2map(ds, mp, init, DENSE_ITERS, force_all=True)
    yield dict(ctx=c, n=n, o=o, truth=truth, init=init)
    c.close()


@pytest.mark.parametrize("ctas", ["sms", "sms-16"])
def test_multi_round_at_default_widths(dense, ctas):
    """A scan of ~165 k points runs three global rounds at both production widths: the per-function grid with no hook at all, and
    liorf_process_frame's width through the hook."""
    n, c = dense["n"], dense["ctx"]
    w = resolve(ctas)
    W, one, rounds = layout(w, n)
    assert rounds >= 3 and n % (W * QPB_GLOBAL), (n, W, rounds)
    hook = 0 if ctas == "sms" else w
    base = solve(c, hook, n, dense["init"], DENSE_ITERS)
    assert_matches_oracle(base, dense["o"], DENSE_ITERS)
    assert_first_selection_exact(c, base, dense["init"], n)
    assert near(base[0], dense["truth"])
    assert_same_bits(solve(c, w, n, dense["init"], DENSE_ITERS, cache=False), base)


# ---------------------------------------------------------------------------------------------- d. liorf_process_frame
N_FRAMES = 14


@pytest.fixture(scope="module")
def drive(synth, oracle):
    import bench
    seq = bench.Sequence(N_FRAMES, 0)
    for i in range(N_FRAMES):
        seq.frame(i)
    return bench, seq


@pytest.mark.parametrize("ctas", ["sms-16", 5])
def test_process_frame_at_pinned_widths(drive, ctas):
    """The 14-frame drive through liorf_process_frame (with look-ahead) against the same frames through the per-function calls on a
    solver of the same width, and against the oracle pipeline.  "sms-16": liorf_process_frame at its own default width, the stepwise
    context pinned to it, so the two are equal by construction.  5 CTAs on both: every frame's solve runs two or three global rounds."""
    bench, seq = drive
    import liorf_b200
    w = resolve(ctas)
    a = bench.GpuPipeline(seq, 0)
    a.stage(range(N_FRAMES))
    if ctas != "sms-16":
        a.ctx.solverGrid(w)
    c = liorf_b200.Context(**{k: seq.filters[k] for k in ("N_SCAN", "downsampleRate", "point_filter_num", "lidarMinRange", "lidarMaxRange")})
    c.solverGrid(w)
    cpu = bench.CpuPipeline(seq)
    for i in range(N_FRAMES):
        raw, (t0, it, rot, ptr) = seq.frame(i)
        guess = seq.initial_guess(i, cpu.prev)                      # all three start every frame from the oracle chain's guess
        a.prev = cpu.prev
        pa = a.step(i, "dev", lookahead=True)
        c.projectPointCloud(raw, t0, it, rot, ptr, True, want_output=False)
        c.downsampleCurrentScan(want_output=False)
        if c.numKeyframes() > 0:
            c.extractSurroundingKeyFrames(c.extractNearby(t0, 2.0), want_count=False)
        c.scan2MapOptimizationAsync(guess, 30, False)
        pc = c.getPose()
        if c.saveFrame(pc, 1.0, 0.2):
            c.addKeyframe(pc, t0)
            c.makeAndSaveScancontextAndKeys()
        if i % 10 == 9:
            c.detectLoopClosureID()
        po = cpu.step(i)
        assert np.array_equal(pa.view(np.uint32), pc.view(np.uint32)), (i, pa, pc)
        assert np.max(np.abs(pa[3:] - po[3:])) < POS_TOL and np.max(np.abs(pa[:3] - po[:3])) < ROT_TOL, (i, pa, po)
        assert a.ctx.numKeyframes() == c.numKeyframes() == len(cpu.kf_clouds), i
        n = a.ctx.lastCounts()["n_ds"]
        if i > 0:
            RUNS.add((w, n, False))
            if ctas == 5:
                assert layout(w, n)[2] >= 2, (i, n)
    a.ctx.close(); c.close()


# ---------------------------------------------------------------------------------------------- e. the iteration clamp
def test_iteration_clamp_and_epoch_stride(oracle, kitti):
    """64 forced iterations (S2M_MAX_ITERS) against the oracle; 80 requested come back as 64.  A launch of 64 iterations uses every
    epoch up to the next launch's first one, so back-to-back launches on one context must give the trace of a fresh context."""
    c, ds = kitti_ctx(kitti, kitti["ds"][::4])
    n = len(ds)
    o = oracle.scan2map(ds, kitti["map"], kitti["init"], 64, force_all=True)
    first = solve(c, 0, n, kitti["init"], 64)
    assert len(first[1]) == 64
    assert_matches_oracle(first, o, 64)
    assert_first_selection_exact(c, first, kitti["init"], n)
    assert near(first[0], kitti["truth"])
    second = solve(c, 0, n, kitti["init"], 64)
    clamped = solve(c, 0, n, kitti["init"], 80)
    assert clamped[3].iters == 64
    f, _ = kitti_ctx(kitti, kitti["ds"][::4])
    fresh = solve(f, 0, n, kitti["init"], 64)
    for r in (second, clamped, first):
        assert_same_bits(r, fresh)
    c.close(); f.close()


def test_hook_rejects_widths_the_device_cannot_hold():
    """the cooperative launch needs every CTA resident at once, one per SM, and the solver needs a worker and the reducer"""
    import liorf_b200
    from liorf_b200.api import LiorfError
    c = liorf_b200.Context()
    for bad in (-1, 1, num_sms() + 1):
        with pytest.raises(LiorfError):
            c.solverGrid(bad)
    c.solverGrid(2); c.solverGrid(num_sms()); c.solverGrid(0)
    c.close()


# ---------------------------------------------------------------------------------------------- coverage of this module
def test_layout_coverage(capsys):
    """Runs last: the solves above reached every layout."""
    runs = sorted(RUNS)
    hits = {"one round": [], "global state, 1 round": [], "2 rounds": [], ">= 3 rounds, partial last round": [], "W = 1": [], "n < W": []}
    for ctas, n, g in runs:
        W, one, rounds = layout(ctas, n, g)
        if one:
            hits["one round"].append((ctas, n))
        elif rounds == 1:
            hits["global state, 1 round"].append((ctas, n))
        elif rounds == 2:
            hits["2 rounds"].append((ctas, n))
        elif n % (W * QPB_GLOBAL):
            hits[">= 3 rounds, partial last round"].append((ctas, n))
        if W == 1:
            hits["W = 1"].append((ctas, n))
        if n < W:
            hits["n < W"].append((ctas, n))
    with capsys.disabled():
        print("\nsolver layouts reached (CTAs, n):")
        for k, v in hits.items():
            print(f"  {k:32s} {len(v):3d}  {v[:6]}{' ...' if len(v) > 6 else ''}")
    missing = [k for k, v in hits.items() if not v]
    assert not missing, missing
