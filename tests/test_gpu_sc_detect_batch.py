"""liorf_sc_detect_loop_closure_id_batch (Context.detectLoopClosureIDBatch): detectLoopClosureID for many calls at once.  Answer q must be
what the live call returns when the database held its first n_db[q] entries and the stale tree covered keys [0, n_tree[q]) — bit for bit:
loop ids and candidate triples exactly, fp32 yaw and fp64 min_dist through their integer bits.  Every case runs with the ring-key search
on auto, forced to the CUDA-core kernel (1) and forced to the tensor-core filter (2).  sc_tree_schedule (the stale-tree rule) is checked
without a GPU."""
import ctypes as C

import numpy as np
import pytest

import liorf_b200
from liorf_b200 import sc_tree_schedule

PATHS = (0, 1, 2)
ERR_ARG = -2


def _live(ctx):
    lid, yaw, md, cand = ctx.detectLoopClosureID()
    return int(lid), np.float32(yaw), np.float64(md), np.array(cand, np.int32)


def _assert_same(batch, q, live, what):
    lid, yaw, md, cand = batch
    assert lid[q] == live[0], (what, q, lid[q], live)
    assert yaw[q].view(np.int32) == np.float32(live[1]).view(np.int32), (what, q, yaw[q], live)
    assert md[q].view(np.int64) == np.float64(live[2]).view(np.int64), (what, q, md[q], live)
    assert np.array_equal(cand[q], live[3]), (what, q, cand[q], live)


def _yaw_of_shift(s):
    """sc_yaw_rad: deg2rad(float) of the decided shift in degrees"""
    return np.float32(np.float64(np.float32(np.float64(s) * 6.0)) * np.pi / 180.0)


def _periodic(rng, period):
    block = rng.uniform(0.5, 6.0, (20, period)) * (rng.random((20, period)) < 0.8)
    return np.tile(block, (1, 60 // period))


def _sequence(synth):
    """~400 entries with planted revisits (no exact duplicates: the reference's order of exact ties is nanoflann's), then the adversarial
    revisits of test_gpu_sc_stages: column-periodic, empty columns, all-zero, identical.  Returns (descs [K, 1200], n_planted)."""
    rng = np.random.default_rng(31)
    base = synth.sc_descriptors(300, seed=301)
    rev, _, _ = synth.sc_queries(base[:150], 100, seed=302)
    seq = list(base[:150])
    for k in range(100):
        seq.append(rev[k]); seq.append(base[150 + k])
    seq += list(base[250:300])
    n_planted = len(seq)
    per = [_periodic(rng, p) for p in (1, 2, 3, 5, 6)]
    seq += [p.reshape(-1) for p in per]
    for i in range(70):
        kind = i % 5
        if kind == 0:
            d = np.roll(per[i // 5 % 5], int(rng.choice([0, 1, 2, 57, 58, 59])), axis=1)
        elif kind == 1:
            d = np.roll(seq[int(rng.integers(0, 300))].reshape(20, 60), int(rng.integers(0, 60)), axis=1).copy()
            d[:, rng.choice(60, 30, replace=False)] = 0.0
        elif kind == 2:
            d = np.zeros((20, 60))
        elif kind == 3:
            d = np.roll(seq[int(rng.integers(0, 300))].reshape(20, 60), int(rng.integers(0, 60)), axis=1)
            d = d + rng.normal(0, 0.05, d.shape) * (d != 0)
        else:
            d = seq[int(rng.integers(0, 300))].reshape(20, 60).copy()          # identical to an earlier entry
        seq.append(np.asarray(d).reshape(-1))
    return np.stack([np.asarray(s, np.float64).reshape(-1) for s in seq]), n_planted


@pytest.fixture(scope="module")
def seq_case(synth):
    return _sequence(synth)


def _replay_every(ctx, descs):
    """one descriptor at a time, detectLoopClosureID after every add"""
    out = []
    for d in descs:
        ctx.scAddDescriptors(d.reshape(1, 1200))
        out.append(_live(ctx))
    return out


# ---------------------------------------------------------------------------------------------------- the schedule (no GPU)

def test_tree_schedule_rule():
    # early-outs do not count; counter 0, 10, 20 ... snapshot n - 30; repeated sizes advance the counter
    calls = [1, 5, 30, 31, 32, 33, 34, 35, 36, 37, 38, 39, 40, 41, 41, 41, 12, 60] + [70] * 9 + [90]
    want = [0, 0, 0, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 11, 11, 11, 0, 11] + [11] * 6 + [40] * 3 + [40]
    assert list(sc_tree_schedule(calls)) == want
    assert sc_tree_schedule([]).shape == (0,)
    assert list(sc_tree_schedule(range(1, 61))) == [0] * 30 + [1] * 10 + [11] * 10 + [21] * 10


# ---------------------------------------------------------------------------------------------------- 1. every live call, replayed

@pytest.mark.gpu
@pytest.mark.parametrize("path", PATHS)
def test_every_live_call_replayed(seq_case, path):
    descs, _ = seq_case
    ctx = liorf_b200.Context()
    ctx.scSetSearchPath(path)
    live = _replay_every(ctx, descs)
    K = len(descs)
    n_db = np.arange(1, K + 1, dtype=np.int32)
    n_tree = sc_tree_schedule(n_db)
    assert set(n_tree[30:40]) == {1} and n_tree[40] == 11              # the first ten calls search a 1-key tree: two substituted slots
    res = ctx.detectLoopClosureIDBatch(n_db, n_tree)
    for q in range(K):
        _assert_same(res, q, live[q], "replay")
    assert np.array_equal(res[3][30], [0, 0, 0])
    n_loop = int((res[0] >= 0).sum())
    print(f"path {path}: {K} calls, {K - 30} on the device, {n_loop} loops")
    assert n_loop >= 40
    ctx.close()


# ---------------------------------------------------------------------------------------------------- 2. irregular histories

@pytest.mark.gpu
@pytest.mark.parametrize("path", PATHS)
def test_irregular_histories_shuffled_with_duplicates(seq_case, path):
    """detect calls at only some sizes, repeated calls at one size (the counter moves, the query row does not), a history that starts
    after the database already held 80 entries; the batch in shuffled order with duplicated entries"""
    descs, _ = seq_case
    rng = np.random.default_rng(100 + path)
    ctx = liorf_b200.Context()
    ctx.scSetSearchPath(path)
    ctx.scAddDescriptors(descs[:80])
    sizes, live = [], []
    for n in range(81, len(descs) + 1):
        ctx.scAddDescriptors(descs[n - 1].reshape(1, 1200))
        if rng.random() < 0.45:
            for _ in range(int(rng.integers(1, 4))):
                sizes.append(n); live.append(_live(ctx))
    sizes = np.array(sizes, np.int32)
    n_tree = sc_tree_schedule(sizes)
    assert (np.diff(sizes) == 0).any() and len(set(n_tree)) > 10
    order = np.concatenate([rng.permutation(len(sizes)), rng.integers(0, len(sizes), 60)])
    res = ctx.detectLoopClosureIDBatch(sizes[order], n_tree[order])
    for q, k in enumerate(order):
        _assert_same(res, q, live[k], "irregular")
    print(f"path {path}: {len(sizes)} calls at {len(set(sizes.tolist()))} sizes, batch of {len(order)}, {int((res[0] >= 0).sum())} loops")
    ctx.close()


# ---------------------------------------------------------------------------------------------------- 3. tensor path at scale

NKT = 80
K3 = 128 * NKT                    # 10 240 keys: every key tile full, so limits close to K leave whole tiles unmasked
DUP = 33 * NKT - 1                # rows DUP and DUP + 1 are identical: a limit of DUP + 1 must keep the tie inside the prefix
OVF = (4000, 7000)                # rows identical to row 17: > SCT_CAP candidate chunks → the exact fallback scan


@pytest.fixture(scope="module")
def scale_case(synth, oracle):
    rng = np.random.default_rng(503)
    db = synth.sc_descriptors(K3, seed=501)
    rev, _, _ = synth.sc_queries(db[:8000], K3 - 9000, seed=502)
    db[9000:] = rev                                                     # planted revisits of rows < 8000
    db[OVF[0]:OVF[1]] = db[17]
    db[DUP + 1] = db[DUP]
    db[8500] = db[17]                                                   # query rows for the two tie cases
    db[8600] = db[DUP]
    lims, rows = [], []

    def add(L, row=None):
        if row is None:
            lo = max(L + 29, 9000) if L + 29 < K3 - 1 else L + 29
            row = int(rng.integers(lo, K3))
        assert 1 <= L <= row + 1 - 30 and row < K3
        lims.append(L); rows.append(row)

    for m in range(128):                                                # every tile residue edge: 0, 1, nkt - 1 (mod nkt)
        for r in (0, 1, NKT - 1):
            if 1 <= m * NKT + r <= K3 - 30:
                add(m * NKT + r)
    for c in (32, 64, 96, 127):                                         # 32-column chunk boundaries and the last column of every tile
        for e in (-1, 0, 1):
            add(c * NKT + e)
    for L in (1, 2, 3, K3 - 30):
        add(L)
    add(DUP + 1, 8600); add(DUP + 2, 8600); add(DUP, 8600)
    for L in (OVF[0] + 1, 5500, 5501, OVF[1] - 1):
        add(L, 8500)
    while len(lims) < 1500:
        L = int(rng.integers(1, K3 - 30)); add(L)
    n_db = np.array(rows, np.int32) + 1
    n_tree = np.array(lims, np.int32)
    keys = oracle.sc_keys_batch(db)
    # oracle.sc_query_batch on each prefix [0, n_tree) (a tree of at least 3 keys: the oracle's batch has no unfilled-slot rule)
    o_loop = np.zeros(len(n_db), np.int32); o_sh = np.zeros(len(n_db), np.int32); o_dist = np.zeros(len(n_db)); o_cand = np.zeros((len(n_db), 3), np.int32)
    for L in sorted(set(lims)):
        if L < 3:
            continue
        sel = np.nonzero(n_tree == L)[0]
        r = n_db[sel] - 1
        lo, sh, di, ca = oracle.sc_query_batch(keys[:L], db[:L], keys[r], db[r])
        o_loop[sel], o_sh[sel], o_dist[sel], o_cand[sel] = lo, sh, di, ca
    return dict(db=db, n_db=n_db, n_tree=n_tree, oracle=(o_loop, o_sh, o_dist, o_cand))


def _live_at(db, N, L):
    """the live call with the database at N entries and the tree at keys [0, L): rows [0, L + 30) then a call (counter 0 snapshots L),
    then row N - 1 appended and the call that answers it — the answer depends on rows [0, L) and row N - 1 only"""
    c = liorf_b200.Context()
    c.scAddDescriptors(db[:L + 30])
    c.detectLoopClosureID()
    c.scAddDescriptors(db[N - 1:N])
    r = _live(c)
    c.close()
    return r


@pytest.fixture(scope="module")
def scale_live(scale_case):
    S = scale_case
    n_db, n_tree = S["n_db"], S["n_tree"]
    picks = []
    for L in (1, 2, 3, NKT - 1, NKT, NKT + 1, 32 * NKT, 32 * NKT + 1, 127 * NKT - 1, 127 * NKT, 127 * NKT + 1, K3 - 30, DUP, DUP + 1, DUP + 2,
              OVF[0] + 1, 5500):
        picks.append(int(np.nonzero(n_tree == L)[0][0]))
    return {q: _live_at(S["db"], int(n_db[q]), int(n_tree[q])) for q in picks}


@pytest.mark.gpu
@pytest.mark.parametrize("path", (1, 0, 2))
def test_tensor_scale_limits_on_every_edge(scale_case, scale_live, path):
    S = scale_case
    n_db, n_tree = S["n_db"], S["n_tree"]
    ctx = liorf_b200.Context()
    ctx.scAddDescriptors(S["db"])
    ctx.scSetSearchPath(path)
    res = ctx.detectLoopClosureIDBatch(n_db, n_tree)
    st = ctx.scTensorStats()
    lid, yaw, md, cand = res
    if path == 1:
        assert st["candidates"] == 0                                    # the CUDA-core kernel ran: no tensor-core search on this context
    else:
        assert st["candidates"] >= 3 * len(n_db) and st["overflow"] >= 3   # auto picked the tensor cores; the identical block overflowed
    for q, live in scale_live.items():
        _assert_same(res, q, live, f"live L={n_tree[q]}")
    o_loop, o_sh, o_dist, o_cand = S["oracle"]
    ok = n_tree >= 3
    assert np.array_equal(cand[ok], o_cand[ok]) and np.array_equal(lid[ok], o_loop[ok])
    assert np.array_equal(yaw[ok].view(np.int32), np.array([_yaw_of_shift(s) for s in o_sh[ok]], np.float32).view(np.int32))
    assert np.array_equal(md[ok].view(np.int64), o_dist[ok].view(np.int64))
    q = np.nonzero((n_db == 8601) & (n_tree == DUP + 1))[0][0]
    assert cand[q][0] == DUP and DUP + 1 not in cand[q] and lid[q] == DUP
    q = np.nonzero((n_db == 8601) & (n_tree == DUP + 2))[0][0]
    assert list(cand[q][:2]) == [DUP, DUP + 1]
    q = np.nonzero((n_db == 8501) & (n_tree == 5500))[0][0]
    assert list(cand[q]) == [17, OVF[0], OVF[0] + 1] and lid[q] == 17
    q = np.nonzero((n_db == 8501) & (n_tree == OVF[0] + 1))[0][0]
    assert list(cand[q][:2]) == [17, OVF[0]]
    edge = np.isin(n_tree % NKT, (0, 1, NKT - 1))
    print(f"path {path}: {len(n_db)} rows, {int(edge.sum())} limits on tile edges, {int((n_tree < 3).sum())} trees under 3 keys, "
          f"overflow queries {st['overflow']}, candidate chunks {st['candidates']}, {int((lid >= 0).sum())} loops")
    ctx.close()


# ---------------------------------------------------------------------------------------------------- 4. reference pin

@pytest.mark.gpu
def test_reference_detect_pin(seq_case, oracle):
    if oracle.refsc() is None:
        pytest.skip("oracle/_ref/libliorf_ref_sc.so was not built (the reference tree is absent and no prebuilt copy travelled)")
    descs, n_planted = seq_case
    ref = oracle.RefSCManager()
    want = []
    for d in descs[:n_planted]:
        ref.save_descriptor(d)
        want.append(ref.detect())
    ctx = liorf_b200.Context()
    ctx.scAddDescriptors(descs)
    n_db = np.arange(1, n_planted + 1, dtype=np.int32)
    lid, yaw, _, _ = ctx.detectLoopClosureIDBatch(n_db, sc_tree_schedule(n_db))
    assert np.array_equal(lid, np.array([w[0] for w in want], np.int32))
    assert np.array_equal(yaw.view(np.int32), np.array([w[1] for w in want], np.float32).view(np.int32))
    assert (lid >= 0).sum() >= 40
    ctx.close()


# ---------------------------------------------------------------------------------------------------- 5. no side effects

@pytest.mark.gpu
def test_no_side_effects(seq_case, synth):
    descs, _ = seq_case
    K0 = 300
    a, b = liorf_b200.Context(), liorf_b200.Context()
    for c in (a, b):
        c.scAddDescriptors(descs[:K0 - 1])
        for _ in range(7):
            c.detectLoopClosureID()                                   # counter 7: the next rebuild is 3 calls away
    qd, _, _ = synth.sc_queries(descs[:K0 - 1], 80, seed=606)
    before = a.scQueryBatch(qd)
    n_db = np.arange(1, K0, dtype=np.int32)
    ref = None
    for path in PATHS:
        a.scSetSearchPath(path)
        r = a.detectLoopClosureIDBatch(n_db, sc_tree_schedule(n_db))
        ref = r if ref is None else ref
        assert all(np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(r, ref))
    a.scSetSearchPath(0)
    after = a.scQueryBatch(qd)
    assert all(np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8)) for x, y in zip(before, after))
    for k in range(K0 - 1, K0 + 24):                                    # live calls across two tree rebuilds: the counter and tree were untouched
        for c in (a, b):
            c.scAddDescriptors(descs[k].reshape(1, 1200))
        la, lb = _live(a), _live(b)
        assert la[0] == lb[0] and la[1].view(np.int32) == lb[1].view(np.int32) and la[2].view(np.int64) == lb[2].view(np.int64) and np.array_equal(la[3], lb[3])
    # a borrowing context answers the same batch from the owner's database, read-only
    br = liorf_b200.Context()
    br.scBorrowDatabase(a)
    n_db2 = np.arange(1, a.scSize() + 1, dtype=np.int32)
    for path in PATHS:
        a.scSetSearchPath(path); br.scSetSearchPath(path)
        ra = a.detectLoopClosureIDBatch(n_db2, sc_tree_schedule(n_db2))
        rb = br.detectLoopClosureIDBatch(n_db2, sc_tree_schedule(n_db2))
        assert all(np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(ra, rb))
    br.close(); a.close(); b.close()


# ---------------------------------------------------------------------------------------------------- 6. arguments

@pytest.mark.gpu
def test_argument_checks_leave_outputs_untouched(seq_case):
    descs, _ = seq_case
    ctx = liorf_b200.Context()
    ctx.scAddDescriptors(descs[:100])
    f = ctx.lib.liorf_sc_detect_loop_closure_id_batch
    P = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None

    def call(n_db, n_tree, Q=None, drop=()):
        n_db = np.asarray(n_db, np.int32); n_tree = np.asarray(n_tree, np.int32)
        Q = len(n_db) if Q is None else Q
        lid = np.full(max(Q, 1), 77, np.int32); yaw = np.full(max(Q, 1), 7.5, np.float32)
        md = np.full(max(Q, 1), 9.25); cand = np.full((max(Q, 1), 3), 55, np.int32)
        arrs = dict(n_db=n_db, n_tree=n_tree, lid=lid, yaw=yaw)
        for k in drop:
            arrs[k] = None
        rc = f(ctx.h, P(arrs["n_db"]), P(arrs["n_tree"]), C.c_int(Q), P(arrs["lid"]), P(arrs["yaw"]), P(md), P(cand))
        return rc, lid, yaw, md, cand

    def untouched(r):
        _, lid, yaw, md, cand = r
        return (lid == 77).all() and (yaw == 7.5).all() and (md == 9.25).all() and (cand == 55).all()

    bad = [([0], [1]), ([101], [1]), ([50, -3], [5, 1]), ([50], [0]), ([50], [21]), ([100], [71]), ([31], [2]), ([40, 60], [5, -1])]
    for n_db, n_tree in bad:
        r = call(n_db, n_tree)
        assert r[0] == ERR_ARG and untouched(r), (n_db, n_tree, r)
    for k in ("n_db", "n_tree", "lid", "yaw"):
        r = call([50], [5], drop=(k,))
        assert r[0] == ERR_ARG and untouched(r), k
    r = call([50], [5], Q=-1)
    assert r[0] == ERR_ARG and untouched(r)
    r = call([], [], Q=0, drop=("n_db", "n_tree", "lid", "yaw"))
    assert r[0] == 0 and untouched(r)
    # early-out entries: loop -1, yaw 0, min_dist / cand3 untouched, their n_tree ignored; the others are answered
    r = call([30, 1, 50, 31], [-5, 999, 20, 1])
    rc, lid, yaw, md, cand = r
    assert rc == 0 and list(lid[:2]) == [-1, -1] and (yaw[:2] == 0).all() and (md[:2] == 9.25).all() and (cand[:2] == 55).all()
    assert md[2] != 9.25 and md[3] != 9.25 and (cand[3] == 0).all()      # a 1-key tree: all three slots are candidate 0
    ctx.close()
