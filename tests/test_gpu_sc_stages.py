"""The ScanContext batch search step by step on caller-owned device buffers (include/liorf_b200.h: liorf_sc_prepare_queries_dev,
liorf_sc_knn_batch_dev, liorf_sc_distance_batch_dev, liorf_sc_decide_dev) — the entry points an integrator chains in their own pipeline.

Stage 2 (k_sc_distance_bulk, csrc/sc_distance.cuh) is fed explicit (query, candidate) pairs of the classes where it can go wrong: every
alignment shift including the wrapping windows, column-periodic descriptors whose sector-key alignment and fine search tie exactly
(first strict minimum in ascending shift order), empty columns down to none, NaN cells, huge and negative heights, unfilled / negative
candidate slots.  Every output is compared with the CPU oracle (oracle/liorf_oracle.hpp, pinned to the reference's Scancontext.cpp) bit
for bit: fp64 values through their int64 bits, NaN exactly where the oracle has NaN, shifts and ids equal.  Query descriptors that are
only 8-byte aligned (a float64 tensor view at an odd element offset) must give the same bits as aligned ones in every stage."""
import ctypes as C
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

INT_MAX = 0x7FFFFFFF
SENT_D = np.int64(0x7FF4DEADBEEFCAFE)       # a NaN payload no kernel produces
SENT_S = 0x5A5A5A5A


def _keys(o, descs):
    return np.stack([o.sc_keys_from_desc(d)[0] for d in descs])


def _same_f64(a, b):
    a = np.asarray(a, np.float64).reshape(-1); b = np.asarray(b, np.float64).reshape(-1)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.int64), b[~nb].view(np.int64))


class _Stages:
    """ctypes calls of the four stage entry points on torch tensors allocated and filled on the context's stream"""

    def __init__(self, ctx):
        import torch
        self.torch, self.ctx = torch, ctx
        self.dev = torch.device(f"cuda:{ctx.params.device}")
        self.st = torch.cuda.ExternalStream(ctx.stream(), device=self.dev)

    def put(self, arr, offset8=False):
        """device copy of a numpy array; offset8: a view 8 bytes into its allocation (8- but not 16-byte aligned)"""
        t = self.torch
        arr = np.ascontiguousarray(arr)
        with t.cuda.stream(self.st):
            src = t.from_numpy(arr).to(self.dev)
            if not offset8:
                return src
            buf = t.empty(arr.size + 1, dtype=src.dtype, device=self.dev)
            v = buf[1:].view(arr.shape)
            v.copy_(src)
        assert v.data_ptr() % 16 == 8
        return v

    def empty(self, shape, dtype):
        with self.torch.cuda.stream(self.st):
            return self.torch.empty(shape, dtype=dtype, device=self.dev)

    def _call(self, name, *args):
        with self.torch.cuda.stream(self.st):
            rc = getattr(self.ctx.lib, name)(self.ctx.h, *args)
        assert rc == 0, (name, rc)

    @staticmethod
    def _p(t):
        return C.c_void_p(t.data_ptr()) if t is not None else None

    def prepare(self, d_q, qkeys=True, qsk=False, qcn=False):
        t, Q = self.torch, int(d_q.shape[0])
        k = self.empty((Q, 20), t.float32) if qkeys else None
        sk = self.empty((Q, 60), t.float64) if qsk else None
        cn = self.empty((Q, 60), t.float64) if qcn else None
        self._call("liorf_sc_prepare_queries_dev", self._p(d_q), Q, self._p(k), self._p(sk), self._p(cn))
        return k, sk, cn

    def knn(self, d_keys, offset):
        t, Q = self.torch, int(d_keys.shape[0])
        d, i = self.empty((Q, 3), t.float32), self.empty((Q, 3), t.int32)
        self._call("liorf_sc_knn_batch_dev", self._p(d_keys), Q, offset, self._p(d), self._p(i))
        return d, i

    def distance(self, d_q, d_cand, offset, pd=None, ps=None):
        t, Q = self.torch, int(d_cand.shape[0])
        pd = self.empty((Q, 3), t.float64) if pd is None else pd
        ps = self.empty((Q, 3), t.int32) if ps is None else ps
        self._call("liorf_sc_distance_batch_dev", self._p(d_q), self._p(d_cand), Q, offset, self._p(pd), self._p(ps))
        return pd, ps

    def decide(self, pd, ps, cand):
        t, Q = self.torch, int(cand.shape[0])
        loop, sh, dist = self.empty(Q, t.int32), self.empty(Q, t.int32), self.empty(Q, t.float64)
        self._call("liorf_sc_decide_dev", self._p(pd), self._p(ps), self._p(cand), Q, self._p(loop), self._p(sh), self._p(dist))
        return loop, sh, dist

    def fill_sentinel(self, pd, ps):
        with self.torch.cuda.stream(self.st):
            pd.view(self.torch.int64).fill_(int(SENT_D)); ps.fill_(SENT_S)

    def host(self, *ts):
        self.ctx.sync()
        return [x.cpu().numpy() for x in ts]


# ---------------------------------------------------------------------------------------------------- adversarial pairs

def _periodic(rng, period):
    block = rng.uniform(0.5, 6.0, (20, period)) * (rng.random((20, period)) < 0.8)
    return np.tile(block, (1, 60 // period))


def _stage2_pairs(synth):
    """(query, candidate, class) triples of the pair classes where stage 2 can go wrong"""
    rng = np.random.default_rng(1234)
    base = synth.sc_descriptors(8, seed=4321).reshape(-1, 20, 60)
    pairs = []
    noisy = lambda d: d + rng.normal(0, 0.05, d.shape) * (d != 0)
    for b in base[:2]:                                              # the alignment lands on every shift, incl. the wrapping windows
        for s in range(60):
            pairs.append((b, noisy(np.roll(b, s, axis=1)), "roll"))
    for p in (1, 2, 3, 5, 6):                                       # exact ties in the alignment AND among the fine shifts
        d = _periodic(rng, p)
        for s in (0, 1, 2, 3, 56, 57, 58, 59):
            pairs.append((d, np.roll(d, s, axis=1), "periodic"))
            pairs.append((np.roll(d, s, axis=1), d, "periodic"))
    for k in range(4):
        b = base[2 + k % 3]; r = noisy(np.roll(b, int(rng.integers(0, 60)), axis=1))
        qe, ce = b.copy(), r.copy()
        qe[:, rng.choice(60, 25, replace=False)] = 0.0; ce[:, rng.choice(60, 25, replace=False)] = 0.0
        pairs += [(qe, r, "empty cols"), (b, ce, "empty cols"), (qe, ce, "empty cols")]
    for k in range(3):
        one = np.zeros((20, 60)); col = int(rng.integers(0, 60)); one[:, col] = base[k][:, col] + 1.0
        pairs += [(one, base[k + 1], "one column"), (base[k + 1], one, "one column"), (one, np.roll(one, k + 1, axis=1), "one column")]
    z = np.zeros((20, 60))
    pairs += [(z, base[0], "all zero"), (base[1], z, "all zero"), (z, z, "all zero")]
    zm_q, zm_c = np.zeros((20, 60)), np.zeros((20, 60))            # zero-mean columns: every sector key 0 (align 0), non-zero norms, but
    zm_q[0, 0], zm_q[1, 0] = 2.0, -2.0                              # no overlap within shifts 57..3 → NaN in all seven → 1e7, shift 0
    zm_c[0, 30], zm_c[1, 30] = 3.0, -3.0
    pairs += [(zm_q, zm_c, "all zero"), (zm_c, zm_q, "all zero")]
    for k in range(4):
        pairs.append((base[k], base[k].copy(), "identical"))
    pairs.append((base[7], base[7], "identical"))
    for k in range(3):
        qn = base[k].copy(); qn[int(rng.integers(0, 20)), int(rng.integers(0, 60))] = np.nan
        cn = noisy(np.roll(base[k], 7 * k + 1, axis=1)); cn[int(rng.integers(0, 20)), int(rng.integers(0, 60))] = np.nan
        pairs += [(qn, base[k + 3], "nan cell"), (base[k + 3], cn, "nan cell")]
    for k in range(3):                                              # every sector-key norm >= 1e7: the alignment argmin stays 0
        pairs.append((base[k] * 1e9, np.roll(base[k], 11 + k, axis=1) * 1e9 + 3e9, "huge"))
        pairs.append((base[k] * 1e9, noisy(np.roll(base[k], 50 + k, axis=1)) * 1e9, "huge"))
    for k in range(6):
        b = base[k] - 3.0 * (base[k] != 0)                          # negative heights (points below the sensor)
        pairs.append((b, noisy(np.roll(b, int(rng.integers(0, 60)), axis=1)), "negative"))
    return pairs


def _restate(q, c):
    """the reference's distanceBtnScanContext restated in numpy, sequential in the reference's order, for the table only:
    (alignment, did the alignment tie, did the fine search tie)"""
    vk1, vk2 = np.zeros(60), np.zeros(60)
    for r in range(20):
        vk1 = vk1 + q[r]; vk2 = vk2 + c[r]
    vk1, vk2 = vk1 / 20, vk2 / 20
    s = np.arange(60); ss = np.zeros(60)
    for k in range(60):
        d = vk1[k] - vk2[(k - s) % 60]; ss = ss + d * d
    nrm = np.sqrt(ss)
    ok = nrm < 1e7
    align = int(np.argmax(nrm == nrm[ok].min())) if ok.any() else 0
    align_tie = bool(ok.any() and (nrm == nrm[ok].min()).sum() > 1)
    sh = np.sort((align + np.arange(-3, 4)) % 60)
    cols = np.arange(60)
    n1, n2, dot = np.zeros((7, 60)), np.zeros((7, 60)), np.zeros((7, 60))
    for r in range(20):
        a = q[r][cols][None, :].repeat(7, 0); b = c[r][(cols[None, :] - sh[:, None]) % 60]
        n1 = n1 + a * a; n2 = n2 + b * b; dot = dot + a * b
    n1, n2 = np.sqrt(n1), np.sqrt(n2)
    tot, eff = np.zeros(7), np.zeros(7)
    with np.errstate(invalid="ignore", divide="ignore"):
        for k in range(60):
            use = (n1[:, k] != 0) & (n2[:, k] != 0)
            tot = np.where(use, tot + dot[:, k] / (n1[:, k] * n2[:, k]), tot); eff = eff + use
        dist = 1.0 - tot / eff
    fin = dist < 1e7
    fine_tie = bool(fin.any() and (dist == dist[fin].min()).sum() > 1)
    return align, align_tie, fine_tie


@pytest.fixture(scope="module")
def stage2_case(synth, oracle):
    """one batch of > 3 000 pairs: query i holds adversarial pair i in slot 0; the other slots (and the queries after the adversarial
    ones) pair synthetic revisits with random rows; some slots are unfilled (INT_MAX) or negative"""
    rng = np.random.default_rng(99)
    pairs = _stage2_pairs(synth)
    filler = synth.sc_descriptors(400, seed=777)
    fq, _, _ = synth.sc_queries(filler, 1101 - len(pairs), seed=778)
    db = np.concatenate([np.stack([p[1].reshape(1200) for p in pairs]), filler], 0)
    qd = np.concatenate([np.stack([p[0].reshape(1200) for p in pairs]), fq], 0)
    Q, A = len(qd), len(pairs)
    cand = rng.integers(0, len(db), (Q, 3)).astype(np.int32)
    cand[:A, 0] = np.arange(A)
    cand[1::5, 2] = INT_MAX; cand[3::5, 1] = -1; cand[A + 7::11, 0] = -123; cand[A + 5] = (INT_MAX, -1, INT_MAX)
    o_d = np.full((Q, 3), np.inf); o_s = np.zeros((Q, 3), np.int32)
    for q in range(Q):
        for j in range(3):
            if 0 <= cand[q, j] < INT_MAX:
                o_d[q, j], o_s[q, j] = oracle.sc_distance(qd[q], db[cand[q, j]])
    return dict(db=db, qd=qd, cand=cand, o_d=o_d, o_s=o_s, pairs=pairs)


def _occupancy(ctx):
    out = (C.c_int * 3)()
    assert ctx.lib.liorf_debug_sc_distance_occupancy(ctx.h, out) == 0
    return out[0], out[1], out[2]


def test_stage2_adversarial_pairs_bit_exact(stage2_case):
    """liorf_sc_distance_batch_dev on the adversarial pairs, at Q = 1, an odd Q and a batch with more pairs than the persistent grid
    has warps: distance bits and shift of every pair == oracle.sc_distance; INT_MAX / negative slots → +inf, shift 0"""
    import liorf_b200
    S = stage2_case
    db, qd, cand, o_d, o_s = S["db"], S["qd"], S["cand"], S["o_d"], S["o_s"]
    G = 5000                                                        # global row of local row 0
    ctx = liorf_b200.Context(); ctx.scAddDescriptors(db)
    st = _Stages(ctx)
    sms, bps16, bps8 = _occupancy(ctx)
    warps = sms * bps16 * 4
    print(f"stage 2 grid: {sms} SMs x {bps16} CTAs/SM (8-byte-aligned queries: {bps8}) x 4 warps = {warps} warps")
    gc = np.where((cand >= 0) & (cand < INT_MAX), cand + G, cand).astype(np.int32)
    for Q in (1, 37, len(qd)):
        pd, ps = st.distance(st.put(qd[:Q]), st.put(gc[:Q]), G)
        pd, ps = st.host(pd, ps)
        for q in range(Q):
            assert _same_f64(pd[q], o_d[q]) and np.array_equal(ps[q], o_s[q]), (Q, q, cand[q], pd[q], o_d[q], ps[q], o_s[q])
    assert 3 * len(qd) > warps                                      # the last batch looped over its pairs
    special = (cand < 0) | (cand == INT_MAX)
    assert special.sum() > 100 and np.all(np.isinf(o_d[special])) and not ps[special].any()
    ctx.close()
    # what the pairs exercised
    rows = {}
    for i, (q, c, cls) in enumerate(S["pairs"]):
        align, at, ft = _restate(q, c)
        r = rows.setdefault(cls, [0, 0, 0, 0])
        r[0] += 1; r[1] += align < 3 or align > 56; r[2] += at; r[3] += ft
    r = rows.setdefault("synthetic", [0, 0, 0, 0]); r[0] += int((~special).sum()) - len(S["pairs"])
    rows["unfilled/negative slot"] = [int(special.sum()), 0, 0, 0]
    print(f"{'class':24s} {'pairs':>6s} {'wrapped':>8s} {'align tie':>10s} {'fine tie':>9s}")
    for k, (n, w, at, ft) in rows.items():
        print(f"{k:24s} {n:6d} {w:8d} {at:10d} {ft:9d}")
    per = rows["periodic"]
    assert per[1] >= 30 and per[2] >= 60 and per[3] >= 30                  # the tie cases really tie, also in wrapped windows
    assert rows["roll"][1] >= 12 and rows["huge"][0] == 6


def test_stage2_ownership_split_over_two_contexts(synth, oracle):
    """a database split over two contexts (rows [0, K1) and [K1, K)): both get the same global candidate triples and write into ONE
    output pair; each writes exactly the slots it owns (+ the INT_MAX / negative ones) and leaves every other slot bit-identical to a
    sentinel; the union == the single-context result == oracle.sc_query_batch"""
    import liorf_b200
    K, K1, Q = 700, 260, 301
    db = synth.sc_descriptors(K, seed=61)
    qd, _, _ = synth.sc_queries(db, Q, seed=62)
    keys = _keys(oracle, db)
    o_loop, o_sh, o_dist, o_cand = oracle.sc_query_batch(keys, db, _keys(oracle, qd), qd)
    cand = np.concatenate([o_cand, [[INT_MAX, -1, 5], [K - 1, INT_MAX, -9]]], 0).astype(np.int32)
    qd2 = np.concatenate([qd, qd[:2]], 0)
    special = (cand < 0) | (cand == INT_MAX)
    owner = np.where(special, -1, (cand >= K1).astype(np.int64))
    assert (owner == 0).sum() > 100 and (owner == 1).sum() > 100
    one = liorf_b200.Context(); one.scAddDescriptors(db)
    s1 = _Stages(one)
    r_d, r_s = s1.host(*s1.distance(s1.put(qd2), s1.put(cand), 0))
    one.close()
    ca, cb = liorf_b200.Context(), liorf_b200.Context()
    ca.scAddDescriptors(db[:K1]); cb.scAddDescriptors(db[K1:])
    sa, sb = _Stages(ca), _Stages(cb)
    pd, ps = sa.empty((Q + 2, 3), sa.torch.float64), sa.empty((Q + 2, 3), sa.torch.int32)
    dq, dc = sa.put(qd2), sa.put(cand)
    ca.sync()
    for g, (s, off) in enumerate(((sa, 0), (sb, K1))):
        s.fill_sentinel(pd, ps); s.ctx.sync()
        s.distance(dq, dc, off, pd, ps)
        d, sh = s.host(pd, ps)
        mine = (owner == g) | special
        assert np.array_equal(d[~mine].view(np.int64), np.full((~mine).sum(), SENT_D)) and np.all(sh[~mine] == SENT_S), g
        assert _same_f64(d[mine], r_d[mine]) and np.array_equal(sh[mine], r_s[mine]), g
    sa.fill_sentinel(pd, ps); ca.sync()
    sa.distance(dq, dc, 0, pd, ps); ca.sync()
    sb.distance(dq, dc, K1, pd, ps)
    d, sh = sb.host(pd, ps)
    assert _same_f64(d, r_d) and np.array_equal(sh, r_s)
    loop, lsh, ldist = sa.host(*sa.decide(pd, ps, dc))
    assert np.array_equal(loop[:Q], o_loop) and np.array_equal(lsh[:Q], o_sh) and _same_f64(ldist[:Q], o_dist)
    for q in range(Q):
        for j in range(3):
            od, os_ = oracle.sc_distance(qd[q], db[cand[q, j]])
            assert _same_f64(d[q, j], od) and sh[q, j] == os_, (q, j)
    ca.close(); cb.close()


def _stage1_queries(synth):
    db = synth.sc_descriptors(500, seed=41)
    q, src, _ = synth.sc_queries(db, 61, seed=42)
    q[3] = 0.0                                                      # empty scan
    q[4] = q[4] * 1e9                                               # huge heights
    q[5] = q[5] - 3.0 * (q[5] != 0)                                 # negative heights
    q[6, :600] = 0.0                                                # empty inner rings
    q[7] = np.tile(q[7].reshape(20, 60)[:, :5], (1, 12)).reshape(1200)   # column-periodic
    return db, q, src


def _colnorm(desc):
    d = desc.reshape(20, 60)
    out = np.empty(60)
    for c in range(60):
        s = 0.0
        for r in range(20):
            v = float(d[r, c]); s += v * v
        out[c] = math.sqrt(s)
    return out


def test_stage1_prepare_outputs_bit_exact(synth, oracle):
    """liorf_sc_prepare_queries_dev three ways (ring keys only: k_sc_ringkeys_batch; with sector keys / column norms: k_sc_keys_batch;
    on an 8-byte-aligned view: the fallback), plus sector keys without column norms: ring keys == oracle.sc_keys_from_desc, sector
    keys == oracle, column norms == a sequential fp64 sum of squares over the rings + sqrt, all bit for bit"""
    import liorf_b200
    _, q, _ = _stage1_queries(synth)
    o_rk = np.stack([oracle.sc_keys_from_desc(d)[0] for d in q]); o_sk = np.stack([oracle.sc_keys_from_desc(d)[1] for d in q])
    o_cn = np.stack([_colnorm(d) for d in q])
    ctx = liorf_b200.Context(); st = _Stages(ctx)
    k1, _, _ = st.prepare(st.put(q))
    k2, sk2, cn2 = st.prepare(st.put(q), qsk=True, qcn=True)
    k3, _, _ = st.prepare(st.put(q, offset8=True))
    k4, sk4, cn4 = st.prepare(st.put(q, offset8=True), qsk=True, qcn=True)
    _, sk5, _ = st.prepare(st.put(q), qkeys=False, qsk=True)
    k1, k2, sk2, cn2, k3, k4, sk4, cn4, sk5 = st.host(k1, k2, sk2, cn2, k3, k4, sk4, cn4, sk5)
    for k in (k1, k2, k3, k4):
        assert np.array_equal(k.view(np.int32), o_rk.view(np.int32))
    for sk in (sk2, sk4, sk5):
        assert np.array_equal(sk.view(np.int64), o_sk.view(np.int64))
    for cn in (cn2, cn4):
        assert np.array_equal(cn.view(np.int64), o_cn.view(np.int64))
    ctx.close()


@pytest.mark.parametrize("offset8", [False, True], ids=["aligned", "offset8"])
def test_chained_stages_on_caller_buffers(synth, oracle, offset8):
    """prepare → knn_batch_dev (global_offset 1000) → distance_batch_dev → decide_dev on caller buffers == liorf_sc_query_batch ==
    oracle.sc_query_batch: candidates, loop ids, shifts, distance bits; the 8-byte-aligned query view gives the same bits"""
    import liorf_b200
    G = 1000
    db, q, src = _stage1_queries(synth)
    ctx = liorf_b200.Context(); ctx.scAddDescriptors(db)
    r_loop, r_sh, r_dist, r_cand = ctx.scQueryBatch(q)
    o_loop, o_sh, o_dist, o_cand = oracle.sc_query_batch(_keys(oracle, db), db, _keys(oracle, q), q)
    st = _Stages(ctx)
    dq = st.put(q, offset8)
    keys, _, _ = st.prepare(dq)
    _, cand = st.knn(keys, G)
    pd, ps = st.distance(dq, cand, G)
    loop, sh, dist = st.decide(pd, ps, cand)
    cand, loop, sh, dist, pd = st.host(cand, loop, sh, dist, pd)
    assert np.array_equal(cand - G, r_cand) and np.array_equal(cand - G, o_cand)
    assert np.array_equal(np.where(loop >= 0, loop - G, -1), r_loop) and np.array_equal(r_loop, o_loop)
    assert np.array_equal(sh, r_sh) and np.array_equal(sh, o_sh)
    assert _same_f64(dist, r_dist) and _same_f64(dist, o_dist)
    for i in range(len(q)):
        for j in range(3):
            assert _same_f64(pd[i, j], oracle.sc_distance(q[i], db[cand[i, j] - G])[0]), (i, j)
    assert (r_loop >= 0).sum() >= 10
    ctx.close()


# ---------------------------------------------------------------------------------------------------- decision

def _decide_ref(pd, ps, cand):
    """include/Scancontext.cpp:319-340 (liorf_oracle.hpp SCManager::detectLoopClosureID): min 1e7, strict < in kNN order, < 0.3"""
    Q = len(pd)
    loop, sh, dist = np.zeros(Q, np.int32), np.zeros(Q, np.int32), np.zeros(Q)
    for q in range(Q):
        mn, al, nn = 10000000.0, 0, 0
        for c in range(3):
            d = float(pd[q, c])
            if d < mn:
                mn, al, nn = d, int(ps[q, c]), int(cand[q, c])
        loop[q] = nn if mn < 0.3 else -1; sh[q] = al; dist[q] = mn
    return loop, sh, dist


def test_decide_on_hand_made_inputs(ctx):
    """liorf_sc_decide_dev on hand-made pair distances: NaN / +inf slots, equal distances (the earlier slot wins), exactly 0.3 (no
    loop), the double just below 0.3 (loop), every slot >= 1e7 (loop -1, shift 0, distance 1e7), then random draws from those values"""
    below = np.nextafter(0.3, 0.0)
    nan, inf = np.nan, np.inf
    rows = [[nan, 0.2, 0.1], [inf, inf, inf], [nan, nan, nan], [0.2, 0.2, 0.5], [0.5, 0.2, 0.2], [0.1, 0.1, 0.1],
            [0.3, 0.5, 0.6], [0.5, 0.3, 0.3], [below, 0.3, 0.4], [0.3, below, below], [1e7, 2e7, inf], [1e7, 1e7, 1e7],
            [0.1, nan, 0.05], [inf, 0.29, nan], [-1e-17, 0.0, -0.0], [0.0, -0.0, 0.25], [1e7, nan, 0.9], [0.31, 0.35, 0.3]]
    rng = np.random.default_rng(5)
    vals = np.array([nan, inf, 0.3, below, 0.1, 0.2, 1e7, 0.0, 0.9])
    pd = np.concatenate([np.array(rows), vals[rng.integers(0, len(vals), (301, 3))]], 0)
    Q = len(pd)
    ps = rng.integers(0, 60, (Q, 3)).astype(np.int32)
    cand = rng.integers(0, 100000, (Q, 3)).astype(np.int32)
    cand[1] = (INT_MAX, INT_MAX, -1)
    st = _Stages(ctx)
    loop, sh, dist = st.host(*st.decide(st.put(pd), st.put(ps), st.put(cand)))
    e_loop, e_sh, e_dist = _decide_ref(pd, ps, cand)
    assert np.array_equal(loop, e_loop) and np.array_equal(sh, e_sh) and _same_f64(dist, e_dist)
    assert (loop[:12] == [cand[0, 2], -1, -1, cand[3, 0], cand[4, 1], cand[5, 0], -1, -1, cand[8, 0], cand[9, 1], -1, -1]).all()
    assert dist[10] == 1e7 and sh[10] == 0 and sh[1] == 0 and dist[6] == 0.3


# ---------------------------------------------------------------------------------------------------- 8-byte-aligned queries

def test_stage2_offset_view_bit_identical(stage2_case):
    """the adversarial batch through liorf_sc_distance_batch_dev from an 8-byte-aligned view: the same bits as the aligned tensor"""
    import liorf_b200
    S = stage2_case
    ctx = liorf_b200.Context(); ctx.scAddDescriptors(S["db"])
    st = _Stages(ctx)
    a_d, a_s = st.host(*st.distance(st.put(S["qd"]), st.put(S["cand"]), 0))
    for Q in (1, 37, len(S["qd"])):
        d, s = st.host(*st.distance(st.put(S["qd"][:Q], offset8=True), st.put(S["cand"][:Q]), 0))
        assert np.array_equal(d.view(np.int64), a_d[:Q].view(np.int64)) and np.array_equal(s, a_s[:Q]), Q
    assert _same_f64(a_d, S["o_d"]) and np.array_equal(a_s, S["o_s"])
    ctx.close()


def test_shard_query_world1_graph_replay_alternating_alignment(synth):
    """liorf_sc_shard_query_dev at world 1: three identical calls (the second is captured, the third replays the graph) on an aligned
    buffer, then on an 8-byte-aligned one, then alternating — every result == liorf_sc_query_batch on the same data"""
    import torch
    import liorf_b200
    from liorf_b200.sc_sharded import PeerShardedSearch
    K, Q = 3000, 257
    db = synth.sc_descriptors(K, seed=83)
    ref = liorf_b200.Context(); ref.scAddDescriptors(db)
    ctx = liorf_b200.Context(); ctx.scAddDescriptors(db)
    S = PeerShardedSearch(ctx, 0, 1, [0, K], Q, torch)
    S.connect_local([S])
    st = _Stages(ctx)
    qs = [synth.sc_queries(db, Q, seed=84 + b)[0] for b in range(2)]
    refs = [ref.scQueryBatch(q) for q in qs]
    bufs = {False: st.empty((Q, 1200), torch.float64), True: st.put(np.zeros((Q, 1200)), offset8=True)}
    for step, (off8, b) in enumerate([(False, 0)] * 3 + [(True, 1)] * 3 + [(False, 1), (True, 0), (False, 0), (True, 1), (True, 1)]):
        with torch.cuda.stream(st.st):
            bufs[off8].copy_(torch.from_numpy(qs[b]).to(st.dev))
        out = S.query(bufs[off8])
        loop, sh, dd, cand = st.host(*out)
        r_loop, r_sh, r_dist, r_cand = refs[b]
        assert np.array_equal(cand, r_cand) and np.array_equal(loop, r_loop) and np.array_equal(sh, r_sh), step
        assert _same_f64(dd, r_dist), step
    ctx.close(); ref.close()


def test_two_rank_phases_offset_view(synth, oracle):
    """the two-rank one-device phases harness of test_gpu_sc_shard.py with an 8-byte-aligned view as every rank's query tensor:
    stage 1 slices, the owner-split stage 2 and the decision == the unsharded search == the oracle"""
    import torch
    import liorf_b200
    from liorf_b200.sc_sharded import PeerShardedSearch
    K, world, bounds = 2005, 2, [0, 1100, 2005]
    db = synth.sc_descriptors(K, seed=87)
    ref = liorf_b200.Context(); ref.scAddDescriptors(db)
    ctxs = [liorf_b200.Context() for _ in range(world)]
    for g, c in enumerate(ctxs):
        c.scAddDescriptors(db[bounds[g]:bounds[g + 1]]); c.scSetSearchPath(1)
    S = [PeerShardedSearch(c, g, world, bounds, 300, torch) for g, c in enumerate(ctxs)]
    for s in S:
        s.connect_local(S)
    PeerShardedSearch.sync_keys_local(S)
    okeys = _keys(oracle, db)
    for b, Q in enumerate((129, 1, 300)):
        qd, _, _ = synth.sc_queries(db, Q, seed=88 + b)
        r_loop, r_sh, r_dist, r_cand = ref.scQueryBatch(qd)
        o_loop, o_sh, o_dist, o_cand = oracle.sc_query_batch(okeys, db, _keys(oracle, qd), qd)
        assert np.array_equal(r_cand, o_cand) and np.array_equal(r_loop, o_loop) and np.array_equal(r_sh, o_sh) and _same_f64(r_dist, o_dist)
        dq = [_Stages(c).put(qd, offset8=True) for c in ctxs]
        res = {}
        for step in (1, 2, 4):
            for g in range(world):
                res[g] = S[g].query(dq[g], phases=step)
        for c in ctxs:
            c.sync()
        torch.cuda.synchronize()
        for g in range(world):
            loop, sh, dd, cand = [t.cpu().numpy() for t in res[g]]
            assert np.array_equal(cand, r_cand) and np.array_equal(loop, r_loop) and np.array_equal(sh, r_sh) and _same_f64(dd, r_dist), (b, g)
    for c in ctxs:
        c.close()
    ref.close()


# ---------------------------------------------------------------------------------------------------- the one-query kernel

def test_detect_loop_closure_sequence_on_adversarial_revisits(ctx, oracle, synth):
    """k_sc_distance (liorf_sc_detect_loop_closure_id) on a sequence with column-periodic, empty-column and all-zero revisits of
    earlier entries: loop id, yaw, the three candidates and min_dist (bits) of every call == oracle.SCManager"""
    rng = np.random.default_rng(17)
    base = synth.sc_descriptors(60, seed=19).reshape(-1, 20, 60)
    per = [_periodic(rng, p) for p in (1, 2, 3, 5, 6)]
    seq = list(base[:40]) + per
    for i in range(70):
        kind = i % 5
        if kind == 0:
            d = np.roll(per[i // 5 % 5], int(rng.choice([0, 1, 2, 57, 58, 59])), axis=1)
        elif kind == 1:
            d = np.roll(seq[int(rng.integers(0, 40))], int(rng.integers(0, 60)), axis=1).copy(); d[:, rng.choice(60, 30, replace=False)] = 0.0
        elif kind == 2:
            d = np.zeros((20, 60))
        elif kind == 3:
            j = int(rng.integers(0, 40)); d = np.roll(seq[j], int(rng.integers(0, 60)), axis=1)
            d = d + rng.normal(0, 0.05, d.shape) * (d != 0)
        else:
            d = base[40 + i % 20]
        seq.append(d)
    sc = oracle.SCManager()
    n_loop = 0
    for i, d in enumerate(seq):
        ctx.scAddDescriptors(d.reshape(1, 1200)); sc.save_descriptor(d)
        g, o = ctx.detectLoopClosureID(), sc.detect()
        assert g[0] == o[0] and np.float32(g[1]).view(np.int32) == np.float32(o[1]).view(np.int32), (i, g, o)
        if i >= 30:
            assert np.array_equal(g[3], o[3]), (i, g, o)
            assert np.float64(g[2]).view(np.int64) == np.float64(o[2]).view(np.int64), (i, g[2], o[2])
        n_loop += g[0] >= 0
    assert n_loop >= 5
