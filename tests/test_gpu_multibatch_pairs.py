"""Pair-driven hash joins (INNER / LEFT against duplicate build keys, every RIGHT and FULL join) whose build side is split into
batches (HJ_NEED_NEW_BATCH, nodeHashjoin.c:709-738; HJ_FILL_INNER_TUPLES after the last batch, :676-706): the probe rows are
grouped by batch once, each batch is loaded and probed in turn, unmatched build rows follow.  CUDA path vs the CPU oracle, the
pair list itself through the C ABI, and TPC-H Q13's join at SF1 on one and on three segments."""
import ctypes as C

import numpy as np
import pytest

from cloudberry_b200 import capi, tpch
from cloudberry_b200 import plan as P
from cloudberry_b200.relation import HostRelation
from gpu_util import canon, to_device
from test_gpu_capacity import _outer_join_plan
from test_gpu_edge import agg_over, dim, fact, make

pytestmark = pytest.mark.gpu

NONE = 0xFFFFFFFF
AGGS = [("s", P.AGG_SUM, "amt"), ("n", P.AGG_COUNT_STAR, None), ("ck", P.AGG_COUNT, "k"), ("sw", P.AGG_SUM, "w")]
NAMES = ["k", "g", "amt", "dk", "w", "c"]


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def _run(ctx, plan, rels_p, generic=False, mem_kb=16):
    dev = to_device(ctx, rels_p)
    ex = capi.Executor(ctx, dev, force_generic=generic, operator_mem_kb=mem_kb)
    try:
        res = ex.run(plan)
        return res, int(ex.estate.contents.es_hashjoin_batches_run)
    finally:
        ex.close()
        for d in dev:
            d.free()


def _check_join(ctx, oracle, jointype, fo, fp, do, dp, generic=False, min_nbatch=4):
    """the joined rows and an aggregate over them, under a 16 KB operator memory, equal the oracle's"""
    j = _outer_join_plan(jointype, fo, do)
    got, batches = _run(ctx, j, [fp, dp], generic)
    assert canon(got.rows) == canon(oracle.execute(j, [[fo, do]]).rows)
    assert max(v["hashjoin_nbatch"] for v in got.instrument.values()) >= min_nbatch
    plan = agg_over(j, NAMES, ["g", "c"], AGGS)
    got2, _ = _run(ctx, plan, [fp, dp], generic)
    assert canon(got2.rows) == canon(oracle.execute(plan, [[fo, do]]).rows)
    return got.rows, batches


@pytest.mark.parametrize("generic", [False, True])
@pytest.mark.parametrize("jointype,dup", [(P.JOIN_INNER, 3), (P.JOIN_LEFT, 3), (P.JOIN_RIGHT, 1), (P.JOIN_RIGHT, 3),
                                          (P.JOIN_FULL, 1), (P.JOIN_FULL, 3)])
def test_join_types(ctx, oracle, jointype, dup, generic):
    """NULL keys on both sides, ~30 000 probe and 8 000 build rows over a key range wide enough that a 16 KB budget splits the
    build side into 16 batches"""
    fo, fp = make(fact, 30011, seed=51, null_frac=0.05, kmax=20000)
    do, dp = make(dim, 8000, seed=52, null_frac=0.05, dup=dup, kmax=20000)
    rows, batches = _check_join(ctx, oracle, jointype, fo, fp, do, dp, generic)
    assert batches > 0
    if jointype in (P.JOIN_RIGHT, P.JOIN_FULL):
        assert any(r[2] is None for r in rows)          # unmatched build rows (no probe side)
    if jointype in (P.JOIN_LEFT, P.JOIN_FULL):
        assert any(r[4] is None for r in rows)          # unmatched probe rows (no build side)


@pytest.mark.parametrize("case", ["probe_keys_all_null", "build_keys_all_null", "empty_probe", "empty_build", "sparse_probe"])
@pytest.mark.parametrize("jointype", [P.JOIN_INNER, P.JOIN_LEFT, P.JOIN_RIGHT, P.JOIN_FULL])
def test_edges(ctx, oracle, case, jointype):
    """every probe key NULL: LEFT / FULL give each probe row once, NULL-extended (NULL-keyed probe rows belong to batch 0); every
    build key NULL: RIGHT / FULL give each build row once; an empty side; a probe side so small that most batches get no row"""
    nf, fnull, nd, dnull = {"probe_keys_all_null": (5000, 1.0, 8000, 0.0), "build_keys_all_null": (5000, 0.0, 8000, 1.0),
                            "empty_probe": (0, 0.0, 8000, 0.0), "empty_build": (5000, 0.1, 0, 0.0),
                            "sparse_probe": (3, 0.0, 8000, 0.0)}[case]
    fo, fp = make(fact, nf, seed=53, null_frac=fnull, kmax=20000)
    do, dp = make(dim, nd, seed=54, null_frac=dnull, dup=3, kmax=20000)
    if case == "sparse_probe":
        for f in (fo, fp):
            f.columns[0][:] = do.columns[0][[0, 3, 6]]      # three probe rows, each with partners
    rows, _ = _check_join(ctx, oracle, jointype, fo, fp, do, dp, min_nbatch=1 if nd == 0 else 4)
    if case == "probe_keys_all_null" and jointype in (P.JOIN_LEFT, P.JOIN_FULL):
        probe = [r for r in rows if r[2] is not None]   # amt: probe side present
        assert len(probe) == fo.nrows and all(r[4] is None for r in probe)
    if case == "build_keys_all_null" and jointype in (P.JOIN_RIGHT, P.JOIN_FULL):
        build = [r for r in rows if r[4] is not None]   # w: build side present
        assert len(build) == do.nrows and all(r[2] is None for r in build)


def _skew_dim(n_unique, n_hot, hot_key, seed=55, kmax=20000):
    rng = np.random.default_rng(seed)
    keys = rng.permutation(np.setdiff1d(np.arange(kmax), [hot_key]))[:n_unique]
    keys = rng.permutation(np.concatenate([keys, np.full(n_hot, hot_key)])).astype(np.int32)
    n = len(keys)
    return HostRelation("dim", ["dk", "w", "c"], [P.INT4, P.INT8, P.DICT8], [keys, rng.integers(0, 100, n), rng.integers(0, 5, n)],
                        nulls=[None, None, None], dict_texts=[None, None, ["c%d" % i for i in range(5)]])


@pytest.mark.parametrize("jointype", [P.JOIN_INNER, P.JOIN_RIGHT, P.JOIN_FULL])
def test_skewed_build_side(ctx, oracle, jointype):
    """one build key ~2 000 times beside 6 000 unique keys: its batch is the fullest and sizes the table"""
    fo, fp = make(fact, 30011, seed=56, null_frac=0.05, kmax=20000)
    hot = int(fo.columns[0][np.flatnonzero(fo.nulls[0] == 0)[0]])
    do, dp = make(_skew_dim, 6000, 2000, hot)
    rows, _ = _check_join(ctx, oracle, jointype, fo, fp, do, dp)
    assert sum(1 for r in rows if r[3] == hot) >= 2000


def _pairs(ctx, ht, rel, fill_outer, fill_inner, pending=None):
    G = ctx.L
    pairs = capi.CbgpuPairs()
    passes = C.c_int64()
    rc = G.cbgpu_ht_probe_pairs_batched(ctx.h, ht, rel.h, (C.c_int32 * 1)(0), 1, fill_outer, fill_inner,
                                        C.cast(pending, C.c_void_p) if pending else None, None, C.byref(passes), C.byref(pairs))
    if rc:
        return rc, None, None, int(passes.value)
    n = int(pairs.npairs)
    o, i = np.zeros(n, dtype=np.uint32), np.zeros(n, dtype=np.uint32)
    if n:
        ctx.check(G.cbgpu_read_u32(ctx.h, pairs.outer_idx, n, o.ctypes.data))
        ctx.check(G.cbgpu_read_u32(ctx.h, pairs.inner_idx, n, i.ctypes.data))
    G.cbgpu_pairs_free(C.byref(pairs))
    return 0, o, i, int(passes.value)


def test_pair_list_through_the_abi(ctx):
    """cbgpu_ht_probe_pairs_batched over an 8-batch table: deterministic, the matches are the join of the keys, each unmatched row
    of either side comes once, the outer part is (batch, outer row) ordered and the unmatched build rows follow in row order"""
    rng = np.random.default_rng(57)
    ik = rng.integers(0, 3000, 6000).astype(np.int32)
    inul = (rng.random(6000) < 0.05).astype(np.uint8)
    ok = rng.integers(0, 4000, 20011).astype(np.int32)
    onul = (rng.random(20011) < 0.05).astype(np.uint8)
    inner = capi.DeviceRelation.from_host(ctx, HostRelation("i", ["k"], [P.INT4], [ik], nulls=[inul]))
    outer = capi.DeviceRelation.from_host(ctx, HostRelation("o", ["k"], [P.INT4], [ok], nulls=[onul]))
    ht = C.c_void_p()
    ctx.check(ctx.L.cbgpu_ht_build_batched(ctx.h, inner.h, (C.c_int32 * 1)(0), 1, 8, C.byref(ht)))
    try:
        assert ctx.L.cbgpu_ht_nbatch(ht) == 8 and ctx.L.cbgpu_ht_has_duplicates(ht)
        rc, o1, i1, passes = _pairs(ctx, ht, outer, 1, 1)
        assert rc == 0 and passes == 8
        rc, o2, i2, _ = _pairs(ctx, ht, outer, 1, 1)
        assert rc == 0 and o1.tobytes() == o2.tobytes() and i1.tobytes() == i2.tobytes()
        # the matches, as a multiset, are the numpy join of the non-NULL keys
        m = (o1 != NONE) & (i1 != NONE)
        by_key = {}
        for r in np.flatnonzero(inul == 0):
            by_key.setdefault(int(ik[r]), []).append(int(r))
        want = sorted((int(r), j) for r in np.flatnonzero(onul == 0) for j in by_key.get(int(ok[r]), []))
        assert sorted(zip(o1[m].tolist(), i1[m].tolist())) == want
        # every unmatched row of either side exactly once
        matched_o, matched_i = set(o1[m].tolist()), set(i1[m].tolist())
        uo = o1[i1 == NONE]
        ui = i1[o1 == NONE]
        assert sorted(uo.tolist()) == sorted(set(range(len(ok))) - matched_o)
        assert sorted(ui.tolist()) == sorted(set(range(len(ik))) - matched_i)
        # order: the outer part first, in at most 8 increasing runs of outer ids (a row's partners in build row order); then the
        # unmatched build rows, increasing
        nout = int(np.count_nonzero(o1 != NONE))
        assert (o1[:nout] != NONE).all() and (o1[nout:] == NONE).all()
        assert int(np.count_nonzero(np.diff(o1[:nout].astype(np.int64)) < 0)) <= 7
        same = np.diff(o1[:nout].astype(np.int64)) == 0
        assert (np.diff(i1[:nout].astype(np.int64))[same] > 0).all()
        assert (np.diff(i1[nout:].astype(np.int64)) > 0).all()
        # the caller's interrupt check is polled before each batch: pending at the 3rd poll stops the call with its code
        polls = {"n": 0}

        def pending(_arg):
            polls["n"] += 1
            return 1 if polls["n"] >= 3 else 0
        cb = capi.PENDING_FN(pending)
        rc, _, _, passes = _pairs(ctx, ht, outer, 1, 1, cb)
        assert rc == -8 and polls["n"] == 3 and passes == 2
        rc, o3, i3, _ = _pairs(ctx, ht, outer, 1, 1)
        assert rc == 0 and o3.tobytes() == o1.tobytes() and i3.tobytes() == i1.tobytes()
    finally:
        ctx.L.cbgpu_ht_free(ht)
        inner.free()
        outer.free()


def _q13_tables(sf):
    n_cust, n_ord = tpch.sizes(sf)["customer"], tpch.sizes(sf)["orders"]
    cust = tpch._rel("customer", tpch.gen_customer(42, n_cust), {"c_mktsegment": tpch.SEGMENTS}).set_dict_hashes(capi.hashbpchar)
    orders = tpch._rel("orders", tpch.gen_orders(42, n_ord, n_cust)).set_dict_hashes(capi.hashbpchar)
    return cust, orders


def _q13_plan(shape, nsegs=1):
    """range table [customer, orders]; the join's count(o_orderkey) per c_custkey.  (a): probe customer, build orders, LEFT;
    (b): probe orders, build customer, RIGHT (on several segments both sides are redistributed on the customer key)"""
    cs = P.SeqScan(1, [("c_custkey", P.Var(1, 1, P.INT4))])
    os_ = P.SeqScan(2, [("o_orderkey", P.Var(2, 1, P.INT8)), ("o_custkey", P.Var(2, 2, P.INT4))])
    if shape == "a":
        h = P.Hash(os_, [P.out_var(os_, 2)])
        j = P.HashJoin(P.JOIN_LEFT, cs, h, [P.out_var(cs, 1)], [("c_custkey", P.out_var(cs, 1)), ("o_orderkey", P.InnerVar(1, P.INT8))])
    else:
        outer, inner = os_, cs
        if nsegs > 1:
            outer = P.Motion(os_, P.MOTIONTYPE_HASH, [P.out_var(os_, 2)], nsegs)
            inner = P.Motion(cs, P.MOTIONTYPE_HASH, [P.out_var(cs, 1)], nsegs)
        h = P.Hash(inner, [P.out_var(inner, 1)])
        j = P.HashJoin(P.JOIN_RIGHT, outer, h, [P.out_var(outer, 2)], [("c_custkey", P.InnerVar(1, P.INT4)), ("o_orderkey", P.out_var(outer, 1))])
    v = tpch._child_var(j)
    agg = P.Agg(j, P.AGG_HASHED, P.AGGSPLIT_SIMPLE, [1], [("c_custkey", v("c_custkey")), ("n", P.Aggref(P.AGG_COUNT, v("o_orderkey")))],
                num_groups=200000)
    return agg if nsegs == 1 else P.Motion(agg, P.MOTIONTYPE_GATHER)


def _counts(rows, n_cust):
    got = np.full(n_cust + 1, -1, dtype=np.int64)
    keys = np.array([r[0] for r in rows], dtype=np.int64)
    assert len(np.unique(keys)) == len(keys) == n_cust
    got[keys] = [r[1] for r in rows]
    return got[1:]


@pytest.mark.parametrize("shape", ["a", "b"])
def test_tpch_q13_join_sf1(ctx, shape):
    """customer LEFT JOIN orders ON c_custkey = o_custkey, count(o_orderkey) per customer, at SF1 under a 256 KB budget (build
    sides of 32 and 256 batches): the counts, zero-order customers included, are numpy's and the unbudgeted run's"""
    cust, orders = _q13_tables(1)
    want = np.bincount(orders.columns[1], minlength=len(cust.columns[0]) + 1)[1:]
    assert (want == 0).any()
    plan = _q13_plan(shape)
    got, batches = _run(ctx, plan, [cust, orders], mem_kb=256)
    assert max(v["hashjoin_nbatch"] for v in got.instrument.values()) >= 8 and batches >= 8
    assert (_counts(got.rows, len(want)) == want).all()
    ref, _ = _run(ctx, plan, [cust, orders], mem_kb=0)
    assert canon(got.rows) == canon(ref.rows)


def test_tpch_q13_join_three_segments(ctx):
    """shape (b) on a 3-segment cluster, Redistribute Motions on the customer key, a 16 KB budget on every segment"""
    cust, orders = _q13_tables(1)
    want = np.bincount(orders.columns[1], minlength=len(cust.columns[0]) + 1)[1:]
    segs = [[cust.take(ci), orders.take(oi)] for ci, oi in zip(np.array_split(np.arange(len(cust.columns[0])), 3),
                                                                  np.array_split(np.arange(len(orders.columns[0])), 3))]
    dsegs = [to_device(ctx, s) for s in segs]
    cl = capi.Cluster(ctx, dsegs, operator_mem_kb=16)
    try:
        got = cl.run(_q13_plan("b", 3))
    finally:
        cl.close()
        for d in dsegs:
            for r in d:
                r.free()
    assert (_counts(got.rows, len(want)) == want).all()
