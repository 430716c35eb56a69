"""TPC-H Q13's join (customer LEFT OUTER JOIN orders ON c_custkey = o_custkey) at SF10 under operator memory budgets that split
its build side into batches: one JSON line per (plan shape, budget).

  shape a: probe customer (1.5 M rows), build orders (15 M rows, duplicate keys), LEFT join
  shape b: probe orders, build customer, RIGHT join

Both go through the pair probe, batch by batch (cbgpu_ht_probe_pairs_batched).  The join's output is materialised on the
device (cb_ExecProcNodeBatch); a run's time is a host clock around it, closed by a device synchronisation: median of --runs
after one warm-up.  "rows_equal" compares each customer's number of orders in the output with the run without a budget.  The
card's name and power limit come from nvidia-smi in the same process.

    python tools/multibatch_join_bench.py [--sf 10] [--budgets-kb 0,65536,8192,1024] [--runs 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from cloudberry_b200 import capi, tpch  # noqa: E402
from cloudberry_b200 import plan as P  # noqa: E402


def q13_join(shape):
    """range table [customer, orders]; output (c_custkey, o_orderkey)"""
    cs = P.SeqScan(1, [("c_custkey", P.Var(1, 1, P.INT4))])
    os_ = P.SeqScan(2, [("o_orderkey", P.Var(2, 1, P.INT8)), ("o_custkey", P.Var(2, 2, P.INT4))])
    if shape == "a":
        h = P.Hash(os_, [P.out_var(os_, 2)])
        return P.HashJoin(P.JOIN_LEFT, cs, h, [P.out_var(cs, 1)], [("c_custkey", P.out_var(cs, 1)), ("o_orderkey", P.InnerVar(1, P.INT8))])
    h = P.Hash(cs, [P.out_var(cs, 1)])
    return P.HashJoin(P.JOIN_RIGHT, os_, h, [P.out_var(os_, 2)], [("c_custkey", P.InnerVar(1, P.INT4)), ("o_orderkey", P.out_var(os_, 1))])


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=60).stdout.strip().splitlines()
        name, power = [x.strip() for x in out[0].split(",")]
        return name, power
    except (OSError, IndexError, ValueError, subprocess.SubprocessError):
        return "unknown", "unknown"


def orders_per_customer(rel, n_cust):
    """per customer, the output rows with an order (count(o_orderkey))"""
    cust, _ = rel.read_column(0)
    _, onull = rel.read_column(1)
    return np.bincount(cust[onull == 0].astype(np.int64), minlength=n_cust + 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sf", type=float, default=10)
    ap.add_argument("--budgets-kb", default="0,65536,8192,1024")
    ap.add_argument("--runs", type=int, default=5)
    a = ap.parse_args()
    budgets = [int(x) for x in a.budgets_kb.split(",")]
    name, power = gpu_info()
    sz = tpch.sizes(a.sf)
    n_cust, n_ord = sz["customer"], sz["orders"]
    cust = tpch._rel("customer", tpch.gen_customer(42, n_cust), {"c_mktsegment": tpch.SEGMENTS}).set_dict_hashes(capi.hashbpchar)
    orders = tpch._rel("orders", tpch.gen_orders(42, n_ord, n_cust)).set_dict_hashes(capi.hashbpchar)
    want = np.bincount(orders.columns[1].astype(np.int64), minlength=n_cust + 1)
    ctx = capi.Context(0)
    dev = [capi.DeviceRelation.from_host(ctx, r) for r in (cust, orders)]
    for shape in ("a", "b"):
        plan = q13_join(shape)
        ref = None
        for kb in budgets:
            ex = capi.Executor(ctx, dev, operator_mem_kb=kb)
            ms = []
            for i in range(a.runs + 1):
                before = ex.estate.contents.es_hashjoin_batches_run
                ctx.sync()
                t0 = time.perf_counter()
                out = ex.run_batch(plan)
                ctx.sync()
                t = (time.perf_counter() - t0) * 1e3
                passes = ex.estate.contents.es_hashjoin_batches_run - before
                if i > 0:
                    ms.append(t)
                if i < a.runs:
                    out.free()
            counts = orders_per_customer(out, n_cust)
            nrows = out.rows()
            out.free()
            ex.close()
            if ref is None:
                ref = counts
            nbatch, build_rows = 1, n_cust if shape == "b" else n_ord
            while kb > 0 and nbatch < 4096 and capi.gpu().cbgpu_ht_bytes_for((build_rows + nbatch - 1) // nbatch) > kb * 1024:
                nbatch <<= 1            # the executor's choice (hash_build, cb_exec.c)
            print(json.dumps({"query": "q13_join", "shape": shape, "sf": a.sf, "operator_mem_kb": kb, "nbatch": nbatch,
                              "passes": int(passes), "rows": int(nrows), "ms_median": round(float(np.median(ms)), 3),
                              "ms_all": [round(x, 3) for x in ms], "rows_equal_unbudgeted": bool((counts == ref).all()),
                              "counts_equal_numpy": bool((counts == want).all()), "gpu": name, "power_limit": power}), flush=True)
    for d in dev:
        d.free()
    ctx.close()


if __name__ == "__main__":
    main()
