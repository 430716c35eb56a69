"""The host side of pair-driven hash joins over a build side split into batches, without a GPU: libcbexec.so + libcbgpu.so over
the CUDA runtime of tests/native/fake_cudart.c, which computes nothing (kernels are no-ops, "device" memory is zeroed host
memory).  INNER and LEFT joins against duplicate build keys, RIGHT and FULL joins under a 16 KB operator memory are accepted,
launch kernels and return no rows; the key checks of the batched branch refuse what the pipelined probe refuses (float8 keys,
dictionary codes of two dictionaries).  The file is its own worker: the test runs it as a script with the fake runtime
preloaded."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_INC = "/usr/local/cuda/include"
UNSUPPORTED = -3


def _plans(P, fact, dim):
    """(name, plan, budget in KB) over the range table [fact, dim]"""
    from test_gpu_capacity import _outer_join_plan
    out = []
    for jt, name in ((P.JOIN_INNER, "inner"), (P.JOIN_LEFT, "left"), (P.JOIN_RIGHT, "right"), (P.JOIN_FULL, "full")):
        out.append((name, _outer_join_plan(jt, fact, dim), 16))

    def keyed(jt, fcol, ftype, dcol, dtype):
        sf = P.SeqScan(1, [("k", P.Var(1, fact.attno(fcol), ftype)), ("amt", P.Var(1, fact.attno("amt"), P.NUMERIC, 2))])
        sd = P.SeqScan(2, [("dk", P.Var(2, dim.attno(dcol), dtype)), ("w", P.Var(2, dim.attno("w"), P.INT8))])
        h = P.Hash(sd, [P.out_var(sd, 1)])
        return P.HashJoin(jt, sf, h, [P.out_var(sf, 1)], [("amt", P.out_var(sf, 2)), ("w", P.InnerVar(2, P.INT8))])
    # a float8 probe key against an int8 build key; dictionary codes of two different dictionaries
    out.append(("float8_key", keyed(P.JOIN_RIGHT, "x", P.FLOAT8, "w", P.INT8), 16))
    out.append(("two_dicts", keyed(P.JOIN_RIGHT, "g", P.DICT8, "c", P.DICT8), 16))
    return out


def worker():
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from cloudberry_b200 import capi
    from cloudberry_b200 import plan as P
    from test_gpu_edge import dim, fact
    fo = fact(30011, seed=61, null_frac=0.05, kmax=20000).set_dict_hashes(capi.hashbpchar)
    do = dim(8000, seed=62, null_frac=0.05, dup=3, kmax=20000).set_dict_hashes(capi.hashbpchar)
    ctx = capi.Context(0)
    dev = [capi.DeviceRelation.from_host(ctx, r) for r in (fo, do)]
    out = {}
    for name, plan, budget in _plans(P, fo, do):
        ex = capi.Executor(ctx, dev, operator_mem_kb=budget)
        before = ctx.launches()
        try:
            res = ex.run(plan)
            out[name] = {"rows": len(res.rows), "error": None, "nbatch": max(v["hashjoin_nbatch"] for v in res.instrument.values())}
        except capi.CbgpuError as e:
            out[name] = {"error": str(e), "code": e.code}
        out[name]["launches"] = ctx.launches() - before
        ex.close()
    for d in dev:
        d.free()
    ctx.close()
    print("MULTIBATCH " + json.dumps(out))


@pytest.mark.skipif(not os.path.exists(os.path.join(CUDA_INC, "cuda_runtime_api.h")), reason="needs the CUDA headers")
def test_multibatch_pair_joins_over_a_runtime_that_computes_nothing(tmp_path):
    so = str(tmp_path / "libfakecudart.so")
    subprocess.check_call(["gcc", "-O1", "-g", "-shared", "-fPIC", "-Wall", "-Werror", "-I" + CUDA_INC, "-o", so,
                           os.path.join(ROOT, "tests", "native", "fake_cudart.c")])
    p = subprocess.run([sys.executable, os.path.abspath(__file__)], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, LD_PRELOAD=so))
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("MULTIBATCH ")]
    assert p.returncode == 0 and lines, (p.stdout[-2000:], p.stderr[-4000:])
    out = json.loads(lines[0][len("MULTIBATCH "):])
    # (the no-op runtime reports no duplicate build keys, so INNER / LEFT take the pipelined probe here; RIGHT / FULL always take
    # the pair probe, and with the build side in batches that is the batched one)
    for name in ("inner", "left", "right", "full"):
        assert out[name]["error"] is None and out[name]["rows"] == 0, out[name]
        assert out[name]["launches"] > 0 and out[name]["nbatch"] >= 4, out[name]
    for name, frag in (("float8_key", "float8 join keys"), ("two_dicts", "two different dictionaries")):
        assert out[name]["code"] == UNSUPPORTED and frag in out[name]["error"], out[name]


if __name__ == "__main__":
    worker()
