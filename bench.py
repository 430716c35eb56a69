#!/usr/bin/env python3
"""bench.py - TPC-H SF100 Q1 (AOCS scan -> hash aggregate) rows/sec on N GPU-segments.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line.
  value      whole-job rows/sec with the projected lineitem columns already resident in HBM
             (a "step" = one full pass of Q1 over the rank's lineitem shard through the ExecProcNode-style
             executor and the C ABI; weak scaling: every GPU-segment holds a full SF100-sized shard)
  e2e        the same query with HOST (pinned) buffers: every step copies the projected columns host->device,
             runs the query, and reads the result rows back
  roofline   algorithmic bytes (38 B/row: SURVEY.md 8d) / CUDA-event duration of the scan+agg kernel, against the
             measured HBM copy bandwidth in MEASURED_PEAKS.json
  cpu_baseline  Q1 on one host core over a bounded sample, rank 0, N=1: kind "reference" = the reference's own per-row code
             (block reader, numeric arithmetic, hash / equality, transition and final functions compiled where they lie into
             oracle/_ref/libexec_ref.so, driven by oracle/ref_q1.c), with the oracle's int64 restatement beside it under "port";
             kind "port" alone where oracle/_ref did not travel
  q3, q5     whole-query lines of the metric's join queries (rows scanned / s, whole-query roofline fraction, Motion bytes), each
             with its own cpu_baseline (the oracle on one core over an SF1 database) at N=1
`--impl reference` times the same reference code on all host cores, one process per core (the reference server itself cannot
be built here: no bison/flex, see DESIGN.md), with the same metric / config keys; CBGPU_BENCH_CPU=port forces the restatement.
`--dump-outputs DIR` also writes every query's result rows from its last timed step as DIR/<query>.npy; the inputs are generated
from fixed seeds, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

Q1_BYTES_PER_ROW = 38       # qty 8 + extendedprice 8 + discount 8 + tax 8 + shipdate 4 + returnflag 1 + linestatus 1
Q1_COLS = ["l_quantity", "l_extendedprice", "l_discount", "l_tax", "l_returnflag", "l_linestatus", "l_shipdate"]


def measured_peak():
    try:
        d = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy bandwidth)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            # only this rank's GPU: querying all eight per sample is too slow for a timed region of ~100 ms
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                                       "-lms", "10"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def ready(self):
        """has nvidia-smi written its first sample yet?"""
        try:
            return self.p is None or os.path.getsize(self.f.name) > 0
        except OSError:
            return True

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.p:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        clocks, reasons, mx = [], set(), None
        for line in open(self.f.name):
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9 or parts[0] != str(self.gpu):
                continue
            try:
                clocks.append(float(parts[1]))
                mx = float(parts[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        if clocks:
            clocks.sort()
            out.update({"sm_mhz": clocks[len(clocks) // 2], "sm_max_mhz": mx, "reasons": sorted(reasons),
                        "samples": len(clocks)})
        return out


def host_cores():
    """cores this process may actually use: the affinity mask, capped by the cgroup's CPU quota if there is one"""
    try:
        n = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return n


def workload_name(sf, world):
    """config.workload: the same string on both arms"""
    return "TPC-H SF%g Q1 on %d GPU-segment(s) (scan + hash-agg kernel%s)" % (
        sf, world, ", two-stage agg over Redistribute Motion" if world > 1 else ", no Motion")


def cpu_q1_sample(nthreads, rows_total, seed=42):
    """Run the oracle's Q1 on a bounded sample of the same synthetic lineitem; returns (rows/s, rows, seconds)."""
    from cloudberry_b200 import tpch
    from oracle import oracle as O
    sz = tpch.sizes(100)
    per = max(1, rows_total // nthreads)
    segs = []
    nation, region = tpch.gen_nation_region()
    for s in range(nthreads):
        cols = tpch.gen_lineitem(seed, sz["lineitem"], sz["supplier"], sz["part"], lo=s * per, hi=(s + 1) * per)
        segs.append([tpch._rel("lineitem", cols)])
    plan = tpch.q1_plan(nthreads) if nthreads > 1 else tpch.q1_plan(1)
    O.lib()
    t0 = time.perf_counter()
    res = O.execute(plan, segs, nthreads=nthreads)
    dt = time.perf_counter() - t0
    assert len(res.rows) >= 1
    return per * nthreads / dt, per * nthreads, dt


REF_Q1_NOTE = ("reference code per row: datumstreamblock.c block reader over reference-written AOCS column files (CRC-32C verified), "
               "numeric.c numeric_sub/_mul/_add + numeric_avg_accum/numeric_sum/numeric_avg, varchar.c hashbpchar/bpchareq, hashfn.c, "
               "compiled where they lie into oracle/_ref/libexec_ref.so; executor glue (ExecScan/ExecAgg/interpreter, not buildable "
               "here: no bison/flex) restated minimally in oracle/ref_q1.c, so a lower bound on the reference's CPU time")


def _ref_q1_worker(idx, per, seed, nsteps, barrier, conn):
    """One CPU segment: its slice of the synthetic lineitem as reference-written column files, then nsteps timed Q1 runs."""
    try:
        from cloudberry_b200 import tpch
        from oracle import oracle as O
        sz = tpch.sizes(100)
        li = tpch._rel("lineitem", tpch.gen_lineitem(seed, sz["lineitem"], sz["supplier"], sz["part"], lo=idx * per, hi=(idx + 1) * per))
        q = O.RefQ1(li)
        times = []
        for _ in range(nsteps):
            barrier.wait()
            t0 = time.perf_counter()
            rows, passed = q.run(tpch.Q1_CUTOFF)
            times.append(time.perf_counter() - t0)
            assert len(rows) >= 1 and passed > 0
        q.free()
        conn.send(times)
    except BaseException as e:      # report instead of leaving the parent waiting on the barrier
        try:
            barrier.abort()
        except Exception:
            pass
        conn.send("error: %r" % (e,))
    finally:
        conn.close()


def ref_q1_steps(nproc, per, nsteps, seed=42):
    """Q1 through the reference's own per-row functions (oracle/ref_q1.c) on nproc CPU segments (one process each, as the
    reference runs one backend per segment); returns the per-step wall times (max over segments), or None if unavailable."""
    import multiprocessing as mp
    from oracle import oracle as O
    if O.ref_exec_lib() is None or os.environ.get("CBGPU_BENCH_CPU") == "port":
        return None
    # spawn, not fork: the main arm calls this from a process that holds a CUDA context and pinned buffers
    ctx = mp.get_context("spawn")
    barrier = ctx.Barrier(nproc)
    pipes, procs = [], []
    for i in range(nproc):
        a, b = ctx.Pipe(duplex=False)
        pr = ctx.Process(target=_ref_q1_worker, args=(i, per, seed, nsteps, barrier, b), daemon=True)
        pr.start()
        b.close()
        pipes.append(a)
        procs.append(pr)
    results = []
    for a in pipes:
        try:
            results.append(a.recv() if a.poll(600) else "error: timed out")
        except (EOFError, OSError):
            results.append("error: a worker process died")
    for pr in procs:
        pr.join(10)
    if any(isinstance(r, str) for r in results):
        sys.stderr.write("ref_q1: %s\n" % [r for r in results if isinstance(r, str)][0])
        return None
    return [max(r[k] for r in results) for k in range(nsteps)]


def cpu_join_samples(sf=1):
    """Q3 / Q5 through the oracle on one thread over an SF`sf` synthetic database -> {q: cpu_baseline object}."""
    from cloudberry_b200 import harness, tpch
    from oracle import oracle as O
    rels = tpch.gen_tables(sf, O.hashbpchar)
    sz = tpch.sizes(sf)
    out = {}
    for q, plan in (("q3", tpch.q3_plan(tpch.SEGMENTS.index("MACHINERY"), 1)), ("q5", tpch.q5_plan(tpch.REGIONS.index("AMERICA"), 1))):
        O.execute(plan, [rels], nthreads=1)         # warm-up (page faults of the hash tables)
        t0 = time.perf_counter()
        res = O.execute(plan, [rels], nthreads=1)
        dt = time.perf_counter() - t0
        rows_in, _ = harness.query_rows_bytes(q, sz)
        assert len(res.rows) >= 1
        out[q] = {"value": rows_in / dt, "unit": "rows/s", "cores": 1, "kind": "port",
                  "sample": "%s over an SF%g synthetic database (%d base-table rows scanned), %.2f s, one thread (row-at-a-time oracle)" % (
                      q.upper(), sf, rows_in, dt)}
    return out


def run_reference(args):
    """CPU arm.  Where oracle/_ref/libexec_ref.so exists: TPC-H Q1 through the reference's own per-row code, one process per host
    core (kind "reference"); else the restated reference path (oracle, kind "port").  Bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    nthreads = min(cores, 256)          # every host core the process may use: one CPU segment (process) each
    from cloudberry_b200 import tpch as _tpch
    per_ref = 1_000_000
    steps = ref_q1_steps(nthreads, per_ref, args.warmup + args.steps)
    if steps is not None:
        timed = steps[args.warmup:]
        dt = sum(timed)
        value = per_ref * nthreads * args.steps / dt
        sample = "Q1 over %d synthetic lineitem rows per step (%d CPU segments = processes x %d rows; %s)" % (
            per_ref * nthreads, nthreads, per_ref, REF_Q1_NOTE)
        line = {
            "impl": "reference", "metric": "TPC-H SF100 Q1 rows/sec", "value": value, "unit": "rows/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "numeric", "data": "synthetic",
            "config": {"workload": workload_name(args.sf, args.gpus),
                       "rows_per_gpu": _tpch.sizes(100)["lineitem"],
                       "note": "the reference's own per-row code for the path on the host cores; the reference server itself needs bison/flex and cannot be built here"},
            "cpu_baseline": {"value": value, "unit": "rows/s", "cores": nthreads, "kind": "reference", "sample": sample},
            "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        print(json.dumps(line))
        return
    rows = min(64_000_000, 2_000_000 * nthreads)
    # generate once, time K steps after W warm-ups
    from cloudberry_b200 import tpch
    from oracle import oracle as O
    sz = tpch.sizes(100)
    per = rows // nthreads
    segs = [[tpch._rel("lineitem", tpch.gen_lineitem(42, sz["lineitem"], sz["supplier"], sz["part"], lo=s * per, hi=(s + 1) * per))]
            for s in range(nthreads)]
    plan = tpch.q1_plan(nthreads) if nthreads > 1 else tpch.q1_plan(1)
    O.lib()
    for _ in range(args.warmup):
        O.execute(plan, segs, nthreads=nthreads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        O.execute(plan, segs, nthreads=nthreads)
    dt = time.perf_counter() - t0
    value = per * nthreads * args.steps / dt
    sample = "Q1 over %d synthetic lineitem rows per step (%d CPU segments x %d rows, two-stage aggregation)" % (per * nthreads, nthreads, per)
    line = {
        "impl": "reference", "metric": "TPC-H SF100 Q1 rows/sec", "value": value, "unit": "rows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": workload_name(args.sf, args.gpus), "rows_per_gpu": sz["lineitem"],
                   "note": "CPU restatement of the reference path (oracle/); the reference server needs bison/flex and cannot be built here"},
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": nthreads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def _rows_as_text(kind, rows):
    from cloudberry_b200 import ssb, tpch
    if kind == "q1":
        return tpch.format_q1(rows)
    if kind == "q3":
        return tpch.format_q3(rows)
    if kind == "q5":
        return tpch.format_q5(rows, tpch.NATIONS)
    return ssb.canon(rows)


def traffic_of(kernel_name):
    """dram bytes per launch of the dominant kernel from the round's ncu --set full capture (tools/gpu_round.sh writes
    profiles/q1_kernel_traffic.json with the sha256 of the kernel source it measured): null when the source has changed since."""
    import hashlib
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "q1_kernel_traffic.json")))
        sha = hashlib.sha256(open(os.path.join(ROOT, "cloudberry_b200", "csrc", "scan_agg.cu"), "rb").read()).hexdigest()
        if d.get("source_sha256") == sha and d.get("kernel", "").split("(")[0] == kernel_name.split("(")[0]:
            return d.get("dram_bytes_per_launch")
    except Exception:
        pass
    return None


def dump_outputs(path, results):
    """--dump-outputs: each query's rows from its last timed step as DIR/<query>.npy, float64 of shape (rows, columns) in
    the plan's output column order; numeric columns hold their decimal value, NULL is NaN.  The rows are sorted so that
    two builds can be compared file by file whatever order their aggregates emit groups in."""
    import math
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, rows in results.items():
        vals = sorted(([float("nan") if x is None else float(x) for x in r] for r in rows),
                      key=lambda r: [(math.isnan(x), 0.0 if math.isnan(x) else x) for x in r])
        a = np.array(vals, dtype=np.float64).reshape(len(vals), len(vals[0]) if vals else 0)
        np.save(os.path.join(path, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of every device-resident query (the end-to-end loop runs --e2e-steps)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--sf", type=float, default=100.0, help="scale factor of each GPU-segment's shard (default: the BASELINE config)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--joins-sf", type=float, default=None,
                    help="scale factor of the ONE database Q5 runs on at N > 1 (default: 300 on 8 GPUs = BASELINE configs[3], else --sf); "
                         "Q3 always runs on SF --sf (configs[2])")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-joins", action="store_true", help="skip the Q3 / Q5 join pipelines (extra keys q3, q5)")
    ap.add_argument("--no-ssb", action="store_true", help="skip SSB Q4.1 - Q4.3 (extra key ssb)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write every query's result rows from its last timed step to DIR/<query>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the GPU path's rows; the reference arm has none")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
        return

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        torch.cuda.set_device(local_rank)
        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist = dist_mod

    from cloudberry_b200 import bench_golden as BG
    from cloudberry_b200 import capi, tpch
    import numpy as np

    gold = BG.load() or {}
    checks = []                 # every result_check of this run; any MISMATCH fails the run (rc 1) after the line is printed

    def result_check(kind, rows, want_rows, missing):
        if want_rows is None:
            return "unchecked: %s" % missing
        c = BG.check(kind, _rows_as_text(kind if kind in ("q1", "q3", "q5") else "ssb", rows), want_rows)
        checks.append(c)
        return c

    ctx = capi.Context(local_rank)
    G = ctx.L
    sz = tpch.sizes(int(args.sf) if float(args.sf).is_integer() else args.sf)
    nrows = sz["lineitem"]
    li_types = [t for _, t in tpch.SCHEMA["lineitem"]]
    li = capi.DeviceRelation(ctx, nrows, li_types, name="lineitem")
    # rank r holds rows [r * nrows, (r + 1) * nrows) of an (N x SF)-sized table: a valid (random) distribution for Q1
    ctx.check(G.cbgpu_gen_lineitem(ctx.h, li.h, 42, rank * nrows, sz["supplier"], sz["part"]))
    ctx.sync()
    rt = [li]
    motion = None
    if world > 1:
        # SetupInterconnect: rank 0 creates the NCCL rendezvous token, everyone joins
        ids = [capi.Motion.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        motion = capi.Motion(ctx, rank, world, ids[0])
    ex = capi.Executor(ctx, rt, motion=motion)
    # one segment: HashAggregate <- Seq Scan.  Several: Gather Motion <- Finalize HashAggregate <-
    # Redistribute Motion <- Partial HashAggregate <- Seq Scan (expected/aggregates.out:3313-3328)
    plan1 = tpch.q1_plan(world)

    def barrier():
        ctx.sync()
        if dist:
            dist.barrier()
        ctx.sync()

    def bcast_rows(rows):
        """the Gather receiver's rows, on every rank (so that all ranks agree on the run's verdict)"""
        if not dist:
            return rows
        box = [rows if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        return box[0]

    def maxr(vals):
        if not dist:
            return [float(v) for v in vals]
        import torch
        t = torch.tensor([float(v) for v in vals], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    def sumr(vals):
        if not dist:
            return [float(v) for v in vals]
        import torch
        t = torch.tensor([float(v) for v in vals], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(x) for x in t.tolist()]

    # ---- device-resident: warm-up, then K timed steps ----
    sampler = ClockSampler(local_rank)
    sampler.start()         # covers warm-up and the timed region: both are the same load
    for _ in range(args.warmup):
        res = ex.run(plan1)
    # keep the same load up (untimed) until the clock sampler is actually sampling; with several ranks the number of
    # extra steps must be the same everywhere (every step holds Motions), so it is fixed there
    if dist:
        for _ in range(80):
            res = ex.run(plan1)
    else:
        t_wait = time.perf_counter()
        while not sampler.ready() and time.perf_counter() - t_wait < 3.0:
            res = ex.run(plan1)
    kernel_ms = []
    barrier()
    l0 = ctx.launches()
    hs0 = (motion.host_syncs(), motion.collectives()) if motion else (0, 0)
    ctx.timer_start()
    knames = []
    for _ in range(args.steps):
        ctx.kernel_log_reset()
        res = ex.run(plan1)
        kn, km = ctx.longest_kernel()     # the step's dominant kernel, timed by its own CUDA events
        kernel_ms.append(km)
        knames.append(kn)
    ms = ctx.timer_stop_ms()
    l1 = ctx.launches()
    hs1 = (motion.host_syncs(), motion.collectives()) if motion else (0, 0)
    barrier()
    clocks = sampler.stop()
    kname = knames[-1]
    q1_rows = bcast_rows(res.rows)
    outputs = {"q1": q1_rows}        # --dump-outputs: each query's rows from its last timed step
    ngroups = len(q1_rows)
    ms = maxr([ms])[0]
    total_rows = nrows * world
    value = total_rows * args.steps / (ms / 1e3)
    peak, peak_src = measured_peak()
    kms = sorted(kernel_ms)[len(kernel_ms) // 2]
    achieved = nrows * Q1_BYTES_PER_ROW / (kms / 1e3) / 1e9
    gq1 = gold.get(BG.key("q1", args.sf))
    q1_check = result_check("q1", q1_rows, BG.q1_rows(gq1, world) if gq1 and len(gq1["shards"]) >= world and gq1["rows_per_shard"] == nrows else None,
                            "no golden rows for SF%g x %d shards" % (args.sf, world))

    # ---- end to end: host (pinned) buffers -> H2D -> query -> rows back ----
    e2e = None
    if not args.no_e2e:
        cols = [tpch.SCHEMA["lineitem"].index(next(c for c in tpch.SCHEMA["lineitem"] if c[0] == n)) for n in Q1_COLS]
        # N = 1: the whole SF100 shard (22.8 GB pinned).
        # N > 1: the same, when the host has the memory to pin a full shard per rank (all ranks must agree); else a sample
        full = nrows * sum(capi.P.TYPE_WIDTH[li_types[c]] for c in cols)
        try:
            import psutil
            roomy = psutil.virtual_memory().available > 2.0 * full * world
        except Exception:
            roomy = False
        if dist:
            roomy = maxr([0.0 if roomy else 1.0])[0] < 0.5
        e2e_rows = nrows if (world == 1 or roomy) else min(nrows, 96_000_000)
        li_e, ex_e = li, ex
        if e2e_rows != nrows:
            li_e = capi.DeviceRelation(ctx, e2e_rows, li_types, name="lineitem_e2e")
            ctx.check(G.cbgpu_gen_lineitem(ctx.h, li_e.h, 42, rank * nrows, sz["supplier"], sz["part"]))
            ex_e = capi.Executor(ctx, [li_e], motion=motion)
        host = {}
        ok = True
        for c in cols:
            w = capi.P.TYPE_WIDTH[li_types[c]]
            p = G.cbgpu_host_alloc(e2e_rows * w)
            if not p:
                ok = False
                break
            host[c] = p
            ctx.check(G.cbgpu_rel_read_column(li_e.h, c, 0, e2e_rows, p, None))
        if dist:
            ok = maxr([0.0 if ok else 1.0])[0] < 0.5          # every step holds Motions: all ranks run it, or none
        narrow = {}
        if ok:
            # what crosses PCIe: every column in the narrowest two's-complement width that holds its values (the loader knows
            # each column's min / max as a storage layer knows its block statistics): numeric(15,2) l_quantity travels as
            # int16, l_extendedprice as int32, l_discount / l_tax as int8 - and is sign-extended on the device
            # (cbgpu_rel_load_column_narrow).  The relation in HBM, the query and its rows are the same as with int64 columns.
            import ctypes as C
            for c in cols:
                w = capi.P.TYPE_WIDTH[li_types[c]]
                if w not in (4, 8) or li_types[c] == capi.P.FLOAT8:
                    continue
                a = np.ctypeslib.as_array(C.cast(host[c], C.POINTER(C.c_int64 if w == 8 else C.c_int32)), shape=(e2e_rows,))
                lo_v, hi_v = (int(a.min()), int(a.max())) if e2e_rows else (0, 0)
                nw = next((k for k in (1, 2, 4) if k < w and -(1 << (8 * k - 1)) <= lo_v and hi_v < (1 << (8 * k - 1))), w)
                if nw == w:
                    continue
                pn = G.cbgpu_host_alloc(e2e_rows * nw)
                if not pn:
                    continue
                dst = np.ctypeslib.as_array(C.cast(pn, C.POINTER({1: C.c_int8, 2: C.c_int16, 4: C.c_int32}[nw])), shape=(e2e_rows,))
                np.copyto(dst, a, casting="unsafe")
                narrow[c] = (pn, nw)
        if ok:
            h2d_full = sum(e2e_rows * capi.P.TYPE_WIDTH[li_types[c]] for c in cols)
            h2d = sum(e2e_rows * (narrow[c][1] if c in narrow else capi.P.TYPE_WIDTH[li_types[c]]) for c in cols)
            d2h = 0

            def e2e_step(packed):
                for c in cols:
                    if packed and c in narrow:
                        li_e.load_column_ptr(c, narrow[c][0], narrow[c][1])
                    else:
                        li_e.load_column_ptr(c, host[c])
                r = ex_e.run(plan1)
                return r

            def e2e_timed(packed):
                e2e_step(packed)
                barrier()
                t0 = time.perf_counter()
                ctx.timer_start()
                for _ in range(args.e2e_steps):
                    r = e2e_step(packed)
                e_ms = ctx.timer_stop_ms()
                wall = time.perf_counter() - t0
                barrier()
                return r, maxr([max(e_ms, wall * 1e3)])[0]
            r_full, full_ms = e2e_timed(False)
            r, e_ms = e2e_timed(True)
            d2h = sum(8 * len(row) for row in r.rows)
            e2e = {"value": e2e_rows * world * args.e2e_steps / (e_ms / 1e3), "unit": "rows/s", "h2d_bytes_per_step": h2d * world,
                   "d2h_bytes_per_step": d2h * world, "steps": args.e2e_steps, "ms_per_step": e_ms / args.e2e_steps,
                   "rows_per_gpu": e2e_rows, "bytes_per_row_shipped": h2d / e2e_rows,
                   "host_column_widths": {Q1_COLS[i]: (narrow[c][1] if c in narrow else capi.P.TYPE_WIDTH[li_types[c]]) for i, c in enumerate(cols)},
                   "note": "projected columns from pinned host memory, each in the narrowest integer width that holds its values "
                           "(chosen from the column's min / max, as a storage layer's block statistics allow), one cudaMemcpyAsync per "
                           "column, sign-extended on the device, then the query; PCIe-bound",
                   "decoded_int64": {"ms_per_step": full_ms / args.e2e_steps, "h2d_bytes_per_step": h2d_full * world,
                                     "value": e2e_rows * world * args.e2e_steps / (full_ms / 1e3), "bytes_per_row_shipped": h2d_full / e2e_rows,
                                     "note": "the same with every column shipped at its decoded width (numerics as int64)"}}
            if e2e_rows == nrows:
                gold_rows = BG.q1_rows(gq1, world) if gq1 and len(gq1["shards"]) >= world else None
                e2e["result_check"] = result_check("q1", bcast_rows(r.rows), gold_rows, "no golden rows")
                e2e["decoded_int64"]["result_check"] = result_check("q1", bcast_rows(r_full.rows), gold_rows, "no golden rows")
        for pn, _ in narrow.values():
            G.cbgpu_host_free(pn)
        for p in host.values():
            G.cbgpu_host_free(p)
        if ex_e is not ex:
            ex_e.close()
            li_e.free()

    # ---- the join queries of the metric (Q3, Q5).  N = 1: on the same resident tables.  N > 1: the BASELINE
    # configs "TPC-H SF100 Q3 on N GPU-segments" and "TPC-H SF300 Q5 on 8 GPU-segments": ONE database distributed over the
    # segments as the reference's DDL would (lineitem / orders by orderkey, customer by c_custkey, supplier by s_suppkey, nation
    # and region replicated), plans with Redistribute Motions; strong scaling ----
    joins = {}

    def timed_query(exq, plan, steps):
        for _ in range(args.warmup):
            r = exq.run(plan)
        barrier()
        l0j = ctx.launches()
        sent0 = motion.bytes_sent() if motion else 0
        h0 = (motion.host_syncs(), motion.collectives()) if motion else (0, 0)
        ctx.timer_start()
        for _ in range(steps):
            ctx.kernel_log_reset()
            r = exq.run(plan)
        qms = ctx.timer_stop_ms() / steps
        kn, km = ctx.longest_kernel()
        sent = (motion.bytes_sent() - sent0) / steps if motion else 0
        h1 = (motion.host_syncs(), motion.collectives()) if motion else (0, 0)
        launches = (ctx.launches() - l0j) // steps
        barrier()
        qms = maxr([qms])[0]
        sent = sumr([sent])[0]
        return {"rows": bcast_rows(r.rows), "ms": qms, "kernel": kn, "kernel_ms": km, "sent": int(sent), "launches": launches,
                "host_syncs": (h1[0] - h0[0]) / steps, "collectives": (h1[1] - h0[1]) / steps}

    def motion_desc():
        if not motion:
            return "none"
        return ("partition fused with the exchange over peer memory (CUDA IPC windows, NVLink stores, device-side epoch signals)"
                if motion.direct() else "staged partition + NCCL send/recv")

    if not args.no_joins:
        from cloudberry_b200 import harness
        q5_sf = args.joins_sf if (args.joins_sf and world > 1) else (300.0 if (world == 8 and args.sf == 100.0) else args.sf)
        runs = [("q3", args.sf)] + [("q5", q5_sf)]
        if world > 1:
            ex.close()
            ex = None
            li.free()           # the weak-scaling Q1 shard makes room for the distributed database
            li = None
        cur_sf, rt_all, owned, exj = None, None, [], None
        for q, jsf in runs:
            if jsf != cur_sf:
                if exj:
                    exj.close()
                for r_ in owned:
                    r_.free()
                if world == 1:
                    rt_all, _ = harness.device_tables(ctx, jsf, lineitem=li if jsf == args.sf else None)
                    owned = rt_all[1:] if jsf == args.sf else rt_all
                    exj = capi.Executor(ctx, rt_all)
                else:
                    rt_all, _ = harness.distributed_tables(ctx, motion, jsf, rank, world)
                    owned = rt_all
                    exj = capi.Executor(ctx, rt_all, motion=motion)
                cur_sf = jsf
            szj = tpch.sizes(int(jsf) if float(jsf).is_integer() else jsf)
            plan = (tpch.q3_plan(tpch.SEGMENTS.index("MACHINERY"), world, customer_replicated=False) if q == "q3"
                    else tpch.q5_plan(tpch.REGIONS.index("AMERICA"), world, replicated=False))
            t = timed_query(exj, plan, args.steps)
            outputs[q] = t["rows"]
            rows_in, nbytes = harness.query_rows_bytes(q, szj)
            g = gold.get(BG.key(q, jsf))
            joins[q] = {"value": rows_in / (t["ms"] / 1e3), "unit": "rows/s", "sf": jsf, "ms_per_step": t["ms"], "steps": args.steps, "rows_scanned": rows_in,
                        "scaling": "strong" if world > 1 else "n/a", "result_rows": len(t["rows"]),
                        "result_check": result_check(q, t["rows"], (BG.q3_rows(g) if q == "q3" else BG.q5_rows(g)) if g else None,
                                                     "no golden rows for SF%g" % jsf),
                        "gpu_launches_per_step": t["launches"],
                        "longest_kernel": t["kernel"], "longest_kernel_ms": t["kernel_ms"], "motion_bytes_per_step": t["sent"],
                        "motion": motion_desc(), "motion_host_syncs_per_step": t["host_syncs"], "motion_collectives_per_step": t["collectives"],
                        "roofline": {"bound": "hbm", "achieved": nbytes / (t["ms"] / 1e3) / 1e9, "peak": peak * world, "unit": "GB/s",
                                     "frac": nbytes / (t["ms"] / 1e3) / 1e9 / (peak * world), "algorithmic_bytes": nbytes,
                                     "note": "whole query (all pipelines, builds, Motions, top-N, host glue) against the projected base columns"}}
        if exj:
            exj.close()
        for r_ in owned:
            r_.free()

    # ---- SSB Q4.1 - Q4.3 (BASELINE configs[4]: wide hash-agg, HBM-bound group-by): ONE SF100 database, lineorder spread over
    # the segments by row range, the four dimensions replicated; star join + two-stage aggregation over Motions at N > 1 ----
    ssbres = None
    if not args.no_ssb:
        from cloudberry_b200 import ssb
        if world > 1 and ex:
            ex.close()
            ex = None
        if li and world > 1:
            li.free()
            li = None
        dev, ssz = ssb.device_tables(ctx, args.sf, capi.hashbpchar, rank, world)
        exs = capi.Executor(ctx, dev, motion=motion)
        rows_in, nbytes = ssb.query_rows_bytes(ssz)
        gs = gold.get(BG.key("ssb", args.sf))
        per, tot_ms = {}, 0.0
        for q in ("q4.1", "q4.2", "q4.3"):
            t = timed_query(exs, ssb.PLANS[q](world), args.steps)
            outputs["ssb_" + q.replace(".", "_")] = t["rows"]
            tot_ms += t["ms"]
            per[q] = {"ms_per_step": t["ms"], "groups": len(t["rows"]), "longest_kernel": t["kernel"], "longest_kernel_ms": t["kernel_ms"],
                      "gpu_launches_per_step": t["launches"], "motion_bytes_per_step": t["sent"],
                      "result_check": result_check(q, t["rows"], BG.ssb_rows(gs, q) if gs else None, "no golden rows for SF%g" % args.sf),
                      "roofline_frac": nbytes / (t["ms"] / 1e3) / 1e9 / (peak * world)}
        ssbres = {"value": 3 * rows_in / (tot_ms / 1e3), "unit": "rows/s", "sf": args.sf, "ms_per_step": tot_ms, "steps": args.steps,
                  "rows_scanned": 3 * rows_in, "scaling": "strong" if world > 1 else "n/a", "queries": per,
                  "result_check": "ok" if all(v["result_check"] == "ok" for v in per.values()) else
                  next(v["result_check"] for v in per.values() if v["result_check"] != "ok"),
                  "motion": motion_desc(),
                  "roofline": {"bound": "hbm", "achieved": 3 * nbytes / (tot_ms / 1e3) / 1e9, "peak": peak * world, "unit": "GB/s",
                               "frac": 3 * nbytes / (tot_ms / 1e3) / 1e9 / (peak * world), "algorithmic_bytes": 3 * nbytes,
                               "note": "Q4.1 + Q4.2 + Q4.3 back to back, each a whole query (dimension builds, star-join pipeline, aggregation, Motions) "
                                       "against the projected base columns (SURVEY.md 8d: 19.3 GB per query)"}}
        exs.close()
        for d in dev:
            d.free()

    # ---- CPU baseline (rank 0, N = 1): the oracle, scalar, on a bounded sample ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        rate, rows, secs = cpu_q1_sample(1, 24_000_000)
        cpu = {"value": rate, "unit": "rows/s", "cores": 1, "kind": "port",
               "sample": "Q1 over the first %d rows of the same synthetic lineitem, %.1f s, one thread (row-at-a-time oracle)" % (rows, secs)}
        # the same through the reference's own per-row code, one core, where oracle/_ref travelled to this box
        try:
            ref_rows = 8_000_000
            st = ref_q1_steps(1, ref_rows, 2)
        except Exception as e:
            sys.stderr.write("ref_q1 baseline skipped: %r\n" % (e,))
            st = None
        if st:
            cpu = {"value": ref_rows / st[1], "unit": "rows/s", "cores": 1, "kind": "reference", "rows_timed": ref_rows,
                   "sample": "Q1 over the first %d rows of the same synthetic lineitem, %.1f s, one process; %s" % (ref_rows, st[1], REF_Q1_NOTE),
                   "port": {"value": rate, "unit": "rows/s", "cores": 1,
                            "sample": "the oracle's int64 restatement (oracle/oracle.c) over the first %d rows, %.1f s, one thread" % (rows, secs)}}

    bad = [c for c in checks if c != "ok"]
    if rank == 0:
        line = {
            "metric": "TPC-H SF100 Q1 rows/sec", "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": {"workload": workload_name(args.sf, world),
                       "rows_per_gpu": nrows, "groups": ngroups, "l2": "inputs (%.1f GB per GPU) larger than L2" % (nrows * Q1_BYTES_PER_ROW / 1e9),
                       "timing": "CUDA events on the executor's stream, max over ranks"},
            "result_check": q1_check, "result_check_source": BG.SOURCE,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic_of(kname), "kernel": kname, "kernel_ms": kms, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": nrows * Q1_BYTES_PER_ROW},
            "clocks": clocks, "gpu_launches": l1 - l0,
        }
        if motion:
            line["motion"] = {"transport": motion_desc(), "host_syncs_per_step": (hs1[0] - hs0[0]) / args.steps,
                              "collectives_per_step": (hs1[1] - hs0[1]) / args.steps}
        if e2e:
            line["e2e"] = e2e
        if cpu:
            line["cpu_baseline"] = cpu
        if joins and world == 1 and not args.no_cpu:
            # the join queries on one host core: the oracle (restated reference path) over an SF1 database of the same generator
            try:
                for q, b in cpu_join_samples().items():
                    joins[q]["cpu_baseline"] = b
            except Exception as e:
                sys.stderr.write("join cpu baselines skipped: %r\n" % (e,))
        line.update(joins)
        if ssbres:
            line["ssb"] = ssbres
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        if bad:
            sys.stderr.write("result_check FAILED: %s\n" % bad[0])
    if ex:
        ex.close()
    if li:
        li.free()
    if motion:
        motion.close()
    ctx.close()
    if dist:
        dist.destroy_process_group()
    if bad:
        sys.exit(1)


if __name__ == "__main__":
    main()
