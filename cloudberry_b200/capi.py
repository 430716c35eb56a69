"""ctypes binding of the C ABI (include/cbgpu.h, include/cb_exec.h): libcbgpu.so + libcbexec.so.

Host-side glue for tests, smoke() and bench.py.  All compute is behind the C ABI; this module never
falls back to numpy / torch / the oracle: if the CUDA library is missing or no GPU is present, the
calls fail loudly.
"""
import ctypes as C
import os
import re

import numpy as np

from . import plan as P
from .relation import HostRelation, NP_DTYPE

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_GPU = None
_EXEC = None


class CbgpuError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("cbgpu error %d: %s" % (code, msg))
        self.code = code


class CbgpuVisimapEntry(C.Structure):
    _fields_ = [("first_row_num", C.c_int64), ("data", C.c_void_p), ("len", C.c_int32)]


class CbAggStateDatum(C.Structure):
    _fields_ = [("n", C.c_int64), ("lo", C.c_int64), ("hi", C.c_int64)]


TUPSER_STATE_NUMERIC, TUPSER_STATE_INT8 = 101, 102


class CbTupAttr(C.Structure):
    _fields_ = [("type", C.c_int32), ("dscale", C.c_int32), ("bpchar_len", C.c_int32), ("ntexts", C.c_int32),
                ("texts", C.POINTER(C.c_char_p)), ("text_lens", C.POINTER(C.c_int32)), ("state", C.POINTER(CbAggStateDatum))]


def _tup_attrs(attrs):
    """[(CbTypeId, dscale, bpchar_len[, texts])] -> (CbTupAttr array, keep-alive list); texts: the column's dictionary in
    byte order (DeviceDict.entries())"""
    arr = (CbTupAttr * max(len(attrs), 1))()
    keep = []
    for i, a in enumerate(attrs):
        arr[i].type, arr[i].dscale, arr[i].bpchar_len = a[0], a[1], a[2]
        if a[0] in (TUPSER_STATE_NUMERIC, TUPSER_STATE_INT8):
            st = CbAggStateDatum()
            keep.append(st)
            arr[i].state = C.pointer(st)
        texts = a[3] if len(a) > 3 and a[3] is not None else []
        if texts:
            bufs = [C.create_string_buffer(bytes(t), len(t)) for t in texts]
            ptrs = (C.c_char_p * len(texts))(*[C.cast(b, C.c_char_p) for b in bufs])
            lens = (C.c_int32 * len(texts))(*[len(t) for t in texts])
            keep += [bufs, ptrs, lens]
            arr[i].ntexts = len(texts)
            arr[i].texts = ptrs
            arr[i].text_lens = lens
    return arr, keep


def tupser_rows(attrs, rows, nulls=None, max_chunk=8160, end=True):
    """rows (lists of ints as the executor holds them) -> the reference's tuple chunk stream (cb_tupser_row);
    attrs: [(CbTypeId, dscale, bpchar_len, DeviceDict or None)]"""
    L = ex()
    n = len(attrs)
    arr, keep = _tup_attrs(attrs)
    out = bytearray()
    buf = C.create_string_buffer(1 << 20)
    for r, row in enumerate(rows):
        cells, held = [], []
        for i, v in enumerate(row):
            if attrs[i][0] in (TUPSER_STATE_NUMERIC, TUPSER_STATE_INT8) and v is not None:
                st = CbAggStateDatum(*[int(x) for x in v])      # (N, lo, hi)
                held.append(st)
                cells.append(C.addressof(st))
            else:
                cells.append(0 if v is None else int(v))
        vals = (C.c_int64 * max(n, 1))(*cells)
        isn = (C.c_uint8 * max(n, 1))(*([int(x) for x in nulls[r]] if nulls is not None else [0] * n))
        k = L.cb_tupser_row(arr, n, vals, isn, max_chunk, buf, len(buf))
        if k < 0:
            raise CbgpuError(int(k), "cb_tupser_row failed")
        out += buf.raw[:k]
    if end:
        k = L.cb_tupser_end_of_stream(buf, len(buf))
        out += buf.raw[:k]
    return bytes(out)


def tupser_parse(attrs, data):
    """a tuple chunk stream -> (rows, nulls, bytes consumed, ended) through cb_tupser_next"""
    L = ex()
    n = len(attrs)
    arr, keep = _tup_attrs(attrs)
    buf = C.create_string_buffer(bytes(data), len(data))
    pos = 0
    rows, nulls = [], []
    vals = (C.c_int64 * max(n, 1))()
    isn = (C.c_uint8 * max(n, 1))()
    used = C.c_int64()
    while True:
        rc = L.cb_tupser_next(arr, n, C.byref(buf, pos), len(data) - pos, C.byref(used), vals, isn)
        if rc == 1:
            row = []
            for i in range(n):
                if attrs[i][0] in (TUPSER_STATE_NUMERIC, TUPSER_STATE_INT8) and not isn[i]:
                    st = arr[i].state.contents
                    row.append((int(st.n), int(st.lo), int(st.hi)))
                else:
                    row.append(int(vals[i]))
            rows.append(row)
            nulls.append([int(isn[i]) for i in range(n)])
            pos += used.value
            continue
        if rc == 0:
            return rows, nulls, pos + used.value, True
        if rc == -1:
            return rows, nulls, pos, False
        raise CbgpuError(int(rc), "cb_tupser_next: malformed chunk stream at byte %d" % pos)


class CbAocsColumnSpec(C.Structure):
    _fields_ = [("relcol", C.c_int32), ("filenum", C.c_int32), ("attlen", C.c_int32), ("varkind", C.c_int32), ("typalign", C.c_int32),
                ("compresstype", C.c_int32), ("eof", C.c_int64), ("dict", C.c_void_p)]


def aocs_column_spec(c):
    """(relcol, filenum, attlen, varkind, typalign, compresstype, eof[, DeviceDict]) -> CbAocsColumnSpec"""
    return CbAocsColumnSpec(*c[:7], c[7].h if len(c) > 7 and c[7] is not None else None)


def aocs_dict_collect_segfile(ctx, basepath, segno, checksum, col):
    """first pass over a string column's segment file (cb_aocs_dict_collect_segfile)"""
    spec = aocs_column_spec(col)
    err = C.create_string_buffer(512)
    rc = ex().cb_aocs_dict_collect_segfile(ctx.h, os.fsencode(basepath), segno, 1 if checksum else 0, C.byref(spec), err, 512)
    if rc != 0:
        raise CbgpuError(rc, err.value.decode() or ctx.error())


def aocs_segfile_path(basepath, segno, filenum):
    """FormatAOSegmentFileName (access/appendonly/aomd.c:84-117) through cb_aocs_segfile_path; None = out of range"""
    buf = C.create_string_buffer(4096)
    if ex().cb_aocs_segfile_path(os.fsencode(basepath), segno, filenum, buf, 4096) != 0:
        return None
    return os.fsdecode(buf.value)


class DeviceDict:
    """dictionary of a bpchar(n) / varchar / text column, built on the device from the column's files (cbgpu_dict)"""

    def __init__(self, ctx, max_entries=4096, arena_bytes=1 << 20, bpchar=True):
        self.ctx = ctx
        h = C.c_void_p()
        ctx.check(ctx.L.cbgpu_dict_create(ctx.h, max_entries, arena_bytes, 1 if bpchar else 0, C.byref(h)))
        self.h = h

    def collect(self, file_bytes, checksum, compresstype=0, typalign=4):
        buf = np.frombuffer(file_bytes, dtype=np.uint8)
        self.ctx.check(self.ctx.L.cbgpu_aocs_dict_collect(self.ctx.h, buf.ctypes.data, len(buf), 1 if checksum else 0, compresstype, typalign,
                                                          self.h))

    def finalize(self):
        n = C.c_int32()
        self.ctx.check(self.ctx.L.cbgpu_dict_finalize(self.h, C.byref(n)))
        return int(n.value)

    def entries(self):
        out = []
        n = self.finalize()
        p = C.c_void_p()
        ln = C.c_int32()
        f = self.ctx.L.cbgpu_dict_entry
        f.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_int32)]
        for i in range(n):
            self.ctx.check(f(self.h, i, C.byref(p), C.byref(ln)))
            out.append(C.string_at(p.value, ln.value))
        return out

    def lookup(self, text):
        b = text if isinstance(text, bytes) else text.encode()
        return int(self.ctx.L.cbgpu_dict_lookup(self.h, b, len(b)))

    def free(self):
        if self.h:
            self.ctx.L.cbgpu_dict_free(self.h)
            self.h = None


class CbNumericDatum(C.Structure):
    _fields_ = [("lo", C.c_int64), ("hi", C.c_int64), ("dscale", C.c_int32), ("text", C.c_char * 84)]


class CbTupleTableSlot(C.Structure):
    _fields_ = [("tts_empty", C.c_bool), ("tts_nvalid", C.c_int32), ("tts_types", C.POINTER(C.c_int32)),
                ("tts_values", C.POINTER(C.c_int64)), ("tts_isnull", C.POINTER(C.c_bool)),
                ("tts_state_n", C.POINTER(C.c_int64)), ("tts_state_lo", C.POINTER(C.c_int64)),
                ("tts_state_hi", C.POINTER(C.c_int64))]


class CbInstrumentation(C.Structure):
    _fields_ = [("ntuples", C.c_double), ("nloops", C.c_double), ("kernels", C.c_int64), ("device_ms", C.c_double),
                ("rows_in", C.c_int64), ("motion_repartitions", C.c_int64), ("hashjoin_nbatch", C.c_int64), ("agg_npartitions", C.c_int64)]


class CbPlanState(C.Structure):
    pass


CbPlanState._fields_ = [
    ("type", C.c_int), ("plan", C.POINTER(P.CbPlan)), ("state", C.c_void_p), ("ExecProcNode", C.c_void_p),
    ("instrument", CbInstrumentation), ("lefttree", C.POINTER(CbPlanState)), ("righttree", C.POINTER(CbPlanState)),
    ("ps_ResultTupleSlot", C.POINTER(CbTupleTableSlot)), ("squelched", C.c_bool), ("priv", C.c_void_p),
]


class CbEState(C.Structure):
    _fields_ = [("es_ctx", C.c_void_p), ("es_nrels", C.c_int32), ("es_range_table", C.POINTER(C.c_void_p)),
                ("es_segindex", C.c_int32), ("es_numsegments", C.c_int32), ("es_interconnect", C.c_void_p),
                ("es_errcode", C.c_int32), ("es_errmsg", C.c_char * 512), ("es_error_hook", C.c_void_p),
                ("es_force_generic", C.c_int32), ("es_processed", C.c_int64), ("es_cluster", C.c_void_p),
                ("es_interrupt_pending", C.c_void_p), ("es_interrupt_arg", C.c_void_p), ("es_operator_mem_kb", C.c_int64),
                ("es_hashjoin_batches_run", C.c_int64), ("es_agg_partitions_run", C.c_int64)]


def header_symbols(header):
    """Function names declared in a C header (used by the not-gpu export test)."""
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    names = set()
    for m in re.finditer(r"\b((?:cbgpu|cb)_[A-Za-z0-9_]+)\s*\(", text):
        name = m.group(1)
        if name.startswith(("cb_type_width",)):
            continue
        names.add(name)
    return sorted(names)


def build():
    import subprocess
    subprocess.check_call(["make", "-s", "-C", os.path.join(HERE, "csrc"), "-j8", "all"])


def _preload_bundled_nccl():
    """libcbgpu.so needs libnccl.so.2.  When the harness also imports torch (rendezvous, barrier), both must
    share ONE NCCL: load the copy bundled with torch's wheels first, so the dynamic loader resolves the
    SONAME to it whichever of the two libraries is imported first.  No such wheel: the system library is used."""
    try:
        import importlib.util
        spec = importlib.util.find_spec("nvidia.nccl")
        for d in (spec.submodule_search_locations if spec else []):
            cand = os.path.join(d, "lib", "libnccl.so.2")
            if os.path.exists(cand):
                C.CDLL(cand, mode=C.RTLD_GLOBAL)
                return
    except Exception:
        pass


def gpu():
    global _GPU
    if _GPU is None:
        so = os.path.join(os.environ.get("CBGPU_LIBDIR") or HERE, "libcbgpu.so")     # CBGPU_LIBDIR: an experimental build (tools/)
        if not os.path.exists(so):
            raise CbgpuError(-1, "libcbgpu.so is not built (run __graft_entry__.build()); there is no CPU fallback")
        _preload_bundled_nccl()
        L = C.CDLL(so, mode=C.RTLD_GLOBAL)
        vp, i32, i64, u64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_double
        sig = {
            "cbgpu_ctx_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
            "cbgpu_ctx_destroy": (None, [vp]),
            "cbgpu_last_error": (C.c_char_p, [vp]),
            "cbgpu_sync": (C.c_int, [vp]),
            "cbgpu_check_status": (C.c_int, [vp]),
            "cbgpu_device_count": (C.c_int, []),
            "cbgpu_sm_count": (C.c_int, [vp]),
            "cbgpu_kernel_launches": (i64, [vp]),
            "cbgpu_timer_start": (C.c_int, [vp]),
            "cbgpu_timer_stop_ms": (C.c_int, [vp, C.POINTER(dbl)]),
            "cbgpu_last_kernel_ms": (dbl, [vp]),
            "cbgpu_last_kernel_name": (C.c_char_p, [vp]),
            "cbgpu_kernel_log_reset": (None, [vp]),
            "cbgpu_kernel_log_longest": (C.c_int, [vp, C.c_char_p, C.c_int, C.POINTER(dbl)]),
            "cbgpu_trace_begin": (C.c_int, [vp]),
            "cbgpu_trace_end": (C.c_int, [vp]),
            "cbgpu_trace_get": (C.c_int, [vp, C.c_int, C.c_char_p, C.c_int, C.POINTER(dbl)]),
            "cbgpu_flush_l2": (C.c_int, [vp]),
            "cbgpu_host_alloc": (vp, [C.c_size_t]),
            "cbgpu_host_free": (None, [vp]),
            "cbgpu_hashbpchar": (C.c_uint32, [C.c_char_p, i32]),
            "cbgpu_rel_create": (C.c_int, [vp, i64, i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(vp)]),
            "cbgpu_rel_free": (None, [vp]),
            "cbgpu_rel_nrows": (i64, [vp]),
            "cbgpu_rel_ncols": (i32, [vp]),
            "cbgpu_rel_col_type": (i32, [vp, i32]),
            "cbgpu_rel_col_dscale": (i32, [vp, i32]),
            "cbgpu_rel_load_column": (C.c_int, [vp, i32, vp, vp]),
            "cbgpu_rel_load_column_narrow": (C.c_int, [vp, i32, vp, i32]),
            "cbgpu_rel_read_column": (C.c_int, [vp, i32, i64, i64, vp, vp]),
            "cbgpu_rel_set_visimap": (C.c_int, [vp, vp]),
            "cbgpu_rel_read_visimap": (C.c_int, [vp, vp]),
            "cbgpu_dict_create": (C.c_int, [vp, i32, i64, i32, C.POINTER(vp)]),
            "cbgpu_dict_free": (None, [vp]),
            "cbgpu_aocs_dict_collect": (C.c_int, [vp, vp, i64, i32, i32, i32, vp]),
            "cbgpu_dict_finalize": (C.c_int, [vp, C.POINTER(i32)]),
            "cbgpu_dict_entry": (C.c_int, [vp, i32, C.POINTER(C.c_char_p), C.POINTER(i32)]),
            "cbgpu_dict_lookup": (i32, [vp, C.c_char_p, i32]),
            "cbgpu_aocs_decode_dict_column": (C.c_int, [vp, vp, i64, i32, i32, i32, vp, vp, i32, i64, C.POINTER(i64)]),
            "cbgpu_aocs_apply_visimap": (C.c_int, [vp, vp, i64, i32, vp, i32, vp, i64, C.POINTER(i64)]),
            "cbgpu_rel_set_dict_hash": (C.c_int, [vp, i32, vp, i32]),
            "cbgpu_rel_set_nrows": (C.c_int, [vp, i64]),
            "cbgpu_rel_copy_rows": (C.c_int, [vp, i64, vp, i64, i64]),
            "cbgpu_rel_col_devptr": (vp, [vp, i32]),
            "cbgpu_rel_nbytes": (C.c_size_t, [vp]),
            "cbgpu_ht_build": (C.c_int, [vp, vp, C.POINTER(i32), i32, C.POINTER(vp)]),
            "cbgpu_ht_build_batched": (C.c_int, [vp, vp, C.POINTER(i32), i32, i32, C.POINTER(vp)]),
            "cbgpu_ht_nbatch": (C.c_int, [vp]),
            "cbgpu_ht_bytes_for": (i64, [i64]),
            "cbgpu_ht_free": (None, [vp]),
            "cbgpu_ht_nrows": (i64, [vp]),
            "cbgpu_ht_has_duplicates": (C.c_int, [vp]),
            "cbgpu_ht_probe_pairs": (C.c_int, [vp, vp, vp, C.POINTER(i32), i32, vp, i64, vp]),
            # pending: a PENDING_FN or None
            "cbgpu_ht_probe_pairs_batched": (C.c_int, [vp, vp, vp, C.POINTER(i32), i32, i32, i32, vp, vp, C.POINTER(i64), vp]),
            "cbgpu_pairs_free": (None, [vp]),
            "cbgpu_merge_sorted_runs": (C.c_int, [vp, vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), i32, i32, C.POINTER(vp),
                                                  C.POINTER(i32)]),
            "cbgpu_dev_free": (None, [vp, vp]),
            "cbgpu_read_u32": (C.c_int, [vp, vp, i64, vp]),
            "cbgpu_motion_unique_id": (C.c_int, [vp]),
            "cbgpu_motion_create": (C.c_int, [vp, C.c_int, C.c_int, vp, C.POINTER(vp)]),
            "cbgpu_motion_create_boot": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, C.POINTER(vp)]),
            "cbgpu_motion_destroy": (None, [vp]),
            "cbgpu_motion_abort": (None, [vp]),
            "cbgpu_motion_host_syncs": (i64, [vp]),
            "cbgpu_motion_collectives": (i64, [vp]),
            "cbgpu_motion_bytes_sent": (i64, [vp]),
            "cbgpu_motion_direct_bytes": (i64, [vp]),
            "cbgpu_motion_direct_available": (C.c_int, [vp]),
            "cbgpu_gen_lineitem": (C.c_int, [vp, vp, u64, i64, i64, i64]),
            "cbgpu_gen_orders": (C.c_int, [vp, vp, u64, i64, i64]),
            "cbgpu_gen_customer": (C.c_int, [vp, vp, u64]),
            "cbgpu_gen_supplier": (C.c_int, [vp, vp, u64]),
            "cbgpu_aocs_decode_column": (C.c_int, [vp, vp, i64, i32, i32, i32, i32, vp, i32, i64, C.POINTER(i64)]),
            "cbgpu_aocs_decode_column_ex": (C.c_int, [vp, vp, i64, i32, i32, i32, i32, i32, vp, i32, i64, C.POINTER(i64)]),
            "cbgpu_gen_customer_range": (C.c_int, [vp, vp, u64, i64]),
            "cbgpu_gen_supplier_range": (C.c_int, [vp, vp, u64, i64]),
            "cbgpu_gen_ssb_lineorder": (C.c_int, [vp, vp, u64, i64, i64, i64, i64]),
        }
        for name, (res, args) in sig.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _GPU = L
    return _GPU


def ex():
    global _EXEC
    if _EXEC is None:
        gpu()
        so = os.path.join(os.environ.get("CBGPU_LIBDIR") or HERE, "libcbexec.so")
        if not os.path.exists(so):
            raise CbgpuError(-1, "libcbexec.so is not built (run __graft_entry__.build())")
        L = C.CDLL(so)
        vp = C.c_void_p
        L.cb_CreateExecutorState.restype = C.POINTER(CbEState)
        L.cb_CreateExecutorState.argtypes = [vp, C.POINTER(vp), C.c_int32]
        L.cb_FreeExecutorState.argtypes = [C.POINTER(CbEState)]
        L.cb_estate_error.restype = C.c_char_p
        L.cb_estate_error.argtypes = [C.POINTER(CbEState)]
        L.cb_ExecInitNode.restype = C.POINTER(CbPlanState)
        L.cb_ExecInitNode.argtypes = [C.POINTER(P.CbPlan), C.POINTER(CbEState), C.c_int]
        L.cb_ExecProcNode.restype = C.POINTER(CbTupleTableSlot)
        L.cb_ExecProcNode.argtypes = [C.POINTER(CbPlanState)]
        L.cb_MultiExecProcNode.restype = vp
        L.cb_MultiExecProcNode.argtypes = [C.POINTER(CbPlanState)]
        L.cb_ExecProcNodeBatch.restype = C.c_int
        L.cb_ExecProcNodeBatch.argtypes = [C.POINTER(CbPlanState), C.POINTER(vp)]
        for n in ("cb_ExecEndNode", "cb_ExecReScan", "cb_ExecSquelchNode"):
            getattr(L, n).restype = None
            getattr(L, n).argtypes = [C.POINTER(CbPlanState)]
        L.cb_slot_text.restype = C.c_int
        L.cb_slot_text.argtypes = [C.POINTER(CbTupleTableSlot), C.c_int, C.c_char_p, C.c_int]
        L.cb_slot_float8.restype = C.c_double
        L.cb_slot_float8.argtypes = [C.POINTER(CbTupleTableSlot), C.c_int]
        L.cb_numeric_sum_text.argtypes = [C.c_int64, C.c_int64, C.c_int32, C.c_char_p, C.c_int32]
        L.cb_numeric_avg_text.argtypes = [C.c_int64, C.c_int64, C.c_int32, C.c_int64, C.c_char_p, C.c_int32]
        L.cb_interconnect_nccl_create.restype = vp
        L.cb_interconnect_nccl_create.argtypes = [vp]
        L.cb_interconnect_destroy.argtypes = [vp]
        L.cb_aocs_segfile_path.restype = C.c_int
        L.cb_aocs_segfile_path.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_char_p, C.c_size_t]
        L.cb_aocs_dict_collect_segfile.restype = C.c_int
        L.cb_aocs_dict_collect_segfile.argtypes = [vp, C.c_char_p, C.c_int, C.c_int, C.POINTER(CbAocsColumnSpec), C.c_char_p, C.c_size_t]
        L.cb_aocs_load_segfile.restype = C.c_int
        L.cb_aocs_load_segfile.argtypes = [vp, C.c_char_p, C.c_int, C.c_int, C.c_int, C.POINTER(CbAocsColumnSpec), vp, C.c_int64,
                                           C.POINTER(CbgpuVisimapEntry), C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                           C.c_char_p, C.c_size_t]
        L.cb_tupser_row.restype = C.c_int64
        L.cb_tupser_row.argtypes = [C.POINTER(CbTupAttr), C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_uint8), C.c_int, vp, C.c_int64]
        L.cb_tupser_end_of_stream.restype = C.c_int
        L.cb_tupser_end_of_stream.argtypes = [vp, C.c_int64]
        L.cb_tupser_next.restype = C.c_int64
        L.cb_tupser_next.argtypes = [C.POINTER(CbTupAttr), C.c_int, vp, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                     C.POINTER(C.c_uint8)]
        L.cb_cluster_create.restype = vp
        L.cb_cluster_create.argtypes = [vp, C.c_int32]
        L.cb_cluster_set_range_table.restype = C.c_int
        L.cb_cluster_set_range_table.argtypes = [vp, C.c_int32, C.POINTER(vp), C.c_int32]
        L.cb_cluster_estate.restype = C.POINTER(CbEState)
        L.cb_cluster_estate.argtypes = [vp, C.c_int32]
        L.cb_cluster_init_plan.restype = C.c_int
        L.cb_cluster_init_plan.argtypes = [vp, C.POINTER(P.CbPlan)]
        L.cb_cluster_next.restype = C.POINTER(CbTupleTableSlot)
        L.cb_cluster_next.argtypes = [vp]
        L.cb_cluster_current_segment.restype = C.c_int32
        L.cb_cluster_current_segment.argtypes = [vp]
        L.cb_cluster_end.argtypes = [vp]
        L.cb_cluster_destroy.argtypes = [vp]
        L.cb_cluster_error.restype = C.c_char_p
        L.cb_cluster_error.argtypes = [vp]
        _EXEC = L
    return _EXEC


def hashbpchar(text):
    b = text.encode() if isinstance(text, str) else text
    return int(gpu().cbgpu_hashbpchar(b, len(b)))


class Context:
    def __init__(self, device=0):
        self.L = gpu()
        h = C.c_void_p()
        rc = self.L.cbgpu_ctx_create(device, C.byref(h))
        self.h = h
        if rc:
            raise CbgpuError(rc, self.error())

    def error(self):
        return (self.L.cbgpu_last_error(self.h) or b"").decode()

    def check(self, rc):
        if rc:
            raise CbgpuError(rc, self.error())

    def sync(self):
        self.check(self.L.cbgpu_sync(self.h))

    def launches(self):
        return int(self.L.cbgpu_kernel_launches(self.h))

    def timer_start(self):
        self.check(self.L.cbgpu_timer_start(self.h))

    def timer_stop_ms(self):
        ms = C.c_double()
        self.check(self.L.cbgpu_timer_stop_ms(self.h, C.byref(ms)))
        return ms.value

    def last_kernel(self):
        return (self.L.cbgpu_last_kernel_name(self.h) or b"").decode(), float(self.L.cbgpu_last_kernel_ms(self.h))

    def kernel_log_reset(self):
        self.L.cbgpu_kernel_log_reset(self.h)

    def longest_kernel(self):
        """(name, ms) of the longest pipeline kernel since kernel_log_reset(); syncs the stream."""
        buf = C.create_string_buffer(128)
        ms = C.c_double()
        self.check(self.L.cbgpu_kernel_log_longest(self.h, buf, 128, C.byref(ms)))
        return buf.value.decode(), ms.value

    def trace_begin(self):
        self.check(self.L.cbgpu_trace_begin(self.h))

    def trace_end(self):
        """[(kernel name, ms)] for every launch since trace_begin(); ms runs from the previous launch's end."""
        n = self.L.cbgpu_trace_end(self.h)
        out = []
        buf = C.create_string_buffer(128)
        ms = C.c_double()
        for i in range(n):
            self.check(self.L.cbgpu_trace_get(self.h, i, buf, 128, C.byref(ms)))
            out.append((buf.value.decode(), ms.value))
        return out

    def flush_l2(self):
        self.check(self.L.cbgpu_flush_l2(self.h))

    def sm_count(self):
        return int(self.L.cbgpu_sm_count(self.h))

    def close(self):
        if self.h:
            self.L.cbgpu_ctx_destroy(self.h)
            self.h = None


ALLGATHER_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t)
PENDING_FN = C.CFUNCTYPE(C.c_int, C.c_void_p)


class CbgpuPairs(C.Structure):
    """cbgpu_pairs: npairs (outer_idx, inner_idx) row-id pairs in two device arrays; 0xFFFFFFFF = the side is missing"""
    _fields_ = [("npairs", C.c_int64), ("outer_idx", C.c_void_p), ("inner_idx", C.c_void_p)]


class Motion:
    """Interconnect endpoint of one GPU-segment (one process per GPU): peer-memory windows with device-side
    signalling, plus NCCL for what the windows cannot take.

    unique_id: the NCCL rendezvous token (rank 0 makes it, everyone gets it).  unique_id=None with
    allgather=f: windows only, bootstrapped through f(my_bytes) -> [bytes of rank 0, 1, ...] (e.g. over a
    torch.distributed gloo group): no NCCL communicator, so two ranks may share one GPU."""

    @staticmethod
    def unique_id():
        buf = C.create_string_buffer(128)
        rc = gpu().cbgpu_motion_unique_id(buf)
        if rc:
            raise CbgpuError(rc, "ncclGetUniqueId failed")
        return buf.raw

    def __init__(self, ctx, rank, nranks, unique_id=None, allgather=None):
        self.ctx = ctx
        self.rank = rank
        self.nranks = nranks
        h = C.c_void_p()
        if unique_id is not None:
            buf = C.create_string_buffer(unique_id, 128)
            ctx.check(ctx.L.cbgpu_motion_create(ctx.h, rank, nranks, buf, C.byref(h)))
        else:
            def _cb(_arg, mine, allp, nbytes):
                try:
                    parts = allgather(C.string_at(mine, nbytes))
                    if len(parts) != nranks or any(len(x) != nbytes for x in parts):
                        return 1
                    C.memmove(allp, b"".join(parts), nbytes * nranks)
                    return 0
                except Exception:       # noqa: BLE001 - reported to the C side as a failed all-gather
                    return 1
            self._cb = ALLGATHER_FN(_cb)        # must outlive the interconnect (tear-down calls it too)
            ctx.check(ctx.L.cbgpu_motion_create_boot(ctx.h, rank, nranks, C.cast(self._cb, C.c_void_p), None, C.byref(h)))
        self.h = h

    def bytes_sent(self):
        """payload bytes this rank moved to other segments: through NCCL (staged path) + stored into peers'
        windows (direct path)"""
        return int(self.ctx.L.cbgpu_motion_bytes_sent(self.h)) + int(self.ctx.L.cbgpu_motion_direct_bytes(self.h))

    def direct(self):
        """True when Redistribute runs fused over peer memory (CUDA IPC windows), False: staged over NCCL"""
        return bool(self.ctx.L.cbgpu_motion_direct_available(self.h))

    def host_syncs(self):
        return int(self.ctx.L.cbgpu_motion_host_syncs(self.h))

    def collectives(self):
        return int(self.ctx.L.cbgpu_motion_collectives(self.h))

    def close(self):
        if self.h:
            self.ctx.L.cbgpu_motion_destroy(self.h)
            self.h = None

    def abort(self):
        """tear down without any collective step (after a failed query)"""
        if self.h:
            self.ctx.L.cbgpu_motion_abort(self.h)
            self.h = None


class DeviceRelation:
    """An HBM-resident relation (the decoded, projected form of an AOCS table)."""

    def __init__(self, ctx, nrows, types, dscales=None, name="rel"):
        self.ctx = ctx
        self.name = name
        self.types = list(types)
        self.dscales = list(dscales) if dscales is not None else [2 if t == P.NUMERIC else 0 for t in types]
        n = len(types)
        h = C.c_void_p()
        ctx.check(ctx.L.cbgpu_rel_create(ctx.h, nrows, n, (C.c_int32 * n)(*self.types), (C.c_int32 * n)(*self.dscales),
                                         C.byref(h)))
        self.h = h
        self.nrows = nrows

    @classmethod
    def adopt(cls, ctx, handle, name="batch"):
        """Wrap a cbgpu_rel the library handed over (cb_ExecProcNodeBatch); this object now owns it."""
        L = ctx.L
        d = cls.__new__(cls)
        d.ctx = ctx
        d.name = name
        d.h = C.c_void_p(handle) if not isinstance(handle, C.c_void_p) else handle
        n = int(L.cbgpu_rel_ncols(d.h))
        d.types = [int(L.cbgpu_rel_col_type(d.h, i)) for i in range(n)]
        d.dscales = [int(L.cbgpu_rel_col_dscale(d.h, i)) for i in range(n)]
        d.nrows = int(L.cbgpu_rel_nrows(d.h))
        return d

    @classmethod
    def from_host(cls, ctx, rel: HostRelation):
        d = cls(ctx, rel.nrows, rel.types, rel.dscales, rel.name)
        d.load(rel)
        return d

    def load(self, rel: HostRelation, sync=True):
        """Host -> device copy of every column (cbgpu_rel_load_column)."""
        L = self.ctx.L
        for i, col in enumerate(rel.columns):
            nl = rel.nulls[i]
            if nl is not None:
                nl = np.ascontiguousarray(nl, dtype=np.uint8)
            self.ctx.check(L.cbgpu_rel_load_column(self.h, i, col.ctypes.data, nl.ctypes.data if nl is not None else None))
            if rel.dict_hashes[i] is not None:
                dh = np.ascontiguousarray(rel.dict_hashes[i], dtype=np.uint32)
                self.ctx.check(L.cbgpu_rel_set_dict_hash(self.h, i, dh.ctypes.data, len(dh)))
        if rel.visimap is not None:
            vm = np.ascontiguousarray(rel.visimap, dtype=np.uint8)
            self.ctx.check(L.cbgpu_rel_set_visimap(self.h, vm.ctypes.data))
        if sync:
            self.ctx.sync()

    def load_aocs_column(self, col, file_bytes, checksum, attlen, varkind=0, typalign=4, row_offset=0, compresstype=0):
        """Decode one column's AOCS segment-file bytes on the device into this relation (cbgpu_aocs_decode_column_ex);
        compresstype 1 = zlib bulk compression.  Returns the number of rows the file held."""
        buf = np.frombuffer(file_bytes, dtype=np.uint8)
        n = C.c_int64()
        self.ctx.check(self.ctx.L.cbgpu_aocs_decode_column_ex(self.ctx.h, buf.ctypes.data, len(buf), 1 if checksum else 0, compresstype,
                                                              attlen, varkind, typalign, self.h, col, row_offset, C.byref(n)))
        return int(n.value)

    def load_aocs_dict_column(self, col, file_bytes, checksum, dictionary, compresstype=0, typalign=4, row_offset=0):
        """rows of a string column as codes of `dictionary` (cbgpu_aocs_decode_dict_column)"""
        buf = np.frombuffer(file_bytes, dtype=np.uint8)
        n = C.c_int64()
        self.ctx.check(self.ctx.L.cbgpu_aocs_decode_dict_column(self.ctx.h, buf.ctypes.data, len(buf), 1 if checksum else 0, compresstype,
                                                                typalign, dictionary.h, self.h, col, row_offset, C.byref(n)))
        return int(n.value)

    def apply_visimap(self, file_bytes, checksum, entries, row_offset=0):
        """entries: [(first_row_no, payload bytes or None)] of the segment file's pg_aovisimap rows; file_bytes: any
        column file of it (cbgpu_aocs_apply_visimap).  Returns the number of rows hidden."""
        buf = np.frombuffer(file_bytes, dtype=np.uint8)
        arr = (CbgpuVisimapEntry * max(len(entries), 1))()
        keep = []
        for i, (first, payload) in enumerate(entries):
            arr[i].first_row_num = first
            if payload is None:
                arr[i].data = None
                arr[i].len = 0
            else:
                b = C.create_string_buffer(bytes(payload), len(payload))
                keep.append(b)
                arr[i].data = C.cast(b, C.c_void_p)
                arr[i].len = len(payload)
        n = C.c_int64()
        self.ctx.check(self.ctx.L.cbgpu_aocs_apply_visimap(self.ctx.h, buf.ctypes.data, len(buf), 1 if checksum else 0, arr, len(entries),
                                                           self.h, row_offset, C.byref(n)))
        return int(n.value)

    def load_segfile(self, basepath, segno, checksum, cols, entries=(), row_offset=0):
        """cols: [(relcol, filenum, attlen, varkind, typalign, compresstype, eof[, DeviceDict])]; entries: [(first_row_no,
        payload or None)].  Reads the segment file set from disk (cb_aocs_load_segfile); returns (rows, rows hidden)."""
        specs = (CbAocsColumnSpec * len(cols))(*[aocs_column_spec(c) for c in cols])
        arr = (CbgpuVisimapEntry * max(len(entries), 1))()
        keep = []
        for i, (first, payload) in enumerate(entries):
            arr[i].first_row_num = first
            if payload is not None:
                b = C.create_string_buffer(bytes(payload), len(payload))
                keep.append(b)
                arr[i].data = C.cast(b, C.c_void_p)
                arr[i].len = len(payload)
        n, h = C.c_int64(), C.c_int64()
        err = C.create_string_buffer(512)
        rc = ex().cb_aocs_load_segfile(self.ctx.h, os.fsencode(basepath), segno, 1 if checksum else 0, len(cols), specs, self.h, row_offset,
                                       arr, len(entries), C.byref(n), C.byref(h), err, 512)
        if rc != 0:
            raise CbgpuError(rc, err.value.decode() or self.ctx.error())
        return int(n.value), int(h.value)

    def read_visimap(self):
        """one bool per row (True = visible)"""
        out = np.zeros((self.rows() + 7) // 8, dtype=np.uint8)
        self.ctx.check(self.ctx.L.cbgpu_rel_read_visimap(self.h, out.ctypes.data))
        return np.unpackbits(out, bitorder="little")[:self.rows()].astype(bool)

    def load_column_ptr(self, col, host_ptr, host_width=None):
        """host_width: the host column's integer width when it is narrower than the column's own (sign-extended on the device)"""
        if host_width is None or host_width == P.TYPE_WIDTH[self.types[col]]:
            self.ctx.check(self.ctx.L.cbgpu_rel_load_column(self.h, col, host_ptr, None))
        else:
            self.ctx.check(self.ctx.L.cbgpu_rel_load_column_narrow(self.h, col, host_ptr, host_width))

    def set_dict_hash(self, col, hashes):
        dh = np.ascontiguousarray(hashes, dtype=np.uint32)
        self.ctx.check(self.ctx.L.cbgpu_rel_set_dict_hash(self.h, col, dh.ctypes.data, len(dh)))

    def read_column(self, col, lo=0, hi=None):
        hi = self.rows() if hi is None else hi
        out = np.empty(hi - lo, dtype=NP_DTYPE[self.types[col]])
        nulls = np.zeros(hi - lo, dtype=np.uint8)
        self.ctx.check(self.ctx.L.cbgpu_rel_read_column(self.h, col, lo, hi, out.ctypes.data, nulls.ctypes.data))
        return out, nulls

    def rows(self):
        return int(self.ctx.L.cbgpu_rel_nrows(self.h))

    def nbytes(self):
        return int(self.ctx.L.cbgpu_rel_nbytes(self.h))

    def free(self):
        if self.h:
            self.ctx.L.cbgpu_rel_free(self.h)
            self.h = None


def _slot_row(E, slot):
    s = slot.contents
    row, states = [], []
    buf = C.create_string_buffer(160)
    for i in range(s.tts_nvalid):
        states.append((s.tts_state_n[i], ((s.tts_state_hi[i] << 64) | (s.tts_state_lo[i] & (2 ** 64 - 1)))))
        if s.tts_isnull[i]:
            row.append(None)
            continue
        t = s.tts_types[i]
        if t == P.FLOAT8:
            row.append(E.cb_slot_float8(slot, i + 1))
        elif t in (P.NUMERIC, P.NUMERIC128):
            E.cb_slot_text(slot, i + 1, buf, 160)
            row.append(buf.value.decode())
        else:
            row.append(int(s.tts_values[i]))
    return row, states


class Result:
    def __init__(self):
        self.rows = []
        self.states = []
        self.segments = []
        self.instrument = {}


def _collect_instrument(ps, out):
    if not ps:
        return
    n = ps.contents
    ins = n.instrument
    out[n.plan.contents.plan_node_id] = {"node": n.type, "ntuples": ins.ntuples, "kernels": ins.kernels,
                                         "device_ms": ins.device_ms, "rows_in": ins.rows_in,
                                         "motion_repartitions": ins.motion_repartitions, "hashjoin_nbatch": ins.hashjoin_nbatch,
                                         "agg_npartitions": ins.agg_npartitions}
    _collect_instrument(n.lefttree, out)
    _collect_instrument(n.righttree, out)


class Executor:
    """ExecutorStart / ExecutorRun / ExecutorEnd for one segment (one GPU)."""

    def __init__(self, ctx, range_table, force_generic=False, motion=None, operator_mem_kb=0):
        self.ctx = ctx
        self.E = ex()
        n = len(range_table)
        arr = (C.c_void_p * max(n, 1))(*[r.h for r in range_table])
        self.estate = self.E.cb_CreateExecutorState(ctx.h, arr, n)
        self.estate.contents.es_force_generic = 1 if force_generic else 0
        # PlanStateOperatorMemKB: hash join build sides / aggregate tables larger than this run in batches / partitions
        self.estate.contents.es_operator_mem_kb = int(operator_mem_kb)
        self._keep = [arr, range_table]
        self.ic = None
        if motion is not None:
            # SetupInterconnect (executor/execMain.c:531): this process is segment `rank` of `nranks`
            self.ic = self.E.cb_interconnect_nccl_create(motion.h)
            self.estate.contents.es_interconnect = self.ic
            self.estate.contents.es_segindex = motion.rank
            self.estate.contents.es_numsegments = motion.nranks
            self._keep.append(motion)

    def run(self, plan_node):
        """Pull every tuple through cb_ExecProcNode, as ExecutePlan does (execMain.c:2772)."""
        E = self.E
        es = self.estate
        es.contents.es_errcode = 0
        ps = E.cb_ExecInitNode(P.plan_ptr(plan_node), es, 0)
        if not ps:
            raise CbgpuError(es.contents.es_errcode, E.cb_estate_error(es).decode())
        res = Result()
        try:
            while True:
                slot = E.cb_ExecProcNode(ps)
                if es.contents.es_errcode:
                    raise CbgpuError(es.contents.es_errcode, E.cb_estate_error(es).decode())
                if not slot or slot.contents.tts_empty:
                    break
                row, st = _slot_row(E, slot)
                res.rows.append(row)
                res.states.append(st)
                res.segments.append(0)
            _collect_instrument(ps, res.instrument)
        finally:
            E.cb_ExecEndNode(ps)
        return res

    def run_batch(self, plan_node, name="batch"):
        """The plan's whole output as one device-resident relation (cb_ExecProcNodeBatch)."""
        E = self.E
        es = self.estate
        es.contents.es_errcode = 0
        ps = E.cb_ExecInitNode(P.plan_ptr(plan_node), es, 0)
        if not ps:
            raise CbgpuError(es.contents.es_errcode, E.cb_estate_error(es).decode())
        try:
            h = C.c_void_p()
            rc = E.cb_ExecProcNodeBatch(ps, C.byref(h))
            if rc or es.contents.es_errcode:
                raise CbgpuError(rc or es.contents.es_errcode, E.cb_estate_error(es).decode())
            return DeviceRelation.adopt(self.ctx, h, name)
        finally:
            E.cb_ExecEndNode(ps)

    def close(self):
        if self.estate:
            self.E.cb_FreeExecutorState(self.estate)
            self.estate = None
        if self.ic:
            self.E.cb_interconnect_destroy(self.ic)
            self.ic = None


class Cluster:
    """N segment executors in one process over one GPU (the reference's gpdemo, on a device)."""

    def __init__(self, ctx, segment_range_tables, force_generic=False, operator_mem_kb=0):
        self.ctx = ctx
        self.E = ex()
        self.nsegs = len(segment_range_tables)
        self.h = self.E.cb_cluster_create(ctx.h, self.nsegs)
        self._keep = []
        for s, rt in enumerate(segment_range_tables):
            arr = (C.c_void_p * max(len(rt), 1))(*[r.h for r in rt])
            self._keep += [arr, rt]
            rc = self.E.cb_cluster_set_range_table(self.h, s, arr, len(rt))
            if rc:
                raise CbgpuError(rc, "bad range table")
            self.E.cb_cluster_estate(self.h, s).contents.es_force_generic = 1 if force_generic else 0
            self.E.cb_cluster_estate(self.h, s).contents.es_operator_mem_kb = int(operator_mem_kb)

    def run(self, plan_node):
        E = self.E
        rc = E.cb_cluster_init_plan(self.h, P.plan_ptr(plan_node))
        if rc:
            msg = E.cb_cluster_error(self.h).decode()
            E.cb_cluster_end(self.h)
            raise CbgpuError(rc, msg)
        res = Result()
        try:
            while True:
                slot = E.cb_cluster_next(self.h)
                err = E.cb_cluster_error(self.h)
                if err:
                    raise CbgpuError(-1, err.decode())
                if not slot or slot.contents.tts_empty:
                    break
                row, st = _slot_row(E, slot)
                res.rows.append(row)
                res.states.append(st)
                res.segments.append(int(E.cb_cluster_current_segment(self.h)))
        finally:
            E.cb_cluster_end(self.h)
        return res

    def close(self):
        if self.h:
            self.E.cb_cluster_destroy(self.h)
            self.h = None
