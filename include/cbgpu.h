/*
 * cbgpu.h - thin C ABI over the sm_100a CUDA kernels (libcbgpu.so).
 *
 * Plain C: pointers, sizes and POD structs only; no CUDA or torch types cross this boundary.
 * The host executor (include/cb_exec.h, cloudberry_b200/csrc/exec/ *.c, plain C) is the only
 * caller on the product path; a Cloudberry backend shim would bind the same entry points
 * (INTEGRATION.md).  Every function returns CBGPU_OK or a negative error code and leaves a
 * message in cbgpu_last_error(ctx); nothing longjmps or throws across the boundary
 * (the reference reports errors with ereport(ERROR) = siglongjmp, utils/elog.h:185; the shim turns
 * a status code into ereport only after the stream is drained and device memory released).
 *
 * What each group of entry points replaces in the reference (paths under /root/reference/src):
 *
 *   relations / columns   the decoded form of an AOCS scan: aocs_beginscan (backend/access/aocs/
 *                         aocsam.c:549) chooses projected columns, datumstreamread_block + the
 *                         block cursor (backend/utils/datumstream/datumstream.c:1364,
 *                         include/utils/datumstreamblock.h:1220-1614) decode them.  Here a column
 *                         is one HBM-resident fixed-width array.
 *   cbgpu_pipeline_run    the per-row inner loops: aocs_getnext (aocsam.c:1418) + ExecScan qual /
 *                         projection (backend/executor/execScan.c:162) + ExecHashJoin probe
 *                         (backend/executor/nodeHashjoin.c:203, nodeHash.c:2089,2255) +
 *                         agg_fill_hash_table / advance_aggregates (backend/executor/nodeAgg.c:2726,
 *                         856) + execMotionSender's evalHashKey (backend/executor/nodeMotion.c:1088),
 *                         fused into one late-materialising kernel per pipeline.
 *   cbgpu_ht_*            MultiExecPrivateHash / ExecHashTableInsert (backend/executor/nodeHash.c:
 *                         167,1877) and ExecScanHashBucket (:2255).
 *   cbgpu_agg_*           TupleHashTable + per-group transition states (backend/executor/
 *                         execGrouping.c:317, nodeAgg.c:2220-2319) and agg_retrieve_hash_table
 *                         (nodeAgg.c:2952).
 *   cbgpu_topn            Limit <- Sort above the Agg (bounded tuplesort), device side so ~1.2M
 *                         Q3 groups are not drained through slots.
 *   cbgpu_motion_*        cdbmotion SendTuple / RecvTupleFrom over a MotionIPCLayer
 *                         (backend/cdb/motion/cdbmotion.c:425,549; include/cdb/ml_ipc.h:36-210),
 *                         replaced by a hash-partition kernel + NCCL grouped send/recv.
 */
#ifndef CBGPU_H
#define CBGPU_H

#include <stdint.h>
#include <stddef.h>
#include "cb_plan.h"

#ifdef __cplusplus
extern "C" {
#endif

#define CBGPU_OK 0
#define CBGPU_ERR_CUDA (-1)			/* a CUDA runtime / NCCL call failed                              */
#define CBGPU_ERR_INVALID (-2)		/* bad argument / malformed descriptor                             */
#define CBGPU_ERR_UNSUPPORTED (-3)	/* valid plan shape the GPU path does not implement: fail loudly,
									 * there is no CPU fallback                                        */
#define CBGPU_ERR_OVERFLOW (-4)		/* integer / numeric value out of range during execution           */
#define CBGPU_ERR_NOMEM (-5)
#define CBGPU_ERR_CORRUPT (-6)		/* stored data fails its checksum (AOCS block CRC-32C)              */
#define CBGPU_ERR_PEER (-7)			/* another segment failed, or did not signal within the interconnect's
									 * time limit (CBGPU_MOTION_TIMEOUT_MS)                             */
#define CBGPU_ERR_INTERRUPTED (-8)	/* the caller's interrupt callback asked for the query to stop      */

typedef struct cbgpu_ctx cbgpu_ctx;
typedef struct cbgpu_rel cbgpu_rel;
typedef struct cbgpu_hashtable cbgpu_hashtable;
typedef struct cbgpu_aggtable cbgpu_aggtable;
typedef struct cbgpu_motion cbgpu_motion;

/* ------------------------------------------------------------------------------------------
 * context
 * ------------------------------------------------------------------------------------------ */
int			cbgpu_ctx_create(int device, cbgpu_ctx **out);	/* lazily initialises CUDA: call after fork */
void		cbgpu_ctx_destroy(cbgpu_ctx *ctx);
const char *cbgpu_last_error(cbgpu_ctx *ctx);
int			cbgpu_sync(cbgpu_ctx *ctx);						/* drain the context's stream              */
/* drain the stream and report (then clear) an error a kernel raised: overflow, full table / buffer */
int			cbgpu_check_status(cbgpu_ctx *ctx);
int			cbgpu_device_count(void);
int			cbgpu_sm_count(cbgpu_ctx *ctx);
int64_t		cbgpu_kernel_launches(cbgpu_ctx *ctx);			/* kernels launched so far on this ctx     */
/* device-side timing on the context's stream (CUDA events) */
int			cbgpu_timer_start(cbgpu_ctx *ctx);
int			cbgpu_timer_stop_ms(cbgpu_ctx *ctx, double *ms);
/* last pipeline kernel's own duration (events around that launch only) and its name */
double		cbgpu_last_kernel_ms(cbgpu_ctx *ctx);
/* log of pipeline kernels launched since the last reset; the longest one's name and duration */
void		cbgpu_kernel_log_reset(cbgpu_ctx *ctx);
int			cbgpu_kernel_log_longest(cbgpu_ctx *ctx, char *name, int namelen, double *ms);
const char *cbgpu_last_kernel_name(cbgpu_ctx *ctx);
/* launch trace (profiling aid): an event after every kernel launch between begin and end; end
 * returns the number of entries, get returns entry i's name and its event-to-event time */
int			cbgpu_trace_begin(cbgpu_ctx *ctx);
int			cbgpu_trace_end(cbgpu_ctx *ctx);
int			cbgpu_trace_get(cbgpu_ctx *ctx, int i, char *name, int namelen, double *ms);
/* NVTX ranges (profilers show one range per plan node around its kernels); no-ops without a profiler attached */
void		cbgpu_range_push(const char *name);
void		cbgpu_range_pop(void);
/* write `bytes` of HBM so the next timed kernel starts with a cold L2 */
int			cbgpu_flush_l2(cbgpu_ctx *ctx);
/* pinned host memory for the end-to-end (host buffers) path */
void	   *cbgpu_host_alloc(size_t bytes);
void		cbgpu_host_free(void *p);

/* hashbpchar (backend/utils/adt/varchar.c:981) on the host, for dictionary columns */
uint32_t	cbgpu_hashbpchar(const char *s, int32_t len);

/* ------------------------------------------------------------------------------------------
 * relations: HBM-resident column batches
 * ------------------------------------------------------------------------------------------ */
int			cbgpu_rel_create(cbgpu_ctx *ctx, int64_t nrows, int32_t ncols, const int32_t *types,
							 const int32_t *dscales, cbgpu_rel **out);
void		cbgpu_rel_free(cbgpu_rel *rel);
int64_t		cbgpu_rel_nrows(const cbgpu_rel *rel);
int32_t		cbgpu_rel_ncols(const cbgpu_rel *rel);
int32_t		cbgpu_rel_col_type(const cbgpu_rel *rel, int32_t col);
int32_t		cbgpu_rel_col_dscale(const cbgpu_rel *rel, int32_t col);
/* host -> device copy of one whole column (asynchronous on the context stream when `host` is
 * pinned); nulls: NULL or one byte per row (1 = NULL) */
int			cbgpu_rel_load_column(cbgpu_rel *rel, int32_t col, const void *host, const uint8_t *nulls);
/* the same for a host column held in a NARROWER two's-complement integer width than the column's own (host_width 1, 2 or 4
 * bytes into an 8- or 4-byte integer / date / scaled-numeric column): copied as it is and sign-extended on the device.  A
 * load is PCIe-bound, so a loader that knows a column's value range (block min / max) ships a numeric(15,2) quantity as
 * int16 instead of int64; the relation in HBM is the same either way.  No NULL map (use cbgpu_rel_load_column for those). */
int			cbgpu_rel_load_column_narrow(cbgpu_rel *rel, int32_t col, const void *host, int32_t host_width);
/* device -> host copy of rows [lo, hi) of a column (blocking) */
int			cbgpu_rel_read_column(cbgpu_rel *rel, int32_t col, int64_t lo, int64_t hi, void *host, uint8_t *nulls);
/* visibility bitmap, one bit per row, 1 = visible (appendonly_visimap.c:198); NULL clears it */
int			cbgpu_rel_set_visimap(cbgpu_rel *rel, const uint8_t *bits);
/* the bitmap back ((nrows + 7) / 8 bytes; all ones when the relation has none) */
int			cbgpu_rel_read_visimap(cbgpu_rel *rel, uint8_t *bits);
/* per-code hashbpchar values of a dictionary column (so it can be a hash key) */
int			cbgpu_rel_set_dict_hash(cbgpu_rel *rel, int32_t col, const uint32_t *hashes, int32_t n);
/* shrink the logical row count (relations allocated at an upper bound, e.g. Motion receive) */
int			cbgpu_rel_set_nrows(cbgpu_rel *rel, int64_t nrows);
/* dst rows [0, n) = src rows dev_idx[0..n) (a DEVICE index list), all columns and NULL maps: an ordered gather (the merged
 * order of a sorted Motion) */
int			cbgpu_rel_take_rows(cbgpu_rel *dst, cbgpu_rel *src, const uint32_t *dev_idx, int64_t n);
/* n rows (host_idx[0..n), or the first n when host_idx is NULL) of EVERY column in one round trip: values widened
 * to int64 (float8: raw bits), row-major out[r * ncols + c], outnull likewise.  For small result sets. */
int			cbgpu_rel_read_rows(cbgpu_rel *rel, const uint32_t *host_idx, int64_t n, int64_t *out, uint8_t *outnull);
/* raw device pointer of a column (for harness-side generators / NCCL); not dereferenceable on host */
void	   *cbgpu_rel_col_devptr(cbgpu_rel *rel, int32_t col);
size_t		cbgpu_rel_nbytes(const cbgpu_rel *rel);

/* ------------------------------------------------------------------------------------------
 * pipelines: driving source -> [filter | probe]* -> sink, one fused kernel
 * ------------------------------------------------------------------------------------------ */
#define CBP_MAX_SRC 8
#define CBP_MAX_COLS 40
#define CBP_MAX_OPS 128
#define CBP_MAX_KEYS 4
#define CBP_MAX_AGGS 16
#define CBP_MAX_OUT 48
#define CBP_STACK 48

typedef enum CbpOpCode
{
	CBP_END = 0,
	CBP_LOAD,			/* a = column index; push value widened to 64 bits (float8: raw bits)        */
	CBP_CONST,			/* push imm                                                                   */
	CBP_ADD, CBP_SUB, CBP_MUL,		/* int64 (ints, dates, scaled numerics); overflow -> error        */
	CBP_FADD, CBP_FSUB, CBP_FMUL,	/* float8                                                         */
	CBP_I2F,			/* int64 scaled by 10^a -> float8                                             */
	CBP_EQ, CBP_NE, CBP_LT, CBP_LE, CBP_GT, CBP_GE,			/* int64 compare -> bool                  */
	CBP_FEQ, CBP_FNE, CBP_FLT, CBP_FLE, CBP_FGT, CBP_FGE,	/* float8 compare (PG NaN ordering)       */
	CBP_AND, CBP_OR, CBP_NOT,		/* three-valued                                                   */
	CBP_FILTER,			/* pop; the row survives only if the value is true (not NULL)                 */
	CBP_PROBE,			/* a = probe index; pops that probe's key values (pushed in key order)        */
	CBP_DUP,			/* push a copy of stack[a] (common sub-expressions)                           */
	CBP_POP,
	CBP_F8ORD			/* float8 bits -> an int64 whose integer order is float8's (float8_cmp_internal, utils/adt/float.c: every
						 * NaN equal and above everything); its own inverse on non-NaN values.  Lets min / max(float8) use
						 * the integer min / max accumulators */
} CbpOpCode;

typedef struct CbpOp
{
	int32_t		code;
	int32_t		a;
	int64_t		imm;
} CbpOp;

typedef struct CbpColumn
{
	const void *data;			/* device pointer                                                     */
	const uint8_t *nulls;		/* device pointer, one byte per row, or NULL                          */
	const uint32_t *dict_hash;	/* device pointer: per-code hash for CB_DICT*, or NULL                */
	int32_t		type;			/* CbTypeId                                                           */
	int32_t		src;			/* which source's row index addresses it: 0 = driving relation,
								 * 1 + j = inner side of probe j                                      */
} CbpColumn;

typedef struct CbpProbe
{
	const cbgpu_hashtable *ht;
	int32_t		jointype;		/* CbJoinType: INNER, LEFT, SEMI, ANTI                                */
	int32_t		nkeys;
	int32_t		keytype[CBP_MAX_KEYS];	/* CbTypeId of each outer key value (for its hash function)   */
	const uint32_t *key_dict_hash[CBP_MAX_KEYS];
	int32_t		null_key_drops;	/* ANTI probe of a NOT IN join over a non-empty build side: an outer row whose key is
								 * NULL is dropped, not kept (x NOT IN (...) is unknown: nodeHashjoin.c:578-590)    */
} CbpProbe;

typedef enum CbpSinkKind
{
	CBP_SINK_AGG = 1,			/* hash aggregate into an agg table                                   */
	CBP_SINK_MATERIALIZE,		/* append the stack values as rows of an output relation              */
	CBP_SINK_PARTITION			/* like MATERIALIZE, rows grouped by destination segment (Motion)     */
} CbpSinkKind;

typedef enum CbpAggKind
{
	CBP_ACC_COUNT = 1,			/* N += 1 (count(*)) or N += (arg not null)                           */
	CBP_ACC_SUM_INT,			/* N, 128-bit exact sum: int4_sum / int8_avg_accum / numeric_avg_accum */
	CBP_ACC_SUM_FLOAT,			/* N, float8 Sx: float8pl / float8_accum                              */
	CBP_ACC_MIN, CBP_ACC_MAX,	/* int64 ordering (ints, dates, scaled numerics)                      */
	CBP_ACC_MERGE_INT,			/* combine: arg pair (N, 128-bit sum) from a partial state            */
	CBP_ACC_MERGE_FLOAT,		/* arg pair (N, Sx bits)                                              */
	CBP_ACC_MERGE_COUNT,		/* arg N                                                              */
	CBP_ACC_MERGE_MIN,			/* arg pair (N, value): ignored when N = 0                            */
	CBP_ACC_MERGE_MAX
} CbpAggKind;

typedef struct CbpAcc
{
	int32_t		kind;			/* CbpAggKind                                                         */
	int32_t		arg;			/* stack position (0-based, after the keys) of the argument, -1 none;
								 * MERGE_INT takes 3 consecutive values: N, sum.lo, sum.hi            */
} CbpAcc;

typedef struct CbpSink
{
	int32_t		kind;
	/* AGG */
	cbgpu_aggtable *agg;
	int32_t		nkeys;
	int32_t		keytype[CBP_MAX_KEYS];
	const uint32_t *key_dict_hash[CBP_MAX_KEYS];
	int32_t		naccs;
	CbpAcc		accs[CBP_MAX_AGGS];
	/* MATERIALIZE / PARTITION: the top `nout` stack values become one output row */
	int32_t		nout;
	cbgpu_rel  *out;			/* preallocated with capacity >= possible rows                        */
	int64_t	   *out_count;		/* device counter(s): [1] or [nsegs]                                  */
	/* PARTITION: cdbhash over the first nhash output values */
	int32_t		nhash;
	int32_t		hashtype[CBP_MAX_KEYS];
	const uint32_t *hash_dict_hash[CBP_MAX_KEYS];
	int32_t		nsegs;
	int64_t		seg_capacity;	/* rows reserved per destination inside `out`                         */
	/* PARTITION, direct mode (cbgpu_motion_direct_begin): rows are stored into the destinations' own
	 * buffers instead of `out` (which then only describes the column types): part_cols[d * nout + c],
	 * part_counts[d]; seg_capacity = rows every destination can take */
	void *const *part_cols;
	unsigned long long *const *part_counts;
	uint8_t *const *part_nulls;	/* direct mode: NULL byte bases, [d * nout + c]                       */
	uint64_t	part_nullmask;	/* direct mode: bit c = store column c's NULL bytes                   */
	/* where a full destination is reported (CBGPU_DX_OVERFLOW is ORed in; the rows beyond the capacity are
	 * dropped, the per-destination counters still count them, the caller redoes the pass with exact sizes).
	 * NULL: a full destination raises CBGPU_ERR_NOMEM in the status word instead. */
	int32_t    *part_flags;
	/* staged mode, exact layout: destination d's rows start at row seg_base[d] of `out` and seg_cap[d] of
	 * them fit (host arrays of nsegs entries); NULL: d * seg_capacity, seg_capacity */
	const int64_t *seg_base;
	const int64_t *seg_cap;
} CbpSink;

typedef struct CbPipeline
{
	int64_t		nrows;			/* rows of the driving source                                         */
	const uint8_t *visimap;		/* driving relation's visibility bits or NULL                         */
	/* optional driver index vectors: row i addresses source s at drv_idx[s][i] (identity if NULL).
	 * Used to continue from join pairs (outer_idx, inner_idx) or a selection vector. */
	int32_t		drv_nsrc;
	const uint32_t *drv_idx[CBP_MAX_SRC];
	int32_t		ncols;
	CbpColumn	cols[CBP_MAX_COLS];
	int32_t		nops;
	CbpOp		ops[CBP_MAX_OPS];
	int32_t		nprobes;
	CbpProbe	probes[CBP_MAX_SRC - 1];
	CbpSink		sink;
	int32_t		force_generic;	/* tests: bypass the pattern-specialised kernels                      */
} CbPipeline;

int			cbgpu_pipeline_run(cbgpu_ctx *ctx, const CbPipeline *p);

/* ------------------------------------------------------------------------------------------
 * hash join tables
 * ------------------------------------------------------------------------------------------ */
/* build over rows of `inner` (all rows, or those listed in sel[0..nsel)); key columns by index.
 * NULL keys are not inserted (strict hash operators, nodeHash.c:2161). */
int			cbgpu_ht_build(cbgpu_ctx *ctx, cbgpu_rel *inner, const int32_t *keycols, int32_t nkeys,
						   cbgpu_hashtable **out);
/* multi-batch hybrid hash join (nodeHash.c:980-990, 1133, 2223-2242): the build side is split into nbatch (a power of two)
 * batches by bits of the key hash that the slot index does not use; the table holds one batch at a time
 * (cbgpu_ht_load_batch) and sizes itself for the fullest.  A pipeline that probes it runs once per batch - probe rows of
 * other batches are skipped in each pass - and its sink accumulates over the passes.  cbgpu_ht_bytes_for(rows) = device
 * bytes of a one-batch table, for choosing nbatch against a budget. */
int			cbgpu_ht_build_batched(cbgpu_ctx *ctx, cbgpu_rel *inner, const int32_t *keycols, int32_t nkeys, int32_t nbatch,
								   cbgpu_hashtable **out);
int			cbgpu_ht_nbatch(const cbgpu_hashtable *ht);
int			cbgpu_ht_load_batch(cbgpu_hashtable *ht, int32_t batch);
int64_t		cbgpu_ht_bytes_for(int64_t rows);
void		cbgpu_ht_free(cbgpu_hashtable *ht);
int64_t		cbgpu_ht_nrows(const cbgpu_hashtable *ht);
int			cbgpu_ht_has_duplicates(const cbgpu_hashtable *ht);
/* the per-code hash table (device pointer) of dictionary key column k of the build side, NULL for other types:
 * the identity of the dictionary the build keys are coded by */
const uint32_t *cbgpu_ht_key_dict_hash(const cbgpu_hashtable *ht, int32_t k);
/* stand-alone probe emitting (outer_idx, inner_idx) pairs for an INNER join (all matches);
 * outer key columns by index.  pairs are written to two device arrays owned by the call result. */
typedef struct cbgpu_pairs
{
	int64_t		npairs;
	uint32_t   *outer_idx;		/* device                                                             */
	uint32_t   *inner_idx;		/* device                                                             */
} cbgpu_pairs;
int			cbgpu_ht_probe_pairs(cbgpu_ctx *ctx, const cbgpu_hashtable *ht, cbgpu_rel *outer,
								 const int32_t *keycols, int32_t nkeys, const uint32_t *sel, int64_t nsel,
								 cbgpu_pairs *out);
/* the same for a LEFT join: an outer row without a partner yields one pair whose inner_idx is 0xFFFFFFFF (a pipeline driven
 * by the pairs reads that source as NULL: HJ_FILL_OUTER_TUPLE, nodeHashjoin.c:640-660) */
int			cbgpu_ht_probe_pairs_left(cbgpu_ctx *ctx, const cbgpu_hashtable *ht, cbgpu_rel *outer, const int32_t *keycols,
									  int32_t nkeys, cbgpu_pairs *out);
/* all outer-join flavours of the pair probe: fill_outer adds (row, 0xFFFFFFFF) for probe rows without a partner (LEFT /
 * FULL), fill_inner adds (0xFFFFFFFF, row) for build rows no probe row matched, NULL-keyed build rows included (RIGHT /
 * FULL: ExecScanHashTableForUnmatched nodeHash.c:2360, HJ_FILL_INNER_TUPLES nodeHashjoin.c:676-706) */
int			cbgpu_ht_probe_pairs_outer(cbgpu_ctx *ctx, const cbgpu_hashtable *ht, cbgpu_rel *outer, const int32_t *keycols,
									   int32_t nkeys, int32_t fill_outer, int32_t fill_inner, cbgpu_pairs *out);
/* every outer-join flavour of the pair probe (as cbgpu_ht_probe_pairs_outer) over a table of any batch count: the probe rows
 * are grouped by batch once (a NULL-keyed row in batch 0), each batch with probe rows is loaded and probed in turn, and the
 * build rows no probe row matched are emitted once after the last batch.  Pairs come in (batch, outer row) order - a row's
 * partners in build row order - then the unmatched build rows in row order.  pending(pending_arg), when given, is polled
 * before each batch (nonzero: CBGPU_ERR_INTERRUPTED); *passes = batches probed.  The table is left on the last batch the
 * call loaded (a single-batch table: the cbgpu_ht_probe_pairs_outer path, unchanged). */
int			cbgpu_ht_probe_pairs_batched(cbgpu_ctx *ctx, cbgpu_hashtable *ht, cbgpu_rel *outer, const int32_t *keycols,
										 int32_t nkeys, int32_t fill_outer, int32_t fill_inner, int (*pending) (void *),
										 void *pending_arg, int64_t *passes, cbgpu_pairs *out);
void		cbgpu_pairs_free(cbgpu_pairs *p);
int			cbgpu_read_u32(cbgpu_ctx *ctx, const uint32_t *dev, int64_t n, uint32_t *host);
/* small device scratch (sink row counters, index vectors): zero-filled allocation, read-back, free */
int			cbgpu_dev_alloc(cbgpu_ctx *ctx, size_t bytes, void **dev);
int			cbgpu_dev_read(cbgpu_ctx *ctx, const void *dev, size_t bytes, void *host);
int			cbgpu_dev_write(cbgpu_ctx *ctx, void *dev, size_t bytes, const void *host);
void		cbgpu_dev_free(cbgpu_ctx *ctx, void *dev);
/* give column `col` of an output relation a NULL byte-map (zero-filled) so sinks may store NULLs */
int			cbgpu_rel_add_nullmap(cbgpu_rel *rel, int32_t col);
/* device -> device copy of rows [src_lo, src_lo + n) of every column of `src` to row dst_lo of `dst`
 * (same column types); the local interconnect and Motion receive buffers use it */
int			cbgpu_rel_copy_rows(cbgpu_rel *dst, int64_t dst_lo, cbgpu_rel *src, int64_t src_lo, int64_t n);
int			cbgpu_rel_has_nulls(const cbgpu_rel *rel, int32_t col);
const uint32_t *cbgpu_rel_dict_hash_dev(const cbgpu_rel *rel, int32_t col);
const uint8_t *cbgpu_rel_nulls_dev(const cbgpu_rel *rel, int32_t col);
const uint8_t *cbgpu_rel_visimap_dev(const cbgpu_rel *rel);
/* share a dictionary hash table between relations (device pointer copy; `dst` does not own it) */
int			cbgpu_rel_share_dict_hash(cbgpu_rel *dst, int32_t dcol, const cbgpu_rel *src, int32_t scol);

/* ------------------------------------------------------------------------------------------
 * aggregate tables
 * ------------------------------------------------------------------------------------------ */
/* acc_kinds[a] (CbpAggKind) fixes each accumulator's initial value (MIN / MAX need one) */
int			cbgpu_agg_create(cbgpu_ctx *ctx, int32_t nkeys, int32_t naccs, const int32_t *acc_kinds,
							 int64_t capacity_groups, cbgpu_aggtable **out);
void		cbgpu_agg_free(cbgpu_aggtable *t);
/* partitioned aggregation for group sets larger than the operator's memory (nodeAgg.c:2149, 3215): with npart (a power of two)
 * partitions set, a pipeline's AGG sink aggregates only the rows whose group hash selects partition `part`; the caller runs
 * the pipeline once per partition and takes each pass's groups away (cbgpu_agg_to_rel) before the next.
 * cbgpu_agg_slot_bytes: device bytes per table slot (two slots are provisioned per group), for sizing against a budget. */
int			cbgpu_agg_set_partition(cbgpu_aggtable *t, int32_t npart, int32_t part);
int64_t		cbgpu_agg_slot_bytes(int32_t nkeys, int32_t naccs);
int			cbgpu_agg_reset(cbgpu_aggtable *t);
/* number of groups present (blocking) */
int			cbgpu_agg_ngroups(cbgpu_aggtable *t, int64_t *ngroups);
/* copy the groups out, compacted, in table order: keys[g*nkeys+k] (64-bit widened),
 * keynull[g] bit k, n[g*naccs+a], sum_lo/sum_hi[g*naccs+a] (float8 states: bits in sum_lo) */
int			cbgpu_agg_read(cbgpu_aggtable *t, int64_t maxgroups, int64_t *keys, uint32_t *keynull,
						   int64_t *n, int64_t *sum_lo, int64_t *sum_hi, int64_t *ngroups);
/* groups as a device relation: columns = keys (typed), then per accumulator N (int8) and the
 * 128-bit sum as two int8 columns (lo, hi); used as the source of the next pipeline (Motion,
 * final aggregation) and by top-N */
int			cbgpu_agg_to_rel(cbgpu_aggtable *t, const int32_t *keytypes, cbgpu_rel **out);

/* device top-N over a relation: ORDER BY up to 4 (column, descending) keys LIMIT n; 128-bit
 * values are ordered through (hi, lo) column pairs: pass hi as the key and lo as the next key.
 * Returns the chosen row indices in order. */
int			cbgpu_topn(cbgpu_ctx *ctx, cbgpu_rel *rel, const int32_t *keycols, const int32_t *descending,
					   const int32_t *unsigned_cmp, int32_t nkeys, int64_t limit, uint32_t *host_idx,
					   int64_t *nout);
/* Merge receive of a sorted Gather Motion (Motion.sendSorted; execMotionSortedReceiver nodeMotion.c:433, CdbMergeComparator
 * :1010): `rel` holds the senders' sorted streams one after another; *order_dev (device, cbgpu_dev_free; NULL when the
 * arrival order already is the order) lists its rows in merged order - equal keys: the earlier sender first.  NULLs sort
 * last ascending, first descending.  More than max_runs sorted runs means a sender broke the order: CBGPU_ERR_INVALID. */
int			cbgpu_merge_sorted_runs(cbgpu_ctx *ctx, cbgpu_rel *rel, const int32_t *keycols, const int32_t *descending,
									const int32_t *unsigned_cmp, int32_t nkeys, int32_t max_runs, uint32_t **order_dev,
									int32_t *nruns_out);

/* ------------------------------------------------------------------------------------------
 * interconnect between GPU-segments, one process per GPU (backend/cdb/motion/cdbmotion.c:425,549 and
 * the MotionIPCLayer implementations under contrib/interconnect are what this replaces).
 *
 * Two transports share one object:
 *   peer-memory windows   every rank owns a receive window in its HBM, mapped into every other rank's
 *                         process (CUDA IPC) at create time.  A Motion is the sender slice's own kernel
 *                         storing rows into the destination's window over NVLink, framed by DEVICE-side
 *                         signals in the windows' control blocks (st.release.sys / ld.acquire.sys epoch
 *                         words): no collective call and one host round trip (the receiver learning its
 *                         row count) per Motion.
 *   NCCL                  staged partition + count all-gather + grouped ncclSend / ncclRecv: the fallback
 *                         for what the windows cannot take (a Motion larger than the window, Broadcast),
 *                         and the only transport where P2P / IPC is unavailable.
 * ------------------------------------------------------------------------------------------ */
/* 128-byte rendezvous token created on one rank and handed to all (the harness broadcasts it) */
int			cbgpu_motion_unique_id(void *out128);
int			cbgpu_motion_create(cbgpu_ctx *ctx, int rank, int nranks, const void *unique_id128, cbgpu_motion **out);
/* Interconnect over the peer-memory windows alone, bootstrapped through an all-gather the CALLER
 * provides (the backend's dispatcher connection, a torch.distributed store ...): every rank passes
 * `bytes` of `mine` and gets nranks * bytes back in rank order; blocking; returns 0 on success.  No
 * NCCL communicator is created (two ranks may share one device: the single-GPU multi-process tests run
 * so), hence no staged fallback: a Motion the windows cannot take is an error. */
typedef int (*cbgpu_allgather_fn) (void *arg, const void *mine, void *all, size_t bytes);
int			cbgpu_motion_create_boot(cbgpu_ctx *ctx, int rank, int nranks, cbgpu_allgather_fn allgather, void *arg,
									 cbgpu_motion **out);
void		cbgpu_motion_destroy(cbgpu_motion *m);
/* tear down WITHOUT any collective step (after a failed query the peers may be gone or out of step:
 * cdbmotion's TeardownInterconnect with hasErrors, include/cdb/ml_ipc.h:106): aborts the NCCL
 * communicator, unmaps the windows */
void		cbgpu_motion_abort(cbgpu_motion *m);
int			cbgpu_motion_rank(const cbgpu_motion *m);
int			cbgpu_motion_nranks(const cbgpu_motion *m);
int64_t		cbgpu_motion_bytes_sent(const cbgpu_motion *m);
/* Redistribute (staged): `send` holds this rank's rows grouped by destination (destination d's rows start
 * at row offsets[d], counts[d] of them); returns the rows addressed to this rank, sender by sender.
 * Receive sizes are exchanged exactly, so no skew can overflow a receiver.  counts[0] < 0 announces "this
 * rank failed before the exchange": every rank then returns CBGPU_ERR_PEER instead of waiting for it. */
int			cbgpu_motion_redistribute(cbgpu_motion *m, cbgpu_rel *send, const int64_t *counts, const int64_t *offsets,
									  cbgpu_rel **recv);
/* this rank failed before its part of the next exchange: tell the peers so that they return CBGPU_ERR_PEER
 * instead of waiting for it.  staged = 0: the peers are entering a direct exchange (or a staged one where
 * there are no windows); staged = 1: they are entering the staged exchange that follows a CBGPU_DX_RETRY. */
int			cbgpu_motion_abandon(cbgpu_motion *m, int staged);
/* Direct Redistribute: partition + exchange fused into the sender slice's own kernel, over the windows.
 *   begin  (local, no synchronisation) lays the exchange out inside every window - the same arithmetic on
 *          every rank, from the column types and the common window size alone - and queues the device-side
 *          wait for "every receiver has emptied its window of the previous exchange".  Returns what the
 *          PARTITION sink needs: per destination d the column bases cols[d * ncols + c], the NULL byte
 *          bases nulls[d * ncols + c], the row counter counts[d] (peer memory, system-scope atomics), the
 *          capacity in rows of every destination, and a device flag word the sink ORs CBGPU_DX_OVERFLOW
 *          into when a destination is full (rows beyond the capacity are dropped, the exchange is redone
 *          staged: the reference never fails on skew, cdbmotion.c:425).
 *          CBGPU_ERR_UNSUPPORTED = no windows, or a row too wide for them: use cbgpu_motion_redistribute
 *          (the answer depends on nothing rank-specific, so all ranks agree).
 *   end    after the pipeline ran (or failed: pass CBGPU_DX_ERROR, the peers must not wait for this rank
 *          for ever): signal "my rows are stored" into every window, wait for every sender's signal, take
 *          delivery.  local_nullmask: bit c = this rank stored NULL bytes for column c.  *outcome:
 *          CBGPU_DX_DELIVERED, or CBGPU_DX_RETRY (some destination overflowed or some rank vetoed;
 *          nothing was delivered anywhere, every rank redoes the Motion through cbgpu_motion_redistribute).
 *          A rank that passed CBGPU_DX_ERROR makes every rank return CBGPU_ERR_PEER.
 *          The sink's own per-destination counters (dev_sent_counts, device) come back in the same round trip. */
#define CBGPU_DX_OVERFLOW 1
#define CBGPU_DX_VETO 2
#define CBGPU_DX_ERROR 4
#define CBGPU_DX_NOFIT 8
#define CBGPU_DX_DELIVERED 0
#define CBGPU_DX_RETRY 1
typedef struct cbgpu_direct_dest
{
	int64_t		capacity;
	void *const *cols;
	uint8_t *const *nulls;
	unsigned long long *const *counts;
	int32_t    *flags;
} cbgpu_direct_dest;
int			cbgpu_motion_direct_available(const cbgpu_motion *m);
int			cbgpu_motion_direct_begin(cbgpu_motion *m, int32_t ncols, const int32_t *types, const int32_t *dscales,
									  cbgpu_direct_dest *dest);
int			cbgpu_motion_direct_end(cbgpu_motion *m, int32_t local_flags, uint64_t local_nullmask,
									const int64_t *dev_sent_counts, int64_t *sent_counts, cbgpu_rel **recv, int32_t *outcome);
int64_t		cbgpu_motion_direct_bytes(const cbgpu_motion *m);
/* host round trips (stream synchronisations) and NCCL collectives spent inside Motions so far: what the
 * device-side signalling is there to keep small (bench.py reports them per step) */
int64_t		cbgpu_motion_host_syncs(const cbgpu_motion *m);
int64_t		cbgpu_motion_collectives(const cbgpu_motion *m);
/* the windows as arenas of the host packet channels (include/cb_chan.h: what the MotionIPCLayer implementation
 * integration/cbgpu_ic_layer.c moves tuple chunks with): fills the channel's memory accessors; the arena (zero-filled at
 * create time) is arena_bytes of every rank's window */
struct CbChanMem;
int			cbgpu_motion_chan_mem(cbgpu_motion *m, struct CbChanMem *mem, size_t *arena_bytes);
/* Gather: the first nrows rows of every rank's `send` to rank `root` (others receive 0 rows) */
int			cbgpu_motion_gather(cbgpu_motion *m, int root, cbgpu_rel *send, int64_t nrows, cbgpu_rel **recv);
/* Broadcast: every rank receives every rank's first nrows rows */
int			cbgpu_motion_broadcast(cbgpu_motion *m, cbgpu_rel *send, int64_t nrows, cbgpu_rel **recv);

/* ------------------------------------------------------------------------------------------
 * AOCS column files decoded on the device (the storage side of aocs_getnext, access/aocs/aocsam.c:1418:
 * datumstreamread_block utils/datumstream/datumstream.c:1364, AppendOnlyStorageRead_GetBlockInfo
 * cdb/cdbappendonlystorageread.c:954, DatumStreamBlockRead_GetReadyOrig / _AdvanceOrig / _Get
 * utils/datumstream/datumstreamblock.c:153, include/utils/datumstreamblock.h:1442,1220)
 * ------------------------------------------------------------------------------------------ */
#define CBGPU_AOCS_VAR_NUMERIC 1	/* numeric varlena -> int64 scaled by the column's dscale             */
#define CBGPU_AOCS_VAR_BPCHAR1 2	/* character(1) varlena -> its byte                                   */
#define CBGPU_AOCS_VAR_DICT 3		/* bpchar(n) / varchar / text -> dictionary code (cbgpu_dict, below)   */
#define CBGPU_AOCS_COMPRESS_NONE 0	/* compresstype=none, or rle_type with compresslevel 1                */
#define CBGPU_AOCS_COMPRESS_ZLIB 1	/* compresstype=zlib (any level), or rle_type with compresslevel 2-4   */
#define CBGPU_AOCS_COMPRESS_ZSTD 2	/* compresstype=zstd (any level)                                       */
/* file_bytes: one column's segment file (<relfilenode>.<n>) as it lies on disk, in host memory:
 * SmallContent / NonBulkDenseContent / BulkDenseContent storage blocks holding Original or Dense (RLE, delta)
 * datum stream blocks.  attlen = pg_type typlen (1/2/4/8, or -1 with varkind), typalign in bytes.  Decodes into
 * rows [row_offset, +nrows) of column `col` (NULL bitmaps become the column's null map).  With checksum != 0 every
 * block's header and block CRC-32C are verified on the device first (CBGPU_ERR_CORRUPT), as the reference does on
 * read (AppendOnlyStorageFormat_VerifyHeaderChecksum / _VerifyBlockChecksum).  LargeContent blocks:
 * CBGPU_ERR_UNSUPPORTED.  Bulk-compressed blocks need the _ex entry point with the column's compresstype. */
int			cbgpu_aocs_decode_column(cbgpu_ctx *ctx, const void *file_bytes, int64_t nbytes, int32_t checksum,
									 int32_t attlen, int32_t varkind, int32_t typalign, cbgpu_rel *rel, int32_t col,
									 int64_t row_offset, int64_t *nrows);
/* The same for a column stored with bulk compression (pg_attribute_encoding compresstype; gp_decompress,
 * cdb/cdbappendonlystorageread.c:1286-1310): blocks whose header carries a compressed length are inflated on the
 * device (zlib streams as catalog/pg_compression.c:272 writes them with compress2(), Zstandard frames as
 * gpcontrib/zstd/zstd_compression.c:104 writes them with ZSTD_compressCCtx()); a bad stream, a wrong Adler-32 /
 * XXH64 or a length other than the header's is CBGPU_ERR_CORRUPT.  quicklz: CBGPU_ERR_UNSUPPORTED. */
int			cbgpu_aocs_decode_column_ex(cbgpu_ctx *ctx, const void *file_bytes, int64_t nbytes, int32_t checksum,
										int32_t compresstype, int32_t attlen, int32_t varkind, int32_t typalign,
										cbgpu_rel *rel, int32_t col, int64_t row_offset, int64_t *nrows);

/* Dictionary of a bpchar(n) / varchar / text column (DESIGN.md data layout: CB_DICT8 / CB_DICT32 codes + per-code
 * hashbpchar).  Built on the device from the column's own files in two passes:
 *   cbgpu_aocs_dict_collect   every segment file of the column: its distinct strings join the set
 *   cbgpu_dict_finalize       codes 0 .. n-1 in byte-wise (memcmp, shorter first on ties) order of the strings
 *   cbgpu_aocs_decode_dict_column   every segment file again: rows become codes; the relation column gets the
 *                             dictionary's per-code hashes (hashbpchar for bpchar: trailing blanks do not count,
 *                             utils/adt/varchar.c:981; hashtext / hash_any of the bytes otherwise)
 * One dictionary can serve several columns / relations (join keys must share one).  bpchar != 0: bpchar semantics,
 * values are compared and kept without their trailing blanks (bpchareq, bcTruelen). */
typedef struct cbgpu_dict cbgpu_dict;
int			cbgpu_dict_create(cbgpu_ctx *ctx, int32_t max_entries, int64_t arena_bytes, int32_t bpchar, cbgpu_dict **out);
void		cbgpu_dict_free(cbgpu_dict *d);
int			cbgpu_aocs_dict_collect(cbgpu_ctx *ctx, const void *file_bytes, int64_t nbytes, int32_t checksum, int32_t compresstype,
									int32_t typalign, cbgpu_dict *dict);
int			cbgpu_dict_finalize(cbgpu_dict *d, int32_t *nentries);
/* entry `code` of a finalized dictionary: *text points at len bytes owned by the dictionary (no terminator) */
int			cbgpu_dict_entry(const cbgpu_dict *d, int32_t code, const char **text, int32_t *len);
/* code of a string (e.g. a Const of the plan), -1 when the column never holds it */
int32_t		cbgpu_dict_lookup(const cbgpu_dict *d, const char *text, int32_t len);
int			cbgpu_aocs_decode_dict_column(cbgpu_ctx *ctx, const void *file_bytes, int64_t nbytes, int32_t checksum,
										  int32_t compresstype, int32_t typalign, const cbgpu_dict *dict, cbgpu_rel *rel,
										  int32_t col, int64_t row_offset, int64_t *nrows);

/* One row of the table's pg_aovisimap_<oid> for the segment file being loaded (access/appendonly/appendonly_visimap_entry.c:
 * AppendOnlyVisimapEntry_Copyout :196-262): first_row_no, and the detoasted `visimap` value after its varlena length
 * word (int32 version + Bitmap_Compress output); data NULL = SQL NULL = every row of the range visible. */
typedef struct cbgpu_visimap_entry
{
	int64_t		first_row_num;
	const void *data;
	int32_t		len;
} cbgpu_visimap_entry;
/* Visibility of the rows of one segment file (AppendOnlyVisimap_IsVisible, access/appendonly/appendonly_visimap.c:198):
 * file_bytes = any one column's file of that segment file (only block headers are read: row numbers run
 * firstRowNum, firstRowNum + 1, ... within a block); entries = the pg_aovisimap rows of that segno, any order.
 * Writes rows [row_offset, +rows of the file) of the relation's visibility bitmap (1 = visible; rows outside keep
 * their state, a relation without a bitmap starts all visible); *nhidden = rows hidden.  The entries are expanded
 * and looked up on the device; a malformed entry is CBGPU_ERR_CORRUPT. */
int			cbgpu_aocs_apply_visimap(cbgpu_ctx *ctx, const void *file_bytes, int64_t nbytes, int32_t checksum,
									 const cbgpu_visimap_entry *entries, int32_t nentries, cbgpu_rel *rel,
									 int64_t row_offset, int64_t *nhidden);

/* ------------------------------------------------------------------------------------------
 * synthetic TPC-H shaped generator (harness; same counter-based formulas as
 * cloudberry_b200/tpch.py so host and device tables are identical)
 * ------------------------------------------------------------------------------------------ */
int			cbgpu_gen_lineitem(cbgpu_ctx *ctx, cbgpu_rel *rel, uint64_t seed, int64_t row_lo,
							   int64_t n_supp, int64_t n_part);
int			cbgpu_gen_orders(cbgpu_ctx *ctx, cbgpu_rel *rel, uint64_t seed, int64_t row_lo, int64_t n_cust);
int			cbgpu_gen_customer(cbgpu_ctx *ctx, cbgpu_rel *rel, uint64_t seed);
int			cbgpu_gen_supplier(cbgpu_ctx *ctx, cbgpu_rel *rel, uint64_t seed);
/* rows [row_lo, row_lo + nrows) of the same tables: every rank generates its slice before the
 * load-time Redistribute that implements DISTRIBUTED BY */
int			cbgpu_gen_customer_range(cbgpu_ctx *ctx, cbgpu_rel *rel, uint64_t seed, int64_t row_lo);
int			cbgpu_gen_supplier_range(cbgpu_ctx *ctx, cbgpu_rel *rel, uint64_t seed, int64_t row_lo);
/* Star Schema Benchmark fact table, rows [row_lo, row_lo + nrows) of cloudberry_b200/ssb.py's lineorder
 * (lo_custkey, lo_partkey, lo_suppkey, lo_orderdate, lo_revenue, lo_supplycost) */
int			cbgpu_gen_ssb_lineorder(cbgpu_ctx *ctx, cbgpu_rel *rel, uint64_t seed, int64_t row_lo, int64_t n_cust,
									int64_t n_part, int64_t n_supp);

#ifdef __cplusplus
}
#endif
#endif							/* CBGPU_H */
