/*
 * cb_exec.c - host executor: ExecInitNode / ExecProcNode / ExecEndNode over the CUDA C ABI.
 *
 * Plain C, like the code it stands in for.  The reference walks the PlanState tree once per tuple
 * (ExecProcNode, backend/executor/execProcnode.c:580-681); this executor walks it once per query:
 * each node describes its output symbolically (a CbStream: driving relation + postfix program +
 * output expressions), parents append their own quals / probes / aggregate arguments, and the
 * first pipeline breaker above (Hash build, Agg, Motion, Limit/Sort, or the top of the plan) runs
 * the whole chain as one fused kernel (cbgpu_pipeline_run).  Only post-aggregation rows are then
 * handed out one slot per ExecProcNode call.
 *
 * Reference functions restated here, node by node:
 *   SeqScan   ExecInitSeqScan / SeqNext            backend/executor/nodeSeqscan.c:58,149
 *             column projection                    backend/access/aocs/aocsam_handler.c:612-634
 *   Hash      MultiExecHash                        backend/executor/nodeHash.c:130
 *   HashJoin  ExecInitHashJoin / ExecHashJoinImpl  backend/executor/nodeHashjoin.c:203,747
 *   Agg       ExecInitAgg / agg_fill_hash_table / agg_retrieve_hash_table / finalize_aggregates
 *                                                  backend/executor/nodeAgg.c:2726,2952
 *             ExecBuildAggTrans (shared transition states)  backend/executor/execExpr.c:3573
 *   Motion    ExecMotion / execMotionSender / execMotionUnsortedReceiver
 *                                                  backend/executor/nodeMotion.c:100,203,307
 */
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../../include/cb_exec.h"

/* ------------------------------------------------------------------------------------------
 * errors
 * ------------------------------------------------------------------------------------------ */
static int
es_fail(CbEState *es, int code, const char *fmt,...)
{
	va_list		ap;

	if (es->es_errcode == 0)
	{
		va_start(ap, fmt);
		vsnprintf(es->es_errmsg, sizeof(es->es_errmsg), fmt, ap);
		va_end(ap);
		es->es_errcode = code;
		if (es->es_error_hook)
			es->es_error_hook(es, code, es->es_errmsg);
	}
	return code;
}

/* wrap a cbgpu_* status */
#define GPU(es, call) \
	do { \
		int rc__ = (call); \
		if (rc__ != CBGPU_OK) \
			return es_fail((es), rc__, "%s", cbgpu_last_error((es)->es_ctx)); \
	} while (0)

#define TRY(call) \
	do { \
		int rc__ = (call); \
		if (rc__ != CBGPU_OK) \
			return rc__; \
	} while (0)

const char *
cb_estate_error(CbEState *estate)
{
	return estate->es_errmsg;
}

/* ------------------------------------------------------------------------------------------
 * streams: the symbolic output of a node
 * ------------------------------------------------------------------------------------------ */
typedef enum PKind { PE_COL = 1, PE_CONST, PE_OP, PE_STATE } PKind;

typedef struct PExpr
{
	int			kind;
	int			type;			/* CbTypeId                                                          */
	int			dscale;
	int			maybe_null;
	int			col;			/* PE_COL: index in pipe.cols                                        */
	int64_t		imm;			/* PE_CONST                                                          */
	int			op;				/* PE_OP: CbpOpCode; l / r children (r = -1 for unary)               */
	int			l, r;
	/* PE_STATE: an aggregate transition state carried as columns (N, sum.lo, sum.hi) */
	int			cn, clo, chi;	/* PE ids                                                            */
	int			acckind;		/* CbpAggKind of the state (COUNT / SUM_INT / SUM_FLOAT / MIN / MAX) */
	int			aggfn;			/* CbAggFn that produced it                                          */
	int			final;			/* finalise when drained (SIMPLE / FINAL agg output)                 */
	int			argtype;		/* input type of the aggregate                                       */
	int			restype;
} PExpr;

#define MAX_PE 768
#define MAX_OUT 64
#define MAX_OWNED 64

typedef struct CbStream
{
	CbPipeline	pipe;			/* cols, ops (quals / probes so far), probes; no sink yet            */
	cbgpu_rel  *col_rel[CBP_MAX_COLS];	/* relation each column belongs to (for bookkeeping)         */
	int			col_idx[CBP_MAX_COLS];
	PExpr		pe[MAX_PE];
	int			npe;
	int			out[MAX_OUT];
	int			nout;
	int			nsrc;			/* sources in use                                                    */
	int64_t		rows_in;
} CbStream;

typedef struct Owned
{
	cbgpu_rel  *rels[MAX_OWNED];
	int			nrels;
	cbgpu_hashtable *hts[MAX_OWNED];
	int			nhts;
	cbgpu_aggtable *aggs[MAX_OWNED];
	int			naggs;
	void	   *devs[MAX_OWNED];
	int			ndevs;
	cbgpu_pairs pairs[8];
	int			npairs;
	CbStream   *streams[8];
	int			nstreams;
} Owned;

static void
owned_free(CbEState *es, Owned *o)
{
	for (int i = 0; i < o->nrels; i++)
		cbgpu_rel_free(o->rels[i]);
	for (int i = 0; i < o->nhts; i++)
		cbgpu_ht_free(o->hts[i]);
	for (int i = 0; i < o->naggs; i++)
		cbgpu_agg_free(o->aggs[i]);
	for (int i = 0; i < o->ndevs; i++)
		cbgpu_dev_free(es->es_ctx, o->devs[i]);
	for (int i = 0; i < o->npairs; i++)
		cbgpu_pairs_free(&o->pairs[i]);
	for (int i = 0; i < o->nstreams; i++)
		free(o->streams[i]);
	memset(o, 0, sizeof(*o));
}

/* result rows on the host */
typedef struct ResultSet
{
	int64_t		nrows;
	int			ncols;
	int		   *types;
	int64_t    *vals;			/* nrows x ncols                                                     */
	uint8_t    *nulls;
	int64_t    *st_n, *st_lo, *st_hi;
	CbNumericDatum *nums;		/* nrows x ncols (only numeric columns used)                         */
	int64_t		cursor;
} ResultSet;

static void
rs_free(ResultSet *rs)
{
	if (!rs)
		return;
	free(rs->types);
	free(rs->vals);
	free(rs->nulls);
	free(rs->st_n);
	free(rs->st_lo);
	free(rs->st_hi);
	free(rs->nums);
	free(rs);
}

static ResultSet *
rs_new(int64_t nrows, int ncols)
{
	ResultSet  *rs = calloc(1, sizeof(ResultSet));
	size_t		n = (size_t) (nrows ? nrows : 1) * (size_t) (ncols ? ncols : 1);

	rs->nrows = nrows;
	rs->ncols = ncols;
	rs->types = calloc((size_t) (ncols ? ncols : 1), sizeof(int));
	rs->vals = calloc(n, sizeof(int64_t));
	rs->nulls = calloc(n, 1);
	rs->st_n = calloc(n, sizeof(int64_t));
	rs->st_lo = calloc(n, sizeof(int64_t));
	rs->st_hi = calloc(n, sizeof(int64_t));
	rs->nums = calloc(n, sizeof(CbNumericDatum));
	return rs;
}

/* node-private state, common to all node types */
typedef struct NodePriv
{
	Owned		owned;
	CbStream   *stream;			/* this node's output stream once opened                             */
	int			opened;
	ResultSet  *rs;
	/* Hash */
	cbgpu_hashtable *ht;
	cbgpu_rel  *inner_rel;
	int			inner_map[MAX_OUT];	/* Hash child output column -> column of inner_rel (first of 3 for states) */
	PExpr		inner_pe[MAX_OUT];	/* metadata of each Hash child output (type, state info)         */
	int			inner_nout;
	/* Motion (local interconnect): received rows deposited by the cluster */
	cbgpu_rel  *recv;
	int			recv_ready;
	int			xstage;			/* 0: no exchange of this Motion yet; 1: its direct attempt is over (peers now
								 * expect the staged one); 2: delivered                               */
	PExpr		send_pe[MAX_OUT];
	int			send_nout;
} NodePriv;

static NodePriv *
np(CbPlanState *ps)
{
	return (NodePriv *) ps->priv;
}

/* ---- PExpr construction with structural sharing ---- */
static int
pe_add(CbStream *s, const PExpr *e)
{
	for (int i = 0; i < s->npe; i++)
	{
		const PExpr *o = &s->pe[i];

		if (o->kind != e->kind || o->type != e->type || o->dscale != e->dscale)
			continue;
		if (e->kind == PE_COL && o->col == e->col)
			return i;
		if (e->kind == PE_CONST && o->imm == e->imm)
			return i;
		if (e->kind == PE_OP && o->op == e->op && o->l == e->l && o->r == e->r && o->imm == e->imm)
			return i;
		if (e->kind == PE_STATE && o->cn == e->cn && o->clo == e->clo && o->chi == e->chi && o->acckind == e->acckind &&
			o->aggfn == e->aggfn && o->final == e->final)
			return i;
	}
	if (s->npe >= MAX_PE)
		return -1;
	s->pe[s->npe] = *e;
	return s->npe++;
}

static int
stream_add_col(CbStream *s, cbgpu_rel *rel, int col, int src)
{
	const void *data = cbgpu_rel_col_devptr(rel, col);

	for (int i = 0; i < s->pipe.ncols; i++)
		if (s->pipe.cols[i].data == data && s->pipe.cols[i].src == src)
			return i;
	if (s->pipe.ncols >= CBP_MAX_COLS)
		return -1;
	CbpColumn  *c = &s->pipe.cols[s->pipe.ncols];

	c->data = data;
	c->nulls = cbgpu_rel_nulls_dev(rel, col);
	c->dict_hash = cbgpu_rel_dict_hash_dev(rel, col);
	c->type = cbgpu_rel_col_type(rel, col);
	c->src = src;
	s->col_rel[s->pipe.ncols] = rel;
	s->col_idx[s->pipe.ncols] = col;
	return s->pipe.ncols++;
}

static int
pe_col(CbStream *s, cbgpu_rel *rel, int col, int src, int force_nullable)
{
	PExpr		e;
	int			c = stream_add_col(s, rel, col, src);

	if (c < 0)
		return -1;
	memset(&e, 0, sizeof(e));
	e.kind = PE_COL;
	e.type = cbgpu_rel_col_type(rel, col);
	e.dscale = cbgpu_rel_col_dscale(rel, col);
	e.col = c;
	e.maybe_null = force_nullable || cbgpu_rel_has_nulls(rel, col);
	e.l = e.r = -1;
	return pe_add(s, &e);
}

static int
pe_const(CbStream *s, int type, int dscale, int64_t v)
{
	PExpr		e;

	memset(&e, 0, sizeof(e));
	e.kind = PE_CONST;
	e.type = type;
	e.dscale = dscale;
	e.imm = v;
	e.l = e.r = -1;
	return pe_add(s, &e);
}

static int
pe_op(CbStream *s, int op, int l, int r, int type, int dscale, int64_t imm)
{
	PExpr		e;

	memset(&e, 0, sizeof(e));
	e.kind = PE_OP;
	e.op = op;
	e.l = l;
	e.r = r;
	e.imm = imm;
	e.type = type;
	e.dscale = dscale;
	e.maybe_null = (l >= 0 && s->pe[l].maybe_null) || (r >= 0 && s->pe[r].maybe_null);
	return pe_add(s, &e);
}

static int64_t
ipow10(int k)
{
	int64_t		r = 1;

	while (k-- > 0)
		r *= 10;
	return r;
}

/* bring an integer / numeric expression to display scale `ds` (numeric add/sub/compare align
 * their operands; constants are folded so `1 - l_discount` becomes `100 - l_discount`) */
static int
pe_rescale(CbStream *s, int e, int ds)
{
	PExpr	   *x = &s->pe[e];
	int			diff = ds - x->dscale;

	if (diff <= 0 || x->type == CB_FLOAT8)
		return e;
	if (diff > 18)
		return -1;
	if (x->kind == PE_CONST)
		return pe_const(s, x->type == CB_NUMERIC ? CB_NUMERIC : x->type, ds, x->imm * ipow10(diff));
	{
		int			c = pe_const(s, CB_INT8, 0, ipow10(diff));

		return pe_op(s, CBP_MUL, e, c, x->type, ds, 0);
	}
}

static int
pe_to_float(CbStream *s, int e)
{
	PExpr	   *x = &s->pe[e];

	if (x->type == CB_FLOAT8)
		return e;
	if (x->kind == PE_CONST)
	{
		double		d = (double) x->imm;
		int64_t		bits;

		for (int k = 0; k < x->dscale; k++)
			d /= 10.0;
		memcpy(&bits, &d, 8);
		return pe_const(s, CB_FLOAT8, 0, bits);
	}
	return pe_op(s, CBP_I2F, e, -1, CB_FLOAT8, 0, x->dscale);
}

/* Var resolution context */
typedef struct VarCtx
{
	CbEState   *es;
	CbStream   *s;
	const int  *outer;			/* PE ids of the OUTER child's output columns                        */
	int			nouter;
	const int  *inner;
	int			ninner;
	cbgpu_rel  *scanrel;		/* for scan-level Vars                                               */
	int			scanrelid;
} VarCtx;

static int	translate(VarCtx *vc, const CbExpr *e, int *out);

static int
translate_op(VarCtx *vc, const CbExpr *e, int *out)
{
	CbStream   *s = vc->s;
	int			l,
				r;

	if (e->nargs != 2)
		return es_fail(vc->es, CBGPU_ERR_INVALID, "operator with %d arguments", e->nargs);
	TRY(translate(vc, e->args[0], &l));
	TRY(translate(vc, e->args[1], &r));
	if (s->pe[l].kind == PE_STATE || s->pe[r].kind == PE_STATE)
		return es_fail(vc->es, CBGPU_ERR_UNSUPPORTED, "arithmetic over an aggregate transition state is not supported on the GPU path");
	int			isfloat = s->pe[l].type == CB_FLOAT8 || s->pe[r].type == CB_FLOAT8;

	if (e->op >= CB_OP_EQ)
	{
		int			code;

		if (isfloat)
		{
			l = pe_to_float(s, l);
			r = pe_to_float(s, r);
			code = CBP_FEQ + (e->op - CB_OP_EQ);
		}
		else
		{
			int			ds = s->pe[l].dscale > s->pe[r].dscale ? s->pe[l].dscale : s->pe[r].dscale;

			l = pe_rescale(s, l, ds);
			r = pe_rescale(s, r, ds);
			code = CBP_EQ + (e->op - CB_OP_EQ);
		}
		if (l < 0 || r < 0)
			return es_fail(vc->es, CBGPU_ERR_UNSUPPORTED, "expression too large for the GPU path");
		*out = pe_op(s, code, l, r, CB_BOOL, 0, 0);
	}
	else if (isfloat)
	{
		l = pe_to_float(s, l);
		r = pe_to_float(s, r);
		*out = pe_op(s, e->op == CB_OP_ADD ? CBP_FADD : e->op == CB_OP_SUB ? CBP_FSUB : CBP_FMUL, l, r, CB_FLOAT8, 0, 0);
	}
	else
	{
		int			ds;

		if (e->op == CB_OP_MUL)
			ds = s->pe[l].dscale + s->pe[r].dscale;	/* numeric_mul: rscale = dscale1 + dscale2 */
		else
		{
			ds = s->pe[l].dscale > s->pe[r].dscale ? s->pe[l].dscale : s->pe[r].dscale;
			l = pe_rescale(s, l, ds);
			r = pe_rescale(s, r, ds);
			if (l < 0 || r < 0)
				return es_fail(vc->es, CBGPU_ERR_UNSUPPORTED, "expression too large for the GPU path");
		}
		if (ds != e->dscale && (e->restype == CB_NUMERIC))
			return es_fail(vc->es, CBGPU_ERR_INVALID, "plan says display scale %d, operands give %d", e->dscale, ds);
		*out = pe_op(s, e->op == CB_OP_ADD ? CBP_ADD : e->op == CB_OP_SUB ? CBP_SUB : CBP_MUL, l, r, e->restype, ds, 0);
	}
	if (*out < 0)
		return es_fail(vc->es, CBGPU_ERR_UNSUPPORTED, "expression too large for the GPU path");
	return CBGPU_OK;
}

static int
translate(VarCtx *vc, const CbExpr *e, int *out)
{
	CbStream   *s = vc->s;

	switch (e->tag)
	{
		case T_CbVar:
			if (e->varno == CB_OUTER_VAR)
			{
				if (e->varattno < 1 || e->varattno > vc->nouter)
					return es_fail(vc->es, CBGPU_ERR_INVALID, "OUTER_VAR attno %d out of range", e->varattno);
				*out = vc->outer[e->varattno - 1];
			}
			else if (e->varno == CB_INNER_VAR)
			{
				if (e->varattno < 1 || e->varattno > vc->ninner)
					return es_fail(vc->es, CBGPU_ERR_INVALID, "INNER_VAR attno %d out of range", e->varattno);
				*out = vc->inner[e->varattno - 1];
			}
			else
			{
				if (!vc->scanrel || e->varno != vc->scanrelid || e->varattno < 1 || e->varattno > cbgpu_rel_ncols(vc->scanrel))
					return es_fail(vc->es, CBGPU_ERR_INVALID, "scan Var (%d, %d) does not belong to this scan", e->varno, e->varattno);
				if (cbgpu_rel_col_type(vc->scanrel, e->varattno - 1) != (int) e->restype)
					return es_fail(vc->es, CBGPU_ERR_INVALID, "Var (%d, %d): plan type %d differs from the relation's column type %d",
								   e->varno, e->varattno, e->restype, cbgpu_rel_col_type(vc->scanrel, e->varattno - 1));
				*out = pe_col(s, vc->scanrel, e->varattno - 1, 0, 0);
			}
			if (*out < 0)
				return es_fail(vc->es, CBGPU_ERR_UNSUPPORTED, "too many columns in one pipeline");
			return CBGPU_OK;
		case T_CbConst:
			if (e->constisnull)
				return es_fail(vc->es, CBGPU_ERR_UNSUPPORTED, "NULL constants are not supported on the GPU path");
			*out = pe_const(s, e->restype, e->dscale, e->constval);
			return CBGPU_OK;
		case T_CbOpExpr:
			return translate_op(vc, e, out);
		case T_CbBoolExpr:
			{
				int			acc = -1;

				if (e->op == CB_NOT_EXPR)
				{
					int			a;

					TRY(translate(vc, e->args[0], &a));
					*out = pe_op(s, CBP_NOT, a, -1, CB_BOOL, 0, 0);
					return CBGPU_OK;
				}
				for (int i = 0; i < e->nargs; i++)
				{
					int			a;

					TRY(translate(vc, e->args[i], &a));
					acc = acc < 0 ? a : pe_op(s, e->op == CB_AND_EXPR ? CBP_AND : CBP_OR, acc, a, CB_BOOL, 0, 0);
				}
				*out = acc;
				return acc < 0 ? es_fail(vc->es, CBGPU_ERR_INVALID, "empty boolean expression") : CBGPU_OK;
			}
		default:
			return es_fail(vc->es, CBGPU_ERR_UNSUPPORTED, "expression node %d is not supported on the GPU path", e->tag);
	}
}

/* ---- emission: PExpr -> postfix ops ---- */
static int
emit_op(CbEState *es, CbStream *s, int code, int a, int64_t imm)
{
	if (s->pipe.nops >= CBP_MAX_OPS - 1)
		return es_fail(es, CBGPU_ERR_UNSUPPORTED, "pipeline program longer than %d ops", CBP_MAX_OPS);
	s->pipe.ops[s->pipe.nops].code = code;
	s->pipe.ops[s->pipe.nops].a = a;
	s->pipe.ops[s->pipe.nops].imm = imm;
	s->pipe.nops++;
	return CBGPU_OK;
}

static int
emit_expr(CbEState *es, CbStream *s, int e)
{
	PExpr	   *x = &s->pe[e];

	switch (x->kind)
	{
		case PE_COL:
			return emit_op(es, s, CBP_LOAD, x->col, 0);
		case PE_CONST:
			return emit_op(es, s, CBP_CONST, 0, x->imm);
		case PE_OP:
			TRY(emit_expr(es, s, x->l));
			if (x->r >= 0)
				TRY(emit_expr(es, s, x->r));
			return emit_op(es, s, x->op, x->op == CBP_I2F ? (int) x->imm : 0, 0);
		default:
			return es_fail(es, CBGPU_ERR_INVALID, "cannot emit a transition state as a scalar");
	}
}

/* ExecQual: every list member must be true; AND trees split into separate FILTERs */
static int
emit_qual(VarCtx *vc, const CbExpr *q)
{
	int			e;

	if (q->tag == T_CbBoolExpr && q->op == CB_AND_EXPR)
	{
		for (int i = 0; i < q->nargs; i++)
			TRY(emit_qual(vc, q->args[i]));
		return CBGPU_OK;
	}
	TRY(translate(vc, q, &e));
	TRY(emit_expr(vc->es, vc->s, e));
	return emit_op(vc->es, vc->s, CBP_FILTER, 0, 0);
}

static CbStream *
stream_new(NodePriv *p)
{
	CbStream   *s = calloc(1, sizeof(CbStream));

	if (p->owned.nstreams < 8)
		p->owned.streams[p->owned.nstreams++] = s;
	return s;
}

/* identity stream over a relation whose columns follow `shape` (column layout of a materialised
 * stream: one column per scalar output, three per transition state) */
static int
stream_over_rel(CbEState *es, CbStream *s, cbgpu_rel *rel, const PExpr *shape, int nshape)
{
	int			c = 0;

	s->pipe.nrows = cbgpu_rel_nrows(rel);
	s->rows_in = s->pipe.nrows;
	s->nsrc = 1;
	s->nout = nshape;
	for (int i = 0; i < nshape; i++)
	{
		if (shape[i].kind == PE_STATE)
		{
			PExpr		e = shape[i];

			e.cn = pe_col(s, rel, c, 0, 0);
			e.clo = pe_col(s, rel, c + 1, 0, 0);
			e.chi = pe_col(s, rel, c + 2, 0, 0);
			if (e.cn < 0 || e.clo < 0 || e.chi < 0)
				return es_fail(es, CBGPU_ERR_UNSUPPORTED, "too many columns in one pipeline");
			s->out[i] = pe_add(s, &e);
			c += 3;
		}
		else
		{
			s->out[i] = pe_col(s, rel, c, 0, 0);
			if (s->out[i] >= 0)
			{
				/* keep the logical type / scale of the producing expression */
				s->pe[s->out[i]].dscale = shape[i].dscale;
			}
			c += 1;
		}
		if (s->out[i] < 0)
			return es_fail(es, CBGPU_ERR_UNSUPPORTED, "too many columns in one pipeline");
	}
	return CBGPU_OK;
}

/* the caller's interrupt check in the form the device library polls between hash join batches */
static int
es_pending(void *arg)
{
	CbEState   *es = (CbEState *) arg;

	return es->es_interrupt_pending && es->es_interrupt_pending(es);
}

/*
 * Run a pipeline.  When one of its probes is a multi-batch hash join (the build side did not fit the operator's memory,
 * nodeHash.c:980-990) the pipeline runs once per batch, each pass with that batch of the build side resident and the
 * probe rows of other batches skipped (ExecHashJoinImpl's HJ_NEED_NEW_BATCH loop, nodeHashjoin.c:709-738, without the
 * spill files: the outer side is scanned again instead of being written out per batch - HBM bandwidth is cheaper than a
 * temp file).  The sink accumulates over the passes: aggregates add up, materialised rows append, partitions fill on.
 */
static int
run_pipeline(CbEState *es, CbPipeline *pl)
{
	int			multi[CBP_MAX_SRC],
				at[CBP_MAX_SRC];
	int			nmulti = 0;
	int64_t		passes = 1;

	for (int j = 0; j < pl->nprobes; j++)
		if (pl->probes[j].ht && cbgpu_ht_nbatch(pl->probes[j].ht) > 1)
		{
			multi[nmulti] = j;
			at[nmulti++] = 0;
			passes *= cbgpu_ht_nbatch(pl->probes[j].ht);
		}
	if (nmulti == 0)
	{
		GPU(es, cbgpu_pipeline_run(es->es_ctx, pl));
		return CBGPU_OK;
	}
	/* several multi-batch joins in one pipeline: a row reaches the sink in the one pass whose batch combination holds all
	 * its partners (the reference's joins each re-read their own spilled batches; stacked here, the passes multiply) */
	if (passes > 65536)
		return es_fail(es, CBGPU_ERR_UNSUPPORTED, "%s%lld passes over the outer side for the multi-batch hash joins of one pipeline (raise the operator memory)", "", (long long) passes);
	for (int k = 0; k < nmulti; k++)
		GPU(es, cbgpu_ht_load_batch((cbgpu_hashtable *) pl->probes[multi[k]].ht, 0));
	for (;;)
	{
		int			k;

		if (es->es_interrupt_pending && es->es_interrupt_pending(es))
			return es_fail(es, CBGPU_ERR_INTERRUPTED, "canceling statement due to user request");
		GPU(es, cbgpu_pipeline_run(es->es_ctx, pl));
		es->es_hashjoin_batches_run++;
		/* next combination: the LAST join's batch changes fastest (its table is usually the smallest to reload) */
		for (k = nmulti - 1; k >= 0; k--)
		{
			if (++at[k] < cbgpu_ht_nbatch(pl->probes[multi[k]].ht))
			{
				GPU(es, cbgpu_ht_load_batch((cbgpu_hashtable *) pl->probes[multi[k]].ht, at[k]));
				break;
			}
			at[k] = 0;
			GPU(es, cbgpu_ht_load_batch((cbgpu_hashtable *) pl->probes[multi[k]].ht, 0));
		}
		if (k < 0)
			break;
	}
	return CBGPU_OK;
}

static int	stream_materialize_ex(CbEState *es, CbPlanState *ps, CbStream *s, Owned *own, cbgpu_rel **out, PExpr *shape, int *nshape,
								  int borrow);
static int	stream_is_plain(const CbStream *s, cbgpu_rel **rel, const uint32_t **sel);

/* the stream's rows as a relation: a new one (MATERIALIZE sink) or, when the stream is a relation already, that one */
static int
stream_materialize(CbEState *es, CbPlanState *ps, CbStream *s, Owned *own, cbgpu_rel **out, PExpr *shape, int *nshape)
{
	return stream_materialize_ex(es, ps, s, own, out, shape, nshape, 1);
}

/* is rel one of the executor's base tables?  (those are never handed out as somebody's result: a consumer may free or
 * re-shape what it is given) */
static int
cbgpu_rel_is_base(const CbEState *es, const cbgpu_rel *rel)
{
	for (int i = 0; i < es->es_nrels; i++)
		if (es->es_range_table[i] == rel)
			return 1;
	return 0;
}

/* run the stream into a new relation (MATERIALIZE sink); columns laid out as stream_over_rel expects */
static int
stream_materialize_ex(CbEState *es, CbPlanState *ps, CbStream *s, Owned *own, cbgpu_rel **out, PExpr *shape, int *nshape, int borrow)
{
	int32_t		types[CBP_MAX_OUT],
				dscales[CBP_MAX_OUT];
	int			ncols = 0;
	int			nullable[CBP_MAX_OUT];
	cbgpu_rel  *rel;
	void	   *counter;
	int64_t		count = 0;
	CbPipeline *p = &s->pipe;
	int			saved_nops = p->nops;

	if (borrow && stream_is_plain(s, &rel, NULL))
	{
		/* the stream already IS a relation with exactly these columns (an aggregate's group relation, a Motion's receive
		 * buffer): hand it over instead of copying it through a kernel.  The caller does not own it - its producer does. */
		int			exact = 1,
					c = 0;

		for (int i = 0; i < s->nout && exact; i++)
		{
			PExpr	   *x = &s->pe[s->out[i]];

			shape[i] = *x;
			if (x->kind == PE_STATE)
			{
				if (s->pe[x->cn].kind != PE_COL || s->col_idx[s->pe[x->cn].col] != c || s->pe[x->clo].kind != PE_COL ||
					s->col_idx[s->pe[x->clo].col] != c + 1 || s->pe[x->chi].kind != PE_COL || s->col_idx[s->pe[x->chi].col] != c + 2)
					exact = 0;
				c += 3;
			}
			else
			{
				if (x->kind != PE_COL || s->col_idx[x->col] != c)
					exact = 0;
				c++;
			}
		}
		if (exact && c == cbgpu_rel_ncols(rel) && !cbgpu_rel_is_base(es, rel) && borrow == 2)
		{
			/* the caller takes the relation over: only if it is this node's own */
			exact = 0;
			for (int i = 0; i < own->nrels; i++)
				if (own->rels[i] == rel)
					exact = 1;
		}
		if (exact && c == cbgpu_rel_ncols(rel) && !cbgpu_rel_is_base(es, rel))
		{
			*nshape = s->nout;
			*out = rel;
			return CBGPU_OK;
		}
	}
	for (int i = 0; i < s->nout; i++)
	{
		PExpr	   *x = &s->pe[s->out[i]];

		shape[i] = *x;
		if (x->kind == PE_STATE)
		{
			if (ncols + 3 > CBP_MAX_OUT)
				return es_fail(es, CBGPU_ERR_UNSUPPORTED, "too many output columns for one pipeline");
			for (int k = 0; k < 3; k++)
			{
				types[ncols] = CB_INT8;
				dscales[ncols] = 0;
				nullable[ncols] = 0;
				ncols++;
			}
			TRY(emit_expr(es, s, x->cn));
			TRY(emit_expr(es, s, x->clo));
			TRY(emit_expr(es, s, x->chi));
		}
		else
		{
			if (ncols + 1 > CBP_MAX_OUT)
				return es_fail(es, CBGPU_ERR_UNSUPPORTED, "too many output columns for one pipeline");
			types[ncols] = x->type == CB_BOOL ? CB_BOOL : x->type;
			dscales[ncols] = x->dscale;
			nullable[ncols] = x->maybe_null;
			ncols++;
			TRY(emit_expr(es, s, s->out[i]));
		}
	}
	*nshape = s->nout;
	TRY(emit_op(es, s, CBP_END, 0, 0));
	GPU(es, cbgpu_rel_create(es->es_ctx, p->nrows, ncols, types, dscales, &rel));
	own->rels[own->nrels++] = rel;
	for (int c = 0; c < ncols; c++)
		if (nullable[c])
			GPU(es, cbgpu_rel_add_nullmap(rel, c));
	/* dictionary columns keep their per-code hashes so they stay usable as hash keys */
	{
		int			c = 0;

		for (int i = 0; i < s->nout; i++)
		{
			PExpr	   *x = &s->pe[s->out[i]];

			if (x->kind == PE_STATE)
			{
				c += 3;
				continue;
			}
			if (x->kind == PE_COL && (x->type == CB_DICT8 || x->type == CB_DICT32) && p->cols[x->col].dict_hash)
				GPU(es, cbgpu_rel_share_dict_hash(rel, c, s->col_rel[x->col], s->col_idx[x->col]));
			c++;
		}
	}
	GPU(es, cbgpu_dev_alloc(es->es_ctx, sizeof(int64_t), &counter));
	own->devs[own->ndevs++] = counter;
	memset(&p->sink, 0, sizeof(p->sink));
	p->sink.kind = CBP_SINK_MATERIALIZE;
	p->sink.nout = ncols;
	p->sink.out = rel;
	p->sink.out_count = (int64_t *) counter;
	p->force_generic = es->es_force_generic;
	{
		int64_t		before = cbgpu_kernel_launches(es->es_ctx);

		TRY(run_pipeline(es, p));
		GPU(es, cbgpu_dev_read(es->es_ctx, counter, sizeof(int64_t), &count));	/* the status word rides along */
		GPU(es, cbgpu_check_status(es->es_ctx));
		ps->instrument.kernels += cbgpu_kernel_launches(es->es_ctx) - before;
		ps->instrument.rows_in += s->rows_in;
		if (cbgpu_last_kernel_ms(es->es_ctx) > 0)
			ps->instrument.device_ms += cbgpu_last_kernel_ms(es->es_ctx);
	}
	GPU(es, cbgpu_rel_set_nrows(rel, count));
	p->nops = saved_nops;		/* the stream itself stays reusable */
	*out = rel;
	return CBGPU_OK;
}

/* does the stream just expose the columns of one relation, untouched? */
static int
stream_is_plain(const CbStream *s, cbgpu_rel **rel, const uint32_t **sel)
{
	cbgpu_rel  *r = NULL;

	if (s->pipe.nops != 0 || s->pipe.nprobes != 0 || s->pipe.visimap)
		return 0;
	/* an ordered selection over the relation (merge receive) is plain too when the caller can take it (sel != NULL) */
	if (s->pipe.drv_nsrc != 0 && !(sel && s->pipe.drv_nsrc == 1 && s->pipe.drv_idx[0]))
		return 0;
	if (sel)
		*sel = s->pipe.drv_nsrc == 1 ? s->pipe.drv_idx[0] : NULL;
	for (int i = 0; i < s->pipe.ncols; i++)
	{
		if (s->pipe.cols[i].src != 0)
			return 0;
		if (r && s->col_rel[i] != r)
			return 0;
		r = s->col_rel[i];
	}
	if (!r || (cbgpu_rel_nrows(r) != s->pipe.nrows && !(sel && *sel)))
		return 0;
	*rel = r;
	return 1;
}

/* ------------------------------------------------------------------------------------------
 * node_open: build (and, at pipeline breakers, run) a node's output stream
 * ------------------------------------------------------------------------------------------ */
static int	node_open(CbPlanState *ps, CbStream **out);
static int	node_open_inner(CbPlanState *ps, CbStream **out);
static const char *node_name(CbNodeTag t);
static int	cluster_run_motion(CbPlanState *ps);
static int	open_limitsort(CbPlanState *ps, CbStream **out);
static int	sort_key_columns(CbEState *es, const PExpr *shape, int nshape, int lead, const CbSortKey *keys, int nkeys, int32_t *keycols,
							 int32_t *desc, int32_t *uns, int *nk_out);

static int
open_seqscan(CbPlanState *ps, CbStream **out)
{
	CbEState   *es = ps->state;
	CbSeqScan  *scan = (CbSeqScan *) ps->plan;
	CbStream   *s = stream_new(np(ps));
	cbgpu_rel  *rel;
	VarCtx		vc;

	if (scan->scanrelid < 1 || scan->scanrelid > es->es_nrels || !es->es_range_table[scan->scanrelid - 1])
		return es_fail(es, CBGPU_ERR_INVALID, "scanrelid %d is not in the range table", scan->scanrelid);
	rel = es->es_range_table[scan->scanrelid - 1];
	s->pipe.nrows = cbgpu_rel_nrows(rel);
	s->pipe.visimap = cbgpu_rel_visimap_dev(rel);
	s->rows_in = s->pipe.nrows;
	s->nsrc = 1;
	memset(&vc, 0, sizeof(vc));
	vc.es = es;
	vc.s = s;
	vc.scanrel = rel;
	vc.scanrelid = scan->scanrelid;
	/* quals first (the AM evaluates pushed-down quals before fetching the remaining columns,
	 * aocs_getnext_withqual, aocsam.c:1269): late materialisation falls out of program order */
	for (int i = 0; i < ps->plan->nquals; i++)
		TRY(emit_qual(&vc, ps->plan->qual[i]));
	if (ps->plan->ntargets > MAX_OUT)
		return es_fail(es, CBGPU_ERR_UNSUPPORTED, "more than %d output columns", MAX_OUT);
	s->nout = ps->plan->ntargets;
	for (int i = 0; i < ps->plan->ntargets; i++)
		TRY(translate(&vc, ps->plan->targetlist[i].expr, &s->out[i]));
	*out = s;
	return CBGPU_OK;
}

/* MultiExecHash: materialise the inner side and build the table */
static int
hash_build(CbPlanState *hashps)
{
	CbEState   *es = hashps->state;
	CbHash	   *h = (CbHash *) hashps->plan;
	NodePriv   *p = np(hashps);
	CbStream   *is;
	cbgpu_rel  *rel = NULL;
	int32_t		keycols[CBP_MAX_KEYS];
	int64_t		before = cbgpu_kernel_launches(es->es_ctx);

	if (p->ht)
		return CBGPU_OK;
	TRY(node_open(hashps->lefttree, &is));
	if (h->nhashkeys < 1 || h->nhashkeys > CBP_MAX_KEYS)
		return es_fail(es, CBGPU_ERR_UNSUPPORTED, "hash join with %d keys is beyond the GPU path's limit", h->nhashkeys);
	p->inner_nout = is->nout;
	if (stream_is_plain(is, &rel, NULL))
	{
		/* a bare scan without quals: build straight over the base relation's columns */
		for (int i = 0; i < is->nout; i++)
		{
			PExpr	   *x = &is->pe[is->out[i]];

			if (x->kind != PE_COL)
			{
				rel = NULL;
				break;
			}
			p->inner_map[i] = is->col_idx[x->col];
			p->inner_pe[i] = *x;
		}
	}
	if (!rel)
	{
		int			n,
					c = 0;

		TRY(stream_materialize(es, hashps, is, &p->owned, &rel, p->inner_pe, &n));
		for (int i = 0; i < n; i++)
		{
			p->inner_map[i] = c;
			c += p->inner_pe[i].kind == PE_STATE ? 3 : 1;
		}
	}
	for (int k = 0; k < h->nhashkeys; k++)
	{
		const CbExpr *ke = h->hashkeys[k];

		if (ke->tag != T_CbVar || ke->varno != CB_OUTER_VAR || ke->varattno < 1 || ke->varattno > is->nout ||
			p->inner_pe[ke->varattno - 1].kind == PE_STATE)
			return es_fail(es, CBGPU_ERR_UNSUPPORTED, "hash keys must be plain columns of the Hash node's child on the GPU path");
		keycols[k] = p->inner_map[ke->varattno - 1];
	}
	{
		/* ExecChooseHashTableSize (nodeHash.c:856): one batch if the table fits the operator's memory, else the smallest
		 * power of two of batches that does */
		int32_t		nbatch = 1;
		const int64_t budget = es->es_operator_mem_kb > 0 ? es->es_operator_mem_kb * 1024 : 0;

		while (budget > 0 && nbatch < 4096 && cbgpu_ht_bytes_for((cbgpu_rel_nrows(rel) + nbatch - 1) / nbatch) > budget)
			nbatch <<= 1;
		if (nbatch > 1)
			GPU(es, cbgpu_ht_build_batched(es->es_ctx, rel, keycols, h->nhashkeys, nbatch, &p->ht));
		else
			GPU(es, cbgpu_ht_build(es->es_ctx, rel, keycols, h->nhashkeys, &p->ht));
		hashps->instrument.hashjoin_nbatch = nbatch;
	}
	p->owned.hts[p->owned.nhts++] = p->ht;
	p->inner_rel = rel;
	hashps->instrument.kernels += cbgpu_kernel_launches(es->es_ctx) - before;
	hashps->instrument.ntuples = (double) cbgpu_ht_nrows(p->ht);
	return CBGPU_OK;
}

static int
inner_out_exprs(CbEState *es, CbStream *s, NodePriv *hp, int src, int nullable, int *inner)
{
	for (int i = 0; i < hp->inner_nout; i++)
	{
		if (hp->inner_pe[i].kind == PE_STATE)
		{
			PExpr		e = hp->inner_pe[i];

			e.cn = pe_col(s, hp->inner_rel, hp->inner_map[i], src, nullable);
			e.clo = pe_col(s, hp->inner_rel, hp->inner_map[i] + 1, src, nullable);
			e.chi = pe_col(s, hp->inner_rel, hp->inner_map[i] + 2, src, nullable);
			inner[i] = pe_add(s, &e);
		}
		else
		{
			inner[i] = pe_col(s, hp->inner_rel, hp->inner_map[i], src, nullable);
			if (inner[i] >= 0)
				s->pe[inner[i]].dscale = hp->inner_pe[i].dscale;
		}
		if (inner[i] < 0)
			return es_fail(es, CBGPU_ERR_UNSUPPORTED, "too many columns in one pipeline");
	}
	return CBGPU_OK;
}

static int
open_hashjoin(CbPlanState *ps, CbStream **out)
{
	CbEState   *es = ps->state;
	CbHashJoin *hj = (CbHashJoin *) ps->plan;
	CbPlanState *hashps = ps->righttree;
	NodePriv   *hp;
	CbStream   *s;
	VarCtx		vc;
	int			keys[CBP_MAX_KEYS];
	int			inner[MAX_OUT];
	int			outer[MAX_OUT];
	int			nouter;

	if (!hashps || hashps->type != T_CbHash)
		return es_fail(es, CBGPU_ERR_INVALID, "HashJoin's inner child must be a Hash node");
	hp = np(hashps);
	/* the reference builds the table before pulling the first outer tuple (HJ_BUILD_HASHTABLE,
	 * nodeHashjoin.c:264; prefetch_inner when a Motion sits below, :271-283) */
	TRY(hash_build(hashps));
	TRY(node_open(ps->lefttree, &s));
	if (hj->nhashkeys != ((CbHash *) hashps->plan)->nhashkeys)
		return es_fail(es, CBGPU_ERR_INVALID, "HashJoin / Hash key count mismatch");
	nouter = s->nout;
	memcpy(outer, s->out, sizeof(int) * (size_t) nouter);
	memset(&vc, 0, sizeof(vc));
	vc.es = es;
	vc.s = s;
	vc.outer = outer;
	vc.nouter = nouter;
	for (int k = 0; k < hj->nhashkeys; k++)
	{
		TRY(translate(&vc, hj->hashkeys[k], &keys[k]));
		if (s->pe[keys[k]].kind == PE_STATE)
			return es_fail(es, CBGPU_ERR_UNSUPPORTED, "join key over a transition state");
	}
	if ((cbgpu_ht_has_duplicates(hp->ht) && (hj->jointype == CB_JOIN_INNER || hj->jointype == CB_JOIN_LEFT)) ||
		hj->jointype == CB_JOIN_RIGHT || hj->jointype == CB_JOIN_FULL)
	{
		const int	fill_outer = hj->jointype == CB_JOIN_LEFT || hj->jointype == CB_JOIN_FULL;
		const int	fill_inner = hj->jointype == CB_JOIN_RIGHT || hj->jointype == CB_JOIN_FULL;

		/* N:M join, or a join that returns unmatched build rows: materialise the outer side, emit (outer, inner) row-id
		 * pairs for every match (ExecScanHashBucket walks the whole chain, nodeHash.c:2255) - plus, per join type, one
		 * pair with a missing side for every unmatched row - and continue from the pairs */
		CbStream   *s2;
		cbgpu_rel  *orel;
		PExpr		shape[MAX_OUT + CBP_MAX_KEYS];
		int			nshape;
		int32_t		keycols[CBP_MAX_KEYS];
		cbgpu_pairs *pairs;
		NodePriv   *me = np(ps);
		int			c;

		const int	multi = cbgpu_ht_nbatch(hp->ht) > 1;

		if (multi)
			/* the batched probe loads build batches by key hash: the same key checks as the pipelined probe below */
			for (int k = 0; k < hj->nhashkeys; k++)
			{
				PExpr	   *kx = &s->pe[keys[k]];

				if (kx->type == CB_FLOAT8)
					return es_fail(es, CBGPU_ERR_UNSUPPORTED, "float8 join keys are not on the GPU path");
				if ((kx->type == CB_DICT8 || kx->type == CB_DICT32) &&
					(kx->kind != PE_COL || !s->pipe.cols[kx->col].dict_hash ||
					 cbgpu_ht_key_dict_hash(hp->ht, k) != s->pipe.cols[kx->col].dict_hash))
					return es_fail(es, CBGPU_ERR_UNSUPPORTED, "join of dictionary columns coded by two different dictionaries (share one dictionary between the columns)");
			}
		/* append the key expressions as extra output columns so the probe can read them */
		for (int k = 0; k < hj->nhashkeys; k++)
		{
			if (s->nout >= MAX_OUT)
				return es_fail(es, CBGPU_ERR_UNSUPPORTED, "too many output columns");
			s->out[s->nout++] = keys[k];
		}
		TRY(stream_materialize(es, ps, s, &me->owned, &orel, shape, &nshape));
		c = 0;
		for (int i = 0; i < nouter; i++)
			c += shape[i].kind == PE_STATE ? 3 : 1;
		for (int k = 0; k < hj->nhashkeys; k++)
			keycols[k] = c + k;
		if (me->owned.npairs >= 8)
			return es_fail(es, CBGPU_ERR_UNSUPPORTED, "too many N:M joins under one node");
		pairs = &me->owned.pairs[me->owned.npairs++];
		if (multi)
		{
			/* build side split into batches: the probe rows are grouped by batch once, each batch is loaded and probed in
			 * turn (HJ_NEED_NEW_BATCH, nodeHashjoin.c:709-738), unmatched build rows follow the last batch */
			int64_t		passes = 0;

			GPU(es, cbgpu_ht_probe_pairs_batched(es->es_ctx, hp->ht, orel, keycols, hj->nhashkeys, fill_outer,
												 fill_inner, es_pending, es, &passes, pairs));
			es->es_hashjoin_batches_run += passes;
		}
		else
			GPU(es, cbgpu_ht_probe_pairs_outer(es->es_ctx, hp->ht, orel, keycols, hj->nhashkeys, fill_outer, fill_inner, pairs));
		s2 = stream_new(me);
		TRY(stream_over_rel(es, s2, orel, shape, nouter));
		if (fill_inner)
			for (int i = 0; i < s2->npe; i++)
				s2->pe[i].maybe_null = 1;	/* the outer side of an unmatched build row is NULL */
		s2->pipe.nrows = pairs->npairs;
		s2->pipe.drv_nsrc = 2;
		s2->pipe.drv_idx[0] = pairs->outer_idx;
		s2->pipe.drv_idx[1] = pairs->inner_idx;
		s2->nsrc = 2;
		s2->rows_in = s->rows_in;
		nouter = s2->nout;
		memcpy(outer, s2->out, sizeof(int) * (size_t) nouter);
		TRY(inner_out_exprs(es, s2, hp, 1, fill_outer, inner));
		s = s2;
		vc.s = s;
	}
	else
	{
		int			j = s->pipe.nprobes;
		int			base = s->pipe.drv_nsrc > 1 ? s->pipe.drv_nsrc : 1;
		CbpProbe   *pr;

		if (base + j + 1 > CBP_MAX_SRC)
			return es_fail(es, CBGPU_ERR_UNSUPPORTED, "more than %d joined sources in one pipeline", CBP_MAX_SRC);
		for (int k = 0; k < hj->nhashkeys; k++)
			TRY(emit_expr(es, s, keys[k]));
		TRY(emit_op(es, s, CBP_PROBE, j, 0));
		pr = &s->pipe.probes[j];
		memset(pr, 0, sizeof(*pr));
		pr->ht = hp->ht;
		pr->jointype = hj->jointype;
		if (hj->jointype == CB_JOIN_LASJ_NOTIN)
		{
			/* x NOT IN (build side): an ANTI probe, except that NULLs are unknowns (nodeHashjoin.c:371-390, 578-590): a NULL
			 * key on the build side leaves nothing (hs_hashkeys_null -> the join returns no row at all); a NULL key on the
			 * probe side drops that row unless the build side is empty */
			const int64_t inner_rows = cbgpu_rel_nrows(hp->inner_rel);

			pr->jointype = CB_JOIN_ANTI;
			pr->null_key_drops = inner_rows > 0;
			if (inner_rows > cbgpu_ht_nrows(hp->ht))
			{
				int			never = pe_const(s, CB_BOOL, 0, 0);

				if (never < 0)
					return es_fail(es, CBGPU_ERR_UNSUPPORTED, "pipeline program too long");
				TRY(emit_expr(es, s, never));
				TRY(emit_op(es, s, CBP_FILTER, 0, 0));
			}
		}
		pr->nkeys = hj->nhashkeys;
		for (int k = 0; k < hj->nhashkeys; k++)
		{
			PExpr	   *kx = &s->pe[keys[k]];

			pr->keytype[k] = kx->type == CB_NUMERIC ? CB_INT8 : kx->type;
			if (kx->type == CB_NUMERIC)
				return es_fail(es, CBGPU_ERR_UNSUPPORTED, "numeric join keys (hash_numeric) are not on the GPU path");
			if (kx->type == CB_FLOAT8)
				/* float8eq makes -0 = +0 and every NaN equal (hashfloat8 maps them to one hash value, hashfunc.c:194); the
				 * tables compare key bits */
				return es_fail(es, CBGPU_ERR_UNSUPPORTED, "float8 join keys are not on the GPU path");
			if (kx->type == CB_DICT8 || kx->type == CB_DICT32)
			{
				if (kx->kind != PE_COL || !s->pipe.cols[kx->col].dict_hash)
					return es_fail(es, CBGPU_ERR_INVALID, "dictionary join key without per-code hashes");
				pr->key_dict_hash[k] = s->pipe.cols[kx->col].dict_hash;
				/* codes are compared, so both sides must be coded by ONE dictionary (cbgpu.h: a dictionary can be shared
				 * between columns that are joined); two private dictionaries would silently lose matches */
				if (cbgpu_ht_key_dict_hash(hp->ht, k) != pr->key_dict_hash[k])
					return es_fail(es, CBGPU_ERR_UNSUPPORTED, "join of dictionary columns coded by two different dictionaries (share one dictionary between the columns)");
			}
		}
		s->pipe.nprobes = j + 1;
		s->nsrc = base + j + 1;
		if (hj->jointype == CB_JOIN_SEMI || hj->jointype == CB_JOIN_ANTI || hj->jointype == CB_JOIN_LASJ_NOTIN)
		{
			/* no inner columns survive a semi / anti join */
			for (int i = 0; i < hp->inner_nout; i++)
				inner[i] = -1;
		}
		else
			TRY(inner_out_exprs(es, s, hp, base + j, hj->jointype == CB_JOIN_LEFT, inner));
	}
	vc.outer = outer;
	vc.nouter = nouter;
	vc.inner = inner;
	vc.ninner = hp->inner_nout;
	if ((hj->njoinquals > 0 || ps->plan->nquals > 0) && hj->jointype != CB_JOIN_INNER)
		return es_fail(es, CBGPU_ERR_UNSUPPORTED, "extra join quals on a non-inner hash join are not implemented on the GPU path");
	for (int i = 0; i < hj->njoinquals; i++)
		TRY(emit_qual(&vc, hj->joinqual[i]));
	for (int i = 0; i < ps->plan->nquals; i++)
		TRY(emit_qual(&vc, ps->plan->qual[i]));
	{
		int			newout[MAX_OUT];

		if (ps->plan->ntargets > MAX_OUT)
			return es_fail(es, CBGPU_ERR_UNSUPPORTED, "more than %d output columns", MAX_OUT);
		for (int i = 0; i < ps->plan->ntargets; i++)
		{
			const CbExpr *te = ps->plan->targetlist[i].expr;

			if (te->tag == T_CbVar && te->varno == CB_INNER_VAR && te->varattno >= 1 && te->varattno <= hp->inner_nout &&
				inner[te->varattno - 1] < 0)
				return es_fail(es, CBGPU_ERR_INVALID, "semi/anti join output references the inner side");
			TRY(translate(&vc, te, &newout[i]));
		}
		s->nout = ps->plan->ntargets;
		memcpy(s->out, newout, sizeof(int) * (size_t) s->nout);
	}
	*out = s;
	return CBGPU_OK;
}

/* ---- Agg ---- */
typedef struct AccMeta
{
	int			kind;			/* CbpAggKind used in the sink                                       */
	int			state_kind;		/* kind of the state it yields (COUNT / SUM_INT / SUM_FLOAT / MIN / MAX) */
	int			arg[3];			/* PE ids of the argument value(s), -1 = none                        */
	int			nargs;
	int			dscale;
	int			argtype;
} AccMeta;

typedef struct AggPlanInfo
{
	int			naccs;
	AccMeta		acc[CBP_MAX_AGGS];
	int			acc_of_target[MAX_OUT];	/* -1: grouping column                                       */
	int			key_of_target[MAX_OUT];
	int			keys[CBP_MAX_KEYS];		/* PE ids                                                    */
	int			nkeys;
	/* HAVING: the Aggref nodes of the qual and the accumulators that hold their states */
#define MAX_HAVING_AGGS 8
	const CbExpr *having_ref[MAX_HAVING_AGGS];
	int			having_acc[MAX_HAVING_AGGS];
	int			nhaving;
} AggPlanInfo;

/* one Aggref of an Agg node's target list or HAVING clause -> its accumulator (transition state): aggregates with the same
 * transition function and input share one (find_compatible_pertrans, nodeAgg.c) */
static int
agg_add_aggref(CbEState *es, VarCtx *vcp, CbStream *s, const CbAgg *agg, AggPlanInfo *info, const CbExpr *te, int *acc_out)
{
	VarCtx		vc = *vcp;
	AccMeta		m;
	int			found = -1;

	memset(&m, 0, sizeof(m));
	m.arg[0] = m.arg[1] = m.arg[2] = -1;
	if (agg->aggsplit == CB_AGGSPLIT_FINAL_DESERIAL)
	{
		/* combine functions over partial states */
		int			a;
		PExpr	   *st;

		if (te->nargs != 1)
			return es_fail(es, CBGPU_ERR_INVALID, "final aggregate needs the partial state as its argument");
		TRY(translate(&vc, te->args[0], &a));
		st = &s->pe[a];
		if (st->kind != PE_STATE)
			return es_fail(es, CBGPU_ERR_INVALID, "final aggregate input is not a partial aggregate state");
		m.state_kind = st->acckind;
		m.dscale = st->dscale;
		m.argtype = st->argtype;
		switch (st->acckind)
		{
			case CBP_ACC_COUNT:
				m.kind = CBP_ACC_MERGE_COUNT;
				m.arg[0] = st->cn;
				m.nargs = 1;
				break;
			case CBP_ACC_SUM_INT:
				m.kind = CBP_ACC_MERGE_INT;
				m.arg[0] = st->cn; m.arg[1] = st->clo; m.arg[2] = st->chi;
				m.nargs = 3;
				break;
			case CBP_ACC_SUM_FLOAT:
				m.kind = CBP_ACC_MERGE_FLOAT;
				m.arg[0] = st->cn; m.arg[1] = st->clo;
				m.nargs = 2;
				break;
			case CBP_ACC_MIN:
			case CBP_ACC_MAX:
				m.kind = st->acckind == CBP_ACC_MIN ? CBP_ACC_MERGE_MIN : CBP_ACC_MERGE_MAX;
				m.arg[0] = st->cn; m.arg[1] = st->clo;
				m.nargs = 2;
				break;
			default:
				return es_fail(es, CBGPU_ERR_INVALID, "unknown partial state kind %d", st->acckind);
		}
	}
	else
	{
		int			a = -1;

		if (te->nargs > 1)
			return es_fail(es, CBGPU_ERR_UNSUPPORTED, "aggregates with %d arguments are not supported", te->nargs);
		if (te->nargs == 1)
		{
			TRY(translate(&vc, te->args[0], &a));
			if (s->pe[a].kind == PE_STATE)
				return es_fail(es, CBGPU_ERR_INVALID, "aggregate argument is a transition state");
			m.argtype = s->pe[a].type;
			m.dscale = s->pe[a].dscale;
		}
		switch (te->op)
		{
			case CB_AGG_COUNT_STAR:
				m.kind = m.state_kind = CBP_ACC_COUNT;
				break;
			case CB_AGG_COUNT:
				m.kind = m.state_kind = CBP_ACC_COUNT;
				/* count(x) over a NOT NULL input is count(*) */
				if (a >= 0 && s->pe[a].maybe_null)
				{
					m.arg[0] = a;
					m.nargs = 1;
				}
				break;
			case CB_AGG_SUM:
			case CB_AGG_AVG:
				if (a < 0)
					return es_fail(es, CBGPU_ERR_INVALID, "sum/avg without an argument");
				m.kind = m.state_kind = (m.argtype == CB_FLOAT8) ? CBP_ACC_SUM_FLOAT : CBP_ACC_SUM_INT;
				m.arg[0] = a;
				m.nargs = 1;
				break;
			case CB_AGG_MIN:
			case CB_AGG_MAX:
				if (a < 0)
					return es_fail(es, CBGPU_ERR_INVALID, "min/max without an argument");
				if (m.argtype == CB_FLOAT8)
				{
					/* float8smaller / float8larger order NaN above everything (float8_cmp_internal, utils/adt/float.c): map the
					 * bits to integers with that order, use the integer accumulators, map back when the state is finalised */
					a = pe_op(s, CBP_F8ORD, a, -1, CB_INT8, 0, 0);
					if (a < 0)
						return es_fail(es, CBGPU_ERR_UNSUPPORTED, "pipeline program too long");
				}
				m.kind = m.state_kind = te->op == CB_AGG_MIN ? CBP_ACC_MIN : CBP_ACC_MAX;
				m.arg[0] = a;
				m.nargs = 1;
				break;
			default:
				return es_fail(es, CBGPU_ERR_UNSUPPORTED, "aggregate function %d is not supported on the GPU path", te->op);
		}
	}
	/* aggregates with the same transition function and input share one state
	 * (find_compatible_pertrans, nodeAgg.c) */
	for (int j = 0; j < info->naccs; j++)
		if (info->acc[j].kind == m.kind && info->acc[j].arg[0] == m.arg[0] && info->acc[j].arg[1] == m.arg[1] &&
			info->acc[j].arg[2] == m.arg[2])
			found = j;
	if (found < 0)
	{
		if (info->naccs >= CBP_MAX_AGGS)
			return es_fail(es, CBGPU_ERR_UNSUPPORTED, "more than %d distinct aggregate states", CBP_MAX_AGGS);
		found = info->naccs++;
		info->acc[found] = m;
	}
	*acc_out = found;
	return CBGPU_OK;
}

/* HAVING: collect the accumulators its Aggrefs need (walks the qual tree) */
static int
agg_collect_having(CbEState *es, VarCtx *vc, CbStream *s, const CbAgg *agg, AggPlanInfo *info, const CbExpr *e)
{
	if (e->tag == T_CbAggref)
	{
		int			a;

		if (info->nhaving >= MAX_HAVING_AGGS)
			return es_fail(es, CBGPU_ERR_UNSUPPORTED, "more than %d aggregates in HAVING", MAX_HAVING_AGGS);
		TRY(agg_add_aggref(es, vc, s, agg, info, e, &a));
		info->having_ref[info->nhaving] = e;
		info->having_acc[info->nhaving] = a;
		info->nhaving++;
		return CBGPU_OK;
	}
	for (int i = 0; i < e->nargs && (e->tag == T_CbOpExpr || e->tag == T_CbBoolExpr); i++)
		TRY(agg_collect_having(es, vc, s, agg, info, e->args[i]));
	return CBGPU_OK;
}

/* the child's rows aggregated: *table_out holds the groups - or, when they did not fit the operator's memory and the
 * aggregation ran in partitions, *parts_out holds them already as a relation (keys, then N / lo / hi per state) */
static int
agg_run(CbPlanState *ps, AggPlanInfo *info, cbgpu_aggtable **table_out, CbStream **child_stream, cbgpu_rel **parts_out)
{
	CbEState   *es = ps->state;
	CbAgg	   *agg = (CbAgg *) ps->plan;
	NodePriv   *p = np(ps);
	CbStream   *s;
	VarCtx		vc;
	int			outer[MAX_OUT];

	TRY(node_open(ps->lefttree, &s));
	*child_stream = s;
	memcpy(outer, s->out, sizeof(int) * (size_t) s->nout);
	memset(&vc, 0, sizeof(vc));
	vc.es = es;
	vc.s = s;
	vc.outer = outer;
	vc.nouter = s->nout;
	memset(info, 0, sizeof(*info));
	if (agg->numCols > CBP_MAX_KEYS)
		return es_fail(es, CBGPU_ERR_UNSUPPORTED, "GROUP BY with %d columns is beyond the GPU path's limit (%d)", agg->numCols, CBP_MAX_KEYS);
	if (agg->aggstrategy != CB_AGG_HASHED && agg->aggstrategy != CB_AGG_PLAIN)
		return es_fail(es, CBGPU_ERR_UNSUPPORTED, "only hashed / plain aggregation runs on the GPU path");
	info->nkeys = agg->numCols;
	for (int k = 0; k < agg->numCols; k++)
	{
		int			att = agg->grpColIdx[k];

		if (att < 1 || att > s->nout || s->pe[s->out[att - 1]].kind == PE_STATE)
			return es_fail(es, CBGPU_ERR_INVALID, "grouping column %d is not a scalar column of the child", att);
		info->keys[k] = s->out[att - 1];
	}
	if (ps->plan->ntargets > MAX_OUT)
		return es_fail(es, CBGPU_ERR_UNSUPPORTED, "more than %d output columns", MAX_OUT);
	for (int i = 0; i < ps->plan->ntargets; i++)
	{
		const CbExpr *te = ps->plan->targetlist[i].expr;
		int			found = -1;

		info->acc_of_target[i] = -1;
		info->key_of_target[i] = -1;
		if (te->tag == T_CbVar)
		{
			for (int k = 0; k < agg->numCols; k++)
				if (te->varno == CB_OUTER_VAR && agg->grpColIdx[k] == te->varattno)
					info->key_of_target[i] = k;
			if (info->key_of_target[i] < 0)
				return es_fail(es, CBGPU_ERR_INVALID, "Agg targetlist Var %d is not a grouping column", te->varattno);
			continue;
		}
		if (te->tag != T_CbAggref)
			return es_fail(es, CBGPU_ERR_UNSUPPORTED, "Agg targetlist entries must be grouping Vars or Aggrefs on the GPU path");
		TRY(agg_add_aggref(es, &vc, s, agg, info, te, &found));
		info->acc_of_target[i] = found;
	}

	for (int i = 0; i < ps->plan->nquals; i++)
		TRY(agg_collect_having(es, &vc, s, agg, info, ps->plan->qual[i]));

	/* program tail: key values, then the accumulators' arguments */
	CbPipeline *pl = &s->pipe;
	int			saved_nops = pl->nops;
	int			pos = 0;

	memset(&pl->sink, 0, sizeof(pl->sink));
	pl->sink.kind = CBP_SINK_AGG;
	pl->sink.nkeys = info->nkeys;
	for (int k = 0; k < info->nkeys; k++)
	{
		PExpr	   *kx = &s->pe[info->keys[k]];

		TRY(emit_expr(es, s, info->keys[k]));
		pl->sink.keytype[k] = kx->type;
		if (kx->type == CB_DICT8 || kx->type == CB_DICT32)
		{
			if (kx->kind != PE_COL || !pl->cols[kx->col].dict_hash)
				return es_fail(es, CBGPU_ERR_INVALID, "dictionary GROUP BY key without per-code hashes");
			pl->sink.key_dict_hash[k] = pl->cols[kx->col].dict_hash;
		}
	}
	pl->sink.naccs = info->naccs;
	for (int a = 0; a < info->naccs; a++)
	{
		pl->sink.accs[a].kind = info->acc[a].kind;
		pl->sink.accs[a].arg = info->acc[a].nargs ? pos : -1;
		for (int k = 0; k < info->acc[a].nargs; k++)
		{
			TRY(emit_expr(es, s, info->acc[a].arg[k]));
			pos++;
		}
	}
	TRY(emit_op(es, s, CBP_END, 0, 0));

	/* table sizing: the planner's numGroups estimate, bounded by the input; grow and retry on overflow */
	int64_t		cap = agg->numGroups > 0 ? agg->numGroups * 2 : 1024;
	int32_t		kinds[CBP_MAX_AGGS];

	if (cap < 1024)
		cap = 1024;
	if (cap > pl->nrows && pl->nrows >= 1024)
		cap = pl->nrows;
	for (int a = 0; a < info->naccs; a++)
		kinds[a] = info->acc[a].kind;
	pl->force_generic = es->es_force_generic;
	*table_out = NULL;
	if (parts_out)
		*parts_out = NULL;
	/* the operator's memory (PlanStateOperatorMemKB, execnodes.h:1166) bounds the table: two slots per group */
	const int64_t max_cap = es->es_operator_mem_kb > 0 && parts_out ?
		(es->es_operator_mem_kb * 1024 / (2 * cbgpu_agg_slot_bytes(info->nkeys, info->naccs)) > 64 ?
		 es->es_operator_mem_kb * 1024 / (2 * cbgpu_agg_slot_bytes(info->nkeys, info->naccs)) : 64) : 0;
	int			npart = 1;

	if (max_cap > 0 && cap > max_cap)
		cap = max_cap;
	for (;;)
	{
		cbgpu_aggtable *t;
		int64_t		ng;
		int			rc;
		int64_t		before = cbgpu_kernel_launches(es->es_ctx);

		if (npart > 1)
			break;
		GPU(es, cbgpu_agg_create(es->es_ctx, info->nkeys, info->naccs, kinds, cap, &t));
		pl->sink.agg = t;
		rc = run_pipeline(es, pl);
		if (rc == CBGPU_OK)
		{
			/* the group count's read-back fetches the status word too: one round trip for both.  A full
			 * table (NOMEM from ngroups) must not hide an overflow raised by the same kernel. */
			int			rc2 = cbgpu_agg_ngroups(t, &ng);

			rc = cbgpu_check_status(es->es_ctx);
			if (rc == CBGPU_OK)
				rc = rc2;
		}
		ps->instrument.kernels += cbgpu_kernel_launches(es->es_ctx) - before;
		ps->instrument.rows_in += s->rows_in;
		if (cbgpu_last_kernel_ms(es->es_ctx) > 0)
			ps->instrument.device_ms += cbgpu_last_kernel_ms(es->es_ctx);
		if (rc == CBGPU_ERR_NOMEM && max_cap > 0 && cap >= max_cap)
		{
			/* the groups do not fit the operator's memory: aggregate in partitions (below) */
			cbgpu_agg_free(t);
			npart = 2;
			continue;
		}
		if (rc == CBGPU_ERR_NOMEM && cap < pl->nrows)
		{
			/* more groups than estimated: the reference grows its table (simplehash SH_GROW) or
			 * spills; here: a larger table and another pass */
			cbgpu_agg_free(t);
			cap = cap * 8 < pl->nrows ? cap * 8 : pl->nrows;
			if (max_cap > 0 && cap > max_cap)
				cap = max_cap;
			continue;
		}
		if (rc != CBGPU_OK)
		{
			cbgpu_agg_free(t);
			return es_fail(es, rc, "%s", cbgpu_last_error(es->es_ctx));
		}
		p->owned.aggs[p->owned.naggs++] = t;
		*table_out = t;
		break;
	}
	/* partitioned aggregation: pass k aggregates the groups whose hash selects partition k into a table of the budget's size
	 * and hands them over as rows; a partition that still overflows doubles the partition count and starts over (the
	 * reference halves its spill partitions recursively, nodeAgg.c:3215 agg_refill_hash_table) */
	while (npart > 1)
	{
		cbgpu_rel  *pieces[256];
		int			npieces = 0;
		int64_t		total = 0;
		int32_t		keytypes[CBP_MAX_KEYS];
		int			rc = CBGPU_OK;
		int			overflow = 0;

		if (npart > 256)
			return es_fail(es, CBGPU_ERR_NOMEM, "hash aggregation does not fit the operator's memory even in 256 partitions");
		for (int k = 0; k < info->nkeys; k++)
			keytypes[k] = s->pe[info->keys[k]].type;
		for (int part = 0; part < npart && rc == CBGPU_OK && !overflow; part++)
		{
			cbgpu_aggtable *t;
			int64_t		ng;
			int			rc2;

			if (es->es_interrupt_pending && es->es_interrupt_pending(es))
				rc = es_fail(es, CBGPU_ERR_INTERRUPTED, "canceling statement due to user request");
			if (rc == CBGPU_OK)
				rc = cbgpu_agg_create(es->es_ctx, info->nkeys, info->naccs, kinds, max_cap, &t);
			if (rc != CBGPU_OK)
				break;
			cbgpu_agg_set_partition(t, npart, part);
			pl->sink.agg = t;
			rc = run_pipeline(es, pl);
			if (rc == CBGPU_OK)
			{
				rc2 = cbgpu_agg_ngroups(t, &ng);
				rc = cbgpu_check_status(es->es_ctx);
				if (rc == CBGPU_OK && rc2 == CBGPU_ERR_NOMEM)
					overflow = 1;
				else if (rc == CBGPU_OK)
					rc = rc2;
			}
			if (rc == CBGPU_OK && !overflow)
			{
				rc = cbgpu_agg_to_rel(t, keytypes, &pieces[npieces]);
				if (rc == CBGPU_OK)
					total += cbgpu_rel_nrows(pieces[npieces++]);
			}
			cbgpu_agg_free(t);
			es->es_agg_partitions_run++;
			ps->instrument.rows_in += s->rows_in;
		}
		if (rc == CBGPU_OK && !overflow)
		{
			/* the pieces back to back: the groups of the whole input */
			cbgpu_rel  *all = NULL;
			int32_t		types[CBP_MAX_OUT];
			const int	ncols = info->nkeys + 3 * info->naccs;
			int64_t		at = 0;

			for (int c = 0; c < ncols; c++)
				types[c] = c < info->nkeys ? keytypes[c] : CB_INT8;
			rc = cbgpu_rel_create(es->es_ctx, total, ncols, types, NULL, &all);
			for (int k = 0; k < info->nkeys && rc == CBGPU_OK; k++)
			{
				int			anynull = 0;

				for (int i = 0; i < npieces; i++)
					anynull |= cbgpu_rel_has_nulls(pieces[i], k);
				if (anynull)
					rc = cbgpu_rel_add_nullmap(all, k);
			}
			for (int i = 0; i < npieces && rc == CBGPU_OK; i++)
			{
				const int64_t n = cbgpu_rel_nrows(pieces[i]);

				if (n > 0)
					rc = cbgpu_rel_copy_rows(all, at, pieces[i], 0, n);
				at += n;
			}
			if (rc == CBGPU_OK)
			{
				p->owned.rels[p->owned.nrels++] = all;
				*parts_out = all;
				ps->instrument.agg_npartitions = npart;
			}
			else if (all)
				cbgpu_rel_free(all);
		}
		for (int i = 0; i < npieces; i++)
			cbgpu_rel_free(pieces[i]);
		if (rc != CBGPU_OK)
			return es->es_errcode ? es->es_errcode : es_fail(es, rc, "%s", cbgpu_last_error(es->es_ctx));
		if (!overflow)
			break;
		npart *= 2;
	}
	pl->nops = saved_nops;
	return CBGPU_OK;
}

/* finalize_aggregates (nodeAgg.c) for one (N, sum) state */
static void
finalize_state(const PExpr *st, int64_t n, int64_t lo, int64_t hi, int64_t *val, uint8_t *isnull, CbNumericDatum *num, int *type)
{
	*isnull = 0;
	*type = st->restype;
	switch (st->aggfn)
	{
		case CB_AGG_COUNT_STAR:
		case CB_AGG_COUNT:
			*val = n;
			*type = CB_INT8;
			return;
		case CB_AGG_SUM:
			if (n == 0)
			{
				*isnull = 1;
				return;
			}
			if (st->acckind == CBP_ACC_SUM_FLOAT)
			{
				*val = lo;
				*type = CB_FLOAT8;
				return;
			}
			if (st->restype == CB_INT8)
			{
				/* int4_sum yields bigint */
				*val = lo;
				return;
			}
			num->lo = lo;
			num->hi = hi;
			num->dscale = st->dscale;
			cb_numeric_sum_text(lo, hi, st->dscale, num->text, sizeof(num->text));
			*val = (int64_t) (intptr_t) num;
			*type = CB_NUMERIC;
			return;
		case CB_AGG_AVG:
			if (n == 0)
			{
				*isnull = 1;
				return;
			}
			if (st->acckind == CBP_ACC_SUM_FLOAT)
			{
				double		sx,
							avg;

				memcpy(&sx, &lo, 8);
				avg = sx / (double) n;	/* float8_avg (float.c:3148) */
				memcpy(val, &avg, 8);
				*type = CB_FLOAT8;
				return;
			}
			num->lo = lo;
			num->hi = hi;
			num->dscale = st->dscale;
			cb_numeric_avg_text(lo, hi, st->dscale, n, num->text, sizeof(num->text));
			*val = (int64_t) (intptr_t) num;
			*type = CB_NUMERIC;
			return;
		case CB_AGG_MIN:
		case CB_AGG_MAX:
			if (n == 0)
			{
				*isnull = 1;
				return;
			}
			if (st->argtype == CB_NUMERIC)
			{
				num->lo = lo;
				num->hi = lo < 0 ? -1 : 0;
				num->dscale = st->dscale;
				cb_numeric_sum_text(num->lo, num->hi, st->dscale, num->text, sizeof(num->text));
				*val = (int64_t) (intptr_t) num;
				*type = CB_NUMERIC;
			}
			else if (st->argtype == CB_FLOAT8)
			{
				/* the state holds the order-preserving integer (CBP_F8ORD): back to float8 bits */
				*val = lo >= 0 ? lo : (int64_t) ((uint64_t) lo ^ 0x7FFFFFFFFFFFFFFFull);
				*type = CB_FLOAT8;
			}
			else
			{
				*val = lo;
				*type = st->argtype;
			}
			return;
	}
	*isnull = 1;
}

static void
fill_state_pe(PExpr *e, const CbAgg *agg, const CbExpr *aggref, const AccMeta *m)
{
	memset(e, 0, sizeof(*e));
	e->kind = PE_STATE;
	e->type = aggref->restype;
	e->restype = aggref->restype;
	e->dscale = m->dscale;
	e->acckind = m->state_kind;
	e->aggfn = aggref->op;
	e->argtype = m->argtype;
	e->final = agg->aggsplit != CB_AGGSPLIT_INITIAL_SERIAL;
	e->l = e->r = -1;
}

/* Agg drained at the top of a slice: read the groups back and finalise on the host */
static int
agg_result(CbPlanState *ps)
{
	CbEState   *es = ps->state;
	CbAgg	   *agg = (CbAgg *) ps->plan;
	NodePriv   *p = np(ps);
	AggPlanInfo info;
	cbgpu_aggtable *t;
	CbStream   *cs;
	int64_t		ng = 0;
	ResultSet  *rs;
	int64_t    *keys, *n, *lo, *hi;
	uint32_t   *keynull;
	int			nk, na;

	TRY(agg_run(ps, &info, &t, &cs, NULL));
	GPU(es, cbgpu_agg_ngroups(t, &ng));
	nk = info.nkeys ? info.nkeys : 1;
	na = info.naccs ? info.naccs : 1;
	keys = calloc((size_t) (ng ? ng : 1) * nk, sizeof(int64_t));
	keynull = calloc((size_t) (ng ? ng : 1), sizeof(uint32_t));
	n = calloc((size_t) (ng ? ng : 1) * na, sizeof(int64_t));
	lo = calloc((size_t) (ng ? ng : 1) * na, sizeof(int64_t));
	hi = calloc((size_t) (ng ? ng : 1) * na, sizeof(int64_t));
	if (ng > 0)
	{
		int			rc = cbgpu_agg_read(t, ng, keys, keynull, n, lo, hi, &ng);

		if (rc)
		{
			free(keys); free(keynull); free(n); free(lo); free(hi);
			return es_fail(es, rc, "%s", cbgpu_last_error(es->es_ctx));
		}
	}
	/* a plain aggregate (no GROUP BY) emits one row even over empty input (nodeAgg.c agg_retrieve_direct) */
	int			synth = (ng == 0 && agg->numCols == 0 && agg->aggstrategy == CB_AGG_PLAIN);

	rs = rs_new(synth ? 1 : ng, ps->plan->ntargets);
	for (int i = 0; i < ps->plan->ntargets; i++)
		rs->types[i] = ps->plan->targetlist[i].expr->restype;
	for (int64_t g = 0; g < rs->nrows; g++)
		for (int i = 0; i < ps->plan->ntargets; i++)
		{
			size_t		o = (size_t) g * rs->ncols + i;

			if (info.key_of_target[i] >= 0)
			{
				int			k = info.key_of_target[i];

				rs->vals[o] = keys[g * nk + k];
				rs->nulls[o] = (keynull[g] >> k) & 1;
				rs->types[i] = cs->pe[info.keys[k]].type;
			}
			else
			{
				int			a = info.acc_of_target[i];
				PExpr		st;
				int64_t		vn = synth ? 0 : n[g * na + a],
							vlo = synth ? 0 : lo[g * na + a],
							vhi = synth ? 0 : hi[g * na + a];
				int			ty;

				fill_state_pe(&st, agg, ps->plan->targetlist[i].expr, &info.acc[a]);
				rs->st_n[o] = vn;
				rs->st_lo[o] = vlo;
				rs->st_hi[o] = vhi;
				if (agg->aggsplit == CB_AGGSPLIT_INITIAL_SERIAL)
				{
					rs->vals[o] = vlo;
					rs->types[i] = CB_INT8;
				}
				else
				{
					finalize_state(&st, vn, vlo, vhi, &rs->vals[o], &rs->nulls[o], &rs->nums[o], &ty);
					rs->types[i] = ty;
				}
			}
		}
	free(keys); free(keynull); free(n); free(lo); free(hi);
	p->rs = rs;
	return CBGPU_OK;
}

/* ------------------------------------------------------------------------------------------
 * HAVING (Agg.plan.qual; ExecQual over the finalised aggregates, nodeAgg.c:2460 / 3100): evaluated on the host over the
 * groups' exact states - a value is the rational num / (den * 10^scale) - so that `sum(x) > 100.00` or `avg(x) <= y` decide
 * exactly as numeric arithmetic does.  The groups that pass become a selection vector over the groups' relation.
 * ------------------------------------------------------------------------------------------ */
typedef struct HVal
{
	__int128	num;
	int64_t		den;			/* > 0                                                                */
	int			scale;
	int			isnull;
	int			isbool;			/* num is 0 / 1                                                       */
} HVal;

typedef struct HCtx
{
	CbEState   *es;
	const CbAgg *agg;
	const AggPlanInfo *info;
	CbStream   *cs;				/* the child's stream: types and scales of the grouping columns           */
	int64_t		g;				/* group (row of the groups' relation)                                */
	int64_t   **keycol;			/* [nkeys] widened key values                                         */
	uint8_t   **keynull;
	int64_t   **st_n, **st_lo, **st_hi;	/* [naccs]                                                  */
	int			err;
} HCtx;

static int
hv_scale_up(__int128 *v, int k)
{
	while (k-- > 0)
		if (__builtin_mul_overflow(*v, (__int128) 10, v))
			return 0;
	return 1;
}

static HVal
having_eval(HCtx *h, const CbExpr *e)
{
	HVal		r;

	memset(&r, 0, sizeof(r));
	r.den = 1;
	switch (e->tag)
	{
		case T_CbConst:
			r.isnull = e->constisnull;
			r.num = e->constval;
			r.scale = e->dscale;
			if (e->restype == CB_FLOAT8)
				h->err = 1;
			return r;
		case T_CbVar:
			for (int k = 0; k < h->agg->numCols; k++)
				if (e->varno == CB_OUTER_VAR && h->agg->grpColIdx[k] == e->varattno)
				{
					r.isnull = h->keynull[k] ? h->keynull[k][h->g] : 0;
					r.num = h->keycol[k][h->g];
					r.scale = h->cs->pe[h->info->keys[k]].dscale;
					if (h->cs->pe[h->info->keys[k]].type == CB_FLOAT8)
						h->err = 1;
					return r;
				}
			h->err = 1;
			return r;
		case T_CbAggref:
			for (int i = 0; i < h->info->nhaving; i++)
				if (h->info->having_ref[i] == e)
				{
					const int	a = h->info->having_acc[i];
					const AccMeta *m = &h->info->acc[a];
					const int64_t n = h->st_n[a][h->g];

					if (m->state_kind == CBP_ACC_SUM_FLOAT)
					{
						h->err = 1;		/* float8 aggregates compare inexactly: not decided here */
						return r;
					}
					r.scale = m->dscale;
					switch (e->op)
					{
						case CB_AGG_COUNT_STAR:
						case CB_AGG_COUNT:
							r.num = n;
							r.scale = 0;
							return r;
						case CB_AGG_SUM:
						case CB_AGG_AVG:
							r.isnull = n == 0;
							r.num = ((__int128) h->st_hi[a][h->g] << 64) | (unsigned __int128) (uint64_t) h->st_lo[a][h->g];
							if (e->op == CB_AGG_AVG && n > 0)
								r.den = n;
							return r;
						case CB_AGG_MIN:
						case CB_AGG_MAX:
							r.isnull = n == 0;
							r.num = h->st_lo[a][h->g];
							return r;
					}
				}
			h->err = 1;
			return r;
		case T_CbOpExpr:
			{
				HVal		a,
							b;
				__int128	L,
							R;
				int			c;

				if (e->nargs != 2 || e->op < CB_OP_EQ)
				{
					h->err = 1;		/* arithmetic over aggregates in HAVING: not on this path */
					return r;
				}
				a = having_eval(h, e->args[0]);
				b = having_eval(h, e->args[1]);
				r.isbool = 1;
				if (a.isnull || b.isnull)
				{
					r.isnull = 1;
					return r;
				}
				/* a.num / (a.den 10^a.scale)  ?  b.num / (b.den 10^b.scale): cross-multiplied, exact or refused */
				L = a.num;
				R = b.num;
				if (__builtin_mul_overflow(L, (__int128) b.den, &L) || __builtin_mul_overflow(R, (__int128) a.den, &R) ||
					!hv_scale_up(&L, b.scale > a.scale ? b.scale - a.scale : 0) || !hv_scale_up(&R, a.scale > b.scale ? a.scale - b.scale : 0))
				{
					h->err = 2;
					return r;
				}
				c = L < R ? -1 : L > R ? 1 : 0;
				switch (e->op)
				{
					case CB_OP_EQ: r.num = c == 0; break;
					case CB_OP_NE: r.num = c != 0; break;
					case CB_OP_LT: r.num = c < 0; break;
					case CB_OP_LE: r.num = c <= 0; break;
					case CB_OP_GT: r.num = c > 0; break;
					default: r.num = c >= 0; break;
				}
				return r;
			}
		case T_CbBoolExpr:
			{
				int			anynull = 0;

				r.isbool = 1;
				if (e->op == CB_NOT_EXPR)
				{
					HVal		a = having_eval(h, e->args[0]);

					r.isnull = a.isnull;
					r.num = !a.num;
					return r;
				}
				/* three-valued AND / OR (ExecEvalBoolAndStep / OrStep, execExprInterp.c) */
				r.num = e->op == CB_AND_EXPR;
				for (int i = 0; i < e->nargs; i++)
				{
					HVal		a = having_eval(h, e->args[i]);

					if (a.isnull)
						anynull = 1;
					else if (e->op == CB_AND_EXPR && !a.num)
					{
						r.num = 0;
						return r;
					}
					else if (e->op == CB_OR_EXPR && a.num)
					{
						r.num = 1;
						return r;
					}
				}
				r.isnull = anynull;
				return r;
			}
		default:
			h->err = 1;
			return r;
	}
}

/* groups relation `rel` (keys, then N / lo / hi per accumulator) -> device selection vector of the groups HAVING keeps */
static int
having_select(CbPlanState *ps, const AggPlanInfo *info, CbStream *cs, cbgpu_rel *rel, uint32_t **sel_dev, int64_t *nsel)
{
	CbEState   *es = ps->state;
	NodePriv   *p = np(ps);
	const CbAgg *agg = (const CbAgg *) ps->plan;
	const int64_t ng = cbgpu_rel_nrows(rel);
	HCtx		h;
	uint32_t   *sel = calloc((size_t) (ng ? ng : 1), sizeof(uint32_t));
	int64_t		kept = 0;
	int			rc = CBGPU_OK;
	const int	nk = info->nkeys,
				na = info->naccs;
	void	   *dev = NULL;

	memset(&h, 0, sizeof(h));
	h.es = es;
	h.agg = agg;
	h.info = info;
	h.cs = cs;
	h.keycol = calloc((size_t) (nk ? nk : 1), sizeof(int64_t *));
	h.keynull = calloc((size_t) (nk ? nk : 1), sizeof(uint8_t *));
	h.st_n = calloc((size_t) (na ? na : 1), sizeof(int64_t *));
	h.st_lo = calloc((size_t) (na ? na : 1), sizeof(int64_t *));
	h.st_hi = calloc((size_t) (na ? na : 1), sizeof(int64_t *));
	for (int k = 0; k < nk && rc == CBGPU_OK; k++)
	{
		const int	w = cb_type_width((CbTypeId) cbgpu_rel_col_type(rel, k));
		char	   *raw = calloc((size_t) (ng ? ng : 1), (size_t) w);

		h.keycol[k] = calloc((size_t) (ng ? ng : 1), sizeof(int64_t));
		h.keynull[k] = calloc((size_t) (ng ? ng : 1), 1);
		if (ng > 0)
			rc = cbgpu_rel_read_column(rel, k, 0, ng, raw, h.keynull[k]);
		for (int64_t g = 0; g < ng; g++)
			h.keycol[k][g] = w == 1 ? ((uint8_t *) raw)[g] : w == 4 ? ((int32_t *) raw)[g] : ((int64_t *) raw)[g];
		free(raw);
	}
	for (int i = 0; i < info->nhaving && rc == CBGPU_OK; i++)
	{
		const int	a = info->having_acc[i];

		if (h.st_n[a])
			continue;
		h.st_n[a] = calloc((size_t) (ng ? ng : 1), sizeof(int64_t));
		h.st_lo[a] = calloc((size_t) (ng ? ng : 1), sizeof(int64_t));
		h.st_hi[a] = calloc((size_t) (ng ? ng : 1), sizeof(int64_t));
		if (ng > 0)
		{
			rc = cbgpu_rel_read_column(rel, nk + 3 * a, 0, ng, h.st_n[a], NULL);
			if (rc == CBGPU_OK)
				rc = cbgpu_rel_read_column(rel, nk + 3 * a + 1, 0, ng, h.st_lo[a], NULL);
			if (rc == CBGPU_OK)
				rc = cbgpu_rel_read_column(rel, nk + 3 * a + 2, 0, ng, h.st_hi[a], NULL);
		}
	}
	for (int64_t g = 0; g < ng && rc == CBGPU_OK && !h.err; g++)
	{
		int			keep = 1;

		h.g = g;
		for (int q = 0; q < ps->plan->nquals && keep; q++)
		{
			HVal		v = having_eval(&h, ps->plan->qual[q]);

			keep = !v.isnull && v.num != 0;	/* ExecQual: NULL counts as false */
		}
		if (keep)
			sel[kept++] = (uint32_t) g;
	}
	if (rc != CBGPU_OK)
		rc = es_fail(es, rc, "%s", cbgpu_last_error(es->es_ctx));
	else if (h.err == 2)
		rc = es_fail(es, CBGPU_ERR_OVERFLOW, "HAVING: a comparison of aggregates left 128 bits");
	else if (h.err)
		rc = es_fail(es, CBGPU_ERR_UNSUPPORTED, "HAVING on the GPU path compares aggregates, grouping columns and constants (no arithmetic, no float8)");
	if (rc == CBGPU_OK)
	{
		rc = cbgpu_dev_alloc(es->es_ctx, sizeof(uint32_t) * (size_t) (kept ? kept : 1), &dev);
		if (rc == CBGPU_OK)
		{
			p->owned.devs[p->owned.ndevs++] = dev;
			if (kept > 0)
				rc = cbgpu_dev_write(es->es_ctx, dev, sizeof(uint32_t) * (size_t) kept, sel);
		}
		if (rc != CBGPU_OK)
			rc = es_fail(es, rc, "%s", cbgpu_last_error(es->es_ctx));
	}
	for (int k = 0; k < nk; k++)
	{
		free(h.keycol[k]);
		free(h.keynull[k]);
	}
	for (int a = 0; a < na; a++)
	{
		free(h.st_n[a]);
		free(h.st_lo[a]);
		free(h.st_hi[a]);
	}
	free(h.keycol); free(h.keynull); free(h.st_n); free(h.st_lo); free(h.st_hi);
	free(sel);
	*sel_dev = (uint32_t *) dev;
	*nsel = kept;
	return rc;
}

/* Agg feeding a parent on the device: groups become a relation (keys, then N / lo / hi per state) */
static int
open_agg(CbPlanState *ps, CbStream **out)
{
	CbEState   *es = ps->state;
	CbAgg	   *agg = (CbAgg *) ps->plan;
	NodePriv   *p = np(ps);
	AggPlanInfo info;
	cbgpu_aggtable *t;
	CbStream   *cs,
			   *s;
	cbgpu_rel  *rel;
	int32_t		keytypes[CBP_MAX_KEYS];

	TRY(agg_run(ps, &info, &t, &cs, &rel));
	for (int k = 0; k < info.nkeys; k++)
		keytypes[k] = cs->pe[info.keys[k]].type;
	if (rel == NULL)
	{
		GPU(es, cbgpu_agg_to_rel(t, keytypes, &rel));
		p->owned.rels[p->owned.nrels++] = rel;
	}
	for (int k = 0; k < info.nkeys; k++)
	{
		PExpr	   *kx = &cs->pe[info.keys[k]];

		if ((kx->type == CB_DICT8 || kx->type == CB_DICT32) && kx->kind == PE_COL)
			GPU(es, cbgpu_rel_share_dict_hash(rel, k, cs->col_rel[kx->col], cs->col_idx[kx->col]));
	}
	s = stream_new(p);
	s->pipe.nrows = cbgpu_rel_nrows(rel);
	s->rows_in = s->pipe.nrows;
	s->nsrc = 1;
	s->nout = ps->plan->ntargets;
	if (ps->plan->nquals > 0)
	{
		/* HAVING: the stream reads the groups' relation through the selection of the groups that pass */
		uint32_t   *sel = NULL;
		int64_t		nsel = 0;

		TRY(having_select(ps, &info, cs, rel, &sel, &nsel));
		s->pipe.drv_nsrc = 1;
		s->pipe.drv_idx[0] = sel;
		s->pipe.nrows = nsel;
	}
	for (int i = 0; i < ps->plan->ntargets; i++)
	{
		if (info.key_of_target[i] >= 0)
		{
			int			k = info.key_of_target[i];

			s->out[i] = pe_col(s, rel, k, 0, 0);
			if (s->out[i] >= 0)
				s->pe[s->out[i]].dscale = cs->pe[info.keys[k]].dscale;
		}
		else
		{
			int			a = info.acc_of_target[i];
			PExpr		e;

			fill_state_pe(&e, agg, ps->plan->targetlist[i].expr, &info.acc[a]);
			e.cn = pe_col(s, rel, info.nkeys + a * 3, 0, 0);
			e.clo = pe_col(s, rel, info.nkeys + a * 3 + 1, 0, 0);
			e.chi = pe_col(s, rel, info.nkeys + a * 3 + 2, 0, 0);
			s->out[i] = (e.cn < 0 || e.clo < 0 || e.chi < 0) ? -1 : pe_add(s, &e);
		}
		if (s->out[i] < 0)
			return es_fail(es, CBGPU_ERR_UNSUPPORTED, "too many columns in one pipeline");
	}
	ps->instrument.ntuples = (double) s->pipe.nrows;
	*out = s;
	return CBGPU_OK;
}

/* ---- Motion ---- */
/* one run of the sender slice's pipeline into a staged PARTITION sink: `out` holds destination d's rows from
 * row base[d] on, cap[d] of them fit.  counts[] = rows ROUTED to each destination, whether they fitted or not. */
static int
partition_pass(CbPlanState *ps, CbStream *s, cbgpu_rel *out, void *counter, void *flagword, const int64_t *base, const int64_t *cap,
			   int nsegs, int64_t *counts)
{
	CbEState   *es = ps->state;
	CbPipeline *pl = &s->pipe;
	int64_t		before = cbgpu_kernel_launches(es->es_ctx);
	int64_t		zeros[65];

	memset(zeros, 0, sizeof(zeros));
	GPU(es, cbgpu_dev_write(es->es_ctx, counter, sizeof(int64_t) * (size_t) nsegs, zeros));
	GPU(es, cbgpu_dev_write(es->es_ctx, flagword, sizeof(int64_t), zeros));
	pl->sink.out = out;
	pl->sink.seg_base = base;
	pl->sink.seg_cap = cap;
	pl->sink.part_flags = (int32_t *) flagword;
	TRY(run_pipeline(es, pl));
	GPU(es, cbgpu_dev_read(es->es_ctx, counter, sizeof(int64_t) * (size_t) nsegs, counts));	/* the status word rides along */
	GPU(es, cbgpu_check_status(es->es_ctx));
	ps->instrument.kernels += cbgpu_kernel_launches(es->es_ctx) - before;
	ps->instrument.rows_in += s->rows_in;
	if (cbgpu_last_kernel_ms(es->es_ctx) > 0)
		ps->instrument.device_ms += cbgpu_last_kernel_ms(es->es_ctx);
	return CBGPU_OK;
}

/* execMotionSender (nodeMotion.c:203): run the child, route every row.  Leaves either the delivered rows in
 * np(ps)->recv (direct Motion: recv_ready set) or this segment's rows grouped by destination in *send
 * (destination d: offsets[d], counts[d]).  np(ps)->xstage tells open_motion how far the exchange got, for
 * the peers' sake, when this fails. */
static int
motion_send_side(CbPlanState *ps, cbgpu_rel **send, int64_t *counts, int64_t *offsets)
{
	CbEState   *es = ps->state;
	CbMotion   *m = (CbMotion *) ps->plan;
	NodePriv   *p = np(ps);
	CbStream   *s;
	int			nsegs = es->es_numsegments;

	TRY(node_open(ps->lefttree, &s));
	if (m->motionType != CB_MOTIONTYPE_HASH)
	{
		TRY(stream_materialize(es, ps, s, &p->owned, send, p->send_pe, &p->send_nout));
		counts[0] = cbgpu_rel_nrows(*send);
		offsets[0] = 0;
		return CBGPU_OK;
	}
	/* hash motion: PARTITION sink = evalHashKey (nodeMotion.c:1088) + per-destination buffers */
	{
		int32_t		types[CBP_MAX_OUT],
					dscales[CBP_MAX_OUT];
		int			ncols = 0,
					nullable[CBP_MAX_OUT];
		CbPipeline *pl = &s->pipe;
		int			saved_nops = pl->nops;
		int			hashpe[CBP_MAX_KEYS];
		int			outer[MAX_OUT];
		VarCtx		vc;
		void	   *counter;
		cbgpu_rel  *rel;
		uint64_t	nullmask = 0;

		if (m->nhashExprs < 1 || m->nhashExprs > CBP_MAX_KEYS)
			return es_fail(es, CBGPU_ERR_UNSUPPORTED, "hash Motion with %d keys is beyond the GPU path's limit", m->nhashExprs);
		memcpy(outer, s->out, sizeof(int) * (size_t) s->nout);
		memset(&vc, 0, sizeof(vc));
		vc.es = es;
		vc.s = s;
		vc.outer = outer;
		vc.nouter = s->nout;
		/* the hash key values go first on the stack (and into the leading output columns),
		 * then every output column */
		memset(&pl->sink, 0, sizeof(pl->sink));
		for (int k = 0; k < m->nhashExprs; k++)
		{
			PExpr	   *kx;

			TRY(translate(&vc, m->hashExprs[k], &hashpe[k]));
			kx = &s->pe[hashpe[k]];
			if (kx->kind == PE_STATE || kx->type == CB_NUMERIC)
				return es_fail(es, CBGPU_ERR_UNSUPPORTED, "Motion hash key type is not supported on the GPU path");
			TRY(emit_expr(es, s, hashpe[k]));
			types[ncols] = kx->type;
			dscales[ncols] = kx->dscale;
			nullable[ncols] = kx->maybe_null;
			pl->sink.hashtype[k] = kx->type;
			if (kx->type == CB_DICT8 || kx->type == CB_DICT32)
			{
				if (kx->kind != PE_COL || !pl->cols[kx->col].dict_hash)
					return es_fail(es, CBGPU_ERR_INVALID, "dictionary Motion key without per-code hashes");
				pl->sink.hash_dict_hash[k] = pl->cols[kx->col].dict_hash;
			}
			ncols++;
		}
		for (int i = 0; i < s->nout; i++)
		{
			PExpr	   *x = &s->pe[s->out[i]];

			p->send_pe[i] = *x;
			if (x->kind == PE_STATE)
			{
				if (ncols + 3 > CBP_MAX_OUT)
					return es_fail(es, CBGPU_ERR_UNSUPPORTED, "too many Motion columns");
				for (int k = 0; k < 3; k++)
				{
					types[ncols] = CB_INT8;
					dscales[ncols] = 0;
					nullable[ncols] = 0;
					ncols++;
				}
				TRY(emit_expr(es, s, x->cn));
				TRY(emit_expr(es, s, x->clo));
				TRY(emit_expr(es, s, x->chi));
			}
			else
			{
				if (ncols + 1 > CBP_MAX_OUT)
					return es_fail(es, CBGPU_ERR_UNSUPPORTED, "too many Motion columns");
				types[ncols] = x->type;
				dscales[ncols] = x->dscale;
				nullable[ncols] = x->maybe_null;
				ncols++;
				TRY(emit_expr(es, s, s->out[i]));
			}
		}
		p->send_nout = s->nout;
		TRY(emit_op(es, s, CBP_END, 0, 0));
		GPU(es, cbgpu_dev_alloc(es->es_ctx, sizeof(int64_t) * (size_t) (nsegs + 1), &counter));
		p->owned.devs[p->owned.ndevs++] = counter;
		pl->sink.kind = CBP_SINK_PARTITION;
		pl->sink.nout = ncols;
		pl->sink.out_count = (int64_t *) counter;
		pl->sink.nhash = m->nhashExprs;
		pl->sink.nsegs = m->numHashSegments > 0 ? m->numHashSegments : nsegs;
		pl->force_generic = es->es_force_generic;
		if (pl->sink.nsegs != nsegs)
			return es_fail(es, CBGPU_ERR_UNSUPPORTED, "Motion to %d hash segments on a %d-segment cluster", pl->sink.nsegs, nsegs);
		for (int c = 0; c < ncols; c++)
			if (nullable[c])
				nullmask |= 1ull << c;

		/* direct Motion (interconnects with peer memory): the PARTITION sink stores every row straight into
		 * its destination segment's receive window - no send buffer, no separate exchange, no collective */
		{
			CbInterconnect *ic = es->es_cluster ? NULL : es->es_interconnect;
			cbgpu_direct_dest dest;

			if (ic && ic->direct_begin && ic->direct_begin(ic, es, m->motionID, ncols, types, dscales, &dest) == CBGPU_OK)
			{
				cbgpu_rel  *recv = NULL;
				int32_t		outcome = CBGPU_DX_DELIVERED;
				int			rc,
							rc2;
				int64_t		before = cbgpu_kernel_launches(es->es_ctx);

				/* from here to direct_end nothing may return early: the peers wait for this segment's signal */
				rc = cbgpu_rel_create(es->es_ctx, 0, ncols, types, dscales, &rel);
				if (rc == CBGPU_OK)
				{
					p->owned.rels[p->owned.nrels++] = rel;
					pl->sink.out = rel;
					pl->sink.seg_capacity = dest.capacity;
					pl->sink.part_cols = dest.cols;
					pl->sink.part_counts = dest.counts;
					pl->sink.part_nulls = dest.nulls;
					pl->sink.part_nullmask = nullmask;
					pl->sink.part_flags = dest.flags;
					rc = run_pipeline(es, pl);
				}
				if (rc && es->es_errcode == 0)
					es_fail(es, rc, "%s", cbgpu_last_error(es->es_ctx));
				rc2 = ic->direct_end(ic, es, m->motionID, rc ? CBGPU_DX_ERROR : 0, nullmask, (const int64_t *) counter, counts, &recv, &outcome);
				p->xstage = 1;
				if (recv)
					p->owned.rels[p->owned.nrels++] = recv;
				if (rc)
					return rc;
				/* an error this segment's own kernels raised (fetched with the completion: no extra round trip) is
				 * the one to report here; the peers see CBGPU_ERR_PEER */
				{
					char		peermsg[512];
					int			st;

					snprintf(peermsg, sizeof(peermsg), "%s", rc2 ? cbgpu_last_error(es->es_ctx) : "");
					st = cbgpu_check_status(es->es_ctx);
					if (st)
					{
						es->es_errcode = 0;
						return es_fail(es, st, "%s", cbgpu_last_error(es->es_ctx));
					}
					if (rc2)
						return es->es_errcode ? es->es_errcode : es_fail(es, rc2, "%s", peermsg);
				}
				ps->instrument.kernels += cbgpu_kernel_launches(es->es_ctx) - before;
				ps->instrument.rows_in += s->rows_in;
				if (cbgpu_last_kernel_ms(es->es_ctx) > 0)
					ps->instrument.device_ms += cbgpu_last_kernel_ms(es->es_ctx);
				if (outcome == CBGPU_DX_DELIVERED)
				{
					/* RecvTupleFrom for the whole stream, done */
					int			c = m->nhashExprs;

					for (int k = 0; k < m->nhashExprs; k++)
					{
						PExpr	   *kx = &s->pe[hashpe[k]];

						if (kx->kind == PE_COL && (kx->type == CB_DICT8 || kx->type == CB_DICT32) && pl->cols[kx->col].dict_hash)
							GPU(es, cbgpu_rel_share_dict_hash(recv, k, s->col_rel[kx->col], s->col_idx[kx->col]));
					}
					for (int i = 0; i < s->nout; i++)
					{
						PExpr	   *x = &s->pe[s->out[i]];

						if (x->kind == PE_STATE)
						{
							c += 3;
							continue;
						}
						if (x->kind == PE_COL && (x->type == CB_DICT8 || x->type == CB_DICT32) && pl->cols[x->col].dict_hash)
							GPU(es, cbgpu_rel_share_dict_hash(recv, c, s->col_rel[x->col], s->col_idx[x->col]));
						c++;
					}
					pl->nops = saved_nops;
					memset(&pl->sink, 0, sizeof(pl->sink));
					p->recv = recv;
					p->recv_ready = 1;
					p->xstage = 2;
					*send = rel;
					return CBGPU_OK;
				}
				/* CBGPU_DX_RETRY: a destination's window was full somewhere (skew, or a Motion larger than the
				 * windows): every segment redoes it staged, with exactly sized buffers */
				pl->sink.part_cols = NULL;
				pl->sink.part_counts = NULL;
				pl->sink.part_nulls = NULL;
				pl->sink.part_nullmask = 0;
			}
		}

		/* staged Motion: partition into a local send buffer, then the interconnect's exchange.  First an
		 * optimistic layout (every destination could receive every row: reserve nrows per destination only
		 * when small, otherwise the even share plus a skew allowance); if a destination turns out fuller -
		 * the reference never fails on skew, it sends tuple by tuple (cdbmotion.c:425) - the counts of that
		 * pass size a second, exact one */
		{
			int64_t		base[64],
						cap[64];
			int64_t		each = pl->nrows;
			int64_t		total = 0;
			int			over = 0;
			void	   *flagword = (char *) counter + sizeof(int64_t) * (size_t) nsegs;

			if (pl->nrows > (1 << 20))
			{
				each = pl->nrows / nsegs + pl->nrows / (4 * nsegs) + 65536;
				if (each > pl->nrows)
					each = pl->nrows;
			}
			for (int d = 0; d < nsegs; d++)
			{
				base[d] = (int64_t) d * each;
				cap[d] = each;
			}
			GPU(es, cbgpu_rel_create(es->es_ctx, each * nsegs, ncols, types, dscales, &rel));
			p->owned.rels[p->owned.nrels++] = rel;
			for (int c = 0; c < ncols; c++)
				if (nullable[c])
					GPU(es, cbgpu_rel_add_nullmap(rel, c));
			TRY(partition_pass(ps, s, rel, counter, flagword, base, cap, nsegs, counts));
			for (int d = 0; d < nsegs; d++)
			{
				over |= counts[d] > cap[d];
				total += counts[d];
			}
			if (over)
			{
				int64_t		again[64];

				for (int d = 0; d < nsegs; d++)
				{
					base[d] = d == 0 ? 0 : base[d - 1] + counts[d - 1];
					cap[d] = counts[d];
				}
				/* the first buffer goes back before the exact one is taken */
				for (int i = 0; i < p->owned.nrels; i++)
					if (p->owned.rels[i] == rel)
						p->owned.rels[i] = p->owned.rels[--p->owned.nrels];
				cbgpu_rel_free(rel);
				GPU(es, cbgpu_rel_create(es->es_ctx, total, ncols, types, dscales, &rel));
				p->owned.rels[p->owned.nrels++] = rel;
				for (int c = 0; c < ncols; c++)
					if (nullable[c])
						GPU(es, cbgpu_rel_add_nullmap(rel, c));
				TRY(partition_pass(ps, s, rel, counter, flagword, base, cap, nsegs, again));
				for (int d = 0; d < nsegs; d++)
					if (again[d] != counts[d])
						return es_fail(es, CBGPU_ERR_INVALID, "Motion %d: the sender slice routed %lld rows to segment %d on its second pass, %lld on its first",
									   m->motionID, (long long) again[d], d, (long long) counts[d]);
				ps->instrument.motion_repartitions += 1;
			}
			for (int d = 0; d < nsegs; d++)
				offsets[d] = base[d];
			{
				int			c = m->nhashExprs;

				for (int i = 0; i < s->nout; i++)
				{
					PExpr	   *x = &s->pe[s->out[i]];

					if (x->kind == PE_STATE)
					{
						c += 3;
						continue;
					}
					if (x->kind == PE_COL && (x->type == CB_DICT8 || x->type == CB_DICT32) && pl->cols[x->col].dict_hash)
						GPU(es, cbgpu_rel_share_dict_hash(rel, c, s->col_rel[x->col], s->col_idx[x->col]));
					c++;
				}
				for (int k = 0; k < m->nhashExprs; k++)
				{
					PExpr	   *kx = &s->pe[hashpe[k]];

					if (kx->kind == PE_COL && (kx->type == CB_DICT8 || kx->type == CB_DICT32) && pl->cols[kx->col].dict_hash)
						GPU(es, cbgpu_rel_share_dict_hash(rel, k, s->col_rel[kx->col], s->col_idx[kx->col]));
				}
			}
			pl->nops = saved_nops;
			pl->sink.seg_base = NULL;	/* they pointed into this frame */
			pl->sink.seg_cap = NULL;
			*send = rel;
		}
	}
	return CBGPU_OK;
}

/* shape of the received relation: hash motions carry their key values in leading columns */
static int
motion_recv_stream(CbPlanState *ps, cbgpu_rel *recv, CbStream **out)
{
	CbEState   *es = ps->state;
	CbMotion   *m = (CbMotion *) ps->plan;
	NodePriv   *p = np(ps);
	CbStream   *s = stream_new(p);
	int			lead = m->motionType == CB_MOTIONTYPE_HASH ? m->nhashExprs : 0;
	int			c = lead;

	s->pipe.nrows = cbgpu_rel_nrows(recv);
	s->rows_in = s->pipe.nrows;
	s->nsrc = 1;
	s->nout = p->send_nout;
	for (int i = 0; i < p->send_nout; i++)
	{
		if (p->send_pe[i].kind == PE_STATE)
		{
			PExpr		e = p->send_pe[i];

			e.cn = pe_col(s, recv, c, 0, 0);
			e.clo = pe_col(s, recv, c + 1, 0, 0);
			e.chi = pe_col(s, recv, c + 2, 0, 0);
			s->out[i] = (e.cn < 0 || e.clo < 0 || e.chi < 0) ? -1 : pe_add(s, &e);
			c += 3;
		}
		else
		{
			s->out[i] = pe_col(s, recv, c, 0, 0);
			if (s->out[i] >= 0)
				s->pe[s->out[i]].dscale = p->send_pe[i].dscale;
			c++;
		}
		if (s->out[i] < 0)
			return es_fail(es, CBGPU_ERR_UNSUPPORTED, "too many columns in one pipeline");
	}
	if (m->nsortkeys > 0 && s->pipe.nrows > 1)
	{
		/* merge receive (execMotionSortedReceiver, nodeMotion.c:433): the senders' sorted streams lie one after another
		 * in the receive buffer; read them in merged order */
		int32_t		keycols[8],
					desc[8],
					uns[8];
		int			nk = 0;
		int32_t		nruns = 0;
		uint32_t   *order = NULL;
		int64_t		before = cbgpu_kernel_launches(es->es_ctx);

		if (m->motionType != CB_MOTIONTYPE_GATHER && m->motionType != CB_MOTIONTYPE_GATHER_SINGLE)
			return es_fail(es, CBGPU_ERR_UNSUPPORTED, "a sorted Motion that is not a Gather");
		TRY(sort_key_columns(es, p->send_pe, p->send_nout, lead, m->sortkeys, m->nsortkeys, keycols, desc, uns, &nk));
		GPU(es, cbgpu_merge_sorted_runs(es->es_ctx, recv, keycols, desc, uns, nk, es->es_numsegments, &order, &nruns));
		ps->instrument.kernels += cbgpu_kernel_launches(es->es_ctx) - before;
		if (order)
		{
			p->owned.devs[p->owned.ndevs++] = order;
			s->pipe.drv_nsrc = 1;
			s->pipe.drv_idx[0] = order;
		}
	}
	ps->instrument.ntuples = (double) s->pipe.nrows;
	*out = s;
	return CBGPU_OK;
}

static int
open_motion(CbPlanState *ps, CbStream **out)
{
	CbEState   *es = ps->state;
	CbMotion   *m = (CbMotion *) ps->plan;
	NodePriv   *p = np(ps);

	if (es->es_numsegments <= 1)
		return node_open(ps->lefttree, out);	/* one segment: every Motion is the identity */
	if (es->es_cluster)
	{
		/* in-process cluster: the first receiver to arrive runs every segment's sender slice */
		if (!p->recv_ready)
			TRY(cluster_run_motion(ps));
		if (!p->recv)
			return es_fail(es, CBGPU_ERR_INVALID, "Motion %d: nothing was delivered to segment %d", m->motionID, es->es_segindex);
		return motion_recv_stream(ps, p->recv, out);
	}
	if (!es->es_interconnect)
		return es_fail(es, CBGPU_ERR_INVALID, "Motion node without an interconnect (SetupInterconnect not done)");
	{
		cbgpu_rel  *send = NULL,
				   *recv = NULL;
		int64_t		counts[64],
					offsets[64];
		CbInterconnect *ic = es->es_interconnect;
		int			rc;

		if (es->es_numsegments > 64)
			return es_fail(es, CBGPU_ERR_UNSUPPORTED, "more than 64 segments");
		memset(counts, 0, sizeof(counts));
		memset(offsets, 0, sizeof(offsets));
		rc = motion_send_side(ps, &send, counts, offsets);
		if (rc)
		{
			/* this segment will not take part in the exchange the others are about to enter (or have entered):
			 * say so instead of leaving them waiting (they then fail with CBGPU_ERR_PEER) */
			if (p->xstage < 2 && ic->abandon)
				ic->abandon(ic, es, m->motionID, p->xstage == 1);
			p->xstage = 2;
			return rc;
		}
		if (p->recv_ready)		/* direct Motion: the sender slice's kernel already delivered */
			return motion_recv_stream(ps, p->recv, out);
		switch (m->motionType)
		{
			case CB_MOTIONTYPE_HASH:
				rc = ic->redistribute(ic, es, m->motionID, send, counts, offsets, &recv);
				break;
			case CB_MOTIONTYPE_GATHER:
			case CB_MOTIONTYPE_GATHER_SINGLE:
				rc = ic->gather(ic, es, m->motionID, 0, send,
								(m->motionType == CB_MOTIONTYPE_GATHER_SINGLE && es->es_segindex != 0) ? 0 : counts[0], &recv);
				break;
			case CB_MOTIONTYPE_BROADCAST:
				rc = ic->broadcast(ic, es, m->motionID, send, counts[0], &recv);
				break;
			default:
				if (ic->abandon)
					ic->abandon(ic, es, m->motionID, 0);
				return es_fail(es, CBGPU_ERR_UNSUPPORTED, "motion type %d", m->motionType);
		}
		p->xstage = 2;
		if (rc)
			return es->es_errcode ? es->es_errcode : es_fail(es, rc, "%s", cbgpu_last_error(es->es_ctx));
		p->recv = recv;
		p->owned.rels[p->owned.nrels++] = recv;
		p->recv_ready = 1;
		return motion_recv_stream(ps, recv, out);
	}
}

static int
node_open(CbPlanState *ps, CbStream **out)
{
	NodePriv   *p = np(ps);

	if (ps->state->es_errcode)
		return ps->state->es_errcode;
	if (p->opened && p->stream)
	{
		*out = p->stream;
		return CBGPU_OK;
	}
	/* CHECK_FOR_INTERRUPTS, once per node = before every pipeline of the query */
	if (ps->state->es_interrupt_pending && ps->state->es_interrupt_pending(ps->state))
	{
		CbInterconnect *ic = ps->state->es_cluster ? NULL : ps->state->es_interconnect;

		/* a Motion this segment will not enter: the peers must not wait for it */
		if (ps->type == T_CbMotion && ic && ic->abandon && ps->state->es_numsegments > 1 && p->xstage < 2)
		{
			ic->abandon(ic, ps->state, ((CbMotion *) ps->plan)->motionID, p->xstage == 1);
			p->xstage = 2;
		}
		return es_fail(ps->state, CBGPU_ERR_INTERRUPTED, "canceling statement due to user request");
	}
	cbgpu_range_push(node_name(ps->type));
	{
		int			rc = node_open_inner(ps, out);

		cbgpu_range_pop();
		return rc;
	}
}

static const char *
node_name(CbNodeTag t)
{
	switch (t)
	{
		case T_CbSeqScan: return "SeqScan";
		case T_CbHash: return "Hash";
		case T_CbHashJoin: return "HashJoin";
		case T_CbAgg: return "Agg";
		case T_CbMotion: return "Motion";
		case T_CbLimitSort: return "Limit/Sort";
		default: return "node";
	}
}

static int
node_open_inner(CbPlanState *ps, CbStream **out)
{
	NodePriv   *p = np(ps);

	switch (ps->type)
	{
		case T_CbSeqScan:
			TRY(open_seqscan(ps, out));
			break;
		case T_CbHashJoin:
			TRY(open_hashjoin(ps, out));
			break;
		case T_CbAgg:
			TRY(open_agg(ps, out));
			break;
		case T_CbMotion:
			TRY(open_motion(ps, out));
			break;
		case T_CbHash:
			return es_fail(ps->state, CBGPU_ERR_INVALID, "a Hash node is driven by MultiExecProcNode, not ExecProcNode (as in the reference, nodeHash.c:113)");
		case T_CbLimitSort:
			TRY(open_limitsort(ps, out));
			break;
		default:
			return es_fail(ps->state, CBGPU_ERR_UNSUPPORTED, "plan node %d is not on the GPU path", ps->type);
	}
	p->stream = *out;
	p->opened = 1;
	return CBGPU_OK;
}

/* ------------------------------------------------------------------------------------------
 * draining: rows to the host
 * ------------------------------------------------------------------------------------------ */
static int
rel_to_result(CbEState *es, cbgpu_rel *rel, const PExpr *shape, int nshape, const uint32_t *rowidx, int64_t nidx, ResultSet **out)
{
	int64_t		nrows = rowidx ? nidx : cbgpu_rel_nrows(rel);
	ResultSet  *rs = rs_new(nrows, nshape);
	int			ncols = cbgpu_rel_ncols(rel);
	int64_t   **colv = calloc((size_t) ncols, sizeof(int64_t *));
	uint8_t   **coln = calloc((size_t) ncols, sizeof(uint8_t *));
	int			rc = CBGPU_OK;

	/* small result sets (groups, top-N rows): every column's rows in one round trip */
	if (nrows > 0 && nrows * ncols <= (1 << 20))
	{
		int64_t    *vals = calloc((size_t) (nrows * ncols), sizeof(int64_t));
		uint8_t    *nls = calloc((size_t) (nrows * ncols), 1);

		rc = cbgpu_rel_read_rows(rel, rowidx, nrows, vals, nls);
		for (int c = 0; c < ncols; c++)
		{
			colv[c] = calloc((size_t) nrows, sizeof(int64_t));
			coln[c] = calloc((size_t) nrows, 1);
			for (int64_t r = 0; r < nrows && rc == CBGPU_OK; r++)
			{
				colv[c][r] = vals[(size_t) r * ncols + c];
				coln[c][r] = nls[(size_t) r * ncols + c];
			}
		}
		free(vals);
		free(nls);
	}
	else
	/* read every column (whole, or the selected rows one by one when an index list is given) */
	for (int c = 0; c < ncols && rc == CBGPU_OK; c++)
	{
		int			w = cb_type_width((CbTypeId) cbgpu_rel_col_type(rel, c));
		char	   *raw = calloc((size_t) (nrows ? nrows : 1), (size_t) w);

		colv[c] = calloc((size_t) (nrows ? nrows : 1), sizeof(int64_t));
		coln[c] = calloc((size_t) (nrows ? nrows : 1), 1);
		if (rowidx)
		{
			for (int64_t r = 0; r < nrows && rc == CBGPU_OK; r++)
				rc = cbgpu_rel_read_column(rel, c, rowidx[r], (int64_t) rowidx[r] + 1, raw + (size_t) r * w, coln[c] + r);
		}
		else if (nrows > 0)
			rc = cbgpu_rel_read_column(rel, c, 0, nrows, raw, coln[c]);
		for (int64_t r = 0; r < nrows; r++)
		{
			switch (w)
			{
				case 1: colv[c][r] = ((uint8_t *) raw)[r]; break;
				case 4: colv[c][r] = ((int32_t *) raw)[r]; break;
				default: colv[c][r] = ((int64_t *) raw)[r]; break;
			}
		}
		free(raw);
	}
	if (rc == CBGPU_OK)
	{
		int			c = 0;

		for (int i = 0; i < nshape; i++)
		{
			if (shape[i].kind == PE_STATE)
			{
				for (int64_t r = 0; r < nrows; r++)
				{
					size_t		o = (size_t) r * nshape + i;
					int			ty;

					rs->st_n[o] = colv[c][r];
					rs->st_lo[o] = colv[c + 1][r];
					rs->st_hi[o] = colv[c + 2][r];
					if (shape[i].final)
					{
						finalize_state(&shape[i], colv[c][r], colv[c + 1][r], colv[c + 2][r], &rs->vals[o], &rs->nulls[o],
									   &rs->nums[o], &ty);
						rs->types[i] = ty;
					}
					else
					{
						rs->vals[o] = colv[c + 1][r];
						rs->types[i] = CB_INT8;
					}
				}
				if (nrows == 0)
					rs->types[i] = shape[i].restype;
				c += 3;
			}
			else
			{
				rs->types[i] = shape[i].type;
				for (int64_t r = 0; r < nrows; r++)
				{
					size_t		o = (size_t) r * nshape + i;

					rs->nulls[o] = coln[c][r];
					if (shape[i].type == CB_NUMERIC)
					{
						CbNumericDatum *nd = &rs->nums[o];

						nd->lo = colv[c][r];
						nd->hi = colv[c][r] < 0 ? -1 : 0;
						nd->dscale = shape[i].dscale;
						cb_numeric_sum_text(nd->lo, nd->hi, nd->dscale, nd->text, sizeof(nd->text));
						rs->vals[o] = (int64_t) (intptr_t) nd;
					}
					else
						rs->vals[o] = colv[c][r];
				}
				c++;
			}
		}
	}
	for (int c = 0; c < ncols; c++)
	{
		free(colv[c]);
		free(coln[c]);
	}
	free(colv);
	free(coln);
	if (rc)
	{
		rs_free(rs);
		return es_fail(es, rc, "%s", cbgpu_last_error(es->es_ctx));
	}
	*out = rs;
	return CBGPU_OK;
}

/* sort keys over a materialised stream (columns laid out as stream_materialize / the Motion receive buffer does: one
 * column per scalar, N / lo / hi per transition state, `lead` leading extra columns) -> the device comparators' key columns.
 * Exact 128-bit sums order through (hi signed, lo unsigned). */
static int
sort_key_columns(CbEState *es, const PExpr *shape, int nshape, int lead, const CbSortKey *keys, int nkeys, int32_t *keycols,
				 int32_t *desc, int32_t *uns, int *nk_out)
{
	int			colstart[MAX_OUT];
	int			c = lead;
	int			nk = 0;

	for (int i = 0; i < nshape; i++)
	{
		colstart[i] = c;
		c += shape[i].kind == PE_STATE ? 3 : 1;
	}
	for (int k = 0; k < nkeys; k++)
	{
		int			att = keys[k].attno;

		if (att < 1 || att > nshape)
			return es_fail(es, CBGPU_ERR_INVALID, "sort key %d out of range", att);
		if (shape[att - 1].kind == PE_STATE)
		{
			/* ORDER BY sum(...): order the exact 128-bit sums through (hi signed, lo unsigned) */
			if (!(shape[att - 1].aggfn == CB_AGG_SUM && shape[att - 1].acckind == CBP_ACC_SUM_INT) &&
				shape[att - 1].aggfn != CB_AGG_COUNT && shape[att - 1].aggfn != CB_AGG_COUNT_STAR)
				return es_fail(es, CBGPU_ERR_UNSUPPORTED, "ORDER BY over this aggregate is not implemented on the GPU path");
			if (nk + 2 > 4)
				return es_fail(es, CBGPU_ERR_UNSUPPORTED, "too many sort keys for the device comparators");
			if (shape[att - 1].aggfn == CB_AGG_SUM)
			{
				keycols[nk] = colstart[att - 1] + 2; desc[nk] = keys[k].descending; uns[nk] = 0; nk++;
				keycols[nk] = colstart[att - 1] + 1; desc[nk] = keys[k].descending; uns[nk] = 1; nk++;
			}
			else
			{
				keycols[nk] = colstart[att - 1]; desc[nk] = keys[k].descending; uns[nk] = 0; nk++;
			}
		}
		else
		{
			if (nk + 1 > 4)
				return es_fail(es, CBGPU_ERR_UNSUPPORTED, "too many sort keys for the device comparators");
			keycols[nk] = colstart[att - 1]; desc[nk] = keys[k].descending; uns[nk] = 0; nk++;
		}
	}
	*nk_out = nk;
	return CBGPU_OK;
}

/* Limit <- Sort: device top-N over the child's materialised rows */
static int
limitsort_run(CbPlanState *ps, cbgpu_rel **out_rel, PExpr *out_shape, int *out_nshape)
{
	CbEState   *es = ps->state;
	CbLimitSort *ls = (CbLimitSort *) ps->plan;
	NodePriv   *p = np(ps);
	CbStream   *s;
	cbgpu_rel  *rel = NULL;
	PExpr		shape[MAX_OUT];
	int			nshape;
	int32_t		keycols[8],
				desc[8],
				uns[8];
	int			nk = 0;
	uint32_t	idx[64];
	int64_t		nout = 0;

	TRY(node_open(ps->lefttree, &s));
	/* the child's rows as a relation */
	TRY(stream_materialize(es, ps, s, &p->owned, &rel, shape, &nshape));
	for (int i = 0; i < ps->plan->ntargets; i++)
	{
		const CbExpr *te = ps->plan->targetlist[i].expr;

		if (te->tag != T_CbVar || te->varno != CB_OUTER_VAR || te->varattno != i + 1)
			return es_fail(es, CBGPU_ERR_UNSUPPORTED, "Limit/Sort must pass its child's columns through unchanged on the GPU path");
	}
	TRY(sort_key_columns(es, shape, nshape, 0, ls->keys, ls->nkeys, keycols, desc, uns, &nk));
	if (ls->limit < 0)
		return es_fail(es, CBGPU_ERR_UNSUPPORTED, "Sort without LIMIT is not on the GPU path (nodeSort.c stays on the CPU)");
	if (ls->limit > 0)
	{
		int64_t		before = cbgpu_kernel_launches(es->es_ctx);

		GPU(es, cbgpu_topn(es->es_ctx, rel, keycols, desc, uns, nk, ls->limit, idx, &nout));
		ps->instrument.kernels += cbgpu_kernel_launches(es->es_ctx) - before;
	}
	/* the chosen rows, in order, as a small relation of their own */
	{
		int32_t		types[CBP_MAX_OUT],
					dscales[CBP_MAX_OUT];
		int			ncols = cbgpu_rel_ncols(rel);
		cbgpu_rel  *small;

		for (int c = 0; c < ncols; c++)
		{
			types[c] = cbgpu_rel_col_type(rel, c);
			dscales[c] = cbgpu_rel_col_dscale(rel, c);
		}
		GPU(es, cbgpu_rel_create(es->es_ctx, nout, ncols, types, dscales, &small));
		p->owned.rels[p->owned.nrels++] = small;
		if (nout > 0)
		{
			/* one gather kernel for all rows and columns (row-by-row copies were 60 tiny memcpys for Q3's ten rows) */
			void	   *didx;

			GPU(es, cbgpu_dev_alloc(es->es_ctx, sizeof(uint32_t) * (size_t) nout, &didx));
			p->owned.devs[p->owned.ndevs++] = didx;
			GPU(es, cbgpu_dev_write(es->es_ctx, didx, sizeof(uint32_t) * (size_t) nout, idx));
			GPU(es, cbgpu_rel_take_rows(small, rel, (const uint32_t *) didx, nout));
		}
		for (int c = 0; c < ncols; c++)
			if (cbgpu_rel_dict_hash_dev(rel, c))
				GPU(es, cbgpu_rel_share_dict_hash(small, c, rel, c));
		*out_rel = small;
	}
	memcpy(out_shape, shape, sizeof(PExpr) * (size_t) nshape);
	*out_nshape = nshape;
	return CBGPU_OK;
}

static int
limitsort_result(CbPlanState *ps)
{
	cbgpu_rel  *small;
	PExpr		shape[MAX_OUT];
	int			nshape;

	TRY(limitsort_run(ps, &small, shape, &nshape));
	return rel_to_result(ps->state, small, shape, nshape, NULL, 0, &np(ps)->rs);
}

static int
open_limitsort(CbPlanState *ps, CbStream **out)
{
	cbgpu_rel  *small;
	PExpr		shape[MAX_OUT];
	int			nshape;
	CbStream   *s;

	TRY(limitsort_run(ps, &small, shape, &nshape));
	s = stream_new(np(ps));
	TRY(stream_over_rel(ps->state, s, small, shape, nshape));
	*out = s;
	return CBGPU_OK;
}

static int
node_result(CbPlanState *ps)
{
	CbEState   *es = ps->state;
	NodePriv   *p = np(ps);

	if (p->rs)
		return CBGPU_OK;
	/* with an operator memory budget the groups may come in partitions: then they are a relation already (open_agg), and the
	 * rows are read from it like any other node's */
	if (ps->type == T_CbAgg && !(es->es_operator_mem_kb > 0 && ((CbAgg *) ps->plan)->numCols > 0) && ps->plan->nquals == 0)
		return agg_result(ps);
	if (ps->type == T_CbLimitSort)
		return limitsort_result(ps);
	{
		CbStream   *s;
		cbgpu_rel  *rel;
		PExpr		shape[MAX_OUT];
		int			nshape;

		const uint32_t *sel = NULL;

		TRY(node_open(ps, &s));
		if (stream_is_plain(s, &rel, &sel))
		{
			/* already a relation with exactly these columns?  (Motion receive buffers, agg relations) */
			int			exact = 1,
						c = 0;

			for (int i = 0; i < s->nout && exact; i++)
			{
				PExpr	   *x = &s->pe[s->out[i]];

				shape[i] = *x;
				if (x->kind == PE_STATE)
				{
					if (s->pe[x->cn].kind != PE_COL || s->col_idx[s->pe[x->cn].col] != c)
						exact = 0;
					c += 3;
				}
				else
				{
					if (x->kind != PE_COL || s->col_idx[x->col] != c)
						exact = 0;
					c++;
				}
			}
			if (exact && c == cbgpu_rel_ncols(rel) && !sel)
				return rel_to_result(es, rel, shape, s->nout, NULL, 0, &p->rs);
			if (exact && c == cbgpu_rel_ncols(rel))
			{
				/* the rows in the stream's order (a MATERIALIZE sink appends in whatever order its warps finish) */
				int32_t		types[CBP_MAX_OUT],
							dscales[CBP_MAX_OUT];
				cbgpu_rel  *ordered;

				for (int k = 0; k < c; k++)
				{
					types[k] = cbgpu_rel_col_type(rel, k);
					dscales[k] = cbgpu_rel_col_dscale(rel, k);
				}
				GPU(es, cbgpu_rel_create(es->es_ctx, s->pipe.nrows, c, types, dscales, &ordered));
				p->owned.rels[p->owned.nrels++] = ordered;
				GPU(es, cbgpu_rel_take_rows(ordered, rel, sel, s->pipe.nrows));
				return rel_to_result(es, ordered, shape, s->nout, NULL, 0, &p->rs);
			}
		}
		TRY(stream_materialize(es, ps, s, &p->owned, &rel, shape, &nshape));
		return rel_to_result(es, rel, shape, nshape, NULL, 0, &p->rs);
	}
}

/* ------------------------------------------------------------------------------------------
 * public API
 * ------------------------------------------------------------------------------------------ */
CbEState *
cb_CreateExecutorState(cbgpu_ctx *ctx, cbgpu_rel **range_table, int32_t nrels)
{
	CbEState   *es = calloc(1, sizeof(CbEState));

	es->es_ctx = ctx;
	es->es_nrels = nrels;
	es->es_range_table = calloc((size_t) (nrels ? nrels : 1), sizeof(cbgpu_rel *));
	for (int i = 0; i < nrels; i++)
		es->es_range_table[i] = range_table[i];
	es->es_numsegments = 1;
	return es;
}

void
cb_FreeExecutorState(CbEState *estate)
{
	if (!estate)
		return;
	free(estate->es_range_table);
	free(estate);
}

static CbTupleTableSlot *
make_slot(int natts)
{
	CbTupleTableSlot *slot = calloc(1, sizeof(CbTupleTableSlot));
	size_t		n = (size_t) (natts ? natts : 1);

	slot->tts_empty = true;
	slot->tts_nvalid = natts;
	slot->tts_types = calloc(n, sizeof(int32_t));
	slot->tts_values = calloc(n, sizeof(int64_t));
	slot->tts_isnull = calloc(n, sizeof(bool));
	slot->tts_state_n = calloc(n, sizeof(int64_t));
	slot->tts_state_lo = calloc(n, sizeof(int64_t));
	slot->tts_state_hi = calloc(n, sizeof(int64_t));
	return slot;
}

static void
free_slot(CbTupleTableSlot *slot)
{
	if (!slot)
		return;
	free(slot->tts_types);
	free(slot->tts_values);
	free(slot->tts_isnull);
	free(slot->tts_state_n);
	free(slot->tts_state_lo);
	free(slot->tts_state_hi);
	free(slot);
}

static CbTupleTableSlot *
exec_generic(CbPlanState *ps)
{
	NodePriv   *p = np(ps);
	CbTupleTableSlot *slot = ps->ps_ResultTupleSlot;
	ResultSet  *rs;

	slot->tts_empty = true;
	if (ps->squelched || ps->state->es_errcode)
		return NULL;
	if (ps->type == T_CbHash)
	{
		es_fail(ps->state, CBGPU_ERR_INVALID, "Hash node does not support ExecProcNode call convention");	/* nodeHash.c:113 */
		return NULL;
	}
	if (!p->rs)
	{
		if (node_result(ps) != CBGPU_OK)
			return NULL;
		ps->instrument.nloops += 1;
	}
	rs = p->rs;
	if (rs->cursor >= rs->nrows)
		return NULL;			/* end of data */
	for (int i = 0; i < rs->ncols; i++)
	{
		size_t		o = (size_t) rs->cursor * rs->ncols + i;

		slot->tts_types[i] = rs->types[i];
		slot->tts_values[i] = rs->vals[o];
		slot->tts_isnull[i] = rs->nulls[o];
		slot->tts_state_n[i] = rs->st_n[o];
		slot->tts_state_lo[i] = rs->st_lo[o];
		slot->tts_state_hi[i] = rs->st_hi[o];
	}
	rs->cursor++;
	slot->tts_empty = false;	/* ExecStoreVirtualTuple */
	ps->instrument.ntuples += 1;
	ps->state->es_processed++;
	return slot;
}

/* Batch-oriented twin of ExecProcNode (SURVEY.md 8b: "new native entry points are batch-oriented"):
 * the node's whole output as ONE device-resident column batch instead of a slot per call.  The
 * relation holds one column per scalar output (three per transition state: N, sum lo, sum hi) and
 * becomes the caller's (cbgpu_rel_free).  For parents that can consume a batch - another GPU
 * operator, a Motion sender, a loader distributing a table with `DISTRIBUTED BY`. */
int
cb_ExecProcNodeBatch(CbPlanState *ps, cbgpu_rel **out)
{
	CbEState   *es = ps->state;
	NodePriv   *p = np(ps);
	CbStream   *s;
	cbgpu_rel  *rel = NULL;
	PExpr		shape[MAX_OUT];
	int			nshape;
	int			found = -1;

	*out = NULL;
	if (ps->squelched || es->es_errcode)
		return es->es_errcode ? es->es_errcode : CBGPU_ERR_INVALID;
	if (ps->type == T_CbHash || ps->type == T_CbAgg || ps->type == T_CbLimitSort)
		return es_fail(es, CBGPU_ERR_UNSUPPORTED, "batch output of node type %d (its result is finalised on the host)", (int) ps->type);
	TRY(node_open(ps, &s));
	TRY(stream_materialize_ex(es, ps, s, &p->owned, &rel, shape, &nshape, 2));
	for (int i = 0; i < p->owned.nrels; i++)
		if (p->owned.rels[i] == rel)
			found = i;
	if (found < 0)
		return es_fail(es, CBGPU_ERR_INVALID, "batch output lost track of its relation");
	p->owned.rels[found] = p->owned.rels[--p->owned.nrels];
	ps->instrument.ntuples += (double) cbgpu_rel_nrows(rel);
	ps->instrument.nloops += 1;
	*out = rel;
	return CBGPU_OK;
}

CbPlanState *
cb_ExecInitNode(CbPlan *node, CbEState *estate, int eflags)
{
	CbPlanState *ps;

	(void) eflags;
	if (!node)
		return NULL;
	switch (node->type)
	{
		case T_CbSeqScan: case T_CbHash: case T_CbHashJoin: case T_CbAgg: case T_CbMotion: case T_CbLimitSort:
			break;
		default:
			es_fail(estate, CBGPU_ERR_UNSUPPORTED, "unrecognized / unsupported node type: %d", (int) node->type);	/* execProcnode.c:525 */
			return NULL;
	}
	ps = calloc(1, sizeof(CbPlanState));
	ps->type = node->type;
	ps->plan = node;
	ps->state = estate;
	ps->ExecProcNode = exec_generic;
	ps->priv = calloc(1, sizeof(NodePriv));
	ps->ps_ResultTupleSlot = make_slot(node->ntargets);
	if (node->lefttree)
	{
		ps->lefttree = cb_ExecInitNode(node->lefttree, estate, eflags);
		if (!ps->lefttree)
			goto fail;
	}
	if (node->righttree)
	{
		ps->righttree = cb_ExecInitNode(node->righttree, estate, eflags);
		if (!ps->righttree)
			goto fail;
	}
	if (node->type != T_CbSeqScan && !ps->lefttree)
	{
		es_fail(estate, CBGPU_ERR_INVALID, "plan node %d needs an outer child", (int) node->type);
		goto fail;
	}
	return ps;
fail:
	cb_ExecEndNode(ps);
	return NULL;
}

CbTupleTableSlot *
cb_ExecProcNode(CbPlanState *node)
{
	return node->ExecProcNode(node);
}

cbgpu_hashtable *
cb_MultiExecProcNode(CbPlanState *node)
{
	if (node->type != T_CbHash)
	{
		es_fail(node->state, CBGPU_ERR_INVALID, "unrecognized node type for MultiExecProcNode: %d", (int) node->type);	/* execProcnode.c:760 */
		return NULL;
	}
	if (hash_build(node) != CBGPU_OK)
		return NULL;
	return np(node)->ht;
}

static void
node_reset(CbPlanState *node)
{
	NodePriv   *p = np(node);

	rs_free(p->rs);
	p->rs = NULL;
	owned_free(node->state, &p->owned);
	p->stream = NULL;
	p->opened = 0;
	p->ht = NULL;
	p->inner_rel = NULL;
	p->recv = NULL;
	p->recv_ready = 0;
	p->xstage = 0;
}

void
cb_ExecReScan(CbPlanState *node)
{
	if (!node)
		return;
	cb_ExecReScan(node->lefttree);
	cb_ExecReScan(node->righttree);
	node_reset(node);
	node->squelched = false;
}

void
cb_ExecSquelchNode(CbPlanState *node)
{
	/* tell the sub-tree no more tuples are wanted (execAmi.c:763) */
	if (!node || node->squelched)
		return;
	node->squelched = true;
	cb_ExecSquelchNode(node->lefttree);
	cb_ExecSquelchNode(node->righttree);
}

void
cb_ExecEndNode(CbPlanState *node)
{
	if (!node)
		return;
	cb_ExecEndNode(node->lefttree);
	cb_ExecEndNode(node->righttree);
	if (node->priv)
	{
		node_reset(node);
		free(node->priv);
	}
	free_slot(node->ps_ResultTupleSlot);
	free(node);
}

int
cb_slot_natts(const CbTupleTableSlot *slot)
{
	return slot->tts_nvalid;
}

int
cb_slot_isnull(const CbTupleTableSlot *slot, int attno)
{
	return slot->tts_isnull[attno - 1];
}

int64_t
cb_slot_int64(const CbTupleTableSlot *slot, int attno)
{
	return slot->tts_values[attno - 1];
}

double
cb_slot_float8(const CbTupleTableSlot *slot, int attno)
{
	double		d;

	memcpy(&d, &slot->tts_values[attno - 1], 8);
	return d;
}

int
cb_slot_text(const CbTupleTableSlot *slot, int attno, char *buf, int buflen)
{
	int			i = attno - 1;

	if (slot->tts_isnull[i])
		return snprintf(buf, (size_t) buflen, "NULL");
	switch (slot->tts_types[i])
	{
		case CB_NUMERIC:
		case CB_NUMERIC128:
			return snprintf(buf, (size_t) buflen, "%s", ((CbNumericDatum *) (intptr_t) slot->tts_values[i])->text);
		case CB_FLOAT8:
			return snprintf(buf, (size_t) buflen, "%.17g", cb_slot_float8(slot, attno));
		default:
			return snprintf(buf, (size_t) buflen, "%lld", (long long) slot->tts_values[i]);
	}
}

/* ------------------------------------------------------------------------------------------
 * NCCL interconnect: the MotionIPCLayer-shaped vtable over cbgpu_motion_*
 * ------------------------------------------------------------------------------------------ */
static int
ic_nccl_redistribute(CbInterconnect *ic, CbEState *es, int32_t motion_id, cbgpu_rel *send, const int64_t *counts,
					 const int64_t *offsets, cbgpu_rel **recv)
{
	(void) motion_id;
	GPU(es, cbgpu_motion_redistribute((cbgpu_motion *) ic->priv, send, counts, offsets, recv));
	return CBGPU_OK;
}

static int
ic_nccl_gather(CbInterconnect *ic, CbEState *es, int32_t motion_id, int32_t root, cbgpu_rel *send, int64_t nrows, cbgpu_rel **recv)
{
	(void) motion_id;
	GPU(es, cbgpu_motion_gather((cbgpu_motion *) ic->priv, root, send, nrows, recv));
	return CBGPU_OK;
}

static int
ic_nccl_broadcast(CbInterconnect *ic, CbEState *es, int32_t motion_id, cbgpu_rel *send, int64_t nrows, cbgpu_rel **recv)
{
	(void) motion_id;
	GPU(es, cbgpu_motion_broadcast((cbgpu_motion *) ic->priv, send, nrows, recv));
	return CBGPU_OK;
}

static int
ic_nccl_direct_begin(CbInterconnect *ic, CbEState *es, int32_t motion_id, int32_t ncols, const int32_t *types, const int32_t *dscales,
					 cbgpu_direct_dest *dest)
{
	(void) motion_id;
	(void) es;
	/* not an error for the query: CBGPU_ERR_UNSUPPORTED here (the same on every segment) sends this Motion
	 * down the staged path */
	return cbgpu_motion_direct_begin((cbgpu_motion *) ic->priv, ncols, types, dscales, dest);
}

static int
ic_nccl_direct_end(CbInterconnect *ic, CbEState *es, int32_t motion_id, int32_t local_flags, uint64_t local_nullmask,
				   const int64_t *dev_sent_counts, int64_t *sent_counts, cbgpu_rel **recv, int32_t *outcome)
{
	int			rc;

	(void) motion_id;
	rc = cbgpu_motion_direct_end((cbgpu_motion *) ic->priv, local_flags, local_nullmask, dev_sent_counts, sent_counts, recv, outcome);
	if (rc != CBGPU_OK && es->es_errcode == 0)
		es_fail(es, rc, "%s", cbgpu_last_error(es->es_ctx));
	return rc;
}

static void
ic_nccl_abandon(CbInterconnect *ic, CbEState *es, int32_t motion_id, int32_t after_direct)
{
	(void) motion_id;
	(void) es;
	cbgpu_motion_abandon((cbgpu_motion *) ic->priv, after_direct);
}

CbInterconnect *
cb_interconnect_nccl_create(cbgpu_motion *motion)
{
	CbInterconnect *ic = calloc(1, sizeof(CbInterconnect));

	if (cbgpu_motion_direct_available(motion))
	{
		ic->direct_begin = ic_nccl_direct_begin;
		ic->direct_end = ic_nccl_direct_end;
	}
	ic->name = cbgpu_motion_direct_available(motion) ? "peer-memory windows + nccl" : "nccl";
	ic->nsegs = cbgpu_motion_nranks(motion);
	ic->segindex = cbgpu_motion_rank(motion);
	ic->redistribute = ic_nccl_redistribute;
	ic->gather = ic_nccl_gather;
	ic->broadcast = ic_nccl_broadcast;
	ic->abandon = ic_nccl_abandon;
	ic->priv = motion;
	return ic;
}

void
cb_interconnect_destroy(CbInterconnect *ic)
{
	free(ic);
}

/* ------------------------------------------------------------------------------------------
 * in-process cluster + local interconnect
 * ------------------------------------------------------------------------------------------ */
struct CbCluster
{
	cbgpu_ctx  *ctx;
	int			nsegs;
	CbEState  **estates;
	CbPlanState **roots;
	int			cur;
	int			singleton;		/* top slice runs on segment 0 only                                  */
	char		err[512];
};

CbCluster *
cb_cluster_create(cbgpu_ctx *ctx, int32_t nsegs)
{
	CbCluster  *c = calloc(1, sizeof(CbCluster));

	c->ctx = ctx;
	c->nsegs = nsegs;
	c->estates = calloc((size_t) nsegs, sizeof(CbEState *));
	c->roots = calloc((size_t) nsegs, sizeof(CbPlanState *));
	for (int s = 0; s < nsegs; s++)
	{
		c->estates[s] = cb_CreateExecutorState(ctx, NULL, 0);
		c->estates[s]->es_segindex = s;
		c->estates[s]->es_numsegments = nsegs;
		c->estates[s]->es_cluster = c;
	}
	return c;
}

int
cb_cluster_set_range_table(CbCluster *c, int32_t seg, cbgpu_rel **range_table, int32_t nrels)
{
	CbEState   *es;

	if (seg < 0 || seg >= c->nsegs)
		return CBGPU_ERR_INVALID;
	es = c->estates[seg];
	free(es->es_range_table);
	es->es_nrels = nrels;
	es->es_range_table = calloc((size_t) (nrels ? nrels : 1), sizeof(cbgpu_rel *));
	for (int i = 0; i < nrels; i++)
		es->es_range_table[i] = range_table[i];
	return CBGPU_OK;
}

CbEState *
cb_cluster_estate(CbCluster *c, int32_t seg)
{
	return (seg >= 0 && seg < c->nsegs) ? c->estates[seg] : NULL;
}

static int
slice_is_singleton(const CbPlan *p)
{
	if (!p)
		return 0;
	if (p->type == T_CbMotion)
	{
		int			t = ((const CbMotion *) p)->motionType;

		return t == CB_MOTIONTYPE_GATHER || t == CB_MOTIONTYPE_GATHER_SINGLE;
	}
	return slice_is_singleton(p->lefttree) || slice_is_singleton(p->righttree);
}

int
cb_cluster_init_plan(CbCluster *c, CbPlan *plan)
{
	for (int s = 0; s < c->nsegs; s++)
	{
		c->roots[s] = cb_ExecInitNode(plan, c->estates[s], 0);
		if (!c->roots[s])
		{
			snprintf(c->err, sizeof(c->err), "segment %d: %.480s", s, c->estates[s]->es_errmsg);
			return c->estates[s]->es_errcode ? c->estates[s]->es_errcode : CBGPU_ERR_INVALID;
		}
	}
	c->singleton = slice_is_singleton(plan);
	c->cur = 0;
	return CBGPU_OK;
}

/* find the PlanState of `plan` in a tree */
static CbPlanState *
find_state(CbPlanState *ps, const CbPlan *plan)
{
	CbPlanState *r;

	if (!ps)
		return NULL;
	if (ps->plan == plan)
		return ps;
	r = find_state(ps->lefttree, plan);
	return r ? r : find_state(ps->righttree, plan);
}

static int
cluster_run_motion(CbPlanState *me)
{
	CbCluster  *c = (CbCluster *) me->state->es_cluster;
	CbMotion   *m = (CbMotion *) me->plan;
	int			nsegs = c->nsegs;
	CbPlanState **mps = calloc((size_t) nsegs, sizeof(CbPlanState *));
	cbgpu_rel **send = calloc((size_t) nsegs, sizeof(cbgpu_rel *));
	int64_t    *counts = calloc((size_t) nsegs * (size_t) nsegs, sizeof(int64_t));
	int64_t    *soff = calloc((size_t) nsegs * (size_t) nsegs, sizeof(int64_t));
	int			rc = CBGPU_OK;

	/* sender side on every segment (a sender slice under a Gather receiver's own singleton slice
	 * still runs everywhere; a slice that itself receives from a Gather runs on segment 0 only) */
	for (int s = 0; s < nsegs && rc == CBGPU_OK; s++)
	{
		mps[s] = find_state(c->roots[s], me->plan);
		if (!mps[s])
		{
			rc = es_fail(me->state, CBGPU_ERR_INVALID, "Motion %d has no peer on segment %d", m->motionID, s);
			break;
		}
		if (slice_is_singleton(m->plan.lefttree) && s != 0)
			continue;
		rc = motion_send_side(mps[s], &send[s], counts + (size_t) s * nsegs, soff + (size_t) s * nsegs);
		if (rc && me->state->es_errcode == 0)
			es_fail(me->state, rc, "segment %d: %s", s, mps[s]->state->es_errmsg);
	}
	/* receiver side: destination d gets sender 0's rows, then sender 1's, ... */
	for (int d = 0; d < nsegs && rc == CBGPU_OK; d++)
	{
		int64_t		total = 0;
		cbgpu_rel  *recv = NULL;
		cbgpu_rel  *shape_src = NULL;
		int32_t		types[CBP_MAX_OUT],
					dscales[CBP_MAX_OUT];
		int			ncols;
		int64_t		off = 0;
		NodePriv   *dp = np(mps[d]);

		for (int s = 0; s < nsegs; s++)
		{
			if (!send[s])
				continue;
			shape_src = send[s];
			switch (m->motionType)
			{
				case CB_MOTIONTYPE_HASH:
					total += counts[(size_t) s * nsegs + d];
					break;
				case CB_MOTIONTYPE_GATHER:
					total += d == 0 ? counts[(size_t) s * nsegs] : 0;
					break;
				case CB_MOTIONTYPE_GATHER_SINGLE:
					total += (d == 0 && s == 0) ? counts[(size_t) s * nsegs] : 0;
					break;
				case CB_MOTIONTYPE_BROADCAST:
					total += counts[(size_t) s * nsegs];
					break;
			}
		}
		if (!shape_src)
		{
			rc = es_fail(me->state, CBGPU_ERR_INVALID, "Motion %d: no sender ran", m->motionID);
			break;
		}
		ncols = cbgpu_rel_ncols(shape_src);
		for (int k = 0; k < ncols; k++)
		{
			types[k] = cbgpu_rel_col_type(shape_src, k);
			dscales[k] = cbgpu_rel_col_dscale(shape_src, k);
		}
		rc = cbgpu_rel_create(c->ctx, total, ncols, types, dscales, &recv);
		if (rc)
		{
			es_fail(me->state, rc, "%s", cbgpu_last_error(c->ctx));
			break;
		}
		dp->owned.rels[dp->owned.nrels++] = recv;
		for (int k = 0; k < ncols; k++)
			if (cbgpu_rel_dict_hash_dev(shape_src, k))
				cbgpu_rel_share_dict_hash(recv, k, shape_src, k);
		for (int s = 0; s < nsegs && rc == CBGPU_OK; s++)
		{
			int64_t		n = 0,
						lo = 0;

			if (!send[s])
				continue;
			switch (m->motionType)
			{
				case CB_MOTIONTYPE_HASH:
					n = counts[(size_t) s * nsegs + d];
					lo = soff[(size_t) s * nsegs + d];
					break;
				case CB_MOTIONTYPE_GATHER:
					n = d == 0 ? counts[(size_t) s * nsegs] : 0;
					break;
				case CB_MOTIONTYPE_GATHER_SINGLE:
					n = (d == 0 && s == 0) ? counts[(size_t) s * nsegs] : 0;
					break;
				case CB_MOTIONTYPE_BROADCAST:
					n = counts[(size_t) s * nsegs];
					break;
			}
			if (n > 0)
				rc = cbgpu_rel_copy_rows(recv, off, send[s], lo, n);
			off += n;
			if (rc)
				es_fail(me->state, rc, "%s", cbgpu_last_error(c->ctx));
		}
		dp->recv = recv;
		dp->recv_ready = 1;
		/* every receiver needs the sender-side column shape */
		if (mps[d] != mps[0] || d == 0)
		{
			for (int s = 0; s < nsegs; s++)
				if (send[s])
				{
					NodePriv   *sp = np(mps[s]);

					if (dp->send_nout == 0)
					{
						dp->send_nout = sp->send_nout;
						memcpy(dp->send_pe, sp->send_pe, sizeof(PExpr) * (size_t) sp->send_nout);
					}
					break;
				}
		}
	}
	if (rc == CBGPU_OK)
		rc = cbgpu_sync(c->ctx) == CBGPU_OK ? CBGPU_OK : es_fail(me->state, CBGPU_ERR_CUDA, "%s", cbgpu_last_error(c->ctx));
	free(mps);
	free(send);
	free(counts);
	free(soff);
	return rc;
}

CbTupleTableSlot *
cb_cluster_next(CbCluster *c)
{
	while (c->cur < c->nsegs)
	{
		CbTupleTableSlot *slot;

		if (c->singleton && c->cur != 0)
			break;
		slot = cb_ExecProcNode(c->roots[c->cur]);
		if (c->estates[c->cur]->es_errcode)
		{
			snprintf(c->err, sizeof(c->err), "segment %d: %.480s", c->cur, c->estates[c->cur]->es_errmsg);
			return NULL;
		}
		if (!CbTupIsNull(slot))
			return slot;
		c->cur++;
	}
	return NULL;
}

int32_t
cb_cluster_current_segment(CbCluster *c)
{
	return c->cur;
}

const char *
cb_cluster_error(CbCluster *c)
{
	for (int s = 0; s < c->nsegs; s++)
		if (c->estates[s]->es_errcode && !c->err[0])
			snprintf(c->err, sizeof(c->err), "segment %d: %.480s", s, c->estates[s]->es_errmsg);
	return c->err;
}

void
cb_cluster_end(CbCluster *c)
{
	for (int s = 0; s < c->nsegs; s++)
	{
		cb_ExecEndNode(c->roots[s]);
		c->roots[s] = NULL;
		c->estates[s]->es_errcode = 0;
		c->estates[s]->es_errmsg[0] = 0;
	}
	c->err[0] = 0;
	c->cur = 0;
}

void
cb_cluster_destroy(CbCluster *c)
{
	if (!c)
		return;
	for (int s = 0; s < c->nsegs; s++)
	{
		if (c->roots[s])
			cb_ExecEndNode(c->roots[s]);
		cb_FreeExecutorState(c->estates[s]);
	}
	free(c->estates);
	free(c->roots);
	free(c);
}
