/*
 * hashtable.cu - hash join build (K2) and the stand-alone pair-emitting probe (K3).
 *
 * Build restates MultiExecPrivateHash -> ExecHashGetHashValue -> ExecHashTableInsert
 * (backend/executor/nodeHash.c:167, 2089, 1877): per inner row hash = rotl1-xor of the per-key
 * hash functions (no finaliser), rows with a NULL key are not inserted (strict operators, :2161).
 * The reference chains MinimalTuples off nbuckets = pow2(ntuples / 5) bucket heads; the device
 * table is open addressing with linear probing over slots = hash32 << 32 | inner row id, at load
 * factor <= 0.5, and late-materialises: the inner payload stays in its column arrays and is
 * gathered by row id only for surviving rows.  The slot position uses the same 32-bit hash value
 * the reference computes (bucketno = hashvalue & (nbuckets - 1), nodeHash.c:2233).
 *
 * Probe restates ExecScanHashBucket (nodeHash.c:2255-2308): compare the stored hash value first,
 * then the key equality (hashqualclauses).
 */
#include "common.cuh"

#include <stdlib.h>

struct BuildParams
{
	HtDev		ht;
	int64_t		nrows;
	int		   *flags;			/* [0] duplicate key seen, [1] rows inserted, [2] a key outside the key-in-slot domain */
};

__device__ __forceinline__ bool
ht_row_hash(const HtDev &ht, uint32_t row, uint32_t *hash, int64_t *key0)
{
	uint32_t	h = 0;

	for (int k = 0; k < ht.nkeys; k++)
	{
		if (ht.keynulls[k] && ht.keynulls[k][row])
			return false;
		int64_t		v = cb_load_widen(ht.keydata[k], ht.keytype[k], row);

		if (k == 0)
			*key0 = v;
		h = pg_hash_combine(h, jh_hash_datum(ht.keytype[k], v, ht.keydict[k]), false);
	}
	*hash = h;
	return true;
}

__device__ __forceinline__ bool
ht_keys_equal_rows(const HtDev &ht, uint32_t ra, uint32_t rb)
{
	for (int k = 0; k < ht.nkeys; k++)
		if (cb_load_widen(ht.keydata[k], ht.keytype[k], ra) != cb_load_widen(ht.keydata[k], ht.keytype[k], rb))
			return false;
	return true;
}

__global__ void
k_ht_clear(unsigned long long *slots, size_t n)
{
	size_t		i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
	size_t		stride = (size_t) gridDim.x * blockDim.x;

	for (; i < n; i += stride)
		slots[i] = HT_EMPTY;
}

/* U rows of a thread in flight: their key loads, then their filter words, then their first slots are issued back to back
 * (a row's chain key -> filter word -> slot -> compare-and-swap is four dependent memory operations, the table rarely fits L2) */
template <int HTB_U>
__global__ void __launch_bounds__(256)
k_ht_build(BuildParams p)
{
	const int64_t stride = (int64_t) gridDim.x * blockDim.x;
	int			inserted = 0;
	bool		dup = false;
	bool		outside = false;

	for (int64_t i0 = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i0 < p.nrows; i0 += stride * HTB_U)
	{
		uint32_t	h[HTB_U], pos[HTB_U], w[HTB_U], bits[HTB_U], word[HTB_U];
		unsigned long long cur[HTB_U], e[HTB_U];
		bool		v[HTB_U];

#pragma unroll
		for (int u = 0; u < HTB_U; u++)
		{
			const int64_t i = i0 + (int64_t) u * stride;
			int64_t		key0 = 0;

			h[u] = 0;
			v[u] = i < p.nrows && ht_row_hash(p.ht, (uint32_t) i, &h[u], &key0);
			if (v[u] && !ht_in_batch(p.ht.nbatch, p.ht.batch_shift, p.ht.batch_id, h[u]))
				v[u] = false;		/* another batch's row */
			if (v[u] && p.ht.keyslot && !ht_key_in_domain(p.ht.keyslot, key0))
			{
				outside = true;		/* the host builds the table again with hash values in the slots */
				v[u] = false;
			}
			e[u] = ((unsigned long long) (p.ht.keyslot ? (uint32_t) key0 : h[u]) << 32) | (uint32_t) i;
			pos[u] = h[u] & p.ht.mask;
			bits[u] = ht_bloom_bits(h[u], &w[u], p.ht.bloom_mask);
		}
		if (p.ht.bloom)
		{
#pragma unroll
			for (int u = 0; u < HTB_U; u++)
				word[u] = v[u] ? p.ht.bloom[w[u]] : 0xFFFFFFFFu;
#pragma unroll
			for (int u = 0; u < HTB_U; u++)
				if ((word[u] & bits[u]) != bits[u])
					atomicOr(p.ht.bloom + w[u], bits[u]);
		}
#pragma unroll
		for (int u = 0; u < HTB_U; u++)
			cur[u] = v[u] ? p.ht.slots[pos[u]] : 0;
#pragma unroll
		for (int u = 0; u < HTB_U; u++)
		{
			if (!v[u])
				continue;
			for (;;)
			{
				unsigned long long c = cur[u];

				if (c == HT_EMPTY)
				{
					c = atomicCAS(p.ht.slots + pos[u], HT_EMPTY, e[u]);
					if (c == HT_EMPTY)
						break;
				}
				/* occupied: the same key -> a duplicate on the build side (key-in-slot tables see it in the slot; the others
				 * compare hash values first, then the keys by row id) */
				if (!dup && (uint32_t) (c >> 32) == (uint32_t) (e[u] >> 32) &&
					(p.ht.keyslot || ht_keys_equal_rows(p.ht, (uint32_t) c, (uint32_t) e[u])))
					dup = true;
				pos[u] = (pos[u] + 1) & p.ht.mask;
				cur[u] = p.ht.slots[pos[u]];
			}
			inserted++;
		}
	}
	if (dup)
		atomicExch(p.flags, 1);
	if (outside)
		atomicExch(p.flags + 2, 1);
	/* one atomic per warp for the inserted count */
	for (int o = 16; o; o >>= 1)
		inserted += __shfl_xor_sync(0xffffffffu, inserted, o);
	if ((threadIdx.x & 31) == 0 && inserted)
		atomicAdd(p.flags + 1, inserted);
}

/* one fill of the table: every build row (nbatch <= 1) or the rows of batch `batch` */
static int
ht_fill(cbgpu_hashtable *ht, int batch)
{
	cbgpu_ctx  *ctx = ht->ctx;
	cbgpu_rel  *inner = ht->inner;
	BuildParams p;
	int			h_flags[3];

	ht->d.batch_id = batch;
	if (ht->d.bloom)
		CB_CUDA(ctx, cudaMemsetAsync(ht->d.bloom, 0, ((size_t) ht->d.bloom_mask + 1) * sizeof(uint32_t), ctx->stream));
	for (;;)
	{
		int			blocks = (int) ((ht->nslots + 255) / 256);

		CB_CUDA(ctx, cudaMemsetAsync(ht->d_flags, 0, 3 * sizeof(int), ctx->stream));
		if (blocks > ctx->sm_count * 8)
			blocks = ctx->sm_count * 8;
		k_ht_clear<<<blocks, 256, 0, ctx->stream>>>(ht->d.slots, (size_t) ht->nslots);
		CB_LAUNCHED(ctx, "k_ht_clear");
		p.ht = ht->d;
		p.nrows = inner->nrows;
		p.flags = ht->d_flags;
		if (inner->nrows > 0)
		{
			const int	u = ctx->opt_htb_u;

			blocks = (int) ((inner->nrows + 256 * u - 1) / (256 * u));
			if (blocks > ctx->sm_count * 8)
				blocks = ctx->sm_count * 8;
			if (u == 4)
				k_ht_build<4><<<blocks, 256, 0, ctx->stream>>>(p);
			else if (u == 2)
				k_ht_build<2><<<blocks, 256, 0, ctx->stream>>>(p);
			else
				k_ht_build<1><<<blocks, 256, 0, ctx->stream>>>(p);
			CB_LAUNCHED(ctx, "k_ht_build");
		}
		CB_CUDA(ctx, cudaMemcpyAsync(h_flags, ht->d_flags, sizeof(h_flags), cudaMemcpyDeviceToHost, ctx->stream));
		CB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
		if (h_flags[2] && ht->d.keyslot)
		{
			/* an int8 key beyond 32 bits: the general layout (hash value in the slot, key verified by row id) */
			ht->d.keyslot = 0;
			if (ht->d.bloom)
				CB_CUDA(ctx, cudaMemsetAsync(ht->d.bloom, 0, ((size_t) ht->d.bloom_mask + 1) * sizeof(uint32_t), ctx->stream));
			continue;
		}
		break;
	}
	if (h_flags[0])
		ht->has_dups = 1;
	ht->ninserted = h_flags[1];
	return CBGPU_OK;
}

/* rows per batch of a build side (the batch number of every row's key hash), to size the resident table for the fullest */
__global__ void
k_ht_batch_histogram(HtDev ht, int64_t nrows, unsigned long long *hist)
{
	for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < nrows; i += (int64_t) gridDim.x * blockDim.x)
	{
		uint32_t	h;
		int64_t		key0;

		if (ht_row_hash(ht, (uint32_t) i, &h, &key0))
			atomicAdd(hist + (h >> ht.batch_shift), 1ull);
	}
}

static int
ht_create(cbgpu_ctx *ctx, cbgpu_rel *inner, const int32_t *keycols, int32_t nkeys, int32_t nbatch, cbgpu_hashtable **out)
{
	cbgpu_hashtable *ht;
	int64_t		nslots = 64;
	int64_t		resident_rows = inner->nrows;

	*out = NULL;
	if (nkeys < 1 || nkeys > CBP_MAX_KEYS)
		return cb_fail(ctx, CBGPU_ERR_UNSUPPORTED, "hash join with %s%lld key columns is beyond the GPU path's limit (4)", "", nkeys);
	if (nbatch < 1 || nbatch > 4096 || (nbatch & (nbatch - 1)) != 0)
		return cb_fail(ctx, CBGPU_ERR_INVALID, "hash join with %s%lld batches (a power of two up to 4096 is expected)", "", nbatch);
	ht = (cbgpu_hashtable *) calloc(1, sizeof(cbgpu_hashtable));
	if (!ht)
		return CBGPU_ERR_NOMEM;
	ht->ctx = ctx;
	ht->inner = inner;
	ht->total_rows = inner->nrows;
	ht->d.nkeys = nkeys;
	ht->d.nbatch = nbatch;
	ht->d.batch_shift = 32;
	for (int b = nbatch; b > 1; b >>= 1)
		ht->d.batch_shift--;
	for (int k = 0; k < nkeys; k++)
	{
		int			c = keycols[k];

		if (c < 0 || c >= inner->ncols)
		{
			free(ht);
			return cb_fail(ctx, CBGPU_ERR_INVALID, "cbgpu_ht_build: bad key column%s %lld", "", c);
		}
		if (inner->types[c] == CB_NUMERIC)
		{
			free(ht);
			return cb_fail(ctx, CBGPU_ERR_UNSUPPORTED, "numeric hash join keys (hash_numeric) are not on the GPU path%s", "", 0);
		}
		if ((inner->types[c] == CB_DICT8 || inner->types[c] == CB_DICT32) && !inner->dict_hash[c])
		{
			free(ht);
			return cb_fail(ctx, CBGPU_ERR_INVALID, "dictionary column %s%lld used as a join key without dict hashes", "", c);
		}
		ht->d.keydata[k] = inner->data[c];
		ht->d.keynulls[k] = inner->nulls[c];
		ht->d.keydict[k] = inner->dict_hash[c];
		ht->d.keytype[k] = inner->types[c];
	}
	CB_CUDA(ctx, cudaSetDevice(ctx->device));
	if (nbatch > 1 && inner->nrows > 0)
	{
		/* the fullest batch sizes the table (hash skew: duplicate keys all land in one batch) */
		unsigned long long *d_hist,
				   *h_hist = (unsigned long long *) calloc((size_t) nbatch, sizeof(unsigned long long));
		int			blocks = (int) ((inner->nrows + 255) / 256);

		if (!h_hist)
		{
			free(ht);
			return CBGPU_ERR_NOMEM;
		}
		if (blocks > ctx->sm_count * 8)
			blocks = ctx->sm_count * 8;
		CB_CUDA(ctx, cudaMallocAsync(&d_hist, sizeof(unsigned long long) * (size_t) nbatch, ctx->stream));
		CB_CUDA(ctx, cudaMemsetAsync(d_hist, 0, sizeof(unsigned long long) * (size_t) nbatch, ctx->stream));
		k_ht_batch_histogram<<<blocks, 256, 0, ctx->stream>>>(ht->d, inner->nrows, d_hist);
		CB_LAUNCHED(ctx, "k_ht_batch_histogram");
		CB_CUDA(ctx, cudaMemcpyAsync(h_hist, d_hist, sizeof(unsigned long long) * (size_t) nbatch, cudaMemcpyDeviceToHost, ctx->stream));
		CB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
		CB_CUDA(ctx, cudaFreeAsync(d_hist, ctx->stream));
		resident_rows = 0;
		for (int b = 0; b < nbatch; b++)
			if ((int64_t) h_hist[b] > resident_rows)
				resident_rows = (int64_t) h_hist[b];
		free(h_hist);
	}
	while (nslots < resident_rows * 2)
		nslots <<= 1;
	if (nslots > (1ll << 32))
	{
		free(ht);
		return cb_fail(ctx, CBGPU_ERR_UNSUPPORTED, "hash join build side too large for 32-bit slots%s (%lld rows)", "", inner->nrows);
	}
	ht->nslots = nslots;
	ht->d.mask = (uint32_t) (nslots - 1);
	CB_CUDA(ctx, cudaMallocAsync(&ht->d.slots, (size_t) nslots * sizeof(unsigned long long), ctx->stream));
	CB_CUDA(ctx, cudaMallocAsync(&ht->d_flags, 3 * sizeof(int), ctx->stream));
	/* one integer key: try the key-in-slot layout (int8 keys: as long as every build value lies in [0, 2^32)) */
	if (nkeys == 1 && !ctx->opt_no_keyslot)
		switch (ht->d.keytype[0])
		{
			case CB_INT8:
				ht->d.keyslot = 2;
				break;
			case CB_INT4: case CB_DATE: case CB_DICT8: case CB_DICT32: case CB_BPCHAR1: case CB_BOOL:
				ht->d.keyslot = 1;
				break;
			default:
				break;
		}
	{
		/* ~16 filter bits per build row, at least one cache line */
		int64_t		words = 32;
		const int	div = ctx->opt_bloom_div;	/* rows per 32-bit filter word (CBGPU_BLOOM_DIV, tuning aid), default 2 */

		while (words < resident_rows / div)
			words <<= 1;
		CB_CUDA(ctx, cudaMallocAsync(&ht->d.bloom, (size_t) words * sizeof(uint32_t), ctx->stream));
		ht->d.bloom_mask = (uint32_t) (words - 1);
		ht->built_bytes = nslots * 8 + words * 4;
	}
	*out = ht;
	return CBGPU_OK;
}

extern "C" int
cbgpu_ht_build(cbgpu_ctx *ctx, cbgpu_rel *inner, const int32_t *keycols, int32_t nkeys, cbgpu_hashtable **out)
{
	int			rc = ht_create(ctx, inner, keycols, nkeys, 1, out);

	if (rc == CBGPU_OK)
		rc = ht_fill(*out, 0);
	if (rc != CBGPU_OK && *out)
	{
		cbgpu_ht_free(*out);
		*out = NULL;
	}
	return rc;
}

/* what a single-batch table over `rows` build rows takes on the device (slots at load factor <= 0.5 + the filter):
 * the caller's figure for choosing nbatch against its memory budget (ExecChooseHashTableSize, nodeHash.c:856-1100) */
extern "C" int64_t
cbgpu_ht_bytes_for(int64_t rows)
{
	int64_t		nslots = 64,
				words = 32;

	while (nslots < rows * 2)
		nslots <<= 1;
	while (words < rows / 2)
		words <<= 1;
	return nslots * 8 + words * 4;
}

extern "C" int
cbgpu_ht_build_batched(cbgpu_ctx *ctx, cbgpu_rel *inner, const int32_t *keycols, int32_t nkeys, int32_t nbatch, cbgpu_hashtable **out)
{
	int			rc = ht_create(ctx, inner, keycols, nkeys, nbatch, out);

	/* every batch is built once now: duplicates on the build side decide the join's shape (N:1 or N:M) before the
	 * first probe, and the key-in-slot layout must hold for all batches alike */
	for (int b = 0; b < nbatch && rc == CBGPU_OK; b++)
		rc = ht_fill(*out, b);
	if (rc == CBGPU_OK && (*out)->d.keyslot == 0 && nbatch > 1)
		rc = ht_fill(*out, nbatch - 1);	/* a late fallback to hash-in-slot: the resident batch must use the final layout */
	if (rc != CBGPU_OK && *out)
	{
		cbgpu_ht_free(*out);
		*out = NULL;
	}
	return rc;
}

extern "C" int
cbgpu_ht_nbatch(const cbgpu_hashtable *ht)
{
	return ht->d.nbatch > 1 ? ht->d.nbatch : 1;
}

extern "C" int
cbgpu_ht_load_batch(cbgpu_hashtable *ht, int32_t batch)
{
	if (batch < 0 || batch >= cbgpu_ht_nbatch(ht))
		return cb_fail(ht->ctx, CBGPU_ERR_INVALID, "hash join batch %s%lld out of range", "", batch);
	if (ht->d.nbatch > 1 && ht->d.batch_id == batch)
		return CBGPU_OK;
	return ht_fill(ht, batch);
}

extern "C" void
cbgpu_ht_free(cbgpu_hashtable *ht)
{
	if (!ht)
		return;
	cudaSetDevice(ht->ctx->device);
	cudaFreeAsync(ht->d.slots, ht->ctx->stream);
	if (ht->d.bloom)
		cudaFreeAsync(ht->d.bloom, ht->ctx->stream);
	cudaFreeAsync(ht->d_flags, ht->ctx->stream);
	free(ht);
}

extern "C" int64_t
cbgpu_ht_nrows(const cbgpu_hashtable *ht)
{
	return ht->d.nbatch > 1 ? ht->total_rows : ht->ninserted;
}

extern "C" int
cbgpu_ht_has_duplicates(const cbgpu_hashtable *ht)
{
	return ht->has_dups;
}

extern "C" const uint32_t *
cbgpu_ht_key_dict_hash(const cbgpu_hashtable *ht, int32_t k)
{
	return (k >= 0 && k < ht->d.nkeys) ? ht->d.keydict[k] : NULL;
}

/* ---------------------------------------------------------------------------------------------
 * K3 stand-alone: (outer_idx, inner_idx) pairs for every match (INNER join), two passes:
 * count matches per outer row -> exclusive scan -> write pairs.  Output order is outer-row major,
 * so the pair list is deterministic.
 * --------------------------------------------------------------------------------------------- */
struct ProbeParams
{
	HtDev		ht;
	const void *okey[CBP_MAX_KEYS];
	const uint8_t *onulls[CBP_MAX_KEYS];
	const uint32_t *odict[CBP_MAX_KEYS];
	int32_t		otype[CBP_MAX_KEYS];
	const uint32_t *sel;
	int64_t		n;
	int32_t		left;			/* LEFT join: an outer row without a partner yields one pair (row, 0xFFFFFFFF)  */
	int32_t		presel;			/* every row of sel belongs to the resident batch (k_ht_partition_*): an unmatched
								 * LEFT row is emitted whatever its key hash - a NULL key's hash is not its batch */
	int32_t		sort_matches;	/* the build side has duplicate keys: a row's partners are written in build row order,
								 * not in the order the table's fill happened to place them */
	uint8_t    *matched;		/* RIGHT / FULL join: [inner rows] set to 1 for every build row that found a partner
								 * (HeapTupleHeaderSetMatch, nodeHashjoin.c:560); NULL otherwise */
	int64_t		ninner;
	unsigned long long *counts;	/* [n + 1] match counts, then their exclusive scan                    */
	uint32_t   *out_outer;
	uint32_t   *out_inner;
};

struct KeyHash
{
	uint32_t	h;
	bool		isnull;			/* some key is NULL: h is not the row's hash (the reference's keep_nulls hash is 0) */
};

/* a probe row's key hash (and its key values, into key[]): the pair probe and the partition of the probe side by batch
 * both hash through here, so a row is probed in the pass of the batch it was filed under */
__device__ __forceinline__ KeyHash
pp_key_hash(const ProbeParams &p, uint32_t row, int64_t *key)
{
	KeyHash		r = {0, false};

	for (int k = 0; k < p.ht.nkeys; k++)
	{
		if (p.onulls[k] && p.onulls[k][row])
			r.isnull = true;
		key[k] = cb_load_widen(p.okey[k], p.otype[k], row);
		r.h = pg_hash_combine(r.h, jh_hash_datum(p.otype[k], key[k], p.odict[k]), false);
	}
	return r;
}

/* heapsort of a short run of row ids, in place: deterministic whatever the input, O(n log n) however many duplicates */
__device__ __forceinline__ void
u32_sift_down(uint32_t *a, int64_t root, int64_t end)
{
	uint32_t	v = a[root];

	for (;;)
	{
		int64_t		c = 2 * root + 1;

		if (c >= end)
			break;
		if (c + 1 < end && a[c + 1] > a[c])
			c++;
		if (a[c] <= v)
			break;
		a[root] = a[c];
		root = c;
	}
	a[root] = v;
}

__device__ void
u32_sort(uint32_t *a, int64_t n)
{
	for (int64_t i = n / 2; i-- > 0;)
		u32_sift_down(a, i, n);
	for (int64_t e = n - 1; e > 0; e--)
	{
		uint32_t	t = a[0];

		a[0] = a[e];
		a[e] = t;
		u32_sift_down(a, 0, e);
	}
}

template <bool WRITE>
__global__ void __launch_bounds__(256)
k_ht_probe_pairs(ProbeParams p)
{
	int64_t		i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	int64_t		stride = (int64_t) gridDim.x * blockDim.x;

	for (; i < p.n; i += stride)
	{
		uint32_t	row = p.sel ? p.sel[i] : (uint32_t) i;
		int64_t		key[CBP_MAX_KEYS];
		const KeyHash kh = pp_key_hash(p, row, key);
		const uint32_t h = kh.h;
		bool		isnull = kh.isnull;
		unsigned long long cnt = 0;
		unsigned long long base = WRITE ? p.counts[i] : 0;

		if (!isnull && p.ht.bloom)
		{
			uint32_t	w;
			uint32_t	bits = ht_bloom_bits(h, &w, p.ht.bloom_mask);

			if ((__ldg(p.ht.bloom + w) & bits) != bits)
				isnull = true;		/* certainly absent */
		}
		if (!isnull && p.ht.keyslot && !ht_key_in_domain(p.ht.keyslot, key[0]))
			isnull = true;			/* outside the build side's key domain: no partner */
		if (!isnull && !ht_in_batch(p.ht.nbatch, p.ht.batch_shift, p.ht.batch_id, h))
			isnull = true;			/* multi-batch join: this row belongs to another pass */
		if (!isnull)
		{
			uint32_t	pos = h & p.ht.mask;

			for (;;)
			{
				unsigned long long e = p.ht.slots[pos];

				if (e == HT_EMPTY)
					break;
				if ((uint32_t) (e >> 32) == (p.ht.keyslot ? (uint32_t) key[0] : h))
				{
					uint32_t	irow = (uint32_t) e;
					bool		eq = true;

					for (int k = 0; k < p.ht.nkeys && !p.ht.keyslot; k++)
						if (cb_load_widen(p.ht.keydata[k], p.ht.keytype[k], irow) != key[k])
							eq = false;
					if (eq)
					{
						if (WRITE)
						{
							p.out_outer[base + cnt] = row;
							p.out_inner[base + cnt] = irow;
						}
						else if (p.matched)
							p.matched[irow] = 1;
						cnt++;
					}
				}
				pos = (pos + 1) & p.ht.mask;
			}
		}
		if (WRITE && p.sort_matches && cnt > 1)
			u32_sort(p.out_inner + base, (int64_t) cnt);	/* this thread's own run of pairs: one outer row */
		if (p.left && cnt == 0 && (p.presel || ht_in_batch(p.ht.nbatch, p.ht.batch_shift, p.ht.batch_id, h)))
		{
			/* no partner (or a NULL key, which never has one): the outer row survives with a NULL inner side */
			if (WRITE)
			{
				p.out_outer[base] = row;
				p.out_inner[base] = 0xFFFFFFFFu;
			}
			cnt = 1;
		}
		if (!WRITE)
			p.counts[i] = cnt;
	}
}

/* single-CTA chained exclusive scan (the pair-emitting probe is the general N:M fallback, not a
 * hot kernel; correctness and determinism matter here, not speed) */
__global__ void
k_exclusive_scan_u64(unsigned long long *a, int64_t n)
{
	__shared__ unsigned long long carry;
	__shared__ unsigned long long warp_tot[32];

	if (threadIdx.x == 0)
		carry = 0;
	__syncthreads();
	for (int64_t base = 0; base < n; base += blockDim.x)
	{
		int64_t		i = base + threadIdx.x;
		unsigned long long v = i < n ? a[i] : 0;
		unsigned long long x = v;
		int			lane = threadIdx.x & 31,
					w = threadIdx.x >> 5;

		for (int o = 1; o < 32; o <<= 1)
		{
			unsigned long long y = __shfl_up_sync(0xffffffffu, x, o);

			if (lane >= o)
				x += y;
		}
		if (lane == 31)
			warp_tot[w] = x;
		__syncthreads();
		if (w == 0)
		{
			unsigned long long t = lane < (int) (blockDim.x >> 5) ? warp_tot[lane] : 0;

			for (int o = 1; o < 32; o <<= 1)
			{
				unsigned long long y = __shfl_up_sync(0xffffffffu, t, o);

				if (lane >= o)
					t += y;
			}
			warp_tot[lane] = t;
		}
		__syncthreads();
		unsigned long long prev = (w ? warp_tot[w - 1] : 0) + carry;

		if (i < n)
			a[i] = prev + x - v;
		__syncthreads();
		if (threadIdx.x == blockDim.x - 1)
			carry = prev + x;
		__syncthreads();
	}
	if (threadIdx.x == 0)
		a[n] = carry;
}

/* RIGHT / FULL join: the build rows no probe row matched, each as a pair (0xFFFFFFFF, row) behind the matches
 * (ExecScanHashTableForUnmatched, nodeHash.c:2360; HJ_FILL_INNER_TUPLES, nodeHashjoin.c:676-706).  Rows whose key is NULL
 * were never inserted and never match: they are emitted too (the reference keeps them in the table for this, keep_nulls
 * nodeHash.c:209). */
__global__ void
k_ht_unmatched_count(ProbeParams p)
{
	int64_t		i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	int64_t		stride = (int64_t) gridDim.x * blockDim.x;

	for (; i < p.ninner; i += stride)
		p.counts[p.n + i] = p.matched[i] ? 0 : 1;
}

__global__ void
k_ht_unmatched_write(ProbeParams p)
{
	int64_t		i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	int64_t		stride = (int64_t) gridDim.x * blockDim.x;

	for (; i < p.ninner; i += stride)
		if (!p.matched[i])
		{
			unsigned long long at = p.counts[p.n + i];

			p.out_outer[at] = 0xFFFFFFFFu;
			p.out_inner[at] = (uint32_t) i;
		}
}

/* ---------------------------------------------------------------------------------------------
 * The probe side grouped by hash-join batch (the reference writes outer tuples to per-batch temp files, ExecHashJoinSaveTuple
 * nodeHashjoin.c:1060; here the row ids are grouped once in HBM): ids[off[b] .. off[b+1]) are the rows of batch b, in row
 * order.  A NULL-keyed row belongs to batch 0, as in the pipelined probe (pipeline.cu, keep_nulls hash 0).  Two passes over
 * the key columns: per-CTA histograms (each CTA owns one contiguous range of rows) into a batch-major [nbatch][nCTA] matrix,
 * its exclusive scan, then an in-order scatter of each range.
 * --------------------------------------------------------------------------------------------- */
#define PART_THREADS 256

__device__ __forceinline__ uint32_t
pp_row_batch(const ProbeParams &p, uint32_t row, int32_t batch_shift)
{
	int64_t		key[CBP_MAX_KEYS];
	const KeyHash kh = pp_key_hash(p, row, key);

	return kh.isnull ? 0 : kh.h >> batch_shift;
}

__global__ void __launch_bounds__(PART_THREADS)
k_ht_partition_count(ProbeParams p, int32_t nbatch, int32_t batch_shift, int64_t chunk, unsigned long long *counts)
{
	extern __shared__ uint32_t s_hist[];
	const int64_t lo = (int64_t) blockIdx.x * chunk;
	const int64_t hi = lo + chunk < p.n ? lo + chunk : p.n;

	for (int b = threadIdx.x; b < nbatch; b += blockDim.x)
		s_hist[b] = 0;
	__syncthreads();
	for (int64_t t = lo; t < hi; t += blockDim.x)
	{
		const int64_t i = t + threadIdx.x;
		const uint32_t b = i < hi ? pp_row_batch(p, (uint32_t) i, batch_shift) : 0xFFFFFFFFu;
		const unsigned peers = __match_any_sync(0xffffffffu, b);

		/* one shared atomic per batch present in the warp (few batches: every lane would hit the same word) */
		if (b != 0xFFFFFFFFu && (threadIdx.x & 31) == __ffs(peers) - 1)
			atomicAdd(&s_hist[b], (uint32_t) __popc(peers));
	}
	__syncthreads();
	for (int b = threadIdx.x; b < nbatch; b += blockDim.x)
		counts[(int64_t) b * gridDim.x + blockIdx.x] = s_hist[b];
}

__global__ void __launch_bounds__(PART_THREADS)
k_ht_partition_scatter(ProbeParams p, int32_t nbatch, int32_t batch_shift, int64_t chunk, const unsigned long long *scan,
					   uint32_t *ids, unsigned long long *off)
{
	extern __shared__ uint32_t s_next[];	/* where this CTA's next row of each batch goes */
	const int64_t lo = (int64_t) blockIdx.x * chunk;
	const int64_t hi = lo + chunk < p.n ? lo + chunk : p.n;
	const int	lane = threadIdx.x & 31,
				warp = threadIdx.x >> 5;

	for (int b = threadIdx.x; b < nbatch; b += blockDim.x)
	{
		s_next[b] = (uint32_t) scan[(int64_t) b * gridDim.x + blockIdx.x];
		if (blockIdx.x == 0)
			off[b] = scan[(int64_t) b * gridDim.x];
	}
	if (blockIdx.x == 0 && threadIdx.x == 0)
		off[nbatch] = scan[(int64_t) nbatch * gridDim.x];
	__syncthreads();
	for (int64_t t = lo; t < hi; t += blockDim.x)
	{
		const int64_t i = t + threadIdx.x;
		const bool	v = i < hi;
		const uint32_t b = v ? pp_row_batch(p, (uint32_t) i, batch_shift) : 0xFFFFFFFFu;
		const unsigned peers = __match_any_sync(0xffffffffu, b);
		const int	rank = __popc(peers & ((1u << lane) - 1));

		/* the warps of the tile take their places in order, so every batch's ids stay in row order */
		for (int w = 0; w < PART_THREADS / 32; w++)
		{
			uint32_t	at = 0;

			if (w == warp && v)
				at = s_next[b];
			__syncwarp();
			if (w == warp && v)
			{
				ids[at + rank] = (uint32_t) i;
				if (lane == __ffs(peers) - 1)
					s_next[b] = at + __popc(peers);
			}
			__syncthreads();
		}
	}
}

#define HT_TRY(call) \
	do { \
		int rc__ = (call); \
		if (rc__ != CBGPU_OK) \
			return rc__; \
	} while (0)

/* device scratch of one batched pair probe, freed whatever the outcome */
struct PairsBatchedScratch
{
	unsigned long long *part;	/* [nbatch * nCTA + 1] histogram matrix, then its scan                */
	unsigned long long *off;	/* [nbatch + 1] batch offsets into ids                                */
	uint32_t   *ids;			/* [outer rows] grouped by batch                                     */
	unsigned long long *counts;	/* [max(rows of a batch, inner rows) + 1]                             */
	uint8_t    *matched;		/* [inner rows] RIGHT / FULL                                          */
	unsigned long long *h_off;	/* host copy of off                                                   */
};

/* p.n probe rows (no selection) -> s->ids grouped by batch, h_off[nbatch + 1] their offsets (one read-back) */
static int
ht_partition_probe(cbgpu_ctx *ctx, const ProbeParams &p, int32_t nbatch, int32_t batch_shift, PairsBatchedScratch *s,
				   unsigned long long *h_off)
{
	const int64_t cap = 262144;	/* matrix entries: its single-CTA scan stays well under a millisecond */
	int64_t		g = (p.n + 8 * PART_THREADS - 1) / (8 * PART_THREADS);

	if (g > 2 * (int64_t) ctx->sm_count)
		g = 2 * (int64_t) ctx->sm_count;
	if (g > cap / nbatch)
		g = cap / nbatch;
	if (g < 1)
		g = 1;
	const int64_t chunk = (p.n + g - 1) / g;
	const size_t shmem = sizeof(uint32_t) * (size_t) nbatch;	/* <= 16 KB */

	CB_CUDA(ctx, cudaMallocAsync(&s->part, sizeof(unsigned long long) * (size_t) (nbatch * g + 1), ctx->stream));
	CB_CUDA(ctx, cudaMallocAsync(&s->off, sizeof(unsigned long long) * (size_t) (nbatch + 1), ctx->stream));
	CB_CUDA(ctx, cudaMallocAsync(&s->ids, sizeof(uint32_t) * (size_t) p.n, ctx->stream));
	k_ht_partition_count<<<(unsigned) g, PART_THREADS, shmem, ctx->stream>>>(p, nbatch, batch_shift, chunk, s->part);
	CB_LAUNCHED(ctx, "k_ht_partition_count");
	k_exclusive_scan_u64<<<1, 1024, 0, ctx->stream>>>(s->part, nbatch * g);
	CB_LAUNCHED(ctx, "k_exclusive_scan_u64");
	k_ht_partition_scatter<<<(unsigned) g, PART_THREADS, shmem, ctx->stream>>>(p, nbatch, batch_shift, chunk, s->part, s->ids, s->off);
	CB_LAUNCHED(ctx, "k_ht_partition_scatter");
	CB_CUDA(ctx, cudaMemcpyAsync(h_off, s->off, sizeof(unsigned long long) * (size_t) (nbatch + 1), cudaMemcpyDeviceToHost, ctx->stream));
	CB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	return CBGPU_OK;
}

static int	ht_probe_pairs(cbgpu_ctx *ctx, const cbgpu_hashtable *ht, cbgpu_rel *outer, const int32_t *keycols, int32_t nkeys,
						   const uint32_t *sel, int64_t nsel, int left, int fill_inner, cbgpu_pairs *out);

extern "C" int
cbgpu_ht_probe_pairs_outer(cbgpu_ctx *ctx, const cbgpu_hashtable *ht, cbgpu_rel *outer, const int32_t *keycols, int32_t nkeys,
						   int32_t fill_outer, int32_t fill_inner, cbgpu_pairs *out)
{
	return ht_probe_pairs(ctx, ht, outer, keycols, nkeys, NULL, 0, fill_outer != 0, fill_inner != 0, out);
}

extern "C" int
cbgpu_ht_probe_pairs(cbgpu_ctx *ctx, const cbgpu_hashtable *ht, cbgpu_rel *outer, const int32_t *keycols, int32_t nkeys,
					 const uint32_t *sel, int64_t nsel, cbgpu_pairs *out)
{
	return ht_probe_pairs(ctx, ht, outer, keycols, nkeys, sel, nsel, 0, 0, out);
}

extern "C" int
cbgpu_ht_probe_pairs_left(cbgpu_ctx *ctx, const cbgpu_hashtable *ht, cbgpu_rel *outer, const int32_t *keycols, int32_t nkeys,
						  cbgpu_pairs *out)
{
	return ht_probe_pairs(ctx, ht, outer, keycols, nkeys, NULL, 0, 1, 0, out);
}

/* the probe side's key columns into a zeroed ProbeParams over the table as it is now */
static int
pp_setup(cbgpu_ctx *ctx, const cbgpu_hashtable *ht, cbgpu_rel *outer, const int32_t *keycols, int32_t nkeys, ProbeParams *p)
{
	if (nkeys != ht->d.nkeys)
		return cb_fail(ctx, CBGPU_ERR_INVALID, "cbgpu_ht_probe_pairs: key count mismatch%s %lld", "", nkeys);
	memset(p, 0, sizeof(*p));
	p->ht = ht->d;
	for (int k = 0; k < nkeys; k++)
	{
		int			c = keycols[k];

		if (c < 0 || c >= outer->ncols)
			return cb_fail(ctx, CBGPU_ERR_INVALID, "cbgpu_ht_probe_pairs: bad key column%s %lld", "", c);
		p->okey[k] = outer->data[c];
		p->onulls[k] = outer->nulls[c];
		p->odict[k] = outer->dict_hash[c];
		p->otype[k] = outer->types[c];
	}
	return CBGPU_OK;
}

/* room for `need` pairs in out's arrays (cudaMalloc'd: cbgpu_pairs_free frees them), growing geometrically */
static int
pairs_reserve(cbgpu_ctx *ctx, cbgpu_pairs *out, int64_t *cap, int64_t need)
{
	uint32_t   *o,
			   *in;
	int64_t		ncap = *cap * 2 > need ? *cap * 2 : need;
	cudaError_t e;

	if (need <= *cap)
		return CBGPU_OK;
	if (ncap > 0xFFFFFFF0ll)
		ncap = 0xFFFFFFF0ll;
	CB_CUDA(ctx, cudaMalloc(&o, (size_t) ncap * sizeof(uint32_t)));
	if ((e = cudaMalloc(&in, (size_t) ncap * sizeof(uint32_t))) != cudaSuccess)
		cudaFree(o);
	CB_CUDA(ctx, e);
	if (out->npairs)
	{
		CB_CUDA(ctx, cudaMemcpyAsync(o, out->outer_idx, (size_t) out->npairs * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx->stream));
		CB_CUDA(ctx, cudaMemcpyAsync(in, out->inner_idx, (size_t) out->npairs * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx->stream));
		CB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	}
	if (out->outer_idx)
		cudaFree(out->outer_idx);
	if (out->inner_idx)
		cudaFree(out->inner_idx);
	out->outer_idx = o;
	out->inner_idx = in;
	*cap = ncap;
	return CBGPU_OK;
}

/* p.counts[0 .. p.n) just counted: scan them, make room and append the pairs the write kernel `write` emits */
template <typename W>
static int
pairs_append(cbgpu_ctx *ctx, ProbeParams &p, int64_t nitems, cbgpu_pairs *out, int64_t *cap, W write)
{
	unsigned long long total = 0;

	k_exclusive_scan_u64<<<1, 1024, 0, ctx->stream>>>(p.counts, nitems);
	CB_LAUNCHED(ctx, "k_exclusive_scan_u64");
	CB_CUDA(ctx, cudaMemcpyAsync(&total, p.counts + nitems, sizeof(total), cudaMemcpyDeviceToHost, ctx->stream));
	CB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	if (total + (unsigned long long) out->npairs > 0xFFFFFFF0ull)
		return cb_fail(ctx, CBGPU_ERR_UNSUPPORTED, "join result of %s%lld pairs exceeds the GPU path's 32-bit row ids", "",
					   (long long) (total + (unsigned long long) out->npairs));
	if (total == 0)
		return CBGPU_OK;
	HT_TRY(pairs_reserve(ctx, out, cap, out->npairs + (int64_t) total));
	p.out_outer = out->outer_idx + out->npairs;
	p.out_inner = out->inner_idx + out->npairs;
	HT_TRY(write());
	out->npairs += (int64_t) total;
	return CBGPU_OK;
}

static int
ht_probe_pairs_batched(cbgpu_ctx *ctx, cbgpu_hashtable *ht, cbgpu_rel *outer, const int32_t *keycols, int32_t nkeys, int left,
					   int fill_inner, int (*pending)(void *), void *pending_arg, int64_t *passes, PairsBatchedScratch *s,
					   cbgpu_pairs *out)
{
	ProbeParams p;
	const int32_t nbatch = ht->d.nbatch;
	const int64_t n = outer->nrows;
	const int64_t ninner = fill_inner ? ht->inner->nrows : 0;
	int64_t		maxrows = ninner,
				cap = 0;

	HT_TRY(pp_setup(ctx, ht, outer, keycols, nkeys, &p));
	if (n + ninner == 0)
		return CBGPU_OK;
	s->h_off = (unsigned long long *) calloc((size_t) nbatch + 1, sizeof(unsigned long long));
	if (!s->h_off)
		return CBGPU_ERR_NOMEM;
	if (n > 0)
	{
		p.n = n;
		HT_TRY(ht_partition_probe(ctx, p, nbatch, ht->d.batch_shift, s, s->h_off));
	}
	for (int b = 0; b < nbatch; b++)
		if ((int64_t) (s->h_off[b + 1] - s->h_off[b]) > maxrows)
			maxrows = (int64_t) (s->h_off[b + 1] - s->h_off[b]);
	CB_CUDA(ctx, cudaMallocAsync(&s->counts, (size_t) (maxrows + 1) * sizeof(unsigned long long), ctx->stream));
	if (ninner)
	{
		CB_CUDA(ctx, cudaMallocAsync(&s->matched, (size_t) ninner, ctx->stream));
		CB_CUDA(ctx, cudaMemsetAsync(s->matched, 0, (size_t) ninner, ctx->stream));
	}
	p.counts = s->counts;
	p.matched = s->matched;
	p.left = left;
	p.presel = 1;
	p.sort_matches = ht->has_dups;
	for (int b = 0; b < nbatch; b++)
	{
		const int64_t lo = (int64_t) s->h_off[b];
		const int64_t cnt = (int64_t) (s->h_off[b + 1] - s->h_off[b]);

		if (cnt <= 0 || lo < 0 || lo + cnt > n)
			continue;			/* no probe row in this batch: its build rows need no table (the unmatched pass reads matched) */
		/* HJ_NEED_NEW_BATCH (nodeHashjoin.c:709): the caller's CHECK_FOR_INTERRUPTS between batches */
		if (pending && pending(pending_arg))
			return cb_fail(ctx, CBGPU_ERR_INTERRUPTED, "canceling statement due to user request%s", "");
		HT_TRY(cbgpu_ht_load_batch(ht, b));
		p.ht = ht->d;
		p.sel = s->ids + lo;
		p.n = cnt;

		const int	blocks = (int) ((cnt + 255) / 256 < ctx->sm_count * 8 ? (cnt + 255) / 256 : ctx->sm_count * 8);

		k_ht_probe_pairs<false><<<blocks, 256, 0, ctx->stream>>>(p);
		CB_LAUNCHED(ctx, "k_ht_probe_pairs<count>");
		HT_TRY(pairs_append(ctx, p, cnt, out, &cap, [&]() {
			k_ht_probe_pairs<true><<<blocks, 256, 0, ctx->stream>>>(p);
			CB_LAUNCHED(ctx, "k_ht_probe_pairs<write>");
			return CBGPU_OK;
		}));
		(*passes)++;
	}
	if (ninner)
	{
		/* HJ_FILL_INNER_TUPLES once, after the last batch: build rows of every batch that no probe row matched, NULL-keyed
		 * ones (never inserted in any batch) included */
		const int	iblocks = (int) ((ninner + 255) / 256 < ctx->sm_count * 8 ? (ninner + 255) / 256 : ctx->sm_count * 8);

		p.sel = NULL;
		p.n = 0;
		p.ninner = ninner;
		k_ht_unmatched_count<<<iblocks, 256, 0, ctx->stream>>>(p);
		CB_LAUNCHED(ctx, "k_ht_unmatched_count");
		HT_TRY(pairs_append(ctx, p, ninner, out, &cap, [&]() {
			k_ht_unmatched_write<<<iblocks, 256, 0, ctx->stream>>>(p);
			CB_LAUNCHED(ctx, "k_ht_unmatched_write");
			return CBGPU_OK;
		}));
	}
	return CBGPU_OK;
}

extern "C" int
cbgpu_ht_probe_pairs_batched(cbgpu_ctx *ctx, cbgpu_hashtable *ht, cbgpu_rel *outer, const int32_t *keycols, int32_t nkeys,
							 int32_t fill_outer, int32_t fill_inner, int (*pending)(void *), void *pending_arg, int64_t *passes,
							 cbgpu_pairs *out)
{
	PairsBatchedScratch s;
	int			rc;

	*passes = 0;
	if (ht->d.nbatch <= 1)
	{
		rc = ht_probe_pairs(ctx, ht, outer, keycols, nkeys, NULL, 0, fill_outer != 0, fill_inner != 0, out);
		*passes = rc == CBGPU_OK && outer->nrows > 0;
		return rc;
	}
	memset(out, 0, sizeof(*out));
	memset(&s, 0, sizeof(s));
	rc = ht_probe_pairs_batched(ctx, ht, outer, keycols, nkeys, fill_outer != 0, fill_inner != 0, pending, pending_arg, passes, &s, out);
	cudaSetDevice(ctx->device);
	if (s.part)
		cudaFreeAsync(s.part, ctx->stream);
	if (s.off)
		cudaFreeAsync(s.off, ctx->stream);
	if (s.ids)
		cudaFreeAsync(s.ids, ctx->stream);
	if (s.counts)
		cudaFreeAsync(s.counts, ctx->stream);
	if (s.matched)
		cudaFreeAsync(s.matched, ctx->stream);
	free(s.h_off);
	if (rc != CBGPU_OK)
		cbgpu_pairs_free(out);
	return rc;
}

static int
ht_probe_pairs(cbgpu_ctx *ctx, const cbgpu_hashtable *ht, cbgpu_rel *outer, const int32_t *keycols, int32_t nkeys,
			   const uint32_t *sel, int64_t nsel, int left, int fill_inner, cbgpu_pairs *out)
{
	ProbeParams p;
	int64_t		n = sel ? nsel : outer->nrows;
	unsigned long long total = 0;
	const int64_t ninner = fill_inner ? ht->inner->nrows : 0;

	memset(out, 0, sizeof(*out));
	HT_TRY(pp_setup(ctx, ht, outer, keycols, nkeys, &p));
	p.sel = sel;
	p.n = n;
	p.left = left;
	p.ninner = ninner;
	if (n + ninner == 0)
		return CBGPU_OK;
	if (fill_inner && ht->d.nbatch > 1)
		return cb_fail(ctx, CBGPU_ERR_UNSUPPORTED, "RIGHT / FULL join over a multi-batch table is not implemented%s", "");
	CB_CUDA(ctx, cudaMallocAsync(&p.counts, (size_t) (n + ninner + 1) * sizeof(unsigned long long), ctx->stream));
	if (ninner)
	{
		CB_CUDA(ctx, cudaMallocAsync(&p.matched, (size_t) ninner, ctx->stream));
		CB_CUDA(ctx, cudaMemsetAsync(p.matched, 0, (size_t) ninner, ctx->stream));
	}
	int			blocks = (int) ((n + 255) / 256);
	int			iblocks = (int) ((ninner + 255) / 256);

	if (blocks > ctx->sm_count * 8)
		blocks = ctx->sm_count * 8;
	if (iblocks > ctx->sm_count * 8)
		iblocks = ctx->sm_count * 8;
	if (n)
	{
		k_ht_probe_pairs<false><<<blocks, 256, 0, ctx->stream>>>(p);
		CB_LAUNCHED(ctx, "k_ht_probe_pairs<count>");
	}
	if (ninner)
	{
		k_ht_unmatched_count<<<iblocks, 256, 0, ctx->stream>>>(p);
		CB_LAUNCHED(ctx, "k_ht_unmatched_count");
	}
	k_exclusive_scan_u64<<<1, 1024, 0, ctx->stream>>>(p.counts, n + ninner);
	CB_LAUNCHED(ctx, "k_exclusive_scan_u64");
	CB_CUDA(ctx, cudaMemcpyAsync(&total, p.counts + n + ninner, sizeof(total), cudaMemcpyDeviceToHost, ctx->stream));
	CB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	if (total > 0xFFFFFFF0ull)
	{
		cudaFreeAsync(p.counts, ctx->stream);
		if (p.matched)
			cudaFreeAsync(p.matched, ctx->stream);
		return cb_fail(ctx, CBGPU_ERR_UNSUPPORTED, "join result of %s%lld pairs exceeds the GPU path's 32-bit row ids", "", (long long) total);
	}
	out->npairs = (int64_t) total;
	if (total)
	{
		CB_CUDA(ctx, cudaMalloc(&out->outer_idx, (size_t) total * sizeof(uint32_t)));
		CB_CUDA(ctx, cudaMalloc(&out->inner_idx, (size_t) total * sizeof(uint32_t)));
		p.out_outer = out->outer_idx;
		p.out_inner = out->inner_idx;
		if (n)
		{
			k_ht_probe_pairs<true><<<blocks, 256, 0, ctx->stream>>>(p);
			CB_LAUNCHED(ctx, "k_ht_probe_pairs<write>");
		}
		if (ninner)
		{
			k_ht_unmatched_write<<<iblocks, 256, 0, ctx->stream>>>(p);
			CB_LAUNCHED(ctx, "k_ht_unmatched_write");
		}
	}
	if (p.matched)
		CB_CUDA(ctx, cudaFreeAsync(p.matched, ctx->stream));
	CB_CUDA(ctx, cudaFreeAsync(p.counts, ctx->stream));
	return CBGPU_OK;
}

extern "C" void
cbgpu_pairs_free(cbgpu_pairs *p)
{
	if (!p)
		return;
	if (p->outer_idx)
		cudaFree(p->outer_idx);
	if (p->inner_idx)
		cudaFree(p->inner_idx);
	p->outer_idx = p->inner_idx = NULL;
	p->npairs = 0;
}
