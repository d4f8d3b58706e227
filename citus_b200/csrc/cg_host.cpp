/*
 * cg_host.cpp -- host side of the path above the kernels: device context, chunk-group
 * skipping, staging of column chunks from 8 KB pages into HBM, the scan driver and the
 * result fetch.  Mirrors the reader of backend/columnar/columnar_reader.c, batch-wise.
 */
#include <algorithm>
#include <chrono>
#include <ctype.h>
#include <omp.h>
#include <sched.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "cg_internal.h"

unsigned long long g_cg_launches = 0;

extern "C" uint64_t cg_kernel_launches(void) { return g_cg_launches; }

static CgContext g_ctx;
static bool g_ctx_ready = false;

CgContext *cg_ctx(void)
{
	if (!g_ctx_ready)
	{
		cg_set_error(CG_EINVAL, "cg_init() has not been called");
		return nullptr;
	}
	return &g_ctx;
}

extern "C" int cg_device_count(int *count)
{
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess)
	{
		*count = 0;
		return cg_set_error(CG_ECUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
	}
	*count = n;
	return CG_OK;
}

extern "C" int cg_init(int device)
{
	if (g_ctx_ready)
	{
		if (g_ctx.device != device)
			return cg_set_error(CG_EINVAL, "already initialised on device %d", g_ctx.device);
		return CG_OK;
	}
	CG_CUDA(cudaSetDevice(device));
	cudaDeviceProp prop;
	CG_CUDA(cudaGetDeviceProperties(&prop, device));
	if (prop.major != 10)
		return cg_set_error(CG_EUNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a (B200) only",
							device, prop.major, prop.minor);
	g_ctx.device = device;
	g_ctx.sm_count = prop.multiProcessorCount;
	CG_CUDA(cudaStreamCreateWithFlags(&g_ctx.compute, cudaStreamNonBlocking));
	g_ctx.own_compute = g_ctx.compute;
	{
		/* keep freed blocks of the stream-ordered allocator: the per-scan arenas are reused */
		cudaMemPool_t pool;
		if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess)
		{
			uint64_t keep = UINT64_MAX;
			cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
		}
	}
	CG_CUDA(cudaStreamCreateWithFlags(&g_ctx.copy, cudaStreamNonBlocking));
	CG_CUDA(cudaEventCreate(&g_ctx.ev_a));
	CG_CUDA(cudaEventCreate(&g_ctx.ev_b));
	CG_CUDA(cudaMalloc((void **) &g_ctx.d_stage_err, sizeof(unsigned long long)));
	CG_CUDA(cudaMemset(g_ctx.d_stage_err, 0, sizeof(unsigned long long)));
	const char *t = getenv("CG_STAGE_THREADS");
	int hw = omp_get_num_procs();
	g_ctx.stage_threads = t ? atoi(t) : std::min(hw, 32);
	if (g_ctx.stage_threads < 1) g_ctx.stage_threads = 1;
	const char *b = getenv("CG_PINNED_BLOCK_MB");
	g_ctx.pinned_block_bytes = (size_t) (b ? atoi(b) : 64) << 20;
	g_ctx_ready = true;
	return CG_OK;
}

/* ------------------------------------------------------------------------------ *
 *  NUMA placement.  On a two-socket host a GPU's PCIe root hangs off one socket; host pages
 *  first touched (and staging threads run) on the other socket cross the inter-socket link on
 *  every DMA read.  cg_numa_bind pins the calling thread -- and the threads it creates later --
 *  to the CPUs of the device's NUMA node, read from sysfs; cg_numa_unbind restores the mask.
 * ------------------------------------------------------------------------------ */
static cpu_set_t g_saved_mask;
static bool g_mask_saved = false;

extern "C" int cg_numa_bind(int32_t *node_out)
{
	CgContext *ctx = cg_ctx();
	if (!ctx) return CG_EINVAL;
	if (node_out) *node_out = -1;
	char bus[32] = {0};
	CG_CUDA(cudaDeviceGetPCIBusId(bus, sizeof bus, ctx->device));
	for (char *c = bus; *c; c++) *c = (char) tolower(*c);
	char path[256];
	snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
	FILE *f = fopen(path, "r");
	int node = -1;
	if (f) { if (fscanf(f, "%d", &node) != 1) node = -1; fclose(f); }
	if (node < 0) return CG_OK;                   /* single node or unknown: nothing to do */
	snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
	f = fopen(path, "r");
	if (!f) return CG_OK;
	char list[4096] = {0};
	if (!fgets(list, sizeof list, f)) { fclose(f); return CG_OK; }
	fclose(f);
	cpu_set_t want, have;
	CPU_ZERO(&want);
	if (sched_getaffinity(0, sizeof have, &have) != 0) return CG_OK;
	int n = 0;
	for (char *tok = strtok(list, ",\n"); tok; tok = strtok(nullptr, ",\n"))
	{
		int a = 0, b = 0;
		int k = sscanf(tok, "%d-%d", &a, &b);
		if (k == 1) b = a;
		if (k < 1) continue;
		for (int c = a; c <= b && c < CPU_SETSIZE; c++)
			if (CPU_ISSET(c, &have)) { CPU_SET(c, &want); n++; }
	}
	if (n == 0) return CG_OK;                     /* the cgroup/cpuset excludes that node: keep what we have */
	if (!g_mask_saved) { g_saved_mask = have; g_mask_saved = true; }
	if (sched_setaffinity(0, sizeof want, &want) != 0) return CG_OK;
	if (node_out) *node_out = node;
	return CG_OK;
}

extern "C" int cg_numa_unbind(void)
{
	if (g_mask_saved) { sched_setaffinity(0, sizeof g_saved_mask, &g_saved_mask); g_mask_saved = false; }
	return CG_OK;
}

int cg_ensure_pinned(CgContext *ctx)
{
	if (ctx->pinned[0]) return CG_OK;
	for (int i = 0; i < CgContext::kPinnedBlocks; i++)
	{
		CG_CUDA(cudaHostAlloc((void **) &ctx->pinned[i], ctx->pinned_block_bytes, cudaHostAllocDefault));
		CG_CUDA(cudaEventCreateWithFlags(&ctx->pinned_free[i], cudaEventDisableTiming));
	}
	return CG_OK;
}

extern "C" int cg_synchronize(void)
{
	CgContext *ctx = cg_ctx();
	if (!ctx) return CG_EINVAL;
	CG_CUDA(cudaStreamSynchronize(ctx->copy));
	CG_CUDA(cudaStreamSynchronize(ctx->compute));
	return CG_OK;
}

extern "C" int cg_set_stream(void *cuda_stream)
{
	CgContext *ctx = cg_ctx();
	if (!ctx) return CG_EINVAL;
	CG_CUDA(cudaStreamSynchronize(ctx->compute));
	ctx->compute = cuda_stream ? (cudaStream_t) cuda_stream : ctx->own_compute;
	return CG_OK;
}

int cg_prof_mark(CgContext *ctx, cudaStream_t stream)
{
	if (!ctx->profiling) return CG_OK;
	if (ctx->prof_used == ctx->prof_events.size())
	{
		cudaEvent_t e;
		CG_CUDA(cudaEventCreate(&e));
		ctx->prof_events.push_back(e);
	}
	CG_CUDA(cudaEventRecord(ctx->prof_events[ctx->prof_used++], stream));
	return CG_OK;
}

extern "C" int cg_profile_begin(void)
{
	CgContext *ctx = cg_ctx();
	if (!ctx) return CG_EINVAL;
	ctx->profiling = true;
	ctx->prof_used = 0;
	return CG_OK;
}

extern "C" int cg_profile_collect(int32_t *launches, double *total_ms, double *max_ms)
{
	CgContext *ctx = cg_ctx();
	if (!ctx) return CG_EINVAL;
	ctx->profiling = false;
	double total = 0, mx = 0;
	size_t n = ctx->prof_used / 2;
	for (size_t i = 0; i < n; i++)
	{
		CG_CUDA(cudaEventSynchronize(ctx->prof_events[2 * i + 1]));
		float ms = 0;
		CG_CUDA(cudaEventElapsedTime(&ms, ctx->prof_events[2 * i], ctx->prof_events[2 * i + 1]));
		total += ms;
		if (ms > mx) mx = ms;
	}
	if (launches) *launches = (int32_t) n;
	if (total_ms) *total_ms = total;
	if (max_ms) *max_ms = mx;
	ctx->prof_used = 0;
	return CG_OK;
}

extern "C" void cg_shutdown(void)
{
	if (!g_ctx_ready) return;
	cudaStreamSynchronize(g_ctx.copy);
	cudaStreamSynchronize(g_ctx.compute);
	for (int i = 0; i < CgContext::kPinnedBlocks; i++)
	{
		if (g_ctx.pinned[i]) cudaFreeHost(g_ctx.pinned[i]);
		if (g_ctx.pinned_free[i]) cudaEventDestroy(g_ctx.pinned_free[i]);
		g_ctx.pinned[i] = nullptr; g_ctx.pinned_free[i] = nullptr;
	}
	cudaEventDestroy(g_ctx.ev_a); cudaEventDestroy(g_ctx.ev_b);
	cudaFree(g_ctx.d_stage_err); g_ctx.d_stage_err = nullptr;
	cudaFree(g_ctx.zstd_scratch); g_ctx.zstd_scratch = nullptr; g_ctx.zstd_scratch_bytes = 0;
	for (int i = 0; i < CgContext::kDmaDepth; i++)
	{
		for (CgContext::DevBuf *b : {&g_ctx.slot_arena[i], &g_ctx.slot_raw[i], &g_ctx.slot_meta[i]})
		{
			cudaFree(b->p);
			b->p = nullptr; b->cap = 0;
		}
		if (g_ctx.meta_pinned[i]) cudaFreeHost(g_ctx.meta_pinned[i]);
		g_ctx.meta_pinned[i] = nullptr; g_ctx.meta_cap[i] = 0;
		if (g_ctx.dma_done[i]) cudaEventDestroy(g_ctx.dma_done[i]);
		g_ctx.dma_done[i] = nullptr;
	}
	for (int i = 0; i < CgContext::kDmaDepth; i++) { if (g_ctx.decode_stream[i]) cudaStreamDestroy(g_ctx.decode_stream[i]); g_ctx.decode_stream[i] = nullptr; }
	for (int i = 0; i < CgContext::kDmaDepth; i++) { if (g_ctx.decoded[i]) cudaEventDestroy(g_ctx.decoded[i]); g_ctx.decoded[i] = nullptr; }
	if (g_ctx.dma_copied) cudaEventDestroy(g_ctx.dma_copied);
	g_ctx.dma_copied = nullptr;
	for (cudaEvent_t e : g_ctx.prof_events) cudaEventDestroy(e);
	g_ctx.prof_events.clear();
	cudaStreamDestroy(g_ctx.copy); cudaStreamDestroy(g_ctx.own_compute);
	g_ctx_ready = false;
}

/* ------------------------------------------------------------------------------ *
 *  K2: chunk-group skipping.
 * ------------------------------------------------------------------------------ */
static int datum_cmp(int type_class, int64_t a, int64_t b)
{
	if (type_class == CG_TYPE_FLOAT)
	{
		double x, y;
		memcpy(&x, &a, 8); memcpy(&y, &b, 8);
		bool xn = x != x, yn = y != y;
		if (xn || yn) return (int) xn - (int) yn;
		return (x > y) - (x < y);
	}
	return (a > b) - (a < b);
}

/*
 * [PG] predicate_refuted_by(base constraint, WHERE list) for an AND-list of
 * "col <op> const": the chunk's (col >= min AND col <= max) is refuted when one conjunct
 * on that column contradicts either half (backend/columnar/columnar_reader.c:1132-1187,
 * 1234-1260, 1358-1384).  A chunk without min/max (all NULL) is never skipped.
 */
static bool atom_refuted(const CgSkipNode &node, int type_class, const CgQual &q)
{
	int64_t k = q.konst;
	int cmin = datum_cmp(type_class, node.min_value, k);
	int cmax = datum_cmp(type_class, node.max_value, k);
	switch (q.op)
	{
		case CG_OP_LT: return cmin >= 0;
		case CG_OP_LE: return cmin > 0;
		case CG_OP_EQ: return cmin > 0 || cmax < 0;
		case CG_OP_GE: return cmax < 0;
		case CG_OP_GT: return cmax <= 0;
		default: return false;   /* <> refutes nothing */
	}
}

/* is the chunk's base constraint on column `col` refuted by the WHERE tree?  The implicit AND-list and an
 * AND node are refuted when any arm is, an OR node when every arm is; an atom on another column is never
 * refuted by this column's range (the reference tests one column's constraint at a time). */
static bool chunk_refuted(const CgSkipNode &node, int type_class, int col, const CgScanDesc *d)
{
	if (!node.has_minmax) return false;
	if (d->nqual_expr == 0)
	{
		for (int q = 0; q < d->nquals; q++)
			if (d->quals[q].column == col && atom_refuted(node, type_class, d->quals[q])) return true;
		return false;
	}
	uint32_t st = 0;
	for (int i = 0; i < d->nqual_expr; i++)
	{
		int t = d->qual_expr[i];
		if (t >= 0) st = (st << 1) | (uint32_t) (d->quals[t].column == col && atom_refuted(node, type_class, d->quals[t]));
		else
		{
			uint32_t b = st & 1u, a = (st >> 1) & 1u;
			st = ((st >> 2) << 1) | (t == CG_QX_AND ? (a | b) : (a & b));
		}
	}
	return st & 1u;
}

static int stripe_chunk_mask(const CgStripe &s, const CgSkipNode *nodes, const CgColumnDesc *columns, int natts,
							 const CgScanDesc *d, uint8_t *mask, int64_t *filtered)
{
	for (uint32_t k = 0; k < s.chunk_count; k++) mask[k] = 1;
	if (!d->enable_qual_pushdown || d->nquals == 0) return CG_OK;
	bool has_qual[256] = {false};
	for (int q = 0; q < d->nquals; q++) has_qual[d->quals[q].column] = true;
	for (int c = 0; c < natts && c < 256; c++)      /* whereClauseVars, in attribute order */
	{
		if (!has_qual[c]) continue;
		/* a column added after the stripe was written has no skip nodes: the reference gives it zeroed
		 * nodes with hasMinMax = false (ReadStripeSkipList, columnar_metadata.c:753-760), which refute nothing */
		if ((uint32_t) c >= s.column_count) continue;
		for (uint32_t k = 0; k < s.chunk_count; k++)
		{
			const CgSkipNode &node = nodes[s.skipnode_base + (uint32_t) c * s.chunk_count + k];
			if (mask[k] && chunk_refuted(node, columns[c].type_class, c, d))
			{
				mask[k] = 0;
				(*filtered)++;
			}
		}
	}
	return CG_OK;
}

static int validate_relation(const CgRelation *rel)
{
	if (!rel || !rel->columns || (rel->nstripes > 0 && (!rel->pages || !rel->stripes || !rel->nodes)))
		return cg_set_error(CG_EINVAL, "NULL relation field");
	if (rel->nstripes < 0 || rel->nnodes < 0) return cg_set_error(CG_EINVAL, "negative count");
	if (rel->natts <= 0 || rel->natts > 256) return cg_set_error(CG_EUNSUPPORTED, "natts %d", rel->natts);
	for (int i = 0; i < rel->nstripes; i++)
	{
		const CgStripe &s = rel->stripes[i];
		if ((int) s.column_count > rel->natts)
			return cg_set_error(CG_ECORRUPT, "stripe %d has %u columns, relation %d", i, s.column_count, rel->natts);
		if ((uint64_t) s.skipnode_base + (uint64_t) s.column_count * s.chunk_count > (uint64_t) rel->nnodes)
			return cg_set_error(CG_ECORRUPT, "stripe %d: skip list exceeds node array", i);
		if (s.file_offset < CG_FIRST_LOGICAL_OFFSET)
			return cg_set_error(CG_ECORRUPT, "stripe %d: invalid logical offset %llu", i, (unsigned long long) s.file_offset);
	}
	return CG_OK;
}

extern "C" int cg_selected_chunk_mask(const CgRelation *rel, int32_t stripe_index, const CgScanDesc *desc,
									  uint8_t *mask, int64_t *filtered)
{
	int rc = validate_relation(rel);
	if (rc) return rc;
	if (stripe_index < 0 || stripe_index >= rel->nstripes) return cg_set_error(CG_EINVAL, "stripe index");
	int64_t f = 0;
	rc = stripe_chunk_mask(rel->stripes[stripe_index], rel->nodes, rel->columns, rel->natts, desc, mask, &f);
	if (filtered) *filtered = f;
	return rc;
}

/* interval arithmetic over the skip lists of the chunk groups that survive skipping */
extern "C" int cg_relation_bounds(const CgRelation *rel, const CgScanDesc *desc, int64_t *key_min, int64_t *key_max,
								  int64_t *term_abs_bound, int64_t *rows)
{
	int rc = validate_relation(rel);
	if (rc) return rc;
	std::vector<int64_t> cmin(rel->natts, INT64_MAX), cmax(rel->natts, INT64_MIN);
	std::vector<uint8_t> unknown(rel->natts, 0);
	int64_t nrows = 0;
	std::vector<uint8_t> mask;
	for (int si = 0; si < rel->nstripes; si++)
	{
		const CgStripe &s = rel->stripes[si];
		mask.resize(s.chunk_count);
		int64_t f = 0;
		stripe_chunk_mask(s, rel->nodes, rel->columns, rel->natts, desc, mask.data(), &f);
		for (uint32_t k = 0; k < s.chunk_count; k++)
		{
			if (!mask[k]) continue;
			nrows += (int64_t) rel->nodes[s.skipnode_base + k].row_count;
			for (uint32_t c = 0; c < s.column_count; c++)
			{
				const CgSkipNode &n = rel->nodes[s.skipnode_base + c * s.chunk_count + k];
				if (rel->columns[c].type_class == CG_TYPE_FLOAT) { unknown[c] = 1; continue; }
				if (!n.has_minmax)
				{
					/* all NULL chunk contributes no values */
					if (n.decompressed_size != 0) unknown[c] = 1;
					continue;
				}
				cmin[c] = std::min(cmin[c], n.min_value);
				cmax[c] = std::max(cmax[c], n.max_value);
			}
		}
	}
	if (rows) *rows = nrows;
	if (key_min && key_max)
	{
		*key_min = 0; *key_max = -1;
		if (desc->ngroup_cols == 1)
		{
			int c = desc->group_cols[0];
			if (!unknown[c] && cmin[c] <= cmax[c]) { *key_min = cmin[c]; *key_max = cmax[c]; }
		}
		if (desc->ngroup_cols == 2)
		{
			/* per-column bounds packed like the key (low 32 bits: first column) */
			int c0 = desc->group_cols[0], c1 = desc->group_cols[1];
			if (!unknown[c0] && !unknown[c1] && cmin[c0] <= cmax[c0] && cmin[c1] <= cmax[c1])
			{
				*key_min = (int64_t) ((uint64_t) (uint32_t) cmin[c0] | ((uint64_t) (uint32_t) cmin[c1] << 32));
				*key_max = (int64_t) ((uint64_t) (uint32_t) cmax[c0] | ((uint64_t) (uint32_t) cmax[c1] << 32));
			}
		}
	}
	if (term_abs_bound)
		for (int a = 0; a < desc->naggs; a++)
		{
			const CgAggSpec &s = desc->aggs[a];
			term_abs_bound[a] = 0;
			if (s.kind != CG_AGG_SUM || s.is_float) continue;
			__int128 bound = 1;
			bool ok = true;
			for (int f = 0; f < s.nfactors && ok; f++)
			{
				int c = s.column[f];
				if (unknown[c]) { ok = false; break; }
				if (cmin[c] > cmax[c]) { bound = 0; continue; }   /* no values at all */
				__int128 lo = (__int128) s.a[f] + (__int128) s.b[f] * cmin[c];
				__int128 hi = (__int128) s.a[f] + (__int128) s.b[f] * cmax[c];
				__int128 m = std::max(lo < 0 ? -lo : lo, hi < 0 ? -hi : hi);
				bound *= m;
				if (bound > ((__int128) 1 << 62)) ok = false;
			}
			if (ok) term_abs_bound[a] = bound == 0 ? 1 : (int64_t) bound;
		}
	return CG_OK;
}

/* ------------------------------------------------------------------------------ *
 *  R1/R4: staging.  ColumnarStorageRead (columnar_storage.c:463-492) copies `amount`
 *  bytes at a logical offset out of consecutive pages, one memcpy per page, after
 *  checking pd_lower (ReadFromBlock :669-689).
 * ------------------------------------------------------------------------------ */
static int storage_read(const uint8_t *pages, uint64_t nblocks, uint64_t logical, uint8_t *out, uint64_t amount)
{
	uint64_t done = 0;
	while (done < amount)
	{
		uint64_t L = logical + done;
		uint64_t blockno = L / CG_BYTES_PER_PAGE;
		uint32_t offset = CG_PAGE_HEADER + (uint32_t) (L % CG_BYTES_PER_PAGE);
		uint64_t n = std::min<uint64_t>(amount - done, CG_BLCKSZ - offset);
		if (blockno >= nblocks) return -1;
		const uint8_t *page = pages + blockno * CG_BLCKSZ;
		uint16_t pd_lower;
		memcpy(&pd_lower, page + 12, 2);
		if (pd_lower < offset + n) return -1;
		memcpy(out + done, page + offset, n);
		done += n;
	}
	return 0;
}

static inline uint64_t pad16(uint64_t x) { return (x + 15) & ~15ull; }

struct StageItem   /* one (chunk group, staged column) */
{
	uint64_t exists_logical, value_logical;
	uint64_t wire_value_off;            /* arena slot of the on-disk value bytes (compressed or not) */
	uint32_t exists_len, value_len;     /* on-disk lengths */
};

struct StagePlan
{
	std::vector<DevChunkCol> cols;      /* [ncg][nstaged] */
	std::vector<StageItem> items;
	std::vector<uint32_t> cg_rows;
	std::vector<uint64_t> cg_begin;     /* arena offset where each chunk group starts; [ncg+1] */
	std::vector<DecodeItem> decode;     /* compressed value streams, in chunk-group order */
	std::vector<uint32_t> dec_first;    /* first decode item of each chunk group; [ncg+1] */
	std::vector<VarlenaItem> varlena;   /* varlena value streams to decode to fixed width, in chunk-group order */
	std::vector<uint32_t> vl_first;     /* first varlena item of each chunk group; [ncg+1] */
	std::vector<uint32_t> stream_bytes; /* per (chunk group, staged column): uncompressed value-stream bytes (the algorithmic bytes) */
	uint64_t wire_bytes = 0;            /* the chunk-group regions: what travels host -> device */
	uint64_t arena_bytes = 0;           /* wire_bytes + the decompressed value slots */
	uint64_t rows = 0;
	bool any_nulls = false;
};

/* lays out the arena for the chunk groups picked by `select` (NULL = all) */
static int plan_staging(const CgRelation *rel, const std::vector<int32_t> &staged,
						const std::vector<std::vector<uint8_t>> *select, StagePlan *sp)
{
	uint64_t off = 0;
	size_t ns = staged.size();
	for (int si = 0; si < rel->nstripes; si++)
	{
		const CgStripe &s = rel->stripes[si];
		for (uint32_t k = 0; k < s.chunk_count; k++)
		{
			if (select && !(*select)[si][k]) continue;
			uint32_t rows = (uint32_t) rel->nodes[s.skipnode_base + k].row_count;
			sp->cg_begin.push_back(off);
			sp->dec_first.push_back((uint32_t) sp->decode.size());
			sp->vl_first.push_back((uint32_t) sp->varlena.size());
			sp->cg_rows.push_back(rows);
			sp->rows += rows;
			for (size_t j = 0; j < ns; j++)
			{
				int c = staged[j];
				DevChunkCol d;
				StageItem it;
				memset(&d, 0, sizeof d);
				d.row_count = rows;
				int comp = CG_COMPRESSION_NONE;
				uint64_t rawlen = 0;
				if ((uint32_t) c >= s.column_count)
				{
					/* column added after the stripe was written and without a default: all NULL
					 * (columnar_reader.c:1626-1650) */
					it.exists_logical = it.value_logical = 0;
					it.exists_len = it.value_len = 0;
					d.value_count = 0;
				}
				else
				{
					const CgSkipNode &n = rel->nodes[s.skipnode_base + (uint32_t) c * s.chunk_count + k];
					comp = n.compression_type;
					if (comp != CG_COMPRESSION_NONE && comp != CG_COMPRESSION_LZ4 && comp != CG_COMPRESSION_PGLZ && comp != CG_COMPRESSION_ZSTD)
						return cg_set_error(CG_ECORRUPT, "unexpected compression type: %d", comp);
					if (n.row_count != rows) return cg_set_error(CG_ECORRUPT, "row count mismatch in chunk group");
					if (n.exists_length * 8 < rows) return cg_set_error(CG_ECORRUPT, "insufficient data for reading boolean array");
					int len = rel->columns[c].attlen;
					const bool varlena = len < 0;
					if (varlena)
					{
						if (comp == CG_COMPRESSION_NONE && n.value_length != n.decompressed_size)
							return cg_set_error(CG_ECORRUPT, "value stream length mismatch in a varlena chunk");
					}
					else if (n.decompressed_size % len != 0 || n.decompressed_size / len > rows ||
						(comp == CG_COMPRESSION_NONE && n.value_length != n.decompressed_size))
						return cg_set_error(CG_ECORRUPT, "value stream of %llu bytes does not fit %u rows of %d bytes",
											(unsigned long long) n.decompressed_size, rows, len);
					if (n.value_length > UINT32_MAX - 64 || n.decompressed_size > UINT32_MAX - 64)
						return cg_set_error(CG_EUNSUPPORTED, "chunk buffer of %llu bytes", (unsigned long long) n.value_length);
					rawlen = n.decompressed_size;
					it.exists_logical = s.file_offset + n.exists_offset;
					it.value_logical = s.file_offset + n.value_offset;
					it.exists_len = (uint32_t) n.exists_length;
					it.value_len = (uint32_t) n.value_length;
					if (varlena)
					{
						/* the number of values of a varlena chunk is the number of set exists bits (NULL rows occupy no bytes) */
						std::vector<uint8_t> bits(n.exists_length);
						if (n.exists_length && storage_read(rel->pages, rel->nblocks, it.exists_logical, bits.data(), n.exists_length))
							return cg_set_error(CG_ECORRUPT, "attempt to read columnar data past pd_lower / end of relation");
						uint32_t nn = 0;
						for (uint32_t r = 0; r < rows; r++) nn += (bits[r >> 3] >> (r & 7)) & 1u;
						d.value_count = nn;
					}
					else
						d.value_count = (uint32_t) (n.decompressed_size / len);
				}
				d.exists_off = off; off += pad16(std::max<uint64_t>((rows + 7) / 8, it.exists_len)) + 16;
				d.values_off = off; off += pad16(it.value_len) + 16;
				it.wire_value_off = d.values_off;
				if (comp != CG_COMPRESSION_NONE)
				{
					/* dst is assigned below, behind the chunk-group regions */
					DecodeItem di;
					di.src = it.wire_value_off; di.dst = sp->cols.size();
					di.comp_len = it.value_len; di.raw_len = (uint32_t) rawlen;
					di.padded = (uint32_t) (pad16(rawlen) + 16); di.kind = (uint32_t) comp;
					sp->decode.push_back(di);
				}
				if (d.value_count != rows)
				{
					d.rank_off = off; off += pad16(4ull * ((rows + 63) / 64));
					sp->any_nulls = true;
				}
				if ((uint32_t) c < s.column_count && cg_is_varlena(rel->columns[c]))
				{
					/* src / dst are assigned below: src = the on-disk stream or its decompressed slot */
					VarlenaItem vi;
					vi.src = comp != CG_COMPRESSION_NONE ? ~0ull : it.wire_value_off; vi.dst = sp->cols.size();
					vi.raw_len = (uint32_t) rawlen; vi.count = d.value_count;
					vi.kind = (uint32_t) cg_type_class(rel->columns[c]); vi.scale = (uint32_t) cg_type_scale(rel->columns[c]);
					sp->varlena.push_back(vi);
				}
				sp->stream_bytes.push_back((uint32_t) rawlen);
				sp->cols.push_back(d);
				sp->items.push_back(it);
			}
		}
	}
	sp->cg_begin.push_back(off);
	sp->dec_first.push_back((uint32_t) sp->decode.size());
	sp->vl_first.push_back((uint32_t) sp->varlena.size());
	sp->wire_bytes = off;
	for (DecodeItem &di : sp->decode)
	{
		DevChunkCol &d = sp->cols[di.dst];
		d.values_off = off;
		di.dst = off;
		off += di.padded;
	}
	for (VarlenaItem &vi : sp->varlena)
	{
		/* the decoded fixed-width array; the stream it is decoded from is where values_off pointed so far */
		DevChunkCol &d = sp->cols[vi.dst];
		if (vi.src == ~0ull) vi.src = d.values_off;
		d.values_off = off;
		vi.dst = off;
		off += pad16((uint64_t) vi.count * (vi.kind == CG_TYPE_NUMERIC ? 8 : 1)) + 16;
	}
	sp->arena_bytes = off;
	return CG_OK;
}

/* fills [cg0, cg1) of the plan into a host buffer laid out like the arena from cg_begin[cg0] */
static int fill_block(const CgRelation *rel, const StagePlan &sp, size_t ns, uint64_t cg0, uint64_t cg1,
					  uint8_t *host, int nthreads)
{
	uint64_t base = sp.cg_begin[cg0];
	int failed = 0;
#pragma omp parallel for schedule(dynamic, 4) num_threads(nthreads)
	for (int64_t g = (int64_t) cg0; g < (int64_t) cg1; g++)
	{
		for (size_t j = 0; j < ns; j++)
		{
			const DevChunkCol &d = sp.cols[g * ns + j];
			const StageItem &it = sp.items[g * ns + j];
			uint8_t *ex = host + (d.exists_off - base);
			uint8_t *va = host + (it.wire_value_off - base);
			uint64_t exspan = it.wire_value_off - d.exists_off;
			memset(ex + (it.exists_len & ~15ull), 0, exspan - (it.exists_len & ~15ull));
			if (it.exists_len && storage_read(rel->pages, rel->nblocks, it.exists_logical, ex, it.exists_len)) failed = 1;
			uint64_t vaspan = pad16(it.value_len) + 16;
			memset(va + (it.value_len & ~15ull), 0, vaspan - (it.value_len & ~15ull));
			if (it.value_len && storage_read(rel->pages, rel->nblocks, it.value_logical, va, it.value_len)) failed = 1;
		}
	}
	if (failed) return cg_set_error(CG_ECORRUPT, "attempt to read columnar data past pd_lower / end of relation");
	return CG_OK;
}

/*
 * Streams the planned chunk groups to the device arena through the pinned ring:
 * host threads de-frame pages into pinned block b while block b-1 is in flight on the
 * copy stream.  after_block(cg0, cg1) is called (on the host) once the H2D of that
 * range has been enqueued; it may enqueue kernels on ctx->compute after making that
 * stream wait on the returned event.
 */
template <typename F>
static int stream_to_device(CgContext *ctx, const CgRelation *rel, const StagePlan &sp, size_t ns,
							uint8_t *d_arena, F after_block)
{
	int rc = cg_ensure_pinned(ctx);
	if (rc) return rc;
	uint64_t ncg = sp.cg_rows.size();
	uint64_t cg = 0;
	int slot = 0;
	static int trace = -1;
	if (trace < 0) { const char *e = getenv("CG_TRACE"); trace = (e && atoi(e)) ? 1 : 0; }
	double t_wait = 0, t_fill = 0, t_enq = 0;
	uint64_t nblk = 0;
	auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
	double t_begin = now();
	while (cg < ncg)
	{
		uint64_t cg1 = cg;
		while (cg1 < ncg && sp.cg_begin[cg1 + 1] - sp.cg_begin[cg] <= ctx->pinned_block_bytes) cg1++;
		if (cg1 == cg)
			return cg_set_error(CG_EUNSUPPORTED, "one chunk group (%llu bytes) exceeds the pinned block size",
								(unsigned long long) (sp.cg_begin[cg + 1] - sp.cg_begin[cg]));
		double t0 = now();
		CG_CUDA(cudaEventSynchronize(ctx->pinned_free[slot]));
		double t1 = now();
		rc = fill_block(rel, sp, ns, cg, cg1, ctx->pinned[slot], ctx->stage_threads);
		if (rc) return rc;
		double t2 = now();
		uint64_t bytes = sp.cg_begin[cg1] - sp.cg_begin[cg];
		CG_CUDA(cudaMemcpyAsync(d_arena + sp.cg_begin[cg], ctx->pinned[slot], bytes, cudaMemcpyHostToDevice, ctx->copy));
		CG_CUDA(cudaEventRecord(ctx->pinned_free[slot], ctx->copy));
		rc = after_block(cg, cg1, ctx->pinned_free[slot]);
		if (rc) return rc;
		double t3 = now();
		t_wait += t1 - t0; t_fill += t2 - t1; t_enq += t3 - t2; nblk++;
		cg = cg1;
		slot = (slot + 1) % CgContext::kPinnedBlocks;
	}
	if (trace)
		fprintf(stderr, "[cg] staged %.1f MB in %llu blocks: total %.1f ms (wait-for-slot %.1f, de-frame %.1f = %.1f GB/s, enqueue %.1f)\n",
				sp.wire_bytes / 1e6, (unsigned long long) nblk, (now() - t_begin) * 1e3, t_wait * 1e3, t_fill * 1e3,
				sp.wire_bytes / 1e9 / (t_fill > 0 ? t_fill : 1), t_enq * 1e3);
	return CG_OK;
}

extern "C" int cg_shard_stage(const CgRelation *rel, const int32_t *columns, int32_t ncolumns, CgShard **out)
{
	CgContext *ctx = cg_ctx();
	if (!ctx) return CG_EINVAL;
	int rc = validate_relation(rel);
	if (rc) return rc;
	CgShard *sh = new CgShard();
	sh->natts = rel->natts;
	sh->columns.assign(rel->columns, rel->columns + rel->natts);
	sh->slot_of_att.assign(rel->natts, -1);
	if (columns && ncolumns > 0)
	{
		for (int i = 0; i < ncolumns; i++)
		{
			if (columns[i] < 0 || columns[i] >= rel->natts) { delete sh; return cg_set_error(CG_EINVAL, "column %d", columns[i]); }
			if (sh->slot_of_att[columns[i]] >= 0) continue;
			sh->slot_of_att[columns[i]] = (int32_t) sh->staged.size();
			sh->staged.push_back(columns[i]);
		}
	}
	else
		for (int c = 0; c < rel->natts; c++) { sh->slot_of_att[c] = c; sh->staged.push_back(c); }
	if (sh->staged.size() > 255) { delete sh; return cg_set_error(CG_EUNSUPPORTED, "more than 255 staged columns"); }
	for (int c : sh->staged)
	{
		int l = rel->columns[c].attlen;
		if (l != 1 && l != 2 && l != 4 && l != 8 && !(l == -1 && (cg_type_class(rel->columns[c]) == CG_TYPE_NUMERIC || cg_type_class(rel->columns[c]) == CG_TYPE_BPCHAR1)))
		{ delete sh; return cg_set_error(CG_EUNSUPPORTED, "column %d: attlen %d", c, l); }
	}

	StagePlan sp;
	rc = plan_staging(rel, sh->staged, nullptr, &sp);
	if (rc) { delete sh; return rc; }
	size_t ns = sh->staged.size();
	sh->rows = sp.rows;
	sh->nchunkgroups = sp.cg_rows.size();
	sh->cg_rows = sp.cg_rows;
	sh->h_chunkcols = sp.cols;
	sh->h_stream_bytes = sp.stream_bytes;
	sh->arena_bytes = sp.arena_bytes;
	sh->stripes.assign(rel->stripes, rel->stripes + rel->nstripes);
	sh->nodes.assign(rel->nodes, rel->nodes + rel->nnodes);
	uint64_t first = 0;
	for (int si = 0; si < rel->nstripes; si++) { sh->stripe_first_cg.push_back(first); first += rel->stripes[si].chunk_count; }

	if (cudaMalloc(&sh->d_arena, std::max<uint64_t>(sp.arena_bytes, 16)) != cudaSuccess ||
		cudaMalloc(&sh->d_chunkcols, std::max<size_t>(sp.cols.size(), 1) * sizeof(DevChunkCol)) != cudaSuccess ||
		cudaMalloc(&sh->d_selected, std::max<uint64_t>(sh->nchunkgroups, 1) * sizeof(uint32_t)) != cudaSuccess)
	{
		cg_shard_free(sh);
		return cg_set_error(CG_ENOMEM, "cudaMalloc of %llu bytes for the shard arena failed", (unsigned long long) sp.arena_bytes);
	}
	cudaError_t e = cudaMemcpyAsync(sh->d_chunkcols, sp.cols.data(), sp.cols.size() * sizeof(DevChunkCol), cudaMemcpyHostToDevice, ctx->copy);
	if (e != cudaSuccess) { cg_shard_free(sh); return cg_set_error(CG_ECUDA, "cudaMemcpyAsync: %s", cudaGetErrorString(e)); }
	/* compressed value streams are decoded block by block behind the H2D copies (K7) */
	DecodeItem *d_decode = nullptr;
	VarlenaItem *d_varlena = nullptr;
	if (!sp.decode.empty() || !sp.varlena.empty())
	{
		if ((!sp.decode.empty() && (cudaMalloc(&d_decode, sp.decode.size() * sizeof(DecodeItem)) != cudaSuccess ||
									cudaMemcpy(d_decode, sp.decode.data(), sp.decode.size() * sizeof(DecodeItem), cudaMemcpyHostToDevice) != cudaSuccess)) ||
			(!sp.varlena.empty() && (cudaMalloc(&d_varlena, sp.varlena.size() * sizeof(VarlenaItem)) != cudaSuccess ||
									 cudaMemcpy(d_varlena, sp.varlena.data(), sp.varlena.size() * sizeof(VarlenaItem), cudaMemcpyHostToDevice) != cudaSuccess)) ||
			cudaMemsetAsync(ctx->d_stage_err, 0, sizeof(unsigned long long), ctx->compute) != cudaSuccess)
		{
			cudaFree(d_decode); cudaFree(d_varlena);
			cg_shard_free(sh);
			return cg_set_error(CG_ECUDA, "staging the decode list failed: %s", cudaGetErrorString(cudaGetLastError()));
		}
	}
	rc = stream_to_device(ctx, rel, sp, ns, sh->d_arena, [&](uint64_t cg0, uint64_t cg1, cudaEvent_t copied) -> int {
		uint32_t f = sp.dec_first[cg0], l = sp.dec_first[cg1];
		uint32_t vf = sp.vl_first[cg0], vl = sp.vl_first[cg1];
		if (f == l && vf == vl) return CG_OK;
		CG_CUDA(cudaStreamWaitEvent(ctx->compute, copied, 0));
		int r = CG_OK;
		if (f != l)
			r = cg_launch_decompress(ctx, sh->d_arena, d_decode + f, sp.decode.data() + f, l - f, ctx->d_stage_err, CG_ERRFLAG_DECOMPRESS,
									 ctx->compute);
		/* varlena value streams (decompressed first when they were compressed) -> dense fixed-width arrays */
		if (r == CG_OK && vf != vl)
			r = cg_launch_varlena_decode(ctx, sh->d_arena, d_varlena + vf, vl - vf, ctx->d_stage_err, CG_ERRFLAG_VARLENA, ctx->compute);
		return r;
	});
	if (rc == CG_OK && sp.any_nulls)
	{
		/* rank directories (K1 prefix popcount), once per staged shard */
		cudaError_t e2 = cudaStreamSynchronize(ctx->copy);
		if (e2 != cudaSuccess) rc = cg_set_error(CG_ECUDA, "%s", cudaGetErrorString(e2));
		else rc = cg_launch_rank(ctx, sh->d_arena, sh->d_chunkcols, 0, sp.cols.size(), ctx->compute);
	}
	if (rc == CG_OK)
	{
		cudaError_t e2 = cudaStreamSynchronize(ctx->copy);
		if (e2 == cudaSuccess) e2 = cudaStreamSynchronize(ctx->compute);
		if (e2 != cudaSuccess) rc = cg_set_error(CG_ECUDA, "%s", cudaGetErrorString(e2));
	}
	else
	{
		cudaStreamSynchronize(ctx->copy);
		cudaStreamSynchronize(ctx->compute);
	}
	if (rc == CG_OK && (d_decode || d_varlena))
	{
		unsigned long long flags = 0;
		cudaError_t e2 = cudaMemcpy(&flags, ctx->d_stage_err, sizeof flags, cudaMemcpyDeviceToHost);
		if (e2 != cudaSuccess) rc = cg_set_error(CG_ECUDA, "%s", cudaGetErrorString(e2));
		else if (flags & CG_ERRFLAG_DECOMPRESS) rc = cg_set_error(CG_ECORRUPT, "cannot decompress the buffer");
		else if (flags & CG_ERRFLAG_VARLENA) rc = cg_set_error(CG_EUNSUPPORTED, "a numeric value is NaN, has more fractional digits than the column's scale or "
																					"does not fit 64 bits, or a varlena stream is malformed");
	}
	cudaFree(d_decode); cudaFree(d_varlena);
	if (rc) { cg_shard_free(sh); return rc; }
	*out = sh;
	return CG_OK;
}

extern "C" void cg_shard_free(CgShard *sh)
{
	if (!sh) return;
	cudaFree(sh->d_arena);
	cudaFree(sh->d_chunkcols);
	cudaFree(sh->d_selected);
	delete sh;
}

extern "C" uint64_t cg_shard_device_bytes(const CgShard *sh) { return sh ? sh->arena_bytes : 0; }
extern "C" uint64_t cg_shard_rows(const CgShard *sh) { return sh ? sh->rows : 0; }

/* ------------------------------------------------------------------------------ *
 *  Scan driver.
 * ------------------------------------------------------------------------------ */
static int g_force_general = -1;
static bool cg_force_general(void)
{
	if (g_force_general < 0) { const char *e = getenv("CG_FORCE_GENERAL_KERNEL"); g_force_general = (e && atoi(e)) ? 1 : 0; }
	return g_force_general == 1;
}

/* run-time switches (the same ones the CG_* environment variables set at first use): which kernel family
 * scans -- "jit" 0 = ahead-of-time kernels only, 1 = plan-specialised where no ahead-of-time specialisation
 * applies (default), 2 = always; "force_general" 1 = the interpretive kernels for everything; "lz4_lanes" 1 / 0 = LZ4 value
 * streams are decoded a lane per stream / eight lanes per stream, 2 or < 0 = by launch size (default); "peer_window" 0 = the
 * combine and the repartition exchange stay on NCCL instead of the IPC-mapped peer window (set it on every rank) */
extern "C" int cg_set_option(const char *name, int64_t value)
{
	if (!name) return cg_set_error(CG_EINVAL, "NULL option name");
	if (strcmp(name, "jit") == 0) { cg_jit_set_level((int) value); return CG_OK; }
	if (strcmp(name, "force_general") == 0) { g_force_general = value ? 1 : 0; return CG_OK; }
	if (strcmp(name, "realign_tma") == 0) { cg_realign_set_tma((int) value); return CG_OK; }
	if (strcmp(name, "lz4_lanes") == 0) { cg_decompress_set_lz4_lanes((int) value); return CG_OK; }
	if (strcmp(name, "lz4_lane_warps") == 0) { cg_decompress_set_lz4_lane_warps((int) value); return CG_OK; }
	if (strcmp(name, "peer_window") == 0) { cg_comm_set_peer_window((int) value); return CG_OK; }     /* the same value on every rank */
	return cg_set_error(CG_EINVAL, "unknown option %s", name);
}

static int check_error_flags(CgPartial *p, unsigned long long flags)
{
	if (flags & CG_ERRFLAG_TABLE_FULL)
		return cg_set_error(CG_ETABLEFULL, "group table (%llu slots) is full: retry with a larger expected_groups",
							(unsigned long long) p->capacity);
	if (flags & CG_ERRFLAG_NULL_MULTIKEY)
		return cg_set_error(CG_EUNSUPPORTED, "NULL in a two-column group key");
	if (flags & CG_ERRFLAG_KEY_RANGE)
		return cg_set_error(CG_EINVAL, "group key outside [key_min, key_max] given to cg_partial_create");
	if (flags & CG_ERRFLAG_SUM_BOUND)
		return cg_set_error(CG_EINVAL, "sum argument exceeds term_abs_bound");
	if (flags & CG_ERRFLAG_DECOMPRESS)
		return cg_set_error(CG_ECORRUPT, "cannot decompress the buffer");
	if (flags & CG_ERRFLAG_VARLENA)
		return cg_set_error(CG_EUNSUPPORTED, "a numeric value is NaN, has more fractional digits than the column's scale or does not fit 64 bits, "
											 "or a varlena stream is malformed");
	return CG_OK;
}

/* CG_PACK_DRAIN_EVERY = n restores a drain every n packed launches (A/B measurements) */
static int drain_every(void)
{
	static int v = -2;
	if (v == -2) { const char *e = getenv("CG_PACK_DRAIN_EVERY"); v = e ? atoi(e) : 0; if (v < 0) v = 0; }
	return v;
}

/*
 * Bookkeeping after a scan launch.  Packed words are drained into the wide accumulators when a group could
 * have come near 2^C rows since the last drain: rows scanned since then exceed capacity * 2^C / 32 (uniform
 * keys would be a factor 32 under the limit; a skewed key that still overflows is detected exactly and
 * reported as CG_ERETRY_UNPACKED).  For C2 (1 M groups, C = 16) that is 2 G rows: a 1 B-row query never
 * drains before its result is read, and a combine can ship the 8-byte packed words alone.
 * packed_only = the launch wrote nothing but packed words.
 */
/* a partial that was read (rows decoded straight from its packed words) and is scanned into again: fold the packed words
 * into the wide accumulators first, as a read used to do, so that reads bound what a packed word accumulates */
static int before_scan(CgContext *ctx, CgPartial *p)
{
	if (!p->read_packed_direct) return CG_OK;
	p->read_packed_direct = false;
	return cg_launch_drain(p, ctx->compute);
}

static int after_launch(CgContext *ctx, CgPartial *p, bool used_packed, bool packed_only, uint64_t rows)
{
	if (!(used_packed && packed_only)) p->wide_dirty = true;
	if (!used_packed) return CG_OK;
	p->packed_dirty = true;
	p->launches_since_drain++;
	p->rows_since_drain += rows;
	const int every = drain_every();
	if (every > 0) return p->launches_since_drain >= every ? cg_launch_drain(p, ctx->compute) : CG_OK;
	const double limit = (double) p->capacity * (double) (1ull << p->pack_shift) / 32.0;
	if ((double) p->rows_since_drain > limit) return cg_launch_drain(p, ctx->compute);
	return CG_OK;
}

static int read_stats(CgContext *ctx, CgPartial *p, unsigned long long before[3], CgScanStats *stats)
{
	unsigned long long after[3];
	CG_CUDA(cudaMemcpyAsync(after, p->d_stats, sizeof after, cudaMemcpyDeviceToHost, ctx->compute));
	CG_CUDA(cudaStreamSynchronize(ctx->compute));
	int rc = check_error_flags(p, after[2]);
	if (rc) return rc;
	if (stats)
	{
		stats->rows_scanned = (int64_t) (after[0] - before[0]);
		stats->rows_removed_by_filter = (int64_t) (after[1] - before[1]);
		stats->rows_passed = stats->rows_scanned - stats->rows_removed_by_filter;
	}
	return CG_OK;
}

extern "C" int cg_scan_shard(const CgShard *sh, const CgScanDesc *desc, CgPartial *into, CgScanStats *stats)
{
	CgContext *ctx = cg_ctx();
	if (!ctx) return CG_EINVAL;
	if (!sh || !desc || !into) return cg_set_error(CG_EINVAL, "NULL argument");
	KPlan plan;
	bool all8 = false;
	int rc = cg_build_plan(desc, sh->columns.data(), sh->natts, &sh->slot_of_att, into, &plan, &all8);
	if (rc) return rc;
	rc = before_scan(ctx, into);
	if (rc) return rc;

	/* K2 on the host: SelectedChunkMask per stripe.  The list of surviving chunk groups is
	 * kept on the device and reused while the WHERE list stays the same. */
	CgShard *msh = const_cast<CgShard *>(sh);
	std::vector<uint8_t> slots(plan.slot, plan.slot + plan.ncols);
	bool same = msh->sel_valid && msh->sel_pushdown == desc->enable_qual_pushdown && msh->sel_nquals == desc->nquals &&
				memcmp(msh->sel_quals, desc->quals, sizeof(CgQual) * desc->nquals) == 0 && msh->sel_slots == slots &&
				msh->sel_nqexpr == desc->nqual_expr && memcmp(msh->sel_qexpr, desc->qual_expr, (size_t) desc->nqual_expr) == 0;
	if (!same)
	{
		std::vector<uint32_t> fastl, slowl;
		uint64_t rows_fast = 0, rows_slow = 0;
		uint32_t nullmask = 0, max_cg_rows = 0;
		fastl.reserve(sh->nchunkgroups);
		int64_t nfiltered = 0;
		std::vector<uint8_t> mask;
		size_t ns = sh->staged.size();
		for (size_t si = 0; si < sh->stripes.size(); si++)
		{
			const CgStripe &s = sh->stripes[si];
			mask.resize(s.chunk_count);
			stripe_chunk_mask(s, sh->nodes.data(), sh->columns.data(), sh->natts, desc, mask.data(), &nfiltered);
			for (uint32_t k = 0; k < s.chunk_count; k++)
			{
				if (!mask[k]) continue;
				uint64_t cg = sh->stripe_first_cg[si] + k;
				bool nulls = false;
				for (int c = 0; c < plan.ncols; c++)
				{
					const DevChunkCol &d = sh->h_chunkcols[cg * ns + plan.slot[c]];
					if (d.value_count != d.row_count) { nulls = true; nullmask |= 1u << c; }
				}
				(nulls ? slowl : fastl).push_back((uint32_t) cg);
				(nulls ? rows_slow : rows_fast) += sh->cg_rows[cg];
				max_cg_rows = std::max(max_cg_rows, sh->cg_rows[cg]);
			}
		}
		msh->sel_nfast = (uint32_t) fastl.size();
		fastl.insert(fastl.end(), slowl.begin(), slowl.end());
		CG_CUDA(cudaStreamSynchronize(ctx->compute));     /* an earlier scan may still read the old list */
		if (!fastl.empty())
			CG_CUDA(cudaMemcpy(msh->d_selected, fastl.data(), fastl.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
		msh->h_selected.swap(fastl);
		msh->sel_filtered = nfiltered;
		msh->sel_pushdown = desc->enable_qual_pushdown;
		msh->sel_nquals = desc->nquals;
		msh->sel_nullmask = nullmask;
		msh->sel_max_cg_rows = max_cg_rows;
		msh->sel_rows_fast = rows_fast;
		msh->sel_rows_total = rows_fast + rows_slow;
		msh->sel_nqexpr = desc->nqual_expr;
		memcpy(msh->sel_qexpr, desc->qual_expr, (size_t) desc->nqual_expr);
		memcpy(msh->sel_quals, desc->quals, sizeof(CgQual) * desc->nquals);
		msh->sel_slots = slots;
		msh->sel_valid = true;
	}
	const std::vector<uint32_t> &selected = sh->h_selected;
	int64_t filtered = sh->sel_filtered;
	uint64_t bytes = 0;
	if (stats)
		for (uint32_t cg : selected)
			for (int c = 0; c < plan.ncols; c++) bytes += sh->algorithmic_bytes_per_cg_col(cg, plan.slot[c]);
	unsigned long long before[3] = {0, 0, 0};
	if (stats)
	{
		CG_CUDA(cudaMemcpyAsync(before, into->d_stats, sizeof before, cudaMemcpyDeviceToHost, ctx->compute));
		CG_CUDA(cudaStreamSynchronize(ctx->compute));
	}
	if (!selected.empty())
	{
		plan.arena = sh->d_arena;
		plan.chunkcols = sh->d_chunkcols;
		plan.nstaged = (int32_t) sh->staged.size();
		plan.selected = sh->d_selected;
		plan.nselected = (uint32_t) selected.size();
		plan.max_cg_rows = sh->sel_max_cg_rows;
		FPlan fast;
		const bool use_small = cg_small_eligible(plan) && !cg_force_general();
		bool use_fast = !use_small && !cg_force_general() && cg_jit_level() < 2 && cg_build_fast_plan(desc, plan, all8, &fast);
		/* the chunk groups without NULLs in the plan columns come first in the selection */
		uint32_t nfast = sh->sel_nfast;
		if (stats) CG_CUDA(cudaEventRecord(ctx->ev_a, ctx->compute));
		rc = cg_prof_mark(ctx, ctx->compute);
		if (rc) return rc;
		if (use_fast && nfast > 0)
		{
			fast.nselected = nfast;
			rc = cg_launch_scan_fast(ctx, fast, ctx->compute);
			if (rc) return rc;
			rc = after_launch(ctx, into, fast.packed != nullptr, fast.nsums == 1, sh->sel_rows_fast);
			if (rc) return rc;
		}
		else if (nfast > 0 && !cg_force_general())
		{
			/* no ahead-of-time specialisation for this shape: the plan-specialised (NVRTC) kernel */
			KPlan piece = plan;
			piece.nselected = nfast;
			bool launched = false, packed = false, ponly = false;
			rc = cg_launch_scan_jit(ctx, piece, 0u, ctx->compute, &launched, &packed, &ponly);
			if (rc) return rc;
			if (launched)
			{
				rc = after_launch(ctx, into, packed, ponly, sh->sel_rows_fast);
				if (rc) return rc;
			}
			if (!launched) nfast = 0;
		}
		else
			nfast = 0;
		if (nfast < plan.nselected)
		{
			/* chunk groups with NULLs in a plan column: the plan-specialised kernel in its nullable form
			 * (exists bitmap + rank directory addressing, columnar_reader.c:1506-1572); the interpretive
			 * kernels only when the JIT is off or unavailable */
			plan.selected = sh->d_selected + nfast;
			plan.nselected -= nfast;
			bool launched = false, packed = false, ponly = false;
			if (!cg_force_general())
			{
				rc = cg_launch_scan_jit(ctx, plan, sh->sel_nullmask ? sh->sel_nullmask : ~0u, ctx->compute, &launched, &packed, &ponly);
				if (rc) return rc;
				if (launched)
				{
					rc = after_launch(ctx, into, packed, ponly, sh->sel_rows_total - sh->sel_rows_fast);
					if (rc) return rc;
				}
			}
			if (!launched)
			{
				if (use_small) rc = cg_launch_scan_small(ctx, plan, all8, ctx->compute);
				else rc = cg_launch_scan(ctx, plan, true, all8, ctx->compute);
				if (rc) return rc;
				into->wide_dirty = true;
			}
		}
		rc = cg_prof_mark(ctx, ctx->compute);
		if (rc) return rc;
		if (stats) CG_CUDA(cudaEventRecord(ctx->ev_b, ctx->compute));
	}
	if (stats)
	{
		memset(stats, 0, sizeof *stats);
		rc = read_stats(ctx, into, before, stats);
		if (rc) return rc;
		stats->chunk_groups_filtered = filtered;
		stats->chunk_groups_scanned = (int64_t) selected.size();
		stats->bytes_scanned = (int64_t) bytes;
		if (!selected.empty())
		{
			float ms = 0;
			CG_CUDA(cudaEventElapsedTime(&ms, ctx->ev_a, ctx->ev_b));
			stats->kernel_ms = ms;
		}
	}
	return CG_OK;
}

/* ------------------------------------------------------------------------------ *
 *  DMA staging: when the relation's pages sit in pinned (registered) host memory the copy
 *  engine moves them itself, so no host core touches the data: one 1-D cudaMemcpyAsync per
 *  run of pages that holds a (stripe, projected column) byte range lands whole pages in a
 *  raw device buffer; cg_realign_kernel then drops the 24-byte page headers and moves every
 *  chunk buffer to its 16-byte aligned arena slot (the GPU half of ColumnarStorageRead's
 *  page de-framing, columnar_storage.c:463-492).
 * ------------------------------------------------------------------------------ */
/* grows one of the context's reusable device buffers; the caller has made sure nothing uses it */
static int devbuf_reserve(CgContext::DevBuf *b, size_t bytes)
{
	if (b->cap >= bytes) return CG_OK;
	if (b->p) CG_CUDA(cudaFree(b->p));
	b->p = nullptr; b->cap = 0;
	size_t cap = bytes + bytes / 8 + 4096;
	if (cudaMalloc((void **) &b->p, cap) != cudaSuccess)
	{
		cudaGetLastError();
		return cg_set_error(CG_ENOMEM, "cudaMalloc of %zu bytes for a staging buffer failed", cap);
	}
	b->cap = cap;
	return CG_OK;
}

extern "C" int cg_relation_register(const CgRelation *rel)
{
	if (!cg_ctx()) return CG_EINVAL;
	if (!rel || !rel->pages || rel->nblocks == 0) return cg_set_error(CG_EINVAL, "empty relation");
	size_t bytes = (size_t) rel->nblocks * CG_BLCKSZ;
	cudaError_t e = cudaHostRegister((void *) rel->pages, bytes, cudaHostRegisterDefault);
	if (e != cudaSuccess)
	{
		/* the OS may refuse to pin the range (an unprivileged process can be refused): the caller can go on
		 * with pageable pages, so the refusal must not linger as the thread's last CUDA error */
		cudaGetLastError();
		return cg_set_error(CG_ECUDA, "cudaHostRegister of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
	}
	return CG_OK;
}

extern "C" int cg_relation_unregister(const CgRelation *rel)
{
	if (!cg_ctx()) return CG_EINVAL;
	if (!rel || !rel->pages) return cg_set_error(CG_EINVAL, "empty relation");
	CG_CUDA(cudaHostUnregister((void *) rel->pages));
	return CG_OK;
}

static bool pages_are_pinned(const CgRelation *rel)
{
	static int disabled = -1;
	if (disabled < 0) { const char *e = getenv("CG_NO_DMA_STAGING"); disabled = (e && atoi(e)) ? 1 : 0; }
	if (disabled || !rel->pages) return false;
	cudaPointerAttributes a;
	if (cudaPointerGetAttributes(&a, rel->pages) != cudaSuccess)
	{
		cudaGetLastError();
		return false;
	}
	return a.type == cudaMemoryTypeHost;
}

struct DmaCopy { uint64_t raw_off; uint64_t first_block; uint64_t nblocks; };

/* builds the page copies and the realign items for the chunk groups of `sp` (same iteration
 * order as plan_staging).  A copy is a run of whole pages sent with one 1-D cudaMemcpyAsync
 * (55 GB/s; the strided 2-D form that drops the headers in the copy engine measured 38-47 GB/s,
 * profiles/r01_pcie_probe.txt); column spans that touch or overlap share one copy. */
static int plan_dma(const CgRelation *rel, const std::vector<int32_t> &staged,
					const std::vector<std::vector<uint8_t>> &select, const StagePlan &sp,
					std::vector<DmaCopy> *copies, std::vector<RealignItem> *items, uint64_t *raw_bytes)
{
	size_t ns = staged.size();
	uint64_t raw_off = 0, g = 0;
	for (int si = 0; si < rel->nstripes; si++)
	{
		const CgStripe &s = rel->stripes[si];
		uint32_t first = UINT32_MAX, last = 0;
		for (uint32_t k = 0; k < s.chunk_count; k++)
			if (select[si][k]) { if (first == UINT32_MAX) first = k; last = k; }
		if (first == UINT32_MAX) continue;
		/* raw offset of logical byte 0 of page p0[j] for staged column j */
		std::vector<uint64_t> base(ns, 0), p0(ns, 0), span_lo(ns, 1), span_hi(ns, 0);
		struct Span { uint64_t b0, b1; size_t j; };
		std::vector<Span> spans;
		for (size_t j = 0; j < ns; j++)
		{
			int c = staged[j];
			if ((uint32_t) c >= s.column_count) continue;
			const CgSkipNode &nf = rel->nodes[s.skipnode_base + (uint32_t) c * s.chunk_count + first];
			const CgSkipNode &nl = rel->nodes[s.skipnode_base + (uint32_t) c * s.chunk_count + last];
			uint64_t lb = s.file_offset + nf.exists_offset;
			uint64_t le = s.file_offset + nl.value_offset + nl.value_length;
			if (le < lb || nl.value_offset + nl.value_length < nl.value_offset)
				return cg_set_error(CG_ECORRUPT, "chunk offsets of column %d run backwards in stripe %d", c, si);
			span_lo[j] = lb; span_hi[j] = le;
			if (le <= lb) le = lb + 1;
			uint64_t b0 = lb / CG_BYTES_PER_PAGE, b1 = (le - 1) / CG_BYTES_PER_PAGE;
			if (b1 >= rel->nblocks) return cg_set_error(CG_ECORRUPT, "attempt to read columnar data past end of relation");
			/* pd_lower of the first and last page of the span (ReadFromBlock, columnar_storage.c:677, checks every
			 * page; touching the header of each of the ~3 M pages of a 24 GB scan would cost more host time than
			 * the copies themselves, so interior pages are trusted to be full) */
			uint16_t lower;
			memcpy(&lower, rel->pages + b1 * CG_BLCKSZ + 12, 2);
			if (lower < CG_PAGE_HEADER + ((le - 1) % CG_BYTES_PER_PAGE) + 1)
				return cg_set_error(CG_ECORRUPT, "attempt to read columnar data past pd_lower of block %llu", (unsigned long long) b1);
			memcpy(&lower, rel->pages + b0 * CG_BLCKSZ + 12, 2);
			if (b0 != b1 && lower != CG_BLCKSZ)
				return cg_set_error(CG_ECORRUPT, "attempt to read columnar data past pd_lower of block %llu", (unsigned long long) b0);
			spans.push_back(Span{b0, b1, j});
		}
		std::sort(spans.begin(), spans.end(), [](const Span &a, const Span &b) { return a.b0 < b.b0; });
		for (size_t i = 0; i < spans.size();)
		{
			uint64_t b0 = spans[i].b0, b1 = spans[i].b1;
			size_t e = i + 1;
			while (e < spans.size() && spans[e].b0 <= b1 + 1) { b1 = std::max(b1, spans[e].b1); e++; }
			for (size_t q = i; q < e; q++)
			{
				p0[spans[q].j] = spans[q].b0;
				base[spans[q].j] = raw_off + (spans[q].b0 - b0) * CG_BLCKSZ;
			}
			copies->push_back(DmaCopy{raw_off, b0, b1 - b0 + 1});
			raw_off += (b1 - b0 + 1) * CG_BLCKSZ;
			i = e;
		}
		for (uint32_t k = 0; k < s.chunk_count; k++)
		{
			if (!select[si][k]) continue;
			for (size_t j = 0; j < ns; j++)
			{
				const DevChunkCol &d = sp.cols[g * ns + j];
				const StageItem &it = sp.items[g * ns + j];
				uint64_t exspan = it.wire_value_off - d.exists_off;
				uint64_t vaspan = pad16(it.value_len) + 16;
				/* every chunk buffer must lie inside the byte range its column's copy covers (the pageable path
				 * reports the same images as past-pd_lower reads; here an unchecked offset would make the
				 * realign kernel read arbitrary device memory) */
				if ((it.exists_len && (it.exists_logical < span_lo[j] || it.exists_logical + it.exists_len > span_hi[j])) ||
					(it.value_len && (it.value_logical < span_lo[j] || it.value_logical + it.value_len > span_hi[j])))
					return cg_set_error(CG_ECORRUPT, "chunk buffer outside its column's byte range in stripe %d", si);
				auto phys = [&](uint64_t logical) {
					uint64_t rel0 = logical - p0[j] * CG_BYTES_PER_PAGE;
					return base[j] + (rel0 / CG_BYTES_PER_PAGE) * CG_BLCKSZ + CG_PAGE_HEADER + rel0 % CG_BYTES_PER_PAGE;
				};
				uint64_t esrc = it.exists_len ? phys(it.exists_logical) : CG_PAGE_HEADER;
				uint64_t vsrc = it.value_len ? phys(it.value_logical) : CG_PAGE_HEADER;
				items->push_back(RealignItem{esrc, d.exists_off, it.exists_len, (uint32_t) exspan});
				items->push_back(RealignItem{vsrc, it.wire_value_off, it.value_len, (uint32_t) vaspan});
			}
			g++;
		}
	}
	*raw_bytes = raw_off + 2 * CG_BLCKSZ;   /* the realign kernel's last vector reads one word past a buffer */
	return CG_OK;
}

/*
 * End to end on host buffers: skip -> stage only the plan's columns of the surviving
 * chunk groups through the pinned ring -> one fused kernel launch per block, the
 * kernel of block b overlapping the H2D of block b+1.
 */
extern "C" int cg_scan_relation(const CgRelation *rel, const CgScanDesc *desc, CgPartial *into, CgScanStats *stats)
{
	CgContext *ctx = cg_ctx();
	if (!ctx) return CG_EINVAL;
	if (!desc || !into) return cg_set_error(CG_EINVAL, "NULL argument");
	int rc = validate_relation(rel);
	if (rc) return rc;

	/* projection */
	std::vector<int32_t> staged, slot_of_att(rel->natts, -1);
	auto need = [&](int c) { if (slot_of_att[c] < 0) { slot_of_att[c] = (int32_t) staged.size(); staged.push_back(c); } };
	for (int q = 0; q < desc->nquals; q++) if (desc->quals[q].column >= 0 && desc->quals[q].column < rel->natts) need(desc->quals[q].column);
	for (int g = 0; g < desc->ngroup_cols; g++) if (desc->group_cols[g] >= 0 && desc->group_cols[g] < rel->natts) need(desc->group_cols[g]);
	for (int a = 0; a < desc->naggs; a++)
		for (int f = 0; f < desc->aggs[a].nfactors && f < 3; f++)
			if (desc->aggs[a].column[f] >= 0 && desc->aggs[a].column[f] < rel->natts) need(desc->aggs[a].column[f]);
	if (staged.empty()) need(0);   /* count(*) only: the reference still reads the first column's skip nodes; we read its chunk row counts */

	KPlan plan;
	bool all8 = false;
	rc = cg_build_plan(desc, rel->columns, rel->natts, &slot_of_att, into, &plan, &all8);
	if (rc) return rc;
	rc = before_scan(ctx, into);
	if (rc) return rc;

	std::vector<std::vector<uint8_t>> select(rel->nstripes);
	int64_t filtered = 0;
	for (int si = 0; si < rel->nstripes; si++)
	{
		select[si].resize(rel->stripes[si].chunk_count);
		stripe_chunk_mask(rel->stripes[si], rel->nodes, rel->columns, rel->natts, desc, select[si].data(), &filtered);
	}
	StagePlan sp;
	rc = plan_staging(rel, staged, &select, &sp);
	if (rc) return rc;
	size_t ns = staged.size();
	uint64_t ncg = sp.cg_rows.size();

	unsigned long long before[3] = {0, 0, 0};
	if (stats)
	{
		CG_CUDA(cudaMemcpyAsync(before, into->d_stats, sizeof before, cudaMemcpyDeviceToHost, ctx->compute));
		CG_CUDA(cudaStreamSynchronize(ctx->compute));
	}
	uint64_t bytes = 0;
	for (uint64_t g = 0; g < ncg; g++)
		for (int c = 0; c < plan.ncols; c++)
		{
			const DevChunkCol &d = sp.cols[g * ns + plan.slot[c]];
			bytes += (uint64_t) sp.stream_bytes[g * ns + plan.slot[c]] + (d.row_count + 7) / 8;
		}

	uint8_t *d_arena = nullptr;
	DevChunkCol *d_cols = nullptr;
	uint32_t *d_ids = nullptr;
	uint64_t dma_bytes = 0;
	bool used_dma = false;
	if (ncg > 0)
	{
		/* small per-call metadata goes through a pinned ring so that its upload is truly
		 * asynchronous (a pageable source would make cudaMemcpyAsync wait for the copy stream) */
		const bool dma = pages_are_pinned(rel);
		std::vector<DmaCopy> copies;
		std::vector<RealignItem> items;
		uint64_t raw_bytes = 0;
		if (dma)
		{
			rc = plan_dma(rel, staged, select, sp, &copies, &items, &raw_bytes);
			if (rc) return rc;
		}
		const size_t cols_bytes = sp.cols.size() * sizeof(DevChunkCol);
		const size_t ids_bytes = ncg * sizeof(uint32_t);
		const size_t items_bytes = items.size() * sizeof(RealignItem);
		const size_t dec_bytes = sp.decode.size() * sizeof(DecodeItem);
		const size_t vl_bytes = sp.varlena.size() * sizeof(VarlenaItem);
		const size_t off_ids = (cols_bytes + 15) & ~15ull, off_items = off_ids + ((ids_bytes + 15) & ~15ull);
		const size_t off_dec = off_items + ((items_bytes + 15) & ~15ull);
		const size_t off_vl = off_dec + ((dec_bytes + 15) & ~15ull);
		const size_t meta_bytes = off_vl + vl_bytes + 64;
		const int mslot = ctx->dma_slot;
		ctx->dma_slot = (mslot + 1) % CgContext::kDmaDepth;
		if (!ctx->dma_done[mslot]) CG_CUDA(cudaEventCreateWithFlags(&ctx->dma_done[mslot], cudaEventDisableTiming));
		if (!ctx->dma_copied) CG_CUDA(cudaEventCreateWithFlags(&ctx->dma_copied, cudaEventDisableTiming));
		CG_CUDA(cudaEventSynchronize(ctx->dma_done[mslot]));      /* bounds the shards in flight; frees the slot */
		/* once work on the slot's buffers has been enqueued, every exit path must leave dma_done[mslot] behind
		 * that work: on an error return the copy and decode streams are drained and the event is recorded, so
		 * the next user of the slot cannot free or overwrite buffers that are still being written */
		struct SlotGuard
		{
			CgContext *ctx; int slot; bool armed = true; cudaStream_t side = nullptr;
			~SlotGuard()
			{
				if (!armed) return;
				cudaStreamSynchronize(ctx->copy);
				if (side) cudaStreamSynchronize(side);
				cudaEventRecord(ctx->dma_done[slot], ctx->compute);
			}
		} slot_guard{ctx, mslot};
		if (ctx->meta_cap[mslot] < meta_bytes)
		{
			if (ctx->meta_pinned[mslot]) CG_CUDA(cudaFreeHost(ctx->meta_pinned[mslot]));
			ctx->meta_pinned[mslot] = nullptr;
			size_t cap = std::max<size_t>(meta_bytes * 2, 4u << 20);
			CG_CUDA(cudaHostAlloc((void **) &ctx->meta_pinned[mslot], cap, cudaHostAllocDefault));
			ctx->meta_cap[mslot] = cap;
		}
		uint8_t *hm = ctx->meta_pinned[mslot];
		/* the slot's device buffers: everything that used them has finished (dma_done above) */
		rc = devbuf_reserve(&ctx->slot_arena[mslot], std::max<uint64_t>(sp.arena_bytes, 16));
		if (rc == CG_OK) rc = devbuf_reserve(&ctx->slot_meta[mslot], meta_bytes);
		if (rc == CG_OK && dma) rc = devbuf_reserve(&ctx->slot_raw[mslot], raw_bytes);
		if (rc) return rc;
		d_arena = ctx->slot_arena[mslot].p;
		uint8_t *d_meta = ctx->slot_meta[mslot].p;
		memcpy(hm, sp.cols.data(), cols_bytes);
		for (uint64_t g = 0; g < ncg; g++) ((uint32_t *) (hm + off_ids))[g] = (uint32_t) g;
		if (items_bytes) memcpy(hm + off_items, items.data(), items_bytes);
		if (dec_bytes) memcpy(hm + off_dec, sp.decode.data(), dec_bytes);
		if (vl_bytes) memcpy(hm + off_vl, sp.varlena.data(), vl_bytes);
		CG_CUDA(cudaMemcpyAsync(d_meta, hm, meta_bytes, cudaMemcpyHostToDevice, ctx->copy));
		d_cols = (DevChunkCol *) d_meta;
		d_ids = (uint32_t *) (d_meta + off_ids);
		const DecodeItem *d_decode = (const DecodeItem *) (d_meta + off_dec);
		const VarlenaItem *d_varlena = (const VarlenaItem *) (d_meta + off_vl);
		plan.arena = d_arena;
		plan.chunkcols = d_cols;
		plan.nstaged = (int32_t) ns;
		for (uint32_t r : sp.cg_rows) plan.max_cg_rows = std::max(plan.max_cg_rows, r);
		FPlan fast;
		const bool use_small = cg_small_eligible(plan) && !cg_force_general();
		const bool use_fast = !use_small && !sp.any_nulls && !cg_force_general() && cg_jit_level() < 2 &&
							  cg_build_fast_plan(desc, plan, all8, &fast);
		const bool try_jit = !use_fast && !cg_force_general();
		/* plan columns with NULLs somewhere in the planned chunk groups: the generated kernel takes the exists
		 * bitmap + rank directory path for those (per chunk, uniformly), dense loads everywhere else */
		uint32_t nullable = 0;
		if (sp.any_nulls)
			for (uint64_t g = 0; g < ncg; g++)
				for (int c = 0; c < plan.ncols; c++)
				{
					const DevChunkCol &d = sp.cols[g * ns + plan.slot[c]];
					if (d.value_count != d.row_count) nullable |= 1u << c;
				}
		if (stats) CG_CUDA(cudaEventRecord(ctx->ev_a, ctx->compute));
		bool decode_done = false;          /* the DMA path may decode on a side stream before launch_block runs */
		auto block_rows = [&](uint64_t cg0, uint64_t cg1) { uint64_t n = 0; for (uint64_t g = cg0; g < cg1; g++) n += sp.cg_rows[g]; return n; };
		auto launch_block = [&](uint64_t cg0, uint64_t cg1, cudaEvent_t copied) -> int {
			CG_CUDA(cudaStreamWaitEvent(ctx->compute, copied, 0));
			/* K7: compressed value streams of the block -> their value slots */
			int r = CG_OK;
			if (!decode_done)
			{
				r = cg_launch_decompress(ctx, d_arena, d_decode + sp.dec_first[cg0], sp.decode.data() + sp.dec_first[cg0],
										 sp.dec_first[cg1] - sp.dec_first[cg0], into->d_stats + 2, CG_ERRFLAG_DECOMPRESS, ctx->compute);
				if (r == CG_OK)
					r = cg_launch_varlena_decode(ctx, d_arena, d_varlena + sp.vl_first[cg0], sp.vl_first[cg1] - sp.vl_first[cg0], into->d_stats + 2,
												 CG_ERRFLAG_VARLENA, ctx->compute);
			}
			if (r) return r;
			if (sp.any_nulls)
			{
				r = cg_launch_rank(ctx, d_arena, d_cols, cg0 * ns, (cg1 - cg0) * ns, ctx->compute);
				if (r) return r;
			}
			r = cg_prof_mark(ctx, ctx->compute);
			if (r) return r;
			bool jitted = false;
			if (try_jit)
			{
				KPlan blk = plan;
				blk.selected = d_ids + cg0;
				blk.nselected = (uint32_t) (cg1 - cg0);
				bool packed = false, ponly = false;
				r = cg_launch_scan_jit(ctx, blk, nullable, ctx->compute, &jitted, &packed, &ponly);
				if (r) return r;
				if (jitted) { r = after_launch(ctx, into, packed, ponly, block_rows(cg0, cg1)); if (r) return r; }
			}
			if (jitted) { }
			else if (use_small)
			{
				KPlan blk = plan;
				blk.selected = d_ids + cg0;
				blk.nselected = (uint32_t) (cg1 - cg0);
				r = cg_launch_scan_small(ctx, blk, all8, ctx->compute);
				into->wide_dirty = true;
			}
			else if (use_fast)
			{
				FPlan blk = fast;
				blk.selected = d_ids + cg0;
				blk.nselected = (uint32_t) (cg1 - cg0);
				r = cg_launch_scan_fast(ctx, blk, ctx->compute);
				if (r == CG_OK) r = after_launch(ctx, into, blk.packed != nullptr, blk.nsums == 1, block_rows(cg0, cg1));
			}
			else
			{
				KPlan blk = plan;
				blk.selected = d_ids + cg0;
				blk.nselected = (uint32_t) (cg1 - cg0);
				r = cg_launch_scan(ctx, blk, sp.any_nulls, all8, ctx->compute);
				into->wide_dirty = true;
			}
			if (r) return r;
			return cg_prof_mark(ctx, ctx->compute);
		};
		if (dma)
		{
			/* whole pages by DMA; the GPU de-frames them */
			static int trace = -1;
			if (trace < 0) { const char *e = getenv("CG_TRACE"); trace = (e && atoi(e)) ? 1 : 0; }
			cudaEvent_t t0 = nullptr, t1 = nullptr;
			auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
			double h0 = now();
			uint8_t *d_raw = ctx->slot_raw[mslot].p;
			if (trace) { cudaEventCreate(&t0); cudaEventCreate(&t1); cudaEventRecord(t0, ctx->copy); }
			for (const DmaCopy &c : copies)
			{
				CG_CUDA(cudaMemcpyAsync(d_raw + c.raw_off, rel->pages + c.first_block * CG_BLCKSZ, c.nblocks * CG_BLCKSZ,
										cudaMemcpyHostToDevice, ctx->copy));
				dma_bytes += c.nblocks * CG_BLCKSZ;
			}
			if (trace)
			{
				double h1 = now();
				cudaEventRecord(t1, ctx->copy);
				cudaEventSynchronize(t1);
				float ms = 0;
				cudaEventElapsedTime(&ms, t0, t1);
				fprintf(stderr, "[cg] dma: %zu copies, %.1f MB, issue %.2f ms, copy-stream %.2f ms = %.1f GB/s\n", copies.size(),
						dma_bytes / 1e6, (h1 - h0) * 1e3, ms, dma_bytes / 1e6 / ms);
				cudaEventDestroy(t0); cudaEventDestroy(t1);
			}
			CG_CUDA(cudaEventRecord(ctx->dma_copied, ctx->copy));
			cudaEvent_t k0 = nullptr, k1 = nullptr, k2 = nullptr;
			if (trace) { cudaEventCreate(&k0); cudaEventCreate(&k1); cudaEventCreate(&k2); cudaEventRecord(k0, ctx->compute); }
			cudaEvent_t ready = ctx->dma_copied;
			/* zstd decoders share one literal scratch area: they stay on the compute stream */
			bool has_zstd = false;
			for (const DecodeItem &di : sp.decode) if (di.kind == CG_COMPRESSION_ZSTD) { has_zstd = true; break; }
			if ((!sp.decode.empty() || !sp.varlena.empty()) && !trace && !has_zstd)
			{
				/* de-framing and decompression run on one of two side streams, the scan follows on the
				 * compute stream: the decode of this shard overlaps the decode (and scan) of the previous one */
				const int ds = (int) (ctx->decode_rr++ % (unsigned) CgContext::kDmaDepth);
				if (!ctx->decode_stream[ds]) CG_CUDA(cudaStreamCreateWithFlags(&ctx->decode_stream[ds], cudaStreamNonBlocking));
				if (!ctx->decoded[mslot]) CG_CUDA(cudaEventCreateWithFlags(&ctx->decoded[mslot], cudaEventDisableTiming));
				cudaStream_t side = ctx->decode_stream[ds];
				slot_guard.side = side;
				CG_CUDA(cudaStreamWaitEvent(side, ctx->dma_copied, 0));
				rc = cg_launch_realign(d_raw, d_arena, (const RealignItem *) (d_meta + off_items), items.size(), side);
				if (rc == CG_OK)
					rc = cg_launch_decompress(ctx, d_arena, d_decode, sp.decode.data(), sp.decode.size(), into->d_stats + 2,
											  CG_ERRFLAG_DECOMPRESS, side);
				if (rc == CG_OK)
					rc = cg_launch_varlena_decode(ctx, d_arena, d_varlena, sp.varlena.size(), into->d_stats + 2, CG_ERRFLAG_VARLENA, side);
				if (rc) return rc;
				CG_CUDA(cudaEventRecord(ctx->decoded[mslot], side));
				ready = ctx->decoded[mslot];
				decode_done = true;
			}
			else
			{
				CG_CUDA(cudaStreamWaitEvent(ctx->compute, ctx->dma_copied, 0));
				rc = cg_launch_realign(d_raw, d_arena, (const RealignItem *) (d_meta + off_items), items.size(), ctx->compute);
			}
			if (trace) cudaEventRecord(k1, ctx->compute);
			if (rc == CG_OK) rc = launch_block(0, ncg, ready);
			if (trace)
			{
				cudaEventRecord(k2, ctx->compute);
				cudaEventSynchronize(k2);
				float a = 0, b = 0;
				cudaEventElapsedTime(&a, k0, k1);
				cudaEventElapsedTime(&b, k1, k2);
				fprintf(stderr, "[cg] dma: realign %.3f ms (%zu items), decode (%zu streams) + scan %.3f ms\n", a, items.size(),
						sp.decode.size(), b);
				cudaEventDestroy(k0); cudaEventDestroy(k1); cudaEventDestroy(k2);
			}
			used_dma = true;
		}
		else
			rc = stream_to_device(ctx, rel, sp, ns, d_arena, launch_block);
		if (stats && rc == CG_OK) CG_CUDA(cudaEventRecord(ctx->ev_b, ctx->compute));
		if (rc) return rc;                  /* slot_guard drains the side streams and records the event */
		CG_CUDA(cudaEventRecord(ctx->dma_done[mslot], ctx->compute));
		slot_guard.armed = false;
	}
	if (stats)
	{
		memset(stats, 0, sizeof *stats);
		rc = read_stats(ctx, into, before, stats);
		if (rc) return rc;
		stats->chunk_groups_filtered = filtered;
		stats->chunk_groups_scanned = (int64_t) ncg;
		stats->bytes_scanned = (int64_t) bytes;
		if (ncg > 0)
		{
			float ms = 0;
			CG_CUDA(cudaEventElapsedTime(&ms, ctx->ev_a, ctx->ev_b));
			stats->kernel_ms = ms;   /* here: first kernel start to last kernel end, H2D overlapped */
			stats->h2d_bytes = (int64_t) ((used_dma ? dma_bytes + 2 * ncg * ns * sizeof(RealignItem) : sp.wire_bytes) +
										  sp.cols.size() * sizeof(DevChunkCol) + ncg * sizeof(uint32_t) +
										  sp.decode.size() * sizeof(DecodeItem));
		}
	}
	return CG_OK;
}

/* ------------------------------------------------------------------------------ *
 *  Results.
 * ------------------------------------------------------------------------------ */
static int ensure_out(CgPartial *p, uint64_t cap)
{
	if (p->out_capacity >= cap && p->d_out_keys) return CG_OK;
	cudaFree(p->d_out_keys); cudaFree(p->d_out_words); cudaFree(p->d_out_nulls);
	p->d_out_keys = nullptr; p->d_out_words = nullptr; p->d_out_nulls = nullptr;
	if (cudaMalloc(&p->d_out_keys, cap * sizeof(int64_t)) != cudaSuccess ||
		cudaMalloc(&p->d_out_words, cap * p->nwords * sizeof(uint64_t)) != cudaSuccess ||
		cudaMalloc(&p->d_out_nulls, cap) != cudaSuccess)
		return cg_set_error(CG_ENOMEM, "cudaMalloc for %llu result rows failed", (unsigned long long) cap);
	p->out_capacity = cap;
	return CG_OK;
}

/* makes the exact accumulators current (drains packed words), then surfaces kernel-side errors */
static int pending_errors(CgContext *ctx, CgPartial *p)
{
	int rc = cg_launch_drain(p, ctx->compute);
	if (rc) return rc;
	unsigned long long st[5];
	CG_CUDA(cudaMemcpyAsync(st, p->d_stats, sizeof st, cudaMemcpyDeviceToHost, ctx->compute));
	CG_CUDA(cudaStreamSynchronize(ctx->compute));
	rc = check_error_flags(p, st[2]);
	if (rc) return rc;
	if (st[CG_STAT_PACKED_ADDED] != st[CG_STAT_PACKED_DRAINED])
		return cg_set_error(CG_ERETRY_UNPACKED,
							"packed accumulators overflowed (%llu rows added, %llu drained): a group received >= 2^%d rows "
							"between drains; disable packing, reset and rescan",
							st[CG_STAT_PACKED_ADDED], st[CG_STAT_PACKED_DRAINED], p->pack_shift);
	return CG_OK;
}

/*
 * Makes the result rows of a partial: surfaces kernel-raised errors, compacts the occupied groups into (keys, NULL flags,
 * accumulator words) and returns their number -- with ONE host synchronisation.  Two forms:
 *   packed-direct  a direct-indexed table that only ever received packed words (the C2 shape, also after an NCCL reduce
 *                  of the packed words): the rows are decoded straight from the 8-byte packed words; the wide table is
 *                  neither read nor written (it is still in its initial state and stays so across cg_partial_reset)
 *   general        drain of any packed words into the wide accumulators, then the compaction of the wide table
 * out_* may be NULL (count only).
 */
static int export_rows(CgContext *ctx, CgPartial *p, uint64_t capacity, int64_t *d_keys, uint8_t *d_nulls, uint64_t *d_words, int64_t *nrows)
{
	unsigned long long st[5], counts[2] = {0, 0};
	const bool direct = p->d_packed && p->packed_dirty && !p->wide_dirty && p->mode == CG_MODE_DENSE && p->desc.ngroup_cols == 1;
	int rc;
	if (direct)
	{
		rc = cg_launch_export_packed(p, capacity, d_keys, d_nulls, d_words, p->d_out_count, ctx->compute);
		p->read_packed_direct = true;
	}
	else
	{
		rc = cg_launch_drain(p, ctx->compute);
		if (rc == CG_OK) rc = cg_launch_export(p, capacity, d_keys, d_nulls, d_words, p->d_out_count, ctx->compute);
	}
	if (rc) return rc;
	/* both read-backs land in pinned memory: truly asynchronous copies, one wait (a pageable destination makes
	 * every small copy a blocking round trip of its own) */
	if (!p->h_ret) CG_CUDA(cudaHostAlloc((void **) &p->h_ret, 8 * sizeof(unsigned long long), cudaHostAllocDefault));
	CG_CUDA(cudaMemcpyAsync(p->h_ret, p->d_stats, sizeof st, cudaMemcpyDeviceToHost, ctx->compute));
	CG_CUDA(cudaMemcpyAsync(p->h_ret + 5, p->d_out_count, sizeof counts, cudaMemcpyDeviceToHost, ctx->compute));
	CG_CUDA(cudaStreamSynchronize(ctx->compute));
	memcpy(st, p->h_ret, sizeof st);
	memcpy(counts, p->h_ret + 5, sizeof counts);
	rc = check_error_flags(p, st[2]);
	if (rc) return rc;
	/* every row added to a packed word must have come out again (drained earlier, or decoded just now) */
	const unsigned long long out = st[CG_STAT_PACKED_DRAINED] + (direct ? counts[1] : 0ull);
	if (st[CG_STAT_PACKED_ADDED] != out)
		return cg_set_error(CG_ERETRY_UNPACKED,
							"packed accumulators overflowed (%llu rows added, %llu decoded): a group received >= 2^%d rows "
							"between drains; disable packing, reset and rescan",
							st[CG_STAT_PACKED_ADDED], out, p->pack_shift);
	*nrows = (int64_t) counts[0];
	return CG_OK;
}

extern "C" int cg_partial_ngroups(CgPartial *p, int64_t *ngroups)
{
	CgContext *ctx = cg_ctx();
	if (!ctx || !p) return CG_EINVAL;
	return export_rows(ctx, p, 0, nullptr, nullptr, nullptr, ngroups);
}

static inline uint64_t f8_unordered(uint64_t u)
{
	return (u >> 63) ? (u & 0x7fffffffffffffffull) : ~u;
}

extern "C" int cg_partial_fetch(CgPartial *p, int64_t capacity, int64_t *keys, uint8_t *key_nulls,
								int64_t *sum_hi, uint64_t *sum_lo, int64_t *count, int64_t *minmax,
								double *fsum, int64_t *ngroups)
{
	CgContext *ctx = cg_ctx();
	if (!ctx || !p) return CG_EINVAL;
	if (capacity < 0) return cg_set_error(CG_EINVAL, "negative capacity");
	int rc = ensure_out(p, std::max<uint64_t>((uint64_t) capacity, 1));
	if (rc) return rc;
	int64_t nrows = 0;
	rc = export_rows(ctx, p, (uint64_t) capacity, p->d_out_keys, p->d_out_nulls, p->d_out_words, &nrows);
	if (rc) return rc;
	unsigned long long n = (unsigned long long) nrows;
	if (ngroups) *ngroups = (int64_t) n;
	if ((int64_t) n > capacity)
		return cg_set_error(CG_EINVAL, "%llu groups do not fit the caller's capacity %lld", n, (long long) capacity);
	if (n == 0) return CG_OK;
	/* result rows come back through a pinned buffer owned by the partial (DMA at link rate,
	 * no page faults on fresh memory), then are unpacked by the staging threads */
	const size_t kbytes = (n * sizeof(int64_t) + 15) & ~15ull, nbytes = (n + 15) & ~15ull;
	const size_t wbytes = (size_t) n * p->nwords * sizeof(uint64_t);
	if (p->h_out_cap < kbytes + nbytes + wbytes)
	{
		if (p->h_out) cudaFreeHost(p->h_out);
		p->h_out = nullptr; p->h_out_cap = 0;
		size_t cap = kbytes + nbytes + wbytes + (1u << 16);
		CG_CUDA(cudaHostAlloc((void **) &p->h_out, cap, cudaHostAllocDefault));
		p->h_out_cap = cap;
	}
	const int64_t *hk = (const int64_t *) p->h_out;
	const uint8_t *hn = p->h_out + kbytes;
	const uint64_t *hw = (const uint64_t *) (p->h_out + kbytes + nbytes);
	CG_CUDA(cudaMemcpyAsync((void *) hk, p->d_out_keys, n * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->compute));
	CG_CUDA(cudaMemcpyAsync((void *) hn, p->d_out_nulls, n, cudaMemcpyDeviceToHost, ctx->compute));
	CG_CUDA(cudaMemcpyAsync((void *) hw, p->d_out_words, wbytes, cudaMemcpyDeviceToHost, ctx->compute));
	CG_CUDA(cudaStreamSynchronize(ctx->compute));
	const int na = p->desc.naggs;
	const int nthreads = n >= 65536 ? std::max(1, std::min(ctx->stage_threads, 16)) : 1;
#pragma omp parallel for schedule(static) num_threads(nthreads)
	for (int64_t i = 0; i < (int64_t) n; i++)
	{
		if (keys) keys[i] = hk[i];
		if (key_nulls) key_nulls[i] = hn[i];
		const uint64_t *w = &hw[i * p->nwords];
		int64_t rows = (int64_t) w[0];
		for (int a = 0; a < na; a++)
		{
			const KAgg &k = p->aggs[a];
			size_t o = i * na + a;
			int64_t hi = 0; uint64_t lo = 0; int64_t cnt = 0; int64_t mm = 0; double fs = 0;
			switch (k.kind)
			{
				case CG_AGG_COUNT_STAR: cnt = rows; break;
				case CG_AGG_COUNT: cnt = rows - (int64_t) w[k.nullword]; break;
				case CG_AGG_SUM:
					cnt = rows - (int64_t) w[k.nullword];
					if (k.is_float) memcpy(&fs, &w[k.word0], 8);
					else
					{
						__int128 s;
						if (k.nlimbs == 1) s = (__int128) (int64_t) w[k.word0];
						else s = (__int128) (unsigned __int128) w[k.word0] + ((__int128) (int64_t) w[k.word0 + 1] << 32);
						hi = (int64_t) (s >> 64); lo = (uint64_t) s;
					}
					break;
				default:
					cnt = rows - (int64_t) w[k.nullword];
					mm = k.is_float ? (int64_t) f8_unordered(w[k.word0]) : (int64_t) w[k.word0];
					break;
			}
			if (sum_hi) sum_hi[o] = hi;
			if (sum_lo) sum_lo[o] = lo;
			if (count) count[o] = cnt;
			if (minmax) minmax[o] = mm;
			if (fsum) fsum[o] = fs;
		}
	}
	return CG_OK;
}

extern "C" int cg_partial_export_device(CgPartial *p, int64_t capacity, int64_t *d_keys, uint8_t *d_key_nulls,
										uint64_t *d_words, int64_t *nrows)
{
	CgContext *ctx = cg_ctx();
	if (!ctx || !p) return CG_EINVAL;
	int64_t got = 0;
	int rc = export_rows(ctx, p, (uint64_t) capacity, d_keys, d_key_nulls, d_words, &got);
	if (rc) return rc;
	unsigned long long n = (unsigned long long) got;
	if (nrows) *nrows = (int64_t) n;
	if ((int64_t) n > capacity) return cg_set_error(CG_EINVAL, "%llu rows exceed capacity %lld", n, (long long) capacity);
	return CG_OK;
}

extern "C" int cg_partial_merge_rows(CgPartial *p, const int64_t *d_keys, const uint8_t *d_key_nulls,
									 const uint64_t *d_words, int64_t nrows)
{
	CgContext *ctx = cg_ctx();
	if (!ctx || !p) return CG_EINVAL;
	int rc = cg_launch_merge(p, d_keys, d_key_nulls, d_words, nrows, ctx->compute);
	if (rc) return rc;
	CG_CUDA(cudaStreamSynchronize(ctx->compute));
	return pending_errors(ctx, p);
}

/* the same without waiting: the drain of the packed words is enqueued on the library's stream, work
 * the caller enqueues behind it on that stream (a collective) sees the drained table; the scan's error
 * flags are NOT looked at here -- cg_partial_check (or any call that reads the partial) does that */
extern "C" int cg_partial_dense_words_enqueue(CgPartial *p, uint64_t **d_words, int64_t *total_words, int32_t *stride)
{
	if (!p || !d_words) return cg_set_error(CG_EINVAL, "NULL partial");
	if (p->mode == CG_MODE_HASH) return cg_set_error(CG_EINVAL, "not a direct-indexed table");
	CgContext *ctx = cg_ctx();
	if (!ctx) return CG_EINVAL;
	int rc = cg_launch_drain(p, ctx->compute);
	if (rc) return rc;
	*d_words = p->d_table;
	if (total_words) *total_words = (int64_t) (p->entries * (uint64_t) p->stride);
	if (stride) *stride = p->stride;
	return CG_OK;
}

/* waits for the partial's pending work and reports what its kernels flagged (table full, key range,
 * sum bound, corrupt compressed stream, packed overflow -> CG_ERETRY_UNPACKED) */
extern "C" int cg_partial_check(CgPartial *p)
{
	CgContext *ctx = cg_ctx();
	if (!ctx || !p) return CG_EINVAL;
	return pending_errors(ctx, p);
}

extern "C" int cg_partial_dense_words(CgPartial *p, uint64_t **d_words, int64_t *total_words, int32_t *stride)
{
	if (!p) return cg_set_error(CG_EINVAL, "NULL partial");
	if (p->mode == CG_MODE_HASH) return cg_set_error(CG_EINVAL, "not a direct-indexed table");
	CgContext *ctx = cg_ctx();
	if (!ctx) return CG_EINVAL;
	int rc = pending_errors(ctx, p);
	if (rc) return rc;
	*d_words = p->d_table;
	if (total_words) *total_words = (int64_t) (p->entries * (uint64_t) p->stride);
	if (stride) *stride = p->stride;
	return CG_OK;
}
