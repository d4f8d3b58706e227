/*
 * citus_gpu.h -- C-ABI of libcitus_gpu.so: the B200 (sm_100a) implementation of Citus's
 * columnar shard-scan / partial-aggregate / combine / hash-repartition hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8(b)).  Plain C, plain pointers and
 * sizes, no CUDA or torch types.  Every entry point returns 0 on success or a CG_E* code;
 * the message is read with cg_last_error() (thread-local).  Nothing here longjmps: the
 * PostgreSQL-side glue turns a non-zero return into ereport(ERROR) (INTEGRATION.md).
 *
 * Reference interfaces each block replaces are cited as file:line under
 * /root/reference/src.
 */
#ifndef CITUS_GPU_H
#define CITUS_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CG_OK 0
#define CG_EINVAL 1        /* bad argument / unsupported plan shape */
#define CG_ECUDA 2         /* CUDA runtime error (message has the cudaError string) */
#define CG_ENOMEM 3
#define CG_ECORRUPT 4      /* relation image inconsistent with its metadata */
#define CG_ETABLEFULL 5    /* group table too small: retry with a larger expected_groups */
#define CG_EUNSUPPORTED 6  /* valid SQL, but outside what the GPU path handles: caller falls
                            * back to the reference's row-at-a-time executor */
#define CG_ECOMM 8          /* NCCL / communicator error, or another rank failed the query */
#define CG_ERETRY_UNPACKED 7 /* an optimistic packed accumulator overflowed (see cg_partial_set_packing):
                            * nothing wrong was returned; call cg_partial_set_packing(p, 0),
                            * cg_partial_reset(p) and scan again */

const char *cg_last_error(void);

/* ---------------------------------------------------------------------------------- *
 *  Device context.  One per process (a PostgreSQL backend is one process; CUDA is
 *  initialised lazily in the backend, never in the postmaster -- SURVEY.md 7.3).
 * ---------------------------------------------------------------------------------- */
int cg_init(int device_ordinal);          /* idempotent */
int cg_device_count(int *count);
int cg_synchronize(void);                 /* waits for the library's streams */
/* Run the kernels on a stream owned by the caller (a CUstream / cudaStream_t handle passed as
 * void *; NULL restores the library's own stream; (void *) 1 is CUDA's legacy default stream,
 * cudaStreamLegacy).  Lets a host that already has a stream -- e.g. the one its NCCL
 * collectives are ordered on -- keep everything in one queue. */
int cg_set_stream(void *cuda_stream);
/* Per-launch device timing of the fused scan kernels: between begin and collect every scan
 * launch is bracketed by CUDA events on the launching stream (no host synchronisation);
 * collect waits for them and returns the launch count and the summed / maximum duration. */
int cg_profile_begin(void);
int cg_profile_collect(int32_t *launches, double *total_ms, double *max_ms);
/* number of CUDA kernels this library has launched so far (all kernels, all entry points) */
uint64_t cg_kernel_launches(void);
/* Plan-specialised kernels (cg_jit.cpp): query shapes without an ahead-of-time specialisation are
 * written out as straight-line CUDA and compiled with NVRTC the first time they are seen (CG_JIT=0
 * turns this off; the interpretive kernels then run everything).  Counters, and a GPU-less check that
 * a query shape generates valid sm_100a code: kind = 0 plain aggregate / 1 shared-memory cells /
 * 2 global table; source (may be NULL) receives the generated CUDA. */
uint64_t cg_jit_launches(void);
uint64_t cg_jit_compiles(void);
/* run-time switches (tests and A/B measurements drive every kernel family through the same C-ABI calls):
 *   "jit" 0 | 1 | 2, "force_general" 0 | 1     which kernel family scans
 *   "realign_tma" 0 | 1                         cp.async.bulk or plain-load form of the page realign kernel
 *   "lz4_lanes" 0 | 1 | 2 (< 0 = default = 2)    LZ4 streams: eight lanes per stream | a lane per stream | by launch size
 *   "lz4_lane_warps" n                          (probe) warps per SM the lane-per-stream kernel spreads a launch over
 *   "peer_window" 0 | 1                         exchange steps over NCCL | over the IPC-mapped peer window; the same
 *                                               value on every rank
 * An unknown name is CG_EINVAL. */
int cg_set_option(const char *name, int64_t value);
struct CgScanDesc;
struct CgColumnDesc;
int cg_jit_compile_check(const struct CgScanDesc *desc, const struct CgColumnDesc *columns, int32_t natts, int64_t key_min,
						 int64_t key_max, int64_t max_rows, int32_t *kind, char *source, size_t source_len);
/* the same for the kernel form that reads NULL-bearing chunks: bit a of nullable_atts = attribute a may be NULL */
int cg_jit_compile_check_nullable(const struct CgScanDesc *desc, const struct CgColumnDesc *columns, int32_t natts, int64_t key_min,
								  int64_t key_max, int64_t max_rows, uint32_t nullable_atts, int32_t *kind, char *source,
								  size_t source_len);
/* Pin the calling thread (and threads it creates afterwards: the staging threads) to the CPUs
 * of the device's NUMA node, so that host pages it first-touches and the DMA reads of them stay
 * on the socket the GPU hangs off.  *node = the node, or -1 when nothing was changed (single
 * node, sysfs unreadable, cpuset excludes the node).  cg_numa_unbind restores the old mask. */
int cg_numa_bind(int32_t *node);
int cg_numa_unbind(void);
void cg_shutdown(void);

/* ---------------------------------------------------------------------------------- *
 *  Relation metadata: field-for-field what the reference keeps per stripe / chunk, in this header's own
 *  layout (NOT memory-compatible with ColumnChunkSkipNode / StripeMetadata: Datum min / max become int64 or
 *  float8 bits, bool / enum fields become int32); pg_glue/gpu_columnar_agg.c build_relation_image() converts.
 * ---------------------------------------------------------------------------------- */

/* include/columnar/columnar_compression.h:17-27 CompressionType */
enum { CG_COMPRESSION_NONE = 0, CG_COMPRESSION_PGLZ = 1, CG_COMPRESSION_LZ4 = 2, CG_COMPRESSION_ZSTD = 3 };

/* include/columnar/columnar.h:85-111 ColumnChunkSkipNode
 * (catalog columnar.chunk, backend/columnar/sql/citus_columnar--11.1-1.sql:48-64) */
typedef struct CgSkipNode
{
	int32_t has_minmax;
	int32_t compression_type;
	int64_t min_value;          /* by-value Datum: sign-extended integer or float8 bits */
	int64_t max_value;
	uint64_t row_count;
	uint64_t value_offset;      /* valueChunkOffset, relative to the stripe's file_offset */
	uint64_t value_length;
	uint64_t exists_offset;
	uint64_t exists_length;
	uint64_t decompressed_size; /* decompressedValueSize */
	int32_t compression_level;
	int32_t reserved;
} CgSkipNode;

/* include/columnar/columnar_metadata.h:21-42 StripeMetadata (catalog columnar.stripe) */
typedef struct CgStripe
{
	uint64_t id;
	uint64_t file_offset;       /* logical offset of the stripe (page aligned) */
	uint64_t data_length;
	uint64_t row_count;
	uint64_t first_row_number;
	uint32_t column_count;
	uint32_t chunk_row_count;   /* chunk_group_row_limit the stripe was written with */
	uint32_t chunk_count;
	uint32_t skipnode_base;     /* node(col,chunk) = nodes[skipnode_base + col*chunk_count + chunk] */
} CgStripe;

enum { CG_TYPE_INT = 0, CG_TYPE_FLOAT = 1,
	   /* by-reference (varlena) types whose values are scaled integers or one character: attlen = -1.
		* numeric(p, s): type_class = CG_TYPE_NUMERIC | s << 8; the column then behaves like an int8 column holding
		* value * 10^s (aggregate results carry the scale; cg_numeric_out prints them), a value with more fractional
		* digits than s, NaN or outside int64 fails the scan with CG_EUNSUPPORTED.  char(1): CG_TYPE_BPCHAR1, behaves
		* like a 1-byte integer column holding the character. */
	   CG_TYPE_NUMERIC = 2, CG_TYPE_BPCHAR1 = 3 };
#define CG_TYPE_NUMERIC_SCALE(s) (CG_TYPE_NUMERIC | ((s) << 8))

/* the slice of the TupleDesc the path needs (Form_pg_attribute attlen / attalign / type class) */
typedef struct CgColumnDesc
{
	int32_t attlen;     /* 1, 2, 4, 8: fixed-width by-value types; -1: varlena (CG_TYPE_NUMERIC / CG_TYPE_BPCHAR1 only) */
	int32_t type_class; /* CG_TYPE_* (low byte) | numeric scale << 8 */
} CgColumnDesc;

/* A columnar relation as the reader sees it: the main fork's 8 KB pages (as they sit in
 * shared_buffers / the file: 24-byte page header + 8168-byte payload, metapage in block 0,
 * data from block 2 -- backend/columnar/columnar_storage.c:21-31,117-126) + its visible
 * stripes and their skip lists (backend/columnar/columnar_metadata.c:717 ReadStripeSkipList). */
typedef struct CgRelation
{
	const uint8_t *pages;
	uint64_t nblocks;
	const CgStripe *stripes;
	int32_t nstripes;
	const CgSkipNode *nodes;
	int32_t nnodes;
	const CgColumnDesc *columns;
	int32_t natts;
} CgRelation;

/* ---------------------------------------------------------------------------------- *
 *  Query description: what the worker task's  Agg <- ColumnarScan  subtree computes
 *  (SURVEY.md 3.3).  Replaces ColumnarBeginRead(projectedColumnList, qualConditions)
 *  include/columnar/columnar.h:251-258 + the plan quals applied by ExecScan
 *  backend/columnar/columnar_customscan.c:1907-1913 + the worker half of the aggregate
 *  split planner/multi_logical_optimizer.c:3160-3484.
 * ---------------------------------------------------------------------------------- */
enum { CG_OP_LT = 0, CG_OP_LE = 1, CG_OP_EQ = 2, CG_OP_GE = 3, CG_OP_GT = 4, CG_OP_NE = 5 };

/* one conjunct "column <op> constant" of the WHERE list (btree operators) */
typedef struct CgQual
{
	int32_t column;   /* 0-based attribute index */
	int32_t op;       /* CG_OP_* */
	int64_t konst;    /* integer, or float8 bits for float columns */
} CgQual;

enum { CG_AGG_COUNT_STAR = 0, CG_AGG_COUNT = 1, CG_AGG_SUM = 2, CG_AGG_MIN = 3, CG_AGG_MAX = 4 };

/* aggregate argument = product over factors of (a + b * column); covers sum(x),
 * sum(x*y), sum(x*(1-d)), sum(x*(1-d)*(1+t)) on scaled-integer decimals (TPC-H Q1/Q6) */
typedef struct CgAggSpec
{
	int32_t kind;        /* CG_AGG_* */
	int32_t nfactors;    /* 0 (count(*)) .. 3 */
	int32_t column[3];
	int32_t is_float;    /* float8 arithmetic (sum is order dependent: tolerance, not bit-exact) */
	int64_t a[3];        /* integers, or float8 bits when is_float */
	int64_t b[3];
	int64_t term_abs_bound; /* integer SUM: caller-proven bound on |argument| (from the skip lists'
							 * min/max), 0 = unknown.  When bound * max_rows < 2^63 the sum is kept in
							 * one 64-bit word instead of two; a row that violates the bound fails the
							 * scan with CG_EINVAL (never a wrong answer). */
} CgAggSpec;

#define CG_MAX_QUALS 8
#define CG_MAX_AGGS 8
#define CG_MAX_GROUP_COLS 2
/* WHERE as a boolean tree over the atoms quals[0..nquals): postfix tokens, >= 0 = atom index,
 * CG_QX_AND / CG_QX_OR combine the two entries on top of the stack (PostgreSQL's BoolExpr; NOT is
 * folded into the operators).  nqual_expr = 0 means the plain AND of all atoms. */
#define CG_MAX_QEXPR 16
#define CG_QX_AND (-1)
#define CG_QX_OR (-2)

typedef struct CgScanDesc
{
	int32_t nquals;
	CgQual quals[CG_MAX_QUALS];
	int32_t enable_qual_pushdown;   /* columnar.enable_qual_pushdown (columnar_customscan.c:225-236) */
	int32_t ngroup_cols;            /* 0 = plain aggregate */
	int32_t group_cols[CG_MAX_GROUP_COLS];
	int32_t naggs;
	CgAggSpec aggs[CG_MAX_AGGS];
	int64_t expected_groups;        /* planner's group estimate; 0 = let the library size the table */
	/* [PG] ExecQual over AND/OR trees (columnar_customscan.c:1907-1913): a row passes iff the tree is TRUE
	 * under three-valued logic -- an atom on a NULL input is not TRUE.  Chunk-group skipping follows
	 * predicate_refuted_by for the base constraint of ONE column at a time (columnar_reader.c:1132-1187):
	 * an AND node is refuted when any arm is, an OR node when all arms are. */
	int32_t nqual_expr;
	int8_t qual_expr[CG_MAX_QEXPR];
	int32_t reserved;
} CgScanDesc;

/* EXPLAIN ANALYZE counters (columnar_customscan.c:1966-1999 and ExecScan instrumentation) */
typedef struct CgScanStats
{
	int64_t rows_scanned;            /* rows handed to the qual */
	int64_t rows_removed_by_filter;  /* "Rows Removed by Filter" */
	int64_t chunk_groups_filtered;   /* "Columnar Chunk Groups Removed by Filter" */
	int64_t rows_passed;
	int64_t chunk_groups_scanned;
	int64_t bytes_scanned;           /* algorithmic bytes: sum over projected columns of
									  * value bytes + exists bytes of the scanned chunk groups */
	double kernel_ms;                /* device time of the fused kernel(s), CUDA events */
	int64_t h2d_bytes;               /* cg_scan_relation: bytes copied host -> device */
} CgScanStats;

/* ---------------------------------------------------------------------------------- *
 *  Staged shards: the projected column chunks of a relation resident in HBM.
 *  Replaces LoadFilteredStripeBuffers / LoadColumnBuffers / ColumnarStorageRead
 *  (backend/columnar/columnar_reader.c:1007-1124, columnar_storage.c:463-492): each
 *  (column, chunk) exists/value buffer is copied out of the 8 KB pages into pinned
 *  memory at a 16-byte aligned slot and sent with cudaMemcpyAsync on a side stream.
 * ---------------------------------------------------------------------------------- */
typedef struct CgShard CgShard;

/* columns: attribute indexes to stage (NULL/0 = all).  The call returns when the shard
 * is resident.  Compressed value streams (lz4, pglz, zstd) are decoded on the GPU behind the copies. */
int cg_shard_stage(const CgRelation *rel, const int32_t *columns, int32_t ncolumns, CgShard **out);
void cg_shard_free(CgShard *shard);
uint64_t cg_shard_device_bytes(const CgShard *shard);
uint64_t cg_shard_rows(const CgShard *shard);

/* ---------------------------------------------------------------------------------- *
 *  Partial aggregate state: the device-resident group table a worker task accumulates
 *  (PostgreSQL nodeAgg's hash table + transition values, and on the coordinator the
 *  combine HashAggregate over sum(sum)/sum(count), multi_logical_optimizer.c:1807-1885,
 *  2231-2275).  One CgPartial may accumulate several shards of the same GPU (legal for
 *  the commutative/associative built-ins) or exactly one (a per-task result).
 * ---------------------------------------------------------------------------------- */
typedef struct CgPartial CgPartial;

/* key_min/key_max: exact bounds of the (packed) group key over the data to be scanned,
 * taken from the skip lists; when the domain is small the table is direct-indexed.
 * Pass key_min > key_max to force the general hash table. */
int cg_partial_create(const CgScanDesc *desc, const CgColumnDesc *columns, int32_t natts,
					  int64_t key_min, int64_t key_max, int64_t max_rows, CgPartial **out);
void cg_partial_free(CgPartial *p);
int cg_partial_reset(CgPartial *p);
/* Optimistic packing (on by default when the plan allows it): for a direct-indexed GROUP BY
 * with count(*) and a bounded integer sum, a row updates ONE 64-bit word
 * (sum << C | count) with one L2 reduction instead of two; packed words are drained into
 * the exact wide accumulators between launches.  A group that receives 2^C or more rows
 * between two drains would overflow its count field: this is detected exactly (the drained
 * counts must add up to the rows added) and reported as CG_ERETRY_UNPACKED by the calls that
 * read the partial -- never as a wrong result. */
int cg_partial_set_packing(CgPartial *p, int32_t enable);

/* Fused decode + filter + partial aggregate of one staged shard into `into`.
 * Chunk-group skipping (SelectedChunkMask, columnar_reader.c:1132-1187) runs on the host
 * from the skip nodes; surviving chunk groups are scanned by one kernel launch.
 * stats may be NULL. The call is asynchronous with respect to the host unless stats is
 * given (counters need the kernel to finish). */
int cg_scan_shard(const CgShard *shard, const CgScanDesc *desc, CgPartial *into, CgScanStats *stats);

/* End-to-end call on HOST buffers: stage + scan.  This is what a GpuColumnarAgg CustomScan
 * node calls once per shard task.  Pageable pages (shared_buffers as it is today) are
 * de-framed by host threads into pinned blocks and sent with cudaMemcpyAsync; pages in
 * pinned memory (cg_relation_register, or a shared_buffers segment registered once at
 * startup) are sent by the copy engine itself as runs of whole pages (1-D copies);
 * the GPU drops the page headers and re-aligns the chunk buffers. */
int cg_relation_register(const CgRelation *rel);      /* cudaHostRegister of the page image; CG_ECUDA if the OS
                                                        * refuses to pin it (the pages stay usable, as pageable) */
int cg_relation_unregister(const CgRelation *rel);
int cg_scan_relation(const CgRelation *rel, const CgScanDesc *desc, CgPartial *into, CgScanStats *stats);

/* Result rows.  Group order is unspecified (it is a hash aggregate).
 * For aggregate j of group i (index i*naggs + j):
 *   sum_hi/sum_lo  128-bit integer sum (two's complement), or float8 sum in fsum
 *   count          count(*) / count(x) value, or for sum/min/max the number of non-NULL
 *                  inputs (0 => the SQL result is NULL)
 *   minmax         min or max (integer, or float8 bits)
 * Any output pointer may be NULL. */
int cg_partial_ngroups(CgPartial *p, int64_t *ngroups);
int cg_partial_fetch(CgPartial *p, int64_t capacity, int64_t *keys, uint8_t *key_nulls,
					 int64_t *sum_hi, uint64_t *sum_lo, int64_t *count, int64_t *minmax,
					 double *fsum, int64_t *ngroups);

/* The inverse of cg_partial_fetch: partial-aggregate ROWS held on the host (group key + per aggregate the 128-bit
 * sum, count, min / max, float sum; arrays [nrows * naggs] laid out like cg_partial_fetch's) are folded into p by the
 * combine kernel.  What the coordinator does with the per-shard result rows it receives (adaptive_executor.c:3964-4189
 * ReceiveResults -> TupleDestination) in place of a CPU HashAggregate over them.  Arrays an aggregate list does not
 * need may be NULL.  count[] of a sum / min / max is its number of non-NULL inputs (0 = the partial was SQL NULL). */
int cg_partial_merge_values(CgPartial *p, int64_t nrows, const int64_t *keys, const uint8_t *key_nulls, const int64_t *sum_hi,
							const uint64_t *sum_lo, const int64_t *count, const int64_t *minmax, const double *fsum);
/* count / exact sum / min / max of one host column (attlen 1, 2, 4, 8; float4 is widened to float8 for min / max; a float
 * sum is not computed: its result depends on the order) in one pass: the batch step of the worker_partial_agg /
 * coord_combine_agg shims (utils/aggregate_utils.c:501-607, 820-1003), which otherwise pay one fmgr call per row. */
int cg_agg_column(int32_t attlen, int32_t is_float, const void *values, const uint8_t *isnull, int64_t n, int64_t *count,
				  int64_t *sum_hi, uint64_t *sum_lo, int64_t *min_value, int64_t *max_value);

/* Raw accumulator export / merge, for the combine step and for collectives.
 * A partial is `nwords` 64-bit accumulator words per group; every word is combined
 * with one commutative op (add / min / max / float add), so partials of different
 * shards or GPUs are merged word by word -- by this library (cg_partial_merge_rows)
 * or by ncclReduce on the dense layout. */
int cg_partial_layout(const CgPartial *p, int32_t *nwords, int32_t *word_ops /* [nwords] CG_WORD_* */,
					  int32_t *is_dense, int64_t *capacity);
enum { CG_WORD_ADD = 0, CG_WORD_MIN = 1, CG_WORD_MAX = 2, CG_WORD_FADD = 3, CG_WORD_FMIN = 4, CG_WORD_FMAX = 5 };

/* Compact occupied groups into device arrays owned by the caller (e.g. torch tensors):
 * d_keys[capacity], d_key_nulls[capacity] (may be NULL), d_words[capacity*nwords];
 * *nrows on the host. */
int cg_partial_export_device(CgPartial *p, int64_t capacity, int64_t *d_keys, uint8_t *d_key_nulls,
							 uint64_t *d_words, int64_t *nrows);
/* Merge rows (device arrays) into p: the coordinator-side combine kernel (K5). */
int cg_partial_merge_rows(CgPartial *p, const int64_t *d_keys, const uint8_t *d_key_nulls,
						  const uint64_t *d_words, int64_t nrows);
/* Plain-aggregate and direct-indexed tables only: device pointer and length (in 64-bit
 * words) of the whole accumulator array, laid out [entry][stride].  Two partials created
 * with the same arguments have identical layouts, so when every word op is CG_WORD_ADD a
 * collective (ncclReduce / ncclAllReduce, sum, int64) combines them in place. */
int cg_partial_dense_words(CgPartial *p, uint64_t **d_words, int64_t *total_words, int32_t *stride);
/* The same without a host synchronisation: pending table maintenance is only enqueued on the library's
 * stream (cg_set_stream), so a collective enqueued behind it on that stream reduces the finished table
 * and the host runs ahead.  The scan's error flags are not examined: call cg_partial_check (every rank,
 * after enqueuing the collective) before trusting the combined result. */
int cg_partial_dense_words_enqueue(CgPartial *p, uint64_t **d_words, int64_t *total_words, int32_t *stride);
/* Waits for the partial's pending work and reports what its kernels flagged. */
int cg_partial_check(CgPartial *p);

/* ---------------------------------------------------------------------------------- *
 *  Hash repartition (map side): worker_partition_query_result's per-row routing
 *  executor/partitioned_intermediate_results.c:493-553 + FindShardInterval
 *  utils/shardinterval_utils.c:260-452.  Keys and payload are device arrays.
 * ---------------------------------------------------------------------------------- */
/* partition index of every row: NULL key -> 0, else binary search of hashint4/8(key) (or of
 * the raw value for range partitioning) over [mins[i], maxs[i]].  key_len 4 or 8.
 * d_index[n] (int32), d_counts[P] (int64).  Returns CG_EINVAL if a hash falls in no range. */
int cg_partition_index(const int64_t *d_keys, const uint8_t *d_nulls, int64_t n, int32_t key_len,
					   int32_t by_hash, const int32_t *mins, const int32_t *maxs, int32_t P,
					   int32_t *d_index, int64_t *d_counts);
/* Stable scatter of `ncols` int64 payload columns into partition-contiguous order:
 * d_out[c][offsets[p] .. offsets[p+1]) holds partition p's rows in input order. */
int cg_partition_scatter(const int32_t *d_index, int64_t n, int32_t P, const int64_t *const *d_cols,
						 int32_t ncols, int64_t *const *d_out, int64_t *h_offsets /* [P+1] */);
/* Same, with the partitions laid out in a caller-chosen order: h_order[p] = output position of
 * partition p (a permutation; e.g. destination-rank-major for an all-to-all);
 * h_offsets[i] .. h_offsets[i+1] then delimit the partition whose position is i. */
int cg_partition_scatter_ordered(const int32_t *d_index, int64_t n, int32_t P, const int32_t *h_order,
								 const int64_t *const *d_cols, int32_t ncols, int64_t *const *d_out,
								 int64_t *h_offsets /* [P+1] */);

/* The return rows of worker_partition_query_result (partitioned_intermediate_results.c:270-291):
 * rows_written[P] and bytes_written[P] (host arrays), the bytes being what each partition's file
 * would hold in COPY text or binary format (worker/worker_sql_task_protocol.c:91-251).  d_cols:
 * ncols device arrays of int64 values; d_nulls: per column a device byte array or NULL; col_len:
 * the binary width of every column (4 for int4, 8 for int8).  A partition without rows has 0
 * bytes unless generate_empty_results (then a binary file still holds header + trailer). */
int cg_partition_copy_bytes(const int32_t *d_index, int64_t n, int32_t P, const int64_t *const *d_cols,
							const uint8_t *const *d_nulls, const int32_t *col_len, int32_t ncols, int32_t binary,
							int32_t generate_empty_results, int64_t *rows_written, int64_t *bytes_written);

/* The partition files themselves (what TaskFileDestReceiver writes, worker/worker_sql_task_protocol.c:91-251): the COPY text or
 * binary encoding of every row, rows of a partition in input order, the P files back to back in the device buffer d_out
 * (out_capacity bytes); file p is [file_offsets[p], file_offsets[p + 1]).  Sizes equal cg_partition_copy_bytes'. */
int cg_partition_copy_serialize(const int32_t *d_index, int64_t n, int32_t P, const int64_t *const *d_cols,
								const uint8_t *const *d_nulls, const int32_t *col_len, int32_t ncols, int32_t binary,
								int32_t generate_empty_results, uint8_t *d_out, int64_t out_capacity, int64_t *file_offsets /* [P + 1] */);

/* The merge side of a dual-repartition join for the aggregate query
 *     SELECT count(*), sum(b.payload + p.payload) FROM build b JOIN probe p USING (key)
 * over two co-located partitions that are already device arrays (what the MERGE task computes with
 * read_intermediate_results() + PostgreSQL's HashJoin + Agg, planner/multi_physical_planner.c:
 * 4304-4328, executor/intermediate_results.c:789-1045).  NULL keys join nothing; the sum is exact
 * (128-bit two's complement in sum_hi:sum_lo).  The joined rows are never materialised. */
int cg_join_count_sum(const int64_t *d_build_keys, const uint8_t *d_build_nulls, const int64_t *d_build_payload,
					  int64_t nbuild, const int64_t *d_probe_keys, const uint8_t *d_probe_nulls,
					  const int64_t *d_probe_payload, int64_t nprobe, int64_t *joined_rows, int64_t *sum_hi,
					  uint64_t *sum_lo);

/* ---------------------------------------------------------------------------------- *
 *  Exchange steps across GPUs (one process per GPU on one node; NVLink / NVSwitch, on the library's streams).
 *  Data moves through a peer window -- every rank's buffers mapped into every other rank with CUDA IPC, written
 *  and read by the library's own kernels -- with NCCL underneath for bootstrap, counts and agreements, and as the
 *  data path when the mapping is refused or switched off (cg_set_option("peer_window", 0) on every rank).
 *  Replaces the libpq funnel of the adaptive executor for GPU-resident results
 *  (executor/adaptive_executor.c:3964-4189 ReceiveResults + the combine query's HashAggregate,
 *  planner/multi_logical_optimizer.c:1807-1885, 2231-2275) and the file exchange of a repartition
 *  (executor/partitioned_intermediate_results.c:115-298, executor/intermediate_results.c:789-1045).
 * ---------------------------------------------------------------------------------- */
#define CG_COMM_ID_BYTES 128
/* rank 0 creates the id; the caller ships the bytes to every rank (over the coordinator's connections) */
int cg_comm_unique_id(uint8_t *id /* [CG_COMM_ID_BYTES] */);
int cg_comm_init(const uint8_t *id, int32_t rank, int32_t nranks);    /* collective; after cg_init; id may be NULL when nranks = 1 */
int cg_comm_rank(int32_t *rank, int32_t *nranks);
int cg_comm_destroy(void);
int cg_comm_barrier(void);
int cg_comm_peer_window(void);               /* 1: the peer window carries the combine and the exchange; 0: NCCL does */
enum { CG_COMM_SUM = 0, CG_COMM_MIN = 1, CG_COMM_MAX = 2 };
/* small host-side agreement (plan constants such as the key range; timings): values[i] <- op over ranks */
int cg_comm_allreduce_i64(int64_t *values, int32_t n, int32_t op);
/* Coordinator-side combine: after the call the partial of rank `root` holds the combined aggregate.  Collective:
 * EVERY rank calls it, passing the status of its own scans in local_status -- a rank that failed still takes
 * part, and every rank then returns an error instead of some of them hanging in a collective.  Direct-indexed
 * tables with additive words are reduced in place (the packed words alone when nothing else was written -- then by
 * the ranks themselves: rank s sums slice s of every rank's words over NVLink into the root's window);
 * other tables send their compacted rows to the root, which merges them.  Asynchronous on the library's
 * stream: errors raised by kernels of any rank surface on the root at the next call that reads the partial. */
int cg_comm_combine(CgPartial *p, int32_t root, int32_t local_status);
/* Hash repartition of this rank's rows (column 0 = the key) into P partitions, partition p owned by rank
 * p mod nranks.  Peer window: routing + histogram, the counts of all ranks, then ONE kernel that is scatter and
 * all-to-all at once -- rows leave shared memory as runs straight into the owner's receive buffer.  NCCL path:
 * scatter into destination-major order and one grouped ncclSend/ncclRecv of all columns on a second stream, so
 * that the next table's routing and scatter overlap this table's exchange.  Results live in the slot (0..3)
 * until its next use. */
int cg_comm_repartition_exchange(int32_t slot, const int64_t *const *d_cols, const uint8_t *d_key_nulls, int64_t n,
								 int32_t ncols, int32_t key_len, int32_t P, const int32_t *mins, const int32_t *maxs,
								 int64_t *recv_rows);
int cg_comm_exchange_wait(int32_t slot);      /* the library's compute stream waits (on the device) for the slot's exchange */
/* received columns (device pointers), rows, rows of every local partition by source rank [nlocal][nranks],
 * bytes sent to other ranks and the duration of the exchange on its stream; any pointer may be NULL */
int cg_comm_exchange_result(int32_t slot, int64_t **d_cols, int64_t *nrows, int64_t *part_counts, int32_t *nlocal,
							uint64_t *sent_bytes, double *exchange_ms);
/* the host-side plan of an exchange (exposed for tests): position[p] = place of partition p in destination-major
 * order; from counts[nranks][P] the rows this rank sends to / receives from every rank and the rows of its local
 * partitions by source rank.  counts may be NULL (positions and nlocal only). */
int cg_comm_exchange_plan(int32_t P, int32_t nranks, int32_t rank, const int64_t *counts, int32_t *position,
						  int64_t *send_rows, int64_t *recv_rows, int64_t *local_part_counts, int32_t *nlocal);
/* peer-window form: where this rank's rows land in the receive buffers of the ranks (pure host arithmetic over the
 * exchanged counts, counts[r * P + p]).  Positions [pos_begin[d], pos_begin[d + 1]) belong to rank d; rank d's buffer
 * has a column stride of total[d] rows; a row at index i of this rank's send order lands at adj[d] + i. */
int cg_comm_peer_plan(int32_t P, int32_t nranks, int32_t rank, const int64_t *counts, int32_t *pos_begin /* [nranks + 1] */,
					  int64_t *total /* [nranks] */, int64_t *adj /* [nranks] */);

/* The same join emitting its rows -- SELECT b.key, b.payload, p.payload FROM build b JOIN probe p USING (key) -- into device
 * arrays of `capacity` rows owned by the caller (row order unspecified, NULL keys join nothing).  *nrows = the number of
 * joined rows; with capacity 0 nothing is written (size the arrays, call again); a too small capacity is CG_EINVAL. */
int cg_join_rows(const int64_t *d_build_keys, const uint8_t *d_build_nulls, const int64_t *d_build_payload, int64_t nbuild,
				 const int64_t *d_probe_keys, const uint8_t *d_probe_nulls, const int64_t *d_probe_payload, int64_t nprobe,
				 int64_t capacity, int64_t *d_out_key, int64_t *d_out_build_payload, int64_t *d_out_probe_payload, int64_t *nrows);

/* exact bounds from the skip lists (min/max of every chunk that survives chunk-group
 * skipping): the packed group key range and |argument| of every aggregate (0 = unknown,
 * e.g. a chunk without min/max).  Feed them to cg_partial_create / CgAggSpec.term_abs_bound. */
int cg_relation_bounds(const CgRelation *rel, const CgScanDesc *desc, int64_t *key_min, int64_t *key_max,
					   int64_t *term_abs_bound /* [naggs] */, int64_t *rows);

/* ---------------------------------------------------------------------------------- *
 *  Host-side helpers that belong to the path.
 * ---------------------------------------------------------------------------------- */
/* SelectedChunkMask (columnar_reader.c:1132-1187): mask[chunk] for one stripe; returns the
 * number of chunk groups filtered through *filtered. */
int cg_selected_chunk_mask(const CgRelation *rel, int32_t stripe_index, const CgScanDesc *desc,
						   uint8_t *mask, int64_t *filtered);

/* numeric text of a 128-bit integer with `scale` fractional digits (sum(numeric) output) and
 * of the quotient sum/count with PostgreSQL's select_div_scale rule (avg output, the
 * master-side sum(sum)/sum(count), multi_logical_optimizer.c:1807-1830).  buf >= 64 bytes. */
int cg_numeric_out(int64_t hi, uint64_t lo, int32_t scale, char *buf, size_t buflen);
int cg_numeric_div_out(int64_t hi, uint64_t lo, int32_t scale, int64_t count, char *buf, size_t buflen);

/* ---------------------------------------------------------------------------------- *
 *  Synthetic shard writer (bench / test tooling; the on-disk encoding of
 *  backend/columnar/columnar_writer.c:391-654, compression none).
 * ---------------------------------------------------------------------------------- */
enum { CG_GEN_UNIFORM = 0, CG_GEN_SEQUENCE = 1 };
typedef struct CgGenColumn
{
	int32_t attlen;
	int32_t kind;           /* CG_GEN_* */
	int64_t lo;             /* uniform in [lo, hi) / sequence start */
	int64_t hi;
	uint32_t null_ppm;      /* NULL probability in parts per million */
	uint32_t reserved;
} CgGenColumn;

typedef struct CgGenRelation CgGenRelation;
/* value(row, col) = lo + splitmix64(seed ^ col<<56 ^ (first_row+row)) % (hi-lo)
 * null(row, col)  = splitmix64(~seed ^ col<<56 ^ (first_row+row)) % 1000000 < null_ppm */
int cg_gen_relation(const CgGenColumn *cols, int32_t natts, uint64_t nrows, uint64_t first_row,
					uint64_t seed, uint64_t stripe_row_limit, uint32_t chunk_row_limit,
					int32_t nthreads, CgGenRelation **out);
/* Encode caller-supplied columns (values[c][row] int64 / float8 bits, nulls[c] may be NULL). */
int cg_write_relation(const CgColumnDesc *cols, int32_t natts, const int64_t *const *values,
					  const uint8_t *const *nulls, uint64_t nrows, uint64_t stripe_row_limit,
					  uint32_t chunk_row_limit, CgGenRelation **out);
/* columnar.compression of the relations written after the call: CG_COMPRESSION_NONE,
 * CG_COMPRESSION_LZ4 or CG_COMPRESSION_ZSTD (liblz4's LZ4_compress_default / libzstd's
 * ZSTD_compress at level 3, as the reference's CompressBuffer) */
int cg_gen_set_compression(int32_t compression);
int cg_gen_relation_view(const CgGenRelation *g, CgRelation *view);
void cg_gen_relation_free(CgGenRelation *g);

#ifdef __cplusplus
}
#endif
#endif /* CITUS_GPU_H */
