/*
 * dbx.h — C-ABI of libdbx, the B200-native replacement for Databend's in-memory
 * vectorised execution hot path (filter -> hash aggregate / hash join / top-k /
 * vector distance).
 *
 * The reference has no FFI on this path: the boundary is a set of Rust traits.
 * Every entry point below names the reference interface it replaces, so that a
 * thin Rust `-sys` crate + shim `impl`s (see INTEGRATION.md) can forward the
 * trait calls here unchanged:
 *
 *   Processor / Transform adaptors     src/query/pipeline/src/core/processor.rs:62-108
 *                                      src/query/pipeline/transforms/src/processors/transforms/transform.rs:30-48
 *                                      .../transform_accumulating.rs:30-37
 *   DataBlock / BlockEntry / Column    src/query/expression/src/block.rs:49-60, values.rs:192-215
 *   Buffer<T> / Bitmap                 src/common/column/src/buffer/immutable.rs:60-73, bitmap/immutable.rs
 *   FilterExecutor / SelectExpr        src/query/expression/src/filter/filter_executor.rs:82-160,
 *                                      filter/select_expr.rs:34-50
 *   AggregateHashTable + transforms    src/query/expression/src/aggregate/aggregate_hashtable.rs:168-408,
 *                                      service/.../aggregator/transform_aggregate_{partial,final}.rs
 *   Join trait                         service/.../new_hash_join/join.rs:26-53
 *   sort / TopN                        src/query/expression/src/kernels/sort.rs:91-111, top_n/
 *   cosine_distance / l2_distance      src/common/vector/src/distance.rs:19-35,65-80
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch types cross this boundary;
 *   - every function returns a dbx_status (0 = ok); the message of the last failure
 *     on a handle is read with dbx_last_error(handle) (NULL handle = thread-local
 *     error of the failed create call).  Nothing aborts or throws across the ABI;
 *   - a handle is thread-compatible (one caller at a time, may migrate between
 *     threads), distinct handles are fully concurrent: each owns one CUDA stream;
 *   - input blocks are borrowed until the operator has consumed them.  Pageable host memory is
 *     consumed before push returns.  PINNED host memory (dbx_host_alloc / dbx_host_register) and
 *     DEVICE memory are read asynchronously on the handle's stream: the caller must not modify or
 *     recycle those buffers before dbx_op_inputs_consumed(op) (or any later dbx_op_finish /
 *     dbx_op_synchronize on the handle) has returned;
 *   - output blocks are owned by the library until dbx_block_release().
 */
#ifndef DBX_H_
#define DBX_H_

#ifndef __CUDACC_RTC__ /* run-time compiled kernels get the fixed-width types from common.cuh */
#include <stddef.h>
#include <stdint.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define DBX_ABI_VERSION 1

/* ---------------------------------------------------------------- status */
typedef enum dbx_status {
  DBX_OK = 0,
  DBX_ERR_INVALID = 1,       /* bad argument / unsupported combination (ErrorCode::BadArguments at build time) */
  DBX_ERR_CUDA = 2,          /* CUDA runtime failure (ErrorCode::Internal) */
  DBX_ERR_BAD_ARGUMENTS = 3, /* per-row evaluation error, e.g. "Division by zero" (evaluator.rs:234-244) */
  DBX_ERR_UNSUPPORTED = 4,   /* valid in the reference but not built here */
  DBX_ERR_OOM = 5,
  DBX_ERR_STATE = 6,         /* call order violated (push after finish, ...) */
  DBX_ERR_NO_DEVICE = 7      /* no usable CUDA device: there is NO CPU fallback */
} dbx_status;

/* ------------------------------------------------------------- data types */
/* NumberDataType subset (src/query/expression/src/types/number.rs) + Boolean + Vector(Float32) */
typedef enum dbx_dtype {
  DBX_BOOL = 0, /* bit-packed, LSB first (Bitmap) */
  DBX_I8 = 1,
  DBX_I16 = 2,
  DBX_I32 = 3,
  DBX_I64 = 4,
  DBX_U8 = 5,
  DBX_U16 = 6,
  DBX_U32 = 7,
  DBX_U64 = 8,
  DBX_F32 = 9,
  DBX_F64 = 10,
  DBX_VEC_F32 = 11 /* VectorColumn::Float32((Buffer<F32>, dim)), flat row-major (types/vector.rs:377-380) */
} dbx_dtype;

/* OR-ed into the entries of dbx_op_create's input_types[] when the column's DataType is
 * Nullable(T) (nullability is part of the schema in the reference: types/nullable.rs). */
#define DBX_NULLABLE 0x100

typedef enum dbx_mem { DBX_MEM_HOST = 0, DBX_MEM_DEVICE = 1 } dbx_mem;

/* A constant (BlockEntry::Const payload, or a literal in an expression). */
typedef struct dbx_scalar {
  int32_t dtype;
  int32_t is_null;
  union {
    int64_t i64;
    uint64_t u64;
    double f64;
  } v;
} dbx_scalar;

/* Column = Buffer<T> (+ optional validity Bitmap with a BIT offset, as left by
 * Bitmap::slice).  `is_const` mirrors BlockEntry::Const(Scalar, DataType, n):
 * the value is in `konst`, `data` is ignored and nothing is materialised. */
typedef struct dbx_column {
  int32_t dtype;               /* dbx_dtype */
  int32_t mem;                 /* dbx_mem: where data/validity live */
  int32_t is_const;
  int32_t vec_dim;             /* DBX_VEC_F32 only */
  int64_t len;                 /* rows */
  const void* data;            /* T[len] (bool: bit-packed; vec: f32[len*vec_dim]) */
  int64_t data_bit_offset;     /* DBX_BOOL only: bit offset of row 0 */
  const uint8_t* validity;     /* NULL = no nulls; else LSB-first bitmap, 1 = valid */
  int64_t validity_bit_offset;
  int64_t null_count;          /* -1 = unknown */
  dbx_scalar konst;
} dbx_column;

/* DataBlock{entries, num_rows, meta}.  `meta` carries BlockMetaInfo-like side
 * channels that stay on the device (partial aggregate payloads, block.rs:370-440). */
typedef struct dbx_block {
  int64_t num_rows;
  int32_t num_cols;
  int32_t reserved;
  dbx_column* cols;
  void* meta;    /* opaque: dbx partial-payload reference, or NULL */
  void* owner;   /* library-owned outputs: released by dbx_block_release */
} dbx_block;

/* ------------------------------------------------------------- predicates */
/* Flattened SelectExpr tree in postfix order (filter/select_expr.rs:34-50):
 *   And / Or                   -> DBX_PRED_AND / DBX_PRED_OR (pop n_children results)
 *   Compare(op, lhs, rhs)      -> DBX_PRED_CMP with two operands
 *   BooleanColumn              -> DBX_PRED_BOOLCOL (a DBX_BOOL column, NULL counts as false)
 *   BooleanScalar              -> DBX_PRED_CONST
 * Operands are column refs, literals, or `column <arith> literal` — the one level of
 * scalar evaluation the configs need (modulo: arithmetic_modulo.rs:29-97).           */
typedef enum dbx_cmp_op { DBX_EQ = 0, DBX_NE = 1, DBX_LT = 2, DBX_LE = 3, DBX_GT = 4, DBX_GE = 5 } dbx_cmp_op;
typedef enum dbx_arith_op { DBX_ARITH_NONE = 0, DBX_ARITH_MODULO = 1 } dbx_arith_op;
typedef enum dbx_pred_kind { DBX_PRED_CMP = 0, DBX_PRED_AND = 1, DBX_PRED_OR = 2, DBX_PRED_BOOLCOL = 3, DBX_PRED_CONST = 4 } dbx_pred_kind;

typedef struct dbx_operand {
  int32_t is_const;   /* 1: literal `c`; 0: column `col` (optionally `col <arith> c`) */
  int32_t col;        /* column index in the pushed block */
  int32_t arith;      /* dbx_arith_op applied as  col <arith> c */
  int32_t reserved;
  dbx_scalar c;
} dbx_operand;

typedef struct dbx_pred_node {
  int32_t kind;       /* dbx_pred_kind */
  int32_t cmp;        /* dbx_cmp_op          (DBX_PRED_CMP) */
  int32_t n_children; /* operand count       (DBX_PRED_AND / DBX_PRED_OR), >= 2 */
  int32_t value;      /* DBX_PRED_CONST: 0/1; DBX_PRED_BOOLCOL: column index */
  dbx_operand lhs, rhs;
} dbx_pred_node;

#define DBX_MAX_PRED_NODES 16
typedef struct dbx_predicate {
  int32_t n_nodes;    /* 0 = no filter (all rows pass) */
  int32_t reserved;
  dbx_pred_node nodes[DBX_MAX_PRED_NODES];
} dbx_predicate;

/* ------------------------------------------------------------- aggregates */
/* AggregateFunctionFactory names (aggregate_function_factory.rs:189-247); all are
 * wrapped by the OrNull adaptor exactly as the factory does:  sum/avg/min/max return
 * Nullable(T) (NULL iff no non-NULL input row), count returns plain UInt64.           */
typedef enum dbx_agg_kind { DBX_AGG_SUM = 0, DBX_AGG_COUNT = 1, DBX_AGG_AVG = 2, DBX_AGG_MIN = 3, DBX_AGG_MAX = 4 } dbx_agg_kind;

typedef struct dbx_agg_desc {
  int32_t kind;     /* dbx_agg_kind */
  int32_t arg_col;  /* argument column index in the pushed block; -1 = count(*) */
} dbx_agg_desc;

#define DBX_MAX_AGGS 8
#define DBX_MAX_GROUP_COLS 4

/* AggregatorParams (aggregator_params.rs:30-78) + the fused predicate. */
typedef struct dbx_agg_params {
  int32_t n_group_cols;                 /* 0 = no GROUP BY (transform_single_key.rs) */
  int32_t group_cols[DBX_MAX_GROUP_COLS];
  int32_t n_aggs;
  dbx_agg_desc aggs[DBX_MAX_AGGS];
  dbx_predicate filter;                 /* fused TransformFilter in front (n_nodes = 0: none) */
  int64_t expected_groups;              /* cardinality hint, 0 = unknown (table grows on demand) */
} dbx_agg_params;

/* ----------------------------------------------------------------- top-k */
/* SortColumnDescription{offset, asc, nulls_first} + LimitType::{LimitRows(k), None}
 * (kernels/sort.rs:41-63).  Order: OrderedFloat (NaN greatest, -0 == +0); ties keep row order.
 * limit = 0 (LimitType::None) sorts the whole input (device radix sort, up to 2^30 - 1 rows);
 * 1 <= limit <= 4 Mi runs the streaming top-k.  Result block: [key, row_id Int64]. */
#define DBX_MAX_SORT_KEYS 4
typedef struct dbx_topk_params {
  int32_t key_col;
  int32_t asc;
  int32_t nulls_first;
  int32_t reserved;
  int64_t limit;
  /* ORDER BY key_col, extra_key_cols[0], extra_key_cols[1], ... (SortColumnDescription list,
   * kernels/sort.rs:43-60): ties on the earlier keys are broken by the later ones, each with its own
   * direction and NULL placement, and finally by input order.  With extra keys the whole input is
   * sorted on the device (one stable radix sort per key, least significant first) and `limit` > 0
   * cuts the sorted result.  Result block: [key (first key), row_id Int64] as for one key. */
  int32_t n_extra_keys; /* 0 .. DBX_MAX_SORT_KEYS - 1 */
  int32_t extra_key_cols[DBX_MAX_SORT_KEYS - 1];
  int32_t extra_asc[DBX_MAX_SORT_KEYS - 1];
  int32_t extra_nulls_first[DBX_MAX_SORT_KEYS - 1];
} dbx_topk_params;

/* ------------------------------------------------------------------ join */
/* INNER: probe columns then build columns per matching pair (inner_join.rs:236-245).
 * LEFT_SEMI / LEFT_ANTI (probe side is "left"): the probe rows with at least one / with no match,
 * probe columns only (left_join_semi.rs, left_join_anti.rs; a NULL probe key never matches, so
 * ANTI keeps the row).
 * LEFT (outer, probe side preserved; left_join.rs): every probe row; rows without a match carry
 * NULL in all build columns, which therefore come back Nullable.  Output row order is unspecified. */
typedef enum dbx_join_kind { DBX_JOIN_INNER = 0, DBX_JOIN_LEFT_SEMI = 1, DBX_JOIN_LEFT_ANTI = 2, DBX_JOIN_LEFT = 3 } dbx_join_kind;
typedef struct dbx_join_params {
  int32_t kind;          /* dbx_join_kind */
  int32_t build_key_col; /* key column index in build blocks */
  int32_t probe_key_col; /* key column index in probe blocks */
  int32_t n_build_cols;  /* dbx_op_create's input_types = build schema (n_build_cols) then probe schema */
  int64_t expected_build_rows; /* hint; 0 = unknown */
} dbx_join_params;

/* -------------------------------------------------------- vector distance */
typedef enum dbx_distance_kind { DBX_DIST_COSINE = 0, DBX_DIST_L2 = 1 } dbx_distance_kind;

/* ----------------------------------------------------------- operator API */
typedef enum dbx_op_kind {
  DBX_OP_FILTER = 0,              /* TransformFilter (filters/filter_predicate.rs:35-104) */
  DBX_OP_AGG_PARTIAL = 1,         /* [TransformFilter ->] TransformPartialAggregate / PartialSingleStateAggregator */
  DBX_OP_AGG_FINAL = 2,           /* TransformFinalAggregate / FinalSingleStateAggregator */
  DBX_OP_TOPK = 3,                /* TransformSortPartial+merge with LIMIT / TransformPartialTopN+FinalTopN */
  DBX_OP_JOIN = 4                 /* Join trait: add_block / final_build / probe_block / final_probe */
} dbx_op_kind;

typedef struct dbx_op dbx_op; /* opaque operator handle */

/* Library / device */
int32_t dbx_abi_version(void);
int32_t dbx_device_count(int32_t* n);                 /* DBX_ERR_NO_DEVICE when none */
const char* dbx_last_error(const dbx_op* op);         /* op == NULL: error of the last failed create on this thread */

/* Pinned host buffers (Buffer::from foreign allocation hook, buffer/mod.rs:26-48) */
int32_t dbx_host_alloc(size_t bytes, void** out);
int32_t dbx_host_free(void* p);
int32_t dbx_host_register(void* p, size_t bytes);     /* pin caller-owned memory for direct DMA */
int32_t dbx_host_unregister(void* p);

/* Device buffers for device-resident pipelines (tests, bench, op->op hand-off) */
int32_t dbx_device_alloc(int32_t device, size_t bytes, void** out);
int32_t dbx_device_free(int32_t device, void* p);
int32_t dbx_memcpy_h2d(int32_t device, void* dst, const void* src, size_t bytes);
int32_t dbx_memcpy_d2h(int32_t device, void* dst, const void* src, size_t bytes);
int32_t dbx_memcpy_d2d(int32_t device, void* dst, const void* src, size_t bytes);
int32_t dbx_device_synchronize(int32_t device);

/* Operator lifecycle.  `params` is the struct matching `kind`
 * (FILTER: dbx_predicate, AGG_*: dbx_agg_params, TOPK: dbx_topk_params, JOIN: dbx_join_params).
 * `input_types[n_input_cols]` are the dbx_dtype of the block columns that will be pushed
 * (DataSchema of the upstream pipe); nullability is taken per block from `validity`. */
int32_t dbx_op_create(int32_t kind, const void* params, const int32_t* input_types, int32_t n_input_cols,
                      int32_t device, dbx_op** out);
int32_t dbx_op_destroy(dbx_op* op);

/* Transform::transform / AccumulatingTransform::transform / Join::add_block(build side) */
int32_t dbx_op_push(dbx_op* op, const dbx_block* block);
/* AccumulatingTransform::on_finish / Join::final_build */
int32_t dbx_op_finish(dbx_op* op);
/* Pull the next output block: *has_block = 0 when drained.  `out_mem` selects where the
 * output columns live (host: pinned, zero-copy wrappable; device: stays in HBM). */
int32_t dbx_op_pull(dbx_op* op, int32_t out_mem, dbx_block* out, int32_t* has_block);
int32_t dbx_block_release(dbx_block* block);
/* Re-arm a finished operator for the next query with the same parameters, keeping its
 * device allocations (operator pooling; the table is re-initialised on the device). */
int32_t dbx_op_reset(dbx_op* op);
/* Block until everything enqueued on the handle's stream has completed. */
int32_t dbx_op_synchronize(dbx_op* op);
/* Block until every block pushed so far has been read completely (host->device copies done,
 * kernels that read device-resident inputs finished): the point after which the caller may
 * reuse pinned-host / device input buffers (the Arc<Buffer> of the reference can be dropped). */
int32_t dbx_op_inputs_consumed(dbx_op* op);

/* Join probe side: Join::probe_block(block) -> JoinStream::next()* ; output blocks are
 * pulled with dbx_op_pull until drained.  Join::final_probe is a no-op for inner joins. */
int32_t dbx_join_probe(dbx_op* op, const dbx_block* block);

/* AGG_FINAL input: hand over a partial operator's device-resident payload
 * (AggregateMeta::AggregatePayload, aggregate_meta.rs) without leaving HBM. */
int32_t dbx_agg_final_merge_partial(dbx_op* final_op, dbx_op* partial_op);

/* Multi-GPU exchange support for the partial->final shuffle (build_partition_bucket.rs:41-131,
 * partitioned_payload.rs:44-57): scatter the finished partial's groups into `n_parts`
 * owner-contiguous runs of fixed-width rows [key:8][state words...] in one device buffer.
 * part_offsets[n_parts+1] is written on the HOST.  Rows are `row_bytes` wide. */
int32_t dbx_agg_partial_partition(dbx_op* partial_op, int32_t n_parts, void** dev_rows, int64_t* part_offsets,
                                  int32_t* row_bytes);
/* AGG_FINAL: merge `n_rows` such rows (device memory, e.g. the all-to-all receive buffer). */
int32_t dbx_agg_final_merge_rows(dbx_op* final_op, const void* dev_rows, int64_t n_rows);

/* Partial states in the reference's spill / cluster wire layout (AggregatorParams::spill_schema,
 * aggregator_params.rs:103-117; aggregator/serde/...): one Tuple column `agg_i` per aggregate function
 * holding its serialised state, then the group columns.  The C-ABI carries each tuple FLATTENED into
 * consecutive columns — [agg_0.0, agg_0.1, ..., agg_{n-1}.k, group_0, ...] — and reports the arity of
 * every tuple, so the binding rebuilds Column::Tuple without copying:
 *   count            (UInt64 count)                          aggregate_count.rs:170
 *   sum(T)           (Sum<T> value, flags...)                aggregate_sum.rs:155
 *   avg(T)           (Sum<T> sum, UInt64 count, flags...)    aggregate_avg.rs:106
 *   min / max(T)     (Boolean has, T value, flags...)        aggregate_min_max_any.rs:315
 * flags = one Boolean for the null adaptor of a Nullable argument, then one for the or-null adaptor
 * (aggregate_null_adaptor.rs:508, aggregate_ornull_adaptor.rs:184); Sum<T> = Int64 / UInt64 / Float64.
 * A GPU partial can so feed the reference's CPU TransformFinalAggregate, and a CPU partial (or a GPU
 * partial on another node) can feed a GPU final. */
int32_t dbx_agg_partial_serialize(dbx_op* partial_op, int32_t out_mem, dbx_block* out, int32_t* tuple_arity /* [n_aggs] */);
int32_t dbx_agg_final_merge_serialized(dbx_op* final_op, const dbx_block* block);

/* Peer-memory exchange of aggregate partials between the GPUs of one box (one process per GPU):
 * the multi-GPU form of the partial -> final shuffle (build_partition_bucket.rs:41-131; between
 * nodes the reference ships AggregateMeta partitions over Arrow Flight,
 * servers/flight/v1/exchange/...).  Every rank creates an exchange (a receive buffer in its HBM),
 * the 64-byte CUDA-IPC handles are all-gathered by the host (torch.distributed / any transport)
 * and passed to connect; then per query
 *     scatter(partial)  partition + store rows straight into the owners' buffers over NVLink
 *     merge(final)      wait (on the device) for every source's release flag, merge the regions
 * with no NCCL call, staging copy or host synchronisation on the data path.
 * region_rows = 0 sizes a region for the worst case (all groups of one source to one owner). */
typedef struct dbx_agg_exchange dbx_agg_exchange;
int32_t dbx_agg_exchange_create(dbx_op* partial_op, int32_t rank, int32_t n_ranks, int64_t region_rows,
                                dbx_agg_exchange** out, void* ipc_handle_out /* 64 bytes, may be NULL */);
int32_t dbx_agg_exchange_local_buffer(dbx_agg_exchange* x, void** base, int64_t* region_rows, int32_t* row_bytes);
int32_t dbx_agg_exchange_connect(dbx_agg_exchange* x, const void* all_handles /* n_ranks x 64 B */,
                                 void* const* same_process_ptrs /* or the buffers themselves */);
int32_t dbx_agg_exchange_scatter(dbx_agg_exchange* x, dbx_op* partial_op);
int32_t dbx_agg_exchange_merge(dbx_agg_exchange* x, dbx_op* final_op);
/* Per-phase device times (ms, CUDA events) of the last scatter/merge pair: out8[0] scatter kernel,
 * [1] wait for the peers' release flags, [2] merge kernel, [3] finalize (merge end -> result
 * columns ready), [4] the wait kernel's own measure of its spin; [5..7] reserved.  Call after the
 * final operator's finish(). */
int32_t dbx_agg_exchange_phase_ms(dbx_agg_exchange* x, float* out8);
int32_t dbx_agg_exchange_destroy(dbx_agg_exchange* x);
const char* dbx_agg_exchange_last_error(const dbx_agg_exchange* x);

/* Hash-partition the rows of a device-resident block by the owner of an integer key column
 * (same owner rule as the aggregate exchange): the step in front of the all-to-all of a
 * partitioned hash join (flight_scatter_hash.rs).  out_cols[c] are caller-allocated device
 * buffers of num_rows values; partition p occupies rows [part_offsets[p], part_offsets[p+1])
 * (part_offsets is HOST memory, n_parts + 1 entries).  Row order inside a partition is unspecified. */
int32_t dbx_hash_partition(int32_t device, const dbx_block* block, int32_t key_col, int32_t n_parts,
                           void* const* out_cols, int64_t* part_offsets);

/* Hash-partitioned row shuffle between the GPUs of one box over peer memory — the exchange in
 * front of a partitioned hash join (flight_scatter_hash.rs:86-125 + the Flight exchange): ONE
 * kernel partitions a device-resident block by the owner of its key (same owner rule as
 * dbx_hash_partition / the aggregate exchange) and stores every row straight into the owner's
 * receive region over NVLink.  Collective protocol: every rank alternates send / recv; recv
 * returns one device-resident block per source rank (views into the receive buffer, valid until
 * this rank's next-but-one send); a rank must be done reading them before its next send.
 * col_types: dbx_dtype per column (fixed-width numeric, not nullable); region_rows: capacity of
 * one (source, owner) region = the largest block a rank may send. */
typedef struct dbx_shuffle dbx_shuffle;
int32_t dbx_shuffle_create(int32_t device, int32_t rank, int32_t n_ranks, const int32_t* col_types, int32_t n_cols, int32_t key_col,
                           int64_t region_rows, dbx_shuffle** out, void* ipc_handle_out /* 64 bytes, may be NULL */);
int32_t dbx_shuffle_local_buffer(dbx_shuffle* s, void** base);
int32_t dbx_shuffle_connect(dbx_shuffle* s, const void* all_handles /* n_ranks x 64 B */, void* const* same_process_ptrs);
int32_t dbx_shuffle_send(dbx_shuffle* s, const dbx_block* block);
int32_t dbx_shuffle_recv(dbx_shuffle* s, dbx_block* blocks /* n_ranks */, dbx_column* cols /* n_ranks x n_cols */);
int32_t dbx_shuffle_last_ms(dbx_shuffle* s, float* send_ms, float* wait_ms);
int32_t dbx_shuffle_destroy(dbx_shuffle* s);
const char* dbx_shuffle_last_error(const dbx_shuffle* s);

/* DataBlock kernels (src/query/expression/src/kernels): every column kind libdbx carries
 * (numeric, Boolean, Vector(Float32), Nullable, Const).  Inputs may live on the host or the
 * device; outputs are library-owned blocks (dbx_block_release) in `out_mem`.
 *   take          take.rs:43-60     out row i = block row indices[i]
 *   take_ranges   take_ranges.rs:40 concatenation of the row ranges [starts[r], starts[r] + lens[r])
 *   scatter       scatter.rs:21     row i goes to outs[indices[i]], input order kept inside each output
 *   concat        concat.rs:62      blocks appended in order (Const entries stay Const only when all agree) */
int32_t dbx_block_take(int32_t device, const dbx_block* block, const uint32_t* indices, int64_t n_indices, int32_t indices_mem,
                       int32_t out_mem, dbx_block* out);
int32_t dbx_block_take_ranges(int32_t device, const dbx_block* block, const uint32_t* starts, const uint32_t* lens, int64_t n_ranges,
                              int32_t out_mem, dbx_block* out);
int32_t dbx_block_scatter(int32_t device, const dbx_block* block, const uint32_t* indices, int32_t indices_mem, int32_t n_parts,
                          int32_t out_mem, dbx_block* outs /* n_parts */);
int32_t dbx_block_concat(int32_t device, const dbx_block* blocks, int32_t n_blocks, int32_t out_mem, dbx_block* out);

/* ------------------------------------------------------------ expressions */
/* Evaluator::run over a block (evaluator.rs:247-465) for numeric / boolean expressions: a postfix
 * program of column refs, constants, casts and function calls.  Result types follow the
 * reference's ResultTypeOfBinary rules (arithmetics_type.rs), values its arithmetic (wrapping
 * integer +,-,*; `/` in Float64 with "divided by zero"; `div` through Float64; modulo in the
 * LeastSuper type with "Division by zero"; to_<type> casts with "number overflowed", rounding
 * float -> int like numeric_cast_option = 'rounding'); NULL propagates (passthrough_nullable),
 * and / or are three-valued.  One fused kernel: inputs read once, one output column written. */
typedef enum dbx_expr_kind { DBX_EXPR_COLUMN = 0, DBX_EXPR_CONST = 1, DBX_EXPR_CAST = 2, DBX_EXPR_CALL = 3 } dbx_expr_kind;
typedef enum dbx_func {
  DBX_FN_PLUS = 0, DBX_FN_MINUS = 1, DBX_FN_MULTIPLY = 2, DBX_FN_DIVIDE = 3, DBX_FN_DIV = 4, DBX_FN_MODULO = 5, DBX_FN_NEGATE = 6,
  DBX_FN_EQ = 7, DBX_FN_NOTEQ = 8, DBX_FN_LT = 9, DBX_FN_LTE = 10, DBX_FN_GT = 11, DBX_FN_GTE = 12,
  DBX_FN_AND = 13, DBX_FN_OR = 14, DBX_FN_NOT = 15, DBX_FN_IS_NULL = 16, DBX_FN_IS_NOT_NULL = 17
} dbx_func;
typedef struct dbx_expr_node {
  int32_t kind;     /* dbx_expr_kind */
  int32_t func;     /* dbx_func (DBX_EXPR_CALL); arguments are the 1 or 2 values below it on the stack */
  int32_t col;      /* DBX_EXPR_COLUMN: column index in the block */
  int32_t cast_to;  /* DBX_EXPR_CAST: dbx_dtype */
  int32_t try_cast; /* DBX_EXPR_CAST: 1 = try_to_<type> (failure gives NULL instead of an error) */
  int32_t reserved;
  dbx_scalar c;     /* DBX_EXPR_CONST */
} dbx_expr_node;
#define DBX_MAX_EXPR_NODES 32
typedef struct dbx_expr {
  int32_t n_nodes;
  int32_t reserved;
  dbx_expr_node nodes[DBX_MAX_EXPR_NODES];
} dbx_expr;
/* out: library-owned block with ONE column (dbx_block_release); *out_dtype = its dbx_dtype
 * (| DBX_NULLABLE).  A per-row evaluation error returns DBX_ERR_BAD_ARGUMENTS with the reference's
 * message in dbx_last_error(NULL) and the first failing row in *first_error_row. */
int32_t dbx_eval_scalar(int32_t device, const dbx_expr* expr, const dbx_block* block, int32_t out_mem, dbx_block* out,
                        int32_t* out_dtype, int64_t* first_error_row);

/* ScalarFunction::eval replacement for the vector distances (scalars/vector.rs:497-556):
 * out[i] = distance(lhs[i], rhs[i]) row-wise, either side may be const.  f32 result. */
int32_t dbx_eval_distance(int32_t kind, int32_t device, const dbx_column* lhs, const dbx_column* rhs,
                          dbx_column* out /* caller-provided f32 buffer, mem as given */);

/* Brute-force kNN: `ORDER BY cosine_distance(c, q) LIMIT k` for a batch of queries, i.e.
 * the EvalScalar -> TopN pipeline of SURVEY 3.5 fused: tensor-core GEMM for candidate
 * selection, exact fp32 re-evaluation of the returned distances.
 * corpus: DBX_VEC_F32 [n, dim]; queries: DBX_VEC_F32 [nq, dim];
 * out_idx[nq*k] (int64 row ids), out_dist[nq*k] (f32), ascending by distance (NaN last). */
typedef struct dbx_knn dbx_knn;
int32_t dbx_knn_create(int32_t kind, int32_t device, const dbx_column* corpus, dbx_knn** out);
int32_t dbx_knn_search(dbx_knn* h, const dbx_column* queries, int32_t k, int32_t out_mem, int64_t* out_idx,
                       float* out_dist);
int32_t dbx_knn_destroy(dbx_knn* h);
/* Device time (ms, CUDA events) and launch count of the tensor-core similarity passes of the last search. */
int32_t dbx_knn_last_gemm_ms(dbx_knn* h, float* ms, int64_t* launches);
/* Instrumentation of the last search: out8[0] queries whose result the certificate proved exact,
 * out8[1] queries answered by the exact (CUDA-core, row-wise) path, out8[2] candidates re-ranked,
 * out8[3] similarity passes, out8[4] cluster size of the GEMM, out8[5] its grid (CTAs),
 * out8[6] / out8[7] host wall microseconds of the similarity passes / of re-rank + certificate. */
int32_t dbx_knn_last_stats(dbx_knn* h, int64_t* out8);
const char* dbx_knn_last_error(const dbx_knn* h);

/* Deterministic synthetic column generator (counter-based: splitmix64(seed + row)),
 * used by tests and bench so host oracle and device data agree bit-for-bit.
 *   kind 0: int64 uniform in [0, a)            (mulhi(r, a))
 *   kind 1: int64 uniform in [-2^31, 2^31)     (sign-extended high 32 bits)
 *   kind 2: float64 = (double)(r >> (64-a))    integer-valued in [0, 2^a)
 *   kind 3: float64 uniform [0,1) from 53 bits
 *   kind 4: float32 ~ N(0,1) (Box-Muller on two 24-bit uniforms), len counts floats
 *   kind 5: int64 unique permutation-ish key: row itself xor-shuffled (bijection on [0,2^a))
 * `first_row` offsets the counter so shards generate their slice of one global column. */
int32_t dbx_synth_fill(int32_t device, int32_t kind, uint64_t seed, int64_t a, int64_t first_row, int64_t len,
                       void* dev_out);

/* Instrumentation: number of kernel launches issued by the library on this thread's
 * handles since process start (bench.py's gpu_launches). */
int64_t dbx_kernel_launch_count(void);
/* Device time (ms) of the dominant kernel of the last push on this handle, measured
 * with CUDA events on the handle's stream (roofline.achieved in bench.py). */
int32_t dbx_op_last_kernel_ms(dbx_op* op, float* ms);
/* Same for an earlier push: back = 0 is the last push, 1 the one before, ... (a ring of 8), so
 * the kernel of query i can be read after query i+1 was enqueued without waiting for it. */
int32_t dbx_op_kernel_ms(dbx_op* op, int32_t back, float* ms);
/* Which build of the hot kernel serves this handle.  Aggregate operators ask for a kernel compiled
 * for their plan at create time (NVRTC, sm_100a; cached per plan shape; DBX_AGG_JIT=0 turns it off):
 * "specialised", or "precompiled kernels (<why>)" when the plan-interpreting kernels serve it.
 * Results are identical either way. */
int32_t dbx_op_kernel_variant(dbx_op* op, char* out, int32_t cap);
/* Compiles the specialised kernels of a canned plan without touching a GPU (is NVRTC usable here?).
 * DBX_OK, or DBX_ERR_UNSUPPORTED with the reason in msg. */
int32_t dbx_agg_jit_selftest(char* msg, int32_t msg_cap);
/* Same for the scalar-expression evaluator: generates and compiles the straight-line kernel of a canned
 * expression (dbx_eval_scalar compiles one per expression shape; DBX_EVAL_JIT=0 keeps the interpreter).
 * DBX_EVAL_JIT=2 is the strict form of the default: when the generated kernel cannot be compiled or
 * launched, dbx_eval_scalar returns DBX_ERR_UNSUPPORTED with the reason (NVRTC's log) in the message
 * instead of falling back to the interpreter.  Unset or any other non-zero value: generated kernel,
 * interpreter as the fall-back.  The variable is read on every call. */
int32_t dbx_eval_jit_selftest(char* msg, int32_t msg_cap);
/* Stream of a handle as a cudaStream_t value (for external event timing). */
int32_t dbx_op_stream(dbx_op* op, void** stream);

#ifdef __cplusplus
}
#endif
#endif /* DBX_H_ */
