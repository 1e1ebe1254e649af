/*
 * b200df.h -- C ABI of libb200df.so: the Blackwell (sm_100a) execution path for rust-dataframe's
 * per-RecordBatch compute.  Plain pointers and sizes only; no C++/torch/arrow types cross this boundary.
 *
 * Reference = nevi-me/rust-dataframe @ a8310afd (paths relative to the reference root).  The reference
 * has no FFI today; the seam is the set of Rust functions below, whose BODIES become one call each
 * (INTEGRATION.md shows the Rust binding).  One call carries ALL chunks of the column(s)
 * (Vec<&PrimitiveArray<T>>, one entry per RecordBatch -- src/table.rs:114-123), so batching, streams and
 * device memory are owned by the library.
 *
 *   bdf_binary      replaces the bodies of ScalarFunctions::{add,subtract,multiply,par_multiply,divide}
 *                   (src/functions/scalar.rs:16-103 -> arrow::compute::{add,subtract,multiply,divide}) and
 *                   atan2/hypot/log (scalar.rs:148,274,291 -> math_op scalar.rs:499-523)
 *   bdf_unary       replaces ScalarFunctions::{abs,sin,cos,tan,acos,...} (scalar.rs:106-457 -> scalar_op
 *                   scalar.rs:525-540)
 *   bdf_cast        replaces the arrow::compute::cast call of Function::Cast (src/evaluation.rs:296-315)
 *   bdf_aggregate   replaces AggregateFunctions::{sum,min,max,count} (src/functions/aggregate.rs:12-93)
 *   bdf_avg         replaces AggregateFunctions::avg (aggregate.rs:32-65)
 *   bdf_*_dev       the same operators on device-resident columns, so a chain of Calculations
 *                   (src/evaluation.rs:66-96 evaluates one after another) uploads once and downloads once.
 *
 * Threads: a context may be called from several threads; calls on one context are serialised (a one-GPU context by a lock around each
 * entry, a multi-GPU context around each fan-out to its GPUs), so the reference's callers need no locking of their own -- but
 * bdf_destroy must not race with another call, and a column or future handle belongs to the thread that is using it.
 * A column may be passed only to the context that made it; any other context returns BDF_INVALID.
 *
 * Error convention: every entry returns a bdf_status; BDF_OK == 0.  bdf_last_error() gives a
 * thread-local message.  No exception or abort crosses the ABI.  Mapping to the reference's errors:
 *   BDF_LENGTH_MISMATCH -> ArrowError::ComputeError("Cannot perform math operation on arrays of different length")
 *                          (text as src/functions/scalar.rs:508-511)
 *   BDF_DIVIDE_BY_ZERO  -> ArrowError::DivideByZero
 *   BDF_UNSUPPORTED     -> a trait bound the reference enforces at compile time (e.g. sin on integers,
 *                          max on floats: T::Native: Float / Ord)
 *   BDF_WOULD_PANIC     -> the reference panics here (max/min .unwrap() on an all-null or empty chunk,
 *                          aggregate.rs:19,29); the binding turns it back into a panic
 *   BDF_CUDA / BDF_OOM / BDF_INVALID -> ArrowError::ComputeError(bdf_last_error())
 * There is NO CPU fallback: without a usable CUDA device bdf_init fails with BDF_CUDA.
 *
 * Ownership: host buffers (inputs and outputs) belong to the caller; the library never frees them and,
 * except for BDF_ASYNC uploads, never touches them after the call returns.  Device memory, streams and
 * events belong to bdf_ctx / bdf_col handles.  A bdf_ctx serialises concurrent callers with a mutex.
 */
#ifndef B200DF_H
#define B200DF_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library is built with -fvisibility=hidden; these are its exports */
#endif

#define BDF_ABI_VERSION 2

/* Arrow primitive types, in arrow::datatypes::DataType order. */
typedef enum {
    BDF_I8 = 0, BDF_I16, BDF_I32, BDF_I64, BDF_U8, BDF_U16, BDF_U32, BDF_U64, BDF_F32, BDF_F64, BDF_NTYPES
} bdf_dtype;

typedef enum { BDF_ADD = 0, BDF_SUB, BDF_MUL, BDF_DIV, BDF_ATAN2, BDF_HYPOT, BDF_LOG, BDF_NBINARY } bdf_binop;

typedef enum {
    BDF_ABS = 0, BDF_SIN, BDF_COS, BDF_TAN,
    BDF_ACOS, BDF_ASIN, BDF_ATAN, BDF_CBRT, BDF_CEIL, BDF_COSH, BDF_DEGREES, BDF_EXP, BDF_EXPM1,
    BDF_FLOOR, BDF_LOG10, BDF_LOG2, BDF_RADIANS, BDF_ROUND, BDF_SINH, BDF_SQRT, BDF_TANH, BDF_NUNARY
} bdf_unop;

typedef enum { BDF_SUM = 0, BDF_MIN, BDF_MAX, BDF_COUNT, BDF_NAGG } bdf_aggop;

/* SURVEY 8(f) N2 (the step after the hot path): boolean columns are Arrow BooleanArrays -- `values` is a bit-packed
 * LSB-first bitmap whose `offset` counts bits -- identified by dtype BDF_BOOL in bdf_upload / bdf_col_describe. */
#define BDF_BOOL 10
typedef enum { BDF_GT = 0, BDF_GE, BDF_EQ, BDF_NE, BDF_LT, BDF_LE } bdf_cmpop;
typedef enum { BDF_AND = 0, BDF_OR, BDF_NOT } bdf_boolop;

typedef enum {
    BDF_OK = 0, BDF_LENGTH_MISMATCH = 1, BDF_DIVIDE_BY_ZERO = 2, BDF_UNSUPPORTED = 3, BDF_CUDA = 4,
    BDF_NCCL = 5 /* the communicator (bdf_comm_*) or a collective failed */, BDF_OOM = 6, BDF_WOULD_PANIC = 7, BDF_INVALID = 8
} bdf_status;

/* One chunk = one PrimitiveArray<T> in Arrow memory layout (ArrayData: buffers[0], null bitmap, len, offset). */
typedef struct {
    const void*    values;     /* base of the values buffer, NOT offset-adjusted                         */
    const uint8_t* validity;   /* LSB-first bitmap, 1 = valid; NULL when the array has no null buffer     */
    int64_t        len;        /* logical length in elements                                              */
    int64_t        offset;     /* element offset, applies to values and to validity bits (sliced arrays)  */
    int64_t        null_count; /* cached ArrayData::null_count, or -1 if unknown                          */
} bdf_view;

/* Output chunk.  values >= len*width bytes, validity >= ceil(len/8) bytes, both caller-allocated
 * (arrow MutableBuffer).  validity is written at bit offset 0 with zero padding bits.  validity may be
 * NULL only if the result carries no bitmap (has_validity == 0 on return), else BDF_INVALID. */
typedef struct {
    void*    values;
    uint8_t* validity;
    int64_t  len;          /* IN: capacity in elements (must equal the result length); OUT: length */
    int64_t  null_count;   /* OUT */
    int32_t  has_validity; /* OUT: 0 => every slot valid and no bitmap was written */
} bdf_out;

/* All four aggregates from one pass.  Each value slot holds T::Native in its low bytes (little endian). */
typedef struct {
    uint64_t sum, min, max;  /* bit patterns of T::Native, zero-padded to 8 bytes                      */
    int64_t  count;          /* non-null slots                                                         */
    int64_t  rows;           /* total slots                                                            */
    int32_t  any_valid;      /* 0 => min/max are None                                                  */
    int32_t  would_panic;    /* 1 => some chunk is empty/all-null: reference max/min .unwrap() panics  */
    int64_t  n_chunks;       /* chunks aggregated (0 => Iterator::max over an empty Vec: None)         */
} bdf_agg4;

typedef struct bdf_ctx bdf_ctx;
typedef struct bdf_col bdf_col;
typedef struct bdf_future bdf_future; /* an aggregate whose kernels are enqueued but not yet waited for */

/* ---- lifecycle ------------------------------------------------------------------------------ */
int          bdf_abi_version(void);
const char*  bdf_last_error(void);
int          bdf_init(int device, bdf_ctx** out);   /* one context per GPU (one process per GPU) */
/* ONE context over n_gpus GPUs of the box (0 = all visible; devices == NULL: 0..n-1): what a single Rust process binds.
 * Every entry below accepts it: the rows of a call are cut into one contiguous range per GPU (the axis the reference's
 * rayon par_iter parallelises, src/functions/scalar.rs:28-31,99-102 -- cuts inside a chunk fall on 64-row boundaries,
 * so a piece is a zero-copy Arrow slice), every GPU moves and computes its pieces over its own PCIe link, and aggregates
 * are combined by the grouped ncclAllReduce (ncclCommInitAll).  Results, chunk structure, null counts and errors are
 * those of the one-GPU context.  Not offered on a multi-GPU context: sort / take / filter (rows change chunks) and the
 * IPC readers (BDF_UNSUPPORTED). */
int          bdf_init_multi(int n_gpus, const int* devices, bdf_ctx** out);
int          bdf_fleet_size(bdf_ctx* ctx);           /* GPUs behind the context (1 for bdf_init) */
void         bdf_destroy(bdf_ctx* ctx);
int          bdf_synchronize(bdf_ctx* ctx);
int          bdf_device_info(bdf_ctx* ctx, int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor, int64_t* hbm_bytes);

/* ---- multi-GPU (SURVEY 8(e)): one context per GPU, the contexts of a job form a communicator ---------------------
 * The Vec<RecordBatch> is sharded over the GPUs by chunk (parallel over the same axis as the reference's rayon
 * par_iter, src/functions/scalar.rs:28-31,99-102): elementwise operators and casts need no exchange at all.  The
 * cross-chunk fold of an aggregate (src/functions/aggregate.rs:12-31,70-93) becomes [this GPU's chunks] -> ONE grouped
 * ncclAllReduce over NVLink (sum/count/rows: ncclSum on the wrapping 64-bit patterns; min/max: ncclMin/ncclMax on
 * order-preserving keys; float sums: all-gathered and folded in rank order), enqueued by the library on the stream
 * that produced the partials -- no host round trip.  After bdf_comm_attach every aggregate entry (bdf_aggregate*,
 * bdf_avg*, bdf_binary_agg_dev*, bdf_eval_expr_agg_dev*) is COLLECTIVE: all ranks make the same calls in the same
 * order and every rank receives the aggregate of the whole column; DivideByZero is agreed on by all ranks.
 * bdf_comm_collective(ctx, 0) switches back to per-rank results.  NCCL is bound at run time (libnccl.so.2).
 *   process per GPU:  rank 0 calls bdf_comm_unique_id, ships the 128 bytes to the others (any side channel), every
 *                     rank calls bdf_comm_attach(ctx, id, rank, world)  [ncclCommInitRank];
 *   one process:      bdf_init_multi (below) owns all GPUs of the box  [ncclCommInitAll]. */
#define BDF_COMM_ID_BYTES 128
int  bdf_comm_unique_id(uint8_t* id /* BDF_COMM_ID_BYTES */);
int  bdf_comm_attach(bdf_ctx* ctx, const uint8_t* id, int rank, int world);
int  bdf_comm_detach(bdf_ctx* ctx);
int  bdf_comm_info(bdf_ctx* ctx, int32_t* rank, int32_t* world, int32_t* nccl_version, int64_t* collectives_enqueued);
int  bdf_comm_collective(bdf_ctx* ctx, int on);
/* How the partial aggregates travel: 0 = the grouped ncclAllReduce, 1 = NVLink peer-memory mailboxes (one small kernel of
 * the library stores every rank's record into every peer and folds in rank order; needs peer access between all GPUs).
 * Default: 1 where available, unless the environment says BDF_COMBINE=nccl.  Results are identical (integers: order
 * independent; float sums: rank-order fold in both).  Collective: every rank switches at the same point. */
int  bdf_comm_set_combine(bdf_ctx* ctx, int mode);
int  bdf_comm_get_combine(bdf_ctx* ctx);
int  bdf_comm_barrier(bdf_ctx* ctx);    /* drains this context's streams, then returns once every rank has arrived */
int  bdf_comm_all_reduce_f64(bdf_ctx* ctx, int op /* BDF_SUM | BDF_MIN | BDF_MAX */, int64_t n, double* inout); /* blocking */

/* Pinned host memory ("Arrow buffers are pinned and copied to device once per batch"). */
int          bdf_host_alloc(bdf_ctx* ctx, size_t bytes, void** out);
int          bdf_host_free(bdf_ctx* ctx, void* p);
int          bdf_host_register(bdf_ctx* ctx, void* p, size_t bytes);
int          bdf_host_unregister(bdf_ctx* ctx, void* p);

/* ---- host in / host out: drop-in bodies for the reference functions --------------------------- */
/* zip() semantics: n = min(n_left, n_right) chunks are processed (scalar.rs:28-31). */
int bdf_binary(bdf_ctx* ctx, int op, int dtype, int64_t n_left, const bdf_view* left, int64_t n_right,
               const bdf_view* right, bdf_out* out);
int bdf_unary(bdf_ctx* ctx, int op, int dtype, int64_t n_chunks, const bdf_view* in, bdf_out* out);
int bdf_cast(bdf_ctx* ctx, int from, int to, int64_t n_chunks, const bdf_view* in, bdf_out* out);
/* out_scalar: T::Native for SUM/MIN/MAX, int64_t for COUNT.  *is_some == 0 <=> Rust None. */
int bdf_aggregate(bdf_ctx* ctx, int op, int dtype, int64_t n_chunks, const bdf_view* in, void* out_scalar,
                  int32_t* is_some);
int bdf_aggregate_all(bdf_ctx* ctx, int dtype, int64_t n_chunks, const bdf_view* in, bdf_agg4* out);
int bdf_avg(bdf_ctx* ctx, int dtype, int64_t n_chunks, const bdf_view* in, double* out, int32_t* is_some);

/* ---- device-resident columns -------------------------------------------------------------------- */
#define BDF_ASYNC 1 /* bdf_upload returns before the copies finish: host buffers must stay valid and
                       unmodified until bdf_col_wait / bdf_synchronize / a download of a dependent column */
int  bdf_upload(bdf_ctx* ctx, int dtype, int64_t n_chunks, const bdf_view* in, int flags, bdf_col** out);
/* Several columns in one call, copies issued chunk-major (a0,b0,a1,b1,...) so that an operator over them
 * can start on chunk i as soon as ITS inputs have landed while later chunks are still crossing PCIe. */
int  bdf_upload_many(bdf_ctx* ctx, int64_t n_cols, const int32_t* dtypes, const int64_t* n_chunks,
                     const bdf_view* const* in, int flags, bdf_col** out /* n_cols entries */);
int  bdf_col_wait(bdf_ctx* ctx, const bdf_col* col);
int  bdf_col_describe(const bdf_col* col, int32_t* dtype, int64_t* n_chunks, int64_t* total_len);
int  bdf_col_chunk_info(bdf_ctx* ctx, const bdf_col* col, int64_t chunk, int64_t* len, int64_t* null_count,
                        int32_t* has_validity);
int  bdf_binary_dev(bdf_ctx* ctx, int op, const bdf_col* left, const bdf_col* right, bdf_col** out);
int  bdf_unary_dev(bdf_ctx* ctx, int op, const bdf_col* in, bdf_col** out);
int  bdf_cast_dev(bdf_ctx* ctx, int to, const bdf_col* in, bdf_col** out);
int  bdf_aggregate_dev(bdf_ctx* ctx, int op, const bdf_col* in, void* out_scalar, int32_t* is_some);
int  bdf_aggregate_all_dev(bdf_ctx* ctx, const bdf_col* in, bdf_agg4* out);
int  bdf_avg_dev(bdf_ctx* ctx, const bdf_col* in, double* out, int32_t* is_some);
int  bdf_download(bdf_ctx* ctx, const bdf_col* col, bdf_out* out /* n_chunks entries */);
/* ---- N2: BooleanFilter comparisons / boolean kernels / filter on device columns ------------------------------
 * bdf_compare_dev  BooleanFilter::{Gt,Ge,Eq,Ne,Lt,Le} (src/expression.rs:820-852): both sides are cast to Float64, then
 *                  compared (IEEE, computed under nulls); validity = AND.  right == NULL compares with `scalar`
 *                  (BooleanInput::Scalar broadcast, :783-802).  Result: a BDF_BOOL column.
 * bdf_boolean_dev  arrow compute::{and,or,not} on boolean columns (values op values, validity AND); b ignored for NOT.
 * bdf_filter_dev   ChunkedArray::filter (src/table.rs:97-107): arrow compute::filter per chunk pair; a slot is kept
 *                  iff the mask is valid and true there.  Result chunk lengths are data dependent (bdf_col_chunk_info). */
int  bdf_compare_dev(bdf_ctx* ctx, int op, const bdf_col* left, const bdf_col* right, double scalar, bdf_col** out);
int  bdf_boolean_dev(bdf_ctx* ctx, int op, const bdf_col* a, const bdf_col* b, bdf_col** out);
int  bdf_filter_dev(bdf_ctx* ctx, const bdf_col* values, const bdf_col* mask, bdf_col** out);
/* ---- N3: consecutive Calculations fused into one pass -----------------------------------------------------------
 * Evaluate::evaluate (src/evaluation.rs:66-96) materialises every Calculation; when the intermediates are not kept, the
 * chain can be evaluated per element in ONE kernel: inputs are read once, only the final column is written
 * (config 2: 40 B/row instead of 88).  The program is straight-line: slots 0..n_inputs-1 are the input columns,
 * node k writes slot n_inputs+k and may read any earlier slot; the last node is the result (Float64).  An input column
 * of another numeric type is read through `as f64` -- a Function::Cast to Float64 (never fails, validity unchanged)
 * folded into the load.  Every node
 * is the same operator the unfused call would run, so arithmetic chains are bit-identical; DivideByZero is raised iff
 * a slot valid for that divide node has a zero divisor.  At most 6 inputs and 12 nodes. */
#define BDF_EXPR_UNARY 100 /* node.op = bdf_binop for binary nodes, BDF_EXPR_UNARY + bdf_unop for unary nodes (operand a) */
typedef struct { int32_t op, a, b; } bdf_expr_node;
int  bdf_eval_expr_dev(bdf_ctx* ctx, int32_t n_inputs, const bdf_col* const* inputs, int32_t n_nodes, const bdf_expr_node* nodes,
                       bdf_col** out);
/* Would bdf_eval_expr_dev accept this program?  Needs no context and no GPU: validates the nodes and runs the host compiler,
 * so a planner can decide what to fuse before it touches data.  input_dtypes may be NULL (all Float64).  Returns the status
 * the evaluation would return for the program itself (BDF_OK, BDF_INVALID, BDF_UNSUPPORTED); on success reports the
 * accumulator program's instruction count and how many of the two temporaries it uses. */
int  bdf_expr_check(int32_t n_inputs, const int32_t* input_dtypes, int32_t n_nodes, const bdf_expr_node* nodes, int32_t* n_instructions,
                    int32_t* n_temporaries);
/* ... with a trailing aggregate (AggregateFunctions::sum / count of the chain's last column, src/functions/aggregate.rs:22-31,
 * 70-93) folded into the same pass, like bdf_binary_agg_dev.  `out` may be NULL: the column is then never written (the
 * chain is only aggregated: sum(sin(((a+b)*c)/d)) reads 32 B/row and writes nothing).  Float64 result: agg->sum and
 * agg->count are set, min/max are not (T::Native: Ord).  The _async form returns a future for bdf_future_wait. */
int  bdf_eval_expr_agg_dev(bdf_ctx* ctx, int32_t n_inputs, const bdf_col* const* inputs, int32_t n_nodes, const bdf_expr_node* nodes,
                           bdf_col** out, bdf_agg4* agg);
int  bdf_eval_expr_agg_dev_async(bdf_ctx* ctx, int32_t n_inputs, const bdf_col* const* inputs, int32_t n_nodes,
                                 const bdf_expr_node* nodes, bdf_col** out, bdf_future** fut);
/* Split download: _begin enqueues the device->host copies (they start as soon as each chunk group is
 * ready), _end waits for them and fills len / null_count / has_validity.  Same `out` array for both. */
int  bdf_download_begin(bdf_ctx* ctx, const bdf_col* col, bdf_out* out);
int  bdf_download_end(bdf_ctx* ctx, const bdf_col* col, bdf_out* out);
/* Fused operator + aggregate (SURVEY K5 / 8(f) N3): out = left (op) right AND sum/min/max/count of `out`,
 * computed while `out` is being written -- one pass, 3 x width bytes/row instead of 4 x.  op in
 * {ADD,SUB,MUL,DIV}.  The column is materialised exactly as bdf_binary_dev would.  agg->would_panic is
 * not evaluated here (always 0); use bdf_aggregate_dev for the reference's unwrap() behaviour. */
int  bdf_binary_agg_dev(bdf_ctx* ctx, int op, const bdf_col* left, const bdf_col* right, bdf_col** out, bdf_agg4* agg);
/* Asynchronous aggregates: the call enqueues the kernels and returns a future; bdf_future_wait blocks until
 * the result has reached the host, converts it and CONSUMES the future (out may be NULL to discard). */
int  bdf_binary_agg_dev_async(bdf_ctx* ctx, int op, const bdf_col* left, const bdf_col* right, bdf_col** out, bdf_future** fut);
int  bdf_aggregate_all_dev_async(bdf_ctx* ctx, const bdf_col* in, bdf_future** fut);
/* sum/min/max/count of up to 64 columns in one call (BASELINE config 3: 8 x Int64): one reduction per column, ONE host
 * wait and -- on a rank of a communicator -- ONE grouped collective for all of them.  out / the future carry n_cols
 * records in column order; the blocking form also evaluates would_panic. */
int  bdf_aggregate_all_many_dev(bdf_ctx* ctx, int32_t n_cols, const bdf_col* const* cols, bdf_agg4* out /* n_cols */);
int  bdf_aggregate_all_many_dev_async(bdf_ctx* ctx, int32_t n_cols, const bdf_col* const* cols, bdf_future** fut);
int  bdf_future_count(const bdf_future* fut);   /* records bdf_future_wait will write */
int  bdf_future_wait(bdf_ctx* ctx, bdf_future* fut, bdf_agg4* out /* bdf_future_count(fut) records */);
void bdf_col_free(bdf_ctx* ctx, bdf_col* col);

/* ---- DataFrame::sort (src/dataframe.rs:194-222): lexsort_to_indices + take ------------------------------------------
 * bdf_sort_indices_dev  arrow compute::lexsort_to_indices over the criteria columns (numeric, equal lengths, any chunking;
 *                       row numbers count through the chunks): a STABLE sort; per criterion ascending or descending,
 *                       nulls always last (the reference passes nulls_first: false), NaN greater than every number,
 *                       -0.0 == 0.0.  Result: one UInt32 chunk of row numbers.  BDF_INVALID for zero criteria
 *                       ("Sort criteria cannot be empty").
 * bdf_take_dev          Column::take (src/table.rs:218-241) -> arrow compute::take: out[i] = values[indices[i]], one
 *                       chunk (the reference's repartitioning loop always produces a single chunk); a null index or a
 *                       null value gives a null slot; an index past the end is an error (BDF_INVALID).  Any numeric
 *                       or boolean values column; indices: a UInt32 column. */
typedef struct { const bdf_col* column; int32_t descending; } bdf_sort_key;
int  bdf_sort_indices_dev(bdf_ctx* ctx, int32_t n_keys, const bdf_sort_key* keys, bdf_col** indices);
int  bdf_take_dev(bdf_ctx* ctx, const bdf_col* values, const bdf_col* indices, bdf_col** out);

/* ---- group-by aggregate (the tail of SURVEY 8(f) N4: `Transformation::GroupAggregate`, a panic! in the reference,
 * src/evaluation.rs:73; its intended shape is src/expression.rs:114-221) ---------------------------------------------------
 * Rows are grouped by ONE numeric key column; every value column is folded per group with the aggregates of
 * AggregateFunctions (sum: wrapping for integers, double accumulation for floats; count of valid slots; min / max for integers).
 * Groups come out in ascending key order, the null key (one group) last -- the order of DataFrame::sort; NaN keys form one
 * group after every number, -0.0 and 0.0 are one group.  Results: one chunk per column, n_groups rows; sum (dtype of the value
 * column, never null: an all-null group sums to 0 like AggregateFunctions::sum), count (Int64), min / max (NULL for a group
 * without a valid value; not produced for float columns -- T::Native: Ord -- the pointers are NULL then). */
typedef struct { bdf_col *sum, *count, *min, *max; } bdf_group_out;
int  bdf_group_aggregate_dev(bdf_ctx* ctx, const bdf_col* key, int32_t n_values, const bdf_col* const* values, bdf_col** out_keys,
                             bdf_group_out* out /* n_values */, int64_t* n_groups);

/* ---- N4: Arrow IPC files either side of the path ---------------------------------------------------------------
 * DataFrame::from_arrow (src/dataframe.rs:391-407: arrow::ipc::reader::FileReader, every RecordBatch -> one chunk per
 * column) and DataFrame::to_arrow (:515-525: arrow::ipc::writer::FileWriter).  The file is mapped and its footer, schema
 * and RecordBatch metadata are decoded by the library itself (Arrow IPC file format, metadata V4/V5, uncompressed,
 * little endian); body buffers are used in place.  Columns of the ten numeric types and Boolean can be read; any other
 * column (strings, lists, structs, dictionaries, temporal types ...) is skipped and reported with dtype -1.
 *   bdf_ipc_open / _close / _describe / _column / _batch_rows / _view need no context (and no GPU);
 *   bdf_ipc_view      a zero-copy bdf_view of one column of one RecordBatch, pointing into the mapping;
 *   bdf_ipc_read      the chosen columns straight to the device, one chunk per RecordBatch (flags: BDF_ASYNC; keep the
 *                     file open until bdf_col_wait / bdf_synchronize then);
 *   bdf_ipc_write_host  write host arrays ([column][batch] views, any offset) as an IPC file (V5, 64-byte aligned bodies);
 *   bdf_ipc_write     device columns (equal chunk structure: chunk b of every column = RecordBatch b) -> IPC file. */
typedef struct bdf_ipc bdf_ipc;
int  bdf_ipc_open(const char* path, bdf_ipc** out);
void bdf_ipc_close(bdf_ipc* file);
int  bdf_ipc_describe(const bdf_ipc* file, int32_t* n_columns, int64_t* n_batches, int64_t* n_rows);
int  bdf_ipc_column(const bdf_ipc* file, int32_t col, const char** name, int32_t* dtype, int32_t* nullable);
int  bdf_ipc_batch_rows(const bdf_ipc* file, int64_t batch, int64_t* rows);
int  bdf_ipc_view(const bdf_ipc* file, int64_t batch, int32_t col, bdf_view* out);
int  bdf_ipc_read(bdf_ctx* ctx, const bdf_ipc* file, int32_t n_cols, const int32_t* cols, int flags, bdf_col** out /* n_cols */);
/* A subset of the RecordBatches, in the given order (multi-GPU: rank r of N reads batches r, r+N, ... -- SURVEY 8(e)). */
int  bdf_ipc_read_batches(bdf_ctx* ctx, const bdf_ipc* file, int32_t n_cols, const int32_t* cols, int64_t n_batches,
                          const int64_t* batches, int flags, bdf_col** out /* n_cols */);
int  bdf_ipc_write_host(const char* path, int32_t n_cols, const char* const* names, const int32_t* dtypes, int64_t n_batches,
                        const bdf_view* const* cols /* [n_cols][n_batches] */);
int  bdf_ipc_write(bdf_ctx* ctx, const char* path, int32_t n_cols, const char* const* names, const bdf_col* const* cols);

/* ---- measurement support ------------------------------------------------------------------------ */
/* Per-launch CUDA-event timing on the library's compute stream (the stream the kernels run on). */
typedef struct {
    int32_t kernel;   /* bdf_kernel_id */
    int32_t dtype;    /* output dtype   */
    int64_t rows;     /* elements processed by the launch */
    int64_t bytes;    /* algorithmic bytes of the launch (SURVEY 8(d) per-row figure x rows) */
    float   ms;       /* device time between the bracketing events */
} bdf_launch_record;
typedef enum { BDF_K_BINARY = 0, BDF_K_UNARY, BDF_K_CAST, BDF_K_REDUCE, BDF_K_GENERATE, BDF_K_AVG, BDF_K_COMPARE, BDF_K_FILTER, BDF_K_EXPR, BDF_K_SORT, BDF_K_TAKE, BDF_K_GROUP } bdf_kernel_id;
int     bdf_profile_enable(bdf_ctx* ctx, int on);
int     bdf_profile_read(bdf_ctx* ctx, bdf_launch_record* buf, int64_t cap, int64_t* n); /* syncs; drains */
int64_t bdf_launch_count(bdf_ctx* ctx);           /* kernels launched since bdf_init */
/* Stream-ordered stopwatch on the compute stream: start/stop record events; stop syncs and reports ms. */
int     bdf_timer_start(bdf_ctx* ctx);
int     bdf_timer_stop(bdf_ctx* ctx, float* ms);
/* Writes `bytes` of device memory (an L2 flush when bytes > L2 size). */
int     bdf_flush_l2(bdf_ctx* ctx, size_t bytes);

/* Counter-based synthetic columns generated on the device (bench / large-config tests; SURVEY 8(d)).
 * Reproduces oracle/oracle.c:orc_generate bit-for-bit.  kind 0: real uniform [lo,hi), 1: real +-[1,2),
 * 2: integer full range, 3: integer uniform [-2^40,2^40).  null_mod 0: no bitmap. */
int bdf_generate(bdf_ctx* ctx, int dtype, int kind, double lo, double hi, uint64_t seed, uint64_t col_id,
                 int64_t n_chunks, const int64_t* chunk_lens, int64_t row0, uint32_t null_mod, bdf_col** out);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* B200DF_H */
