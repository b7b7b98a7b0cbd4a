/*
 * srj_b200.h -- C ABI of libsrj_b200.so: the B200-native (sm_100a) replacement for the
 * row<->columnar + Spark row-hash hot path of NVIDIA/spark-rapids-jni.
 *
 * This is the drop-in boundary (SURVEY.md 8b).  Every entry point below is what the reference's
 * JNI layer for this path would bind; each cites the reference interface it replaces.  Paths are
 * relative to the reference tree; RC = src/main/cpp/src/row_conversion.cu.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only.  All data pointers are DEVICE pointers owned by the
 *     caller (the JNI shim allocates them with rmm exactly where the reference does); functions
 *     whose name ends in _host take HOST pointers and stage through the device themselves.
 *   - Every function returns SRJ_OK (0) or a negative srj_status; nothing throws across the
 *     boundary.  srj_last_error() returns a thread-local message for the last failure.
 *     The JNI shim maps codes to the reference's exception classes (INTEGRATION.md):
 *       SRJ_EINVAL/SRJ_EUNSUPPORTED -> ai.rapids.cudf.CudfException (cudf::logic_error, error.hpp:233-239)
 *       SRJ_EOVERFLOW -> CudfColumnSizeOverflowException, SRJ_ENOMEM -> OutOfMemoryError,
 *       SRJ_ECUDA -> CudaException / CudaFatalException.
 *   - Work is enqueued on the caller's `stream` (the reference uses the per-thread default
 *     stream, CMakeLists.txt:322-326); functions are re-entrant and keep no global mutable state.
 *     Functions documented "synchronizes" block until `stream` is idle because they return
 *     host-visible sizes (the reference synchronises at the same points: RC:1534-1544, 2389).
 *   - Bitmasks are cudf bitmasks: uint32 words, bit (i % 32) of word (i / 32), 1 = valid
 *     (thirdparty/cudf/cpp/include/cudf/utilities/bit.hpp:48-106).  NULL mask = all valid.
 *   - Row counts are int64 at this ABI; the JNI shim passes cudf::size_type (int32) values.
 */
#ifndef SRJ_B200_H
#define SRJ_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SRJ_API __attribute__((visibility("default")))
#else
#define SRJ_API
#endif

/* ---- status codes --------------------------------------------------------------------------- */
typedef enum srj_status {
  SRJ_OK           = 0,
  SRJ_EINVAL       = -1, /* bad argument / layout precondition (CUDF_EXPECTS -> cudf::logic_error)  */
  SRJ_EUNSUPPORTED = -2, /* type not supported on this path (RowConversion.java:131, hive_hash.cu:63) */
  SRJ_EOVERFLOW    = -3, /* a column would exceed the int32 size_type limit (std::overflow_error)    */
  SRJ_ECUDA        = -4, /* CUDA runtime error (cudf::cuda_error)                                    */
  SRJ_ENOMEM       = -5  /* device allocation failed (rmm::out_of_memory)                            */
} srj_status;

/* ---- cudf type ids: thirdparty/cudf/cpp/include/cudf/types.hpp:191-224 ----------------------- */
typedef enum srj_type_id {
  SRJ_EMPTY = 0, SRJ_INT8, SRJ_INT16, SRJ_INT32, SRJ_INT64, SRJ_UINT8, SRJ_UINT16, SRJ_UINT32, SRJ_UINT64,
  SRJ_FLOAT32, SRJ_FLOAT64, SRJ_BOOL8, SRJ_TIMESTAMP_DAYS, SRJ_TIMESTAMP_SECONDS,
  SRJ_TIMESTAMP_MILLISECONDS, SRJ_TIMESTAMP_MICROSECONDS, SRJ_TIMESTAMP_NANOSECONDS,
  SRJ_DURATION_DAYS, SRJ_DURATION_SECONDS, SRJ_DURATION_MILLISECONDS, SRJ_DURATION_MICROSECONDS,
  SRJ_DURATION_NANOSECONDS, SRJ_DICTIONARY32, SRJ_STRING, SRJ_LIST, SRJ_DECIMAL32, SRJ_DECIMAL64,
  SRJ_DECIMAL128, SRJ_STRUCT, SRJ_NUM_TYPE_IDS
} srj_type_id;

/*
 * srj_column: the cudf::column_view fields this path reads/writes
 * (thirdparty/cudf/cpp/include/cudf/column/column_view.hpp:237-244).  One struct serves inputs and
 * outputs; for outputs the caller allocates every buffer and the library fills it.
 *   fixed-width column : data = size * size_of(type) bytes
 *   STRING column      : data = chars, offsets = int32[size + 1]   (RC:1919-1923, 2421-2428)
 *   LIST column        : offsets = int32[size + 1], children[0] = the element column     (hash entry points only)
 *   STRUCT column      : children[0 .. num_children) = the fields, each `size` rows        (hash entry points only)
 * Sliced views (offset != 0) are not supported, as in the reference (RC:1809-1811).
 */
typedef struct srj_column {
  int32_t type_id;     /* srj_type_id                                        */
  int32_t scale;       /* decimals only; carried, never interpreted           */
  int64_t size;        /* rows                                                */
  void* data;          /* device                                              */
  uint32_t* null_mask; /* device, ceil(size/32) words, or NULL (= all valid)  */
  int32_t* offsets;    /* device, STRING / LIST                               */
  const struct srj_column* children; /* HOST array of child descriptors (LIST / STRUCT), else NULL */
  int32_t num_children;
  int32_t reserved;
} srj_column;

/* One output batch of convert_to_rows = one LIST<INT8> column of <= INT32_MAX bytes (RC:174-190). */
typedef struct srj_row_batch {
  int64_t row_start; /* first table row in this batch                     */
  int64_t row_count; /* rows in this batch (multiple of 32 except the last, RC:1515-1517) */
  int64_t num_bytes; /* size of the INT8 child                            */
} srj_row_batch;

/* ---- library --------------------------------------------------------------------------------- */
SRJ_API const char* srj_version(void);
SRJ_API const char* srj_last_error(void);
SRJ_API const char* srj_status_string(int status);

/* ---- layout: compute_column_information, RC:1332-1371 ---------------------------------------- */
typedef struct srj_layout {
  int32_t num_columns;
  int32_t num_string_columns;
  int32_t validity_offset;    /* byte offset of the validity bytes in a row                 */
  int32_t size_per_row;       /* validity_offset + ceil(ncols/8): UNPADDED fixed+validity   */
  int32_t fixed_row_size;     /* round_up(size_per_row, 8): the row stride of a fixed-width-only table */
  int32_t reserved;
} srj_layout;

/* col_starts/col_sizes (each num_columns entries) may be NULL. */
SRJ_API int srj_compute_layout(const int32_t* type_ids, int32_t num_columns, srj_layout* out,
                               int32_t* col_starts, int32_t* col_sizes);

/*
 * A plan caches the per-schema device metadata (column starts/sizes, width-class schedule) so the
 * hot calls do no host->device metadata traffic.  Create once per schema per device (the JNI shim
 * keeps a small schema-keyed cache); destroy when done.  Plans are immutable => thread-safe.
 */
typedef struct srj_plan srj_plan;
SRJ_API int srj_plan_create(const int32_t* type_ids, const int32_t* scales /* may be NULL */,
                            int32_t num_columns, srj_plan** out);
SRJ_API void srj_plan_destroy(srj_plan* plan);
SRJ_API int srj_plan_layout(const srj_plan* plan, srj_layout* out);

/* ---- convert_to_rows: RowConversion.convertToRows / RC:1994-2055 ------------------------------ */
/*
 * Step 1 (synchronizes when the table has STRING columns): per-row sizes (RC:201-257) and the
 * <= 2 GiB / 32-row batch cut (build_batches, RC:1466-1557).  `workspace` must hold
 * srj_to_rows_workspace_bytes(plan, num_rows) bytes (0 for fixed-width-only tables) and must be
 * passed unchanged to step 2.  Writes up to max_batches entries; *num_batches gets the count
 * (0 for an empty table: the caller then returns one empty LIST column, SURVEY App. C.4).
 */
SRJ_API int64_t srj_to_rows_workspace_bytes(const srj_plan* plan, int64_t num_rows);
SRJ_API int srj_to_rows_plan_batches(const srj_plan* plan, const srj_column* cols, int64_t num_rows,
                                     void* workspace, srj_row_batch* batches, int32_t max_batches,
                                     int32_t* num_batches, void* stream);
/*
 * Step 2 (async): fill each batch's LIST offsets child (int32[row_count + 1]) and INT8 data child
 * (num_bytes).  Fuses copy_to_rows + copy_validity_to_rows + copy_strings_to_rows
 * (RC:574-688, 706-798, 816-861).  Padding bytes are written as zeros (undefined in the reference).
 * `workspace` is the buffer step 1 filled: its cumulative row sizes are only read, the scratch
 * words behind them (scan partials, dead after step 1) carry a 4-byte device flag of the fast
 * variable-width kernel -- so two step-2 calls must not share one workspace concurrently.
 */
SRJ_API int srj_convert_to_rows(const srj_plan* plan, const srj_column* cols, int64_t num_rows,
                                const void* workspace, const srj_row_batch* batches,
                                int32_t num_batches, int32_t* const* batch_offsets,
                                uint8_t* const* batch_data, void* stream);

/* ---- convert_from_rows: RowConversion.convertFromRows / RC:2149-2441 -------------------------- */
/*
 * Phase 1 (async): fixed-width columns, every column's validity mask, exact null counts
 * (replaces fixup_null_counts, RC:2130-2136) and, for STRING columns, the offsets child
 * (lengths + exclusive scan, RC:2375-2388).  Fuses copy_from_rows + copy_validity_from_rows
 * (RC:879-969, 987-1094).
 *   rows        : the LIST's INT8 child
 *   row_offsets : the LIST's offsets child (int32[num_rows + 1]) or NULL for a fixed-width-only
 *                 schema, where rows are read at stride fixed_row_size exactly as the reference
 *                 does (RC:2317; it ignores the offsets there too, SURVEY App. C.5)
 *   rows_bytes  : size of `rows`; checked against size_per_row * num_rows (RC:2197)
 *   cols        : num_columns outputs; data (fixed-width), null_mask and (STRING) offsets must be
 *                 allocated; STRING data (chars) may be NULL in this phase
 *   d_null_counts : device int64[num_columns] or NULL
 *   d_char_totals : device int64[num_columns + 1] or NULL.  Entries [0, num_columns) receive the chars size
 *                 of each STRING column (0 for the others); the caller reads them back (that read is the
 *                 one sync the reference also has, RC:2389) to size the chars.  Entry [num_columns] is a
 *                 status word for phase 2: bit 0 set = some row does not use the canonical string layout
 *                 (pair.offset != size_per_row + lengths of the preceding STRING columns); phase 2 then
 *                 follows the stored pair offsets exactly like copy_strings_from_rows (RC:1143) instead of
 *                 its fast path.  Bit 1 set = a STRING column's chars exceed INT32_MAX (the caller maps it to
 *                 SRJ_EOVERFLOW / CudfColumnSizeOverflowException; the totals themselves are exact int64).
 *                 The STRING offsets children are complete only after phase 2.
 * If hash_kind != SRJ_HASH_NONE the row hash of the listed key columns is computed from the same
 * shared-memory tile and written to hash_out (int64 for xxhash64, int32 otherwise): the fused
 * from_rows + partition-hash of BASELINE config 4.  Keys must be fixed-width columns.
 */
/*
 * Workspace of one phase-1 / phase-2 call pair: srj_from_rows_workspace_bytes(plan, num_rows) bytes of device memory
 * (0 for schemas that need none; then NULL may be passed).  Phase 1 leaves there what phase 2 needs besides the
 * offsets children (for wide tables: the chars of every STRING column before each 32-row group -- the offsets
 * children themselves hold group-local sums between the two calls and are finished by phase 2), so the same
 * buffer must be passed to both calls and must not be shared by two conversions in flight.
 */
SRJ_API int64_t srj_from_rows_workspace_bytes(const srj_plan* plan, int64_t num_rows);

typedef enum srj_hash_kind { SRJ_HASH_NONE = 0, SRJ_HASH_XXHASH64 = 1, SRJ_HASH_MURMUR3_32 = 2, SRJ_HASH_HIVE = 3 } srj_hash_kind;

typedef struct srj_fused_hash {
  int32_t kind;            /* srj_hash_kind */
  int32_t num_keys;        /* <= 16 */
  int32_t key_columns[16]; /* indices into the schema, hashed in this order */
  int64_t seed;            /* xxhash64: int64 seed; murmur: low 32 bits; hive: ignored */
  void* out;               /* device, num_rows elements */
} srj_fused_hash;

SRJ_API int srj_convert_from_rows_fixed(const srj_plan* plan, const uint8_t* rows,
                                        const int32_t* row_offsets, int64_t rows_bytes,
                                        int64_t num_rows, const srj_column* cols,
                                        int64_t* d_null_counts, int64_t* d_char_totals,
                                        const srj_fused_hash* hash /* may be NULL */, void* workspace,
                                        void* stream);
/* Phase 2 (async): gather the chars of every STRING column (copy_strings_from_rows, RC:1110-1150).
 * d_char_totals is the buffer phase 1 filled (its status word selects the fast path); NULL = always
 * follow the stored pair offsets. */
SRJ_API int srj_convert_from_rows_strings(const srj_plan* plan, const uint8_t* rows,
                                          const int32_t* row_offsets, int64_t rows_bytes, int64_t num_rows,
                                          const srj_column* cols, const int64_t* d_char_totals,
                                          const void* workspace, void* stream);

/* ---- row hashes: Hash.xxhash64 / murmurHash32 / hiveHash, hash/hash.hpp:40-74 ------------------ */
#define SRJ_DEFAULT_XXHASH64_SEED 42 /* hash/hash.hpp:27 */
#define SRJ_MAX_STACK_DEPTH 8        /* hash/hash.hpp:28: nesting limit of LIST / STRUCT keys */
SRJ_API int srj_get_max_stack_depth(void); /* Hash.getMaxStackDepth, HashJni.cpp:26-30 */
/* out has no null mask (xxhash64.cu:556-562).  num_columns == 0 or num_rows == 0 is a no-op.
 * LIST / STRUCT keys are hashed like the reference (xxhash64.cu:446-506, murmur_hash.cu:119-144,
 * hive_hash.cu:363-433): xxhash64 / murmur chain the leaf values depth first (nulls keep the accumulator; murmur
 * rejects LIST<STRUCT>, murmur_hash.cu:167-187), hive folds 31 * h + x over the fields of a struct and over the
 * elements of a list.  Nesting beyond SRJ_MAX_STACK_DEPTH returns SRJ_EINVAL (CudfException). */
SRJ_API int srj_xxhash64(const srj_column* cols, int32_t num_columns, int64_t num_rows, int64_t seed,
                         int64_t* out, void* stream);
SRJ_API int srj_murmur_hash3_32(const srj_column* cols, int32_t num_columns, int64_t num_rows,
                                uint32_t seed, int32_t* out, void* stream);
SRJ_API int srj_hive_hash(const srj_column* cols, int32_t num_columns, int64_t num_rows, int32_t* out,
                          void* stream);

/* ---- multi-GPU configuration (SURVEY 8e: row-range shards + one all-gather of per-column chunks) ---------------- */
/* ---- Spark HashPartitioning on the device (SURVEY 8f rank 1) ---------------------------------------------------
 * The consumer of Hash.murmurHash32: GpuHashPartitioning computes pmod(murmur3_32(42, keys), P) per row and then
 * partitions the batch (cudf Table.partition) into the P slices shuffle_split takes
 * (src/main/cpp/src/shuffle_split.hpp:60-189: a table plus exactly these split offsets).
 *
 *   srj_partition_workspace_bytes : bytes of the caller-provided workspace of the calls below.
 *   srj_hash_partition            : d_partition_ids[r] = pmod(murmur3_32(seed, keys of row r), P) (null keys keep the
 *                                   accumulator, hash/murmur_hash.cu:111-117); then srj_partition_plan.
 *   srj_partition_plan            : ids -> d_partition_offsets[P + 1] (row index where each partition starts; [P] = rows)
 *                                   and the STABLE partition maps: d_scatter_map[src] = dest, d_gather_map[dest] = src
 *                                   (rows of one partition keep their input order).  Ids outside [0, P) are reduced
 *                                   with Spark's pmod in place.  <= INT32_MAX rows, <= 16384 partitions.  The workspace
 *                                   keeps the plan's tile order: pass it, unmodified, to srj_partition_columns.
 *   srj_partition_columns         : (same num_partitions, maps and workspace as the plan) moves fixed-width data and
 *                                   null masks into `out`; for STRING columns writes the
 *                                   output offsets (out.offsets[rows] = the chars the column needs: read it, allocate
 *                                   out.data, then call srj_partition_strings).  d_null_counts (device int64[ncols],
 *                                   may be NULL) receives the null count of every column that has a mask.
 *   srj_partition_strings         : the chars of every STRING column.
 * All pointers device pointers owned by the caller; asynchronous on `stream`.
 */
SRJ_API int64_t srj_partition_workspace_bytes(int64_t num_rows, int32_t num_partitions);
SRJ_API int srj_hash_partition(const srj_column* keys, int32_t num_keys, int64_t num_rows, uint32_t seed, int32_t num_partitions,
                               int32_t* d_partition_ids, int32_t* d_partition_offsets, int32_t* d_scatter_map,
                               int32_t* d_gather_map, void* workspace, void* stream);
SRJ_API int srj_partition_plan(int32_t* d_partition_ids, int64_t num_rows, int32_t num_partitions, int32_t* d_partition_offsets,
                               int32_t* d_scatter_map, int32_t* d_gather_map, void* workspace, void* stream);
SRJ_API int srj_partition_columns(const srj_column* in, const srj_column* out, int32_t num_columns, int64_t num_rows,
                                  int32_t num_partitions, const int32_t* d_scatter_map, const int32_t* d_gather_map,
                                  int64_t* d_null_counts, void* workspace, void* stream);
SRJ_API int srj_partition_strings(const srj_column* in, const srj_column* out, int32_t num_columns, int64_t num_rows,
                                  const int32_t* d_gather_map, void* stream);

/* ---- Kudo shuffle wire format: split / assemble (SURVEY 8f rank 2) -------------------------------------------------
 * shuffle_split / shuffle_assemble of the reference (src/main/cpp/src/shuffle_split.hpp:60-189) for FLAT tables
 * (fixed-width, decimal, STRING columns): a table is cut at `splits` (P + 1 row indices, e.g. the partition offsets
 * of srj_hash_partition) into P partitions written back to back, each in the Kudo format of
 * kudo/KudoSerializer.java:49-171 (header "KUD0" + 6 big-endian ints + hasValidity bits | validity | offsets | data);
 * assemble concatenates partitions (of one or several splits) back into one table.
 *   srj_kudo_split_sizes    : d_partition_offsets[P + 1] (byte offset of every partition) and *total_bytes (host; one
 *                             stream synchronisation).
 *   srj_kudo_split          : writes the partitions into `out` (total_bytes, 4-byte aligned).
 *   srj_kudo_assemble_sizes : parses the headers; *total_rows and, per STRING column, char_totals[c] (host arrays);
 *                             SRJ_EINVAL on a malformed header.  The workspace keeps what srj_kudo_assemble needs.
 *   srj_kudo_assemble       : fills `out` (total_rows rows per column; null masks, where given, are produced for every
 *                             column -- partitions without validity contribute valid rows).
 * <= 256 columns, <= 65535 partitions.  LIST / STRUCT columns are not supported here (SRJ_EUNSUPPORTED); nested tables
 * are assembled by srj_kudo_assemble_nested below.
 */
SRJ_API int64_t srj_kudo_workspace_bytes(int32_t num_columns, int32_t num_partitions);
SRJ_API int srj_kudo_split_sizes(const srj_column* cols, int32_t num_columns, int64_t num_rows, const int32_t* d_splits,
                                 int32_t num_partitions, int64_t* d_partition_offsets, int64_t* total_bytes, void* workspace,
                                 void* stream);
SRJ_API int srj_kudo_split(const srj_column* cols, int32_t num_columns, int64_t num_rows, const int32_t* d_splits,
                           int32_t num_partitions, const int64_t* d_partition_offsets, uint8_t* out, void* workspace, void* stream);
SRJ_API int srj_kudo_assemble_sizes(const uint8_t* partitions, const int64_t* d_partition_offsets, int32_t num_partitions,
                                    const int32_t* type_ids, int32_t num_columns, int64_t* total_rows, int64_t* char_totals,
                                    void* workspace, void* stream);
SRJ_API int srj_kudo_assemble(const uint8_t* partitions, const int64_t* d_partition_offsets, int32_t num_partitions,
                              const srj_column* out, int32_t num_columns, int64_t total_rows, void* workspace, void* stream);

/* Assemble of NESTED tables (LIST / STRUCT columns; a map is LIST<STRUCT<K, V>>).  The schema is flattened in pre-order
 * (a LIST / STRUCT before its children), exactly as the reader's Schema gives it (getFlattenedTypeIds /
 * getFlattenedNumChildren); the partitions may come from any Kudo writer, including the reference's host
 * KudoSerializer (KudoTableHeaderCalc.java:77-195, SlicedBufferSerializer.java:72-247).
 *   srj_kudo_nested_workspace_bytes : workspace of the two calls below (kept between them).
 *   srj_kudo_assemble_nested_sizes  : per flattened column its assembled rows flat_rows[c] and, for STRING, chars
 *                                     char_totals[c] (host arrays of num_flat; one stream synchronisation).
 *                                     SRJ_EINVAL: the child counts do not describe the columns, a LIST does not have
 *                                     exactly one child, or a partition is malformed (a section outside the partition's
 *                                     bytes, offsets with off[0] < 0 or off[n] < off[0]).  SRJ_EOVERFLOW: a column's
 *                                     rows or chars exceed INT32_MAX.
 *   srj_kudo_assemble_nested        : fills the srj_column trees `out` (num_columns roots) of that schema: every column
 *                                     flat_rows[c] rows, LIST / STRING offsets int32[rows + 1], STRING chars, LIST
 *                                     children[0], STRUCT children; null masks, where given, are produced.
 * <= 256 flattened columns, <= 65535 partitions.
 */
SRJ_API int64_t srj_kudo_nested_workspace_bytes(int32_t num_flat, int32_t num_partitions);
SRJ_API int srj_kudo_assemble_nested_sizes(const uint8_t* partitions, const int64_t* d_partition_offsets, int32_t num_partitions,
                                           const int32_t* flat_type_ids, const int32_t* flat_num_children, int32_t num_flat,
                                           int64_t* flat_rows, int64_t* char_totals, void* workspace, void* stream);
SRJ_API int srj_kudo_assemble_nested(const uint8_t* partitions, const int64_t* d_partition_offsets, int32_t num_partitions,
                                     const srj_column* out, int32_t num_columns, void* workspace, void* stream);

/* ---- Apache Spark UnsafeRow codec (SURVEY 8f rank 3) -----------------------------------------------------------
 * The row format Spark's own operators consume (org.apache.spark.sql.catalyst.expressions.UnsafeRow /
 * codegen.UnsafeRowWriter); the reference speaks only JCUDF (RowConversion.java:44-117) and leaves the adaptation to
 * the plugin's CudfUnsafeRow.  Row = null bitset (ceil(n/64) 8-byte words, bit SET = NULL) | one 8-byte slot per
 * field | variable region (strings: (offset << 32) | length, padded to 8; DECIMAL128: 16 bytes always reserved,
 * BigInteger.toByteArray() big-endian minimal bytes, slot (offset << 32) | byte count).  DECIMAL32/64 are longs.
 * Supported: the fixed-width types of the row path, STRING, DECIMAL32/64/128; <= 256 columns; rows 8-byte aligned.
 *
 *   srj_unsafe_row_layout   : bitset bytes and the size of a row without its strings.
 *   srj_unsafe_row_sizes    : d_row_offsets[rows + 1] (byte offset of every row) and *total_bytes (host; the call
 *                             synchronises the stream once); SRJ_EOVERFLOW beyond INT32_MAX bytes.
 *   srj_convert_to_unsafe_rows   : columns -> rows (d_row_offsets may be NULL for tables without STRING columns:
 *                                  rows are then fixed_bytes apart).
 *   srj_convert_from_unsafe_rows : rows -> fixed-width / decimal values, null masks (+ counts), and for STRING
 *                                  columns the output offsets (out.offsets[rows] = chars needed: read it, allocate
 *                                  out.data, then call srj_convert_from_unsafe_rows_strings).
 */
SRJ_API int srj_unsafe_row_layout(const int32_t* type_ids, int32_t num_columns, int32_t* bitset_bytes, int32_t* fixed_bytes);
SRJ_API int64_t srj_unsafe_row_workspace_bytes(int32_t num_columns, int64_t num_rows);
SRJ_API int srj_unsafe_row_sizes(const srj_column* cols, int32_t num_columns, int64_t num_rows, int32_t* d_row_offsets,
                                 int64_t* total_bytes, void* workspace, void* stream);
SRJ_API int srj_convert_to_unsafe_rows(const srj_column* cols, int32_t num_columns, int64_t num_rows, const int32_t* d_row_offsets,
                                       uint8_t* rows, void* workspace, void* stream);
SRJ_API int srj_convert_from_unsafe_rows(const uint8_t* rows, const int32_t* d_row_offsets, int64_t num_rows, const srj_column* out,
                                         int32_t num_columns, int64_t* d_null_counts, void* workspace, void* stream);
SRJ_API int srj_convert_from_unsafe_rows_strings(const uint8_t* rows, const int32_t* d_row_offsets, int64_t num_rows,
                                                 const srj_column* out, int32_t num_columns, void* stream);

/*
 * After the NCCL all-gather of every rank's packed column slab, add to the STRING offsets of rank r's rows the chars
 * the ranks before r hold for that column, so that the gathered chunks form one column.  No reference counterpart
 * (the reference has no collective); the plugin-side caller owns the NCCL communicator.
 *   gathered     : [world][slab_bytes] device buffer (the all-gather's output)
 *   d_offs_at    : device int64[num_string_columns]: byte offset of each STRING column's int32 offsets[rows + 1] in a slab
 *   d_scol       : device int32[num_string_columns]: schema column of each STRING column
 *   d_totals     : device int64[world][num_columns + 1]: every rank's d_char_totals, all-gathered
 */
SRJ_API int srj_shard_rebase_offsets(void* gathered, int64_t slab_bytes, const int64_t* d_offs_at, const int32_t* d_scol,
                                     const int64_t* d_totals, int64_t rows_per_shard, int32_t num_columns,
                                     int32_t num_string_columns, int32_t world, void* stream);

/* ---- host-buffer entry points (end-to-end path: H2D + convert + D2H inside the call) ---------------------- */
/*
 * What a caller holding HOST buffers uses (the plugin's row<->columnar transitions hand over host memory: the
 * reference's consumers copy to the device, call convertFromRows / convertToRows, copy back).  Device staging
 * buffers and streams live in a small per-plan pool and are reused by later calls (no cudaMalloc per call); calls are
 * re-entrant (concurrent calls take different pool entries) and synchronize before returning.  Pinned host buffers
 * give full PCIe speed.  Two calls in flight on two threads overlap one's H2D with the other's D2H (full duplex).
 *
 * srj_host_alloc_fn: the library calls it when an output buffer's size is known only during the call; it returns HOST
 * memory of `bytes` bytes (JNI shim: HostMemoryBuffer.allocate) or NULL on failure (-> SRJ_ENOMEM).
 *   from_rows: index = schema column of a STRING column -> its chars buffer
 *   to_rows  : index = 2 * batch -> int32 offsets[row_count + 1] of the batch, 2 * batch + 1 -> its row bytes
 */
typedef void* (*srj_host_alloc_fn)(void* ctx, int32_t index, int64_t bytes);

/*
 * Rows -> columns.  h_rows / h_row_offsets are the LIST's children in host memory (h_row_offsets may be NULL for a
 * fixed-width-only schema: rows at stride fixed_row_size); rows_bytes = size of h_rows.  h_cols[i].data / null_mask /
 * offsets are HOST buffers to fill (null_mask may be NULL to skip it); a STRING column's data pointer is an OUTPUT:
 * obtained from `alloc` and stored into h_cols[i].data.  Fixed-width-only schemas are streamed through the device in
 * chunks of `chunk_rows` rows (0 = library default) so that H2D, kernel and D2H of consecutive chunks overlap.
 */
SRJ_API int srj_convert_from_rows_host(const srj_plan* plan, const uint8_t* h_rows, const int32_t* h_row_offsets,
                                       int64_t rows_bytes, int64_t num_rows, srj_column* h_cols, int64_t* h_null_counts,
                                       int64_t chunk_rows, srj_host_alloc_fn alloc, void* alloc_ctx);
/*
 * Columns -> rows.  h_cols are HOST columns; batches[] receives the <= 2 GiB batch cut (build_batches, RC:1466-1557),
 * h_batch_offsets[b] / h_batch_data[b] the host buffers obtained from `alloc` for each batch.
 */
SRJ_API int srj_convert_to_rows_host(const srj_plan* plan, const srj_column* h_cols, int64_t num_rows,
                                     srj_row_batch* batches, int32_t max_batches, int32_t* num_batches,
                                     int32_t** h_batch_offsets, uint8_t** h_batch_data, srj_host_alloc_fn alloc,
                                     void* alloc_ctx);

#ifdef __cplusplus
}
#endif
#endif /* SRJ_B200_H */
