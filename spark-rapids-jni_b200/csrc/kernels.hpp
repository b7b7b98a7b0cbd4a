// kernels.hpp -- host-side launchers implemented in the .cu files.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/srj_b200.h"
#include "plan.hpp"

namespace srj {

// from_rows.cu
int launch_from_rows(const srj_plan* plan, const uint8_t* rows, const int32_t* row_offsets, int64_t rows_bytes,
                     int64_t num_rows, void* const* d_ent_dst, uint32_t* const* d_masks, int64_t* d_null_counts,
                     int64_t* d_status, const srj_fused_hash* fh, cudaStream_t stream);

size_t from_rows_smem_bytes(const Tiling& tl, int nentries, int ncols, int nstr);  // dynamic shared memory of from_rows_kernel

// from_rows_wide.cu: wide variable-width tables (per-row TMA slabs; offsets leave as group-local inclusive sums +
// absolute group bases unless `finalize`)
bool plan_wide(srj_plan* plan);
int64_t wide_workspace_bytes(const srj_plan* plan, int64_t num_rows);
const uint32_t* wide_workspace_bases(const srj_plan* plan, int64_t num_rows, const void* workspace);  // [nstr][ngroups]
int launch_from_rows_wide(const srj_plan* plan, const uint8_t* rows, const int32_t* row_offsets, int64_t rows_bytes,
                          int64_t num_rows, const srj_column* cols /* host array of the output columns */,
                          int64_t* d_null_counts, int64_t* d_char_totals, void* d_scratch /* wide_workspace_bytes() */,
                          bool finalize, cudaStream_t stream);

// strings.cu
// In-place inclusive scan of the int32 lengths stored at offsets[c][1..n] for every STRING column
// (offsets[c][0] = 0), per-column totals to d_char_totals[schema col] (int64), a total beyond INT32_MAX sets bit 1 of *d_status.
int launch_string_offsets_scan(int32_t* const* d_offsets /* device array [nstr] */, const int32_t* d_string_cols,
                               int nstr, int64_t num_rows, int64_t* d_char_totals, int64_t* d_status,
                               void* d_partials /* int64 [nstr * nchunks] */,
                               bool mark_finished /* set bit 2 of *d_status: the offsets are complete */, cudaStream_t stream);
int64_t string_scan_partials_bytes(int nstr, int64_t num_rows);
// copy_strings_from_rows replacement.  cols = the caller's columns (host array); d_tab = device table
// [offsets nstr][chars nstr], needed (and uploaded by the caller) only when !strings_fast_path().
int launch_strings_from_rows(const srj_plan* plan, const uint8_t* rows, const int32_t* row_offsets,
                             int64_t rows_bytes, int64_t num_rows, const srj_column* cols, void* const* d_tab,
                             const int64_t* d_status,
                             const uint32_t* d_bases /* non-NULL: offsets hold group-local inclusive sums, the chars before
                                                        each 32-row group are d_bases[nstr][ngroups] (wide tables) */,
                             cudaStream_t stream);
bool strings_wide_eligible(const srj_plan* plan);
bool strings_fast_path(const srj_plan* plan, const int64_t* d_status);

// to_rows.cu
int launch_row_sizes(const srj_plan* plan, const int32_t* const* d_str_offsets, int64_t num_rows,
                     uint64_t* d_cum_sizes, cudaStream_t stream);
// batch cut on the device: d_out = int64[1 + 3 * max_batches]
int launch_batch_cut(const uint64_t* d_cum, int64_t num_rows, int32_t max_batches, int64_t* d_out, cudaStream_t stream);
int launch_to_rows(const srj_plan* plan, const void* const* d_col_data, const uint32_t* const* d_masks,
                   const int32_t* const* d_str_offsets, const uint8_t* const* d_str_chars, int64_t row_start,
                   int64_t row_count, const uint64_t* d_cum_sizes /* NULL for fixed */, int32_t* out_offsets,
                   uint8_t* out_data, int64_t out_bytes, cudaStream_t stream,
                   const void* const* h_col_data /* host copy of the column pointers (alignment checks) */,
                   int32_t* d_fail_flag /* 4 bytes of device scratch (variable-width tables), may be NULL */);
// to_rows_var.cu: wide rows with STRING columns.  *launched = 0: table not eligible, nothing was launched.
int launch_to_rows_var(const srj_plan* plan, const void* const* d_col_data, const uint32_t* const* d_masks,
                       const int32_t* const* d_str_offsets, const uint8_t* const* d_str_chars, int64_t row_start,
                       int64_t row_count, const int32_t* out_offsets, uint8_t* out_data, int64_t out_bytes,
                       int32_t* d_fail_flag, cudaStream_t stream, const void* const* h_col_data, int* launched);

// hash_nested.cu: tables with LIST / STRUCT key columns
bool hash_has_nested(const srj_column* cols, int32_t num_columns);
int launch_hash_nested(int kind, const srj_column* cols, int32_t num_columns, int64_t num_rows, int64_t seed, void* out,
                       void* d_scratch, void* h_pinned, size_t scratch_bytes, cudaStream_t stream);

// hash.cu
int launch_hash(int kind, const srj_column* cols, int32_t num_columns, int64_t num_rows, int64_t seed, void* out,
                cudaStream_t stream);

// ---- partition.cu: Spark HashPartitioning (ids, stable partition maps, moving the columns) ----
int64_t partition_workspace_bytes(int64_t num_rows, int32_t num_partitions);
int launch_partition_plan(int32_t* d_ids, int64_t num_rows, int32_t num_partitions, int32_t* d_part_offsets, int32_t* d_scatter_map,
                          int32_t* d_gather_map, void* workspace, cudaStream_t stream);
int launch_partition_scatter_fixed(const void* in, void* out, int elem_size, const int32_t* d_scatter_map, int64_t n, cudaStream_t stream);
int launch_partition_gather_mask(const uint32_t* in, uint32_t* out, const int32_t* d_gather_map, int64_t n, unsigned long long* d_null_count,
                                 cudaStream_t stream);
int launch_partition_move_tiles(const srj_column* in, const srj_column* out, const int* elem_size, int32_t ncols, int64_t n, int32_t P,
                                const int32_t* d_scatter_map, const void* workspace, unsigned long long* d_null_counts, cudaStream_t stream);
int launch_partition_string_offsets(const int32_t* in_off, int32_t* out_off, const int32_t* d_gather_map, int64_t n, void* scan_ws,
                                    cudaStream_t stream);
int launch_partition_gather_chars(const uint8_t* in_chars, const int32_t* in_off, uint8_t* out_chars, const int32_t* out_off,
                                  const int32_t* d_gather_map, int64_t n, cudaStream_t stream);

// exclusive scan of int32 in place (partition.cu); `sums` = i32_scan_nchunks(n) ints of scratch; *tail (may be NULL) <- grand total
int64_t i32_scan_nchunks(int64_t n);
int launch_i32_exclusive_scan(int32_t* v, int64_t n, int32_t* sums, int32_t* tail, cudaStream_t stream);

// ---- unsafe_row.cu: columns <-> Apache Spark UnsafeRow ----
int unsafe_row_layout(const int32_t* type_ids, int32_t ncols, int32_t* bitset_bytes, int32_t* fixed_bytes, int32_t* ndec, int32_t* nstr);
int64_t unsafe_row_workspace_bytes(int32_t ncols, int64_t n);
int launch_unsafe_row_sizes(const srj_column* cols, int32_t ncols, int64_t n, int32_t* d_row_offsets, void* workspace, int64_t* h_total,
                            cudaStream_t stream);
int launch_unsafe_to_rows(const srj_column* cols, int32_t ncols, int64_t n, const int32_t* d_row_offsets, uint8_t* rows, void* workspace,
                          cudaStream_t stream);
int launch_unsafe_from_rows(const srj_column* out, int32_t ncols, int64_t n, const uint8_t* rows, const int32_t* d_row_offsets,
                            int64_t* d_null_counts, void* workspace, cudaStream_t stream);
int launch_unsafe_from_rows_strings(const srj_column* out, int32_t ncols, int64_t n, const uint8_t* rows, const int32_t* d_row_offsets,
                                    cudaStream_t stream);

// ---- kudo.cu: the Kudo shuffle wire format (split of flat tables / assemble of flat and nested tables) ----
int64_t kudo_workspace_bytes(int32_t ncols, int32_t P);
int launch_kudo_split_sizes(const srj_column* cols, int32_t ncols, const int32_t* d_splits, int32_t P, int64_t* d_part_offsets, int64_t* h_total,
                            void* workspace, cudaStream_t stream);
int launch_kudo_split(const srj_column* cols, int32_t ncols, const int32_t* d_splits, int32_t P, const int64_t* d_part_offsets, uint8_t* out,
                      void* workspace, cudaStream_t stream);
int launch_kudo_assemble_sizes(const uint8_t* buf, const int64_t* d_part_offsets, int32_t P, const int32_t* type_ids, int32_t ncols, int64_t* h_rows,
                               int64_t* h_char_totals, void* workspace, cudaStream_t stream);
int launch_kudo_assemble(const uint8_t* buf, const int64_t* d_part_offsets, int32_t P, const srj_column* out, int32_t ncols, int64_t total_rows,
                         void* workspace, cudaStream_t stream);
// nested (LIST / STRUCT) schemas, flattened in pre-order; the flat entry points above are these over a schema of leaves
int launch_kudo_assemble_nested_sizes(const uint8_t* buf, const int64_t* d_part_offsets, int32_t P, const int32_t* type_ids, const int32_t* num_children,
                                      int32_t F, int64_t* h_rows, int64_t* h_char_totals, void* workspace, cudaStream_t stream);
int launch_kudo_assemble_nested(const uint8_t* buf, const int64_t* d_part_offsets, int32_t P, const srj_column* out, int32_t ncols, void* workspace,
                                cudaStream_t stream);

}  // namespace srj
