// capi.cu -- the extern "C" boundary declared in include/srj_b200.h: argument checking, plans,
// per-call pointer tables, launch sequencing.  No kernels here.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <nvtx3/nvToolsExt.h>

#include "common.cuh"
#include "hash_device.cuh"
#include "kernels.hpp"
#include "plan.hpp"

namespace srj {

static thread_local char g_err[512] = "";

// NVTX range of one C-ABI call (the reference wraps its entry points the same way: nvtx_ranges.hpp:24-46,
// SRJ_FUNC_RANGE); header-only NVTX v3, a no-op unless a profiler is attached.
struct ApiRange {
  explicit ApiRange(const char* name) { nvtxRangePushA(name); }
  ~ApiRange() { nvtxRangePop(); }
};
#define SRJ_API_RANGE() ::srj::ApiRange _srj_range(__func__)

void set_error(const char* fmt, ...)
{
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what)
{
  set_error("CUDA error %d (%s) at %s", static_cast<int>(e), cudaGetErrorString(e), what);
  return e == cudaErrorMemoryAllocation ? SRJ_ENOMEM : SRJ_ECUDA;
}

static int size_of_type(int32_t t)
{
  switch (t) {
    case SRJ_INT8: case SRJ_UINT8: case SRJ_BOOL8: return 1;
    case SRJ_INT16: case SRJ_UINT16: return 2;
    case SRJ_INT32: case SRJ_UINT32: case SRJ_FLOAT32: case SRJ_TIMESTAMP_DAYS: case SRJ_DURATION_DAYS:
    case SRJ_DECIMAL32: return 4;
    case SRJ_INT64: case SRJ_UINT64: case SRJ_FLOAT64: case SRJ_TIMESTAMP_SECONDS: case SRJ_TIMESTAMP_MILLISECONDS:
    case SRJ_TIMESTAMP_MICROSECONDS: case SRJ_TIMESTAMP_NANOSECONDS: case SRJ_DURATION_SECONDS:
    case SRJ_DURATION_MILLISECONDS: case SRJ_DURATION_MICROSECONDS: case SRJ_DURATION_NANOSECONDS:
    case SRJ_DECIMAL64: return 8;
    case SRJ_DECIMAL128: return 16;
    default: return 0;
  }
}

// compute_column_information, RC:1332-1371
static int compute_layout(const int32_t* types, int32_t n, srj_layout* out, std::vector<int32_t>* starts,
                          std::vector<int32_t>* sizes)
{
  if (n < 0 || (n > 0 && !types)) { set_error("layout: bad schema"); return SRJ_EINVAL; }
  int64_t off = 0;
  int nstr    = 0;
  if (starts) starts->clear();
  if (sizes) sizes->clear();
  for (int32_t i = 0; i < n; ++i) {
    const bool compound = types[i] == SRJ_STRING;
    const int sz        = compound ? 8 : size_of_type(types[i]);
    if (sz == 0) {
      set_error("column %d: type id %d is not supported by the row format (only fixed-width and STRING, RowConversion.java:131)", i, types[i]);
      return SRJ_EUNSUPPORTED;
    }
    const int al = compound ? 4 : sz;
    off          = (off + al - 1) / al * al;
    if (starts) starts->push_back(static_cast<int32_t>(off));
    if (sizes) sizes->push_back(sz);
    off += sz;
    nstr += compound;
    if (off > INT32_MAX - 8) { set_error("layout: row too large"); return SRJ_EOVERFLOW; }
  }
  out->num_columns        = n;
  out->num_string_columns = nstr;
  out->validity_offset    = static_cast<int32_t>(off);
  off += (n + 7) / 8;
  out->size_per_row   = static_cast<int32_t>(off);
  out->fixed_row_size = static_cast<int32_t>((off + 7) / 8 * 8);
  out->reserved       = 0;
  return SRJ_OK;
}

// RAII lease of one TableRing slot (see plan.hpp).  upload() copies `host_bytes` of pointer tables to the
// device buffer; the device buffer may be larger (`total_bytes`) to carry device-only scratch behind them.
struct TableLease {
  const srj_plan* plan;
  cudaStream_t stream;
  TableSlot* slot = nullptr;
  TableLease(const srj_plan* p, cudaStream_t s) : plan(p), stream(s) {}
  int acquire(size_t total_bytes)
  {
    TableRing& r = plan->ring;
    {
      std::lock_guard<std::mutex> lk(r.mu);
      slot = &r.slots[r.next++ % TableRing::kSlots];
    }
    slot->busy.lock();  // > kSlots concurrent callers: the 9th waits for the 1st call to return
    if (slot->used) SRJ_CUDA_TRY(cudaEventSynchronize(slot->ev));  // previous user of this slot has drained
    if (!slot->ev) SRJ_CUDA_TRY(cudaEventCreateWithFlags(&slot->ev, cudaEventDisableTiming));
    if (slot->cap < total_bytes) {
      const size_t cap = std::max<size_t>(total_bytes * 2, 16384);
      if (slot->d_buf) cudaFree(slot->d_buf);
      if (slot->h_pinned) cudaFreeHost(slot->h_pinned);
      slot->d_buf = slot->h_pinned = nullptr;
      slot->cap = 0;
      SRJ_CUDA_TRY(cudaMalloc(&slot->d_buf, cap));
      SRJ_CUDA_TRY(cudaMallocHost(&slot->h_pinned, cap));
      slot->cap = cap;
    }
    return SRJ_OK;
  }
  void* host() const { return slot->h_pinned; }
  void* dev() const { return slot->d_buf; }
  int upload(size_t host_bytes)
  {
    SRJ_CUDA_TRY(cudaMemcpyAsync(slot->d_buf, slot->h_pinned, host_bytes, cudaMemcpyHostToDevice, stream));
    return SRJ_OK;
  }
  ~TableLease()
  {
    if (!slot) return;
    if (slot->ev) {
      cudaEventRecord(slot->ev, stream);
      slot->used = true;
    }
    slot->busy.unlock();
  }
};

// Phase 1 of a wide variable-width table runs from_rows_wide_kernel (no fused hash there).
static bool use_wide_from_rows(const srj_plan* plan, const int32_t* row_offsets, const srj_fused_hash* hash)
{
  return plan->wide.enabled && row_offsets != nullptr && !(hash && hash->kind != SRJ_HASH_NONE);
}

static int check_cols(const srj_plan* plan, const srj_column* cols, int64_t num_rows, const char* who)
{
  if (!plan || (plan->num_columns > 0 && !cols)) { set_error("%s: null argument", who); return SRJ_EINVAL; }
  if (num_rows < 0) { set_error("%s: negative row count", who); return SRJ_EINVAL; }
  for (int c = 0; c < plan->num_columns; ++c) {
    if (cols[c].type_id != plan->type_ids[c]) { set_error("%s: column %d type %d does not match the plan (%d)", who, c, cols[c].type_id, plan->type_ids[c]); return SRJ_EINVAL; }
    if (cols[c].size != num_rows) { set_error("%s: column %d has %lld rows, expected %lld", who, c, (long long)cols[c].size, (long long)num_rows); return SRJ_EINVAL; }
  }
  return SRJ_OK;
}

}  // namespace srj

using namespace srj;

extern "C" {

const char* srj_version(void) { return "srj_b200 0.1.0 (sm_100a)"; }
const char* srj_last_error(void) { return g_err; }
const char* srj_status_string(int s)
{
  switch (s) {
    case SRJ_OK: return "SRJ_OK";
    case SRJ_EINVAL: return "SRJ_EINVAL";
    case SRJ_EUNSUPPORTED: return "SRJ_EUNSUPPORTED";
    case SRJ_EOVERFLOW: return "SRJ_EOVERFLOW";
    case SRJ_ECUDA: return "SRJ_ECUDA";
    case SRJ_ENOMEM: return "SRJ_ENOMEM";
    default: return "SRJ_E?";
  }
}

int srj_compute_layout(const int32_t* type_ids, int32_t num_columns, srj_layout* out, int32_t* col_starts,
                       int32_t* col_sizes)
{
  if (!out) { set_error("layout: out is null"); return SRJ_EINVAL; }
  std::vector<int32_t> st, sz;
  const int rc = compute_layout(type_ids, num_columns, out, &st, &sz);
  if (rc != SRJ_OK) return rc;
  if (col_starts) std::copy(st.begin(), st.end(), col_starts);
  if (col_sizes) std::copy(sz.begin(), sz.end(), col_sizes);
  return SRJ_OK;
}

int srj_plan_create(const int32_t* type_ids, const int32_t* scales, int32_t num_columns, srj_plan** out)
{
  SRJ_API_RANGE();
  if (!out) { set_error("plan_create: out is null"); return SRJ_EINVAL; }
  *out = nullptr;
  srj_layout lay{};
  std::vector<int32_t> st, sz;
  int rc = compute_layout(type_ids, num_columns, &lay, &st, &sz);
  if (rc != SRJ_OK) return rc;
  auto* p               = new srj_plan();
  p->num_columns        = num_columns;
  p->num_string_columns = lay.num_string_columns;
  p->validity_offset    = lay.validity_offset;
  p->size_per_row       = lay.size_per_row;
  p->fixed_row_size     = lay.fixed_row_size;
  p->type_ids.assign(type_ids, type_ids + num_columns);
  p->scales.assign(num_columns, 0);
  if (scales) p->scales.assign(scales, scales + num_columns);
  p->col_start = st;
  p->col_size  = sz;
  std::vector<int32_t> string_start;
  for (int c = 0; c < num_columns; ++c)
    if (type_ids[c] == SRJ_STRING) {
      p->string_columns.push_back(c);
      string_start.push_back(st[c]);
    }
  // schedules: entries grouped by width class
  for (int k = 0; k < kNumClasses; ++k) {
    p->fr_class_begin[k] = static_cast<int32_t>(p->fr_entries.size());
    p->tr_class_begin[k] = static_cast<int32_t>(p->tr_entries.size());
    for (int c = 0; c < num_columns; ++c) {
      if (type_ids[c] == SRJ_STRING) {
        if (k == 2) p->fr_entries.push_back(Entry{st[c] + 4, c});  // the length word, RC:2163-2172
      } else if (class_of_size(sz[c]) == k) {
        p->fr_entries.push_back(Entry{st[c], c});
        p->tr_entries.push_back(Entry{st[c], c});
      }
    }
  }
  p->fr_class_begin[kNumClasses] = static_cast<int32_t>(p->fr_entries.size());
  p->tr_class_begin[kNumClasses] = static_cast<int32_t>(p->tr_entries.size());

  // from_rows tiling (shared memory budget 227 KB/CTA on sm_100)
  Tiling& tl = p->tiling;
  const int S = p->fixed_row_size;
  // Narrow rows (512 rows fit 64 KB): three 64 KB stages.  Wider rows: two 100 KB stages -- taller tiles mean longer
  // contiguous pieces per column and per CTA, which is what the DRAM likes once the part is warm (C2, 200 B rows:
  // 256-row tiles 92.3 %, 512-row tiles 94.7 % of the measured copy bandwidth on the same box).
  if (S <= 128) { tl.num_stages = 3; tl.stage_bytes = 64 * 1024; }
  else          { tl.num_stages = 2; tl.stage_bytes = 100 * 1024; }
  int fitrows = tl.stage_bytes / S;
  int R       = fitrows / 32 * 32;
  if (R > 512) R = 512;
  if (R >= 128) R = R / 128 * 128;  // 4 row groups per unit => predicate-free fast path
  if (R < 32) R = fitrows >= 16 ? 16 : 8;
  // development knobs (tuning only)
  if (const int v = SRJ_KNOB("SRJ_FR_STAGES", 0)) tl.num_stages = v;
  if (const int v = SRJ_KNOB("SRJ_FR_TILE_ROWS", 0)) { R = v; tl.stage_bytes = std::max(R * S, 4096); }
  if (const int v = SRJ_KNOB("SRJ_FR_STAGE_KB", 0)) tl.stage_bytes = v * 1024;
  tl.tile_rows     = R;
  tl.rows_per_item = R >= 32 ? 32 : R;
  // The per-schema shared-memory tables (entry starts, column and mask pointers, null counters) come on top of the
  // stages: for very wide schemas shrink the stages until the kernel's request fits the 227 KB limit.
  {
    const int nent_fr = static_cast<int>(p->fr_entries.size());
    while (from_rows_smem_bytes(tl, nent_fr, num_columns, lay.num_string_columns) > 232448 && tl.stage_bytes > 8 * 1024) {
      tl.stage_bytes   = (tl.stage_bytes * 3 / 4) & ~127;
      int fit          = tl.stage_bytes / S;
      int r2           = fit / 32 * 32;
      if (r2 > 512) r2 = 512;
      if (r2 >= 128) r2 = r2 / 128 * 128;
      if (r2 < 32) r2 = fit >= 16 ? 16 : 8;
      tl.tile_rows     = r2;
      tl.rows_per_item = r2 >= 32 ? 32 : r2;
    }
    if (from_rows_smem_bytes(tl, nent_fr, num_columns, lay.num_string_columns) > 232448) {
      delete p;
      set_error("plan_create: schema too wide for the kernels' shared-memory tables (%d columns)", num_columns);
      return SRJ_EUNSUPPORTED;
    }
  }

  plan_wide(p);  // slabs of a wide variable-width table (from_rows_wide.cu); p->wide.enabled says whether it applies

  // device mirror
  {
    const cudaError_t e0 = cudaGetDevice(&p->device);
    if (e0 != cudaSuccess) { delete p; return cuda_fail(e0, "cudaGetDevice"); }
  }
  const size_t b_fr = p->fr_entries.size() * sizeof(Entry);
  const size_t b_tr = p->tr_entries.size() * sizeof(Entry);
  const size_t b_cs = static_cast<size_t>(num_columns) * 4;
  const size_t b_sc = p->string_columns.size() * 4;
  std::vector<int32_t> tr_chunk(p->tr_entries.size());
  {
    // staging layout of to_rows2: widest class first so that every piece stays 16-byte aligned
    int32_t acc = 0;
    for (int k = kNumClasses - 1; k >= 0; --k)
      for (int e = p->tr_class_begin[k]; e < p->tr_class_begin[k + 1]; ++e) { tr_chunk[e] = acc; acc += 1 << k; }
  }
  const size_t b_tc = tr_chunk.size() * 4;
  const size_t b_we = p->wide.enabled ? p->wide.entries.size() * sizeof(WideEntry) : 0;
  const size_t b_ws = p->wide.enabled ? p->wide.slabs.size() * sizeof(WideSlab) : 0;
  const size_t tot  = b_fr + b_tr + b_cs + 2 * b_sc + b_tc + b_we + b_ws + 96;
  std::vector<uint8_t> blob(tot, 0);
  size_t o = 0;
  auto put = [&](const void* src, size_t n) { size_t at = o; if (n) memcpy(blob.data() + o, src, n); o += (n + 7) & ~size_t{7}; return at; };
  const size_t o_fr = put(p->fr_entries.data(), b_fr);
  const size_t o_tr = put(p->tr_entries.data(), b_tr);
  const size_t o_cs = put(st.data(), b_cs);
  const size_t o_sc = put(p->string_columns.data(), b_sc);
  const size_t o_ss = put(string_start.data(), b_sc);
  const size_t o_tc = put(tr_chunk.data(), b_tc);
  const size_t o_we = put(p->wide.entries.data(), b_we);
  const size_t o_ws = put(p->wide.slabs.data(), b_ws);
  cudaError_t e = cudaMalloc(&p->d_blob, tot);
  if (e != cudaSuccess) { delete p; return cuda_fail(e, "cudaMalloc(plan)"); }
  e = cudaMemcpy(p->d_blob, blob.data(), tot, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { cudaFree(p->d_blob); delete p; return cuda_fail(e, "cudaMemcpy(plan)"); }
  auto* base        = static_cast<uint8_t*>(p->d_blob);
  p->d_fr_entries   = reinterpret_cast<const Entry*>(base + o_fr);
  p->d_tr_entries   = reinterpret_cast<const Entry*>(base + o_tr);
  p->d_col_start    = reinterpret_cast<const int32_t*>(base + o_cs);
  p->d_string_cols  = reinterpret_cast<const int32_t*>(base + o_sc);
  p->d_string_start = reinterpret_cast<const int32_t*>(base + o_ss);
  p->d_tr_chunk_off = reinterpret_cast<const int32_t*>(base + o_tc);
  p->wide.d_entries = reinterpret_cast<const WideEntry*>(base + o_we);
  p->wide.d_slabs   = reinterpret_cast<const WideSlab*>(base + o_ws);
  *out              = p;
  return SRJ_OK;
}

void srj_plan_destroy(srj_plan* plan)
{
  if (!plan) return;
  if (plan->d_blob) cudaFree(plan->d_blob);
  for (auto& ar : plan->host_pool.a) {
    for (auto& s : ar.st) if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
    for (auto& d : ar.d_buf) if (d) cudaFree(d);
    if (ar.h_pin) cudaFreeHost(ar.h_pin);
  }
  for (auto& sl : plan->ring.slots) {
    if (sl.used && sl.ev) cudaEventSynchronize(sl.ev);
    if (sl.d_buf) cudaFree(sl.d_buf);
    if (sl.h_pinned) cudaFreeHost(sl.h_pinned);
    if (sl.ev) cudaEventDestroy(sl.ev);
  }
  delete plan;
}

int srj_plan_layout(const srj_plan* plan, srj_layout* out)
{
  if (!plan || !out) { set_error("plan_layout: null argument"); return SRJ_EINVAL; }
  out->num_columns        = plan->num_columns;
  out->num_string_columns = plan->num_string_columns;
  out->validity_offset    = plan->validity_offset;
  out->size_per_row       = plan->size_per_row;
  out->fixed_row_size     = plan->fixed_row_size;
  out->reserved           = 0;
  return SRJ_OK;
}

// ---------------------------------------------------------------------------------------------------
// convert_to_rows
// ---------------------------------------------------------------------------------------------------
static const int kRsChunkHost = 4096;  // must match kRsChunk in to_rows.cu

int64_t srj_to_rows_workspace_bytes(const srj_plan* plan, int64_t num_rows)
{
  if (!plan || plan->num_string_columns == 0 || num_rows <= 0) return 0;
  const int64_t nchunks = (num_rows + kRsChunkHost - 1) / kRsChunkHost;
  return (num_rows + nchunks) * 8;
}

int srj_to_rows_plan_batches(const srj_plan* plan, const srj_column* cols, int64_t num_rows, void* workspace,
                             srj_row_batch* batches, int32_t max_batches, int32_t* num_batches, void* stream_)
{
  SRJ_API_RANGE();
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int rc              = check_cols(plan, cols, num_rows, "to_rows_plan_batches");
  if (rc != SRJ_OK) return rc;
  if (!batches || !num_batches || max_batches < 1) { set_error("to_rows_plan_batches: bad batch array"); return SRJ_EINVAL; }
  *num_batches = 0;
  if (num_rows == 0) return SRJ_OK;
  const uint64_t MAXB = INT32_MAX;  // MAX_BATCH_SIZE, RC:65
  if (plan->num_string_columns == 0) {
    // constant row size: build_batches (RC:1466-1557) in closed form.
    const uint64_t S = plan->fixed_row_size;
    int64_t last     = 0;
    while (last < num_rows) {
      // lower_bound over (i - last) * S >= MAXB  (cum[i] - cum[last] with cum inclusive)
      const int64_t k      = static_cast<int64_t>((MAXB + S - 1) / S);  // first i - last reaching MAXB
      const bool to_end    = last + k >= num_rows;
      int64_t rows         = to_end ? num_rows - last : k / 32 * 32;
      while (static_cast<uint64_t>(rows) * S > MAXB) rows -= (rows % 32) ? (rows % 32) : 32;  // overflow guard
      if (rows <= 0) { set_error("to_rows: a single row exceeds 2 GiB"); return SRJ_EOVERFLOW; }
      if (*num_batches >= max_batches) { set_error("to_rows: more than %d batches", max_batches); return SRJ_EINVAL; }
      batches[*num_batches] = srj_row_batch{last, rows, static_cast<int64_t>(static_cast<uint64_t>(rows) * S)};
      ++*num_batches;
      last += rows;
    }
    return SRJ_OK;
  }
  if (!workspace) { set_error("to_rows_plan_batches: workspace is null"); return SRJ_EINVAL; }
  // device: per-row sizes + inclusive scan
  const int nstr = plan->num_string_columns;
  std::vector<const int32_t*> h_off(nstr);
  for (int s = 0; s < nstr; ++s) {
    h_off[s] = cols[plan->string_columns[s]].offsets;
    if (!h_off[s]) { set_error("to_rows: STRING column %d has no offsets", plan->string_columns[s]); return SRJ_EINVAL; }
  }
  // pointer table of the STRING offsets + room for the batch list the device computes
  const int cap          = std::min<int>(max_batches, 4096);
  const size_t tab_bytes = (sizeof(void*) * nstr + 15) & ~size_t{15};
  const size_t out_bytes = sizeof(int64_t) * (1 + 3 * static_cast<size_t>(cap));
  TableLease sc(plan, stream);
  rc = sc.acquire(tab_bytes + out_bytes);
  if (rc != SRJ_OK) return rc;
  memcpy(sc.host(), h_off.data(), sizeof(void*) * nstr);
  rc = sc.upload(sizeof(void*) * nstr);
  if (rc != SRJ_OK) return rc;
  uint64_t* cum = static_cast<uint64_t*>(workspace);
  rc            = launch_row_sizes(plan, static_cast<const int32_t* const*>(sc.dev()), num_rows, cum, stream);
  if (rc != SRJ_OK) return rc;
  // build_batches on the device, one read-back (the sync of RC:1534-1544, once instead of once per batch)
  int64_t* d_out = reinterpret_cast<int64_t*>(static_cast<uint8_t*>(sc.dev()) + tab_bytes);
  int64_t* h_out = reinterpret_cast<int64_t*>(static_cast<uint8_t*>(sc.host()) + tab_bytes);
  rc             = launch_batch_cut(cum, num_rows, cap, d_out, stream);
  if (rc != SRJ_OK) return rc;
  const size_t first = sizeof(int64_t) * (1 + 3 * static_cast<size_t>(std::min(cap, 8)));   // nearly always one batch
  SRJ_CUDA_TRY(cudaMemcpyAsync(h_out, d_out, first, cudaMemcpyDeviceToHost, stream));
  SRJ_CUDA_TRY(cudaStreamSynchronize(stream));
  if (h_out[0] > 8) {
    SRJ_CUDA_TRY(cudaMemcpyAsync(h_out, d_out, sizeof(int64_t) * (1 + 3 * static_cast<size_t>(h_out[0])), cudaMemcpyDeviceToHost, stream));
    SRJ_CUDA_TRY(cudaStreamSynchronize(stream));
  }
  if (h_out[0] == -1) { set_error("to_rows: a single row exceeds 2 GiB"); return SRJ_EOVERFLOW; }
  if (h_out[0] < 0) { set_error("to_rows: more than %d batches", cap); return SRJ_EINVAL; }
  *num_batches = static_cast<int32_t>(h_out[0]);
  for (int b = 0; b < *num_batches; ++b) batches[b] = srj_row_batch{h_out[1 + 3 * b], h_out[2 + 3 * b], h_out[3 + 3 * b]};
  return SRJ_OK;
}

int srj_convert_to_rows(const srj_plan* plan, const srj_column* cols, int64_t num_rows, const void* workspace,
                        const srj_row_batch* batches, int32_t num_batches, int32_t* const* batch_offsets,
                        uint8_t* const* batch_data, void* stream_)
{
  SRJ_API_RANGE();
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int rc              = check_cols(plan, cols, num_rows, "convert_to_rows");
  if (rc != SRJ_OK) return rc;
  if (num_batches == 0 || num_rows == 0) return SRJ_OK;
  if (!batches || !batch_offsets || !batch_data) { set_error("convert_to_rows: null batch arrays"); return SRJ_EINVAL; }
  const int nc = plan->num_columns, nstr = plan->num_string_columns;
  if (nstr > 0 && !workspace) { set_error("convert_to_rows: workspace is null"); return SRJ_EINVAL; }
  // pointer tables: [col_data nc][masks nc][str_offsets nstr][str_chars nstr]
  std::vector<const void*> tab(2 * static_cast<size_t>(nc) + 2 * static_cast<size_t>(nstr));
  for (int c = 0; c < nc; ++c) {
    if (plan->type_ids[c] != SRJ_STRING && !cols[c].data) { set_error("convert_to_rows: column %d has no data", c); return SRJ_EINVAL; }
    tab[c]      = cols[c].data;
    tab[nc + c] = cols[c].null_mask;
  }
  for (int s = 0; s < nstr; ++s) {
    const srj_column& c = cols[plan->string_columns[s]];
    if (!c.offsets) { set_error("convert_to_rows: STRING column %d has no offsets", plan->string_columns[s]); return SRJ_EINVAL; }
    tab[2 * nc + s]        = c.offsets;
    tab[2 * nc + nstr + s] = c.data;
  }
  TableLease sc(plan, stream);
  rc = sc.acquire(tab.size() * sizeof(void*));
  if (rc != SRJ_OK) return rc;
  memcpy(sc.host(), tab.data(), tab.size() * sizeof(void*));
  rc = sc.upload(tab.size() * sizeof(void*));
  if (rc != SRJ_OK) return rc;
  auto** d = static_cast<const void**>(sc.dev());
  for (int b = 0; b < num_batches; ++b) {
    if (!batch_offsets[b] || (!batch_data[b] && batches[b].num_bytes > 0)) { set_error("convert_to_rows: batch %d buffers are null", b); return SRJ_EINVAL; }
    rc = launch_to_rows(plan, d, reinterpret_cast<const uint32_t* const*>(d + nc),
                        reinterpret_cast<const int32_t* const*>(d + 2 * nc),
                        reinterpret_cast<const uint8_t* const*>(d + 2 * nc + nstr), batches[b].row_start,
                        batches[b].row_count, nstr ? static_cast<const uint64_t*>(workspace) : nullptr,
                        batch_offsets[b], batch_data[b], batches[b].num_bytes, stream, tab.data(),
                        // the scan partials behind the cumulative sizes are dead after plan_batches: 4 bytes of
                        // them carry the "fast kernel gave up" flag
                        nstr ? reinterpret_cast<int32_t*>(const_cast<uint64_t*>(static_cast<const uint64_t*>(workspace)) + num_rows) : nullptr);
    if (rc != SRJ_OK) return rc;
  }
  return SRJ_OK;
}

// ---------------------------------------------------------------------------------------------------
// convert_from_rows
// ---------------------------------------------------------------------------------------------------
int64_t srj_from_rows_workspace_bytes(const srj_plan* plan, int64_t num_rows)
{
  if (!plan || num_rows <= 0 || !plan->wide.enabled) return 0;
  return wide_workspace_bytes(plan, num_rows);
}

int srj_convert_from_rows_fixed(const srj_plan* plan, const uint8_t* rows, const int32_t* row_offsets,
                                int64_t rows_bytes, int64_t num_rows, const srj_column* cols, int64_t* d_null_counts,
                                int64_t* d_char_totals, const srj_fused_hash* hash, void* workspace, void* stream_)
{
  SRJ_API_RANGE();
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int rc              = check_cols(plan, cols, num_rows, "convert_from_rows");
  if (rc != SRJ_OK) return rc;
  const int nc = plan->num_columns, nstr = plan->num_string_columns;
  if (nstr > 0 && !row_offsets && num_rows > 0) { set_error("convert_from_rows: a schema with STRING columns needs the LIST offsets"); return SRJ_EINVAL; }
  if (nstr == 0) row_offsets = nullptr;  // fixed-width schemas ignore the offsets like the reference (RC:2317)
  // RC:2197: size_per_row * num_rows <= child.size()
  if (static_cast<int64_t>(plan->fixed_row_size) * num_rows > rows_bytes) {
    set_error("convert_from_rows: The layout of the data appears to be off (%lld rows x %d bytes > %lld)", (long long)num_rows, plan->fixed_row_size, (long long)rows_bytes);
    return SRJ_EINVAL;
  }
  if (num_rows > 0 && !rows) { set_error("convert_from_rows: rows is null"); return SRJ_EINVAL; }
  if (hash && hash->kind != SRJ_HASH_NONE) {
    if (hash->num_keys < 0 || hash->num_keys > 16 || !hash->out) { set_error("fused hash: bad key list / output"); return SRJ_EINVAL; }
    for (int k = 0; k < hash->num_keys; ++k) {
      const int c = hash->key_columns[k];
      if (c < 0 || c >= nc) { set_error("fused hash: key column %d out of range", c); return SRJ_EINVAL; }
      if (plan->type_ids[c] == SRJ_STRING) { set_error("fused hash: STRING keys are not supported in the fused path"); return SRJ_EUNSUPPORTED; }
      if (hash->kind == SRJ_HASH_HIVE && !hash::hive_supported(plan->type_ids[c])) { set_error("fused hive hash: unsupported key type %d", plan->type_ids[c]); return SRJ_EUNSUPPORTED; }
    }
  }
  for (int c = 0; c < nc; ++c) {
    if (plan->type_ids[c] == SRJ_STRING) {
      if (!cols[c].offsets) { set_error("convert_from_rows: STRING column %d has no offsets buffer", c); return SRJ_EINVAL; }
    } else if (!cols[c].data && num_rows > 0) {
      set_error("convert_from_rows: column %d has no data buffer", c); return SRJ_EINVAL;
    }
    if (!cols[c].null_mask && num_rows > 0) { set_error("convert_from_rows: column %d has no null mask buffer (always allocated, RC:2220)", c); return SRJ_EINVAL; }
  }
  // The hash of a "fused" call can run inside the conversion kernel (no extra traffic: the consumer warps hash the key
  // fields they already hold) or as the streaming hash kernel over the key columns just written (12 more bytes per row
  // for two integer keys, but the conversion kernel keeps its issue slots for the transpose and the hash its own kernel
  // shape).  SRJ_FUSE_SPLIT picks the second; it also lets wide variable-width tables keep their fast path.
  const bool want_hash  = hash && hash->kind != SRJ_HASH_NONE;
  const bool split_hash = want_hash && SRJ_KNOB("SRJ_FUSE_SPLIT", 1) != 0;
  const srj_fused_hash* fused = split_hash ? nullptr : hash;
  auto hash_after = [&]() -> int {
    if (!split_hash || num_rows == 0) return SRJ_OK;
    srj_column keys[16];
    for (int k = 0; k < hash->num_keys; ++k) keys[k] = cols[hash->key_columns[k]];
    return launch_hash(hash->kind, keys, hash->num_keys, num_rows, hash->seed, hash->out, stream);
  };
  if (use_wide_from_rows(plan, row_offsets, fused)) {
    // wide variable-width table: per-row slabs; the pointer tables travel as kernel parameters and the kernels publish
    // null counts / totals / status themselves: no memset, no staging copy, no hidden allocation
    if (num_rows > 0 && !workspace) { set_error("convert_from_rows: this schema needs a workspace (srj_from_rows_workspace_bytes)"); return SRJ_EINVAL; }
    rc = launch_from_rows_wide(plan, rows, row_offsets, rows_bytes, num_rows, cols, d_null_counts, d_char_totals, workspace,
                               SRJ_KNOB("SRJ_W_FINALIZE", 0) != 0, stream);
    return rc != SRJ_OK ? rc : hash_after();
  }
  if (d_null_counts) SRJ_CUDA_TRY(cudaMemsetAsync(d_null_counts, 0, sizeof(int64_t) * nc, stream));
  if (d_char_totals) SRJ_CUDA_TRY(cudaMemsetAsync(d_char_totals, 0, sizeof(int64_t) * (nc + 1), stream));
  const size_t nent = plan->fr_entries.size();
  // pointer tables: [ent_dst nent][masks nc][str_offsets nstr] + scan partials
  std::vector<void*> tab(nent + nc + nstr);
  for (size_t e = 0; e < nent; ++e) {
    const int c = plan->fr_entries[e].column;
    tab[e]      = plan->type_ids[c] == SRJ_STRING ? static_cast<void*>(reinterpret_cast<uint8_t*>(cols[c].offsets) + 4)  // lengths land at offsets[1..n]
                                                  : cols[c].data;
  }
  for (int c = 0; c < nc; ++c) tab[nent + c] = cols[c].null_mask;
  for (int s = 0; s < nstr; ++s) tab[nent + nc + s] = cols[plan->string_columns[s]].offsets;
  const size_t tab_bytes  = (tab.size() * sizeof(void*) + 15) & ~size_t{15};
  const size_t part_bytes = static_cast<size_t>(string_scan_partials_bytes(nstr, num_rows));
  TableLease sc(plan, stream);
  rc = sc.acquire(tab_bytes + part_bytes + 16);
  if (rc != SRJ_OK) return rc;
  memcpy(sc.host(), tab.data(), tab.size() * sizeof(void*));
  rc = sc.upload(tab.size() * sizeof(void*));
  if (rc != SRJ_OK) return rc;
  auto** d = static_cast<void**>(sc.dev());
  rc = launch_from_rows(plan, rows, row_offsets, rows_bytes, num_rows, d, reinterpret_cast<uint32_t* const*>(d + nent),
                        d_null_counts, d_char_totals ? d_char_totals + nc : nullptr, fused, stream);
  if (rc != SRJ_OK) return rc;
  if (nstr > 0) {
    uint8_t* tail = static_cast<uint8_t*>(sc.dev()) + tab_bytes;
    rc = launch_string_offsets_scan(reinterpret_cast<int32_t* const*>(d + nent + nc), plan->d_string_cols, nstr, num_rows,
                                    d_char_totals, d_char_totals ? d_char_totals + nc : nullptr, tail, plan->wide.enabled, stream);
    if (rc != SRJ_OK) return rc;
  }
  return hash_after();
}

int srj_convert_from_rows_strings(const srj_plan* plan, const uint8_t* rows, const int32_t* row_offsets,
                                  int64_t rows_bytes, int64_t num_rows, const srj_column* cols,
                                  const int64_t* d_char_totals, const void* workspace, void* stream_)
{
  SRJ_API_RANGE();
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int rc              = check_cols(plan, cols, num_rows, "convert_from_rows_strings");
  if (rc != SRJ_OK) return rc;
  const int nstr = plan->num_string_columns;
  if (nstr == 0 || num_rows == 0) return SRJ_OK;
  if (!rows || !row_offsets) { set_error("convert_from_rows_strings: rows / offsets are null"); return SRJ_EINVAL; }
  for (int s = 0; s < nstr; ++s)
    if (!cols[plan->string_columns[s]].offsets) { set_error("convert_from_rows_strings: STRING column %d has no offsets", plan->string_columns[s]); return SRJ_EINVAL; }
  const int64_t* d_status = d_char_totals ? d_char_totals + plan->num_columns : nullptr;
  // wide tables: phase 1 (from_rows_wide.cu) left group-local offsets + the group bases in the workspace
  const uint32_t* d_bases = nullptr;
  if (plan->wide.enabled && SRJ_KNOB("SRJ_W_FINALIZE", 0) == 0) {
    if (!workspace) { set_error("convert_from_rows_strings: this schema needs the workspace phase 1 filled"); return SRJ_EINVAL; }
    d_bases = wide_workspace_bases(plan, num_rows, workspace);
  }
  if (strings_fast_path(plan, d_status))   // pointer tables travel as kernel parameters
    return launch_strings_from_rows(plan, rows, row_offsets, rows_bytes, num_rows, cols, nullptr, d_status, d_bases, stream);
  std::vector<void*> tab(2 * static_cast<size_t>(nstr));
  for (int s = 0; s < nstr; ++s) {
    const srj_column& c = cols[plan->string_columns[s]];
    tab[s]        = c.offsets;
    tab[nstr + s] = c.data;  // may be NULL only when the column has no chars at all
  }
  TableLease sc(plan, stream);
  rc = sc.acquire(tab.size() * sizeof(void*));
  if (rc != SRJ_OK) return rc;
  memcpy(sc.host(), tab.data(), tab.size() * sizeof(void*));
  rc = sc.upload(tab.size() * sizeof(void*));
  if (rc != SRJ_OK) return rc;
  return launch_strings_from_rows(plan, rows, row_offsets, rows_bytes, num_rows, cols, static_cast<void* const*>(sc.dev()),
                                  d_status, d_bases, stream);
}

// ---------------------------------------------------------------------------------------------------
// hashes
// ---------------------------------------------------------------------------------------------------
int srj_get_max_stack_depth(void) { return SRJ_MAX_STACK_DEPTH; }

// Tables with LIST / STRUCT keys: the column trees are uploaded through a process-wide staging ring (there is no plan
// on the hash entry points) and hashed by hash_nested.cu.
static int hash_any(int kind, const srj_column* cols, int32_t num_columns, int64_t num_rows, int64_t seed, void* out, cudaStream_t stream)
{
  if (!hash_has_nested(cols, num_columns)) return launch_hash(kind, cols, num_columns, num_rows, seed, out, stream);
  if (num_columns == 0 || num_rows == 0) return SRJ_OK;
  static srj_plan staging{};              // only its pointer-table ring is used
  constexpr size_t kBytes = 256 * 1024;   // ~5000 tree nodes
  TableLease sc(&staging, stream);
  int rc = sc.acquire(kBytes);
  if (rc != SRJ_OK) return rc;
  return launch_hash_nested(kind, cols, num_columns, num_rows, seed, out, sc.dev(), sc.host(), kBytes, stream);
}

int srj_xxhash64(const srj_column* cols, int32_t num_columns, int64_t num_rows, int64_t seed, int64_t* out, void* stream)
{
  SRJ_API_RANGE();
  if (num_columns < 0 || num_rows < 0 || (num_columns > 0 && !cols) || (num_rows > 0 && !out)) { set_error("xxhash64: bad argument"); return SRJ_EINVAL; }
  return hash_any(SRJ_HASH_XXHASH64, cols, num_columns, num_rows, seed, out, static_cast<cudaStream_t>(stream));
}

int srj_murmur_hash3_32(const srj_column* cols, int32_t num_columns, int64_t num_rows, uint32_t seed, int32_t* out,
                        void* stream)
{
  SRJ_API_RANGE();
  if (num_columns < 0 || num_rows < 0 || (num_columns > 0 && !cols) || (num_rows > 0 && !out)) { set_error("murmur_hash3_32: bad argument"); return SRJ_EINVAL; }
  return hash_any(SRJ_HASH_MURMUR3_32, cols, num_columns, num_rows, seed, out, static_cast<cudaStream_t>(stream));
}

int srj_hive_hash(const srj_column* cols, int32_t num_columns, int64_t num_rows, int32_t* out, void* stream)
{
  SRJ_API_RANGE();
  if (num_columns < 0 || num_rows < 0 || (num_columns > 0 && !cols) || (num_rows > 0 && !out)) { set_error("hive_hash: bad argument"); return SRJ_EINVAL; }
  return hash_any(SRJ_HASH_HIVE, cols, num_columns, num_rows, 0, out, static_cast<cudaStream_t>(stream));
}

// ---------------------------------------------------------------------------------------------------
// Spark HashPartitioning: pmod(murmur3_32(seed, keys), P) + stable partition (partition.cu)
// ---------------------------------------------------------------------------------------------------
int64_t srj_partition_workspace_bytes(int64_t num_rows, int32_t num_partitions)
{
  return partition_workspace_bytes(num_rows, num_partitions);
}

int srj_partition_plan(int32_t* d_partition_ids, int64_t num_rows, int32_t num_partitions, int32_t* d_partition_offsets,
                       int32_t* d_scatter_map, int32_t* d_gather_map, void* workspace, void* stream)
{
  SRJ_API_RANGE();
  if (num_rows < 0 || num_partitions <= 0 || !d_partition_offsets || (num_rows > 0 && (!d_partition_ids || !workspace))) {
    set_error("partition_plan: bad argument");
    return SRJ_EINVAL;
  }
  if (num_rows > INT32_MAX || num_partitions > (1 << 14)) {
    set_error("partition_plan: %lld rows / %d partitions exceed the int32 row index / 16384 partitions", static_cast<long long>(num_rows), num_partitions);
    return SRJ_EUNSUPPORTED;
  }
  return launch_partition_plan(d_partition_ids, num_rows, num_partitions, d_partition_offsets, d_scatter_map, d_gather_map, workspace,
                               static_cast<cudaStream_t>(stream));
}

int srj_hash_partition(const srj_column* keys, int32_t num_keys, int64_t num_rows, uint32_t seed, int32_t num_partitions,
                       int32_t* d_partition_ids, int32_t* d_partition_offsets, int32_t* d_scatter_map, int32_t* d_gather_map,
                       void* workspace, void* stream)
{
  SRJ_API_RANGE();
  if (num_keys <= 0 || !keys) { set_error("hash_partition: no key columns"); return SRJ_EINVAL; }
  if (num_rows > 0 && !d_partition_ids) { set_error("hash_partition: bad argument"); return SRJ_EINVAL; }
  // the hashes go where the ids will be: part_ids_kernel turns them into ids in place
  int rc = hash_any(SRJ_HASH_MURMUR3_32, keys, num_keys, num_rows, seed, d_partition_ids, static_cast<cudaStream_t>(stream));
  if (rc != SRJ_OK) return rc;
  return srj_partition_plan(d_partition_ids, num_rows, num_partitions, d_partition_offsets, d_scatter_map, d_gather_map, workspace, stream);
}

int srj_partition_columns(const srj_column* in, const srj_column* out, int32_t num_columns, int64_t num_rows, int32_t num_partitions,
                          const int32_t* d_scatter_map, const int32_t* d_gather_map, int64_t* d_null_counts, void* workspace, void* stream)
{
  SRJ_API_RANGE();
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (num_columns < 0 || num_rows < 0 || num_partitions <= 0 || (num_columns > 0 && (!in || !out))) { set_error("partition_columns: bad argument"); return SRJ_EINVAL; }
  if (num_rows > 0 && (!d_scatter_map || !d_gather_map || !workspace)) { set_error("partition_columns: the maps and the plan's workspace are needed"); return SRJ_EINVAL; }
  if (d_null_counts && num_columns > 0) SRJ_CUDA_TRY(cudaMemsetAsync(d_null_counts, 0, sizeof(int64_t) * num_columns, st));
  std::vector<int> esz(static_cast<size_t>(num_columns), 0);
  for (int32_t c = 0; c < num_columns; ++c) {
    const srj_column& a = in[c];
    const srj_column& b = out[c];
    if (a.type_id != b.type_id || a.size != num_rows || b.size != num_rows) { set_error("partition_columns: column %d: type / size mismatch", c); return SRJ_EINVAL; }
    if (a.type_id == SRJ_STRING) {
      if (!a.offsets || !b.offsets) { set_error("partition_columns: STRING column %d needs offsets", c); return SRJ_EINVAL; }
    } else {
      esz[c] = size_of_type(a.type_id);
      if (esz[c] <= 0) { set_error("partition_columns: column %d: unsupported type %d", c, a.type_id); return SRJ_EUNSUPPORTED; }
      if (num_rows > 0 && (!a.data || !b.data)) { set_error("partition_columns: column %d: NULL data", c); return SRJ_EINVAL; }
    }
    if (a.null_mask && !b.null_mask) { set_error("partition_columns: column %d has a null mask but its output has none", c); return SRJ_EINVAL; }
    if (!a.null_mask && b.null_mask && num_rows > 0) SRJ_CUDA_TRY(cudaMemsetAsync(b.null_mask, 0xff, static_cast<size_t>((num_rows + 31) / 32) * 4, st));
  }
  // fixed-width data and every null mask: tile by tile, staged in destination order (plans of <= 1024 partitions) ...
  int rc = launch_partition_move_tiles(in, out, esz.data(), num_columns, num_rows, num_partitions, d_scatter_map, workspace,
                                       reinterpret_cast<unsigned long long*>(d_null_counts), st);
  if (rc == SRJ_EUNSUPPORTED) {
    // ... or row by row
    rc = SRJ_OK;
    for (int32_t c = 0; c < num_columns && rc == SRJ_OK && num_rows > 0; ++c) {
      if (esz[c] > 0) rc = launch_partition_scatter_fixed(in[c].data, out[c].data, esz[c], d_scatter_map, num_rows, st);
      if (rc == SRJ_OK && in[c].null_mask)
        rc = launch_partition_gather_mask(in[c].null_mask, out[c].null_mask, d_gather_map, num_rows,
                                          d_null_counts ? reinterpret_cast<unsigned long long*>(d_null_counts + c) : nullptr, st);
    }
  }
  if (rc != SRJ_OK) return rc;
  // STRING columns: the output offsets (lengths through the gather map, then a scan; partials behind the plan's tile order)
  for (int32_t c = 0; c < num_columns; ++c) {
    if (in[c].type_id != SRJ_STRING) continue;
    if (num_rows == 0) {
      SRJ_CUDA_TRY(cudaMemsetAsync(out[c].offsets, 0, 4, st));   // an empty STRING column still has its offsets[0] = 0
      continue;
    }
    rc = launch_partition_string_offsets(in[c].offsets, out[c].offsets, d_gather_map, num_rows, static_cast<int32_t*>(workspace) + num_rows, st);
    if (rc != SRJ_OK) return rc;
  }
  return SRJ_OK;
}

int srj_partition_strings(const srj_column* in, const srj_column* out, int32_t num_columns, int64_t num_rows, const int32_t* d_gather_map,
                          void* stream)
{
  SRJ_API_RANGE();
  if (num_columns < 0 || num_rows < 0 || (num_columns > 0 && (!in || !out))) { set_error("partition_strings: bad argument"); return SRJ_EINVAL; }
  for (int32_t c = 0; c < num_columns; ++c) {
    if (in[c].type_id != SRJ_STRING || num_rows == 0) continue;
    if (!out[c].offsets || !in[c].offsets) { set_error("partition_strings: column %d: NULL offsets", c); return SRJ_EINVAL; }
    const int rc = launch_partition_gather_chars(static_cast<const uint8_t*>(in[c].data), in[c].offsets, static_cast<uint8_t*>(out[c].data),
                                                 out[c].offsets, d_gather_map, num_rows, static_cast<cudaStream_t>(stream));
    if (rc != SRJ_OK) return rc;
  }
  return SRJ_OK;
}

// ---------------------------------------------------------------------------------------------------
// Apache Spark UnsafeRow codec (unsafe_row.cu)
// ---------------------------------------------------------------------------------------------------
int srj_unsafe_row_layout(const int32_t* type_ids, int32_t num_columns, int32_t* bitset_bytes, int32_t* fixed_bytes)
{
  if (!type_ids || !bitset_bytes || !fixed_bytes) { set_error("unsafe_row_layout: bad argument"); return SRJ_EINVAL; }
  int32_t ndec = 0, nstr = 0, fb = 0;
  const int rc = unsafe_row_layout(type_ids, num_columns, bitset_bytes, &fb, &ndec, &nstr);
  if (rc != SRJ_OK) { set_error("unsafe_row_layout: 1..256 columns of fixed-width, decimal or STRING type"); return rc; }
  *fixed_bytes = fb + 16 * ndec;   // every DECIMAL128 field reserves 16 bytes of the variable region
  return SRJ_OK;
}

int64_t srj_unsafe_row_workspace_bytes(int32_t num_columns, int64_t num_rows) { return unsafe_row_workspace_bytes(num_columns, std::max<int64_t>(0, num_rows)); }

static int ur_check(const char* what, const srj_column* cols, int32_t ncols, int64_t n, const void* workspace)
{
  if (ncols <= 0 || n < 0 || !cols || !workspace) { set_error("%s: bad argument", what); return SRJ_EINVAL; }
  if (n > INT32_MAX) { set_error("%s: more than INT32_MAX rows", what); return SRJ_EOVERFLOW; }
  for (int32_t c = 0; c < ncols; ++c)
    if (cols[c].size != n) { set_error("%s: column %d has %lld rows, expected %lld", what, c, static_cast<long long>(cols[c].size), static_cast<long long>(n)); return SRJ_EINVAL; }
  return SRJ_OK;
}

int srj_unsafe_row_sizes(const srj_column* cols, int32_t num_columns, int64_t num_rows, int32_t* d_row_offsets, int64_t* total_bytes,
                         void* workspace, void* stream)
{
  SRJ_API_RANGE();
  int rc = ur_check("unsafe_row_sizes", cols, num_columns, num_rows, workspace);
  if (rc != SRJ_OK) return rc;
  if (!d_row_offsets || !total_bytes) { set_error("unsafe_row_sizes: bad argument"); return SRJ_EINVAL; }
  rc = launch_unsafe_row_sizes(cols, num_columns, num_rows, d_row_offsets, workspace, total_bytes, static_cast<cudaStream_t>(stream));
  if (rc == SRJ_EOVERFLOW) set_error("unsafe_row_sizes: %lld bytes of rows exceed one LIST<INT8> column (INT32_MAX): convert fewer rows per call", static_cast<long long>(*total_bytes));
  else if (rc == SRJ_EUNSUPPORTED) set_error("unsafe_row_sizes: unsupported column type or more than 256 columns");
  return rc;
}

int srj_convert_to_unsafe_rows(const srj_column* cols, int32_t num_columns, int64_t num_rows, const int32_t* d_row_offsets, uint8_t* rows,
                               void* workspace, void* stream)
{
  SRJ_API_RANGE();
  int rc = ur_check("convert_to_unsafe_rows", cols, num_columns, num_rows, workspace);
  if (rc != SRJ_OK) return rc;
  if ((num_rows > 0 && !rows) || (reinterpret_cast<uintptr_t>(rows) & 7)) { set_error("convert_to_unsafe_rows: rows must be 8-byte aligned"); return SRJ_EINVAL; }
  if (!d_row_offsets)
    for (int32_t c = 0; c < num_columns; ++c)
      if (cols[c].type_id == SRJ_STRING) { set_error("convert_to_unsafe_rows: STRING columns need the row offsets of srj_unsafe_row_sizes"); return SRJ_EINVAL; }
  rc = launch_unsafe_to_rows(cols, num_columns, num_rows, d_row_offsets, rows, workspace, static_cast<cudaStream_t>(stream));
  if (rc == SRJ_EUNSUPPORTED) set_error("convert_to_unsafe_rows: unsupported column type or more than 256 columns");
  return rc;
}

int srj_convert_from_unsafe_rows(const uint8_t* rows, const int32_t* d_row_offsets, int64_t num_rows, const srj_column* out, int32_t num_columns,
                                 int64_t* d_null_counts, void* workspace, void* stream)
{
  SRJ_API_RANGE();
  int rc = ur_check("convert_from_unsafe_rows", out, num_columns, num_rows, workspace);
  if (rc != SRJ_OK) return rc;
  if ((num_rows > 0 && !rows) || (reinterpret_cast<uintptr_t>(rows) & 7)) { set_error("convert_from_unsafe_rows: rows must be 8-byte aligned"); return SRJ_EINVAL; }
  if (!d_row_offsets)
    for (int32_t c = 0; c < num_columns; ++c)
      if (out[c].type_id == SRJ_STRING) { set_error("convert_from_unsafe_rows: variable-width rows need their offsets"); return SRJ_EINVAL; }
  rc = launch_unsafe_from_rows(out, num_columns, num_rows, rows, d_row_offsets, d_null_counts, workspace, static_cast<cudaStream_t>(stream));
  if (rc == SRJ_EUNSUPPORTED) set_error("convert_from_unsafe_rows: unsupported column type or more than 256 columns");
  return rc;
}

int srj_convert_from_unsafe_rows_strings(const uint8_t* rows, const int32_t* d_row_offsets, int64_t num_rows, const srj_column* out,
                                         int32_t num_columns, void* stream)
{
  SRJ_API_RANGE();
  if (num_columns <= 0 || num_rows < 0 || !out || (num_rows > 0 && (!rows || !d_row_offsets))) { set_error("convert_from_unsafe_rows_strings: bad argument"); return SRJ_EINVAL; }
  if (reinterpret_cast<uintptr_t>(rows) & 7) { set_error("convert_from_unsafe_rows_strings: rows must be 8-byte aligned"); return SRJ_EINVAL; }
  return launch_unsafe_from_rows_strings(out, num_columns, num_rows, rows, d_row_offsets, static_cast<cudaStream_t>(stream));
}

// ---------------------------------------------------------------------------------------------------
// Kudo shuffle wire format: split / assemble (kudo.cu)
// ---------------------------------------------------------------------------------------------------
int64_t srj_kudo_workspace_bytes(int32_t num_columns, int32_t num_partitions) { return kudo_workspace_bytes(std::max(num_columns, 0), std::max(num_partitions, 0)); }

static int kudo_check(const char* what, int32_t ncols, int32_t P, const void* a, const void* b, const void* ws)
{
  if (ncols <= 0 || P < 0 || !a || !b || !ws) { set_error("%s: bad argument", what); return SRJ_EINVAL; }
  if (ncols > 256 || P > 65535) { set_error("%s: at most 256 columns and 65535 partitions", what); return SRJ_EUNSUPPORTED; }
  return SRJ_OK;
}

int srj_kudo_split_sizes(const srj_column* cols, int32_t num_columns, int64_t num_rows, const int32_t* d_splits, int32_t num_partitions,
                         int64_t* d_partition_offsets, int64_t* total_bytes, void* workspace, void* stream)
{
  SRJ_API_RANGE();
  int rc = kudo_check("kudo_split_sizes", num_columns, num_partitions, cols, d_partition_offsets, workspace);
  if (rc != SRJ_OK) return rc;
  if (!d_splits || !total_bytes || num_rows < 0 || num_rows > INT32_MAX) { set_error("kudo_split_sizes: bad argument"); return SRJ_EINVAL; }
  for (int32_t c = 0; c < num_columns; ++c)
    if (cols[c].size != num_rows) { set_error("kudo_split_sizes: column %d: row count mismatch", c); return SRJ_EINVAL; }
  rc = launch_kudo_split_sizes(cols, num_columns, d_splits, num_partitions, d_partition_offsets, total_bytes, workspace, static_cast<cudaStream_t>(stream));
  if (rc == SRJ_EUNSUPPORTED) set_error("kudo_split_sizes: only fixed-width, decimal and STRING columns");
  else if (rc == SRJ_EOVERFLOW) set_error("kudo_split_sizes: a partition exceeds the 32-bit section lengths of the Kudo header, or the splits are not increasing");
  return rc;
}

int srj_kudo_split(const srj_column* cols, int32_t num_columns, int64_t num_rows, const int32_t* d_splits, int32_t num_partitions,
                   const int64_t* d_partition_offsets, uint8_t* out, void* workspace, void* stream)
{
  SRJ_API_RANGE();
  int rc = kudo_check("kudo_split", num_columns, num_partitions, cols, d_partition_offsets, workspace);
  if (rc != SRJ_OK) return rc;
  if (!d_splits || (num_partitions > 0 && !out) || (reinterpret_cast<uintptr_t>(out) & 3)) { set_error("kudo_split: out must be a 4-byte aligned device buffer"); return SRJ_EINVAL; }
  if (num_partitions == 0) return SRJ_OK;
  (void)num_rows;
  rc = launch_kudo_split(cols, num_columns, d_splits, num_partitions, d_partition_offsets, out, workspace, static_cast<cudaStream_t>(stream));
  if (rc == SRJ_EUNSUPPORTED) set_error("kudo_split: only fixed-width, decimal and STRING columns");
  return rc;
}

int srj_kudo_assemble_sizes(const uint8_t* partitions, const int64_t* d_partition_offsets, int32_t num_partitions, const int32_t* type_ids,
                            int32_t num_columns, int64_t* total_rows, int64_t* char_totals, void* workspace, void* stream)
{
  SRJ_API_RANGE();
  int rc = kudo_check("kudo_assemble_sizes", num_columns, num_partitions, type_ids, d_partition_offsets, workspace);
  if (rc != SRJ_OK) return rc;
  if ((num_partitions > 0 && !partitions) || !total_rows || !char_totals) { set_error("kudo_assemble_sizes: bad argument"); return SRJ_EINVAL; }
  rc = launch_kudo_assemble_sizes(partitions, d_partition_offsets, num_partitions, type_ids, num_columns, total_rows, char_totals, workspace,
                                  static_cast<cudaStream_t>(stream));
  if (rc == SRJ_EINVAL) set_error("kudo_assemble_sizes: a partition is not a well-formed Kudo partition of %d columns", num_columns);
  else if (rc == SRJ_EUNSUPPORTED) set_error("kudo_assemble_sizes: only fixed-width, decimal and STRING columns");
  else if (rc == SRJ_EOVERFLOW) set_error("kudo_assemble_sizes: the assembled rows or chars of a column exceed INT32_MAX");
  else if (rc == SRJ_OK && *total_rows > INT32_MAX) { set_error("kudo_assemble_sizes: %lld rows exceed a column", static_cast<long long>(*total_rows)); return SRJ_EOVERFLOW; }
  return rc;
}

int srj_kudo_assemble(const uint8_t* partitions, const int64_t* d_partition_offsets, int32_t num_partitions, const srj_column* out,
                      int32_t num_columns, int64_t total_rows, void* workspace, void* stream)
{
  SRJ_API_RANGE();
  int rc = kudo_check("kudo_assemble", num_columns, num_partitions, out, d_partition_offsets, workspace);
  if (rc != SRJ_OK) return rc;
  for (int32_t c = 0; c < num_columns; ++c)
    if (out[c].size != total_rows) { set_error("kudo_assemble: column %d: expected %lld rows", c, static_cast<long long>(total_rows)); return SRJ_EINVAL; }
  rc = launch_kudo_assemble(partitions, d_partition_offsets, num_partitions, out, num_columns, total_rows, workspace, static_cast<cudaStream_t>(stream));
  if (rc == SRJ_EUNSUPPORTED) set_error("kudo_assemble: only fixed-width, decimal and STRING columns");
  return rc;
}

int64_t srj_kudo_nested_workspace_bytes(int32_t num_flat, int32_t num_partitions)
{
  return kudo_workspace_bytes(std::max(num_flat, 0), std::max(num_partitions, 0));
}

int srj_kudo_assemble_nested_sizes(const uint8_t* partitions, const int64_t* d_partition_offsets, int32_t num_partitions, const int32_t* flat_type_ids,
                                   const int32_t* flat_num_children, int32_t num_flat, int64_t* flat_rows, int64_t* char_totals, void* workspace,
                                   void* stream)
{
  SRJ_API_RANGE();
  int rc = kudo_check("kudo_assemble_nested_sizes", num_flat, num_partitions, flat_type_ids, d_partition_offsets, workspace);
  if (rc != SRJ_OK) return rc;
  if ((num_partitions > 0 && !partitions) || !flat_num_children || !flat_rows || !char_totals) { set_error("kudo_assemble_nested_sizes: bad argument"); return SRJ_EINVAL; }
  rc = launch_kudo_assemble_nested_sizes(partitions, d_partition_offsets, num_partitions, flat_type_ids, flat_num_children, num_flat, flat_rows, char_totals,
                                         workspace, static_cast<cudaStream_t>(stream));
  if (rc == SRJ_EINVAL) set_error("kudo_assemble_nested_sizes: the flattened schema is not a forest of %d columns (a LIST has one child), or a partition is not a well-formed Kudo partition of it", num_flat);
  else if (rc == SRJ_EUNSUPPORTED) set_error("kudo_assemble_nested_sizes: a type outside fixed-width, decimal, STRING, LIST and STRUCT");
  else if (rc == SRJ_EOVERFLOW) set_error("kudo_assemble_nested_sizes: the assembled rows or chars of a column exceed INT32_MAX");
  return rc;
}

int srj_kudo_assemble_nested(const uint8_t* partitions, const int64_t* d_partition_offsets, int32_t num_partitions, const srj_column* out,
                             int32_t num_columns, void* workspace, void* stream)
{
  SRJ_API_RANGE();
  int rc = kudo_check("kudo_assemble_nested", num_columns, num_partitions, out, d_partition_offsets, workspace);
  if (rc != SRJ_OK) return rc;
  rc = launch_kudo_assemble_nested(partitions, d_partition_offsets, num_partitions, out, num_columns, workspace, static_cast<cudaStream_t>(stream));
  if (rc == SRJ_EINVAL) set_error("kudo_assemble_nested: malformed column tree (a LIST has one child and offsets, children are given)");
  else if (rc == SRJ_EUNSUPPORTED) set_error("kudo_assemble_nested: more than 256 flattened columns, or a type outside the format");
  return rc;
}

}  // extern "C"
