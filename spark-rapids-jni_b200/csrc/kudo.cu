// kudo.cu -- the reference's Kudo shuffle wire format for flat tables (SURVEY §8f rank 2): split a table at row indices
// into P self-describing partitions laid back to back in one buffer (shuffle_split, src/main/cpp/src/shuffle_split.hpp:60-136,
// shuffle_split.cu:640-690,940-1075) and assemble such partitions back into one table (shuffle_assemble,
// shuffle_split.hpp:174-189).  The bytes are the format of kudo/KudoSerializer.java:49-171:
//   partition = header | hasValidity bits | validity | offsets | data
//   header    = "KUD0", row offset, row count, validity length, offsets length, total length, column count: seven
//               BIG-ENDIAN 32-bit integers (kudo/KudoTableHeader.java:186-200); then (ncols + 7) / 8 bytes, bit c = column
//               c carries validity in this partition (it has a mask and the partition has rows)
//   validity  = per such column the mask bytes [row / 8, (row + n - 1) / 8] copied as they are (the reader skips row % 8
//               bits, kudo/SlicedValidityBufferInfo.java:63-77); the section is padded so that header + validity is a
//               multiple of 4 (KudoSerializer.java:497-499)
//   offsets   = per STRING column the n + 1 raw int32 offsets (not rebased), when n > 0; data = per column n * size bytes
//               or the chars; both sections padded to 4
// Split writes flat tables (fixed-width, decimals, STRING).  Assemble also reads nested tables (LIST / STRUCT columns,
// KudoTableHeaderCalc.java:77-195, SlicedBufferSerializer.java:72-247, KudoTableMerger.java:96-295): the columns are
// flattened in pre-order (a LIST / STRUCT before its children) and the column count and hasValidity bits index that
// list; every flattened column has a slice (offset, rows): the header's at the root, the parent's below a STRUCT,
// (off[0], off[n] - off[0]) of the list's raw offsets below a LIST.  Validity comes for STRUCT, LIST and leaf columns,
// offsets for LIST and STRING columns, data for leaves, each in pre-order.  A flat table is a schema of leaves.
//
// Kernels: split -- a thread per partition sizes it; one CTA per (column, partition) moves that column's buffers.
// Assemble -- a thread per partition checks its header and walks the flattened schema once, recording per (column,
// partition) the slice and where the column's buffers lie (every read is checked against the partition's bytes); one
// CTA per column scans the partitions for row and char bases; one CTA per (column, partition) moves the buffers with
// the widest accesses the two addresses allow.  Validity bits reach the output words with atomicOr (a slice starts at
// an arbitrary row); LIST offsets are rebased onto the child's row base.
#include <algorithm>
#include <vector>

#include "common.cuh"
#include "kernels.hpp"

namespace srj {

constexpr int kKudoMaxCols   = 256;
constexpr uint32_t kKudoMagic = 0x4B554430u;

enum : int32_t { KK_FIXED = 0, KK_STRING = 1, KK_LIST = 2, KK_STRUCT = 3 };

struct KCol {
  uint8_t* data;        // fixed-width values or chars
  uint8_t* mask;        // validity bytes (bit r%8 of byte r/8), or NULL
  int32_t* offsets;     // STRING / LIST
  int32_t size;         // element bytes, 0 for STRING / LIST / STRUCT
  int32_t kind;         // KK_*
  int32_t parent;       // flattened index of the parent column, -1 at the root
  int32_t pad;
};

__host__ __device__ __forceinline__ int64_t pad4(int64_t x) { return (x + 3) & ~int64_t{3}; }
__device__ __forceinline__ uint32_t bswap32(uint32_t v) { return __byte_perm(v, 0, 0x0123); }
__host__ __device__ __forceinline__ int kudo_header_bytes(int ncols) { return 28 + (ncols + 7) / 8; }

// bytes of the three buffers of column c for rows [s, s + n)
__device__ __forceinline__ void kudo_col_sizes(const KCol& c, int32_t s, int32_t n, int64_t& v, int64_t& o, int64_t& d)
{
  v = (c.mask && n > 0) ? (s + n - 1) / 8 - s / 8 + 1 : 0;
  if (c.size == 0) {
    o = n > 0 ? 4 * (static_cast<int64_t>(n) + 1) : 0;
    d = c.offsets ? static_cast<int64_t>(c.offsets[s + n]) - c.offsets[s] : 0;
  } else {
    o = 0;
    d = static_cast<int64_t>(n) * c.size;
  }
}

// cooperative byte copy by the CTA.  The destination is written with aligned 16-byte stores; the source is read with
// aligned 16-byte loads when it is congruent to the destination mod 16, else as aligned 32-bit words funnel-shifted
// into place (the buffers of a Kudo partition have no alignment guarantees: KudoSerializer.java:157-159).
__device__ void cta_copy_bytes(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, int64_t n)
{
  const int tid = threadIdx.x, nt = blockDim.x;
  if (n <= 0) return;
  const uintptr_t da = reinterpret_cast<uintptr_t>(dst);
  const int64_t head = tmin<int64_t>(n, (16 - (da & 15)) & 15);
  for (int64_t i = tid; i < head; i += nt) dst[i] = src[i];
  const uintptr_t sa = reinterpret_cast<uintptr_t>(src + head);
  int64_t body       = (n - head) >> 4;
  uint4* d16         = reinterpret_cast<uint4*>(dst + head);
  if ((sa & 15) == 0) {
    const uint4* s16 = reinterpret_cast<const uint4*>(src + head);
    for (int64_t i = tid; i < body; i += nt) d16[i] = s16[i];
  } else {
    if (body > 0) --body;   // the last chunk's fifth word could lie past the source: it goes with the tail bytes
    const uint32_t* sw = reinterpret_cast<const uint32_t*>(sa & ~uintptr_t{3});
    const uint32_t sh  = static_cast<uint32_t>(sa & 3) * 8u;
    for (int64_t i = tid; i < body; i += nt) {
      const uint32_t* w = sw + 4 * i;
      const uint32_t w0 = w[0], w1 = w[1], w2 = w[2], w3 = w[3], w4 = w[4];
      d16[i] = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh));
    }
  }
  for (int64_t i = head + body * 16 + tid; i < n; i += nt) dst[i] = src[i];
}

// ---- split ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) kudo_split_sizes_kernel(const KCol* __restrict__ cols, int ncols, const int32_t* __restrict__ splits, int P,
                                                              int64_t* __restrict__ part_sizes, int32_t* __restrict__ bad)
{
  const int p = blockIdx.x * 256 + threadIdx.x;
  if (p >= P) return;
  const int32_t s = splits[p], n = splits[p + 1] - s;
  int64_t V = 0, O = 0, D = 0;
  for (int c = 0; c < ncols; ++c) {
    int64_t v, o, d;
    kudo_col_sizes(cols[c], s, n, v, o, d);
    V += v;
    O += o;
    D += d;
  }
  const int hs  = kudo_header_bytes(ncols);
  part_sizes[p] = pad4(hs + V) + pad4(O) + pad4(D);
  // the header holds the section lengths as 32-bit integers (KudoTableHeaderCalc.java:70-77: toIntExact)
  if (n < 0 || pad4(hs + V) - hs + pad4(O) + pad4(D) > INT32_MAX) atomicExch(bad, 1);
}

// exclusive scan of n values by one CTA of 1024 threads (n <= a few 10^4): put(i, sum of get(0 .. i - 1)) for i <= n
template <class Get, class Put>
__device__ void cta_exclusive_scan(int n, Get get, Put put)
{
  __shared__ int64_t s_warp[32];
  __shared__ int64_t s_carry;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  const int lane = lane_id(), w = warp_id();
  for (int b = 0; b < n + 1; b += 1024) {
    const int i     = b + threadIdx.x;
    const int64_t x = i < n ? get(i) : 0;
    int64_t inc     = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t y = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += y;
    }
    if (lane == 31) s_warp[w] = inc;
    __syncthreads();
    if (w == 0) {
      int64_t t = s_warp[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int64_t y = __shfl_up_sync(0xffffffffu, t, o);
        if (lane >= o) t += y;
      }
      s_warp[lane] = t;
    }
    __syncthreads();
    const int64_t base = s_carry + (w > 0 ? s_warp[w - 1] : 0);
    if (i <= n) put(i, base + inc - x);
    __syncthreads();
    if (threadIdx.x == 0) s_carry += s_warp[31];
    __syncthreads();
  }
}

// exclusive scan of P + 1 int64 in place by one CTA; element P receives the total
__global__ void __launch_bounds__(1024) i64_scan_small_kernel(int64_t* v, int n)
{
  cta_exclusive_scan(n, [&](int i) { return v[i]; }, [&](int i, int64_t x) { v[i] = x; });
}

__global__ void __launch_bounds__(256) kudo_split_kernel(const KCol* __restrict__ cols, int ncols, const int32_t* __restrict__ splits,
                                                        const int64_t* __restrict__ part_offsets, uint8_t* __restrict__ out)
{
  const int c = blockIdx.x, p = blockIdx.y;
  const int32_t s = splits[p], n = splits[p + 1] - s;
  const int hs   = kudo_header_bytes(ncols);
  uint8_t* part  = out + part_offsets[p];
  // where this column's buffers go: the sizes of the columns before it (and, for the section starts, of all columns)
  __shared__ int64_t s_pos[6];   // V, O, D before column c; V, O, D of the partition
  if (threadIdx.x == 0) {
    int64_t bv = 0, bo = 0, bd = 0, V = 0, O = 0, D = 0;
    for (int k = 0; k < ncols; ++k) {
      int64_t v, o, d;
      kudo_col_sizes(cols[k], s, n, v, o, d);
      if (k < c) { bv += v; bo += o; bd += d; }
      V += v; O += o; D += d;
    }
    s_pos[0] = bv; s_pos[1] = bo; s_pos[2] = bd; s_pos[3] = V; s_pos[4] = O; s_pos[5] = D;
  }
  __syncthreads();
  const int64_t V = s_pos[3], O = s_pos[4], D = s_pos[5];
  const int64_t vlen = pad4(hs + V) - hs, olen = pad4(O), dlen = pad4(D);
  uint8_t* v_at = part + hs;
  uint8_t* o_at = v_at + vlen;
  uint8_t* d_at = o_at + olen;
  if (c == 0) {
    // header (big endian), hasValidity bits, and the zero padding of the three sections
    if (threadIdx.x < 7) {
      const uint32_t f[7] = {kKudoMagic, static_cast<uint32_t>(s), static_cast<uint32_t>(n), static_cast<uint32_t>(vlen), static_cast<uint32_t>(olen),
                             static_cast<uint32_t>(vlen + olen + dlen), static_cast<uint32_t>(ncols)};
      reinterpret_cast<uint32_t*>(part)[threadIdx.x] = bswap32(f[threadIdx.x]);   // partitions start 4-byte aligned
    }
    for (int b = threadIdx.x; b < (ncols + 7) / 8; b += 256) {
      uint32_t bits = 0;
      for (int k = 8 * b; k < tmin(ncols, 8 * b + 8); ++k) bits |= (cols[k].mask && n > 0 ? 1u : 0u) << (k - 8 * b);
      part[28 + b] = static_cast<uint8_t>(bits);
    }
    if (threadIdx.x < 12) {
      const int sec     = threadIdx.x / 4, k = threadIdx.x % 4;
      uint8_t* end      = sec == 0 ? v_at + V : sec == 1 ? o_at + O : d_at + D;
      const int64_t pad = sec == 0 ? vlen - V : sec == 1 ? olen - O : dlen - D;
      if (k < pad) end[k] = 0;
    }
  }
  const KCol col = cols[c];
  int64_t v, o, d;
  kudo_col_sizes(col, s, n, v, o, d);
  if (v) cta_copy_bytes(v_at + s_pos[0], col.mask + s / 8, v);
  if (o) cta_copy_bytes(o_at + s_pos[1], reinterpret_cast<const uint8_t*>(col.offsets + s), o);
  if (d) cta_copy_bytes(d_at + s_pos[2], col.size ? col.data + static_cast<int64_t>(s) * col.size : col.data + col.offsets[s], d);
}

// ---- assemble ------------------------------------------------------------------------------------------------------------
struct KPartInfo {   // per partition, parsed from its header
  int32_t row_offset, rows, vlen, olen;
};

struct KRec {        // per (flattened column, partition)
  int32_t off, rows;    // the column's slice in this partition
  int32_t v, o, d;      // where its validity / offsets / data bytes start inside the three sections
  int32_t has_v;        // validity bytes present
  int64_t row_base;     // rows of the column in the partitions before this one
  int64_t char_base;    // STRING: chars of the partition, then (scanned) chars before it
};

__device__ __forceinline__ uint32_t ld_be32(const uint8_t* p) { return (uint32_t{p[0]} << 24) | (uint32_t{p[1]} << 16) | (uint32_t{p[2]} << 8) | p[3]; }
__device__ __forceinline__ int32_t ld_le32(const uint8_t* p) { return static_cast<int32_t>(uint32_t{p[0]} | (uint32_t{p[1]} << 8) | (uint32_t{p[2]} << 16) | (uint32_t{p[3]} << 24)); }

// thread per partition: checks the header, walks the flattened schema in pre-order and fills rec[c * P + p].  The bytes
// arrive over the network, so every section must lie inside [offs[p], offs[p + 1]) and every offsets pair read must
// satisfy 0 <= off[0] <= off[n]; otherwise *bad is set and the partition contributes no rows.
__global__ void __launch_bounds__(256) kudo_parse_kernel(const uint8_t* __restrict__ buf, const int64_t* __restrict__ part_offsets, int P, int F,
                                                        const KCol* __restrict__ cols, KPartInfo* __restrict__ info, KRec* __restrict__ rec,
                                                        int32_t* __restrict__ bad)
{
  const int p = blockIdx.x * 256 + threadIdx.x;
  if (p >= P) return;
  const int64_t plen = part_offsets[p + 1] - part_offsets[p];
  const int hs       = kudo_header_bytes(F);
  const uint8_t* h   = buf + part_offsets[p];
  KPartInfo pi{0, 0, 0, 0};
  bool ok = plen >= hs;
  int64_t dlen = 0;
  if (ok) {
    pi = KPartInfo{static_cast<int32_t>(ld_be32(h + 4)), static_cast<int32_t>(ld_be32(h + 8)), static_cast<int32_t>(ld_be32(h + 12)),
                   static_cast<int32_t>(ld_be32(h + 16))};
    const int32_t total = static_cast<int32_t>(ld_be32(h + 20));
    dlen = static_cast<int64_t>(total) - pi.vlen - pi.olen;
    ok = ld_be32(h) == kKudoMagic && static_cast<int>(ld_be32(h + 24)) == F && pi.rows >= 0 && pi.row_offset >= 0 && pi.vlen >= 0 &&
         pi.olen >= 0 && dlen >= 0 && hs + static_cast<int64_t>(total) <= plen;
  }
  const uint8_t* os = h + hs + (ok ? pi.vlen : 0);
  int64_t v = 0, o = 0, d = 0;
  for (int c = 0; ok && c < F; ++c) {
    const KCol col = cols[c];
    KRec r{};
    if (col.parent < 0) {
      r.off = pi.row_offset;
      r.rows = pi.rows;
    } else {
      const KRec& from = rec[static_cast<int64_t>(cols[col.parent].kind == KK_STRUCT ? col.parent : c) * P + p];   // below a LIST: set by the list
      r.off = from.off;
      r.rows = from.rows;
    }
    const int32_t s = r.off, n = r.rows;
    r.has_v = n > 0 && ((h[28 + c / 8] >> (c % 8)) & 1);
    r.v = static_cast<int32_t>(v);
    r.o = static_cast<int32_t>(o);
    r.d = static_cast<int32_t>(d);
    if (r.has_v) v += (static_cast<int64_t>(s) + n - 1) / 8 - s / 8 + 1;
    if (col.kind == KK_STRING || col.kind == KK_LIST) {
      int32_t a = 0, b = 0;
      if (n > 0) {
        const int64_t ob = 4 * (static_cast<int64_t>(n) + 1);
        if (o + ob > pi.olen) { ok = false; break; }
        a = ld_le32(os + o);
        b = ld_le32(os + o + 4 * static_cast<int64_t>(n));
        if (a < 0 || b < a) { ok = false; break; }
        o += ob;
      }
      if (col.kind == KK_LIST) {
        KRec& child = rec[static_cast<int64_t>(c + 1) * P + p];   // pre-order: a LIST's only child follows it
        child.off   = a;
        child.rows  = b - a;
      } else {
        r.char_base = b - a;
        d += b - a;
      }
    } else if (col.kind == KK_FIXED) {
      d += static_cast<int64_t>(n) * col.size;
    }
    if (v > pi.vlen || d > dlen) { ok = false; break; }
    rec[static_cast<int64_t>(c) * P + p] = r;
  }
  if (!ok) {
    atomicExch(bad, 1);
    pi.rows = 0;
    for (int c = 0; c < F; ++c) rec[static_cast<int64_t>(c) * P + p] = KRec{};
  }
  info[p] = pi;
}

// CTA per flattened column: row_base / char_base of every partition (exclusive scans); totals[2c] = rows, [2c + 1] = chars
__global__ void __launch_bounds__(1024) kudo_scan_kernel(KRec* __restrict__ rec, int P, int64_t* __restrict__ totals)
{
  const int c = blockIdx.x;
  KRec* r     = rec + static_cast<int64_t>(c) * P;
  cta_exclusive_scan(P, [&](int i) { return static_cast<int64_t>(r[i].rows); },
                     [&](int i, int64_t x) { if (i < P) r[i].row_base = x; else totals[2 * c] = x; });
  cta_exclusive_scan(P, [&](int i) { return r[i].char_base; },
                     [&](int i, int64_t x) { if (i < P) r[i].char_base = x; else totals[2 * c + 1] = x; });
}

// 5 CTAs per SM (<= 51 registers, no spills): the copy is bound by loads in flight, and the unconstrained build's 62
// registers would leave 4
__global__ void __launch_bounds__(256, 5) kudo_assemble_kernel(const uint8_t* __restrict__ buf, const int64_t* __restrict__ part_offsets, int P, int F,
                                                           const KCol* __restrict__ out, const KPartInfo* __restrict__ info, const KRec* __restrict__ rec)
{
  const int c = blockIdx.x, p = blockIdx.y;
  const KRec r = rec[static_cast<int64_t>(c) * P + p];
  const int n  = r.rows;
  if (n == 0) return;
  const KPartInfo pi  = info[p];
  const uint8_t* vs   = buf + part_offsets[p] + kudo_header_bytes(F);
  const uint8_t* os   = vs + pi.vlen;
  const uint8_t* ds   = os + pi.olen;
  const KCol col      = out[c];
  const int64_t rb    = r.row_base;
  // ---- validity: output bits [rb, rb + n) <- input bits [off % 8, ... ) of the slice's bytes, or ones ----
  if (col.mask) {
    const uint8_t* vb   = vs + r.v;
    const int shift     = r.off & 7;
    uint32_t* om        = reinterpret_cast<uint32_t*>(col.mask);
    const int64_t w0    = rb >> 5, w1 = (rb + n - 1) >> 5;
    for (int64_t w = w0 + threadIdx.x; w <= w1; w += 256) {
      const int64_t r_lo = tmax<int64_t>(rb, w << 5), r_hi = tmin<int64_t>(rb + n, (w + 1) << 5);   // rows of this word
      uint32_t bits = 0;
      if (r.has_v) {
        const int64_t i0 = r_lo - rb + shift;   // first input bit
        uint64_t acc     = 0;
        const int64_t nbytes = ((i0 & 7) + (r_hi - r_lo) + 7) >> 3;   // <= 5
        for (int64_t b = 0; b < nbytes; ++b) acc |= static_cast<uint64_t>(vb[(i0 >> 3) + b]) << (8 * b);
        bits = static_cast<uint32_t>(acc >> (i0 & 7));
      } else {
        bits = 0xffffffffu;
      }
      const int cnt = static_cast<int>(r_hi - r_lo);
      if (cnt < 32) bits &= (1u << cnt) - 1u;
      bits <<= (r_lo & 31);
      if (bits) atomicOr(om + w, bits);
    }
  }
  // ---- offsets (rebased onto the child's rows or the chars before the partition) + chars, or fixed-width data ----
  if (col.kind == KK_STRING || col.kind == KK_LIST) {
    const uint8_t* ob  = os + r.o;
    const int64_t base = col.kind == KK_LIST ? rec[static_cast<int64_t>(c + 1) * P + p].row_base : r.char_base;
    const int32_t o0   = ld_le32(ob);
    for (int i = threadIdx.x; i <= n; i += 256) col.offsets[rb + i] = static_cast<int32_t>(base + (ld_le32(ob + 4 * static_cast<int64_t>(i)) - o0));
    if (col.kind == KK_STRING) cta_copy_bytes(col.data + base, ds + r.d, ld_le32(ob + 4 * static_cast<int64_t>(n)) - o0);
  } else if (col.kind == KK_FIXED) {
    cta_copy_bytes(col.data + rb * col.size, ds + r.d, static_cast<int64_t>(n) * col.size);
  }
}

// ---- host side -------------------------------------------------------------------------------------------------------------
static int kudo_elem_size(int32_t t)
{
  switch (t) {
    case SRJ_INT8: case SRJ_UINT8: case SRJ_BOOL8: return 1;
    case SRJ_INT16: case SRJ_UINT16: return 2;
    case SRJ_INT32: case SRJ_UINT32: case SRJ_FLOAT32: case SRJ_TIMESTAMP_DAYS: case SRJ_DURATION_DAYS: case SRJ_DECIMAL32: return 4;
    case SRJ_INT64: case SRJ_UINT64: case SRJ_FLOAT64: case SRJ_TIMESTAMP_SECONDS: case SRJ_TIMESTAMP_MILLISECONDS:
    case SRJ_TIMESTAMP_MICROSECONDS: case SRJ_TIMESTAMP_NANOSECONDS: case SRJ_DURATION_SECONDS: case SRJ_DURATION_MILLISECONDS:
    case SRJ_DURATION_MICROSECONDS: case SRJ_DURATION_NANOSECONDS: case SRJ_DECIMAL64: return 8;
    case SRJ_DECIMAL128: return 16;
    case SRJ_STRING: return 0;
    default: return -1;
  }
}

// workspace: [KCol x 256 | bad flag (64 B) | totals int64 x 2 x 256 | KPartInfo x P | KRec x F x P]
struct KudoWs {
  KCol* cols;
  int32_t* bad;
  int64_t* totals;
  KPartInfo* info;
  KRec* rec;
};
static KudoWs kudo_ws(void* workspace, int P)
{
  uint8_t* w = static_cast<uint8_t*>(workspace);
  KudoWs k;
  k.cols = reinterpret_cast<KCol*>(w);
  w += kKudoMaxCols * sizeof(KCol);
  k.bad = reinterpret_cast<int32_t*>(w);
  w += 64;
  k.totals = reinterpret_cast<int64_t*>(w);
  w += 2 * kKudoMaxCols * 8;
  k.info = reinterpret_cast<KPartInfo*>(w);
  w += (static_cast<size_t>(P) * sizeof(KPartInfo) + 63) & ~size_t{63};
  k.rec = reinterpret_cast<KRec*>(w);
  return k;
}
int64_t kudo_workspace_bytes(int32_t ncols, int32_t P)
{
  return static_cast<int64_t>(kKudoMaxCols) * (sizeof(KCol) + 16) + 64 + static_cast<int64_t>(P) * sizeof(KPartInfo) + 64 +
         static_cast<int64_t>(std::max(ncols, 1)) * P * sizeof(KRec) + 256;
}

static int kudo_upload(const srj_column* cols, int32_t ncols, const KudoWs& ws, cudaStream_t stream)
{
  if (ncols <= 0 || ncols > kKudoMaxCols) return SRJ_EUNSUPPORTED;
  KCol h[kKudoMaxCols];
  for (int c = 0; c < ncols; ++c) {
    const int sz = kudo_elem_size(cols[c].type_id);
    if (sz < 0) return SRJ_EUNSUPPORTED;
    h[c] = KCol{static_cast<uint8_t*>(cols[c].data), reinterpret_cast<uint8_t*>(cols[c].null_mask), cols[c].offsets, sz,
                sz == 0 ? KK_STRING : KK_FIXED, -1, 0};
  }
  SRJ_CUDA_TRY(cudaMemcpyAsync(ws.cols, h, sizeof(KCol) * ncols, cudaMemcpyHostToDevice, stream));
  return SRJ_OK;
}

int launch_kudo_split_sizes(const srj_column* cols, int32_t ncols, const int32_t* d_splits, int32_t P, int64_t* d_part_offsets, int64_t* h_total,
                            void* workspace, cudaStream_t stream)
{
  const KudoWs ws = kudo_ws(workspace, P);
  const int rc = kudo_upload(cols, ncols, ws, stream);
  if (rc != SRJ_OK) return rc;
  SRJ_CUDA_TRY(cudaMemsetAsync(ws.bad, 0, 4, stream));
  kudo_split_sizes_kernel<<<(P + 255) / 256, 256, 0, stream>>>(ws.cols, ncols, d_splits, P, d_part_offsets, ws.bad);
  i64_scan_small_kernel<<<1, 1024, 0, stream>>>(d_part_offsets, P);
  SRJ_CUDA_TRY(cudaGetLastError());
  int32_t bad = 0;
  SRJ_CUDA_TRY(cudaMemcpyAsync(h_total, d_part_offsets + P, 8, cudaMemcpyDeviceToHost, stream));
  SRJ_CUDA_TRY(cudaMemcpyAsync(&bad, ws.bad, 4, cudaMemcpyDeviceToHost, stream));
  SRJ_CUDA_TRY(cudaStreamSynchronize(stream));
  return bad ? SRJ_EOVERFLOW : SRJ_OK;
}

int launch_kudo_split(const srj_column* cols, int32_t ncols, const int32_t* d_splits, int32_t P, const int64_t* d_part_offsets, uint8_t* out,
                      void* workspace, cudaStream_t stream)
{
  const KudoWs ws = kudo_ws(workspace, P);
  const int rc = kudo_upload(cols, ncols, ws, stream);
  if (rc != SRJ_OK) return rc;
  kudo_split_kernel<<<dim3(ncols, P), 256, 0, stream>>>(ws.cols, ncols, d_splits, d_part_offsets, out);
  SRJ_CUDA_TRY(cudaGetLastError());
  return SRJ_OK;
}

// the flattened schema -> kind / size / parent of every column; SRJ_EINVAL when the child counts do not describe a
// forest of `F` columns or a LIST has other than one child, SRJ_EUNSUPPORTED for a type outside the format
static int kudo_schema(const int32_t* type_ids, const int32_t* num_children, int F, KCol* h)
{
  if (F <= 0) return SRJ_EINVAL;
  if (F > kKudoMaxCols) return SRJ_EUNSUPPORTED;
  int stack[kKudoMaxCols], left[kKudoMaxCols], depth = 0;
  for (int c = 0; c < F; ++c) {
    while (depth > 0 && left[depth - 1] == 0) --depth;
    h[c] = KCol{nullptr, nullptr, nullptr, 0, KK_FIXED, depth > 0 ? stack[depth - 1] : -1, 0};
    if (depth > 0) --left[depth - 1];
    const int32_t t = type_ids[c], k = num_children[c];
    if (t == SRJ_LIST || t == SRJ_STRUCT) {
      if (k < 0 || (t == SRJ_LIST && k != 1)) return SRJ_EINVAL;
      h[c].kind   = t == SRJ_LIST ? KK_LIST : KK_STRUCT;
      stack[depth] = c;
      left[depth++] = k;
    } else {
      const int sz = kudo_elem_size(t);
      if (sz < 0) return SRJ_EUNSUPPORTED;
      if (k != 0) return SRJ_EINVAL;
      h[c].size = sz;
      h[c].kind = sz == 0 ? KK_STRING : KK_FIXED;
    }
  }
  while (depth > 0 && left[depth - 1] == 0) --depth;
  return depth == 0 ? SRJ_OK : SRJ_EINVAL;
}

int launch_kudo_assemble_nested_sizes(const uint8_t* buf, const int64_t* d_part_offsets, int32_t P, const int32_t* type_ids, const int32_t* num_children,
                                      int32_t F, int64_t* h_rows, int64_t* h_char_totals, void* workspace, cudaStream_t stream)
{
  const KudoWs ws = kudo_ws(workspace, P);
  KCol h[kKudoMaxCols];
  const int rc = kudo_schema(type_ids, num_children, F, h);
  if (rc != SRJ_OK) return rc;
  SRJ_CUDA_TRY(cudaMemcpyAsync(ws.cols, h, sizeof(KCol) * F, cudaMemcpyHostToDevice, stream));
  SRJ_CUDA_TRY(cudaMemsetAsync(ws.bad, 0, 4, stream));
  if (P > 0) kudo_parse_kernel<<<(P + 255) / 256, 256, 0, stream>>>(buf, d_part_offsets, P, F, ws.cols, ws.info, ws.rec, ws.bad);
  kudo_scan_kernel<<<F, 1024, 0, stream>>>(ws.rec, P, ws.totals);
  SRJ_CUDA_TRY(cudaGetLastError());
  int32_t bad = 0;
  std::vector<int64_t> totals(2 * static_cast<size_t>(F));
  SRJ_CUDA_TRY(cudaMemcpyAsync(&bad, ws.bad, 4, cudaMemcpyDeviceToHost, stream));
  SRJ_CUDA_TRY(cudaMemcpyAsync(totals.data(), ws.totals, 16 * static_cast<size_t>(F), cudaMemcpyDeviceToHost, stream));
  SRJ_CUDA_TRY(cudaStreamSynchronize(stream));
  if (bad) return SRJ_EINVAL;
  bool over = false;
  for (int c = 0; c < F; ++c) {
    h_rows[c]        = totals[2 * c];
    h_char_totals[c] = totals[2 * c + 1];
    over |= h_rows[c] > INT32_MAX || h_char_totals[c] > INT32_MAX;   // int32 offsets / size_type rows
  }
  return over ? SRJ_EOVERFLOW : SRJ_OK;
}

// the srj_column trees in pre-order
static int kudo_flatten(const srj_column* cols, int32_t n, std::vector<const srj_column*>& flat)
{
  for (int32_t i = 0; i < n; ++i) {
    if (static_cast<int>(flat.size()) >= kKudoMaxCols) return SRJ_EUNSUPPORTED;
    flat.push_back(&cols[i]);
    const int32_t t = cols[i].type_id;
    if (t == SRJ_LIST || t == SRJ_STRUCT) {
      if (cols[i].num_children > 0 && !cols[i].children) return SRJ_EINVAL;
      const int rc = kudo_flatten(cols[i].children, cols[i].num_children, flat);
      if (rc != SRJ_OK) return rc;
    }
  }
  return SRJ_OK;
}

int launch_kudo_assemble_nested(const uint8_t* buf, const int64_t* d_part_offsets, int32_t P, const srj_column* out, int32_t ncols, void* workspace,
                                cudaStream_t stream)
{
  const KudoWs ws = kudo_ws(workspace, P);
  std::vector<const srj_column*> flat;
  int rc = kudo_flatten(out, ncols, flat);
  if (rc != SRJ_OK) return rc;
  const int F = static_cast<int>(flat.size());
  int32_t ids[kKudoMaxCols], nch[kKudoMaxCols];
  for (int c = 0; c < F; ++c) {
    ids[c] = flat[c]->type_id;
    nch[c] = (ids[c] == SRJ_LIST || ids[c] == SRJ_STRUCT) ? flat[c]->num_children : 0;
  }
  KCol h[kKudoMaxCols];
  rc = kudo_schema(ids, nch, F, h);
  if (rc != SRJ_OK) return rc;
  for (int c = 0; c < F; ++c) {
    const srj_column& o = *flat[c];
    h[c].data    = static_cast<uint8_t*>(o.data);
    h[c].mask    = reinterpret_cast<uint8_t*>(o.null_mask);
    h[c].offsets = o.offsets;
    if (o.null_mask && o.size > 0) SRJ_CUDA_TRY(cudaMemsetAsync(o.null_mask, 0, static_cast<size_t>((o.size + 31) / 32) * 4, stream));
    if (h[c].kind == KK_STRING || h[c].kind == KK_LIST) {
      if (!o.offsets) return SRJ_EINVAL;
      if (o.size == 0) SRJ_CUDA_TRY(cudaMemsetAsync(o.offsets, 0, 4, stream));
    }
  }
  SRJ_CUDA_TRY(cudaMemcpyAsync(ws.cols, h, sizeof(KCol) * F, cudaMemcpyHostToDevice, stream));
  if (P > 0) kudo_assemble_kernel<<<dim3(F, P), 256, 0, stream>>>(buf, d_part_offsets, P, F, ws.cols, ws.info, ws.rec);
  SRJ_CUDA_TRY(cudaGetLastError());
  return SRJ_OK;
}

// flat tables: a schema of leaves
int launch_kudo_assemble_sizes(const uint8_t* buf, const int64_t* d_part_offsets, int32_t P, const int32_t* type_ids, int32_t ncols, int64_t* h_rows,
                               int64_t* h_char_totals, void* workspace, cudaStream_t stream)
{
  if (ncols <= 0 || ncols > kKudoMaxCols) return SRJ_EUNSUPPORTED;
  for (int c = 0; c < ncols; ++c)
    if (kudo_elem_size(type_ids[c]) < 0) return SRJ_EUNSUPPORTED;
  const std::vector<int32_t> leaves(ncols, 0);
  std::vector<int64_t> rows(ncols);
  const int rc = launch_kudo_assemble_nested_sizes(buf, d_part_offsets, P, type_ids, leaves.data(), ncols, rows.data(), h_char_totals, workspace, stream);
  if (rc == SRJ_OK || rc == SRJ_EOVERFLOW) *h_rows = rows[0];
  return rc;
}

int launch_kudo_assemble(const uint8_t* buf, const int64_t* d_part_offsets, int32_t P, const srj_column* out, int32_t ncols, int64_t total_rows,
                         void* workspace, cudaStream_t stream)
{
  if (ncols <= 0 || ncols > kKudoMaxCols) return SRJ_EUNSUPPORTED;
  for (int c = 0; c < ncols; ++c)
    if (kudo_elem_size(out[c].type_id) < 0) return SRJ_EUNSUPPORTED;
  (void)total_rows;   // = out[c].size, checked by the caller
  return launch_kudo_assemble_nested(buf, d_part_offsets, P, out, ncols, workspace, stream);
}

}  // namespace srj
