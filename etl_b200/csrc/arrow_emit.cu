// arrow_emit.cu — columnar emitter (SURVEY §8f N2): the rows of ONE replicated-schema version of a decoded batch as
// Arrow-layout column buffers, built on the device from the cell plane.
//
// Replaces the per-row walk of the destinations' encoders — build_array_for_field / build_primitive_array /
// build_boolean_array / build_string_array / build_binary_array / build_uuid_array and the cell_to_* converters of
// crates/etl-destinations/src/iceberg/encoding.rs:61-330 (the DuckLake and BigQuery encoders walk the same
// Vec<TableRow>) — for the column types whose Arrow value is a function of the decoded cell alone:
//   Bool → Boolean (bit-packed) · I16/I32 → Int32 · I64/U32 → Int64 (:200-221) · F32 · F64 · Date → Date32 days (:257-262)
//   Time → Time64 µs (:270-275) · Timestamp / TimestampTz → Timestamp µs (:284-301) · Uuid → FixedSizeBinary(16) (:313-318)
//   String → Utf8 (int32 offsets) · Bytes → LargeBinary (int64 offsets) (:245-250).
// A cell of another variant in such a column becomes null, exactly as the converters return None.
// With ETL_ARROW_FORMATTED (etl_dec_arrow_emit_ex) two more column classes are built here:
//   Numeric → Utf8 holding PgNumeric::to_string() (cell_to_string, :349; the text comes from numeric_text.cuh)
//   Array of a non-json element kind → List<child> (build_list_array and its typed builders, :386-776), the child type
//   being the element's column type above (a numeric element → Utf8, formatted the same way).
// Json columns and json / jsonb arrays (serde_json text) stay ETL_ARROW_UNSUPPORTED: they stay on the shim's row path.
// Pure gather / scan / copy / format kernels over planes that are already in HBM: HBM-bound, no parsing.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include <string>
#include <type_traits>
#include <vector>

#include "etl_decode.h"
#include "numeric_text.cuh"

namespace {

constexpr int kSelThreads = 1024;

struct SelParams {
  const uint8_t* rec_kind; const uint8_t* rec_flags; const int32_t* rec_schema; const uint64_t* rec_cell_base;
  uint64_t n_records;
  int32_t schema; uint32_t row_kinds; uint32_t n_cols;
  uint32_t* blk;          // per-block counts → exclusive offsets
  uint64_t* row_cell0;    // out: first cell of the row's image, per selected row
  uint64_t* row_rec;      // out: record index per selected row
  unsigned long long* n_rows;
};
// which image of record r is a row of this batch? returns false or the cell offset of the image inside the record
__device__ __forceinline__ bool row_of(const SelParams& S, uint64_t r, uint64_t* cell0) {
  if (r >= S.n_records || S.rec_schema[r] != S.schema) return false;
  const uint32_t k = S.rec_kind[r], f = S.rec_flags[r];
  if (!(f & ETL_RF_EVENT)) return false;
  const uint64_t c0 = S.rec_cell_base[r];
  if (k == 'I' && (S.row_kinds & 1u)) { *cell0 = c0; return true; }
  if (k == 'U' && (S.row_kinds & 2u) && !(f & ETL_RF_NEW_PARTIAL)) {      // UpdatedTableRow::Full only: a partial row has holes
    *cell0 = S.rec_cell_base[r + 1] - S.n_cols;                           // the new image is the record's last n_cols cells
    return true;
  }
  if (k == 'D' && (S.row_kinds & 4u) && (f & ETL_RF_OLD_FULL)) { *cell0 = c0; return true; }
  return false;
}
__global__ void __launch_bounds__(kSelThreads) k_sel_count(SelParams S) {
  uint64_t c0;
  const int c = __syncthreads_count(row_of(S, (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, &c0));
  if (threadIdx.x == 0) S.blk[blockIdx.x] = (uint32_t)c;
}
__global__ void __launch_bounds__(kSelThreads) k_blk_scan(uint32_t* blk, uint32_t nb, unsigned long long* total) {
  __shared__ uint32_t sh[kSelThreads];
  const uint32_t per = (nb + blockDim.x - 1) / blockDim.x;
  const uint32_t lo = threadIdx.x * per, hi = min(lo + per, nb);
  uint32_t acc = 0;
  for (uint32_t i = lo; i < hi; i++) acc += blk[i];
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (uint32_t d = 1; d < blockDim.x; d <<= 1) {
    uint32_t v = sh[threadIdx.x];
    if (threadIdx.x >= d) v += sh[threadIdx.x - d];
    __syncthreads();
    sh[threadIdx.x] = v;
    __syncthreads();
  }
  uint32_t run = threadIdx.x ? sh[threadIdx.x - 1] : 0u;
  for (uint32_t i = lo; i < hi; i++) { const uint32_t c = blk[i]; blk[i] = run; run += c; }
  if (threadIdx.x == blockDim.x - 1) *total = sh[blockDim.x - 1];
}
__global__ void __launch_bounds__(kSelThreads) k_sel_scatter(SelParams S) {
  __shared__ uint32_t warp_cnt[kSelThreads / 32];
  const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint64_t c0 = 0;
  const bool sel = row_of(S, r, &c0);
  const unsigned bal = __ballot_sync(0xffffffffu, sel);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) warp_cnt[wid] = __popc(bal);
  __syncthreads();
  uint32_t before = 0;
  for (int k = 0; k < wid; k++) before += warp_cnt[k];
  if (sel) {
    const uint64_t at = (uint64_t)S.blk[blockIdx.x] + before + __popc(bal & ((1u << lane) - 1u));
    S.row_cell0[at] = c0; S.row_rec[at] = r;
  }
}

struct ColParams {
  const uint8_t* cell_tag; const uint64_t* cell_val; const uint32_t* cell_aux; const uint8_t* heap; const uint8_t* stream;
  const uint64_t* row_cell0; uint64_t n_rows; uint32_t col; uint32_t arrow_type;
  uint32_t* validity;     // one word per 32 rows
  void* values;           // fixed width
  uint32_t* lens;         // var width: byte length per row (→ scanned into offsets)
  uint32_t src_kind;      // ETL_K_* of the column: a Utf8 column is String- or (ETL_ARROW_FORMATTED) Numeric-backed
};
// iceberg/encoding.rs:200-318: value of a cell for the column's Arrow type, or "null"
__device__ __forceinline__ bool fixed_value(uint32_t at, uint32_t tag, uint64_t val, uint32_t aux, int64_t* out) {
  switch (at) {
    case ETL_ARROW_BOOLEAN: if (tag != ETL_CELL_BOOL) return false; *out = (int64_t)(val & 1u); return true;
    case ETL_ARROW_INT32: if (tag != ETL_CELL_I16 && tag != ETL_CELL_I32) return false; *out = (int64_t)val; return true;
    case ETL_ARROW_INT64: if (tag != ETL_CELL_I64 && tag != ETL_CELL_U32) return false; *out = tag == ETL_CELL_U32 ? (int64_t)(uint32_t)val : (int64_t)val; return true;
    case ETL_ARROW_FLOAT32: if (tag != ETL_CELL_F32) return false; *out = (int64_t)(uint32_t)val; return true;
    case ETL_ARROW_FLOAT64: if (tag != ETL_CELL_F64) return false; *out = (int64_t)val; return true;
    case ETL_ARROW_DATE32: if (tag != ETL_CELL_DATE) return false; *out = (int64_t)val; return true;
    case ETL_ARROW_TIME64_US: if (tag != ETL_CELL_TIME) return false; *out = (int64_t)val * 1000000ll + (int64_t)(aux / 1000u); return true;
    case ETL_ARROW_TIMESTAMP_US: if (tag != ETL_CELL_TIMESTAMP) return false; *out = (int64_t)val * 1000000ll + (int64_t)(aux / 1000u); return true;
    case ETL_ARROW_TIMESTAMPTZ_US: if (tag != ETL_CELL_TIMESTAMPTZ) return false; *out = (int64_t)val * 1000000ll + (int64_t)(aux / 1000u); return true;
    default: return false;
  }
}
// one thread per row of one column: value / length + the validity word of its warp
__global__ void __launch_bounds__(256) k_col_fixed(ColParams C) {
  const uint64_t row = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool valid = false;
  int64_t v = 0;
  uint32_t len = 0;
  if (row < C.n_rows) {
    const uint64_t cell = C.row_cell0[row] + C.col;
    const uint32_t tag = C.cell_tag[cell];
    const uint64_t val = C.cell_val[cell];
    const uint32_t aux = C.cell_aux[cell];
    switch (C.arrow_type) {
      case ETL_ARROW_UTF8:
        if (C.src_kind == ETL_K_NUMERIC) {
          valid = tag == ETL_CELL_NUMERIC;
          if (valid) len = etl::numeric_text_len(*reinterpret_cast<const etl_numeric_hdr*>(C.heap + val), aux,
                                                 reinterpret_cast<const int16_t*>(C.heap + val + sizeof(etl_numeric_hdr)));
        } else {
          valid = tag == ETL_CELL_STRING; len = valid ? aux : 0u;
        }
        break;
      case ETL_ARROW_LARGE_BINARY: valid = tag == ETL_CELL_BYTES; len = valid ? aux : 0u; break;
      case ETL_ARROW_UUID: valid = tag == ETL_CELL_UUID; break;
      default: valid = fixed_value(C.arrow_type, tag, val, aux, &v); break;
    }
    switch (C.arrow_type) {
      case ETL_ARROW_INT32: case ETL_ARROW_DATE32: case ETL_ARROW_FLOAT32: static_cast<int32_t*>(C.values)[row] = valid ? (int32_t)v : 0; break;
      case ETL_ARROW_INT64: case ETL_ARROW_FLOAT64: case ETL_ARROW_TIME64_US: case ETL_ARROW_TIMESTAMP_US: case ETL_ARROW_TIMESTAMPTZ_US:
        static_cast<int64_t*>(C.values)[row] = valid ? v : 0; break;
      case ETL_ARROW_UUID: {
        uint64_t a = 0, b = 0;
        if (valid) { const uint64_t* s = reinterpret_cast<const uint64_t*>(C.heap + val); a = s[0]; b = s[1]; }   // heap reservations are 8-byte aligned
        static_cast<uint64_t*>(C.values)[2 * row] = a; static_cast<uint64_t*>(C.values)[2 * row + 1] = b;
        break;
      }
      case ETL_ARROW_UTF8: case ETL_ARROW_LARGE_BINARY: C.lens[row] = len; break;
      default: break;
    }
  }
  const unsigned vb = __ballot_sync(0xffffffffu, valid);
  const unsigned bb = __ballot_sync(0xffffffffu, valid && v != 0);
  if ((threadIdx.x & 31) == 0 && (row >> 5) < ((C.n_rows + 31) >> 5)) {
    C.validity[row >> 5] = vb;
    if (C.arrow_type == ETL_ARROW_BOOLEAN) static_cast<uint32_t*>(C.values)[row >> 5] = bb;   // Boolean values are bit-packed too
  }
}
// exclusive scan of lens → int32 / int64 offsets (n + 1 entries): block sums, scan of the sums, final pass
__global__ void __launch_bounds__(1024) k_len_blocks(const uint32_t* lens, uint64_t n, unsigned long long* blk) {
  __shared__ unsigned long long sh[32];
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long v = i < n ? lens[i] : 0ull;
  for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < 32) {
    v = sh[threadIdx.x];
    for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
    if (threadIdx.x == 0) blk[blockIdx.x] = v;
  }
}
__global__ void __launch_bounds__(1024) k_blk_scan64(unsigned long long* blk, uint32_t nb, unsigned long long* total) {
  __shared__ unsigned long long sh[1024];
  const uint32_t per = (nb + blockDim.x - 1) / blockDim.x;
  const uint32_t lo = threadIdx.x * per, hi = min(lo + per, nb);
  unsigned long long acc = 0;
  for (uint32_t i = lo; i < hi; i++) acc += blk[i];
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (uint32_t d = 1; d < blockDim.x; d <<= 1) {
    unsigned long long v = sh[threadIdx.x];
    if (threadIdx.x >= d) v += sh[threadIdx.x - d];
    __syncthreads();
    sh[threadIdx.x] = v;
    __syncthreads();
  }
  unsigned long long run = threadIdx.x ? sh[threadIdx.x - 1] : 0ull;
  for (uint32_t i = lo; i < hi; i++) { const unsigned long long c = blk[i]; blk[i] = run; run += c; }
  if (threadIdx.x == blockDim.x - 1) *total = sh[blockDim.x - 1];
}
template <typename OffT>
__global__ void __launch_bounds__(1024) k_offsets(const uint32_t* lens, uint64_t n, const unsigned long long* blk, OffT* offs) {
  __shared__ unsigned long long sh[1024];
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned long long mine = i < n ? lens[i] : 0ull;
  sh[threadIdx.x] = mine;
  __syncthreads();
  for (uint32_t d = 1; d < blockDim.x; d <<= 1) {
    unsigned long long v = sh[threadIdx.x];
    if (threadIdx.x >= d) v += sh[threadIdx.x - d];
    __syncthreads();
    sh[threadIdx.x] = v;
    __syncthreads();
  }
  const unsigned long long excl = blk[blockIdx.x] + sh[threadIdx.x] - mine;
  if (i < n) offs[i] = (OffT)excl;
  if (i + 1 == n) offs[n] = (OffT)(excl + mine);
}
// warp per row: copy the row's bytes to their place in the column's data buffer (16 B per lane where aligned)
template <typename OffT>
__global__ void __launch_bounds__(256) k_gather(ColParams C, const OffT* offs, uint8_t* data) {
  const uint64_t row = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31;
  if (row >= C.n_rows) return;
  const uint64_t cell = C.row_cell0[row] + C.col;
  const uint32_t tag = C.cell_tag[cell];
  const bool str = C.arrow_type == ETL_ARROW_UTF8;
  if (tag != (str ? (uint32_t)ETL_CELL_STRING : (uint32_t)ETL_CELL_BYTES)) return;
  const uint8_t* src = (str ? C.stream : C.heap) + C.cell_val[cell];
  const uint32_t n = C.cell_aux[cell];
  uint8_t* dst = data + (uint64_t)offs[row];
  for (uint32_t i = lane; i < n; i += 32) dst[i] = src[i];
}
// warp per row of a Numeric column: PgNumeric::to_string() at the row's place, lane l taking digit groups l, l+32, …
__global__ void __launch_bounds__(256) k_numeric_text(ColParams C, const int32_t* offs, uint8_t* data) {
  const uint64_t row = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31;
  if (row >= C.n_rows) return;
  const uint64_t cell = C.row_cell0[row] + C.col;
  if (C.cell_tag[cell] != ETL_CELL_NUMERIC) return;
  const uint8_t* e = C.heap + C.cell_val[cell];
  etl::numeric_text_write(*reinterpret_cast<const etl_numeric_hdr*>(e), C.cell_aux[cell],
                          reinterpret_cast<const int16_t*>(e + sizeof(etl_numeric_hdr)), data + offs[row], lane, 32);
}

// ---- List columns (ETL_ARROW_FORMATTED): cell = etl_array_hdr + etl_array_elem[n] in the heap; element payloads
// (strings, numerics, bytes, uuids) are heap offsets too, unlike top-level string cells (stream offsets).
struct ListParams {
  const uint8_t* cell_tag; const uint64_t* cell_val; const uint8_t* heap;
  const uint64_t* row_cell0; uint64_t n_rows; uint32_t col; uint32_t child_type;
  uint32_t* validity;                  // list validity, one word per 32 rows (zeroed beforehand)
  uint32_t* n_elems;                   // pass 1: elements per row (→ int32 list offsets)
  uint32_t* child_lens;                // pass 1, Utf8 / LargeBinary child: child bytes per row (→ child_base)
  const int32_t* list_offs;            // pass 2
  const unsigned long long* child_base;// pass 2, var-width child: first child byte of each row, [n_rows] = total
  uint32_t* cvalid;                    // child validity (zeroed beforehand)
  void* cvalues;                       // fixed-width child values (Boolean: bit-packed, zeroed beforehand)
  void* coffs;                         // var-width child offsets (int32 Utf8, int64 LargeBinary)
  uint8_t* cdata;
  uint64_t n_values;
};
__device__ __forceinline__ const etl_array_elem* list_elems(const uint8_t* heap, uint64_t hdr_off, uint32_t* n) {
  *n = reinterpret_cast<const etl_array_hdr*>(heap + hdr_off)->n_elems;
  return reinterpret_cast<const etl_array_elem*>(heap + hdr_off + sizeof(etl_array_hdr));
}
// a var-width child element: valid? and its byte length (string / bytes as stored, numeric as formatted)
__device__ __forceinline__ bool elem_var_len(const uint8_t* heap, uint32_t child_type, const etl_array_elem& e, uint32_t* len) {
  if (child_type == ETL_ARROW_LARGE_BINARY) { *len = e.aux; return e.tag == ETL_CELL_BYTES; }
  if (e.tag == ETL_CELL_STRING) { *len = e.aux; return true; }
  if (e.tag == ETL_CELL_NUMERIC) {
    *len = etl::numeric_text_len(*reinterpret_cast<const etl_numeric_hdr*>(heap + e.val), e.aux,
                                 reinterpret_cast<const int16_t*>(heap + e.val + sizeof(etl_numeric_hdr)));
    return true;
  }
  *len = 0;
  return false;
}
__device__ __forceinline__ void elem_var_write(const uint8_t* heap, const etl_array_elem& e, uint8_t* dst, uint32_t len,
                                               uint32_t w, uint32_t n_w) {
  if (e.tag == ETL_CELL_NUMERIC) {
    etl::numeric_text_write(*reinterpret_cast<const etl_numeric_hdr*>(heap + e.val), e.aux,
                            reinterpret_cast<const int16_t*>(heap + e.val + sizeof(etl_numeric_hdr)), dst, w, n_w);
  } else {
    const uint8_t* src = heap + e.val;
    for (uint32_t i = w; i < len; i += n_w) dst[i] = src[i];
  }
}
// OR 32 bits that start at bit p of a bitmap: a row's element range is not 32-aligned, neighbours share words
__device__ __forceinline__ void or_bits(uint32_t* words, uint64_t p, unsigned bits) {
  if (!bits) return;
  const uint32_t sh = (uint32_t)(p & 31u);
  atomicOr(&words[p >> 5], bits << sh);
  if (sh && (bits >> (32u - sh))) atomicOr(&words[(p >> 5) + 1], bits >> (32u - sh));
}
// pass 1, warp per row: list validity, elements per row and, for var-width children, the row's child bytes
__global__ void __launch_bounds__(256) k_list_count(ListParams L) {
  const uint64_t row = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31;
  if (row >= L.n_rows) return;
  const uint64_t cell = L.row_cell0[row] + L.col;
  const bool valid = L.cell_tag[cell] == ETL_CELL_ARRAY;
  uint32_t n = 0;
  unsigned long long bytes = 0;
  if (valid) {
    const etl_array_elem* el = list_elems(L.heap, L.cell_val[cell], &n);
    if (L.child_lens) {
      for (uint32_t i = lane; i < n; i += 32) { uint32_t len; if (elem_var_len(L.heap, L.child_type, el[i], &len)) bytes += len; }
      for (int d = 16; d > 0; d >>= 1) bytes += __shfl_down_sync(0xffffffffu, bytes, d);
    }
  }
  if (lane == 0) {
    L.n_elems[row] = n;
    if (L.child_lens) L.child_lens[row] = (uint32_t)min(bytes, 0xFFFFFFFFull);   // saturates: the column is then refused as > 2 GiB
    if (valid) atomicOr(&L.validity[row >> 5], 1u << (row & 31));
  }
}
// pass 2, warp per row, 32 elements at a time: child validity, child values or child offsets + bytes
__global__ void __launch_bounds__(256) k_list_fill(ListParams L) {
  const uint64_t row = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31;
  if (row >= L.n_rows) return;
  const uint32_t ct = L.child_type;
  const bool var = ct == ETL_ARROW_UTF8 || ct == ETL_ARROW_LARGE_BINARY;
  if (var && lane == 0 && row + 1 == L.n_rows) {     // closing child offset
    if (ct == ETL_ARROW_UTF8) static_cast<int32_t*>(L.coffs)[L.n_values] = (int32_t)L.child_base[L.n_rows];
    else static_cast<int64_t*>(L.coffs)[L.n_values] = (int64_t)L.child_base[L.n_rows];
  }
  const uint64_t cell = L.row_cell0[row] + L.col;
  if (L.cell_tag[cell] != ETL_CELL_ARRAY) return;
  uint32_t n;
  const etl_array_elem* el = list_elems(L.heap, L.cell_val[cell], &n);
  const uint64_t o = (uint64_t)(uint32_t)L.list_offs[row];
  unsigned long long run = var ? L.child_base[row] : 0ull;
  for (uint32_t b = 0; b < n; b += 32) {
    const uint32_t i = b + lane;
    const bool in = i < n;
    etl_array_elem e;
    e.val = 0; e.aux = 0; e.tag = ETL_CELL_NULL;
    if (in) e = el[i];
    bool valid = false;
    int64_t v = 0;
    uint32_t len = 0;
    if (in) {
      if (var) valid = elem_var_len(L.heap, ct, e, &len);
      else if (ct == ETL_ARROW_UUID) valid = e.tag == ETL_CELL_UUID;
      else valid = fixed_value(ct, e.tag, e.val, e.aux, &v);
    }
    const unsigned vb = __ballot_sync(0xffffffffu, valid);
    const unsigned bb = __ballot_sync(0xffffffffu, valid && v != 0);
    if (lane == 0) {
      or_bits(L.cvalid, o + b, vb);
      if (ct == ETL_ARROW_BOOLEAN) or_bits(static_cast<uint32_t*>(L.cvalues), o + b, bb);
    }
    if (!var) {
      if (in) {
        switch (ct) {
          case ETL_ARROW_INT32: case ETL_ARROW_DATE32: case ETL_ARROW_FLOAT32: static_cast<int32_t*>(L.cvalues)[o + i] = valid ? (int32_t)v : 0; break;
          case ETL_ARROW_INT64: case ETL_ARROW_FLOAT64: case ETL_ARROW_TIME64_US: case ETL_ARROW_TIMESTAMP_US: case ETL_ARROW_TIMESTAMPTZ_US:
            static_cast<int64_t*>(L.cvalues)[o + i] = valid ? v : 0; break;
          case ETL_ARROW_UUID: {
            uint64_t a = 0, c = 0;
            if (valid) { const uint64_t* s = reinterpret_cast<const uint64_t*>(L.heap + e.val); a = s[0]; c = s[1]; }
            static_cast<uint64_t*>(L.cvalues)[2 * (o + i)] = a; static_cast<uint64_t*>(L.cvalues)[2 * (o + i) + 1] = c;
            break;
          }
          default: break;
        }
      }
      continue;
    }
    // var-width child: warp exclusive scan of the lengths → offsets, then the bytes
    uint32_t incl = len;
    for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= (uint32_t)d) incl += t; }
    const unsigned long long at = run + incl - len;
    run += __shfl_sync(0xffffffffu, incl, 31);
    if (in) {
      if (ct == ETL_ARROW_UTF8) static_cast<int32_t*>(L.coffs)[o + i] = (int32_t)at;
      else static_cast<int64_t*>(L.coffs)[o + i] = (int64_t)at;
    }
    const bool longv = valid && len > 64;              // short values: one lane each; long ones: the whole warp
    if (valid && !longv) elem_var_write(L.heap, e, L.cdata + at, len, 0, 1);
    for (unsigned lb = __ballot_sync(0xffffffffu, longv); lb; lb &= lb - 1) {
      const int src = __ffs(lb) - 1;
      etl_array_elem f;
      f.val = __shfl_sync(0xffffffffu, e.val, src); f.aux = __shfl_sync(0xffffffffu, e.aux, src);
      f.tag = (uint8_t)__shfl_sync(0xffffffffu, (uint32_t)e.tag, src);
      const unsigned long long fat = __shfl_sync(0xffffffffu, at, src);
      const uint32_t flen = __shfl_sync(0xffffffffu, len, src);
      elem_var_write(L.heap, f, L.cdata + fat, flen, lane, 32);
    }
  }
}

uint32_t arrow_type_of(uint32_t k) {
  switch (k) {
    case ETL_K_BOOL: return ETL_ARROW_BOOLEAN;
    case ETL_K_I16: case ETL_K_I32: return ETL_ARROW_INT32;
    case ETL_K_I64: case ETL_K_U32: return ETL_ARROW_INT64;
    case ETL_K_F32: return ETL_ARROW_FLOAT32;
    case ETL_K_F64: return ETL_ARROW_FLOAT64;
    case ETL_K_STRING: return ETL_ARROW_UTF8;
    case ETL_K_BYTES: return ETL_ARROW_LARGE_BINARY;
    case ETL_K_DATE: return ETL_ARROW_DATE32;
    case ETL_K_TIME: return ETL_ARROW_TIME64_US;
    case ETL_K_TIMESTAMP: return ETL_ARROW_TIMESTAMP_US;
    case ETL_K_TIMESTAMPTZ: return ETL_ARROW_TIMESTAMPTZ_US;
    case ETL_K_UUID: return ETL_ARROW_UUID;
    default: return ETL_ARROW_UNSUPPORTED;    // numeric / json / arrays: cell_to_string formatting stays with the shim
  }
}
// ETL_ARROW_FORMATTED also formats numerics and lays out arrays of a non-json element kind (iceberg/schema.rs:9-37)
uint32_t arrow_type_of(uint32_t k, uint32_t flags) {
  if (!(flags & ETL_ARROW_FORMATTED)) return arrow_type_of(k);
  if (k == ETL_K_NUMERIC) return ETL_ARROW_UTF8;
  if ((k & ETL_K_ARRAY) && (k & ~(uint32_t)ETL_K_ARRAY) != ETL_K_JSON)
    return arrow_type_of(k & ~(uint32_t)ETL_K_ARRAY, flags) == ETL_ARROW_UNSUPPORTED ? ETL_ARROW_UNSUPPORTED : ETL_ARROW_LIST;
  return arrow_type_of(k);
}
uint32_t value_width(uint32_t at) {
  switch (at) {
    case ETL_ARROW_INT32: case ETL_ARROW_DATE32: case ETL_ARROW_FLOAT32: return 4;
    case ETL_ARROW_INT64: case ETL_ARROW_FLOAT64: case ETL_ARROW_TIME64_US: case ETL_ARROW_TIMESTAMP_US: case ETL_ARROW_TIMESTAMPTZ_US: return 8;
    case ETL_ARROW_UUID: return 16;
    default: return 0;
  }
}
struct Col {
  uint32_t arrow_type = 0, src_kind = 0;
  uint64_t validity_off = 0, values_off = 0, offsets_off = 0, data_off = 0, data_bytes = 0, values_bytes = 0, offsets_bytes = 0;
  // List columns: the child column (validity / values / offsets + data over n_values elements)
  uint32_t child_type = 0;
  uint64_t n_values = 0, c_validity_off = 0, c_validity_bytes = 0, c_values_off = 0, c_values_bytes = 0, c_offsets_off = 0,
           c_offsets_bytes = 0, c_data_off = 0, c_data_bytes = 0;
};
bool var_width(uint32_t at) { return at == ETL_ARROW_UTF8 || at == ETL_ARROW_LARGE_BINARY; }

}  // namespace

struct etl_arrow_batch {
  uint64_t n_rows = 0;
  std::vector<Col> cols;
  uint8_t* dev = nullptr;     // one device allocation: row_rec | per column validity, values / offsets, data | list children
  uint8_t* host = nullptr;    // pinned host image (to_host)
  uint64_t bytes = 0, row_rec_off = 0;
  std::string error;
};

extern "C" {

int etl_dec_arrow_emit(const etl_dec_batch* batch, uint32_t schema_index, uint32_t row_kinds, int to_host, etl_arrow_batch** out) {
  return etl_dec_arrow_emit_ex(batch, schema_index, row_kinds, 0, to_host, out);
}

int etl_dec_arrow_emit_ex(const etl_dec_batch* batch, uint32_t schema_index, uint32_t row_kinds, uint32_t flags, int to_host,
                          etl_arrow_batch** out) {
  if (!batch || !out || (flags & ~(uint32_t)ETL_ARROW_FORMATTED)) return ETL_ERR_INVALID_ARG;
  const uint8_t* dev_stream = etl_dec_batch_device_stream(batch);
  etl_dec_planes P;
  etl_dec_summary S;
  etl_dec_schema_info sc;
  if (etl_dec_batch_planes(batch, 0, &P) != ETL_OK || etl_dec_batch_summary(batch, &S) != ETL_OK) return ETL_ERR_INVALID_ARG;
  if (etl_dec_batch_schema(batch, schema_index, &sc) != ETL_OK) return ETL_ERR_INVALID_ARG;
  cudaStream_t st = cudaStreamPerThread;
  etl_arrow_batch* A = new etl_arrow_batch();
  auto fail = [&](int rc) { if (A->dev) cudaFree(A->dev); if (A->host) cudaFreeHost(A->host); delete A; return rc; };
#define CKA(call) do { if ((call) != cudaSuccess) { cudaGetLastError(); return fail(ETL_ERR_CUDA); } } while (0)
  // rows of the valid prefix only
  const uint64_t n_valid = S.first_error.record_index == UINT64_MAX ? P.n_records : std::min<uint64_t>(P.n_records, S.first_error.record_index - S.record_index_base);
  const uint32_t nb = (uint32_t)((n_valid + kSelThreads - 1) / kSelThreads);
  uint32_t* d_blk = nullptr; uint64_t* d_cell0 = nullptr; uint64_t* d_rec = nullptr; unsigned long long* d_n = nullptr;
  CKA(cudaMalloc(&d_blk, (nb + 1) * 4ull)); CKA(cudaMalloc(&d_cell0, (n_valid + 1) * 8)); CKA(cudaMalloc(&d_rec, (n_valid + 1) * 8)); CKA(cudaMalloc(&d_n, 16));
  auto free_tmp = [&]() { cudaFree(d_blk); cudaFree(d_cell0); cudaFree(d_rec); cudaFree(d_n); };
  SelParams Sp{P.rec_kind, P.rec_flags, P.rec_schema, P.rec_cell_base, n_valid, (int32_t)schema_index, row_kinds, sc.n_cols, d_blk, d_cell0, d_rec, d_n};
  unsigned long long n_rows = 0;
  if (nb) {
    k_sel_count<<<nb, kSelThreads, 0, st>>>(Sp);
    k_blk_scan<<<1, kSelThreads, 0, st>>>(d_blk, nb, d_n);
    k_sel_scatter<<<nb, kSelThreads, 0, st>>>(Sp);
    if (cudaMemcpyAsync(&n_rows, d_n, 8, cudaMemcpyDeviceToHost, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess) { free_tmp(); return fail(ETL_ERR_CUDA); }
  }
  A->n_rows = n_rows;
  // pass 1: validity + fixed values + lengths (into a scratch), per column; var-width sizes need a sync before the data buffers exist
  const uint64_t vbytes = ((n_rows + 31) / 32 * 4 + 63) & ~63ull;
  uint64_t cur = ((n_rows * 8) + 63) & ~63ull;        // row_rec first
  A->row_rec_off = 0;
  A->cols.resize(sc.n_cols);
  uint32_t n_var = 0, n_list = 0;
  for (uint32_t c = 0; c < sc.n_cols; c++) {
    Col& col = A->cols[c];
    col.src_kind = sc.col_kind[c];
    col.arrow_type = arrow_type_of(sc.col_kind[c], flags);
    if (col.arrow_type == ETL_ARROW_UNSUPPORTED) continue;
    col.validity_off = cur; cur += vbytes;
    if (col.arrow_type == ETL_ARROW_BOOLEAN) { col.values_off = cur; col.values_bytes = vbytes; cur += vbytes; }
    else if (value_width(col.arrow_type)) { col.values_off = cur; col.values_bytes = (n_rows * value_width(col.arrow_type) + 63) & ~63ull; cur += col.values_bytes; }
    else if (col.arrow_type == ETL_ARROW_LIST) {
      col.child_type = arrow_type_of(col.src_kind & ~(uint32_t)ETL_K_ARRAY, flags);
      col.offsets_off = cur; col.offsets_bytes = ((n_rows + 1) * 4 + 63) & ~63ull; cur += col.offsets_bytes; n_list++;
    }
    else { col.offsets_off = cur; col.offsets_bytes = ((n_rows + 1) * (col.arrow_type == ETL_ARROW_UTF8 ? 4 : 8) + 63) & ~63ull; cur += col.offsets_bytes; n_var++; }
  }
  const uint64_t fixed_bytes = cur;
  // length slots: one per var-width column, then two per list column (elements per row, child bytes per row); the
  // scan totals of all of them come back in one copy
  const uint32_t n_slots = n_var + 2 * n_list;
  uint32_t* d_lens = nullptr; unsigned long long* d_lblk = nullptr; unsigned long long* d_tot = nullptr; unsigned long long* d_cbase = nullptr;
  uint8_t* d_fixed = nullptr;
  auto free_scratch = [&]() { free_tmp(); cudaFree(d_lens); cudaFree(d_lblk); cudaFree(d_tot); cudaFree(d_cbase); cudaFree(d_fixed); };
  const uint32_t lb = (uint32_t)((n_rows + 1023) / 1024);
  if (n_slots) { if (cudaMalloc(&d_lens, (size_t)n_slots * (n_rows + 1) * 4) != cudaSuccess || cudaMalloc(&d_lblk, (size_t)n_slots * (lb + 1) * 8) != cudaSuccess || cudaMalloc(&d_tot, n_slots * 8 + 8) != cudaSuccess) { free_scratch(); return fail(ETL_ERR_ALLOC); } }
  if (n_list && cudaMalloc(&d_cbase, (size_t)n_list * (n_rows + 1) * 8) != cudaSuccess) { free_scratch(); return fail(ETL_ERR_ALLOC); }
  if (cudaMalloc(&d_fixed, fixed_bytes + 64) != cudaSuccess) { free_scratch(); return fail(ETL_ERR_ALLOC); }
  cudaMemsetAsync(d_fixed, 0, fixed_bytes + 64, st);
  if (n_rows) cudaMemcpyAsync(d_fixed, d_rec, n_rows * 8, cudaMemcpyDeviceToDevice, st);
  std::vector<unsigned long long> totals(n_slots + 1, 0);
  // exclusive scan of a length slot into offsets, its total into d_tot[slot]
  auto scan = [&](uint32_t slot, auto* offs) {
    using OffT = typename std::remove_pointer<decltype(offs)>::type;
    const uint32_t* lens = d_lens + (size_t)slot * (n_rows + 1);
    unsigned long long* blk = d_lblk + (size_t)slot * (lb + 1);
    k_len_blocks<<<lb, 1024, 0, st>>>(lens, n_rows, blk);
    k_blk_scan64<<<1, 1024, 0, st>>>(blk, lb, d_tot + slot);
    k_offsets<OffT><<<lb, 1024, 0, st>>>(lens, n_rows, blk, offs);
  };
  auto list_params = [&](uint32_t c, const Col& col) {
    ListParams Lp{};
    Lp.cell_tag = P.cell_tag; Lp.cell_val = P.cell_val; Lp.heap = P.heap; Lp.row_cell0 = d_cell0; Lp.n_rows = n_rows; Lp.col = c;
    Lp.child_type = col.child_type;
    return Lp;
  };
  const uint32_t warp_grid = (uint32_t)((n_rows * 32 + 255) / 256);
  uint32_t vi = 0, li = 0;
  for (uint32_t c = 0; c < sc.n_cols && n_rows; c++) {
    Col& col = A->cols[c];
    if (col.arrow_type == ETL_ARROW_UNSUPPORTED) continue;
    if (col.arrow_type == ETL_ARROW_LIST) {
      const uint32_t slot = n_var + 2 * li;
      ListParams Lp = list_params(c, col);
      Lp.validity = (uint32_t*)(d_fixed + col.validity_off);
      Lp.n_elems = d_lens + (size_t)slot * (n_rows + 1);
      if (var_width(col.child_type)) Lp.child_lens = d_lens + (size_t)(slot + 1) * (n_rows + 1);
      k_list_count<<<warp_grid, 256, 0, st>>>(Lp);
      scan(slot, (int32_t*)(d_fixed + col.offsets_off));
      if (Lp.child_lens) scan(slot + 1, (int64_t*)(d_cbase + (size_t)li * (n_rows + 1)));
      li++;
      continue;
    }
    ColParams Cp{P.cell_tag, P.cell_val, P.cell_aux, P.heap, dev_stream, d_cell0, n_rows, c, col.arrow_type,
                 (uint32_t*)(d_fixed + col.validity_off), col.values_bytes ? (void*)(d_fixed + col.values_off) : nullptr, nullptr, col.src_kind};
    const bool var = var_width(col.arrow_type);
    if (var) Cp.lens = d_lens + (size_t)vi * (n_rows + 1);
    k_col_fixed<<<(uint32_t)((n_rows + 255) / 256), 256, 0, st>>>(Cp);
    if (var) {
      if (col.arrow_type == ETL_ARROW_UTF8) scan(vi, (int32_t*)(d_fixed + col.offsets_off));
      else scan(vi, (int64_t*)(d_fixed + col.offsets_off));
      vi++;
    }
  }
  if (n_slots && n_rows) cudaMemcpyAsync(totals.data(), d_tot, n_slots * 8, cudaMemcpyDeviceToHost, st);
  if (cudaStreamSynchronize(st) != cudaSuccess) { free_scratch(); return fail(ETL_ERR_CUDA); }
  // pass 2: data buffers and list children
  vi = 0; li = 0;
  for (uint32_t c = 0; c < sc.n_cols; c++) {
    Col& col = A->cols[c];
    if (col.arrow_type == ETL_ARROW_LIST) {
      const uint32_t slot = n_var + 2 * li++;
      const uint64_t nv = col.n_values = n_rows ? totals[slot] : 0;
      if (nv > 0x7FFFFFFFull) A->error = "List column has 2^31 or more values: split the batch";
      const uint64_t cvb = ((nv + 31) / 32 * 4 + 63) & ~63ull;
      col.c_validity_off = cur; col.c_validity_bytes = cvb; cur += cvb;
      if (col.child_type == ETL_ARROW_BOOLEAN) { col.c_values_off = cur; col.c_values_bytes = cvb; cur += cvb; }
      else if (value_width(col.child_type)) { col.c_values_off = cur; col.c_values_bytes = (nv * value_width(col.child_type) + 63) & ~63ull; cur += col.c_values_bytes; }
      else {
        col.c_offsets_off = cur; col.c_offsets_bytes = ((nv + 1) * (col.child_type == ETL_ARROW_UTF8 ? 4 : 8) + 63) & ~63ull; cur += col.c_offsets_bytes;
        col.c_data_off = cur; col.c_data_bytes = n_rows ? totals[slot + 1] : 0; cur += (col.c_data_bytes + 63) & ~63ull;
        if (col.child_type == ETL_ARROW_UTF8 && col.c_data_bytes > 0x7FFFFFFFull) A->error = "Utf8 list values exceed 2 GiB: split the batch";
      }
      continue;
    }
    if (!var_width(col.arrow_type)) continue;
    col.data_off = cur; col.data_bytes = n_rows ? totals[vi] : 0; cur += (col.data_bytes + 63) & ~63ull;
    if (col.arrow_type == ETL_ARROW_UTF8 && col.data_bytes > 0x7FFFFFFFull) { A->error = "Utf8 column exceeds 2 GiB: split the batch"; }
    vi++;
  }
  A->bytes = cur + 64;
  bool ok = A->error.empty() && cudaMalloc(&A->dev, A->bytes) == cudaSuccess;
  if (ok) ok = cudaMemcpyAsync(A->dev, d_fixed, fixed_bytes, cudaMemcpyDeviceToDevice, st) == cudaSuccess;
  li = 0;
  for (uint32_t c = 0; ok && c < sc.n_cols; c++) {
    Col& col = A->cols[c];
    if (col.arrow_type == ETL_ARROW_LIST) {
      // bitmaps are OR-ed into; with no rows nothing writes the closing child offset
      ok = cudaMemsetAsync(A->dev + col.c_validity_off, 0, n_rows ? col.c_validity_bytes + (col.child_type == ETL_ARROW_BOOLEAN ? col.c_values_bytes : 0)
                                                                   : A->bytes - col.c_validity_off, st) == cudaSuccess;
      if (ok && n_rows) {
        ListParams Lp = list_params(c, col);
        Lp.list_offs = (const int32_t*)(A->dev + col.offsets_off);
        Lp.child_base = d_cbase + (size_t)li * (n_rows + 1);
        Lp.cvalid = (uint32_t*)(A->dev + col.c_validity_off);
        Lp.cvalues = col.c_values_bytes ? (void*)(A->dev + col.c_values_off) : nullptr;
        Lp.coffs = col.c_offsets_bytes ? (void*)(A->dev + col.c_offsets_off) : nullptr;
        Lp.cdata = A->dev + col.c_data_off;
        Lp.n_values = col.n_values;
        k_list_fill<<<warp_grid, 256, 0, st>>>(Lp);
      }
      li++;
      continue;
    }
    if (!var_width(col.arrow_type) || !n_rows) continue;
    ColParams Cp{P.cell_tag, P.cell_val, P.cell_aux, P.heap, dev_stream, d_cell0, n_rows, c, col.arrow_type, nullptr, nullptr, nullptr, col.src_kind};
    if (col.src_kind == ETL_K_NUMERIC) k_numeric_text<<<warp_grid, 256, 0, st>>>(Cp, (const int32_t*)(A->dev + col.offsets_off), A->dev + col.data_off);
    else if (col.arrow_type == ETL_ARROW_UTF8) k_gather<int32_t><<<warp_grid, 256, 0, st>>>(Cp, (const int32_t*)(A->dev + col.offsets_off), A->dev + col.data_off);
    else k_gather<int64_t><<<warp_grid, 256, 0, st>>>(Cp, (const int64_t*)(A->dev + col.offsets_off), A->dev + col.data_off);
  }
  if (ok && to_host) {
    ok = cudaHostAlloc((void**)&A->host, A->bytes, cudaHostAllocDefault) == cudaSuccess;
    if (ok) ok = cudaMemcpyAsync(A->host, A->dev, A->bytes, cudaMemcpyDeviceToHost, st) == cudaSuccess;
  }
  if (ok) ok = cudaStreamSynchronize(st) == cudaSuccess && cudaGetLastError() == cudaSuccess;
  free_scratch();
  if (!ok) return fail(A->error.empty() ? ETL_ERR_CUDA : ETL_ERR_INVALID_ARG);
  *out = A;
  return ETL_OK;
#undef CKA
}
uint64_t etl_dec_arrow_rows(const etl_arrow_batch* a) { return a ? a->n_rows : 0; }
uint32_t etl_dec_arrow_cols(const etl_arrow_batch* a) { return a ? (uint32_t)a->cols.size() : 0; }
const uint64_t* etl_dec_arrow_row_records(const etl_arrow_batch* a, int host) {
  if (!a) return nullptr;
  const uint8_t* base = host ? a->host : a->dev;
  return base ? reinterpret_cast<const uint64_t*>(base + a->row_rec_off) : nullptr;
}
int etl_dec_arrow_column(const etl_arrow_batch* a, uint32_t c, int host, etl_arrow_column* out) {
  if (!a || !out || c >= a->cols.size()) return ETL_ERR_INVALID_ARG;
  const uint8_t* base = host ? a->host : a->dev;
  if (!base) return ETL_ERR_INVALID_ARG;
  const Col& col = a->cols[c];
  memset(out, 0, sizeof *out);
  out->arrow_type = col.arrow_type;
  if (col.arrow_type == ETL_ARROW_UNSUPPORTED) return ETL_OK;
  out->validity = base + col.validity_off;
  if (col.values_bytes) out->values = base + col.values_off;
  if (col.arrow_type == ETL_ARROW_LIST) out->offsets = base + col.offsets_off;
  else if (col.offsets_bytes) { out->offsets = base + col.offsets_off; out->data = base + col.data_off; out->data_bytes = col.data_bytes; }
  return ETL_OK;
}
int etl_dec_arrow_list_values(const etl_arrow_batch* a, uint32_t c, int host, etl_arrow_column* child, uint64_t* n_values) {
  if (!a || !child || c >= a->cols.size() || a->cols[c].arrow_type != ETL_ARROW_LIST) return ETL_ERR_INVALID_ARG;
  const uint8_t* base = host ? a->host : a->dev;
  if (!base) return ETL_ERR_INVALID_ARG;
  const Col& col = a->cols[c];
  memset(child, 0, sizeof *child);
  child->arrow_type = col.child_type;
  child->validity = base + col.c_validity_off;
  if (col.c_values_bytes) child->values = base + col.c_values_off;
  if (col.c_offsets_bytes) { child->offsets = base + col.c_offsets_off; child->data = base + col.c_data_off; child->data_bytes = col.c_data_bytes; }
  if (n_values) *n_values = col.n_values;
  return ETL_OK;
}
void etl_dec_arrow_free(etl_arrow_batch* a) {
  if (!a) return;
  if (a->dev) cudaFree(a->dev);
  if (a->host) cudaFreeHost(a->host);
  delete a;
}

}  // extern "C"
