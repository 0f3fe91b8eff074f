/*
 * etl_decode.h — C ABI of the B200 batched pgoutput (CDC) decode engine.
 *
 * This is the drop-in boundary for supabase/etl's streaming-replication hot path. The reference
 * has no FFI seam at the decoder; the entry points below are what a Rust shim in `crates/etl`
 * binds in place of:
 *
 *   reference interface replaced                                   | entry point here
 *   ---------------------------------------------------------------+-----------------------------
 *   EventsStream::poll_next  (crates/etl/src/replication/stream.rs:291-306): one parsed message
 *     per poll → raw CopyData bodies appended to a pinned staging buffer              | etl_stage_*
 *   SchemaStore / SharedTableCache lookups done per message
 *     (crates/etl/src/replication/apply.rs:2062-2079, :3324-3357)                   | etl_dec_put_table_schema
 *   ApplyLoop::handle_replication_message → handle_logical_replication_message →
 *     handle_{begin,commit,relation,insert,update,delete,truncate}_message
 *     (apply.rs:1687-2248) + conversions::event::parse_event_from_*_message
 *     (crates/etl/src/conversions/event.rs:276-543) + parse_cell_from_postgres_text
 *     (crates/etl/src/conversions/text.rs:28-173) for a whole batch at once          | etl_dec_decode
 *   Vec<Event> handed to ApplyLoopState::add_event_to_batch (apply.rs:433-439)        | etl_dec_batch_* accessors
 *
 * Conventions (SURVEY.md §8b): every function returns 0 on success and a non-zero
 * `etl_status` on infrastructure failure (CUDA, allocation, bad arguments). DATA errors are not
 * return codes: they are reported as `first_error` inside a successfully returned batch whose
 * records [0, first_error.record_index) are valid — mirroring apply.rs:1595-1599 where earlier
 * events stay in the batch and the failing message returns Err. One ctx per apply loop; calls on
 * one ctx are not re-entrant. All integers are host (little-endian) order. No torch / C++ types
 * cross this boundary.
 */
#ifndef ETL_DECODE_H
#define ETL_DECODE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ETL_DECODE_ABI_VERSION 2u

/* ---------------------------------------------------------------- status codes */
typedef enum etl_status {
  ETL_OK = 0,
  ETL_ERR_INVALID_ARG = 1,
  ETL_ERR_CUDA = 2,
  ETL_ERR_ALLOC = 3,
  ETL_ERR_NO_DEVICE = 4,
  ETL_ERR_INTERNAL = 5,
} etl_status;

/* ---------------------------------------------------------------- record kinds
 * rec_kind is the pgoutput tag byte of the frame (XLogData 'w' frames), or 'k' for a primary
 * keepalive frame. Grammar: SURVEY.md Appendix B. */
enum {
  ETL_REC_BEGIN = 'B',
  ETL_REC_COMMIT = 'C',
  ETL_REC_ORIGIN = 'O',
  ETL_REC_RELATION = 'R',
  ETL_REC_TYPE = 'Y',
  ETL_REC_INSERT = 'I',
  ETL_REC_UPDATE = 'U',
  ETL_REC_DELETE = 'D',
  ETL_REC_TRUNCATE = 'T',
  ETL_REC_MESSAGE = 'M',
  ETL_REC_KEEPALIVE = 'k',
};

/* rec_flags bits */
enum {
  ETL_RF_OLD_FULL = 0x01,    /* 'O' image present: OldTableRow::Full   (event.rs:445-448) */
  ETL_RF_OLD_KEY = 0x02,     /* 'K' image present: OldTableRow::Key    (event.rs:441-444) */
  ETL_RF_NEW_PARTIAL = 0x04, /* UpdatedTableRow::Partial               (event.rs:662-667) */
  ETL_RF_DDL_MESSAGE = 0x08, /* 'M' whose prefix is supabase_etl_ddl   (event.rs:31)      */
  ETL_RF_EVENT = 0x80,       /* the reference emits an Event for this frame               */
};

/* ---------------------------------------------------------------- cell tags = Cell variants
 * crates/etl/src/types/cell.rs:38-76, in declaration order. */
enum {
  ETL_CELL_NULL = 0,
  ETL_CELL_BOOL = 1,        /* val = 0|1 */
  ETL_CELL_STRING = 2,      /* val = byte offset into the staged stream, aux = byte length (zero copy) */
  ETL_CELL_I16 = 3,         /* val = sign-extended value */
  ETL_CELL_I32 = 4,
  ETL_CELL_U32 = 5,
  ETL_CELL_I64 = 6,
  ETL_CELL_F32 = 7,         /* val = IEEE-754 bits (low 32) */
  ETL_CELL_F64 = 8,         /* val = IEEE-754 bits */
  ETL_CELL_NUMERIC = 9,     /* val = heap offset of etl_numeric_hdr, aux = number of base-10000 digits */
  ETL_CELL_DATE = 10,       /* val = days since 1970-01-01 (signed) */
  ETL_CELL_TIME = 11,       /* val = seconds since midnight, aux = nanoseconds (>= 1e9 only for :60 leap second) */
  ETL_CELL_TIMESTAMP = 12,  /* val = seconds since 1970-01-01T00:00:00 (naive), aux = nanoseconds */
  ETL_CELL_TIMESTAMPTZ = 13,/* val = UTC seconds since the unix epoch, aux = nanoseconds */
  ETL_CELL_UUID = 14,       /* val = heap offset of 16 big-endian bytes */
  ETL_CELL_JSON = 15,       /* val = stream byte offset, aux = byte length of the VALIDATED json text */
  ETL_CELL_BYTES = 16,      /* val = heap offset of decoded bytes, aux = length */
  ETL_CELL_ARRAY = 17,      /* val = heap offset of etl_array_hdr, aux = element count */
  ETL_CELL_MISSING = 254,   /* unresolved UnchangedToast → PartialTableRow missing index (event.rs:641-656) */
};

/* column decode classes derived from the type oid exactly as text.rs:28-173 dispatches */
enum {
  ETL_K_BOOL = 1, ETL_K_STRING = 2, ETL_K_I16 = 3, ETL_K_I32 = 4, ETL_K_U32 = 5, ETL_K_I64 = 6,
  ETL_K_F32 = 7, ETL_K_F64 = 8, ETL_K_NUMERIC = 9, ETL_K_DATE = 10, ETL_K_TIME = 11,
  ETL_K_TIMESTAMP = 12, ETL_K_TIMESTAMPTZ = 13, ETL_K_UUID = 14, ETL_K_JSON = 15, ETL_K_BYTES = 16,
  ETL_K_ARRAY = 0x20, /* ETL_K_ARRAY | element kind */
};

/* numeric heap entry: header followed by `aux` little-endian int16 base-10000 digits.
 * crates/etl/src/conversions/numeric.rs:67-88 */
typedef struct etl_numeric_hdr {
  uint8_t kind;   /* 0 value, 1 NaN, 2 +Infinity, 3 -Infinity */
  uint8_t sign;   /* 0 positive, 1 negative */
  int16_t weight;
  uint16_t scale;
  uint16_t pushed_groups; /* base-10000 groups the reference pushes onto its digit Vec before stripping zero groups
                             (numeric.rs:441-448; 0 for canonical zero and the specials, saturates at 65535): the
                             Vec's capacity — and with it the row's size hint — follows from this count */
} etl_numeric_hdr;

/* array heap entry: header followed by n_elems etl_array_elem (8-byte aligned). Element payloads
 * (unescaped strings, numerics, bytes, uuids) live in the heap at elem.val. text.rs:184-249 */
typedef struct etl_array_hdr {
  uint8_t elem_kind; /* ETL_K_* of the element type */
  uint8_t _pad[3];
  uint32_t n_elems;
} etl_array_hdr;
typedef struct etl_array_elem {
  uint64_t val;
  uint32_t aux;
  uint8_t tag;   /* ETL_CELL_* (ETL_CELL_NULL for a NULL element) */
  uint8_t _pad[3];
} etl_array_elem;

/* ---------------------------------------------------------------- data-error descriptions
 * (ErrorKind, description) pairs the path can raise. crates/etl/src/error.rs */
typedef enum etl_error_kind {
  ETL_EK_NONE = 0,
  ETL_EK_CONVERSION_ERROR = 1,
  ETL_EK_INVALID_DATA = 2,
  ETL_EK_DESERIALIZATION_ERROR = 3,
  ETL_EK_INVALID_STATE = 4,
  ETL_EK_VALIDATION_ERROR = 5,
  ETL_EK_CORRUPTED_TABLE_SCHEMA = 6,
  ETL_EK_MISSING_TABLE_SCHEMA = 7,
  ETL_EK_SOURCE_ERROR = 8, /* malformed frame: the third-party parser returns io::Error */
} etl_error_kind;

typedef enum etl_error_code {
  ETL_E_NONE = 0,
  ETL_E_UTF8 = 1,               /* ConversionError  "UTF-8 conversion failed"            error.rs:480-489 */
  ETL_E_PARSE_INT = 2,          /* ConversionError  "Integer parsing failed"             error.rs:510    */
  ETL_E_PARSE_FLOAT = 3,        /* ConversionError  "Float parsing failed"               error.rs:525    */
  ETL_E_DATETIME = 4,           /* ConversionError  "Datetime parsing failed"            error.rs:878    */
  ETL_E_NUMERIC = 5,            /* ConversionError  "Numeric parsing failed"             error.rs:893    */
  ETL_E_UUID = 6,               /* InvalidData      "UUID parsing failed"                error.rs:863    */
  ETL_E_JSON = 7,               /* DeserializationError "JSON deserialization failed"    error.rs:456-463 */
  ETL_E_BOOL = 8,               /* InvalidData      "Invalid boolean value"              bool.rs:17      */
  ETL_E_BYTEA = 9,              /* ConversionError  "Bytea hex string conversion failed" hex.rs:12-29    */
  ETL_E_BINARY_FORMAT = 10,     /* ConversionError  "Binary format not supported in tuple data" event.rs:976 */
  ETL_E_NOT_NULL = 11,          /* InvalidData      "Required column missing from tuple" event.rs:947-955 */
  ETL_E_FIELD_COUNT = 12,       /* ConversionError  "Tuple data field count does not match schema" event.rs:556,608 */
  ETL_E_FULL_ROW_MISSING = 13,  /* ConversionError  "Tuple missing source value for full row image" event.rs:568 */
  ETL_E_KEY_NO_COLUMNS = 14,    /* ConversionError  "Replica-identity tuple missing key columns" event.rs:890 */
  ETL_E_KEY_SHAPE = 15,         /* ConversionError  "Replica-identity tuple shape does not match schema" event.rs:907 */
  ETL_E_KEY_MISSING_VALUE = 16, /* ConversionError  "Replica-identity tuple missing source value" event.rs:803,847 */
  ETL_E_TX_STATE = 17,          /* InvalidState     "Invalid transaction state"          apply.rs:1955,2018,2098,... */
  ETL_E_COMMIT_LSN = 18,        /* ValidationError  "Invalid commit LSN"                 apply.rs:1960-1969 */
  ETL_E_MISSING_TABLE_STATE = 19,/* InvalidState    "Missing shared table state"         apply.rs:3328-3337 */
  ETL_E_ARRAY_SHORT = 20,       /* ConversionError  "Array input too short"              text.rs:190 */
  ETL_E_ARRAY_BRACES = 21,      /* ConversionError  "Array input missing braces"         text.rs:194 */
  ETL_E_UNKNOWN_COLUMNS = 22,   /* CorruptedTableSchema "Received columns during replication that are not in the stored table schema" error.rs:960-975 */
  ETL_E_MISSING_TABLE_SCHEMA = 23,/* MissingTableSchema  stored TableSchema absent for a Relation (apply.rs:2062-2072) */
  ETL_E_MALFORMED_FRAME = 24,   /* SourceError: truncated frame / unknown tag (postgres-replication parse error) */
  ETL_E_COPY_NOT_TERMINATED = 25, /* ConversionError "Row data not properly terminated"                  table_row.rs:88-92 */
  ETL_E_COPY_COLUMN_COUNT = 26,  /* ConversionError "Column count mismatch between schema and row"     table_row.rs:103-113,150-160 */
  ETL_E__COUNT
} etl_error_code;

typedef struct etl_first_error {
  uint64_t record_index; /* UINT64_MAX when the batch decoded cleanly */
  uint32_t seq;          /* evaluation step inside the record (old tuple cells, then new tuple cells) */
  uint32_t code;         /* etl_error_code */
  uint32_t kind;         /* etl_error_kind */
  uint32_t _pad;
} etl_first_error;

/* ---------------------------------------------------------------- schema catalogue
 * ColumnSchema — crates/etl-postgres/src/types/schema.rs:165-179 */
typedef struct etl_column_schema {
  const char* name;        /* UTF-8, NUL terminated */
  uint32_t type_oid;
  int32_t modifier;
  int32_t ordinal_position;
  int32_t primary_key_ordinal_position; /* -1 = not part of the primary key */
  uint8_t nullable;
  uint8_t _pad[7];
} etl_column_schema;

/* stream state carried between batches — ApplyLoopState {remote_final_lsn, next_tx_ordinal}
 * apply.rs:600-626 */
typedef struct etl_stream_state {
  uint64_t final_lsn;       /* valid when in_tx != 0 */
  uint64_t next_tx_ordinal;
  uint8_t in_tx;            /* remote_final_lsn.is_some() */
  uint8_t _pad[7];
} etl_stream_state;

/* ---------------------------------------------------------------- staging
 * The stager is the replacement for the per-message parse in EventsStream: each CopyData body
 * (what `copy_both_simple::<Bytes>` yields, crates/etl/src/replication/client.rs:1098-1099) is
 * appended as 'd' + int32(len+4, big-endian) + body into one pinned host buffer. While appending
 * it records, for free, (a) sparse anchors: anchors[k] = offset of the first frame that starts at
 * or after k*anchor_stride (len if none), and (b) the offsets of Relation frames. */
typedef struct etl_stager etl_stager;
int etl_stage_create(uint64_t capacity_bytes, uint32_t anchor_stride, etl_stager** out);
void etl_stage_destroy(etl_stager*);
void etl_stage_reset(etl_stager*);
int etl_stage_append(etl_stager*, const uint8_t* copydata_body, uint32_t body_len);
/* adopt an already framed stream (bench/tests): walks it once on the host to build the indexes */
int etl_stage_append_framed(etl_stager*, const uint8_t* framed, uint64_t len);

typedef struct etl_dec_input {
  const uint8_t* host_buf;       /* framed stream in host memory (pinned if from the stager) */
  const uint8_t* dev_buf;        /* optional: same bytes already resident in HBM (NULL → library copies). PRECONDITION:
                                    16-byte aligned and followed by at least 64 readable bytes after `len` — the
                                    kernels read whole aligned words / 16-byte copy granules around a cell. The
                                    library's own copy of host_buf is padded for you. */
  uint64_t len;
  const uint64_t* anchors;       /* host array, n_anchors entries, see etl_stager */
  const uint64_t* dev_anchors;   /* optional: n_anchors + 1 entries resident in HBM, last entry = len. Anchors are
                                    not trusted: the kernels clamp them to `len` and treat a non-ascending pair as an
                                    empty segment; an anchor that is not a frame start yields ETL_E_MALFORMED_FRAME. */
  uint64_t n_anchors;
  uint32_t anchor_stride;
  uint32_t max_frame_len;        /* 0 = unknown; else an upper bound of the longest frame in bytes ('d' + length field +
                                    body; the stager fills it).  A hint: when no frame can hold a 512-byte value the
                                    passes that exist for long values are skipped (and run after all if it was wrong) */
  const uint64_t* relation_offsets; /* host array: frame offsets of every 'R' frame, ascending */
  uint64_t n_relations;
  etl_stream_state carry_in;
} etl_dec_input;
int etl_stage_view(const etl_stager*, etl_dec_input* out);

/* ---------------------------------------------------------------- decoder */
typedef struct etl_dec_ctx etl_dec_ctx;
typedef struct etl_dec_batch etl_dec_batch;

/* One context = one apply loop on one GPU (the harness and the shim run one process / thread per GPU).  SURVEY §8b
 * sketched `etl_dec_create(const int* device_ids, int n_dev, …)`; with one owner per device the multi-GPU form is
 * etl_dec_create + etl_dec_comm_init(rank, n_ranks) below, which gives the context its NCCL communicator. */
int etl_dec_create(int device_id, etl_dec_ctx** out);
/* run on the caller's CUDA stream (a cudaStream_t, e.g. torch.cuda.current_stream().cuda_stream);
 * default: a private stream created by etl_dec_create */
int etl_dec_set_stream(etl_dec_ctx*, void* cuda_stream);
void etl_dec_destroy(etl_dec_ctx*);
const char* etl_dec_last_error(const etl_dec_ctx*);
uint32_t etl_dec_abi_version(void);

/* store (or replace) the TableSchema the SchemaStore would return for table_id */
int etl_dec_put_table_schema(etl_dec_ctx*, uint32_t table_id, uint64_t snapshot_id,
                             const etl_column_schema* cols, uint32_t n_cols);
/* forget replicated-schema state (new connection: Postgres re-sends Relation messages) */
int etl_dec_reset_relations(etl_dec_ctx*);
/* ETL_K_* decode class of a type oid, exactly as text.rs:28-173 dispatches (utils.rs:7-16 for unknown oids) */
uint32_t etl_dec_kind_for_type_oid(uint32_t type_oid);
/* free / total device memory as the CUDA runtime reports it (leak checks) */
int etl_dec_mem_info(etl_dec_ctx*, uint64_t* free_bytes, uint64_t* total_bytes);

/* ---------------------------------------------------------------- multi-GPU (SURVEY §8e)
 * The staged stream shards by byte range at record starts, one range per GPU of a box; the library owns the
 * exchange: an NCCL communicator over the ranks (libnccl.so.2 is resolved at run time — the copy already loaded
 * into the process if there is one).  etl_dec_decode_sharded runs
 *   relation-update exchange (the Relation frames of every range, one all-gather; apply.rs:2012-2089,
 *   table_cache.rs:36-130) → index pass → ncclAllGather of the 64-byte seam summaries ON THE DECODE STREAM →
 *   device-side fold of the ranks before this one into the carry-in (apply.rs:600-626) → record + tuple passes
 * with no host round trip between the index and the record pass.  `carry_in` of the input is the state before the
 * FIRST shard (pass the same value on every rank); summary.carry_out is the state after the LAST shard and
 * summary.record_index_base the global index of this rank's first record.  Output order = rank order. */
#define ETL_COMM_ID_BYTES 128u
int etl_dec_comm_unique_id(uint8_t* out, uint32_t cap);   /* rank 0; broadcast the bytes to the other ranks */
int etl_dec_comm_init(etl_dec_ctx*, const uint8_t* unique_id, uint32_t id_bytes, int rank, int n_ranks);
/* The same protocol with the two exchanges carried by the HOST (a box without NVLink/NCCL between the processes, tests
 * on one GPU): `fn(user, send, recv, bytes)` must fill recv with the n_ranks blocks of `bytes` in rank order, return 0. */
typedef int (*etl_host_allgather_fn)(void* user, const void* send, void* recv, uint64_t bytes);
int etl_dec_comm_init_host(etl_dec_ctx*, int rank, int n_ranks, etl_host_allgather_fn fn, void* user);

/* flags for etl_dec_decode */
enum {
  ETL_DECODE_RESULTS_TO_HOST = 0x1, /* copy result planes to pinned host memory before returning */
  ETL_DECODE_SEAM_DEFER = 0x2,      /* multi-GPU shard: carry_in unknown, run only the local scan;
                                       caller exchanges etl_dec_seam and calls etl_dec_decode_finish */
  ETL_DECODE_NO_TIMING = 0x4,       /* leave the *_ms fields of the summary at 0: the CUDA-event queries behind them cost
                                       ~25 us of host time per call, which an 8 MiB batch notices */
};

/* per-shard seam summary exchanged with ONE all-gather across the GPUs of a box (SURVEY §8e) */
typedef struct etl_dec_seam {
  uint64_t n_records;
  uint64_t n_cells;
  uint64_t heap_bytes;
  uint64_t lsn;        /* final_lsn of the last Begin in the shard (valid if has_begin) */
  uint64_t ord;        /* has_begin: next_tx_ordinal at shard end; else ordinal consumers in shard */
  uint8_t has_begin;
  uint8_t closed;      /* a Commit follows the last Begin (or any Commit when !has_begin) */
  uint8_t _pad[6];
} etl_dec_seam;

/* Limits of one call: len < 1 TiB and fewer than 2^32 frames (record indices inside a batch are 32-bit: a 64 GiB
 * stream of nothing but 23-byte keepalives is still below it); a longer stream is decoded in several calls chained
 * through carry_in / carry_out, like the reference's batches. */
int etl_dec_decode(etl_dec_ctx*, const etl_dec_input*, uint32_t flags, etl_dec_batch** out);
int etl_dec_decode_sharded(etl_dec_ctx*, const etl_dec_input*, uint32_t flags, etl_dec_batch** out);
/* two-phase form: the caller exchanges the seam summaries itself (tests; hosts without NCCL) */
int etl_dec_decode_begin(etl_dec_ctx*, const etl_dec_input*, uint32_t flags, etl_dec_seam* seam_out);
int etl_dec_decode_finish(etl_dec_ctx*, const etl_stream_state* carry_in, uint64_t record_index_base,
                          etl_dec_batch** out);
void etl_dec_batch_free(etl_dec_batch*);

/* result planes. Device planes are owned by the batch. Host planes exist only when
 * ETL_DECODE_RESULTS_TO_HOST was set; they live in a pinned buffer cached on the ctx and stay
 * valid until the next decode on the same ctx. All arrays are in stream order. */
typedef struct etl_dec_planes {
  uint64_t n_records;
  uint64_t n_cells;
  uint64_t heap_bytes;
  /* record plane (n_records entries; rec_cell_base has n_records + 1) */
  const uint64_t* rec_off;
  const uint8_t* rec_kind;
  const uint8_t* rec_flags;
  const uint32_t* rec_rel;       /* relation id (R/I/U/D), relation count (T) */
  const int32_t* rec_schema;     /* schema version index (see etl_dec_batch_schema), -1 if none */
  const uint64_t* rec_start_lsn;
  const uint64_t* rec_commit_lsn;
  const uint64_t* rec_tx_ordinal;
  const uint64_t* rec_cell_base;
  const uint32_t* rec_tuple_bytes; /* DML: Σ text lengths of the frame's tuples = the ETL_ROW_SIZE_BYTES histogram sample
                                      (calculate_tuple_bytes, event.rs:260-270, :388, :462, :507); 0 for other records */
  const uint32_t* rec_heap_hint;   /* DML: Σ estimate_cell_allocated_bytes (types/table_row.rs:295-345) over the String,
                                      Bytes and Numeric cells of the event's rows — the part of Event::size_hint
                                      (types/event.rs:288-312) that depends on the data; the struct sizes and Vec<Cell>
                                      capacities follow from rec_kind / rec_flags / the schema. Json and Array payloads
                                      are estimated by whoever builds the serde_json::Value / ArrayCell. */
  /* cell plane */
  const uint8_t* cell_tag;
  const uint64_t* cell_val;
  const uint32_t* cell_aux;
  /* heap */
  const uint8_t* heap;
} etl_dec_planes;

typedef struct etl_dec_summary {
  etl_first_error first_error;
  etl_stream_state carry_out;
  uint64_t insert_bytes;  /* ETL_BYTES_PROCESSED_TOTAL{insert}: calculate_tuple_bytes event.rs:260-270 */
  uint64_t update_bytes;
  uint64_t delete_bytes;
  uint64_t n_events;      /* frames with ETL_RF_EVENT */
  uint32_t n_schemas;     /* schema versions referenced by rec_schema */
  uint32_t gpu_launches;  /* kernels launched for this batch */
  float kernel_ms;        /* CUDA-event time of the kernel sequence (resident input → resident output) */
  float h2d_ms, d2h_ms;
  float index_ms;         /* pass A: k_act_* + k_chase (frame offsets) [+ the totals-only k_records pass] */
  float emit_ms;          /* pass B+C: k_records … k_long_cells */
  float frames_ms;        /* k_records (stream-state scan + record plane) */
  float walk_ms;          /* k_bin_scan + k_perm (shape bins) */
  float spans_ms;         /* k_utf8_dead (structure-blind UTF-8 pass over segments without a frame start) */
  float cells_ms;         /* k_rows (tuples → rows: staging, walk, UTF-8, per-kind parsers, cell plane) */
  float long_ms;          /* k_long_cells (verdicts of the long text cells: line bitmap + edges) */
  uint64_t h2d_bytes, d2h_bytes; /* bytes copied host→device / device→host for this batch */
  uint64_t span_bytes;    /* bytes streamed by k_utf8_dead (its algorithmic bytes) */
  uint64_t record_index_base; /* global index of this batch's first record (sharded decode: Σ records of the ranks before) */
  uint32_t abi_version;
  uint32_t _pad2;
} etl_dec_summary;

int etl_dec_batch_planes(const etl_dec_batch*, int host, etl_dec_planes* out);
int etl_dec_batch_summary(const etl_dec_batch*, etl_dec_summary* out);

/* replicated schema version i: what ReplicatedTableSchema exposes to events (schema.rs:651-900) */
typedef struct etl_dec_schema_info {
  uint32_t table_id;
  uint32_t n_cols;          /* replicated columns */
  uint32_t n_identity;
  uint32_t _pad;
  uint64_t snapshot_id;
  uint64_t effective_off;   /* stream offset of the Relation frame that installed it (0 = carried in) */
  const uint8_t* col_kind;  /* n_cols ETL_K_* */
  const uint8_t* col_flags; /* bit0 nullable, bit1 identity */
  const int32_t* col_index; /* index into the stored TableSchema's column list */
} etl_dec_schema_info;
int etl_dec_batch_schema(const etl_dec_batch*, uint32_t index, etl_dec_schema_info* out);

/* ---------------------------------------------------------------- initial-sync COPY rows (SURVEY §8f N1)
 * Replaces parse_table_row_from_postgres_copy_bytes (crates/etl/src/conversions/table_row.rs:25-165) applied row by
 * row by TableCopyStream::poll_next (crates/etl/src/replication/stream.rs:75-101) for a whole buffer of rows.
 * `buf` holds the COPY-text rows back to back exactly as the CopyData bodies arrive (each ends with its LF);
 * row_offsets has n_rows + 1 ascending entries (row r = [row_offsets[r], row_offsets[r+1])).  Same device-buffer
 * precondition as etl_dec_input.dev_buf (16-byte aligned, 64 readable bytes after len).  The table's columns are those
 * of etl_dec_put_table_schema, in order.  Result: an etl_dec_batch whose planes hold n_records = n_rows,
 * n_cells = n_rows * n_cols (row-major: cell r * n_cols + c), rec_off = the row offsets, rec_kind..rec_heap_hint NULL;
 * a string / json cell is a span of `buf` (val = offset) unless the field needed unescaping: then bit 63 of val is
 * set and the low bits are a heap offset.  first_error: record_index = row, seq = 0 for the row's UTF-8 check,
 * 1 + column otherwise; rows before it are valid. */
#define ETL_COPY_VAL_IN_HEAP (1ull << 63)
typedef struct etl_copy_input {
  const uint8_t* host_buf;
  const uint8_t* dev_buf;          /* optional, resident copy */
  uint64_t len;
  const uint64_t* row_offsets;     /* host, n_rows + 1 entries */
  const uint64_t* dev_row_offsets; /* optional, resident copy */
  uint64_t n_rows;
} etl_copy_input;
int etl_dec_copy_decode(etl_dec_ctx*, uint32_t table_id, const etl_copy_input*, uint32_t flags, etl_dec_batch** out);

/* ---------------------------------------------------------------- columnar emitter (SURVEY §8f N2)
 * The rows of ONE replicated-schema version of a decoded batch as Arrow-layout column buffers, built on the device.
 * Replaces the per-row walk of the destinations' encoders (crates/etl-destinations/src/iceberg/encoding.rs:61-330:
 * build_array_for_field and the cell_to_* converters; the DuckLake / BigQuery encoders walk the same Vec<TableRow>) for
 * the column types whose Arrow value depends on the decoded cell alone.  Numeric / Json / Array columns (cell_to_string
 * formatting in the reference) come back as ETL_ARROW_UNSUPPORTED and stay on the shim's row path, unless
 * etl_dec_arrow_emit_ex is asked for ETL_ARROW_FORMATTED (below).
 * row_kinds: bit 0 inserts, bit 1 updates (new image, Full rows only), bit 2 deletes (old image, when Full); rows keep
 * stream order and etl_dec_arrow_row_records gives the record index of each (for the CDC columns). */
enum {
  ETL_ARROW_UNSUPPORTED = 0,
  ETL_ARROW_BOOLEAN = 1,        /* values bit-packed like the validity bitmap */
  ETL_ARROW_INT32 = 2,          /* Cell::I16 | I32   (encoding.rs:200-206) */
  ETL_ARROW_INT64 = 3,          /* Cell::I64 | U32   (:214-220) */
  ETL_ARROW_FLOAT32 = 4,
  ETL_ARROW_FLOAT64 = 5,
  ETL_ARROW_UTF8 = 6,           /* int32 offsets[n_rows + 1] + data */
  ETL_ARROW_LARGE_BINARY = 7,   /* int64 offsets[n_rows + 1] + data */
  ETL_ARROW_DATE32 = 8,         /* days since 1970-01-01 (:257-262) */
  ETL_ARROW_TIME64_US = 9,      /* microseconds since midnight (:270-275) */
  ETL_ARROW_TIMESTAMP_US = 10,  /* naive, microseconds since the epoch (:284-289) */
  ETL_ARROW_TIMESTAMPTZ_US = 11,/* UTC, microseconds since the epoch (:297-302) */
  ETL_ARROW_UUID = 12,          /* FixedSizeBinary(16) */
  ETL_ARROW_LIST = 13,          /* ETL_ARROW_FORMATTED only: validity = list validity, offsets = int32 list offsets
                                   [n_rows + 1], values / data NULL; the elements: etl_dec_arrow_list_values */
};
typedef struct etl_arrow_column {
  uint32_t arrow_type;
  uint32_t _pad;
  const uint8_t* validity;  /* bit i = row i is non-null (LSB first), ceil(n_rows / 8) bytes, zero padded to 64 */
  const void* values;       /* fixed-width values, n_rows entries (Boolean: bit-packed); NULL for var-width columns */
  const void* offsets;      /* var-width: n_rows + 1 offsets (int32 for UTF8, int64 for LARGE_BINARY) */
  const uint8_t* data;      /* var-width: the bytes */
  uint64_t data_bytes;
} etl_arrow_column;
typedef struct etl_arrow_batch etl_arrow_batch;
int etl_dec_arrow_emit(const etl_dec_batch*, uint32_t schema_index, uint32_t row_kinds, int to_host, etl_arrow_batch** out);
/* flags for etl_dec_arrow_emit_ex; flags == 0 is etl_dec_arrow_emit, other bits are ETL_ERR_INVALID_ARG */
#define ETL_ARROW_FORMATTED 0x1u   /* Numeric → ETL_ARROW_UTF8, arrays (non-json elements) → ETL_ARROW_LIST */
/* With ETL_ARROW_FORMATTED (crates/etl-destinations/src/iceberg/encoding.rs, cell_to_string :349 and
 * build_list_array :386-776; element types as iceberg/schema.rs:9-37):
 *   Numeric column → ETL_ARROW_UTF8 holding PgNumeric::to_string() (conversions/numeric.rs:502-590)
 *   array column → ETL_ARROW_LIST whose child type is the element's: bool → BOOLEAN, int2 / int4 → INT32,
 *     int8 / oid → INT64, float4 / float8 → FLOAT32 / FLOAT64, text-like and numeric → UTF8 (numeric formatted as
 *     above), date → DATE32, time → TIME64_US, timestamp / timestamptz → TIMESTAMP_US / TIMESTAMPTZ_US,
 *     uuid → UUID, bytea → LARGE_BINARY.  A null cell is a null list; a NULL element a null child value.
 *   Json columns and json / jsonb arrays stay ETL_ARROW_UNSUPPORTED.
 * Limits, as for Utf8 columns: a Utf8 column or child over 2 GiB, or a list column of 2^31 or more values, fails the
 * call with ETL_ERR_INVALID_ARG (split the batch). */
int etl_dec_arrow_emit_ex(const etl_dec_batch*, uint32_t schema_index, uint32_t row_kinds, uint32_t flags, int to_host,
                          etl_arrow_batch** out);
uint64_t etl_dec_arrow_rows(const etl_arrow_batch*);
uint32_t etl_dec_arrow_cols(const etl_arrow_batch*);
const uint64_t* etl_dec_arrow_row_records(const etl_arrow_batch*, int host);
int etl_dec_arrow_column(const etl_arrow_batch*, uint32_t column, int host, etl_arrow_column* out);
/* the child column of an ETL_ARROW_LIST column: an etl_arrow_column over n_values elements (its own validity, values
 * or offsets + data, same conventions); ETL_ERR_INVALID_ARG for any other column */
int etl_dec_arrow_list_values(const etl_arrow_batch*, uint32_t column, int host, etl_arrow_column* child,
                              uint64_t* n_values);
void etl_dec_arrow_free(etl_arrow_batch*);
/* device address of the staged stream a batch was decoded from (string / json cells are offsets into it); valid until
 * the next decode on the same context (library-owned copy) or as long as the caller's dev_buf lives */
const uint8_t* etl_dec_batch_device_stream(const etl_dec_batch*);

/* ---------------------------------------------------------------- shim stand-in (host only, no GPU work)
 * What the Rust shim does with the planes (INTEGRATION.md §3; replaces nothing in the reference — it is the glue that
 * rebuilds the reference's own types): materialise the AoS Vec<Event> handed to add_event_to_batch (apply.rs:433-439)
 * — one owned copy per String / Bytes / Numeric, a serde_json-style tree per Json cell, ArrayCells — and compute
 * Event::size_hint (types/event.rs:288-312, types/table_row.rs:250-345) per event.  C++ here because the image has no
 * Rust toolchain; the Rust struct sizes are parameters (pass std::mem::size_of values; NULL = x86-64 estimates). */
typedef struct etl_rust_layout {
  uint32_t size_of_cell, size_of_table_row, size_of_partial_table_row;
  uint32_t size_of_begin_event, size_of_commit_event, size_of_insert_event, size_of_update_event, size_of_delete_event,
           size_of_truncate_event, size_of_replicated_table_schema, size_of_relation_event;
  uint32_t size_of_json_value, size_of_usize;
} etl_rust_layout;
typedef struct etl_event_list etl_event_list;
/* batch must have been decoded with ETL_DECODE_RESULTS_TO_HOST; host_stream = the staged bytes (string / json spans) */
int etl_shim_materialise(const etl_dec_batch*, const uint8_t* host_stream, const etl_rust_layout*, etl_event_list** out);
uint64_t etl_shim_event_count(const etl_event_list*);
uint64_t etl_shim_size_hint(const etl_event_list*, uint64_t event_index);  /* Event::size_hint */
uint64_t etl_shim_total_size_hint(const etl_event_list*);                  /* what events_batch_bytes would hold */
uint64_t etl_shim_owned_bytes(const etl_event_list*);                      /* bytes copied into owned buffers */
/* serde_json::to_string of the Json cell at `new_row_cell` of an insert/update event (tests); returns its length */
int64_t etl_shim_json_text(const etl_event_list*, uint64_t event_index, uint32_t new_row_cell, char* buf, uint64_t cap);
void etl_shim_event_list_free(etl_event_list*);

#ifdef __cplusplus
}
#endif
#endif /* ETL_DECODE_H */
