"""Restatements of the reference's Arrow text forms, for the columnar emitter's formatted mode (ETL_ARROW_FORMATTED).

format_numeric restates PgNumeric's Display (crates/etl/src/conversions/numeric.rs:502-590) line by line over the
decoder's numeric heap entry (etl_numeric_hdr + base-10000 digits, include/etl_decode.h).  list_expected restates
build_list_array and its typed builders (crates/etl-destinations/src/iceberg/encoding.rs:386-776) for one column of
one row selection, from a decoded batch's planes."""
import struct

import numpy as np

NUMERIC_HDR = struct.Struct("<BBhHH")   # kind, sign, weight, scale, pushed_groups

# Arrow types of etl_arrow_column.arrow_type
(A_UNSUP, A_BOOL, A_I32, A_I64, A_F32, A_F64, A_UTF8, A_LBIN, A_DATE32, A_TIME64, A_TS, A_TSTZ, A_UUID, A_LIST) = range(14)
# ETL_K_* → Arrow type of a column (or of an array element) in formatted mode; Json (15) stays unsupported
KIND2ARROW = {1: A_BOOL, 2: A_UTF8, 3: A_I32, 4: A_I32, 5: A_I64, 6: A_I64, 7: A_F32, 8: A_F64, 9: A_UTF8, 10: A_DATE32,
              11: A_TIME64, 12: A_TS, 13: A_TSTZ, 14: A_UUID, 16: A_LBIN}
K_ARRAY, K_JSON = 0x20, 15


def formatted_type(kind: int) -> int:
    if kind & K_ARRAY:
        return A_LIST if (kind & ~K_ARRAY) in KIND2ARROW else A_UNSUP
    return KIND2ARROW.get(kind, A_UNSUP)


def format_numeric(kind: int, sign: int, weight: int, scale: int, digits) -> str:
    """numeric.rs:502-590 (Display for PgNumeric, format_numeric_value)."""
    if kind == 1:
        return "NaN"
    if kind == 2:
        return "Infinity"
    if kind == 3:
        return "-Infinity"
    if not digits:
        return "0"
    out = "-" if sign else ""
    if weight < 0:
        out += "0"
    else:
        for d in range(weight + 1):
            dd = "%04d" % (digits[d] if d < len(digits) else 0)
            if d == 0:
                t = dd.lstrip("0")
                out += t if t else "0"
            else:
                out += dd
    if scale > 0:
        out += "."
        remaining, d = scale, weight + 1
        while remaining > 0:
            dd = "%04d" % (digits[d] if 0 <= d < len(digits) else 0)
            k = min(4, remaining)
            out += dd[:k]
            remaining -= k
            d += 1
    return out


def numeric_entry(heap: bytes, off: int, n_digits: int):
    """(kind, sign, weight, scale, digits) of the numeric heap entry at off"""
    kind, sign, weight, scale, _ = NUMERIC_HDR.unpack_from(heap, off)
    digits = list(struct.unpack_from("<%dh" % n_digits, heap, off + 8)) if n_digits else []
    return kind, sign, weight, scale, digits


def numeric_text(heap: bytes, off: int, n_digits: int) -> bytes:
    return format_numeric(*numeric_entry(heap, off, n_digits)).encode()


def selected_rows(p, schema_index: int, row_kinds: int):
    """(record index, first cell of the row image) of every row the emitter selects, in stream order"""
    sc = p.schemas[schema_index]
    rows = []
    for r in range(p.n_records):
        if int(p.rec_schema[r]) != schema_index or not int(p.rec_flags[r]) & 0x80:
            continue
        k, f = chr(int(p.rec_kind[r])), int(p.rec_flags[r])
        c0, c1 = int(p.rec_cell_base[r]), int(p.rec_cell_base[r + 1])
        if k == "I" and row_kinds & 1:
            rows.append((r, c0))
        elif k == "U" and row_kinds & 2 and not f & 4:
            rows.append((r, c1 - sc.n_cols))
        elif k == "D" and row_kinds & 4 and f & 1:
            rows.append((r, c0))
    return rows


def numeric_column(p, rows, c):
    """Utf8 column of a Numeric column: (validity, int64 offsets, data)"""
    heap = p.heap.tobytes()
    valid, chunks = [], []
    for _, c0 in rows:
        cell = c0 + c
        ok = int(p.cell_tag[cell]) == 9
        valid.append(ok)
        chunks.append(numeric_text(heap, int(p.cell_val[cell]), int(p.cell_aux[cell])) if ok else b"")
    offs = np.zeros(len(rows) + 1, dtype=np.int64)
    offs[1:] = np.cumsum([len(x) for x in chunks])
    return np.array(valid, dtype=bool), offs, b"".join(chunks)


ELEM = np.dtype([("val", "<u8"), ("aux", "<u4"), ("tag", "u1"), ("pad", "u1", 3)])


def list_column(p, rows, c, child_type: int):
    """List column: (list validity, int64 list offsets, child validity, child values) where child values are an array
    for fixed-width children (bool / int / float as numpy, uuid as bytes) and (int64 offsets, data) for Utf8 /
    LargeBinary children.  Vectorised over the elements: the array workload has millions of them."""
    heap = p.heap.tobytes()
    hv = p.heap
    n = len(rows)
    cells = np.array([c0 + c for _, c0 in rows], dtype=np.int64)
    tags = p.cell_tag[cells] if n else np.zeros(0, np.uint8)
    lvalid = tags == 17
    hoff = p.cell_val[cells].astype(np.int64) if n else np.zeros(0, np.int64)
    ne = np.zeros(n, dtype=np.int64)
    if lvalid.any():
        ne[lvalid] = hv[hoff[lvalid][:, None] + np.arange(4, 8)].copy().view("<u4").ravel()
    loffs = np.zeros(n + 1, dtype=np.int64)
    loffs[1:] = np.cumsum(ne)
    nv = int(loffs[-1])
    # element records: heap offset of element j of row r = hoff[r] + 8 + 16 j
    row_of = np.repeat(np.arange(n), ne)
    j = np.arange(nv) - loffs[row_of]
    eoff = hoff[row_of] + 8 + 16 * j
    raw = hv[eoff[:, None] + np.arange(16)] if nv else np.zeros((0, 16), np.uint8)
    el = np.ascontiguousarray(raw).view(ELEM).ravel()
    etag, evalu, eaux = el["tag"].astype(np.int64), el["val"], el["aux"].astype(np.int64)
    want = {A_BOOL: (1,), A_I32: (3, 4), A_I64: (5, 6), A_F32: (7,), A_F64: (8,), A_UTF8: (2, 9), A_LBIN: (16,),
            A_DATE32: (10,), A_TIME64: (11,), A_TS: (12,), A_TSTZ: (13,), A_UUID: (14,)}[child_type]
    cvalid = np.isin(etag, want)
    sv = evalu.view(np.int64)
    if child_type == A_BOOL:
        v = (evalu & 1).astype(bool) & cvalid
    elif child_type in (A_I32, A_DATE32):
        v = np.where(cvalid, sv, 0).astype(np.int32)
    elif child_type == A_F32:
        v = np.where(cvalid, evalu & 0xFFFFFFFF, 0).astype(np.uint32)
    elif child_type == A_I64:
        v = np.where(cvalid, np.where(etag == 5, (evalu & 0xFFFFFFFF).view(np.int64), sv), 0).astype(np.int64)
    elif child_type == A_F64:
        v = np.where(cvalid, sv, 0).astype(np.int64)
    elif child_type in (A_TIME64, A_TS, A_TSTZ):
        v = np.where(cvalid, sv * 1000000 + eaux // 1000, 0).astype(np.int64)
    elif child_type == A_UUID:
        idx = np.where(cvalid, evalu.astype(np.int64), 0)
        b = hv[idx[:, None] + np.arange(16)] if nv else np.zeros((0, 16), np.uint8)
        b = np.where(cvalid[:, None], b, 0).astype(np.uint8)
        v = b.tobytes()
    else:
        lens = np.where(cvalid, eaux, 0)
        num = cvalid & (etag == 9)
        texts = {}
        for k in np.flatnonzero(num):               # numerics: formatted (memoised by heap entry bytes)
            o, d = int(evalu[k]), int(eaux[k])
            key = heap[o:o + 8 + 2 * d]
            t = texts.get(key)
            if t is None:
                t = texts[key] = numeric_text(heap, o, d)
            texts[int(k)] = t
            lens[k] = len(t)
        coffs = np.zeros(nv + 1, dtype=np.int64)
        coffs[1:] = np.cumsum(lens)
        total = int(coffs[-1])
        data = np.zeros(total, dtype=np.uint8)
        plain = cvalid & ~num
        if plain.any():                              # strings / bytes: one gather over the heap
            pl = lens[plain]
            starts = np.repeat(evalu[plain].astype(np.int64) - coffs[:-1][plain], pl)
            dst = np.repeat(coffs[:-1][plain], pl) + (np.arange(int(pl.sum())) - np.repeat(np.cumsum(pl) - pl, pl))
            data[dst] = hv[starts + dst]
        for k in np.flatnonzero(num):
            t = texts[int(k)]
            data[coffs[k]:coffs[k] + len(t)] = np.frombuffer(t, np.uint8)
        v = (coffs, data.tobytes())
    return lvalid, loffs, cvalid, v
