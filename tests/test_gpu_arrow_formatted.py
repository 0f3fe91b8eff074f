"""Columnar emitter, formatted mode (etl_dec_arrow_emit_ex with ETL_ARROW_FORMATTED): Numeric columns as Utf8 and array
columns as List<child>, against the restatements of tests/arrow_ref.py (PgNumeric::to_string and the iceberg list
builders) evaluated on the ORACLE's planes, as test_gpu_arrow.py does for the plain columns.  Also: flags == 0 is
etl_dec_arrow_emit byte for byte."""
import ctypes as C

import numpy as np
import pytest

import arrow_ref as R
from etl_b200 import abi, pgoutput as pg, workloads as wl
from test_gpu_parity import ARRAY_COLS

pytestmark = pytest.mark.gpu

FMT = abi.ARROW_FORMATTED
WIDTH = {R.A_I32: 4, R.A_DATE32: 4, R.A_F32: 4, R.A_I64: 8, R.A_F64: 8, R.A_TIME64: 8, R.A_TS: 8, R.A_TSTZ: 8, R.A_UUID: 16}


@pytest.fixture(scope="module")
def lib():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return abi.load()


_cudart = None


def _device_bytes(ptr, n):
    """n bytes at a device address (the to_host=0 image): cudaMemcpy of the runtime the library already loaded"""
    global _cudart
    if _cudart is None:
        path = next(l.split()[-1] for l in open("/proc/self/maps") if "libcudart" in l)
        _cudart = C.CDLL(path)
        _cudart.cudaMemcpy.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]
    buf = (C.c_uint8 * max(n, 1))()
    assert _cudart.cudaMemcpy(buf, C.c_void_p(ptr), n, 2) == 0
    return bytes(buf[:n])


def _bytes(ptr, n, host):
    if n == 0:
        return b""
    return bytes((C.c_uint8 * n).from_address(ptr)) if host else _device_bytes(ptr, n)


def _bits(raw, n):
    return np.unpackbits(np.frombuffer(raw, np.uint8), bitorder="little")[:n].astype(bool)


def column_buffers(col: abi.ArrowColumn, n: int, host: int) -> dict:
    """the meaningful bytes of every buffer of a column of n entries"""
    at = col.arrow_type
    out = {"type": at}
    if at == R.A_UNSUP:
        return out
    out["validity"] = _bytes(col.validity, (n + 7) // 8, host)
    if at == R.A_BOOL:
        out["values"] = _bytes(col.values, (n + 7) // 8, host)
    elif at in WIDTH:
        out["values"] = _bytes(col.values, n * WIDTH[at], host)
    else:
        ow = 8 if at == R.A_LBIN else 4
        out["offsets"] = _bytes(col.offsets, (n + 1) * ow, host)
        if at != R.A_LIST:
            out["data"] = _bytes(col.data, col.data_bytes, host)
    return out


class Emitted:
    def __init__(self, lib, bh, si, kinds, flags, to_host=1):
        self.lib, self.a, self.host = lib, C.c_void_p(), to_host
        if flags is None:
            assert lib.etl_dec_arrow_emit(bh._h, si, kinds, to_host, C.byref(self.a)) == 0
        else:
            assert lib.etl_dec_arrow_emit_ex(bh._h, si, kinds, flags, to_host, C.byref(self.a)) == 0
        self.n = lib.etl_dec_arrow_rows(self.a)
        self.n_cols = lib.etl_dec_arrow_cols(self.a)

    def records(self):
        return np.frombuffer(_bytes(self.lib.etl_dec_arrow_row_records(self.a, self.host) or 0, 8 * self.n, self.host), np.uint64)

    def column(self, c):
        col = abi.ArrowColumn()
        assert self.lib.etl_dec_arrow_column(self.a, c, self.host, C.byref(col)) == 0
        return col

    def buffers(self, c):
        return column_buffers(self.column(c), self.n, self.host)

    def child(self, c):
        ch, nv = abi.ArrowColumn(), C.c_uint64()
        assert self.lib.etl_dec_arrow_list_values(self.a, c, self.host, C.byref(ch), C.byref(nv)) == 0
        return ch, nv.value

    def free(self):
        self.lib.etl_dec_arrow_free(self.a)


def _decode(w_tables, raw: bytes, stream: np.ndarray, oracle_mod):
    from etl_b200 import decoder
    orc = oracle_mod.Oracle()
    dec = decoder.Decoder(0)
    for tid, cols in w_tables.items():
        orc.put_table_schema(tid, cols)
        dec.put_table_schema(tid, cols)
    want = orc.decode(raw)
    st = decoder.Stager(stream.nbytes + 64, 2048)
    st.append_framed(stream)
    return dec, st, want


def check_numeric(e: Emitted, c: int, want_planes, rows):
    valid, offs, data = R.numeric_column(want_planes, rows, c)
    b = e.buffers(c)
    assert b["type"] == R.A_UTF8
    assert np.array_equal(_bits(b["validity"], e.n), valid), f"numeric validity of column {c}"
    assert np.array_equal(np.frombuffer(b["offsets"], np.int32).astype(np.int64), offs), f"numeric offsets of column {c}"
    assert b["data"] == data, f"numeric text of column {c}"


def check_list(e: Emitted, c: int, want_planes, rows, elem_kind: int):
    ct = R.KIND2ARROW[elem_kind]
    lvalid, loffs, cvalid, v = R.list_column(want_planes, rows, c, ct)
    b = e.buffers(c)
    assert b["type"] == R.A_LIST
    assert np.array_equal(_bits(b["validity"], e.n), lvalid), f"list validity of column {c}"
    assert np.array_equal(np.frombuffer(b["offsets"], np.int32).astype(np.int64), loffs), f"list offsets of column {c}"
    ch, nv = e.child(c)
    assert ch.arrow_type == ct and nv == int(loffs[-1]), (c, ch.arrow_type, ct, nv)
    cb = column_buffers(ch, nv, e.host)
    assert np.array_equal(_bits(cb["validity"], nv), cvalid), f"child validity of column {c}"
    if ct == R.A_BOOL:
        assert np.array_equal(_bits(cb["values"], nv), v)
    elif ct == R.A_UUID:
        assert cb["values"] == v
    elif ct in WIDTH:
        assert cb["values"] == np.ascontiguousarray(v).tobytes(), f"child values of column {c}"
    else:
        offs, data = v
        got = np.frombuffer(cb["offsets"], np.int32 if ct == R.A_UTF8 else np.int64).astype(np.int64)
        assert np.array_equal(got, offs), f"child offsets of column {c}"
        assert ch.data_bytes == len(data) and cb["data"] == data, f"child data of column {c}"
    return nv


SMALL = [("c2", 0.01), ("c3", 0.001), ("c4", 0.002), ("c5", 0.002)]


@pytest.mark.parametrize("name,scale", SMALL)
def test_flags0_is_emit_and_formatted_adds_numeric(lib, oracle_mod, name, scale):
    w = wl.make(name, scale, n_segments=1)
    stream, _ = w.generate()
    raw = stream.tobytes()
    dec, st, want = _decode(w.table_schemas(), raw, stream, oracle_mod)
    n_numeric = 0
    with dec.decode_input(st.view(), to_host=True) as bh:
        for kinds in (1, 3, 7):
            for si in range(min(len(want.schemas), 6)):
                base, ex0, fmt = Emitted(lib, bh, si, kinds, None), Emitted(lib, bh, si, kinds, 0), Emitted(lib, bh, si, kinds, FMT)
                assert base.n == ex0.n == fmt.n and base.n_cols == ex0.n_cols == fmt.n_cols
                assert np.array_equal(base.records(), ex0.records()) and np.array_equal(base.records(), fmt.records())
                rows = R.selected_rows(want, si, kinds)
                assert len(rows) == base.n
                kinds_of = want.schemas[si].col_kind
                for c in range(base.n_cols):
                    b0 = base.buffers(c)
                    assert ex0.buffers(c) == b0, (name, si, kinds, c)
                    k = int(kinds_of[c])
                    if b0["type"] != R.A_UNSUP:
                        assert fmt.buffers(c) == b0, (name, si, kinds, c)
                    elif k == 9:
                        check_numeric(fmt, c, want, rows)
                        n_numeric += 1
                    else:
                        assert R.formatted_type(k) == R.A_UNSUP, k
                        assert fmt.column(c).arrow_type == R.A_UNSUP, (c, k)   # json stays unsupported
                for e in (base, ex0, fmt):
                    e.free()
    st.close()
    dec.close()
    if name in ("c3", "c4"):
        assert n_numeric > 0


def _fixture_table():
    usable = [(oid, v) for oid, v, _ in ARRAY_COLS]
    cols = [dict(name="id", type_oid=20, pk=1, nullable=False, ordinal_position=1),
            dict(name="n", type_oid=1700, nullable=True, ordinal_position=2)]
    cols += [dict(name=f"a{oid}", type_oid=oid, nullable=True, ordinal_position=i + 3) for i, (oid, _) in enumerate(usable)]
    rel = pg.relation(95, "public", "arrays_full", "f", [(1 if c["name"] == "id" else 0, c["name"], c["type_oid"], -1) for c in cols])
    return usable, cols, rel


NUMS = ["1.50", "-0.0001", "NaN", "123456789012345678901234567890.123456789", "-Infinity", "0.000", "1e40", None]


def _fixture_stream(n_rows: int, bad_at=None):
    """every valid ARRAY_COLS spelling, in inserts, Full-image updates and deletes (replident full); bad_at: a row whose
    int4[] cell fails to parse (first_error in the middle of the batch)"""
    usable, cols, rel = _fixture_table()
    w = pg.StreamWriter()
    final = w.lsn + 10**9
    w.emit(pg.begin(final, w.clock, 1))
    w.emit(rel)
    prev = None
    for r in range(n_rows):
        row = [str(r), NUMS[r % len(NUMS)]] + [None if (r + j) % 11 == 10 else v[(r + j) % len(v)] for j, (_, v) in enumerate(usable)]
        if r == bad_at:
            row[2] = "{1,x}"
        if prev is not None and r % 5 == 4:
            w.emit(pg.delete(95, old=prev))
        elif prev is not None and r % 3 == 2:
            w.emit(pg.update(95, row, old=prev))
        else:
            w.emit(pg.insert(95, row))
        prev = row
    w.emit(pg.commit(0, final, final + 8, w.clock))
    raw = w.bytes()
    return {95: cols}, raw


def _check_all_columns(lib, bh, want, kinds, flags=FMT, to_host=1):
    e = Emitted(lib, bh, 0, kinds, flags, to_host)
    rows = R.selected_rows(want, 0, kinds)
    if want.first_error[0] is not None:
        rows = [(r, c0) for r, c0 in rows if r < want.first_error[0]]
    assert e.n == len(rows)
    assert np.array_equal(e.records(), np.array([r for r, _ in rows], np.uint64))
    kinds_of = want.schemas[0].col_kind
    n_lists = n_values = 0
    for c in range(e.n_cols):
        k = int(kinds_of[c])
        if k == 9:
            check_numeric(e, c, want, rows)
        elif k & R.K_ARRAY and (k & ~R.K_ARRAY) != R.K_JSON:
            n_values += check_list(e, c, want, rows, k & ~R.K_ARRAY)
            n_lists += 1
        elif k & R.K_ARRAY:
            assert e.column(c).arrow_type == R.A_UNSUP                         # json[] / jsonb[]
            assert lib.etl_dec_arrow_list_values(e.a, c, to_host, C.byref(abi.ArrowColumn()), None) == 1
    e.free()
    return e.n, n_lists, n_values


@pytest.mark.parametrize("kinds", [1, 7])
def test_array_fixture_lists(lib, oracle_mod, kinds):
    tables, raw = _fixture_stream(600)
    stream = np.frombuffer(raw, np.uint8)
    dec, st, want = _decode(tables, raw, stream, oracle_mod)
    assert want.first_error[0] is None, want.first_error
    with dec.decode_input(st.view(), to_host=True) as bh:
        n, n_lists, n_values = _check_all_columns(lib, bh, want, kinds)
    assert n > 300 and n_lists >= 14 and n_values > 1000, (n, n_lists, n_values)
    st.close()
    dec.close()


def test_first_error_keeps_valid_prefix(lib, oracle_mod):
    tables, raw = _fixture_stream(400, bad_at=250)
    stream = np.frombuffer(raw, np.uint8)
    dec, st, want = _decode(tables, raw, stream, oracle_mod)
    assert want.first_error[0] is not None
    with dec.decode_input(st.view(), to_host=True) as bh:
        s = bh.summary()
        assert s.first_error.record_index == want.first_error[0]
        n, n_lists, _ = _check_all_columns(lib, bh, want, 7)
    assert n == 250 and n_lists >= 14           # rows 0..249: every DML image before the failing insert is a row
    st.close()
    dec.close()


def test_array_workload_at_size(lib, oracle_mod):
    """the array workload at 200 k rows: multi-block scans, child bitmap words shared by neighbouring rows, rows of
    70 000 elements; the device image (to_host=0) and the host image (to_host=1) both checked"""
    stream, tables, stats = wl.array_stream(200_000)
    raw = stream.tobytes()
    dec, st, want = _decode(tables, raw, stream, oracle_mod)
    assert want.first_error[0] is None
    with dec.decode_input(st.view(), to_host=False) as bh:
        for to_host in (0, 1):
            n, n_lists, n_values = _check_all_columns(lib, bh, want, 7, to_host=to_host)
            assert n == stats["rows"] and n_lists == 6 and n_values > 10_000_000, (n, n_lists, n_values)
    st.close()
    dec.close()
