"""The BASELINE.json stream shapes C1..C5 (SURVEY.md §8d) as deterministic synthetic generators.

`make(name, scale)` returns a `Workload`: table schemas (what the reference's SchemaStore would
hold) + a segment generator backed by csrc/walgen.c.  Segments are independent sub-streams
(begin with the Relation messages of a connection epoch, end on a Commit), so a rank can generate
only the byte range it owns.  Host-side tooling; not on the decode path.
"""
from __future__ import annotations

import ctypes as C
import os
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import numpy as np

from . import build as _build

# generator kinds (csrc/walgen.c)
(SEQ_INT8, INT4_FULL, INT4_RANGE, INT8_FULL, BOOLG, TEXT_LOGNORMAL, TEXT_UNIFORM, TIMESTAMPTZG, NUMERICG, JSONBG,
 TOAST_TEXT, UUIDG, DATEG, FLOAT8G, BYTEAG, TIMESTAMPG, TIMEG, INT2G, FLOAT4G, OIDG) = range(1, 21)

OID = dict(bool=16, bytea=17, int8=20, int2=21, int4=23, text=25, oid=26, float4=700, float8=701, date=1082,
           time=1083, timestamp=1114, timestamptz=1184, numeric=1700, uuid=2950, jsonb=3802)


class _Col(C.Structure):
    _fields_ = [("type_oid", C.c_uint32), ("nullable", C.c_uint8), ("is_pk", C.c_uint8), ("gen", C.c_uint8),
                ("_pad", C.c_uint8), ("p0", C.c_uint32), ("p1", C.c_uint32), ("name", C.c_char * 32)]


class _Table(C.Structure):
    _fields_ = [("rel_id", C.c_uint32), ("replident", C.c_uint8), ("_pad", C.c_uint8), ("n_cols", C.c_uint16),
                ("cols", C.POINTER(_Col)), ("name", C.c_char * 32)]


class _Cfg(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("n_tables", C.c_uint32), ("_pad0", C.c_uint32), ("tables", C.POINTER(_Table)),
                ("n_msgs", C.c_uint64), ("target_bytes", C.c_uint64), ("pct_insert", C.c_uint32),
                ("pct_update", C.c_uint32), ("pct_delete", C.c_uint32), ("pct_key_change", C.c_uint32),
                ("tx_mean", C.c_uint32), ("tx_fixed", C.c_uint32), ("null_pct", C.c_uint32),
                ("nonascii_pct", C.c_uint32), ("toast_row_pct", C.c_uint32), ("toast_unchanged_pct", C.c_uint32),
                ("keepalive_every", C.c_uint32), ("schema_bump_ppm", C.c_uint32), ("relations_once", C.c_uint32),
                ("_pad1", C.c_uint32)]


class _Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("bytes", "frames", "dml", "inserts", "updates", "deletes", "txs", "relations", "cells")]


_lib = None


def _walgen():
    global _lib
    if _lib is None:
        L = C.CDLL(_build.WALGEN_LIB if os.path.exists(_build.WALGEN_LIB) else _build.build_walgen())
        L.wg_generate_segment.argtypes = [C.POINTER(_Cfg), C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(_Stats)]
        L.wg_generate_segment.restype = C.c_uint64
        _lib = L
    return _lib


@dataclass
class ColSpec:
    name: str
    typ: str
    gen: int
    nullable: bool = False
    pk: Optional[int] = None
    p0: int = 0
    p1: int = 0


@dataclass
class TableSpec:
    rel_id: int
    name: str
    replident: str
    cols: List[ColSpec]

    def column_schemas(self) -> List[dict]:
        """etl_column_schema list (ColumnSchema, etl-postgres/src/types/schema.rs:165-179)."""
        return [dict(name=c.name, type_oid=OID[c.typ], pk=c.pk, nullable=c.nullable, ordinal_position=i + 1)
                for i, c in enumerate(self.cols)]


@dataclass
class Workload:
    name: str
    tables: List[TableSpec]
    seed: int
    msgs_per_segment: int = 0
    bytes_per_segment: int = 0
    n_segments: int = 1
    mix: Tuple[int, int, int] = (10000, 0, 0)
    pct_key_change: int = 0
    tx_mean: int = 20
    tx_fixed: int = 0
    null_pct: int = 0
    nonascii_pct: int = 0
    toast_row_pct: int = 0
    toast_unchanged_pct: int = 0
    keepalive_every: int = 0
    schema_bump_ppm: int = 0
    relations_once: bool = False      # ONE stream: only segment 0 carries the Relation messages
    description: str = ""
    _keep: list = field(default_factory=list, repr=False)

    def _cfg(self) -> _Cfg:
        tabs = (_Table * len(self.tables))()
        for i, t in enumerate(self.tables):
            cols = (_Col * len(t.cols))()
            for j, c in enumerate(t.cols):
                cols[j].type_oid = OID[c.typ]
                cols[j].nullable = int(c.nullable)
                cols[j].is_pk = int(c.pk is not None)
                cols[j].gen = c.gen
                cols[j].p0, cols[j].p1 = c.p0, c.p1
                cols[j].name = c.name.encode()
            self._keep.append(cols)
            tabs[i].rel_id = t.rel_id
            tabs[i].replident = ord(t.replident)
            tabs[i].n_cols = len(t.cols)
            tabs[i].cols = cols
            tabs[i].name = t.name.encode()
        self._keep.append(tabs)
        cfg = _Cfg()
        cfg.seed = self.seed
        cfg.n_tables = len(self.tables)
        cfg.tables = tabs
        cfg.n_msgs = self.msgs_per_segment
        cfg.target_bytes = self.bytes_per_segment
        cfg.pct_insert, cfg.pct_update, cfg.pct_delete = self.mix
        cfg.pct_key_change = self.pct_key_change
        cfg.tx_mean, cfg.tx_fixed = self.tx_mean, self.tx_fixed
        cfg.null_pct, cfg.nonascii_pct = self.null_pct, self.nonascii_pct
        cfg.toast_row_pct, cfg.toast_unchanged_pct = self.toast_row_pct, self.toast_unchanged_pct
        cfg.keepalive_every, cfg.schema_bump_ppm = self.keepalive_every, self.schema_bump_ppm
        cfg.relations_once = int(self.relations_once)
        return cfg

    def segment_capacity(self) -> int:
        if self.bytes_per_segment:
            return int(self.bytes_per_segment * 1.05) + (4 << 20)
        per_msg = 64 + sum(5 + max(32, c.p1 if c.gen in (TEXT_LOGNORMAL, TEXT_UNIFORM) else 48) for c in max(self.tables, key=lambda t: len(t.cols)).cols) * 2
        return int(self.msgs_per_segment * per_msg * 1.2) + (1 << 20)

    def generate_segment(self, seg: int, out: Optional[np.ndarray] = None) -> Tuple[np.ndarray, dict]:
        cfg = self._cfg()
        cap = self.segment_capacity() if out is None else out.nbytes
        while True:
            buf = np.empty(cap, dtype=np.uint8) if out is None else out
            st = _Stats()
            n = _walgen().wg_generate_segment(C.byref(cfg), seg, buf.ctypes.data, buf.nbytes, C.byref(st))
            if n != 2**64 - 1:
                break
            if out is not None:
                raise RuntimeError("segment buffer too small")
            cap *= 2
        stats = {k: int(getattr(st, k)) for k, _ in _Stats._fields_}
        return buf[:n], stats

    def generate(self, segments: Optional[range] = None, threads: int = 8) -> Tuple[np.ndarray, dict]:
        """Concatenated stream of the given segments (default: all)."""
        segs = list(segments if segments is not None else range(self.n_segments))
        with ThreadPoolExecutor(max_workers=max(1, min(threads, len(segs)))) as ex:
            parts = list(ex.map(self.generate_segment, segs))
        total = {k: sum(p[1][k] for p in parts) for k in parts[0][1]}
        stream = parts[0][0] if len(parts) == 1 else np.concatenate([p[0] for p in parts])
        return stream, total

    def table_schemas(self) -> Dict[int, List[dict]]:
        return {t.rel_id: t.column_schemas() for t in self.tables}


def _c2_cols() -> List[ColSpec]:
    cols = [ColSpec("id", "int4", INT4_FULL, False, 1)]
    cols += [ColSpec(f"n{i}", "int4", INT4_FULL, True) for i in range(1, 5)]
    cols += [ColSpec(f"t{i}", "text", TEXT_LOGNORMAL, True, None, 16, 256) for i in range(5)]
    return cols


_C3_CYCLE = [("int4", INT4_FULL, 0, 0), ("int8", INT8_FULL, 0, 0), ("numeric", NUMERICG, 0, 0),
             ("text", TEXT_LOGNORMAL, 24, 256), ("timestamptz", TIMESTAMPTZG, 0, 0), ("jsonb", JSONBG, 0, 0)]


def _c3_cols(n: int = 100) -> List[ColSpec]:
    cols = []
    for i in range(n):
        typ, gen, p0, p1 = _C3_CYCLE[i % 6]
        cols.append(ColSpec(f"c{i}", typ, gen, i != 0, 1 if i == 0 else None, p0, p1))
    return cols


def _c4_tables(seed: int) -> List[TableSpec]:
    rng = np.random.Generator(np.random.PCG64(seed))
    pool = _C3_CYCLE + [("bool", BOOLG, 0, 0), ("uuid", UUIDG, 0, 0), ("date", DATEG, 0, 0), ("float8", FLOAT8G, 0, 0)]
    tabs = []
    for k in range(64):
        ncols = int(rng.integers(4, 25))
        cols = [ColSpec("id", "int8", SEQ_INT8, False, 1)]
        for j in range(1, ncols):
            typ, gen, p0, p1 = pool[int(rng.integers(0, len(pool)))]
            cols.append(ColSpec(f"c{j}", typ, gen, True, None, p0, p1))
        tabs.append(TableSpec(16384 + k, f"t{k}", "f" if k % 4 == 3 else "d", cols))
    return tabs


def relation_preamble(stream: np.ndarray, n_tables: int) -> np.ndarray:
    """Prefix of a stream up to the first Commit after every table's Relation message has been seen: decoding it
    gives a fresh decoder the replicated-schema state the rest of a `relations_once` stream relies on."""
    pos, seen, n = 0, 0, int(stream.nbytes)
    while pos + 5 <= n:
        fl = int.from_bytes(stream[pos + 1:pos + 5].tobytes(), "big")
        tag = int(stream[pos + 30]) if stream[pos + 5] == ord("w") else 0
        pos += 1 + fl
        if tag == ord("R"):
            seen += 1
        elif tag == ord("C") and seen >= n_tables:
            return stream[:pos]
    return stream


def mid_transaction_cut(stream: np.ndarray, target: int) -> int:
    """Offset of the first frame at or after `target` that is a DML record preceded by a DML record — a cut there
    falls inside a transaction (bench.py --scaling strong puts the shard seams at such offsets)."""
    pos, prev, n = 0, 0, int(stream.nbytes)
    dml = (ord("I"), ord("U"), ord("D"))
    while pos + 5 <= n:
        fl = int.from_bytes(stream[pos + 1:pos + 5].tobytes(), "big")
        tag = int(stream[pos + 30]) if stream[pos + 5] == ord("w") else 0
        if pos >= target and tag in dml and prev in dml:
            return pos
        prev = tag
        pos += 1 + fl
    return 0


def make(name: str, scale: float = 1.0, n_segments: Optional[int] = None, one_stream: bool = False) -> Workload:
    """name ∈ {c1, c2, c3, c4, c5}.  `scale` multiplies the message count / byte size of the named
    configuration (1.0 = the BASELINE.json size)."""
    name = name.lower()
    if name == "c1":
        cols = [ColSpec("id", "int8", SEQ_INT8, False, 1), ColSpec("name", "text", TEXT_UNIFORM, True, None, 8, 24),
                ColSpec("age", "int4", INT4_RANGE, True, None, 0, 120), ColSpec("active", "bool", BOOLG, True),
                ColSpec("created", "timestamptz", TIMESTAMPTZG, True)]
        segs = n_segments or 1
        return Workload("c1", [TableSpec(16384, "users", "d", cols)], 0xE7100001, msgs_per_segment=max(1, int(10_000 * scale / segs)),
                        n_segments=segs, mix=(10000, 0, 0), tx_fixed=100,
                        description="single-table 5-col INSERT-only pgoutput stream, 10k msgs")
    if name == "c2":
        segs = n_segments or 8
        return Workload("c2", [TableSpec(16384, "orders", "d", _c2_cols())], 0xE7100002,
                        msgs_per_segment=max(1, int(1_000_000 * scale / segs)), n_segments=segs, mix=(5000, 3500, 1500),
                        pct_key_change=1000, tx_mean=20, null_pct=500, nonascii_pct=200,
                        description="mixed Insert/Update/Delete, 10-col int4+text table, 1M msgs")
    if name == "c3":
        segs = n_segments or 8
        return Workload("c3", [TableSpec(16384, "wide", "f", _c3_cols())], 0xE7100003,
                        msgs_per_segment=max(1, int(1_000_000 * scale / segs)), n_segments=segs, mix=(7000, 3000, 0),
                        tx_mean=20, null_pct=500, nonascii_pct=200,
                        description="wide 100-col table (int4/int8/numeric/text/timestamptz/jsonb), 1M msgs")
    if name == "c4":
        segs = n_segments or 16
        return Workload("c4", _c4_tables(0xE7100004), 0xE7100004, msgs_per_segment=max(1, int(10_000_000 * scale / segs)),
                        n_segments=segs, mix=(5000, 3500, 1500), pct_key_change=1000, tx_mean=20, null_pct=500,
                        nonascii_pct=200, schema_bump_ppm=100,
                        description="64-table publication with interleaved Relation/schema msgs, 10M msgs")
    if name == "c5":
        segs = n_segments or 64
        cols_d = _c2_cols() + [ColSpec("doc", "text", TOAST_TEXT, True, None, 2048, 65536)]
        cols_f = _c2_cols() + [ColSpec("doc", "text", TOAST_TEXT, True, None, 2048, 65536)]
        total = int((10 << 30) * scale)
        return Workload("c5", [TableSpec(16384, "docs_default", "d", cols_d), TableSpec(16385, "docs_full", "f", cols_f)],
                        0xE7100005, bytes_per_segment=max(1 << 16, total // segs), n_segments=segs, mix=(5000, 3500, 1500),
                        pct_key_change=1000, tx_mean=20, null_pct=500, nonascii_pct=200, toast_row_pct=500,
                        toast_unchanged_pct=6000, keepalive_every=4096, relations_once=one_stream,
                        description="10 GiB synthetic pgoutput buffer, mixed ops + TOASTed text")
    raise ValueError(f"unknown workload {name}")


# ---- array-heavy stream (none of C1..C5 has array columns): the columnar emitter's List columns at size
ARRAY_TABLE_COLS = [("id", 20), ("a_int4", 1007), ("a_text", 1009), ("a_numeric", 1231), ("a_uuid", 2951), ("a_bool", 1000),
                    ("a_tstz", 1185)]
HUGE_ARRAY_ELEMS = 70_000


def _element_pools(rng: np.random.Generator, n: int = 4096) -> List[List[str]]:
    """n spellings per array column (NULL elements included), in ARRAY_TABLE_COLS order after id"""
    def nulls(vals):
        return [("NULL" if rng.random() < 0.06 else v) for v in vals]
    i4 = [str(int(x)) for x in rng.integers(-2**31, 2**31, n)]
    words = ["alpha", "b c", "quote\\\"d", "comma,here", "é✓", "", "NULL", "back\\\\slash", "x" * 40, "tab\tbed"]
    txt = ['"' + words[int(k)] + str(int(j)) + '"' if k < len(words) else str(int(j)) for k, j in zip(rng.integers(0, 14, n), rng.integers(0, 10**6, n))]
    num_forms = ["%d", "%d.%d", "-%d.%d", "0.000%d", "%de5", "%d.%de-7"]
    num = []
    for k, a, b in zip(rng.integers(0, len(num_forms) + 1, n), rng.integers(0, 10**9, n), rng.integers(0, 10**6, n)):
        if k == len(num_forms):
            num.append(["NaN", "Infinity", "-Infinity", "0.000", "-0"][int(a) % 5])
        else:
            f = num_forms[int(k)]
            num.append(f % ((int(a),) if f.count("%") == 1 else (int(a), int(b))))
    uu = ["%08x-%04x-%04x-%04x-%012x" % (int(a) & 0xFFFFFFFF, int(b) & 0xFFFF, (int(a) >> 40) & 0xFFFF, (int(b) >> 20) & 0xFFFF, int(a) * 7919 & 0xFFFFFFFFFFFF)
          for a, b in zip(rng.integers(0, 2**62, n), rng.integers(0, 2**62, n))]
    bo = ["t" if x else "f" for x in rng.integers(0, 2, n)]
    ts = ['"%04d-%02d-%02d %02d:%02d:%02d%s%s"' % (1990 + int(y) % 60, 1 + int(y) % 12, 1 + int(y) % 28, int(s) % 24, int(s) % 60, int(s) // 60 % 60,
                                                 "." + str(int(s) % 1000000) if int(s) % 3 == 0 else "", ["+00", "-07", "+05:30"][int(s) % 3])
          for y, s in zip(rng.integers(0, 10**6, n), rng.integers(0, 10**9, n))]
    return [nulls(p) for p in (i4, txt, num, uu, bo, ts)]


def array_stream(n_rows: int, seed: int = 0xE71000A0) -> Tuple[np.ndarray, Dict[int, List[dict]], dict]:
    """Deterministic pgoutput stream of one 'replident full' table with int4[] / text[] / numeric[] / uuid[] / bool[] /
    timestamptz[] columns: inserts, Full-image updates and deletes (about 70 / 20 / 10 %) over n_rows row images.
    Cells are NULL (6 %), empty arrays (8 %), 1-8 elements (mostly) or 9-400 elements (3 %); elements are NULL about
    6 % of the time; rows 1000 and n_rows // 2 (when they exist) carry HUGE_ARRAY_ELEMS-element int4[] and numeric[]
    cells.  Returns (stream, table schemas, stats)."""
    from . import pgoutput as pg
    rng = np.random.Generator(np.random.PCG64(seed))
    pools = _element_pools(rng)
    dbl = [p + p for p in pools]
    npool = len(pools[0])
    n_acols = len(pools)
    u = rng.random((n_rows, n_acols))
    lens = np.where(u < 0.06, -1, np.where(u < 0.14, 0, np.where(u < 0.97, rng.integers(1, 9, (n_rows, n_acols)),
                                                                rng.integers(9, 401, (n_rows, n_acols)))))
    starts = rng.integers(0, npool, (n_rows, n_acols))
    ops = rng.random(n_rows)
    huge = {r for r in (1000, n_rows // 2) if r < n_rows}

    def cell(r, j):
        n = int(lens[r, j])
        if r in huge and j in (0, 2):
            n = HUGE_ARRAY_ELEMS
        if n < 0:
            return None
        s, p = int(starts[r, j]), dbl[j]
        if n <= npool:
            return "{" + ",".join(p[s:s + n]) + "}"
        return "{" + ",".join(p[(s + k) % npool] for k in range(n)) + "}"

    rel_id = 16500
    cols = [dict(name=nm, type_oid=oid, pk=1 if nm == "id" else None, nullable=nm != "id", ordinal_position=i + 1)
            for i, (nm, oid) in enumerate(ARRAY_TABLE_COLS)]
    w = pg.StreamWriter()
    xid, n_ins, n_upd, n_del, prev = 1, 0, 0, 0, None
    final = w.lsn + 10**9           # Begin's final_lsn = its Commit's commit_lsn
    w.emit(pg.begin(final, w.clock, xid))
    w.emit(pg.relation(rel_id, "public", "arrays", "f", [(1 if nm == "id" else 0, nm, oid, -1) for nm, oid in ARRAY_TABLE_COLS]))
    for r in range(n_rows):
        row = [str(r)] + [cell(r, j) for j in range(n_acols)]
        if prev is not None and ops[r] >= 0.9:
            w.emit(pg.delete(rel_id, old=prev)); n_del += 1
        elif prev is not None and ops[r] >= 0.7:
            w.emit(pg.update(rel_id, row, old=prev)); n_upd += 1
        else:
            w.emit(pg.insert(rel_id, row)); n_ins += 1
        prev = row
        if r % 50 == 49:
            w.emit(pg.commit(0, final, final + 8, w.clock))
            xid += 1
            final += 10**9
            w.emit(pg.begin(final, w.clock, xid))
    w.emit(pg.commit(0, final, final + 8, w.clock))
    stream = np.frombuffer(w.bytes(), dtype=np.uint8)
    return stream, {rel_id: cols}, dict(bytes=int(stream.nbytes), rows=n_rows, inserts=n_ins, updates=n_upd, deletes=n_del)
