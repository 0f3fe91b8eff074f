"""Time the columnar emitter (etl_dec_arrow_emit_ex, to_host=0) with flags 0 and with ETL_ARROW_FORMATTED, alternately in
one process, on a decoded batch that stays resident: C3 (numeric columns) and the array workload (List columns).

    python tools/bench_arrow.py [--c3-scale 1.0] [--array-rows 400000] [--iters 30] [--warmup 5] [--out FILE]

Each call is bracketed by CUDA events on the legacy default stream (the emitter runs on the per-thread default stream,
which is ordered with it), so a time covers the whole call: row selection, both passes, its allocations and its two
host synchronisations.  The median of --iters calls after --warmup calls is reported.

bytes = what the emitter has to move: the output buffers it returns (validity, values, offsets, data, list children)
plus what it reads for them: 13 bytes of cell plane (tag, val, aux) per row and emitted column, 16 bytes per list
element record, and the var-width payload, counted as equal to the output data bytes.  GB/s = bytes / median time.
Prints one JSON line with the card name and power limit read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from etl_b200 import abi, decoder, workloads as wl  # noqa: E402

WIDTH = {abi.ARROW_INT32: 4, abi.ARROW_DATE32: 4, abi.ARROW_FLOAT32: 4, abi.ARROW_INT64: 8, abi.ARROW_FLOAT64: 8,
         abi.ARROW_TIME64_US: 8, abi.ARROW_TIMESTAMP_US: 8, abi.ARROW_TIMESTAMPTZ_US: 8, abi.ARROW_UUID: 16}


def _column_bytes(at, n, data_bytes):
    """(output bytes, payload bytes) of a column of n entries"""
    out = (n + 7) // 8
    if at == abi.ARROW_BOOLEAN:
        out += (n + 7) // 8
    elif at in WIDTH:
        out += n * WIDTH[at]
    else:
        out += (n + 1) * (8 if at == abi.ARROW_LARGE_BINARY else 4) + data_bytes
    return out, data_bytes


def traffic(lib, a, n_rows):
    out = 8 * n_rows                           # row_records
    read = 8 * n_rows                          # row → first cell
    for c in range(lib.etl_dec_arrow_cols(a)):
        col = abi.ArrowColumn()
        lib.etl_dec_arrow_column(a, c, 0, C.byref(col))
        if col.arrow_type == abi.ARROW_UNSUPPORTED:
            continue
        read += 13 * n_rows
        if col.arrow_type == abi.ARROW_LIST:
            ch, nv = abi.ArrowColumn(), C.c_uint64()
            lib.etl_dec_arrow_list_values(a, c, 0, C.byref(ch), C.byref(nv))
            o, p = _column_bytes(abi.ARROW_LIST, n_rows, 0)
            co, cp = _column_bytes(ch.arrow_type, nv.value, ch.data_bytes)
            out += o + co
            read += 16 * nv.value + cp
        else:
            o, p = _column_bytes(col.arrow_type, n_rows, col.data_bytes)
            out += o
            read += p
    return out, read


def bench_batch(lib, bh, schema_index, kinds, iters, warmup):
    import torch
    res = {}
    times = {0: [], abi.ARROW_FORMATTED: []}
    a = C.c_void_p()
    for it in range(warmup + iters):
        for flags in (0, abi.ARROW_FORMATTED):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            s.record(torch.cuda.default_stream())
            rc = lib.etl_dec_arrow_emit_ex(bh._h, schema_index, kinds, flags, 0, C.byref(a))
            e.record(torch.cuda.default_stream())
            e.synchronize()
            assert rc == 0, rc
            if it >= warmup:
                times[flags].append(s.elapsed_time(e))
            if it == warmup + iters - 1:
                n = lib.etl_dec_arrow_rows(a)
                out, read = traffic(lib, a, n)
                res[flags] = dict(rows=int(n), out_bytes=int(out), bytes=int(out + read))
            lib.etl_dec_arrow_free(a)
    line = {}
    for flags, name in ((0, "flags0"), (abi.ARROW_FORMATTED, "formatted")):
        ms = float(np.median(times[flags]))
        r = res[flags]
        line[name] = dict(rows=r["rows"], out_bytes=r["out_bytes"], bytes_read_written=r["bytes"], ms=round(ms, 4),
                          ms_min=round(float(np.min(times[flags])), 4), GBps=round(r["bytes"] / ms / 1e6, 2))
    return line


def run(lib, stream, tables, kinds, iters, warmup):
    dec = decoder.Decoder(0)
    for tid, cols in tables.items():
        dec.put_table_schema(tid, cols)
    st = decoder.Stager(stream.nbytes + 64, 2048)
    st.append_framed(stream)
    try:
        with dec.decode_input(st.view(), to_host=False) as bh:
            s = bh.summary()
            assert s.first_error.record_index == 2**64 - 1, "the stream must decode cleanly"
            out = bench_batch(lib, bh, 0, kinds, iters, warmup)
            out["stream_bytes"] = int(stream.nbytes)
            return out
    finally:
        st.close()
        dec.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--c3-scale", type=float, default=1.0)
    ap.add_argument("--array-rows", type=int, default=400_000)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_arrow.py needs a CUDA device")
    lib = abi.load()
    line = {"tool": "bench_arrow", "iters": a.iters, "warmup": a.warmup, "row_kinds": 7, "to_host": 0}
    w = wl.make("c3", a.c3_scale)
    stream, _ = w.generate()
    line["c3"] = dict(scale=a.c3_scale, **run(lib, stream, w.table_schemas(), 7, a.iters, a.warmup))
    del stream
    stream, tables, stats = wl.array_stream(a.array_rows)
    line["arrays"] = dict(array_rows=a.array_rows, **run(lib, stream, tables, 7, a.iters, a.warmup))
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True)
    name, limit = (q.stdout.strip().splitlines()[0].split(", ") + [""])[:2] if q.returncode == 0 and q.stdout.strip() else (torch.cuda.get_device_name(0), "unknown")
    line["gpu"], line["power_limit"] = name, limit
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
