#!/usr/bin/env python
"""bench.py — WAL GB/s and events/s of the batched pgoutput decode path on N B200s of one node.

  python bench.py --gpus 1 --steps 5 --warmup 3                      (driver launches N>1 via torchrun)
  python bench.py --impl reference ...                                (the CPU path on the host cores)

A "step" is one pass of the decode hot path over the staged synthetic stream:
  value  — stream + anchor index already resident in HBM, results left in HBM (CUDA-event timed)
  e2e    — the same call through the C ABI with HOST (pinned) buffers: H2D of the stream and its
           anchor index, the kernels, and the D2H of every result plane are inside the timed region
Workload (default c5): BASELINE.json configs[4], "10 GiB synthetic pgoutput buffer, mixed ops + TOASTed text" —
ONE stream (its Relation messages appear once, in the first megabytes).  With N GPUs the stream is cut into N
byte ranges at record starts that fall INSIDE transactions (strong scaling: total work fixed, default); the
library exchanges the Relation frames and the 64-byte seam summaries over NCCL (etl_dec_decode_sharded) — no host
round trip between the index pass and the record pass.  `--scaling weak` gives every GPU a full 10 GiB range.
Inputs are far larger than L2 (126 MB), so no flush is needed between steps.

After the timed legs, and outside them, rank 0 of a single-GPU run also (a) checks the CUDA path against the CPU
oracle on EVERY segment of c5 and of c2 / c3 / c4 at their BASELINE sizes (canonical plane digests), (b) times
c2 / c3 / c4 the same way as the headline and (c) times back-to-back decodes at the reference's own batch size
(BatchConfig::DEFAULT_MAX_BYTES = 8 MiB, etl-config/src/shared/pipeline.rs:54-68) with carry-in/out chaining.
All of it goes into the ONE JSON line.

`--dump-outputs DIR` writes a seeded sample of the planes the last timed step decoded (sample_outputs) as float64 .npy
files.  The workloads are generated from fixed seeds, so two builds run with the same arguments can be compared output
for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GIB = 1 << 30
NO_ERROR = 2**64 - 1
DATA_ERRORS = []      # first_error of any timed / warm-up decode: a clean synthetic stream must not produce one


_REAL_STDOUT = None


def emit_line(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c5", choices=["c1", "c2", "c3", "c4", "c5"])
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the BASELINE.json size of the workload")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="N>1: strong = ONE stream of the BASELINE size cut into N byte ranges; weak = a full-size range per GPU")
    ap.add_argument("--stride", type=int, default=2048, help="anchor stride of the staged stream")
    ap.add_argument("--cpu-sample-gib", type=float, default=10.0, help="bounded sample for the CPU baseline")
    ap.add_argument("--gen-threads", type=int, default=0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the post-timing legs (parity at size, c2/c3/c4, 8 MiB batches)")
    ap.add_argument("--extras-scale", type=float, default=1.0, help="scale of the c2/c3/c4 legs (1.0 = BASELINE sizes)")
    ap.add_argument("--batch-calls", type=int, default=1000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed sample of the planes the last timed step decoded to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the planes of the CUDA path (--impl ours)")
    return args


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, STREAM-style copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def host_cores():
    """(cores the process may run on, cores of the box)."""
    try:
        usable = len(os.sched_getaffinity(0))
    except Exception:
        usable = os.cpu_count() or 1
    return usable, (os.cpu_count() or usable)


class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU while a timed region runs."""

    def __init__(self, index: int):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv = None

    def _run(self):
        nv = self._nv
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
                 0x80: "hw_power_brake_slowdown"}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop.wait(0.002)

    def __enter__(self):
        if self._nv:
            self._stop.clear()
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        return self

    def __exit__(self, *a):
        if self._t:
            self._stop.set()
            self._t.join()

    def report(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def generate_segments(w, segs, threads):
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=max(1, min(threads, len(segs)))) as ex:
        parts = list(ex.map(w.generate_segment, segs))
    return [p[0] for p in parts], [p[1] for p in parts]


# ------------------------------------------------------------------------------------------------ CPU side (oracle)
def _new_oracle(w, preamble):
    from oracle import pyoracle
    o = pyoracle.Oracle()
    for tid, cols in w.table_schemas().items():
        o.put_table_schema(tid, cols)
    if preamble is not None:                          # ONE stream: the Relation messages live in its first bytes
        b = o.decode_raw(preamble)
        o.free(b)
    return o


def cpu_decode_segments(w, seg_arrays, threads, preamble=None, digests=False):
    """Decode independent pieces with the CPU oracle on `threads` host threads (each worker owns an oracle context
    that has seen the stream's Relation preamble).  Returns (seconds, records[, digests])."""
    from concurrent.futures import ThreadPoolExecutor

    def work(idx):
        o = _new_oracle(w, preamble)
        n, out = 0, {}
        for i in idx:
            if digests:
                d, nr, fe = o.digest(seg_arrays[i])
                assert fe is None
                out[i] = (d, nr)
                n += nr
            else:
                b = o.decode_raw(seg_arrays[i])
                assert b.first_error.record_index == NO_ERROR
                n += b.n_records
                o.free(b)
        return n, out

    threads = max(1, min(threads, len(seg_arrays)))
    chunks = [list(range(t, len(seg_arrays), threads)) for t in range(threads)]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:
        res = list(ex.map(work, chunks))
    dt = time.perf_counter() - t0
    recs = sum(r[0] for r in res)
    if digests:
        merged = {}
        for r in res:
            merged.update(r[1])
        return dt, recs, merged
    return dt, recs


def run_reference(args, rank, world):
    """The reference arm: the CPU implementation of the path (oracle port — the Rust reference cannot be built in
    this image) on every host core this process may use, on a bounded sample of the same workload."""
    if rank != 0:
        return
    from etl_b200 import workloads as wl
    w = wl.make(args.workload, args.scale, one_stream=(args.workload == "c5"))
    usable, box = host_cores()
    seg_bytes = w.bytes_per_segment or (w.segment_capacity() // 2)
    n_sample = max(1, min(w.n_segments, max(usable, int(args.cpu_sample_gib * 4 * GIB / max(seg_bytes, 1)))))
    n_sample = min(n_sample, w.n_segments)
    arrays, stats = generate_segments(w, list(range(n_sample)), args.gen_threads or usable)
    pre = wl.relation_preamble(arrays[0], len(w.tables)) if w.relations_once else None
    total_bytes = sum(a.nbytes for a in arrays)
    frames = sum(s["frames"] for s in stats)
    threads = min(usable, n_sample)
    for _ in range(max(1, min(args.warmup, 1))):
        cpu_decode_segments(w, arrays, threads, pre)
    secs = 0.0
    for _ in range(args.steps):
        dt, _ = cpu_decode_segments(w, arrays, threads, pre)
        secs += dt
    ms = secs / args.steps * 1e3
    val = total_bytes / (secs / args.steps) / 1e9
    sample = (f"{n_sample} of {w.n_segments} segments ({total_bytes / GIB:.2f} GiB) of workload {w.name}, {threads} threads "
              f"(box: {box} cores, {usable} usable by this process)")
    line = {"impl": "reference", "metric": "wal_decode_throughput", "value": val, "unit": "GB/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": args.scaling if args.gpus > 1 else "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "events_per_s": frames / (secs / args.steps),
            "config": {"workload": f"{w.name}: {w.description}", "scale": args.scale},
            "cpu_baseline": {"value": val, "unit": "GB/s", "cores": threads, "box_cores": box, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit_line(line)


# ------------------------------------------------------------------------------------------------ GPU side
class Staged:
    """One staged stream: pinned host copy (Stager) + resident device copy + anchors."""

    def __init__(self, pieces, stride, dev, torch):
        from etl_b200 import abi, decoder
        self.nbytes = int(sum(p.nbytes for p in pieces))
        self.stager = decoder.Stager(max(self.nbytes, 1), stride)
        for p in pieces:
            if p.nbytes:
                self.stager.append_framed(p)
        v = self.stager.view()
        self.n_anchors = int(v.n_anchors)
        host = self.stager.host_array()
        self.d_stream = torch.empty(max(self.nbytes, 1) + 64, dtype=torch.uint8, device=dev)
        self.d_stream[self.nbytes:].zero_()
        if self.nbytes:
            self.d_stream[:self.nbytes].copy_(torch.from_numpy(host))
        an = np.ctypeslib.as_array(C.cast(v.anchors, abi.u64p), shape=(self.n_anchors,)) if self.n_anchors else np.zeros(0, np.uint64)
        self.d_anchors = torch.from_numpy(np.concatenate([an, np.array([self.nbytes], dtype=np.uint64)]).view(np.int64)).to(dev)

    def view(self, resident: bool, carry=None):
        inp = self.stager.view()
        if resident:
            inp.dev_buf = self.d_stream.data_ptr()
            inp.dev_anchors = self.d_anchors.data_ptr()
        if carry:
            inp.carry_in.in_tx, inp.carry_in.final_lsn, inp.carry_in.next_tx_ordinal = int(carry[0]), carry[1], carry[2]
        return inp

    def close(self):
        self.stager.close()
        self.d_stream = self.d_anchors = None


def decode_once(dec, st, resident, sharded, carry=None, timing=True):
    inp = st.view(resident, carry)
    bh = dec.decode_sharded(inp, to_host=not resident, timing=timing) if sharded else dec.decode_input(inp, to_host=not resident, timing=timing)
    s = bh.summary()
    if s.first_error.record_index != NO_ERROR:
        # never raise between collectives (the other ranks would wait for this one for ever): remember it, fail the line later
        DATA_ERRORS.append((int(s.first_error.record_index), int(s.first_error.seq), int(s.first_error.code)))
    return bh, s


# ------------------------------------------------------------------------------------------------ --dump-outputs
DUMP_BYTES = 64 << 20                 # all files of one dump together
DUMP_RECORDS, DUMP_CELLS = 1 << 17, 1 << 19
DUMP_SEED = 0xD0D0
PLANE_DTYPES = {"rec_off": np.uint64, "rec_kind": np.uint8, "rec_flags": np.uint8, "rec_rel": np.uint32, "rec_schema": np.int32,
                "rec_start_lsn": np.uint64, "rec_commit_lsn": np.uint64, "rec_tx_ordinal": np.uint64, "rec_cell_base": np.uint64,
                "rec_tuple_bytes": np.uint32, "rec_heap_hint": np.uint32, "cell_tag": np.uint8, "cell_val": np.uint64,
                "cell_aux": np.uint32}
SUMMARY_FIELDS = ("n_records", "n_cells", "first_error_record", "first_error_seq", "first_error_code", "first_error_kind",
                  "carry_in_tx", "carry_final_lsn", "carry_next_tx_ordinal", "insert_bytes", "update_bytes", "delete_bytes", "n_events")


def _halves(a):
    """Unsigned 64-bit integers as two float64 arrays that hold them exactly: (high 32 bits, low 32 bits)."""
    a = np.asarray(a, dtype=np.uint64)
    return (a >> np.uint64(32)).astype(np.float64), (a & np.uint64(0xFFFFFFFF)).astype(np.float64)


def sample_outputs(summary, schemas, fetch, heap, share=1.0):
    """The outputs of one decoded batch as float64 arrays, keyed by file name.

    summary: SUMMARY_FIELDS -> unsigned int (first_error_record 2**64 - 1: no error); schemas: objects with table_id,
    n_cols, n_identity, snapshot_id, effective_off; fetch(plane, idx): the named plane of PLANE_DTYPES at the indices
    idx; heap(): the batch's heap as bytes.
    Records and cells are sampled from a fixed seed, so two batches with the same record and cell counts are sampled at
    the same indices (record_sample, cell_sample).  64-bit planes and the summary are split into exact 32-bit halves.
    A numeric, uuid, bytes or array cell points into the heap, and where a value lands there depends on the order in
    which warps reserve space: its cell_val is written as 0 and cell_var_crc32 holds the CRC-32 of the value it points
    to (0 for every other cell).  share scales the sample (one rank's part of a multi-GPU dump)."""
    import zlib
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from canon import _VAR_TAGS, decode_cell
    n, m = int(summary["n_records"]), int(summary["n_cells"])
    rng = np.random.default_rng(DUMP_SEED)
    rec_idx = np.sort(rng.choice(n, size=min(n, int(DUMP_RECORDS * share)), replace=False)).astype(np.int64)
    cell_idx = np.sort(rng.choice(m, size=min(m, int(DUMP_CELLS * share)), replace=False)).astype(np.int64)
    planes = {}
    for name, dt in PLANE_DTYPES.items():
        idx = rec_idx if name.startswith("rec_") else cell_idx
        planes[name] = np.asarray(fetch(name, idx), dtype=dt) if len(idx) else np.zeros(0, dt)
    var_cells = np.isin(planes["cell_tag"], _VAR_TAGS)
    crc = np.zeros(len(cell_idx), dtype=np.float64)
    if var_cells.any():
        h = heap()
        crc[var_cells] = [zlib.crc32(repr(decode_cell(int(t), int(v), int(a), b"", h, strict=True)).encode())
                          for t, v, a in zip(planes["cell_tag"][var_cells], planes["cell_val"][var_cells], planes["cell_aux"][var_cells])]
    planes["cell_val"] = np.where(var_cells, np.uint64(0), planes["cell_val"])
    out = {"summary": np.stack(_halves([summary[f] for f in SUMMARY_FIELDS]), axis=1),
           "schemas": np.array([(s.table_id, s.n_cols, s.n_identity, s.snapshot_id, s.effective_off) for s in schemas],
                               dtype=np.float64).reshape(-1, 5),
           "record_sample": rec_idx.astype(np.float64), "cell_sample": cell_idx.astype(np.float64), "cell_var_crc32": crc}
    for name, vals in planes.items():
        if vals.dtype == np.uint64:
            out[name + "_hi"], out[name + "_lo"] = _halves(vals)
        else:
            out[name] = vals.astype(np.float64)
    return out


class _DevicePlane:
    """A device array of the library, seen by torch.as_tensor through the CUDA array interface (no copy)."""

    def __init__(self, ptr, count, dtype):
        self.__cuda_array_interface__ = {"shape": (int(count),), "typestr": np.dtype(dtype).str, "data": (int(ptr), False),
                                         "version": 2}


def dump_outputs(torch, dev, bh, out_dir, prefix="", share=1.0):
    """--dump-outputs for one decoded batch whose planes are resident in HBM: the sampled elements are gathered on the
    device and copied to the host, the heap only if a sampled cell points into it."""
    p, s = bh.planes(False), bh.summary()
    n = int(p.n_records)
    counts = {"rec_cell_base": n + 1, "cell_tag": int(p.n_cells), "cell_val": int(p.n_cells), "cell_aux": int(p.n_cells)}

    def fetch(name, idx):
        dt = np.dtype(PLANE_DTYPES[name])
        signed = np.dtype(f"i{dt.itemsize}") if dt.itemsize > 1 else dt     # torch gathers signed 32/64-bit integers
        t = torch.as_tensor(_DevicePlane(getattr(p, name), counts.get(name, n), signed), device=dev)
        return t[torch.from_numpy(idx).to(dev)].cpu().numpy().view(dt)

    def heap():
        nb = int(p.heap_bytes)
        return torch.as_tensor(_DevicePlane(p.heap, nb, np.uint8), device=dev).cpu().numpy().tobytes() if nb else b""

    fe = s.first_error
    summary = dict(n_records=n, n_cells=int(p.n_cells), first_error_record=int(fe.record_index), first_error_seq=int(fe.seq),
                   first_error_code=int(fe.code), first_error_kind=int(fe.kind), carry_in_tx=int(s.carry_out.in_tx), carry_final_lsn=int(s.carry_out.final_lsn),
                   carry_next_tx_ordinal=int(s.carry_out.next_tx_ordinal), insert_bytes=int(s.insert_bytes),
                   update_bytes=int(s.update_bytes), delete_bytes=int(s.delete_bytes), n_events=int(s.n_events))
    arrays = sample_outputs(summary, bh.schemas(), fetch, heap, share)
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_BYTES * share, f"--dump-outputs would write {total} bytes"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{prefix}{name}.npy"), a)


def time_steps(torch, dist, dec, st, resident, sharded, steps, dev, world, on_last=None):
    """K decode calls as a production caller makes them (ETL_DECODE_NO_TIMING: no per-kernel event queries on the host),
    bracketed by barrier + synchronize and CUDA events, max over ranks.  The per-kernel breakdown comes from two more calls
    with the summary timings on, after the timed region.  on_last(batch), if given, sees the last timed call's batch after
    the timed region, before it is freed."""
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    rows, launches, last = [], 0, None
    e0.record()
    for i in range(steps):
        bh, s = decode_once(dec, st, resident, sharded, timing=False)
        launches += s.gpu_launches
        last = dict(h2d=int(s.h2d_bytes), d2h=int(s.d2h_bytes), span_bytes=int(s.span_bytes), n_records=int(bh.planes(False).n_records),
                    n_cells=int(bh.planes(False).n_cells))
        if on_last is None or i < steps - 1:
            bh.free()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    if on_last is not None:
        on_last(bh)
        bh.free()
    for _ in range(2):                                   # every rank (the sharded call is collective)
        bh, s = decode_once(dec, st, resident, sharded, timing=True)
        rows.append((s.index_ms, s.frames_ms, s.walk_ms, s.cells_ms, s.spans_ms, s.kernel_ms, s.long_ms))
        bh.free()
    return float(ms.item()), np.mean(np.array(rows, dtype=np.float64), axis=0), launches, last


def materialise_leg(dec, st):
    """The shim's share (INTEGRATION.md §3), timed: one decode to host planes, then etl_shim_materialise builds owned
    Vec<Event>-shaped rows from them (one copy per String / Bytes, numerics from the heap, JSON trees) on ONE host thread."""
    from etl_b200 import abi
    lib = abi.load()
    bh, _ = decode_once(dec, st, False, False)
    lst = C.c_void_p()
    t0 = time.perf_counter()
    rc = lib.etl_shim_materialise(bh._h, st.view(False).host_buf, None, C.byref(lst))
    dt = time.perf_counter() - t0
    out = {"error": f"etl_shim_materialise rc={rc}"}
    if rc == 0:
        out = {"ms": dt * 1e3, "events": int(lib.etl_shim_event_count(lst)), "owned_bytes": int(lib.etl_shim_owned_bytes(lst)),
               "total_size_hint": int(lib.etl_shim_total_size_hint(lst)), "threads": 1}
        lib.etl_shim_event_list_free(lst)
    bh.free()
    return out


def roofline_block(wname, nbytes, n_anchors, km, ms_per_step, last, scale):
    """roofline of the dominant kernel + the whole pipeline.  km = mean (index, records, bins, rows, dead, kernel, long cells) ms."""
    peak, peak_src = measured_peak()
    algo_bytes = nbytes + 8 * (n_anchors + 1)              # SURVEY §8d: every staged byte once + the anchor index
    span = int(last["span_bytes"])
    live = algo_bytes - span
    # bytes each kernel is responsible for: k_utf8_dead streams the segments without a frame start (the inside of
    # TOAST-sized values); k_rows every live byte (frames staged once) + the 13-byte cell it writes per output cell
    fused_dead = span > 0 and float(km[4]) < 0.02       # the dead-segment pass runs inside k_rows (its warps stream the segments after their rows)
    kbytes = {"k_utf8_dead": 0 if fused_dead else span, "k_rows": live + 13 * int(last["n_cells"]) + (span if fused_dead else 0)}
    ktime = {"k_utf8_dead": float(km[4]), "k_rows": float(km[3])}
    dominant = max(ktime, key=lambda k: ktime[k])
    achieved = kbytes[dominant] / max(ktime[dominant], 1e-9) / 1e6
    traffic, alone_us = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        traffic = tj.get(f"{wname}/{dominant}")
        alone_us = tj.get(f"{wname}/{dominant}/serialised_us") if scale == 1.0 else None
    except Exception:
        pass
    kern = {"k_act*+k_chase": float(km[0]), "k_records": float(km[1]), "k_bin_scan+k_perm": float(km[2]),
            "k_rows+k_heavy+k_fix" + (" (k_rows streams the dead segments too)" if fused_dead else ""): float(km[3]),
            "k_utf8_dead (separate launch)": float(km[4]), "k_long_cells": float(km[6])}
    return {"bound": "hbm", "kernel": dominant, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": kbytes[dominant],
            "avg_launch_ms": ktime[dominant],
            "alone_under_ncu": ({"ms": alone_us / 1e3, "achieved": kbytes[dominant] / (alone_us * 1e-6) / 1e9,
                                 "frac": kbytes[dominant] / (alone_us * 1e-6) / 1e9 / peak,
                                 "source": "profiles/traffic.json (ncu launch list: kernels serialised, not sharing HBM)"} if alone_us else None),
            "kernels_ms": kern,
            "k_rows": {"algorithmic_bytes": kbytes["k_rows"], "ms": ktime["k_rows"], "frac": kbytes["k_rows"] / max(ktime["k_rows"], 1e-9) / 1e6 / peak},
            "k_utf8_dead": {"algorithmic_bytes": span, "ms": ktime["k_utf8_dead"], "fused_into_k_rows": fused_dead,
                            "frac": (span / max(ktime["k_utf8_dead"], 1e-9) / 1e6 / peak) if (span and not fused_dead) else None},
            "pipeline": {"algorithmic_bytes": algo_bytes, "ms": ms_per_step,
                         "achieved": algo_bytes / (ms_per_step * 1e-3) / 1e9,
                         "frac": algo_bytes / (ms_per_step * 1e-3) / 1e9 / peak,
                         "note": "algorithmic bytes ÷ the driver-visible step time (CUDA events around whole decode calls: every launch, memset, allocation and the final sync included)"}}


def gpu_parity(dec_factory, w, arrays, preamble_needed, threads):
    """CUDA path vs oracle on every segment, full planes, by canonical digest.  Returns a verdict string."""
    from oracle import pyoracle
    pre = None
    if preamble_needed:
        from etl_b200 import workloads as wl
        pre = wl.relation_preamble(arrays[0], len(w.tables))
    t0 = time.perf_counter()
    _, recs, want = cpu_decode_segments(w, arrays, threads, pre, digests=True)
    dec = dec_factory()
    if pre is not None:                               # the same starting state as the oracle workers: the stream's Relation preamble
        from etl_b200 import decoder as _d
        pst = _d.Stager(max(pre.nbytes, 1), 2048)
        pst.append_framed(pre)
        dec.decode_input(pst.view(), to_host=True).free()
        pst.close()
    bad = []
    for i, a in enumerate(arrays):
        if not w.relations_once:
            dec.reset_relations()                     # every segment is its own connection epoch
        from etl_b200 import decoder
        st = decoder.Stager(max(a.nbytes, 1), 2048)
        st.append_framed(a)
        bh = dec.decode_input(st.view(), to_host=True)
        s = bh.summary()
        p = bh.planes(True)
        nv = p.n_records if s.first_error.record_index == NO_ERROR else s.first_error.record_index
        got = (pyoracle.planes_digest(p, nv), int(p.n_records))
        if s.first_error.record_index != NO_ERROR or got != want[i]:
            bad.append(i)
        bh.free()
        st.close()
    dec.close()
    dt = time.perf_counter() - t0
    if bad:
        return f"MISMATCH in segments {bad[:8]} of {len(arrays)}"
    return f"bit-exact ({len(arrays)}/{len(arrays)} segments, {recs} records, every plane; {dt:.1f} s)"


def batch_leg(torch, dev, name, scale, calls, stride):
    """Back-to-back decodes at the reference's batch size (8 MiB of staged stream per call) with carry-in/out chaining."""
    from etl_b200 import decoder, workloads as wl
    w = wl.make(name, scale, n_segments=1)
    stream, stats = w.generate()
    target = 8 << 20
    # cut at record starts: walk the frame chain once on the host
    cuts, pos, n = [0], 0, int(stream.nbytes)
    nxt = target
    mv = memoryview(stream)
    while pos + 5 <= n:
        if pos >= nxt:
            cuts.append(pos)
            nxt = pos + target
        pos += 1 + int.from_bytes(mv[pos + 1:pos + 5], "big")
    cuts.append(n)
    parts = [stream[a:b] for a, b in zip(cuts[:-1], cuts[1:]) if b > a]
    staged = [Staged([p], stride, dev, torch) for p in parts]
    dec = decoder.Decoder(dev.index, stream=torch.cuda.current_stream().cuda_stream)
    for tid, cols in w.table_schemas().items():
        dec.put_table_schema(tid, cols)

    def sweep(resident, n_calls, lat):
        done, carry, nb = 0, None, 0
        while done < n_calls:
            carry = None
            for st in staged:
                t0 = time.perf_counter()
                bh, s = decode_once(dec, st, resident, False, carry, timing=False)   # ETL_DECODE_NO_TIMING: what a production caller passes
                if not resident:
                    bh.planes(True)
                carry = (int(s.carry_out.in_tx), int(s.carry_out.final_lsn), int(s.carry_out.next_tx_ordinal))
                bh.free()
                lat.append(time.perf_counter() - t0)
                nb += st.nbytes
                done += 1
                if done >= n_calls:
                    break
        return nb

    out = {"batch_bytes_target": target, "batches_in_stream": len(parts), "workload": f"{name} x{scale}", "calls": calls,
           "source": "BatchConfig::DEFAULT_MAX_BYTES (etl-config/src/shared/pipeline.rs:54-68)"}
    for label, resident in (("resident", True), ("e2e", False)):
        sweep(resident, 2 * len(staged), [])
        torch.cuda.synchronize()
        lat = []
        t0 = time.perf_counter()
        nb = sweep(resident, calls, lat)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        la = np.sort(np.array(lat)) * 1e6
        out[label] = {"GBps": nb / dt / 1e9, "p50_us": float(la[len(la) // 2]), "p99_us": float(la[min(len(la) - 1, int(len(la) * 0.99))]),
                      "mean_us": float(la.mean())}
    # the 1-thread CPU port on the same batches, same chaining
    o = _new_oracle(w, None)
    t0 = time.perf_counter()
    nb, carry, done = 0, None, 0
    budget = max(len(parts), min(calls, 4 * len(parts)))
    while done < budget:
        carry = None
        o.reset_relations()
        for p in parts:
            b = o.decode_raw(p, carry)
            assert b.first_error.record_index == NO_ERROR
            carry = (int(b.carry_out.in_tx), int(b.carry_out.final_lsn), int(b.carry_out.next_tx_ordinal))
            o.free(b)
            nb += p.nbytes
            done += 1
    dt = time.perf_counter() - t0
    out["cpu_port_1thread_GBps"] = nb / dt / 1e9
    out["e2e_vs_cpu_1thread"] = out["e2e"]["GBps"] / out["cpu_port_1thread_GBps"]
    for st in staged:
        st.close()
    dec.close()
    return out


def copy_leg(torch, dev, n_rows, steps):
    """Initial-sync COPY rows (SURVEY §8f N1): a 10-column int4 + text table (the C2 shape) as COPY text, decoded by
    etl_dec_copy_decode with the buffer resident in HBM; rows/s next to the 1-thread CPU port and parity by digest.
    The reference's own figure for its copy phase (87 738 rows/s end to end, etl-benchmarks/README.md:302-308) includes
    the network read and the destination write — context only."""
    from etl_b200 import abi, decoder
    from oracle import pyoracle
    rng = np.random.default_rng(0xC0B7)
    ints = rng.integers(-2**31, 2**31, size=(n_rows, 5))
    lens = np.minimum(256, np.maximum(1, np.exp(np.log(16) + 0.8 * rng.standard_normal((n_rows, 5))).astype(np.int64)))
    alnum = np.frombuffer(b"abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789      ", dtype=np.uint8)
    pool = alnum[rng.integers(0, len(alnum), size=1 << 20)].tobytes()
    starts = rng.integers(0, (1 << 20) - 256, size=(n_rows, 5))
    nulls = rng.integers(0, 20, size=(n_rows, 9)) == 0
    rows = []
    for r in range(n_rows):
        f = [str(ints[r, 0])]
        for c in range(1, 5):
            f.append("\\N" if nulls[r, c - 1] else str(ints[r, c]))
        for c in range(5):
            f.append("\\N" if nulls[r, 4 + c] else pool[starts[r, c]:starts[r, c] + lens[r, c]].decode())
        rows.append("\t".join(f))
    blob = ("\n".join(rows) + "\n").encode()
    buf = np.frombuffer(blob, dtype=np.uint8)
    offs = np.zeros(n_rows + 1, dtype=np.uint64)
    offs[1:] = np.flatnonzero(buf == 10) + 1
    oids = [23] * 5 + [25] * 5
    cols = [dict(name=f"c{i}", type_oid=o, pk=1 if i == 0 else None, nullable=i != 0) for i, o in enumerate(oids)]
    dec = decoder.Decoder(dev.index, stream=torch.cuda.current_stream().cuda_stream)
    dec.put_table_schema(9, cols)
    d_buf = torch.zeros(buf.nbytes + 64, dtype=torch.uint8, device=dev)
    d_buf[:buf.nbytes].copy_(torch.from_numpy(buf.copy()))
    d_off = torch.from_numpy(offs.view(np.int64).copy()).to(dev)
    lib = abi.load()

    def once(to_host):
        inp = abi.CopyInput()
        inp.dev_buf, inp.dev_row_offsets, inp.len, inp.n_rows = d_buf.data_ptr(), d_off.data_ptr(), buf.nbytes, n_rows
        inp.row_offsets = offs.ctypes.data
        h = C.c_void_p()
        rc = lib.etl_dec_copy_decode(dec._ctx, 9, C.byref(inp), abi.RESULTS_TO_HOST if to_host else 0, C.byref(h))
        if rc:
            raise RuntimeError(lib.etl_dec_last_error(dec._ctx).decode())
        return decoder.BatchHandle(dec, h)

    for _ in range(3):
        once(False).free()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        once(False).free()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    bh = once(True)
    p, s = bh.planes(True), bh.summary()
    m = int(p.n_cells)
    got = pyoracle.copy_planes_digest(decoder._np_from(p.cell_tag, m, np.uint8), decoder._np_from(p.cell_val, m, np.uint64),
                                      decoder._np_from(p.cell_aux, m, np.uint32), n_rows, len(oids), buf, decoder._np_from(p.heap, p.heap_bytes, np.uint8))
    clean = s.first_error.record_index == NO_ERROR
    bh.free()
    dec.close()
    t0 = time.perf_counter()
    want, err = pyoracle.copy_rows_digest(oids, buf, offs)
    cpu_s = time.perf_counter() - t0
    return {"table": "10 columns (5 x int4, 5 x text, 5 % NULL), COPY text", "rows": n_rows, "bytes": int(buf.nbytes), "ms_per_step": ms,
            "rows_per_s": n_rows / (ms * 1e-3), "GBps": buf.nbytes / (ms * 1e-3) / 1e9,
            "cpu_port_1thread_rows_per_s": n_rows / cpu_s, "parity": "bit-exact (every cell, strings by content)" if (clean and err is None and got == want) else "MISMATCH",
            "reference_context": "87 738 rows/s end to end on other hardware (etl-benchmarks/README.md:302-308), incl. network and destination"}


def measure_workload(torch, dev, name, scale, steps, warmup, stride, threads, cpu_budget_s=6.0):
    """One of the other BASELINE configs on one GPU: value, e2e, roofline, 1-thread CPU port, parity at size."""
    from etl_b200 import decoder, workloads as wl
    w = wl.make(name, scale)
    arrays, stats = generate_segments(w, list(range(w.n_segments)), threads)
    nbytes = sum(a.nbytes for a in arrays)
    frames = sum(s["frames"] for s in stats)
    st = Staged(arrays, stride, dev, torch)
    dec = decoder.Decoder(dev.index, stream=torch.cuda.current_stream().cuda_stream)
    for tid, cols in w.table_schemas().items():
        dec.put_table_schema(tid, cols)
    for _ in range(max(warmup, 3)):
        decode_once(dec, st, True, False)[0].free()
    ms, km, _, last = time_steps(torch, None, dec, st, True, False, steps, dev, 1)
    ms_step = ms / steps
    for _ in range(2):
        decode_once(dec, st, False, False)[0].free()
    e_ms, _, _, elast = time_steps(torch, None, dec, st, False, False, steps, dev, 1)
    mat = materialise_leg(dec, st)
    dec.close()
    # 1-thread CPU port on a bounded sample (first segments)
    pick, acc = [], 0
    est_rate = 0.15e9                                    # bytes/s guess, only to bound the sample
    for i, a in enumerate(arrays):
        if pick and acc + a.nbytes > est_rate * cpu_budget_s:
            break
        pick.append(i)
        acc += a.nbytes
    secs, recs = cpu_decode_segments(w, [arrays[i] for i in pick], 1)
    _, box = host_cores()
    res = {"config": f"{w.name}: {w.description}", "scale": scale, "bytes": int(nbytes), "msgs": int(frames),
           "value": nbytes / (ms_step * 1e-3) / 1e9, "unit": "GB/s", "events_per_s": frames / (ms_step * 1e-3), "ms_per_step": ms_step,
           "roofline": roofline_block(w.name, nbytes, st.n_anchors, km, ms_step, last, scale),
           "e2e": {"value": nbytes / (e_ms / steps * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": e_ms / steps,
                   "h2d_bytes_per_step": elast["h2d"], "d2h_bytes_per_step": elast["d2h"]},
           "e2e_materialised": ({"value": nbytes / ((e_ms / steps + mat["ms"]) * 1e-3) / 1e9, "unit": "GB/s", "shim": mat,
                                 "cpu_port_1thread_plus_shim": nbytes / (nbytes / (acc / secs) + mat["ms"] * 1e-3) / 1e9,
                                 "note": "e2e + the shim stand-in building owned events from the host planes on one thread; the same "
                                         "materialisation after the 1-thread CPU port for comparison (the reference builds its owned events inside its decode)"}
                                if "ms" in mat else mat),
           "cpu_baseline": {"value": acc / secs / 1e9, "unit": "GB/s", "events_per_s": recs / secs, "cores": 1, "box_cores": box, "kind": "port",
                            "sample": f"first {len(pick)} of {len(arrays)} segments ({acc / GIB:.2f} GiB, {recs} msgs) in {secs:.1f} s"}}
    st.close()
    parity = gpu_parity(lambda: _fresh_decoder(dev, w), w, arrays, False, threads)
    return res, parity


def _fresh_decoder(dev, w):
    from etl_b200 import decoder
    d = decoder.Decoder(dev.index)
    for tid, cols in w.table_schemas().items():
        d.put_table_schema(tid, cols)
    return d


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries the ONE JSON line and nothing else: whatever native code writes to fd 1 (NCCL prints its version banner
    # there) lands on stderr from here on, and the line goes to the saved descriptor
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    if world > 1:
        # NCCL's init lines (incl. "nranks N") on stderr
        os.environ["NCCL_DEBUG"] = os.environ.get("ETL_NCCL_DEBUG", "INFO")
        os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
    import torch
    import torch.distributed as dist
    from etl_b200 import decoder, workloads as wl

    assert torch.cuda.is_available(), "bench.py needs CUDA devices (the decode path has no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # the decode chain runs on torch's CURRENT stream (the CUDA events below see only that one): a high-priority stream,
    # so that the library's low-priority side pass yields thread slots to it
    main_stream = torch.cuda.Stream(device=dev, priority=-1)
    torch.cuda.set_stream(main_stream)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world
    usable, box = host_cores()

    # ---- this rank's byte range of the workload
    one = args.workload == "c5"
    w = wl.make(args.workload, args.scale, one_stream=one)
    S = w.n_segments
    strong = world > 1 and args.scaling == "strong"
    t0 = time.perf_counter()
    gen_threads = args.gen_threads or max(1, usable // world)
    if strong:
        assert S % world == 0, "segments must divide over the ranks"
        per = S // world
        r0, r1 = rank * per, (rank + 1) * per
        segs = list(range(r0, r1)) + ([r1] if rank < world - 1 else [])
        arrays, stats = generate_segments(w, segs, gen_threads)
        # seams fall INSIDE a transaction, ~1 MiB after a segment boundary
        d_lo = wl.mid_transaction_cut(arrays[0], 1 << 20) if rank > 0 else 0
        pieces = [arrays[0][d_lo:]] + arrays[1:per]
        frames = sum(s["frames"] for s in stats[:per])
        if rank < world - 1:
            d_hi = wl.mid_transaction_cut(arrays[per], 1 << 20)
            pieces.append(arrays[per][:d_hi])
        arrays = None
    else:
        my_segs = list(range(rank * S, (rank + 1) * S))   # weak: a full-size range of one longer stream per GPU
        arrays, stats = generate_segments(w, my_segs, gen_threads)
        pieces = arrays
        frames = sum(s["frames"] for s in stats)
    st = Staged(pieces, args.stride, dev, torch)
    nbytes = st.nbytes
    gen_s = time.perf_counter() - t0
    keep_arrays = rank == 0 and world == 1 and not (args.no_cpu_baseline and args.no_extras)
    if not keep_arrays:
        arrays = None
    pieces = None

    dec = decoder.Decoder(local_rank, stream=torch.cuda.current_stream().cuda_stream)
    for tid, cols in w.table_schemas().items():
        dec.put_table_schema(tid, cols)
    sharded = world > 1
    if sharded:                                        # the library owns the communicator (NCCL inside libetl_decode.so)
        uid = [dec.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        dec.comm_init(uid[0], rank, world)

    for _ in range(max(args.warmup, 3)):
        decode_once(dec, st, True, sharded)[0].free()
    dump = None
    if args.dump_outputs:
        def dump(bh):
            dump_outputs(torch, dev, bh, args.dump_outputs, f"rank{rank}_" if world > 1 else "", 1.0 / world)
    sampler = ClockSampler(local_rank)
    with sampler:
        total_ms, km, launches, last = time_steps(torch, dist, dec, st, True, sharded, args.steps, dev, world, on_last=dump)
    ms_per_step = total_ms / args.steps

    e2e = None
    if not args.no_e2e:
        for _ in range(2):
            decode_once(dec, st, False, sharded)[0].free()
        e2e_ms, _, _, elast = time_steps(torch, dist, dec, st, False, sharded, args.steps, dev, world)
        e2e = {"ms_per_step": e2e_ms / args.steps, "h2d": elast["h2d"], "d2h": elast["d2h"]}
        if rank == 0 and world == 1 and not args.no_extras:
            e2e["materialise"] = materialise_leg(dec, st)

    # ---- totals over ranks
    tot = torch.tensor([nbytes, frames, last["n_records"], last["n_cells"], e2e["h2d"] if e2e else 0, e2e["d2h"] if e2e else 0, len(DATA_ERRORS)],
                       dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    if tot[6].item() > 0:
        if DATA_ERRORS:
            print(f"rank {rank}: decode reported data errors on a clean stream: {DATA_ERRORS[:3]}", file=sys.stderr, flush=True)
        if world > 1:
            dist.destroy_process_group()
        sys.exit(3)
    total_bytes, total_frames = float(tot[0].item()), float(tot[1].item())
    n_anchors = st.n_anchors
    dec.close()
    st.close()
    st = None
    torch.cuda.empty_cache()

    cpu_baseline = None
    if rank == 0 and n_gpus == 1 and not args.no_cpu_baseline:
        # the scalar oracle port, one thread (the reference's streaming decode is a single task, apply.rs:839-967)
        budget = int(args.cpu_sample_gib * GIB)
        pick, acc = [], 0
        for i, a in enumerate(arrays):
            if pick and acc + a.nbytes > budget:
                break
            pick.append(i)
            acc += a.nbytes
        pre = wl.relation_preamble(arrays[0], len(w.tables)) if w.relations_once else None
        secs, recs = cpu_decode_segments(w, [arrays[i] for i in pick], 1, pre)
        cpu_baseline = {"value": acc / secs / 1e9, "unit": "GB/s", "cores": 1, "box_cores": box, "kind": "port",
                        "sample": f"first {len(pick)} of {len(arrays)} segments of this run's stream ({acc / GIB:.2f} GiB, {recs} msgs) in {secs:.1f} s",
                        "events_per_s": recs / secs}

    extras = {}
    if rank == 0 and n_gpus == 1 and not args.no_extras:
        parity = {}
        try:
            parity[w.name] = gpu_parity(lambda: _fresh_decoder(dev, w), w, arrays, w.relations_once, usable)
        except Exception as e:  # noqa: BLE001 — the verdict is part of the line, not a crash
            parity[w.name] = f"ERROR {type(e).__name__}: {e}"
        arrays = None
        workloads = {}
        for name in ("c2", "c3", "c4"):
            if name == w.name:
                continue
            try:
                res, par = measure_workload(torch, dev, name, args.extras_scale, args.steps, args.warmup, args.stride, usable)
                workloads[name] = res
                parity[name] = par
            except Exception as e:  # noqa: BLE001
                workloads[name] = {"error": f"{type(e).__name__}: {e}"}
            torch.cuda.empty_cache()
        batches = {}
        for name in ("c2", "c3"):
            try:
                batches[name] = batch_leg(torch, dev, name, min(1.0, args.extras_scale) * (1.0 if name == "c2" else 0.1), args.batch_calls, args.stride)
            except Exception as e:  # noqa: BLE001
                batches[name] = {"error": f"{type(e).__name__}: {e}"}
        try:
            copy = copy_leg(torch, dev, int(1_000_000 * min(1.0, args.extras_scale)), args.steps)
        except Exception as e:  # noqa: BLE001
            copy = {"error": f"{type(e).__name__}: {e}"}
        extras = {"parity": parity, "workloads": workloads, "batch_8MiB": batches, "copy_rows": copy}

    if rank == 0:
        line = {
            "metric": "wal_decode_throughput", "value": total_bytes / (ms_per_step * 1e-3) / 1e9, "unit": "GB/s",
            "n_gpus": n_gpus, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": ("strong" if strong else "weak"), "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "events_per_s": total_frames / (ms_per_step * 1e-3),
            "config": {"workload": f"{w.name}: {w.description}", "scale": args.scale, "bytes_total": int(total_bytes),
                       "msgs_total": int(total_frames), "records": int(tot[2].item()), "cells": int(tot[3].item()),
                       "parallelism": (f"ONE stream cut into {n_gpus} byte ranges at mid-transaction record starts (strong scaling; Relation frames only in "
                                       f"range 0), seam + relation-update exchange over NCCL inside the library" if strong else
                                       (f"{n_gpus} full-size byte ranges of one longer stream (weak scaling), seam + relation-update exchange over NCCL inside the library"
                                        if n_gpus > 1 else "single GPU")),
                       "scaling_note": "efficiency = value_N / (N * value_1): total bytes are fixed under strong scaling, per-GPU bytes under weak",
                       "anchor_stride": args.stride, "l2_policy": "inputs (>=1.25 GiB per GPU) larger than the 126 MB L2",
                       "timed_calls": "etl_dec_decode(_sharded) with ETL_DECODE_NO_TIMING; roofline.kernels_ms from two more calls with the summary timings on, outside the timed region",
                       "generate_s": round(gen_s, 2), "host_cores": {"box": box, "usable": usable}},
            "roofline": roofline_block(w.name, nbytes, n_anchors, km, ms_per_step, last, args.scale),
            "gpu_launches": launches,
            "clocks": sampler.report(),
        }
        if e2e:
            line["e2e"] = {"value": total_bytes / (e2e["ms_per_step"] * 1e-3) / 1e9, "unit": "GB/s",
                           "h2d_bytes_per_step": int(tot[4].item()), "d2h_bytes_per_step": int(tot[5].item()),
                           "ms_per_step": e2e["ms_per_step"]}
            mat = e2e.get("materialise")
            if mat:
                line["e2e_materialised"] = ({"value": total_bytes / ((e2e["ms_per_step"] + mat["ms"]) * 1e-3) / 1e9, "unit": "GB/s", "shim": mat,
                                             "cpu_port_1thread_plus_shim": (total_bytes / (total_bytes / (cpu_baseline["value"] * 1e9) + mat["ms"] * 1e-3) / 1e9
                                                                            if cpu_baseline else None),
                                             "note": "e2e + the shim stand-in building owned events from the host planes on one thread; the same "
                                                     "materialisation after the 1-thread CPU port for comparison (the reference builds its owned events inside its decode)"}
                                            if "ms" in mat else mat)
        if cpu_baseline:
            line["cpu_baseline"] = cpu_baseline
        line.update(extras)
        emit_line(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
