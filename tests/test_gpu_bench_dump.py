"""bench.py --dump-outputs: two runs write the same files (float64, within 64 MB), and what they hold is the oracle's
decode of the same stream, sampled the same way."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from etl_b200 import workloads as wl

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# c3: numeric and jsonb columns, so heap-backed cells are in the sample
ARGS = ["--workload", "c3", "--scale", "0.002", "--warmup", "1", "--no-e2e", "--no-cpu-baseline", "--no-extras"]


def _bench_dump(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *ARGS, "--steps", str(steps), "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout)
    assert line["steps"] == steps
    files = sorted(os.listdir(out_dir))
    assert all(f.endswith(".npy") for f in files), files
    assert sum(os.path.getsize(os.path.join(out_dir, f)) for f in files) <= bench.DUMP_BYTES
    return {f[:-4]: np.load(os.path.join(out_dir, f)) for f in files}


def test_dump_outputs_repeat_and_match_oracle(oracle_mod, tmp_path):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    a = _bench_dump(tmp_path / "a", 2)
    b = _bench_dump(tmp_path / "b", 3)
    assert a.keys() == b.keys()
    for k in a:
        assert a[k].dtype == np.float64, k
        assert np.array_equal(a[k], b[k]), k

    w = wl.make("c3", 0.002)
    stream = np.concatenate([w.generate_segment(i)[0] for i in range(w.n_segments)]).tobytes()
    orc = oracle_mod.Oracle()
    for tid, cols in w.table_schemas().items():
        orc.put_table_schema(tid, cols)
    orc.decode(stream)                  # bench decodes the same stream on one context again and again
    p = orc.decode(stream)
    fe = p.first_error
    summary = dict(n_records=p.n_records, n_cells=p.n_cells, first_error_record=bench.NO_ERROR if fe[0] is None else fe[0],
                   first_error_seq=fe[1], first_error_code=fe[2], first_error_kind=fe[3], carry_in_tx=p.carry_out[0],
                   carry_final_lsn=p.carry_out[1], carry_next_tx_ordinal=p.carry_out[2], insert_bytes=p.insert_bytes,
                   update_bytes=p.update_bytes, delete_bytes=p.delete_bytes, n_events=p.n_events)
    want = bench.sample_outputs(summary, p.schemas, lambda name, idx: getattr(p, name)[idx], lambda: p.heap.tobytes())
    assert a.keys() == want.keys()
    assert np.count_nonzero(want["cell_var_crc32"]) > 0
    for k in want:
        assert np.array_equal(a[k], want[k]), k
