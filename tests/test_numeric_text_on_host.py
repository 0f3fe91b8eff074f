"""Numeric → Utf8 text of the columnar emitter's formatted mode, on the CPU.

1. The Python restatement of PgNumeric::to_string() (tests/arrow_ref.py) against the reference's own known answers
   (crates/etl/src/conversions/numeric.rs:730-958), on the headers and digits the oracle's parser produces.
2. The device formatter (etl_b200/csrc/numeric_text.cuh) compiled for the host (tests/emul/numeric_text_host.cpp — test
   infrastructure, not a product path) against the restatement on fuzzed spellings and on every numeric element of
   the array fixtures, written by one writer and by 32 interleaved writers (the warp-cooperative split).
3. The ABI guards of etl_dec_arrow_emit_ex that need no GPU."""
import ctypes as C
import os
import random
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.normpath(os.path.join(HERE, ".."))
sys.path.insert(0, HERE)
from arrow_ref import ELEM, format_numeric, numeric_entry, numeric_text  # noqa: E402

N_FUZZ = int(os.environ.get("ETL_HOST_FUZZ_N", "100000"))


def parsed(oracle_mod, text: str):
    e, tag, val, aux, heap = oracle_mod.parse_cell(1700, text.encode())
    assert e == 0 and tag & 0xFF == 9, (text, e, tag)
    return heap, val, aux


KNOWN = [  # (input, to_string) — numeric.rs:730-958
    ("NaN", "NaN"), ("Infinity", "Infinity"), ("-Infinity", "-Infinity"),
    ("123", "123"), ("-456", "-456"), ("1234.50", "1234.50"), ("0", "0"), ("0.0", "0"), ("000", "0"), ("000.000", "0"),
    ("-0", "0"), ("-0.00", "0"), ("0.000", "0"), ("12345678", "12345678"), ("0.1234", "0.1234"),
    ("0.0012000", "0.0012000"), ("9999.9999", "9999.9999"), ("10000.0001", "10000.0001"), ("0000120.00", "120.00"),
    ("1200000", "1200000"),
]
ROUNDTRIP = ["120.00", "1.2000", "0.0120", "9999.9999", "10000.0001", "-120.00", "1200000"]   # :916-933
SPECIAL = ["NaN", "Infinity", "-Infinity"]                                                        # :950-958


@pytest.mark.parametrize("text,want", KNOWN)
def test_restatement_matches_reference_known_answers(oracle_mod, text, want):
    heap, val, aux = parsed(oracle_mod, text)
    assert numeric_text(heap, val, aux).decode() == want


@pytest.mark.parametrize("text", ROUNDTRIP + SPECIAL)
def test_restatement_roundtrip_stability(oracle_mod, text):
    """print → parse → print is stable, and the internal value survives (roundtrip_stability, :916-933)"""
    heap, val, aux = parsed(oracle_mod, text)
    printed = numeric_text(heap, val, aux).decode()
    heap2, val2, aux2 = parsed(oracle_mod, printed)
    assert numeric_text(heap2, val2, aux2).decode() == printed
    assert numeric_entry(heap, val, aux)[:4] == numeric_entry(heap2, val2, aux2)[:4]


def test_restatement_edge_cases():
    assert format_numeric(0, 1, 0, 5, []) == "0"                  # no digits: "0" whatever the scale and sign
    assert format_numeric(0, 0, -2, 8, [12]) == "0.00000012"      # weight < 0: leading "0", groups before 0 are 0000
    assert format_numeric(0, 0, 2, 0, [7]) == "700000000"         # groups past the end count as 0000
    assert format_numeric(0, 1, 0, 2, [1, 2345]) == "-1.23"       # fraction cut to scale digits
    assert format_numeric(0, 0, 0, 0, [0]) == "0"                 # a zero first group prints "0"


@pytest.fixture(scope="module")
def emu():
    src = os.path.join(HERE, "emul", "numeric_text_host.cpp")
    so = os.path.join(HERE, "emul", "libnumeric_text_host.so")
    deps = [src, os.path.join(ROOT, "etl_b200", "csrc", "numeric_text.cuh"), os.path.join(ROOT, "include", "etl_decode.h")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                               "-I", os.path.join(ROOT, "etl_b200", "csrc"), "-o", so, src])
    L = C.CDLL(so)
    L.emu_numeric_text.restype = C.c_int64
    L.emu_numeric_text.argtypes = [C.c_char_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint64]
    cap = 1 << 18
    buf = (C.c_uint8 * cap)()

    def fmt(heap: bytes, off: int, n_digits: int, writers: int) -> bytes:
        n = L.emu_numeric_text(heap[off:off + 8 + 2 * n_digits], n_digits, writers, buf, cap)
        assert n >= 0
        return bytes(buf[:n])
    return fmt


def _spellings(rng):
    def digits(n):
        return "".join(rng.choice("0123456789") for _ in range(n))
    while True:
        k = rng.randint(0, 9)
        if k == 0:
            yield rng.choice(["NaN", "nan", "Infinity", "-Infinity", "inf", "-inf", "+Infinity", "-0.000", "0", "-0", "0.0000"])
        elif k == 1:     # huge weights
            yield rng.choice(["", "-"]) + rng.choice("123456789") + digits(rng.randint(0, 6)) + "e" + str(rng.randint(100, 131000))
        elif k == 2:     # tiny weights
            yield rng.choice(["", "-"]) + "0." + "0" * rng.randint(0, 200) + digits(rng.randint(1, 12)) + rng.choice(["", "e-" + str(rng.randint(0, 500))])
        elif k == 3:     # scale up to the maximum, trailing zero groups
            yield rng.choice(["", "-"]) + digits(rng.randint(1, 8)) + "." + digits(rng.randint(0, 40)) + "0" * rng.randint(0, 1000)
        elif k == 4:     # zero groups in the middle and at the end of the integer part
            yield rng.choice(["", "-"]) + rng.choice("123456789") + "0" * rng.randint(0, 40) + digits(rng.randint(0, 5)) + "0" * rng.randint(0, 12)
        elif k == 5:
            yield rng.choice(["", "-", "+"]) + digits(rng.randint(0, 40)) + rng.choice(["", ".", "." + digits(rng.randint(1, 30))]) + \
                rng.choice(["", "", "e" + str(rng.randint(-50, 50)), "E+" + digits(2)])
        elif k == 6:
            yield "%.*f" % (rng.randint(0, 30), rng.uniform(-1e6, 1e6))
        elif k == 7:     # exponents that move the point past the scale
            yield digits(rng.randint(1, 20)) + "." + digits(rng.randint(0, 20)) + "e" + str(rng.randint(-60, 60))
        else:
            yield str(rng.randint(-10 ** 30, 10 ** 30)) + rng.choice(["", ".", ".0", ".00000", "." + digits(rng.randint(1, 9))])


def test_device_formatter_matches_restatement_on_fuzzed_spellings(emu, oracle_mod):
    rng = random.Random(0x4E554D)
    gen = _spellings(rng)
    n_ok = n_long = 0
    for _ in range(N_FUZZ):
        text = next(gen)
        e, tag, val, aux, heap = oracle_mod.parse_cell(1700, text.encode())
        if e:
            continue
        n_ok += 1
        want = numeric_text(heap, val, aux)
        n_long += len(want) > 128
        w = 32 if rng.random() < 0.5 else 1
        got = emu(heap, val, aux, w)
        assert got == want, (text, w, got[:80], want[:80])
        assert b"\xff" not in got
    assert n_ok > N_FUZZ // 2 and n_long > N_FUZZ // 20, (n_ok, n_long)


def test_device_formatter_on_array_fixture_elements(emu, oracle_mod):
    """every numeric element of the array fixtures (the spellings test_gpu_parity decodes), element by element"""
    from test_gpu_parity import ARRAY_COLS
    seen = 0
    for oid, valid, _ in ARRAY_COLS:
        for text in valid:
            e, tag, val, aux, heap = oracle_mod.parse_cell(oid, text.encode())
            assert e == 0
            if tag != 17:
                continue
            n = int.from_bytes(heap[val + 4:val + 8], "little")
            for j in range(n):
                r = np.frombuffer(heap[val + 8 + 16 * j:val + 24 + 16 * j], ELEM)[0]
                if int(r["tag"]) != 9:
                    continue
                want = numeric_text(heap, int(r["val"]), int(r["aux"]))
                for w in (1, 32):
                    assert emu(heap, int(r["val"]), int(r["aux"]), w) == want
                seen += 1
    assert seen >= 4, seen


def test_emit_ex_rejects_bad_arguments():
    from etl_b200 import abi
    lib = abi.load()
    out = C.c_void_p()
    assert lib.etl_dec_arrow_emit_ex(None, 0, 7, 0, 1, C.byref(out)) == 1            # NULL batch
    assert lib.etl_dec_arrow_emit_ex(None, 0, 7, abi.ARROW_FORMATTED, 1, C.byref(out)) == 1
    for bit in (0x2, 0x4, 0x80000000):    # unknown flag bits: refused before the (here bogus) batch is read
        assert lib.etl_dec_arrow_emit_ex(C.c_void_p(1), 0, 7, abi.ARROW_FORMATTED | bit, 1, C.byref(out)) == 1
    assert lib.etl_dec_arrow_list_values(None, 0, 1, C.byref(abi.ArrowColumn()), None) == 1
