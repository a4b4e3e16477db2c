"""CSV source: pins the oracle (oracle/csv_oracle.c) and checks the host build of the device code against it.

1. Known-answer vectors restated from the reference's row-parser tests (tuplex/test/core/CSVRowParseGeneratorTests.cc:256-980):
   input text, column types / serialize mask, expected status and values.
2. Cell splitting equals the reference's own csvmonkey reader (its output stored under tests/golden/) on the Zillow
   fixture and on fuzzed inputs with pathological quoting.
3. The device code (tuplex_b200/csrc/csvops.cuh) compiled for the host — including the quote-parity speculation, its
   verification and the sequential repair — equals the oracle on seeded random CSV.
"""
import gzip
import math
import os
import random
import struct

import numpy as np
import pytest

from oracle import pyoracle as po
from csv_helpers import T_BOOL, T_F64, T_I64, T_SKIP, T_STR, assert_same_parse, gen_csv, host_parse

HERE = os.path.dirname(os.path.abspath(__file__))
I, F, B, S, X = T_I64, T_F64, T_BOOL, T_STR, T_SKIP

# (text, types, ok?, expected values of the parsed columns)  — CSVRowParseGeneratorTests.cc line in the comment
VECTORS = [
    ("10", [I], True, [10]),                                    # :269
    ("\n\r\n10", [I], True, [10]),                              # :282
    ("10\n", [I], True, [10]),                                  # :295
    ("10,", [I], False, None),                                  # :308 CSV_OVERRUN
    ("10,\n", [I], False, None),                                # :321
    ("10,\r", [I], False, None),                                # :335
    ("10$", [I], False, None),                                  # :348 ValueError
    ("10$", [X], True, []),                                     # :361 not serialized -> no conversion
    ("$10", [I], False, None),                                  # :375
    ("\t10   \n", [I], True, [10]),                             # :389 whitespace is trimmed
    ('""', [I], False, None),                                   # :402 quoted empty string is no integer
    ('"10"', [I], True, [10]),                                  # :422
    ('"10"\n', [I], True, [10]),                                # :438
    ('"10",""', [I], False, None),                              # :451
    ('"10",\n', [I], False, None),                              # :464
    ('"10$"', [I], False, None),                                # :491
    ('"10$"', [X], True, []),                                   # :504
    ('"$10"', [I], False, None),                                # :518
    ('"\t10   "\n', [I], True, [10]),                           # :532
    ('10,"20",30', [I, I, I], True, [10, 20, 30]),              # :561
    ("10,20,30", [I, I, I], True, [10, 20, 30]),                # :578
    ('10,20,"30"', [I, X, I], True, [10, 30]),                  # :595
    ('0,"1",2,3,"4"\n', [I] * 5, True, [0, 1, 2, 3, 4]),        # :611
    ("7", [I], True, [7]),                                      # :635
    ('12.5,"7.5",1.0', [F, F, F], True, [12.5, 7.5, 1.0]),      # :653
    ("\n\r\n12.5,7.5,1.0", [F, F, F], True, [12.5, 7.5, 1.0]),  # :670
    ('10,20,"30"', [X, F, X], True, [20.0]),                    # :687
    ('10,20.34$,"30"', [F, F, F], False, None),                 # :702
    ('TRUE,"false",y', [B, B, B], True, [True, False, True]),   # :717
    ("\n\r\nYes,no,T,f", [B] * 4, True, [True, False, True, False]),  # :734
    ('"TRUE",false,NO', [X, B, X], True, [False]),              # :753
    ('true,20.34$,"falsch!"', [B, B, B], False, None),          # :768
    ('"test"" this"', [S], True, ['test" this']),               # :783
    ('"quoted text can contain \n \r or """', [S], True, ['quoted text can contain \n \r or "']),  # :799
    ("hello", [S], True, ["hello"]),                            # :814
    ("a", [S], True, ["a"]),                                    # :828
    ('"a"', [S], True, ["a"]),                                  # :842
    ('some text here,"quoted text can contain \n \r or """,Hello world!', [S, S, S], True,
     ["some text here", 'quoted text can contain \n \r or "', "Hello world!"]),                    # :857
    ('"ab""","\n""","""haha"""', [S, S, S], True, ['ab"', '\n"', '"haha"']),                       # :875
    ('some text here,ignore this,"speaking in "" is stupid"', [S, X, S], True,
     ["some text here", 'speaking in " is stupid']),                                               # :893
    ('1234, dhfgj,-20,WRONG,"""hello!"""\n', [I, X, F, X, S], True, [1234, -20.0, '"hello!"']),    # :921 (first row)
]


def _values(res):
    out = []
    for col, t in zip(res.columns, res.types):
        if t == T_STR:
            by, offs = col
            out.append(by[offs[0]:offs[1]].decode())
        elif t == T_BOOL:
            out.append(bool(col[0]))
        else:
            out.append(col[0].item())
    return out


@pytest.mark.parametrize("parser", ["oracle", "device_code_on_host"])
def test_reference_row_parser_vectors(parser):
    for text, types, ok, expect in VECTORS:
        data = text.encode()
        res = po.csv_parse(data, types, null_values=[]) if parser == "oracle" else host_parse(data, types, null_values=[])
        assert res.n_rows == 1, text
        if not ok:
            assert len(res.bad) == 1 and len(res.rowmap) == 0, text
            assert res.bad[0][1] == 70, text  # BADPARSE_STRING_INPUT
        else:
            assert len(res.bad) == 0, (text, res.bad)
            assert _values(res) == expect, (text, _values(res), expect)


def test_unterminated_quote_yields_no_row():
    # DoubleQuoteError vector (:910): csvmonkey's reader (yield_incomplete_row = false) drops the row
    for parse in (lambda d: po.csv_parse(d, [S], null_values=[]), lambda d: host_parse(d, [S], null_values=[])):
        r = parse(b'"user forgot to close doublequote')
        assert r.n_rows == 0 and not r.bad
        r = parse(b'ok\n"user forgot')
        assert r.n_rows == 1 and len(r.rowmap) == 1


def test_scalar_parsers_known_answers():
    f = lambda s: po.csv_scalar("f64", s)
    assert f("12.5") == 12.5 and f("7.5") == 7.5 and f("-20") == -20.0 and f("1801.0") == 1801.0
    assert f("20.34$") is None and f("") is None and f("  ") is None
    assert math.isnan(f("nan")) and math.isnan(f("NaN")) and f("inf") == math.inf and f("Infinity") == math.inf
    assert f("-inf") is None and f("+nan") is None            # special values only without a sign (StringUtils.cc:140-150)
    assert f("n") == 0.0 and f("infi") == 0.0                  # prefix quirk of the reference's matcher
    assert f("1e5") == 100000.0 and f("1e-2") == 0.01 and f("1e400") == 1e50 * 1e50 * 1e50 * 1e50 * 1e50 * 1e50 * 1e8 and f(" 3.5\t") == 3.5
    # the accumulation is not correctly rounded: 0.3 -> 3/10, 0.07 -> 0/10 + 7/100
    assert f("0.07") == 0.0 + 7 / 100.0
    assert po.csv_scalar("i64", " 42 ") == 42 and po.csv_scalar("i64", "-") == 0 and po.csv_scalar("i64", "+5") is None
    assert po.csv_scalar("i64", "9223372036854775808") == -2**63  # wraps, no overflow detection
    for s, v in (("t", True), ("Y", True), ("yes", True), ("TRUE", True), ("f", False), ("n", False), ("No", False), ("false", False)):
        assert po.csv_scalar("bool", s) is v
    for s in ("1", "0", "tr", "yess", " true", ""):
        assert po.csv_scalar("bool", s) is None


def test_device_scalar_decoders_equal_oracle():
    from csv_helpers import host_shim
    import ctypes as ct
    L = host_shim()
    rng = random.Random(5)
    alpha = "0123456789.eE+-naifNIty \t"
    for it in range(60000):
        s = "".join(rng.choice(alpha) for _ in range(rng.randint(0, 12)))
        if it % 3 == 0:
            s = f"{rng.uniform(-1e9, 1e9):.{rng.randint(0, 15)}g}"
        d = ct.c_double()
        ok = L.hcsv_atod(s.encode(), len(s), ct.byref(d))
        want = po.csv_scalar("f64", s)
        assert bool(ok) == (want is not None), s
        if ok:
            assert struct.pack("<d", d.value) == struct.pack("<d", want) or (math.isnan(d.value) and math.isnan(want)), s
    for s in ["t", "T", "y", "n", "F", "no", "NO", "yes", "YeS", "true", "TRUE", "false", "False", "1", "0", "", "tru", "falsee", "on"]:
        b = ct.c_longlong()
        ok = L.hcsv_atob(s.encode(), len(s), ct.byref(b))
        want = po.csv_scalar("bool", s)
        assert bool(ok) == (want is not None) and (not ok or bool(b.value) == want), s


def _zillow_csv():
    return gzip.open(os.path.join(HERE, "golden", "zillow_noexc.csv.gz"), "rb").read()


def test_cells_equal_reference_csvmonkey():
    """the reader's cell dumps are stored in tests/golden/csvmonkey_cells.npz (written by make_golden.py:csvmonkey_cells)"""
    import hashlib
    g = np.load(os.path.join(HERE, "golden", "csvmonkey_cells.npz"))
    data = _zillow_csv()
    dump = po.csv_parse(data, [S] * 10, null_values=[], dump_cells=True).dump
    assert hashlib.sha256(dump).digest() == g["zillow_sha256"].tobytes()
    inputs, io_, cells, co = g["inputs"].tobytes(), g["input_offsets"], g["cells"].tobytes(), g["cell_offsets"]
    assert len(io_) == len(co) == 1541
    for it in range(1540):
        s, ref = inputs[io_[it]:io_[it + 1]], cells[co[it]:co[it + 1]]
        ncols = 1 if it < 1500 else 5  # seeded byte soup, then gen_csv tables of 5 columns
        assert po.csv_parse(s, [S] * ncols, null_values=[], dump_cells=True).dump == ref, s


def test_device_code_on_host_equals_oracle_fuzz():
    rng = random.Random(11)
    seq = 0
    for it in range(400):
        ncols = rng.randint(1, 7)
        types = [rng.choice([I, F, B, S, S, X]) for _ in range(ncols)]
        data = gen_csv(rng, rng.randint(0, 80), types, dirty=rng.choice([0.0, 0.05, 0.3]), weird_quotes=rng.choice([0.0, 0.0, 0.02]))
        kw = dict(header=rng.random() < 0.5, null_values=rng.choice([[], [""], ["", "NULL"]]))
        a = host_parse(data, types, **kw)
        b = po.csv_parse(data, types, **kw)
        assert_same_parse(a, b, what=(it, data[:200]))
        seq += a.sequential
    assert seq > 0  # the repair path was exercised
    # raw byte soup around the structural characters
    alpha = ["a", '"', ",", "\n", "\r", "1", '""', ',"', '",']
    for it in range(3000):
        data = "".join(rng.choice(alpha) for _ in range(rng.randint(0, 200))).encode()
        types = [S, I][: rng.randint(1, 2)]
        assert_same_parse(host_parse(data, types), po.csv_parse(data, types), what=data)


def test_zillow_fixture_parses_to_the_pipeline_columns():
    """The raw CSV fixture of the reference (header + 32,661 rows, quoted cells with commas) parsed with projection
    pushdown gives exactly the pre-split column fixture the Zillow parity tests use."""
    import csv as pycsv
    import io
    data = _zillow_csv()
    types = [S, S, S, S, F, S, S, X, S, X]  # postal_code is f64 in the inferred schema; provider / sales_date unused
    for parse in (po.csv_parse, host_parse):
        r = parse(data, types, header=True, null_values=[""])
        assert r.n_rows == 32661 and not r.bad
        rows = list(pycsv.reader(io.StringIO(data.decode())))[1:]
        for c, src in zip(range(8), [0, 1, 2, 3, 4, 5, 6, 8]):
            if r.types[c] == T_STR:
                by, offs = r.columns[c]
                for i in (0, 1, 17, 4000, 32660):
                    assert by[offs[i]:offs[i + 1]].decode() == rows[i][src]
            else:
                assert r.columns[c][0] == 1801.0 and r.columns[c][32660] == float(rows[32660][src])


# ---- CSV sink (K7) -----------------------------------------------------------------------------------------------------
def _cols_from(values_by_col, types):
    from tuplex_b200.backend import Column
    return [Column.from_values(v, t) for v, t in zip(values_by_col, types)]


def test_quote_for_csv_known_answers():
    """tuplex/test/runtime/RuntimeTest.cc:207-213 (quoteForCSV) through the oracle and through the device code on the host"""
    from csv_helpers import host_csv_write
    cases = [("", ""), ("hello", "hello"), (",,,,", '",,,,"'), ("\n\r", '"\n\r"'), ('"', '""""'), ('""', '""""""'), (',"a"\n', '",""a""\n"')]
    for raw, want in cases:
        cols = _cols_from([[raw]], [T_STR])
        assert po.csv_write(cols, 1) == (want + "\n").encode(), raw
        assert host_csv_write(cols, 1) == (want + "\n").encode(), raw


def test_sink_device_code_on_host_equals_oracle_fuzz():
    from csv_helpers import host_csv_write
    rng = random.Random(99)
    words = ["", "a", "x,y", 'q"q', "l\nb", "r\rb", "plain text", "é", '""', ";", "tab\t"]
    for it in range(300):
        ncols = rng.randint(1, 6)
        types = [rng.choice([T_I64, T_BOOL, T_STR, T_STR]) for _ in range(ncols)]
        n = rng.randint(0, 40)
        vals = []
        for t in types:
            if t == T_I64:
                vals.append([rng.choice([0, -1, 9, 10, -10, 2**63 - 1, -2**63, rng.randint(-10**18, 10**18)]) for _ in range(n)])
            elif t == T_BOOL:
                vals.append([rng.random() < 0.5 for _ in range(n)])
            else:
                vals.append([rng.choice(words) for _ in range(n)])
        cols = _cols_from(vals, types)
        d = rng.choice([",", ";", "|"])
        assert host_csv_write(cols, n, delimiter=d) == po.csv_write(cols, n, delimiter=d), (it, types)


def test_sink_zillow_output_is_the_golden_file():
    """the Z1 output columns (oracle run of the stage) through the sink oracle = the reference baselines' output file"""
    from tuplex_b200 import workloads
    from tuplex_b200.backend import Column
    from csv_helpers import host_csv_write
    cols, n = workloads.load_zillow_fixture()
    ora = po.run_program(workloads.zillow_program(), cols, n)
    out_cols = [Column(t, d, o) for t, d, o in ora.columns]
    golden = workloads.zillow_golden_csv()
    body = golden.split(b"\n", 1)[1]
    assert po.csv_write(out_cols, ora.n_out) == body
    assert host_csv_write(out_cols, ora.n_out) == body


def test_sink_f64_fixed8_exact():
    """device f64 formatter (exact 128-bit integer arithmetic) vs the oracle's printf("%.8f") on ties, boundaries, specials"""
    import struct as st
    from csv_helpers import host_csv_write
    rng = random.Random(123)
    vals = [0.0, -0.0, 1.5, -2.25, 2**-9, 3 * 2**-9, 0.000000005, 0.000000015, 0.999999995, 0.9999999949999999, 1e-9, -1e-10, 123456789.123456789,
            9.007199254740992e15, 2**62 * 1.0, -(2**63 - 1024) * 1.0, 5e-324, 2.2250738585072014e-308, 1 / 3, 2 / 3, 1801.0, 0.07, 99999999.999999994,
            float("inf"), float("-inf"), float("nan")]
    for _ in range(20000):
        r = rng.random()
        if r < 0.3:
            vals.append(st.unpack("<d", st.pack("<Q", rng.getrandbits(64)))[0])
        elif r < 0.6:
            vals.append(rng.uniform(-1e6, 1e6))
        elif r < 0.8:
            vals.append(rng.randint(-10**9, 10**9) / 10 ** rng.randint(0, 12))
        else:
            vals.append(rng.randint(0, 2**20) * 2.0 ** -rng.randint(1, 40))  # many exact ties at the 8th decimal
    small = [v for v in vals if v != v or abs(v) == float("inf") or abs(v) < 2.0**63]
    cols = _cols_from([small], [T_F64])
    assert host_csv_write(cols, len(small)) == po.csv_write(cols, len(small))


def test_numeric_cells_decode_fuzz():
    """numeric / bool cells through the register-resident cell path (<= 32 bytes), the memory path (longer cells) and the
    dequoting path (escaped cells), all against the oracle"""
    rng = random.Random(77)

    def cell():
        r = rng.random()
        if r < 0.3:
            return str(rng.randint(-10**18, 10**18))
        if r < 0.5:
            return f"{rng.uniform(-1e9, 1e9):.{rng.randint(0, 17)}f}"
        if r < 0.6:
            return " " * rng.randint(0, 20) + str(rng.randint(0, 99999)) + "\t" * rng.randint(0, 20)
        if r < 0.7:
            return "0" * rng.randint(25, 60) + str(rng.randint(0, 9))
        if r < 0.8:
            return '"' + str(rng.randint(0, 999)) + '"'
        if r < 0.85:
            return '"1""2"'
        if r < 0.9:
            return rng.choice(["true", "F", "yes", "No", "nan", "inf", "1e5", "-", "+3", ""])
        return rng.choice(["abc", "1.2.3", "--1", "9" * 40])
    for it in range(400):
        types = [rng.choice([I, F, B]) for _ in range(rng.randint(1, 5))]
        rows = [",".join(cell() for _ in types) for _ in range(rng.randint(1, 40))]
        data = ("\n".join(rows) + "\n").encode()
        assert_same_parse(host_parse(data, types), po.csv_parse(data, types), what=data[:100])
