"""Generates the golden fixtures under tests/golden/ from the reference's own test resources and the
reference's own hand-written C++ Zillow pipeline (built by oracle/Makefile into oracle/_ref/).
Run in the build container (needs /root/reference); the outputs are committed, this script documents
how they were made. Nothing at test/bench time reads /root/reference.

  zillow_noexc_cols.csv.gz   the 8 columns the Z1 pipeline reads (benchmarks/zillow/Z1/baseline/zillow.cpp:19-27)
                             of tuplex/test/resources/pipelines/zillow/zillow_noexc.csv (32,661 rows)
  zillow_noexc_out.csv.gz    output of oracle/_ref/zillow_ref (= unmodified zillow.cpp) on that file,
                             md5 4d5ca0263b1a5058341a369116dee83a (also produced by benchmarks/zillow/Z1/runpython.py)
  lineitem_q6.npz            l_quantity, l_extendedprice, l_discount, l_shipdate(yyyymmdd) of
                             tuplex/test/resources/tpch/lineitem.tbl (60,175 rows); golden Q6 = 1193053.2252999984
                             (tuplex/test/core/TPCH.cc:85-97)
"""
import csv, gzip, hashlib, io, os, subprocess, sys, tempfile
import numpy as np

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
COLS = ["title", "address", "city", "state", "postal_code", "price", "facts and features", "url"]

src = os.path.join(REF, "tuplex/test/resources/pipelines/zillow/zillow_noexc.csv")
rows = list(csv.DictReader(open(src, newline="")))
buf = io.StringIO()
w = csv.writer(buf, lineterminator="\n")
w.writerow(COLS)
for r in rows:
    w.writerow([r[c] for c in COLS])
with gzip.GzipFile(os.path.join(HERE, "zillow_noexc_cols.csv.gz"), "wb", mtime=0) as fp:
    fp.write(buf.getvalue().encode())

with tempfile.TemporaryDirectory() as td:
    subprocess.check_call([os.path.join(ROOT, "oracle/_ref/zillow_ref"), "--path", src, "--output_path", td, "--preload"],
                          stdout=subprocess.DEVNULL)
    out = open(os.path.join(td, "part0.csv"), "rb").read()
assert hashlib.md5(out).hexdigest() == "4d5ca0263b1a5058341a369116dee83a", hashlib.md5(out).hexdigest()
with gzip.GzipFile(os.path.join(HERE, "zillow_noexc_out.csv.gz"), "wb", mtime=0) as fp:
    fp.write(out)

q, p, d, s = [], [], [], []
for line in open(os.path.join(REF, "tuplex/test/resources/tpch/lineitem.tbl")):
    f = line.split("|")
    q.append(int(f[4])); p.append(float(f[5])); d.append(float(f[6])); s.append(int(f[10].replace("-", "")))
np.savez_compressed(os.path.join(HERE, "lineitem_q6.npz"), l_quantity=np.array(q, np.int64), l_extendedprice=np.array(p, np.float64),
                    l_discount=np.array(d, np.float64), l_shipdate=np.array(s, np.int64))
# the gtest golden, recomputed as a sequential sum in file order with the literal bounds of runtuplex.py:96-99
acc = 0.0
for qq, pp, dd, ss in zip(q, p, d, s):
    if 19940101 <= ss < 19950101 and 0.05 <= dd <= 0.07 and qq < 24:
        acc = acc + pp * dd
assert repr(acc) == "1193053.2252999984", repr(acc)
print("golden fixtures written; q6 =", repr(acc), "rows", len(q))


def zillow_full_fixture():
    """tests/golden/zillow_noexc.csv.gz = the reference's fixture file as is (10 columns, header, quoted cells),
    gzip'ed with mtime 0: input of the CSV-source (K6) parity tests."""
    import gzip
    import shutil
    src = "/root/reference/tuplex/test/resources/pipelines/zillow/zillow_noexc.csv"
    with open(src, "rb") as f, gzip.GzipFile(os.path.join(os.path.dirname(os.path.abspath(__file__)), "zillow_noexc.csv.gz"), "wb", mtime=0) as g:
        shutil.copyfileobj(f, g)


zillow_full_fixture()


def zillow_reference_udfs():
    """tests/golden/zillow_z1_udfs_ref.py = the UDF definitions of the reference's Z1 benchmark script, LITERALLY
    (benchmarks/zillow/Z1/runtuplex.py: extractBd ... filterBd). A fixture (the workload's user code), so that a parity test can
    lower the reference's own statements (intermediate variables and all) instead of this repo's re-worded workloads.py."""
    src = open("/root/reference/benchmarks/zillow/Z1/runtuplex.py").read()
    a = src.index("def extractBd(x):")
    b = src.index("if __name__ == \"__main__\":") if "if __name__ == \"__main__\":" in src else src.index("if __name__ == '__main__':")
    body = src[a:b].rstrip() + "\n"
    hdr = ('"""LITERAL copy of the UDFs of /root/reference/benchmarks/zillow/Z1/runtuplex.py (test fixture: the workload\'s user code),\n'
           'written by tests/golden/make_golden.py:zillow_reference_udfs. Do not edit."""\n\n')
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "zillow_z1_udfs_ref.py"), "w") as fp:
        fp.write(hdr + body)


zillow_reference_udfs()


def csvmonkey_cells():
    """tests/golden/csvmonkey_cells.npz = what the reference's own csvmonkey reader (oracle/_ref/csv_ref) makes of
    the cell-splitting vectors of tests/test_csv_oracle.py::test_cells_equal_reference_csvmonkey:
      inputs / input_offsets   1,540 inputs with pathological quoting (seeded), concatenated
      cells / cell_offsets     the reader's cell dump of each input
      zillow_sha256            sha256 of its cell dump of tests/golden/zillow_noexc.csv.gz (the dump itself is 7.7 MB)"""
    import random
    sys.path[:0] = [ROOT, os.path.dirname(HERE)]
    from oracle import pyoracle as po
    from csv_helpers import T_BOOL, T_F64, T_I64, T_STR, gen_csv
    rng = random.Random(7)
    alpha = ["a", "b", '"', ",", "\n", "\r", " ", "1", "x", '""', ',"', '"\n', '",', "\r\n"]
    inputs = ["".join(rng.choice(alpha) for _ in range(rng.randint(0, 60))).encode() for _ in range(1500)]
    inputs += [gen_csv(rng, 30, [T_I64, T_STR, T_F64, T_STR, T_BOOL], dirty=0.2, weird_quotes=0.05) for _ in range(40)]
    cells = [po.csv_ref_cells(s) for s in inputs]
    offs = lambda parts: np.cumsum([0] + [len(p) for p in parts], dtype=np.uint64)
    zillow = gzip.open(os.path.join(HERE, "zillow_noexc.csv.gz"), "rb").read()
    np.savez_compressed(os.path.join(HERE, "csvmonkey_cells.npz"),
                        inputs=np.frombuffer(b"".join(inputs), np.uint8), input_offsets=offs(inputs),
                        cells=np.frombuffer(b"".join(cells), np.uint8), cell_offsets=offs(cells),
                        zillow_sha256=np.frombuffer(hashlib.sha256(po.csv_ref_cells(zillow)).digest(), np.uint8))


csvmonkey_cells()
