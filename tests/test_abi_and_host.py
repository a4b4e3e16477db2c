"""No-GPU checks: the C-ABI library builds for sm_100a, loads, and exports every symbol include/tplx_gpu.h
declares; compute entry points fail loudly without a device (no CPU fallback); host-side logic."""
import ctypes as ct
import os
import re

import numpy as np
import pytest

from tuplex_b200 import backend, frontend, ir, pyexec, workloads
from tuplex_b200.context import Context
from tuplex_b200.dataset import _merge_by_rowno
from tuplex_b200.ir import T_F64, T_I64, T_STR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol(built):
    hdr = open(os.path.join(ROOT, "include", "tplx_gpu.h")).read()
    declared = sorted(set(re.findall(r"\b(tplx_gpu_[a-z_0-9]+)\s*\(", hdr)))
    assert len(declared) >= 25
    L = ct.CDLL(os.path.join(ROOT, "tuplex_b200", "lib", "libtplx_gpu.so"))
    for name in declared:
        assert hasattr(L, name), f"{name} declared in tplx_gpu.h but not exported"
    assert sorted(backend.lib()._declared) == declared  # the Python binding covers the whole ABI


def test_sass_is_sm100a(built):
    import subprocess
    out = subprocess.run(["cuobjdump", "-lelf", os.path.join(ROOT, "tuplex_b200", "lib", "libtplx_gpu.so")], capture_output=True, text=True).stdout
    assert "sm_100a" in out


# every GPU hidden from a child process: the checks of a machine without a device hold on a GPU machine too
NO_DEVICE_ENV = dict(os.environ, CUDA_VISIBLE_DEVICES="")

NO_CPU_FALLBACK = r'''
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from tuplex_b200 import backend, workloads
from tuplex_b200.ir import T_I64
assert backend.device_count() == 0
try:
    backend.init([0])
    sys.exit("init([0]) succeeded without a device")
except backend.GpuBackendError:
    pass
st = backend.Stage(workloads.c1_program())  # descriptor validation works without a device
try:
    st.run_host(0, [backend.Column(T_I64, np.arange(4))], 4)
    sys.exit("run_host succeeded without a device")
except backend.GpuBackendError:
    pass
print("no cpu fallback ok")
'''


def test_no_cpu_fallback(built):
    import subprocess
    import sys
    r = subprocess.run([sys.executable, "-c", NO_CPU_FALLBACK, ROOT], env=NO_DEVICE_ENV, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "no cpu fallback ok" in r.stdout, r.stdout + r.stderr


def test_descriptor_validation(built):
    blob = bytearray(workloads.zillow_program().serialize())
    bad = bytes(blob[:-8])
    h = ct.c_void_p()
    buf = ct.create_string_buffer(bad, len(bad))
    assert backend.lib().tplx_gpu_stage_create(buf, len(bad), ct.byref(h)) == ir.C.get("TPLX_E_BADDESC", -3)
    blob[0] ^= 0xFF
    buf = ct.create_string_buffer(bytes(blob), len(blob))
    assert backend.lib().tplx_gpu_stage_create(buf, len(blob), ct.byref(h)) != 0
    assert b"magic" in backend.lib().tplx_gpu_last_error()


def test_frontend_lowering_shapes():
    p = workloads.zillow_program()
    assert p.prefilter is not None and p.hidden_out_cols == 1 and len(p.out_cols) == 12
    assert [t for _, t in p.out_cols][:11].count(T_STR) == 7
    assert len(p.opids) >= 12 and p.opids[0] == 100001
    q = workloads.q6_program()
    assert q.endpoint == ir.C["TPLX_EP_AGGREGATE"] and len(q.accs) == 1 and q.accs[0].kind == ir.C["TPLX_ACC_SUM_F64"]
    # unsupported constructs fall back instead of miscompiling
    sc = frontend.StageCompiler([T_I64], [None])
    with pytest.raises(frontend.UnsupportedUDF):
        sc.add_map(lambda x: [x, x], 100001)
    sc = frontend.StageCompiler([T_STR], [None])
    with pytest.raises(frontend.UnsupportedUDF):
        sc.add_map(lambda x: x.split(","), 100001)
    with pytest.raises(frontend.UnsupportedUDF):
        frontend.StageCompiler([T_I64], [None]).finish_aggregate(lambda a, x: a * x, lambda a, b: a * b, 1, 1)


def test_parallelize_majority_type_and_fallback_rows():
    ctx = Context({"tuplex.gpu.optionColumns": False})  # rows with None leave the normal case
    src = ctx._source_from_rows([1, 2, None, 4], None)
    assert [c.type for c in src.cols] == [T_I64] and src.n_rows == 3
    assert src.fallback == [(2, None)] and src.orig_index.tolist() == [0, 1, 3]
    ctx = Context()  # default: None stays in the normal case, the column becomes Option[i64] (validity bitmap)
    src = ctx._source_from_rows([1, 2, None, 4], None)
    assert [c.type for c in src.cols] == [T_I64] and src.n_rows == 4 and not src.fallback
    assert src.cols[0].valid.tolist() == [0b1011] and src.cols[0].to_values() == [1, 2, None, 4]
    src = ctx._source_from_rows([(1, "a"), (2, "b"), (3.5, "c"), ("x", "d")], ["n", "s"])
    assert [c.type for c in src.cols] == [T_I64, T_STR] and src.n_rows == 2 and len(src.fallback) == 2


def test_merge_by_row_number():
    """ResolveTask::executeInOrder semantics: exception k sits at slot row_no_k of the output stream."""
    exc = np.array([(2, 2, 136, 1), (5, 4, 136, 1)], dtype=backend.EXC_DTYPE)  # rows 2 and 5 raised
    normal = ["r0", "r1", "r3", "r4", "r6"]
    assert _merge_by_rowno(normal, exc, [(2, 2, "R2"), (5, 4, "R5")]) == ["r0", "r1", "R2", "r3", "R5", "r4", "r6"][:0] + ["r0", "r1", "R2", "r3", "R5", "r4", "r6"]
    assert _merge_by_rowno(normal, exc, [(5, 4, "R5")]) == ["r0", "r1", "r3", "R5", "r4", "r6"]
    assert _merge_by_rowno(normal, exc[:0], []) == normal


def test_cpython_slow_path_with_resolvers():
    op = pyexec.Op("map", lambda x: 10 // x)
    op.resolvers.append((ZeroDivisionError, lambda x: -1))
    assert pyexec.run_row([op], 0, [None])[0] == -1
    op2 = pyexec.Op("map", lambda x: 10 // x)
    op2.ignores.append(ZeroDivisionError)
    with pytest.raises(pyexec.Dropped):
        pyexec.run_row([op2], 0, [None])
    ops = [pyexec.Op("withColumn", lambda x: x["a"] + 1, column="b"), pyexec.Op("filter", lambda x: x["b"] > 2),
           pyexec.Op("selectColumns", columns=["b"])]
    assert pyexec.run_row(ops, (5,), ["a"]) == (6, ["b"])
    assert pyexec.exception_code(ValueError()) == 135 and pyexec.exception_code(ZeroDivisionError()) == 136


def test_shard_ranges():
    from tuplex_b200.dist import shard_range
    for n in (0, 1, 7, 600):
        for w in (1, 2, 4, 8):
            parts = [shard_range(n, r, w) for r in range(w)]
            assert parts[0][0] == 0 and parts[-1][1] == n
            assert all(parts[i][1] == parts[i + 1][0] for i in range(w - 1))
            assert max(h - l for l, h in parts) - min(h - l for l, h in parts) <= 1


def test_frontend_breadth_vs_cpython(built):
    """Constructs beyond the benchmark UDFs: membership in literal containers, min/max, str.format / f-strings with
    integer specs, dict-valued map; each lowered program run by the oracle must equal CPython."""
    from oracle import pyoracle
    rows = [(i - 5, "w%d" % (i % 3), float(i) / 4) for i in range(40)]
    cols = [backend.Column.from_values([r[0] for r in rows], T_I64), backend.Column.from_values([r[1] for r in rows], T_STR),
            backend.Column.from_values([r[2] for r in rows], T_F64)]
    udfs = [
        lambda x: (x['a'] in (1, -2, 7), x['s'] not in ['w0', 'zz'], min(x['a'], 3), max(x['f'], 1.5), min(x['a'], x['f'])),
        lambda x: ('{:03}|{}'.format(x['a'], x['s']), f"{x['a']:04}:{x['s']}!", '{1}-{0:4d}'.format(x['a'], x['s']), f"{x['s']}{x['a']}"),
        lambda x: {'k': x['s'].upper(), 'v': x['a'] * 2},
    ]
    for f in udfs:
        sc = frontend.StageCompiler([T_I64, T_STR, T_F64], ["a", "s", "f"])
        sc.add_map(f, 100001)
        prog = sc.finish_memory()
        res = pyoracle.run_program(prog, cols, len(rows))
        got = list(zip(*[res.values(c) for c in range(len(res.columns))]))
        exp = []
        for r in rows:
            v = f(pyexec.Row(r, ["a", "s", "f"]))
            exp.append(tuple(v.values()) if isinstance(v, dict) else v)
        assert got == exp
    sc = frontend.StageCompiler([T_I64, T_STR, T_F64], ["a", "s", "f"])
    sc.add_map(udfs[2], 100001)
    sc.finish_memory()
    assert sc.names == ["k", "v"]


def test_csv_source_planning_and_chunking(tmp_path, monkeypatch):
    """host side of Context.csv: sniffing / header / type inference from a sample, and chunking of large inputs at row
    boundaries (quote parity) — chunks re-joined must give the same rows as one pass."""
    import numpy as np
    from tuplex_b200 import csvsource as cs
    from tuplex_b200.ir import T_F64, T_I64, T_STR
    from csv_helpers import gen_csv
    import random
    rng = random.Random(4)
    body = gen_csv(rng, 400, [T_I64, T_STR, T_F64, T_STR], dirty=0.0)
    p = tmp_path / "t.csv"
    p.write_bytes(b"id,name,score,note\n" + body)
    import tuplex_b200
    ds = tuplex_b200.Context().csv(str(p))
    src = ds._source
    assert src.names == ["id", "name", "score", "note"] and src.header and src.delimiter == ","
    assert src.types == [T_I64, T_STR, T_F64, T_STR]
    whole = [cells for cells, _, _ in cs.iter_rows(src.files[0].tobytes(), 44, 34)]
    monkeypatch.setattr(cs, "MAX_CHUNK", 997)
    parts = list(src.chunks())
    assert len(parts) > 10 and parts[0][1] is True and not any(h for _, h in parts[1:])
    assert b"".join(d.tobytes() for d, _ in parts) == src.files[0].tobytes()
    joined = [cells for d, _ in parts for cells, _, _ in cs.iter_rows(d.tobytes(), 44, 34)]
    assert joined == whole
    # interpreter-path decoders: typed (as the device decodes) vs general (`parse` of the reference's fallback code)
    assert src.line_object(b'7,"a,b",1.50,x', True) == (7, "a,b", 1.5, "x")
    assert src.line_object(b"n/a,t,,x", False) == ("n/a", True, None, "x")
    hs = src.to_host_source()
    assert hs.n_rows + len(hs.fallback) == 400


def test_csv_missing_file_gives_empty_dataset(tmp_path):
    """tuplex/python/tests/test_csv.py:66-69 (test_non_existent_file): no exception, nothing to show"""
    import tuplex_b200
    ctx = tuplex_b200.Context()
    ds = ctx.csv(str(tmp_path / "missing_file.ccc"))
    assert ds.collect() == []
    ds.show()
    assert any("no such file" in m for m in ctx._messages)


def test_cpp_host_join_fails_loudly_without_a_device(built, tmp_path):
    """tplx_host_run --join (GpuBackend::execute(GpuHashJoinStage&)) has no CPU path either: without a device it exits non-zero with the
    library's message instead of producing rows."""
    import subprocess
    from oracle import pyoracle
    cols = [backend.Column(T_I64, np.arange(4, dtype=np.int64))]
    (part,) = pyoracle.to_partitions(cols, 4, 1 << 16)
    f = tmp_path / "p.bin"
    f.write_bytes(part)
    exe = os.path.join(ROOT, "tuplex_b200", "lib", "tplx_host_run")
    r = subprocess.run([exe, "--join", "0", "0", "0", "0", "0", str(1 << 16), str(tmp_path / "out"), "0", "1", str(f), str(f)],
                       env=NO_DEVICE_ENV, capture_output=True, text=True, timeout=60)
    assert r.returncode != 0 and "error" in r.stderr.lower()
    assert not (tmp_path / "out.out0").exists()
