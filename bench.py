#!/usr/bin/env python
"""bench.py — rows/s of the hot path on B200, next to the HBM roofline and the reference's CPU path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload zillow|q6|c1] [--rows R] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the stage over the whole synthetic workload. Default workload = BASELINE.json
configs[1]: the Zillow Z1 pipeline over 100M synthetic rows (cyclic replication of the reference's 32,661-row
fixture, the reference's own generator benchmarks/zillow/Z1/sample_zillow.py:20-45), column-blocked, one GPU.
Prints ONE JSON line (rank 0). See the prompt contract in DESIGN.md §Measurement for every key.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# Steady-state measurement: the stage specialiser (csrc/jit.inl) compiles a stage once per process; by default that happens on a
# background thread while the interpreting kernels keep working. Here the first warm-up step waits for it, so that every timed step
# runs the same kernels (TPLX_JIT=0 measures the interpreting kernels).
os.environ.setdefault("TPLX_JIT_SYNC", "1")

import numpy as np  # noqa: E402


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="both", choices=["both", "zillow", "q6", "c1", "aggbykey", "zillow_csv", "q6_csv"],
                    help="both (default) = BASELINE.json's metric: Zillow Z1 (top level of the line) + TPC-H Q6 (nested under \"q6\")")
    ap.add_argument("--rows", type=int, default=0, help="rows per GPU (default: 100M zillow / 600M q6 / 1e6*100 c1)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-sample-rows", type=int, default=1_000_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--keys", type=int, default=0, help="distinct keys of the aggbykey workload (default rows/100)")
    ap.add_argument("--min-region-s", type=float, default=0.0,
                    help="repeat the K-step timed region (each repeat bracketed by barrier + synchronize) until this much time has "
                         "been measured and report the median repeat; by default the K steps run once")
    ap.add_argument("--no-pageable", action="store_true", help="skip the pageable-host-memory end-to-end variant")
    ap.add_argument("--no-extras", action="store_true", help="default workload only: skip the brief c1 / aggregateByKey measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the headline workloads' last timed step returned to DIR/*.npy "
                         f"(float32 / float64, at most {DUMP_LIMIT >> 20} MB; rank 0; see OutputDump)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what this project's timed path computed: use it with --impl ours")
    return args


DUMP_LIMIT = 64 << 20  # bytes of .npy data one --dump-outputs run writes at most


class OutputDump:
    """--dump-outputs DIR: what a workload's timed path returned in its last timed step, as DIR/<workload>.<array>.npy in float32 or
    float64, so that two builds of the project can be compared output for output (the inputs are generated from fixed seeds).

      <wl>.result            aggregate stages: the aggregate of every block (one value per block)
      <wl>.rows              row stages: number of output rows; the rows are the output of every block in block order (hash
                             tables: the groups sorted by value, their order in the table is not part of the result)
      <wl>.sample            indices of the rows written: all of them, or a fixed, seeded sample when they exceed the size limit
      <wl>.<NN_col>          a fixed-width output column (float64; i64 values beyond 2^53 are rounded)
      <wl>.<NN_col>.bytes    a string column: the bytes of the sampled rows (float32, one value per byte; absent when all are empty) ...
      <wl>.<NN_col>.lengths  ... and their lengths
      <wl>.<NN_col>.valid    an Option column: 1 = the row holds a value
      <wl>.exceptions.*      the same for the exception records (row in block, row number, code, operator id)
    No array of length 0 is written: a table without rows is only its .rows file."""

    def __init__(self, path, n_workloads):
        os.makedirs(path, exist_ok=True)
        self.path = path
        self.limit = (DUMP_LIMIT - (1 << 20)) // n_workloads  # 1 MB left for the .npy headers and the one-value arrays

    def _save(self, name, a):
        np.save(os.path.join(self.path, name + ".npy"), a)

    def aggregate(self, wl_name, values):
        self._save(f"{wl_name}.result", np.array(values, np.float64))

    def rows(self, wl_name, prog, blocks, exceptions, sort=False):
        """blocks: the output columns (backend.Column) of every block of stage `prog`; exceptions: the EXC_DTYPE records of every block."""
        from tuplex_b200.backend import EXC_DTYPE, Column
        from tuplex_b200.ir import T_I64
        names = [(prog.out_names[i] if i < len(prog.out_names) else None) or f"col{i}" for i in range(len(blocks[0]))]
        exc = np.concatenate(exceptions) if exceptions else np.zeros(0, EXC_DTYPE)
        exc_cols = [Column(T_I64, np.ascontiguousarray(exc[f])) for f in EXC_DTYPE.names]
        self._table(f"{wl_name}.exceptions", list(EXC_DTYPE.names), [[c] for c in exc_cols], self.limit // 8, False)
        self._table(wl_name, names, [[b[c] for b in blocks] for c in range(len(names))], self.limit - self.limit // 8, sort)

    def _table(self, prefix, names, parts, limit, sort):
        from tuplex_b200.ir import T_STR
        cols = []
        for ps in parts:  # one column over the blocks: fixed-width values, or string bytes + row starts + lengths
            present = None
            if any(p.valid is not None for p in ps):
                present = np.concatenate([p.present() if p.valid is not None else np.ones(len(p), bool) for p in ps])
            if ps[0].type == T_STR:
                base = np.cumsum([0] + [len(p.data) for p in ps])
                starts = np.concatenate([p.offsets[:-1].astype(np.int64) + b for p, b in zip(ps, base)])
                lens = np.concatenate([np.diff(p.offsets.astype(np.int64)) for p in ps])
                cols.append((np.concatenate([p.data for p in ps]), starts, lens, present))
            else:
                cols.append((np.concatenate([p.data for p in ps]).astype(np.float64), None, None, present))
        n = len(cols[0][0]) if cols[0][1] is None else len(cols[0][1])
        order = np.arange(n)
        if sort and n:
            keys = []
            for data, starts, lens, present in cols:
                if starts is not None:
                    data = np.unique(np.array([data[s:s + l].tobytes() for s, l in zip(starts, lens)], dtype=object).astype(bytes),
                                     return_inverse=True)[1]
                keys += [data] + ([present] if present is not None else [])
            order = np.lexsort(keys[::-1])
        row_bytes = np.full(n, 8, np.int64)  # its index in <prefix>.sample
        for _, starts, lens, present in cols:
            row_bytes += 8 if starts is None else 8 + 4 * lens
            row_bytes += 0 if present is None else 4
        idx = np.arange(n)
        if row_bytes.sum() > limit:
            cand = np.random.default_rng(0).choice(n, size=min(n, limit // 8), replace=False)
            idx = np.sort(cand[np.cumsum(row_bytes[order[cand]]) <= limit])
        rows = order[idx]
        self._save(f"{prefix}.rows", np.array([n], np.float64))
        if n == 0:  # no arrays of length 0: the row count says that there is nothing
            return
        self._save(f"{prefix}.sample", idx.astype(np.float64))
        for i, (name, (data, starts, lens, present)) in enumerate(zip(names, cols)):
            stem = "%s.%02d_%s" % (prefix, i, "".join(ch if ch.isalnum() else "_" for ch in name))
            if starts is None:
                self._save(stem, data[rows])
            else:
                ln = lens[rows]
                pos = np.repeat(starts[rows] - (np.cumsum(ln) - ln), ln) + np.arange(int(ln.sum()))
                if len(pos):
                    self._save(stem + ".bytes", data[pos].astype(np.float32))
                self._save(stem + ".lengths", ln.astype(np.float64))
            if present is not None:
                self._save(stem + ".valid", present[rows].astype(np.float32))


# ------------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------------
class Clocks:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 8:
                self.samples.append(f)

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        mx = [float(s[2]) for s in self.samples if s[2].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(self.samples)}


STAGE_KERNEL_SOURCES = ("strops.cuh", "csvops.cuh", "vm.cuh", "kernels.cuh", "vecvm.cuh", "fused.cuh", "mask.cuh", "jit.inl")


def kernel_source_hash():
    """sha256 over the sources of the stage kernels the headline workloads launch (row / mask / vector / fused kernels, the VM, the string
    primitives, the specialiser): the key that ties profiles/traffic.json (DRAM bytes from an `ncu --set full` capture, tools/make_traffic.py)
    to the code it was captured from. Sources of other kernels (CSV, join, merge, hash) do not enter it."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "tuplex_b200", "csrc")
    for f in STAGE_KERNEL_SOURCES:
        h.update(f.encode())
        h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def ncu_traffic(wl, n_launch):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed ncu capture summarised in
    profiles/traffic.json, scaled to this run's rows per launch. The file records the hash of the kernel sources it was
    captured from: when the sources have changed since, the number is stale and None is reported instead."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    t = json.load(open(p))
    if t.get("kernel_source_hash") != kernel_source_hash():
        return None
    per_row = t.get("dram_bytes_per_row", {}).get(wl["name"])
    if per_row is None:
        return None
    return per_row * wl["rows"] / n_launch


def host_cores(calibrate=True):
    """CPU cores this process may really use: scheduler affinity, capped by the cgroup CPU quota (a quota-limited container
    still sees every core in os.cpu_count(); oversubscribing it made round 1's CPU arm 7x too slow on the 1-GPU lease)."""
    visible = os.cpu_count() or 1
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = visible
    quota = None
    try:
        txt = open("/sys/fs/cgroup/cpu.max").read().split()
        if txt and txt[0] != "max":
            quota = float(txt[0]) / float(txt[1])
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    used = aff if quota is None else max(1, min(aff, int(quota + 0.5)))
    out = {"cores_visible": visible, "cores_affinity": aff, "cores_quota": quota, "cores_used": used}
    if calibrate:
        # what the box really delivers (catches limits the cgroup files do not show): use no more processes than that
        par = effective_parallelism(used)
        out["parallelism_measured"] = round(par, 1)
        if par < 0.7 * used:  # suspicious: the CPU arm is then ALSO run with this many processes and the faster run is reported
            out["cores_alt"] = max(1, int(par + 0.5))
    return out


def effective_parallelism(procs: int) -> float:
    """Measured: aggregate throughput of `procs` spinning processes / one spinning process (what the box really gives us,
    whatever the cgroup files say)."""
    code = ("import sys,time\nT0=float(sys.argv[1])\nwhile time.time()<T0: pass\nn=0\nwhile time.time()<T0+0.8:\n"
            "    for _ in range(20000): n+=1\nprint(n)")

    def run(k):  # k processes spin over the SAME 0.8 s window (interpreter start-up is kept out of it)
        t0 = time.time() + 0.5 + 0.01 * k
        ps = [subprocess.Popen([sys.executable, "-S", "-E", "-c", code, repr(t0)], stdout=subprocess.PIPE, text=True) for _ in range(k)]
        return sum(int(p.communicate()[0].strip() or 0) for p in ps)
    one = max(1, sorted(run(1) for _ in range(3))[1])
    return max(run(procs) for _ in range(2)) / one


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------------
def pinned(arr: np.ndarray):
    """Copy a numpy array into page-locked host memory (torch is plumbing here: allocator only)."""
    import torch
    t = torch.empty(arr.shape, dtype=torch.from_numpy(arr[:0]).dtype, pin_memory=True)
    out = t.numpy()
    out[...] = arr
    out_flags_keep = t  # keep the tensor alive through the numpy view's base
    return out, out_flags_keep


def unpin(blocks):
    """The same blocks in ordinary pageable memory (plain numpy copies; blocks that share arrays keep sharing the copy)."""
    from tuplex_b200.backend import Column
    memo = {}

    def cp(a):
        if a is None:
            return None
        k = a.ctypes.data
        if k not in memo:
            memo[k] = np.array(a, copy=True)
        return memo[k]
    return [([Column(c.type, cp(c.data), cp(c.offsets)) for c in cols], n) for cols, n in blocks]


def build_workload(args):
    from tuplex_b200 import workloads as W
    from tuplex_b200.backend import Column
    keep = []

    def pin_cols(cols):
        out = []
        for c in cols:
            d, k1 = pinned(c.data)
            keep.append(k1)
            o = None
            if c.offsets is not None:
                o, k2 = pinned(c.offsets)
                keep.append(k2)
            out.append(Column(c.type, d, o))
        return out

    if args.workload == "zillow":
        total = args.rows or 100_000_000
        src, n0 = W.load_zillow_fixture()
        cycles_per_block = 500
        bn = cycles_per_block * n0
        blocks = []
        full = W.replicate(src, n0, min(bn, total))
        full = pin_cols(full)
        done = 0
        while done < total:
            m = min(bn, total - done)
            if m == len(full[0]):
                blocks.append((full, m))
            else:
                blocks.append((pin_cols(W.replicate(src, n0, m)), m))
            done += m
        prog = W.zillow_program()
        in_bytes = sum(sum(c.nbytes() for c in cols) for cols, _ in blocks)
        return dict(name="zillow_z1", prog=prog, blocks=blocks, rows=total, in_bytes=in_bytes, keep=keep, pageable_blocks=lambda: unpin(blocks),
                    desc=f"Zillow Z1 map/withColumn/filter pipeline, {total} synthetic rows (cyclic replication of the 32,661-row "
                         f"zillow_noexc fixture), 8 column-blocked inputs, {len(blocks)} blocks of <= {bn} rows")
    if args.workload == "q6":
        total = args.rows or 600_000_000
        bn = 100_000_000
        blocks = []
        done = 0
        base = pin_cols(W.gen_lineitem(min(bn, total), seed=42))
        while done < total:
            m = min(bn, total - done)
            blocks.append((base if m == len(base[0].data) else [c.slice(0, m) for c in base], m))
            done += m
        prog = W.q6_program()
        return dict(name="tpch_q6", prog=prog, blocks=blocks, rows=total, in_bytes=total * 32, keep=keep, pageable_blocks=lambda: unpin(blocks),
                    desc=f"TPC-H Q6 filter+aggregate, {total} synthetic lineitem rows (SF100 ~ 600M), 4 columns i64,f64,f64,i64")
    if args.workload == "c1":
        total = args.rows or 100_000_000
        x = np.arange(1, total + 1, dtype=np.int64)
        blocks = [(pin_cols([Column(0, x)]), total)]
        return dict(name="c1_map_filter", prog=W.c1_program(), blocks=blocks, rows=total, in_bytes=total * 8, keep=keep,
                    desc=f"parallelize([1..{total}]).map(x*x).filter(x%2==0)")
    total = args.rows or 100_000_000
    nkeys = args.keys or max(1000, total // 100)
    blocks = [(pin_cols(W.gen_keyed(total, nkeys, seed=42 + int(os.environ.get("RANK", "0")))), total)]  # every rank its own shard of rows
    return dict(name="aggbykey_str", prog=W.keyed_program(), blocks=blocks, rows=total, in_bytes=total * 20, keep=keep, nkeys=nkeys,
                desc=f"aggregateByKey string key, {total} rows, {nkeys} distinct keys")


# ------------------------------------------------------------------------------------------------------
# CPU arms
# ------------------------------------------------------------------------------------------------------
def cpu_zillow_reference(sample_rows: int, procs: int):
    """The reference's own hand-written C++ Z1 pipeline (benchmarks/zillow/Z1/baseline/zillow.cpp, built unmodified
    into oracle/_ref/zillow_ref), --preload compute stage, `procs` processes in parallel over the host cores."""
    import gzip
    exe = os.path.join(ROOT, "oracle", "_ref", "zillow_ref")
    if not os.path.exists(exe):
        return None
    with gzip.open(os.path.join(ROOT, "tests", "golden", "zillow_noexc_cols.csv.gz"), "rb") as fp:
        raw = fp.read()
    header, body = raw.split(b"\n", 1)
    n0 = body.count(b"\n")
    reps = max(1, sample_rows // n0)
    rows = reps * n0
    td = tempfile.mkdtemp(prefix="tplx_cpu_")
    path = os.path.join(td, "sample.csv")
    with open(path, "wb") as fp:
        fp.write(header + b"\n")
        for _ in range(reps):
            fp.write(body)
    ps = [subprocess.Popen([exe, "--path", path, "--output_path", os.path.join(td, f"out{i}"), "--preload"], stdout=subprocess.PIPE,
                           stderr=subprocess.DEVNULL, text=True) for i in range(procs)]
    ns = []
    for p in ps:
        out, _ = p.communicate()
        for line in out.splitlines():
            if line.startswith("compute stage:"):
                ns.append(float(line.split()[2]))
    subprocess.call(["rm", "-rf", td])
    if len(ns) != procs:
        return None
    return dict(value=procs * rows / (max(ns) * 1e-9), unit="rows/s", cores=procs, kind="reference", rows_total=procs * rows,
                sample=f"{procs} processes x {rows} rows (cyclic replication of the fixture, CSV preloaded), compute stage of "
                       f"oracle/_ref/zillow_ref = reference benchmarks/zillow/Z1/baseline/zillow.cpp; slowest process {max(ns) * 1e-6:.1f} ms")


def cpu_zillow_csv_reference(sample_rows: int, procs: int):
    """File-to-result arm of the CSV workload: the reference's C++ Z1 baseline in its streaming mode (csvmonkey parse +
    pipeline per row, `transform stage`; benchmarks/zillow/Z1/baseline/zillow.cpp built unmodified into
    oracle/_ref/zillow_ref), `procs` processes in parallel, each over the same CSV file (full 10-column fixture rows)."""
    import gzip
    exe = os.path.join(ROOT, "oracle", "_ref", "zillow_ref")
    if not os.path.exists(exe):
        return None
    with gzip.open(os.path.join(ROOT, "tests", "golden", "zillow_noexc.csv.gz"), "rb") as fp:
        raw = fp.read()
    header, body = raw.split(b"\n", 1)
    n0 = body.count(b"\n")
    reps = max(1, sample_rows // n0)
    rows = reps * n0
    td = tempfile.mkdtemp(prefix="tplx_cpu_")
    path = os.path.join(td, "sample.csv")
    with open(path, "wb") as fp:
        fp.write(header + b"\n")
        for _ in range(reps):
            fp.write(body)
    ps = [subprocess.Popen([exe, "--path", path, "--output_path", os.path.join(td, f"out{i}")], stdout=subprocess.PIPE,
                           stderr=subprocess.DEVNULL, text=True) for i in range(procs)]
    ns = []
    for p in ps:
        out, _ = p.communicate()
        for line in out.splitlines():
            if line.startswith("transform stage:"):
                ns.append(float(line.split()[2]))
    subprocess.call(["rm", "-rf", td])
    if len(ns) != procs:
        return None
    return dict(value=procs * rows / (max(ns) * 1e-9), unit="rows/s", cores=procs, kind="reference", rows_total=procs * rows,
                sample=f"{procs} processes x {rows} rows of raw CSV (cyclic replication of the fixture file), "
                       f"transform stage (csvmonkey parse + pipeline) of oracle/_ref/zillow_ref = reference "
                       f"benchmarks/zillow/Z1/baseline/zillow.cpp; slowest process {max(ns) * 1e-6:.1f} ms")


def _q6_csv_worker(path):
    import time as _t
    from oracle import pyoracle
    from tuplex_b200 import ir
    data = open(path, "rb").read()
    t0 = _t.perf_counter()
    r = pyoracle.csv_parse(data, [ir.T_I64, ir.T_F64, ir.T_F64, ir.T_I64], delimiter="|", header=False)
    v = pyoracle.q6(*r.columns)
    return _t.perf_counter() - t0, r.n_rows, v


def cpu_q6_csv_port(sample_rows: int, procs: int):
    """CPU arm of q6_csv (kind 'port'): oracle/csv_oracle.c (csvmonkey restatement + fast_atoi64 / fast_atod) followed by
    oracle/workloads.c's Q6 loop, one process per host core over the same text (the reference's own LLVM path cannot be
    built here; its C++ Q6 baseline needs weld.h)."""
    import multiprocessing as mp
    from tuplex_b200 import workloads as W
    n = max(100_000, min(sample_rows, 2_000_000))
    q, p_, d_, s_ = (c.data for c in W.gen_lineitem(n, seed=42))
    td = tempfile.mkdtemp(prefix="tplx_cpu_")
    path = os.path.join(td, "lineitem.tbl")
    with open(path, "wb") as fp:
        fp.write(b"\n".join(b"%d|%.2f|%.2f|%d" % (int(a), float(b), float(c), int(e)) for a, b, c, e in zip(q, p_, d_, s_)) + b"\n")
    with mp.get_context("fork").Pool(procs) as pool:
        res = pool.map(_q6_csv_worker, [path] * procs)
    subprocess.call(["rm", "-rf", td])
    slow = max(r[0] for r in res)
    return dict(value=procs * n / slow, unit="rows/s", cores=procs, kind="port", rows_total=procs * n,
                sample=f"{procs} processes x {n} rows of '|'-separated text: oracle/csv_oracle.c parse + oracle/workloads.c Q6 loop; "
                       f"slowest process {slow * 1e3:.1f} ms")


def cpu_port(wl, sample_rows: int, threads: int):
    """oracle port (kind 'port') on a bounded sample."""
    from oracle import pyoracle
    if wl["name"] == "tpch_q6":
        cols = wl["blocks"][0][0]
        m = min(len(cols[0].data), max(sample_rows, 50_000_000))
        a = [c.data[:m] for c in cols]
        t0 = time.perf_counter()
        pyoracle.q6(*a, part_rows=1 << 20, threads=threads)
        dt = time.perf_counter() - t0
        return dict(value=m / dt, unit="rows/s", cores=threads, kind="port",
                    sample=f"{m} rows, oracle/workloads.c Q6 loop, {threads} threads over 1Mi-row partitions, inputs in memory")
    if wl["name"] == "c1_map_filter":
        x = wl["blocks"][0][0][0].data
        m = min(len(x), max(sample_rows, 50_000_000))
        t0 = time.perf_counter()
        pyoracle.c1(x[:m], part_rows=1 << 20, threads=threads)
        dt = time.perf_counter() - t0
        return dict(value=m / dt, unit="rows/s", cores=threads, kind="port",
                    sample=f"{m} rows, oracle/workloads.c C1 loop, {threads} threads")
    cols, n = wl["blocks"][0]
    m = min(n, sample_rows)
    t0 = time.perf_counter()
    pyoracle.run_program(wl["prog"], [c.slice(0, m) for c in cols], m)
    dt = time.perf_counter() - t0
    return dict(value=m / dt, unit="rows/s", cores=1, kind="port", sample=f"{m} rows through oracle/tplx_oracle.c (scalar interpreter)")


def cpu_arm(args, wl_key, wl, hc):
    """One bounded CPU sample of workload `wl_key` on hc['cores_used'] host cores -> cpu_baseline dict."""
    if hc.get("cores_alt") and not hc.get("_in_alt"):
        a = cpu_arm(args, wl_key, wl, dict(hc, cores_alt=None))
        b = cpu_arm(args, wl_key, wl, dict(hc, cores_used=hc["cores_alt"], cores_alt=None))
        best = a if a["value"] >= b["value"] else b
        best["also_tried"] = {"cores": (b if best is a else a)["cores_used"], "value": (b if best is a else a)["value"]}
        return best
    cores = hc["cores_used"]
    if wl_key == "zillow":
        r = cpu_zillow_reference(args.cpu_sample_rows, cores)
    elif wl_key == "zillow_csv":
        r = cpu_zillow_csv_reference(args.cpu_sample_rows, cores)
    elif wl_key == "q6_csv":
        r = cpu_q6_csv_port(args.cpu_sample_rows, cores)
    else:
        r = None
    if r is None:
        r = cpu_port(wl, args.cpu_sample_rows, cores)
    r.update(cores_visible=hc["cores_visible"], cores_affinity=hc["cores_affinity"], cores_quota=hc["cores_quota"], cores_used=cores)
    return r


WL_NAMES = {"zillow": "zillow_z1", "q6": "tpch_q6", "c1": "c1_map_filter", "aggbykey": "aggbykey_str", "zillow_csv": "zillow_z1_from_csv",
            "q6_csv": "tpch_q6_from_csv"}
DEFAULT_ROWS = {"zillow": 100_000_000, "q6": 600_000_000, "c1": 100_000_000, "aggbykey": 100_000_000}


def static_config(args, wl_key):
    """The workload description both arms print (`config`): nothing measured in here, so the driver can compare the two lines."""
    rows = args.rows or DEFAULT_ROWS.get(wl_key, 0)
    desc = {"zillow": "Zillow Z1 map/withColumn/filter pipeline (benchmarks/zillow/Z1), synthetic rows = cyclic replication of the 32,661-row "
                      "zillow_noexc fixture (the reference's own generator), 8 column-blocked inputs, blocks of <= 16,330,500 rows",
            "q6": "TPC-H Q6 filter+aggregate (benchmarks/tpch/Q06, pre-processed columns), synthetic lineitem rows (SF100 ~ 600M), "
                  "4 columns i64,f64,f64,i64, blocks of 100M rows",
            "c1": "parallelize([1..n]).map(x*x).filter(x%2==0)", "aggbykey": "aggregateByKey string key"}[wl_key]
    return {"workload": WL_NAMES[wl_key], "rows_per_gpu": rows, "description": desc,
            "l2": "inputs larger than L2 (every block >> 126 MB, distinct HBM buffers per block)"}


def reference_line(args):
    """`--impl reference`: the reference's own CPU implementation of the path (oracle/_ref/zillow_ref = the reference's zillow.cpp
    compiled unmodified; the C port of oracle/workloads.c for Q6/C1) on the host cores this process may use. Every step is a
    bounded sample of the workload named in `config`."""
    import types
    hc = host_cores()
    keys = ["zillow", "q6"] if args.workload == "both" else [args.workload]
    out = {}
    for wl_key in keys:
        wl_args = types.SimpleNamespace(**vars(args))
        wl_args.workload = wl_key
        wl_args.rows = min(args.rows or 10**9, 2_000_000) if wl_key != "q6" else min(args.rows or 10**9, 100_000_000)
        wl = None
        if wl_key not in ("zillow", "zillow_csv", "q6_csv"):
            os.environ.setdefault("CUDA_VISIBLE_DEVICES", "")
            wl = build_workload_nopin(wl_args)
        vals, last = [], None
        # the secondary workload of the default pair gets fewer repeats so that the whole arm stays within a few minutes
        steps, warm = (args.steps, args.warmup) if wl_key == keys[0] else (max(3, args.steps // 4), 1)
        for i in range(warm + steps):
            last = cpu_arm(args, wl_key, wl, hc)
            if i >= warm:
                vals.append(last["value"])
        v = float(np.mean(vals))
        out[wl_key] = (v, last, steps, warm)
    k0 = keys[0]
    v, last, _, _ = out[k0]
    cfg = static_config(args, k0)
    if args.workload == "both":
        cfg["q6"] = static_config(args, "q6")
    line = {"metric": "rows/sec on Zillow pipeline + TPC-H Q6" if args.workload in ("both", "zillow", "q6") else "rows/sec",
            "impl": "reference", "value": v, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": (last["rows_total"] / v * 1e3) if last.get("rows_total") else None, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8/i64/f64", "data": "synthetic", "config": cfg,
            "cpu_baseline": dict(last, value=v),
            "e2e": {"value": v, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "host": hc}
    if args.workload == "both":
        v6, last6, st6, w6 = out["q6"]
        line["q6"] = {"value": v6, "unit": "rows/s", "steps": st6, "warmup": w6, "cpu_baseline": dict(last6, value=v6),
                      "e2e": {"value": v6, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------------
def measure_join(args, rank, world, local, dist):
    """K8 (csrc/join.cuh): a flights-like broadcast join, measured briefly next to the headline workloads. Probe side = 50 M rows
    (i64 key, i64 payload) resident in HBM, build side = a 1 M-row dimension table (i64 key, i64 payload, 8-byte string), inner join,
    90 % of the probe rows find exactly one partner. A step = one probe of the whole block (count, scan, emit, gather of every output
    column); the table is built once outside the timed region (its time is reported). value = probe rows / s over all ranks."""
    import time
    import torch
    from tuplex_b200 import backend, ir
    from tuplex_b200.backend import Column
    n_probe, n_build = 50_000_000, 1_000_000
    rng = np.random.default_rng(42 + rank)
    bkeys = rng.permutation(n_build).astype(np.int64) * 2 + 1
    names = np.frombuffer(b"".join(b"%08d" % i for i in range(n_build)), dtype=np.uint8).copy()
    build = [Column(ir.T_I64, bkeys), Column(ir.T_I64, rng.integers(0, 1 << 40, n_build)),
             Column(ir.T_STR, names, (np.arange(n_build + 1, dtype=np.uint64) * 8).astype(np.uint32))]
    pkeys = bkeys[rng.integers(0, n_build, n_probe)]
    miss = rng.random(n_probe) < 0.1
    pkeys[miss] = pkeys[miss] + 1  # even keys never match
    probe = [Column(ir.T_I64, pkeys), Column(ir.T_I64, rng.integers(0, 1 << 40, n_probe))]
    bb = backend.Block.upload(local, build, n_build)
    pb = backend.Block.upload(local, probe, n_probe)
    jn = backend.Join(bb, [c.type for c in build], 0)
    ptypes = [c.type for c in probe]

    def sync_all():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    steps = max(3, min(args.steps, 5))
    kms, n_out, out_bytes, launches = [], 0, 0, 0
    for _ in range(3):
        jn.probe(pb, ptypes, 0).free()
    sync_all()
    t0 = time.perf_counter()
    for _ in range(steps):
        res = jn.probe(pb, ptypes, 0)
        info = res.info
        kms.append(float(info.kernel_ms))
        n_out, launches = int(info.n_out_rows), int(info.kernel_launches)
        out_bytes = n_out * 8 * 3 + int(sum(info.out_str_bytes[:4])) + (n_out + 1) * 4
        res.free()
    sync_all()
    dt = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([dt], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    # end to end: pageable host columns in, every output column out (Block.upload + probe + fetch), one step
    sync_all()
    t1 = time.perf_counter()
    pb2 = backend.Block.upload(local, probe, n_probe)
    res = jn.probe(pb2, ptypes, 0)
    cols = res.columns()
    e2e_s = time.perf_counter() - t1
    d2h = sum(c.nbytes() for c in cols)
    res.free()
    pb2.free()
    binfo = jn.info
    jn.free()
    pb.free()
    bb.free()
    if rank != 0:
        return None
    peak, peak_src = peaks()
    alg = n_probe * 16 + out_bytes  # probe columns read once + output columns written once (table traffic not counted)
    km = float(np.median(kms))
    out = {"workload": "join_broadcast", "description": "inner hash join, 50 M probe rows (i64 key, i64) x 1 M-row table (i64 key, i64, str8), 90 % hit rate; "
           "K8 build + probe (csrc/join.cuh) through tplx_gpu_join_build / tplx_gpu_join_probe", "rows_per_gpu": n_probe, "build_rows": n_build,
           "value": n_probe * world * steps / dt, "unit": "rows/s", "ms_per_step": dt / steps * 1e3, "steps": steps, "out_rows_per_gpu": n_out,
           "build_ms": binfo["build_ms"], "gpu_launches": launches * steps,
           "roofline": {"bound": "hbm", "kernel": "join_probe_count/emit + join_gather_* (K8)", "achieved": alg / (km * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": alg / (km * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_row": alg / n_probe,
                        "kernel_ms_per_launch": km},
           "e2e": {"value": n_probe / e2e_s, "unit": "rows/s", "h2d_bytes_per_step": n_probe * 16, "d2h_bytes_per_step": int(d2h), "steps": 1,
                   "inputs_prepinned": False}}
    if not args.no_cpu_baseline:
        # CPU arm: the join oracle (oracle/join_oracle.c, one thread) on a bounded sample of the same probe rows
        from oracle import pyoracle
        ns = 5_000_000
        t2 = time.perf_counter()
        op, _ = pyoracle.join_pairs(build[0], n_build, Column(ir.T_I64, pkeys[:ns]), ns, False)
        cs = time.perf_counter() - t2
        out["cpu_baseline"] = {"value": ns / cs, "unit": "rows/s", "cores": 1, "kind": "port",
                               "sample": f"{ns} probe rows against the same {n_build}-row table, index pairs only (oracle/join_oracle.c)", "out_rows": int(len(op))}
    return out


def measure(args, wl_key, rank, world, local, dist, hc, dump=None):
    """Device-resident `value`, `roofline`, end-to-end `e2e` (page-locked and pageable host inputs) and the CPU arm of one workload;
    with `dump` (an OutputDump), what the last timed step returned is written. Returns the fields of its JSON object (rank 0) or None."""
    import torch
    from tuplex_b200 import backend, ir
    wargs = argparse.Namespace(**vars(args))
    wargs.workload = wl_key
    wl = build_workload(wargs)
    prog = wl["prog"]
    st = backend.Stage(prog)
    ep = prog.endpoint
    if ep == ir.C["TPLX_EP_HASH"]:
        st.hash_reserve(local, wl.get("nkeys", 1 << 20))

    # device-resident copies of every block (distinct HBM: the working set is far larger than the 126 MB L2)
    dev_blocks = [backend.Block.upload(local, cols, n) for cols, n in wl["blocks"]]
    torch.cuda.synchronize()

    def sync_all():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    stats = {}
    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(max_workers=3)

    def combine_partials(partials):
        tot = 0.0
        for p in partials:
            tot = tot + p
        if dist is not None:  # the one collective of the path, inside the C ABI: ncclAllGather + fold in rank order
            stats["local_partial"] = tot
            tot = ir.bits_f64(st.agg_finish(local, [ir.f64_bits(tot)])[0])
        return tot

    kept = []  # with keep=True: the results a caller of the step receives, freed once they are dumped

    def step_resident(keep=False):
        kms = 0.0
        launches = 0
        n_out = 0
        partials = []
        keep_rows = keep and ep == ir.C["TPLX_EP_MEMORY"]
        if ep == ir.C["TPLX_EP_HASH"]:
            st.hash_reset(local)
            st.hash_reserve(local, wl.get("nkeys", 1 << 20))

        def one_resident(b):
            r = st.run(b, 0)   # every block is its own task (row numbers per task), so blocks need not run in sequence
            inf = r.info
            out = (inf.kernel_ms, inf.kernel_launches, int(inf.n_out_rows),
                   ir.bits_f64(r.aggregate_bits()[0]) if ep == ir.C["TPLX_EP_AGGREGATE"] else None, int(inf.specialised_launches))
            if keep_rows:
                return out, r
            r.free()
            return out, None
        # row stages: blocks in flight on the GPU's execution lanes (the latency-bound dense launch of one block overlaps the
        # prefilter of the next). Aggregate scans are DRAM-bound (nothing to overlap) and hash stages share one table per
        # device: those run one block at a time.
        runner = pool.map if ep == ir.C["TPLX_EP_MEMORY"] else map
        spec = 0
        for (km, kl, no, part, sl), r in runner(one_resident, dev_blocks):
            kms += km
            launches += kl
            spec += sl
            n_out += no
            if part is not None:
                partials.append(part)
            if r is not None:
                kept.append(r)
        if ep == ir.C["TPLX_EP_AGGREGATE"]:
            stats["result"] = combine_partials(partials)
        if ep == ir.C["TPLX_EP_HASH"]:
            if dist is not None:  # hash-partitioned all-to-all between the GPUs' tables (tplx_gpu_stage_hash_exchange)
                st.hash_exchange(local)
            fin = st.hash_finish(local)
            n_out = int(fin.info.n_out_rows)
            kms += fin.info.kernel_ms
            launches += fin.info.kernel_launches
            if keep:
                kept.append(fin)
            else:
                fin.free()
        stats.update(kernel_ms=kms, launches=launches, n_out=n_out, specialised=spec)

    def step_e2e(blocks):
        d2h = 0
        h2d = 0
        zc = 0
        if ep == ir.C["TPLX_EP_HASH"]:
            st.hash_reset(local)
            st.hash_reserve(local, wl.get("nkeys", 1 << 20))
        # three blocks in flight: the H2D copy of the next blocks (copy stream) overlaps the kernels and the result
        # fetch (D2H stream) of earlier ones.
        # Every block is its own task (row numbers start at 0 per task, like one TransformTask per partition group).
        partials = []

        def one(block):
            cols, n = block
            r = st.run_host(local, cols, n, 0)
            inf = r.info
            nb = 0
            part = None
            if ep == ir.C["TPLX_EP_MEMORY"]:
                for c in r.columns():
                    nb += c.nbytes()
                nb += r.exceptions().nbytes
            elif ep == ir.C["TPLX_EP_AGGREGATE"]:
                part = ir.bits_f64(r.aggregate_bits()[0])
                nb += 8 * len(prog.accs)
            out = (int(inf.h2d_bytes), int(inf.zero_copy_cols), nb, part)
            r.free()
            return out
        for hb, z, nb, part in pool.map(one, blocks):
            h2d += hb
            zc = max(zc, z)
            d2h += nb
            if part is not None:
                partials.append(part)
        if ep == ir.C["TPLX_EP_AGGREGATE"]:
            stats["result_e2e"] = combine_partials(partials)
        if ep == ir.C["TPLX_EP_HASH"]:
            if dist is not None:
                st.hash_exchange(local)
            fin = st.hash_finish(local)
            for c in fin.columns():
                d2h += c.nbytes()
            fin.free()
        stats["d2h"] = d2h
        stats["h2d"] = h2d
        stats["zero_copy_cols"] = zc

    def timed(fn, k):
        """K steps bracketed by barrier + synchronize on both sides; wall time of this rank."""
        sync_all()
        t0 = time.perf_counter()
        for _ in range(k):
            fn()
        sync_all()
        return time.perf_counter() - t0

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    # the sampler starts before the warm-up, so that starting nvidia-smi does not compete with the timed steps for the host
    clocks = Clocks(local)
    clocks.start()
    W = max(args.warmup, 3)
    for i in range(W):
        # with --dump-outputs the last warm-up step holds its results like the dumped step will, so that the device memory pool
        # already holds that much when the timed steps run
        step_resident(keep=dump is not None and i == W - 1)
    # K steps between barrier + synchronize; with --min-region-s the region is repeated until that much time has been measured
    # and the median repeat is reported (max over ranks)
    reps = []
    kms = 0.0
    launches = 0
    spent = 0.0
    while True:
        kacc = lacc = done = 0
        for r in kept:  # held by the last warm-up step or a previous repeat's last step
            r.free()
        kept.clear()

        def one_step():
            nonlocal kacc, lacc, done
            done += 1
            step_resident(keep=dump is not None and done == args.steps)
            kacc += stats["kernel_ms"]
            lacc += stats["launches"]
        dt_r = max_over_ranks(timed(one_step, args.steps))
        reps.append((dt_r, kacc, lacc))
        spent += dt_r
        if spent >= args.min_region_s or len(reps) >= 200:
            break
    reps.sort()
    dt, kms, launches = reps[len(reps) // 2]
    if dump is not None:
        if ep == ir.C["TPLX_EP_AGGREGATE"]:
            dump.aggregate(wl["name"], [stats["result"]])
        else:
            dump.rows(wl["name"], prog, [r.columns() for r in kept], [r.exceptions() for r in kept] if ep == ir.C["TPLX_EP_MEMORY"] else [],
                      sort=ep == ir.C["TPLX_EP_HASH"])
        for r in kept:
            r.free()
        kept.clear()

    # end-to-end through the C ABI with host buffers (H2D of inputs + D2H of results inside the timed region), K steps
    step_e2e(wl["blocks"])
    dt_e2e = max_over_ranks(timed(lambda: step_e2e(wl["blocks"]), args.steps))
    e2e_stats = dict(stats)
    # the same with ordinary (pageable) host memory: what a caller pays who hands over plain malloc'ed partitions
    dt_pg = None
    pg_steps = max(1, min(args.steps, 3))
    if world == 1 and not args.no_pageable and wl.get("pageable_blocks") is not None:
        try:
            pb = wl["pageable_blocks"]()
            step_e2e(pb)
            dt_pg = timed(lambda: step_e2e(pb), pg_steps)
            pg_stats = dict(stats)
            del pb
        except MemoryError:
            dt_pg = None
    clk = clocks.stop()  # sampled over the warm-up and all timed regions (device-resident steps and end-to-end steps)

    line = None
    if rank == 0:
        rows_all = wl["rows"] * world
        ms_step = dt / args.steps * 1e3
        peak, peak_src = peaks()
        # algorithmic bytes: every input byte read once + output bytes written once
        out_bytes = e2e_stats.get("d2h", 0) if ep == ir.C["TPLX_EP_MEMORY"] else 0
        alg_bytes = wl["in_bytes"] + out_bytes
        n_launch = max(1, len(dev_blocks))
        k_ms_per_launch = kms / args.steps / n_launch
        # launches of different blocks overlap on the GPU's execution lanes, so the per-launch event times can add up
        # to more than the step: the device time the kernels really occupied is at most the step itself
        k_ms_step = min(kms / args.steps, ms_step)
        achieved = alg_bytes / (k_ms_step * 1e-3) / 1e9 if k_ms_step > 0 else 0.0
        kname = {"zillow_z1": "stage_mask_kernel<true> (K1f: prefilter evaluated from the string-scan hint) + mask_count/scan/expand + "
                              "stage_rows_kernel (dense launch over the survivors)",
                 "tpch_q6": "fused_scan_agg_tma_kernel", "aggbykey_str": "stage_hash_kernel",
                 "c1_map_filter": "stage_rows_vec_kernel<4> (K1v)"}.get(
            wl["name"], {0: "stage_rows_kernel", 1: "stage_agg_kernel", 2: "stage_hash_kernel"}[ep])
        if stats.get("specialised", 0):  # the stage specialiser's build of the same kernel source ran (tplx_jit_kernel)
            kname = kname.replace("stage_rows_kernel (dense", "stage_rows_kernel specialised for this stage at run time (NVRTC, tplx_jit_kernel; dense") \
                         .replace("stage_rows_vec_kernel<4> (K1v)", "tplx_jit_kernel = K1r (vecvm.cuh), the fixed-width row kernel specialised for this stage at run time "
                                                                    "(NVRTC): fates + counts in pass 1, outputs in pass 2 from L2, nothing staged")
        line = {
            "value": rows_all / (dt / args.steps), "unit": "rows/s", "ms_per_step": ms_step,
            "timed_region": {"repeats": len(reps), "seconds_measured": spent, "reported": "median repeat of K steps, max over ranks",
                             "min_ms_per_step": reps[0][0] / args.steps * 1e3, "max_ms_per_step": reps[-1][0] / args.steps * 1e3},
            "checks": {"out_rows_per_gpu": stats.get("n_out"), "blocks": len(dev_blocks)},
            "clocks": clk,
            "e2e": {"value": rows_all / (dt_e2e / args.steps), "unit": "rows/s", "h2d_bytes_per_step": e2e_stats.get("h2d", wl["in_bytes"]),
                    "d2h_bytes_per_step": e2e_stats.get("d2h", 0), "steps": args.steps, "inputs_prepinned": True,
                    "host_input_bytes_per_step": wl["in_bytes"], "zero_copy_cols": e2e_stats.get("zero_copy_cols", 0),
                    "note": "inputs lie in page-locked host memory before the timed region (inputs_prepinned); h2d = explicit copies of the "
                            "columns the prefilter reads; zero_copy_cols input columns stay in host memory and are read over PCIe for "
                            "surviving rows only (late materialisation); every output column and the exception records are fetched"},
            "gpu_launches": launches,
            "specialised_launches_per_step": stats.get("specialised", 0),  # of the step's launches: kernels the stage specialiser (csrc/jit.inl) compiled for this stage at run time
            "roofline": {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic(wl, n_launch), "peak_source": peak_src, "algorithmic_bytes_per_row": alg_bytes / wl["rows"],
                         "kernel_ms_per_launch": k_ms_per_launch, "kernel_share_of_step": k_ms_step / ms_step,
                         "launches_overlap": (kms / args.steps) > ms_step},
        }
        if dt_pg is not None:
            line["e2e"]["pageable"] = {"value": wl["rows"] / (dt_pg / pg_steps), "unit": "rows/s", "steps": pg_steps,
                                       "h2d_bytes_per_step": pg_stats.get("h2d"), "zero_copy_cols": pg_stats.get("zero_copy_cols", 0),
                                       "note": "same call with ordinary pageable numpy buffers (every column is copied; the driver stages the copies)"}
        if "result" in stats:
            line["checks"]["result"] = repr(stats["result"])
            line["checks"]["collective"] = ("tplx_gpu_agg_finish: ncclAllGather of the per-GPU partial + fold in rank order on the device"
                                            if world > 1 else None)
    if dist is not None and "local_partial" in stats:
        # self-test of the collective under the launcher (every rank takes part): the device-side fold must equal, bit for bit, the
        # same fold of the ranks' partials done on the host after a torch.distributed all_gather
        import torch as _t
        mine = _t.tensor([stats["local_partial"]], dtype=_t.float64, device="cuda")
        allp = [_t.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allp, mine)
        exp = 0.0
        for t_ in allp:
            exp = exp + float(t_.item())
        got = st.agg_finish(local, [ir.f64_bits(stats["local_partial"])])[0]
        if rank == 0:
            line["checks"]["collective_parity"] = bool(ir.f64_bits(exp) == got)
        if not args.no_cpu_baseline and world == 1:  # the CPU arm is reported at N = 1 only
            line["cpu_baseline"] = cpu_arm(args, wl_key, wl, hc)
    # free this workload's device and pinned memory before the next one is built
    for b in dev_blocks:
        b.free()
    st.close()
    del dev_blocks, wl
    import gc
    gc.collect()
    torch.cuda.synchronize()
    return line


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return 0
        return reference_line(args)

    if args.workload in ("zillow_csv", "q6_csv"):
        return main_csv(args, rank, world, local)
    import torch
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from tuplex_b200 import backend
    backend.init([local])
    if dist is not None:
        from tuplex_b200 import dist as tdist
        tdist.init_comm(local)  # this rank's NCCL communicator inside libtplx_gpu.so (id broadcast over the launcher's group)
    hc = host_cores()
    keys = ["zillow", "q6"] if args.workload == "both" else [args.workload]
    dump = OutputDump(args.dump_outputs, len(keys)) if args.dump_outputs and rank == 0 else None
    parts = {k: measure(args, k, rank, world, local, dist, hc, dump) for k in keys}
    extras = {}
    if args.workload == "both" and not args.no_extras:
        # the other two configurations of BASELINE.json, measured briefly in the same run (device-resident value + roofline + e2e):
        # config 0 (fixed-width map/filter through the vector kernel K1v) and one shard of config 5 (aggregateByKey, string keys;
        # under torchrun every rank aggregates its shard and the tables are exchanged on the device)
        xa = argparse.Namespace(**vars(args))
        xa.steps, xa.min_region_s, xa.no_pageable, xa.no_cpu_baseline = max(3, min(args.steps, 5)), 0.3, True, True
        xa.rows = 0
        extras["c1"] = measure(xa, "c1", rank, world, local, dist, hc)
        xb = argparse.Namespace(**vars(xa))
        xb.rows, xb.keys = 125_000_000, 10_000_000
        extras["aggbykey"] = measure(xb, "aggbykey", rank, world, local, dist, hc)
        xj = argparse.Namespace(**vars(xa))
        xj.no_cpu_baseline = args.no_cpu_baseline
        try:
            extras["join"] = measure_join(xj, rank, world, local, dist)
        except Exception as e:  # noqa: BLE001 — an extra must never take the headline line down with it
            extras["join"] = {"workload": "join_broadcast", "error": repr(e)[:300]}
    if rank == 0:
        k0 = keys[0]
        cfg = static_config(args, k0)
        if args.workload == "both":
            cfg["q6"] = static_config(args, "q6")
        line = {"metric": "rows/sec on Zillow pipeline + TPC-H Q6" if args.workload in ("both", "zillow", "q6") else "rows/sec",
                "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8/i64/f64", "data": "synthetic", "config": cfg}
        line.update(parts[k0])
        if args.workload == "both":
            line["q6"] = parts["q6"]
            line["gpu_launches"] += parts["q6"]["gpu_launches"]
            for k, v in extras.items():
                line[k] = v
        line["host"] = hc
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main_csv(args, rank, world, local):
    """Z1 from raw CSV text: K6 (device CSV parse, csrc/csv.cuh) in front of the Z1 stage. A step parses every block of
    CSV bytes into a column block and runs the stage on it; `value` has the bytes resident in HBM, `e2e` starts from
    page-locked host bytes (H2D of the text inside the timed region) and fetches the result rows."""
    import gzip
    import torch
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from tuplex_b200 import backend, ir, workloads as W
    from concurrent.futures import ThreadPoolExecutor
    backend.init([local])
    S, F, I, X = ir.T_STR, ir.T_F64, ir.T_I64, backend.CSV_SKIP
    if args.workload == "zillow_csv":
        with gzip.open(os.path.join(ROOT, "tests", "golden", "zillow_noexc.csv.gz"), "rb") as fp:
            raw = fp.read()
        header, body = raw.split(b"\n", 1)
        n0 = body.count(b"\n")
        total = args.rows or 32_661_000
        cycles = 125
        bn = cycles * n0
        n_blocks = max(1, total // bn)
        total = n_blocks * bn
        text = np.frombuffer(header + b"\n" + body * cycles, dtype=np.uint8)
        types, has_header, delim = [S, S, S, S, F, S, S, X, S, X], True, ","
        prog = W.zillow_program()
        expect_out = 577 * cycles * n_blocks
        name = "zillow_z1_from_csv"
        desc = (f"Zillow Z1 from raw CSV text: {total} rows = {n_blocks} buffers of {cycles} cycles of the reference's 10-column "
                f"zillow_noexc.csv (header + quoted cells), parsed on the device (8 of 10 columns, projection pushdown) and fed to the Z1 stage")
        expect_agg = None
    else:
        # TPC-H Q6 in the reference benchmark's own end-to-end form (benchmarks/tpch/Q06/runtuplex.py:96-99, --preprocessed):
        # '|'-separated text of l_quantity|l_extendedprice|l_discount|l_shipdate, no header, parse + 3 filters + sum
        n0 = 2_000_000
        cols = W.gen_lineitem(n0, seed=42)
        q, p_, d_, s_ = (c.data for c in cols)
        lines = [b"%d|%.2f|%.2f|%d" % (int(a), float(b), float(c), int(e)) for a, b, c, e in zip(q, p_, d_, s_)]
        body = b"\n".join(lines) + b"\n"
        total = args.rows or 600_000_000
        cycles = max(1, (1 << 30) // len(body))  # ~1 GiB per buffer
        bn = cycles * n0
        n_blocks = max(1, total // bn)
        total = n_blocks * bn
        text = np.frombuffer(body * cycles, dtype=np.uint8)
        types, has_header, delim = [I, F, F, I], False, "|"
        prog = W.q6_program()
        expect_out = None
        name = "tpch_q6_from_csv"
        desc = (f"TPC-H Q6 from '|'-separated text (the reference benchmark's --preprocessed end-to-end form): {total} rows = {n_blocks} "
                f"buffers of {cycles} cycles of 2,000,000 generated lineitem rows (4 columns, 2-decimal prices and discounts), parsed on the "
                f"device (fast_atoi64 / fast_atod) and reduced by the fused scan-aggregate; published reference, end-to-end from the full "
                f"16-column .tbl at SF10 on 16 threads of an r5d.8xlarge: 37 M rows/s (BASELINE.md)")
        # expected aggregate: the stage over the generator's own binary columns, summed per cycle like the blocks below
        from oracle import pyoracle
        expect_agg = pyoracle.q6(q, p_, d_, s_)
    host, keep = pinned(text)
    st = backend.Stage(prog)
    is_agg = prog.endpoint == ir.C["TPLX_EP_AGGREGATE"]
    # late materialisation: string columns the prefilter does not read stay as cell references in the CSV buffer
    from tuplex_b200.dataset import csv_lazy_columns
    lazy = csv_lazy_columns(prog, [c for c, t in enumerate(types) if t != X], types)
    bufs = [backend.CsvBuffer(local, host) for _ in range(n_blocks)]  # distinct HBM buffers, each >> L2
    torch.cuda.synchronize()
    pool = ThreadPoolExecutor(max_workers=3)
    stats = {}

    def sync_all():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    kept = []  # with keep=True: (parse, result) of every buffer, freed once they are dumped

    def run_block(buf, fetch, keep=False):
        p = buf.parse(types, delimiter=delim, header=has_header, lazy=lazy)
        r = st.run(p.block, 0)
        inf, pinf = r.info, p.info
        nb = 0
        if is_agg:
            stats["agg"] = ir.bits_f64(r.aggregate_bits()[0])
            nb = 8
        elif fetch:
            for c in r.columns():
                nb += c.nbytes()
        out = (float(pinf.parse_ms), float(inf.kernel_ms), int(pinf.kernel_launches) + int(inf.kernel_launches), int(inf.n_out_rows),
               int(pinf.n_rows), int(pinf.n_bad), sum(int(x) for x in p.block_bytes()), nb)
        if keep:
            kept.append((p, r))
        else:
            r.free()
            p.free()
        return out

    def step_resident(keep=False):
        acc = [0.0, 0.0, 0, 0, 0, 0, 0, 0]
        for o in map(lambda b: run_block(b, False, keep), bufs):
            for i, v in enumerate(o):
                acc[i] += v
        stats.update(parse_ms=acc[0], stage_ms=acc[1], launches=acc[2], n_out=acc[3], rows=acc[4], bad=acc[5], col_bytes=acc[6])

    def step_e2e():
        def one(_):
            b = backend.CsvBuffer(local, host)
            o = run_block(b, True)
            b.free()
            return o
        d2h = 0
        for o in pool.map(one, range(n_blocks)):
            d2h += o[7]
        stats["d2h"] = d2h

    dumping = args.dump_outputs is not None and rank == 0
    n_warm = max(args.warmup, 3)
    for i in range(n_warm):
        step_resident(keep=dumping and i == n_warm - 1)  # the device memory pool grows to what the dumped step holds
    assert stats["rows"] == total and stats["bad"] == 0 and (expect_out is None or stats["n_out"] == expect_out), stats
    if expect_agg is not None:  # one buffer = `cycles` copies of the generated rows
        assert abs(stats["agg"] - cycles * expect_agg) <= 1e-9 * abs(cycles * expect_agg), (stats["agg"], cycles * expect_agg)
    for p, r in kept:
        r.free()
        p.free()
    kept.clear()
    clocks = Clocks(local)
    sync_all()
    clocks.start()
    t0 = time.perf_counter()
    pms = sms = 0.0
    launches = 0
    for i in range(args.steps):
        step_resident(keep=dumping and i == args.steps - 1)
        pms += stats["parse_ms"]
        sms += stats["stage_ms"]
        launches += stats["launches"]
    sync_all()
    dt = time.perf_counter() - t0
    if kept:
        dump = OutputDump(args.dump_outputs, 1)
        if is_agg:
            dump.aggregate(name, [ir.bits_f64(r.aggregate_bits()[0]) for _, r in kept])
        else:
            dump.rows(name, prog, [r.columns() for _, r in kept], [r.exceptions() for _, r in kept])
        for p, r in kept:
            r.free()
            p.free()
        kept.clear()
    e2e_steps = max(1, min(args.steps, 3))
    step_e2e()
    sync_all()
    t1 = time.perf_counter()
    for _ in range(e2e_steps):
        step_e2e()
    sync_all()
    dt_e2e = time.perf_counter() - t1
    clk = clocks.stop()
    times = torch.tensor([dt, dt_e2e], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dt, dt_e2e = float(times[0]), float(times[1])
    if rank == 0:
        rows_all = total * world
        ms_step = dt / args.steps * 1e3
        peak, peak_src = peaks()
        csv_bytes = int(text.size) * n_blocks
        # algorithmic bytes of the dominant (parse) kernels: every CSV byte read once + the column block written once
        alg = csv_bytes + stats["col_bytes"]
        parse_ms_step = pms / args.steps
        achieved = alg / (parse_ms_step * 1e-3) / 1e9
        line = {"metric": "rows/sec on Zillow pipeline + TPC-H Q6", "value": rows_all / (dt / args.steps), "unit": "rows/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8/i64/f64", "data": "synthetic",
                "config": {"workload": name, "rows_per_gpu": total, "blocks": n_blocks, "csv_bytes_per_gpu": csv_bytes,
                           "description": desc,
                           "l2": "inputs larger than L2 (every buffer >> 126 MB, distinct HBM buffers)", "out_rows_per_gpu": stats["n_out"]},
                "clocks": clk,
                "e2e": {"value": rows_all / (dt_e2e / e2e_steps), "unit": "rows/s", "h2d_bytes_per_step": csv_bytes,
                        "d2h_bytes_per_step": stats.get("d2h", 0), "steps": e2e_steps,
                        "note": "host CSV bytes (page-locked) -> tplx_gpu_csv_upload -> tplx_gpu_csv_parse -> tplx_gpu_stage_run -> result columns fetched"},
                "gpu_launches": launches,
                "roofline": {"bound": "hbm", "kernel": "csv_tile_states + csv_row_ends + csv_parse_rows + scans + csv_compact + csv_copy_strings (K6)",
                             "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             # dram__bytes_read + dram__bytes_write of the six K6 kernels per parse, ncu --set full (profiles/r01_csv_k6.md:
                             # 5.47 GB for 804.1 MB of text), scaled to this buffer size
                             "traffic": (5.47e9 / 804.1e6 * int(text.size)) if args.workload == "zillow_csv" else None, "peak_source": peak_src,
                             "algorithmic_bytes_per_row": alg / total, "kernel_ms_per_launch": parse_ms_step / n_blocks,
                             "kernel_share_of_step": parse_ms_step / ms_step, "stage_ms_per_step": sms / args.steps,
                             "csv_gb_per_s": csv_bytes / (parse_ms_step * 1e-3) / 1e9}}
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_arm(args, args.workload, None, host_cores())
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def build_workload_nopin(args):
    """CPU arm: same generators, no pinned memory / no CUDA."""
    from tuplex_b200 import workloads as W
    from tuplex_b200.backend import Column
    if args.workload == "q6":
        n = args.rows
        return dict(name="tpch_q6", prog=W.q6_program(), blocks=[(W.gen_lineitem(n, 42), n)], rows=n)
    if args.workload == "c1":
        n = args.rows
        return dict(name="c1_map_filter", prog=W.c1_program(), blocks=[([Column(0, np.arange(1, n + 1, dtype=np.int64))], n)], rows=n)
    n = args.rows
    return dict(name="aggbykey_str", prog=W.keyed_program(), blocks=[(W.gen_keyed(n, max(1000, n // 100), 42), n)], rows=n)


if __name__ == "__main__":
    sys.exit(main())
