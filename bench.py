#!/usr/bin/env python
"""bench.py — joined rows/sec of the B200 hash join on BASELINE.json's headline config.

  python bench.py --gpus N --steps K --warmup W          (N>1: launched under torchrun, one rank per GPU)
  python bench.py --impl reference ...                   (the CPU restatement of the reference design)
  python bench.py --workload {join,agg,expr}             (secondary configs C4 / C2; default join = C3)

A "step" = one full pass of the hot path over the synthetic tables of the workload (for the join:
build 1e7 rows + probe 1e8 rows -> 1e8 joined rows materialised in HBM), inputs resident in HBM.
`e2e` = the same job through the C-ABI with pinned HOST buffers, PCIe copies inside the timed region.
Prints ONE JSON line on rank 0.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True   # the benchmark leaves the tree as it found it (it may be read-only)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

HBM_FALLBACK_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback


def join_config(n_build, n_probe):
    return {"workload": f"C3: int64 equi-join, uniform keys, build={n_build} probe={n_probe}, 100% match, output (B.k,B.v,P.k,P.v) materialised",
            "build_rows": n_build, "probe_rows": n_probe, "l2": "inputs (1.76 GB) and output (3.2 GB) exceed the 126 MB L2; no flush needed",
            "step": "tq_join create + build + probe + result, inputs resident in HBM",
            "e2e_step": "same through the C-ABI with HOST buffers: pinned inputs (tq_pinned_alloc, declared TQ_JOIN_STABLE_INPUT so uploads overlap "
                        "result downloads), 8M-row probe pieces, every result column copied back to pinned host memory; all copies inside the timed region"}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------ --dump-outputs
DUMP_SAMPLE_ROWS = 1 << 19   # rows kept of each large result: 4 MB per float64 array, the whole dump stays far below the limit
DUMP_LIMIT_BYTES = 64 << 20


def sample_rows(n):
    """sorted positions of a fixed, seeded sample of n rows (all of them when n is small): the same rows in every run"""
    if n <= DUMP_SAMPLE_ROWS:
        return np.arange(n)
    return np.sort(np.random.default_rng(12345).choice(n, DUMP_SAMPLE_ROWS, replace=False))


def write_dump(dump_dir, arrays):
    """one DIR/<name>.npy per array; float32 / float64 only, DUMP_LIMIT_BYTES in all"""
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(dump_dir, exist_ok=True)
    for name, a in arrays.items():
        if a.dtype not in (np.float32, np.float64):
            raise TypeError(f"--dump-outputs: {name} is {a.dtype}, not float32 / float64")
        np.save(os.path.join(dump_dir, name + ".npy"), a)


def int64_halves(name, v):
    """an int64 column float64 cannot hold exactly, as its high (signed) and low 32-bit halves: both exact in float64"""
    return {name + "_hi32": (v >> 32).astype(np.float64), name + "_lo32": (v & 0xFFFFFFFF).astype(np.float64)}


# ------------------------------------------------------------------ synthetic tables (SURVEY §8d)
def gen_join_tables(n_build, n_probe, key_range, seed_b=3, seed_p=4, rank=0):
    """C3: B.k = permutation of [0, n_build) (seed 3), B.v = 7k+1; P.k uniform [0, key_range) (seed 4), P.v = row id."""
    rb = np.random.default_rng(seed_b + 1000 * rank)
    rp = np.random.default_rng(seed_p + 1000 * rank)
    if key_range == n_build:
        bk = rb.permutation(n_build).astype(np.int64)
    else:  # a shard of a bigger table: distinct keys of this rank's residue class
        bk = rb.permutation(n_build).astype(np.int64)
    bv = bk * 7 + 1
    pk = rp.integers(0, key_range, n_probe, dtype=np.int64)
    pv = np.arange(n_probe, dtype=np.int64)
    return bk, bv, pk, pv


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.proc, self.lines = device, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.device)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------ CPU arm (oracle/cpu_ref.c)
def cpu_join_sample(n_build, n_probe_full, sample_probe, workers, seed_rank=0, tables=None):
    import oracle_py as O
    lib = O.load()
    bk, bv, pk, pv = tables if tables is not None else gen_join_tables(n_build, sample_probe, n_build, rank=seed_rank)
    bs, ps, ck = C.c_double(0), C.c_double(0), C.c_uint64(0)
    rows = lib.orc_mt_join_bench(C.c_int64(n_build), C.c_void_p(bk.ctypes.data), C.c_void_p(bv.ctypes.data), C.c_int64(sample_probe),
                                 C.c_void_p(pk.ctypes.data), C.c_void_p(pv.ctypes.data), C.c_int(workers), C.byref(bs), C.byref(ps), C.byref(ck))
    assert rows == sample_probe, (rows, sample_probe)
    # whole-job estimate: the build is paid once, the probe scales with the probe rows
    est_total_s = bs.value + ps.value * (n_probe_full / sample_probe)
    return {"value": n_probe_full / est_total_s, "unit": "joined rows/s", "cores": workers, "kind": "port",
            "sample": f"full serial build of {n_build} rows ({bs.value:.2f} s) + probe of the first {sample_probe} of {n_probe_full} probe rows "
                      f"({ps.value:.2f} s, {workers} worker threads), extrapolated to the whole probe side; "
                      "oracle/cpu_ref.c = C restatement of the reference's goroutine design (no Go toolchain in this image)",
            "build_s": bs.value, "probe_s": ps.value}


def verify_join_result(rows, cols, pk, n_probe_expected, id_base=0):
    """Size-independent properties of the C3 join, checked on EVERY row: B.v = 7*B.k + 1, B.k = P.k, P.k is the key the
    probe row P.v really carried, and every probe row id appears exactly once (100 % match, unique build keys)."""
    bk, bv, pkk, pv = cols
    checks = {"row_count": rows == n_probe_expected,
              "B.v == 7*B.k + 1": bool(np.array_equal(bv, bk * 7 + 1)),
              "B.k == P.k": bool(np.array_equal(bk, pkk))}
    ids = pv - id_base
    in_range = bool(((ids >= 0) & (ids < len(pk))).all()) if rows else True
    checks["P.v in range"] = in_range
    if in_range and rows:
        checks["P.k == probe_keys[P.v]"] = bool(np.array_equal(pkk, pk[ids]))
        checks["every probe row exactly once"] = bool((np.bincount(ids, minlength=len(pk)) == 1).all()) if rows == len(pk) else False
    return {"ok": all(checks.values()), "rows": int(rows), "checks": checks}


# ------------------------------------------------------------------ GPU arm
class JoinBench:
    def __init__(self, lib, L, n_build, n_probe, rank=0, world=1):
        from tinysql_b200.chunk import INT64, Column, DeviceColumn
        self.lib, self.L = lib, L
        self.n_build, self.n_probe = n_build, n_probe
        self.bk, self.bv, self.pk, self.pv = gen_join_tables(n_build, n_probe, n_build, rank=rank)
        self.d_b = [DeviceColumn.from_host(Column(INT64, self.bk)), DeviceColumn.from_host(Column(INT64, self.bv))]
        self.d_p = [DeviceColumn.from_host(Column(INT64, self.pk)), DeviceColumn.from_host(Column(INT64, self.pv))]
        self.INT64 = INT64

    def desc(self, batch=0, flags=0):
        L = self.L
        t = (C.c_int32 * 2)(1, 1)
        k = (C.c_int32 * 1)(0)
        self._keep = (t, k)
        return L.TQJoinDesc(0, 1, 2, t, 2, t, 1, k, k, batch, flags)

    def step_device(self, keep=False, hold=False):
        """build + probe with inputs resident in HBM; returns (joined rows, probe kernel ns, build ns).  keep=True copies the
        four result columns to the host (verification leg, outside every timed region).  hold=True leaves the handle and the
        result it lends alive until take_held() (the last timed step of a --dump-outputs run)."""
        L, lib = self.L, self.lib
        h = C.c_void_p()
        d = self.desc()
        L.check(lib.tq_join_create(C.byref(d), C.byref(h)))
        barr = (L.TQColumn * 2)(self.d_b[0].tq(), self.d_b[1].tq())
        for i in range(2):
            barr[i].null_bitmap = None
        parr = (L.TQColumn * 2)(self.d_p[0].tq(), self.d_p[1].tq())
        for i in range(2):
            parr[i].null_bitmap = None
        L.check(lib.tq_join_put_build(h, barr, L.TQ_MEM_DEVICE))
        L.check(lib.tq_join_finalize_build(h))
        L.check(lib.tq_join_put_probe(h, parr, None, L.TQ_MEM_DEVICE))
        L.check(lib.tq_join_probe_eof(h))
        out = (L.TQColumn * 4)()
        n, eof = C.c_int64(0), C.c_int32(0)
        L.check(lib.tq_join_next_device(h, out, C.byref(n), C.byref(eof)))
        st = (C.c_int64 * 8)()
        lib.tq_join_stats(h, st)
        rows = n.value
        self.last_out = self._copy_out(out, rows) if keep else None
        if hold:
            self.held = (h, out, rows)
        else:
            L.check(lib.tq_join_destroy(h))
        return rows, st[5], st[6]

    def _copy_out(self, out, rows):
        cols = []
        for c in range(4):
            a = np.empty(rows, dtype=np.int64)
            self.L.check(self.lib.tq_memcpy_d2h(a.ctypes.data, out[c].data, rows * 8))
            cols.append(a)
        return cols

    def take_held(self):
        """the result of the held step as --dump-outputs arrays: the rows of a seeded sample of probe rows, in probe-row
        order (the hash join's output order is not part of its result), plus the row count; then the handle is destroyed"""
        h, out, rows = self.held
        self.held = None
        bk, bv, pkk, pv = self._copy_out(out, rows)
        self.L.check(self.lib.tq_join_destroy(h))
        mark = np.zeros(self.n_probe, dtype=bool)
        mark[sample_rows(self.n_probe)] = True
        pos = np.flatnonzero(mark[pv])
        pos = pos[np.argsort(pv[pos], kind="stable")]
        # every value of C3 is below 2^53 (keys < n_build, B.v = 7k+1, row ids < n_probe): float64 holds it exactly
        return {"join_rows": np.array([rows], dtype=np.float64), "join_build_key": bk[pos].astype(np.float64),
                "join_build_value": bv[pos].astype(np.float64), "join_probe_key": pkk[pos].astype(np.float64),
                "join_probe_value": pv[pos].astype(np.float64)}

    def verify(self):
        """Full-size value check of the device-resident join (outside the timed region): output = (B.k, B.v, P.k, P.v)."""
        return verify_join_result(*self.step_and_keep(), self.pk, self.n_probe)

    def step_and_keep(self):
        rows, _, _ = self.step_device(keep=True)
        return rows, self.last_out

    def setup_e2e(self):
        """pinned host inputs / outputs for the C-ABI host path"""
        lib, L = self.lib, self.L

        def pinned(n_items, src=None):
            p = C.c_void_p()
            L.check(lib.tq_pinned_alloc(n_items * 8, C.byref(p)))
            arr = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_int64)), shape=(n_items,))
            if src is not None:
                arr[:] = src
            return p, arr

        self.h_b = [pinned(self.n_build, self.bk), pinned(self.n_build, self.bv)]
        self.h_p = [pinned(self.n_probe, self.pk), pinned(self.n_probe, self.pv)]
        self.out_rows = 1 << 23
        self.h_out = [pinned(self.out_rows) for _ in range(4)]
        self.h_out_bm = [np.zeros((self.out_rows + 7) // 8 + 8, dtype=np.uint8) for _ in range(4)]

    def step_e2e(self):
        """Open/build/probe/Next-until-EOF/Close through the C-ABI with HOST buffers."""
        L, lib = self.L, self.lib
        h = C.c_void_p()
        # the host buffers are C-owned pinned memory (tq_pinned_alloc) that nobody rewrites during the step: declare them
        # stable so the upload of piece i+1 overlaps the download of result i (both still inside the timed region)
        d = self.desc(batch=1 << 23, flags=L.TQ_JOIN_STABLE_INPUT)
        L.check(lib.tq_join_create(C.byref(d), C.byref(h)))

        def cols(bufs, n):
            a = (L.TQColumn * len(bufs))()
            for i, (p, _) in enumerate(bufs):
                a[i].length, a[i].data, a[i].null_bitmap, a[i].offsets = n, p.value, None, None
            return a
        L.check(lib.tq_join_put_build(h, cols(self.h_b, self.n_build), L.TQ_MEM_HOST))
        L.check(lib.tq_join_finalize_build(h))
        out = (L.TQColumn * 4)()
        for i in range(4):
            out[i].data = self.h_out[i][0].value
            out[i].null_bitmap = self.h_out_bm[i].ctypes.data
        n, eof = C.c_int64(0), C.c_int32(0)
        total = 0
        checksum = 0
        # feed the probe side in 8M-row host pieces and drain whatever is ready after each one (the Next contract:
        # 0 rows with eof == 0 means "feed more"); result copies of piece i overlap the upload + kernels of piece i+1
        piece = 1 << 23

        def drain():
            nonlocal total, checksum
            while True:
                L.check(lib.tq_join_next(h, self.out_rows, out, C.byref(n), C.byref(eof)))
                if n.value == 0:
                    return bool(eof.value)
                total += n.value
                self.last_e2e_rows = n.value
                checksum += int(self.h_out[1][1][0])  # touch the result on the host
        for lo in range(0, self.n_probe, piece):
            rows = min(piece, self.n_probe - lo)
            a = (L.TQColumn * 2)()
            for i, (p, _) in enumerate(self.h_p):
                a[i].length, a[i].data, a[i].null_bitmap, a[i].offsets = rows, p.value + lo * 8, None, None
            L.check(lib.tq_join_put_probe(h, a, None, L.TQ_MEM_HOST))
            drain()
        L.check(lib.tq_join_probe_eof(h))
        while not drain():
            pass
        L.check(lib.tq_join_destroy(h))
        return total


    def free(self):
        """give the join tables back before the secondary workloads allocate theirs"""
        for c in self.d_b + self.d_p:
            c.free()
        for bufs in (getattr(self, "h_b", []), getattr(self, "h_p", []), getattr(self, "h_out", [])):
            for p, _ in bufs:
                self.lib.tq_pinned_free(p)
        self.h_b = self.h_p = self.h_out = []

    def verify_e2e_tail(self):
        """the host buffers still hold the LAST result piece of the last e2e step: its rows must satisfy the row-wise properties"""
        n = self.last_e2e_rows
        bk, bv, pkk, pv = (self.h_out[c][1][:n] for c in range(4))
        ok = bool(n > 0 and np.array_equal(bv, bk * 7 + 1) and np.array_equal(bk, pkk) and np.array_equal(pkk, self.pk[pv]))
        return {"rows": int(n), "ok": ok}

    def step_e2e_chunked(self):
        """The reference's own calling pattern (executor/join.go:194-221, the shim in INTEGRATION.md): ONE <=1024-row chunk per
        tq_join_put_build / tq_join_put_probe call from ordinary (pageable) host memory, no TQ_JOIN_STABLE_INPUT, results drained
        through tq_join_next with 1024-row chunks.  ~2e5 C-ABI calls per step; the caller here is a Python loop, so the
        figure includes ~1 us of ctypes overhead per call (a cgo call costs about the same)."""
        L, lib = self.L, self.lib
        h = C.c_void_p()
        d = self.desc()
        L.check(lib.tq_join_create(C.byref(d), C.byref(h)))
        CH = 1024
        t0 = time.perf_counter()
        a = (L.TQColumn * 2)()
        for lo in range(0, self.n_build, CH):
            rows = min(CH, self.n_build - lo)
            for i, src in enumerate((self.bk, self.bv)):
                a[i].length, a[i].data, a[i].null_bitmap, a[i].offsets = rows, src.ctypes.data + lo * 8, None, None
            L.check(lib.tq_join_put_build(h, a, L.TQ_MEM_HOST))
        L.check(lib.tq_join_finalize_build(h))
        outs = [np.empty(CH, dtype=np.int64) for _ in range(4)]
        bms = [np.zeros(CH // 8 + 8, dtype=np.uint8) for _ in range(4)]
        out = (L.TQColumn * 4)()
        for i in range(4):
            out[i].data, out[i].null_bitmap = outs[i].ctypes.data, bms[i].ctypes.data
        n, eof = C.c_int64(0), C.c_int32(0)
        total, ok = 0, True

        def drain():
            nonlocal total, ok
            while True:
                L.check(lib.tq_join_next(h, CH, out, C.byref(n), C.byref(eof)))
                if n.value == 0:
                    return bool(eof.value)
                total += n.value
                ok = ok and int(outs[1][0]) == int(outs[0][0]) * 7 + 1   # touch the chunk on the host
        for lo in range(0, self.n_probe, CH):
            rows = min(CH, self.n_probe - lo)
            for i, src in enumerate((self.pk, self.pv)):
                a[i].length, a[i].data, a[i].null_bitmap, a[i].offsets = rows, src.ctypes.data + lo * 8, None, None
            L.check(lib.tq_join_put_probe(h, a, None, L.TQ_MEM_HOST))
            drain()
        L.check(lib.tq_join_probe_eof(h))
        while not drain():
            pass
        dt = time.perf_counter() - t0
        L.check(lib.tq_join_destroy(h))
        calls = 2 * ((self.n_probe + CH - 1) // CH) + (self.n_build + CH - 1) // CH
        return {"value": total / dt, "unit": "joined rows/s", "ms_per_step": dt * 1e3, "rows": int(total), "ok": bool(ok and total == self.n_probe),
                "chunk_rows": CH, "c_abi_calls_per_step": int(calls), "h2d_bytes_per_step": 16 * (self.n_build + self.n_probe),
                "d2h_bytes_per_step": 32 * self.n_probe,
                "note": "one <=1024-row chunk per call from pageable host memory (no STABLE_INPUT), 1 step, driven from Python"}


def run_join_bench(args, rank, world, local_rank, dist):
    from tinysql_b200 import _lib as L
    lib = L.load()
    L.check(lib.tq_init(local_rank))
    n_build, n_probe = args.build_rows, args.probe_rows
    peak, peak_src = measured_peak()
    if world > 1:
        from tinysql_b200 import dist as D
        return D.bench_distributed_join(args, rank, world, local_rank, dist, peak, peak_src)
    jb = JoinBench(lib, L, n_build, n_probe, rank, world)
    for _ in range(args.warmup):
        rows, _, _ = jb.step_device()
        assert rows == n_probe, rows
    sampler = ClockSampler(local_rank)
    sampler.start()
    lib.tq_device_synchronize()
    launches1 = lib.tq_kernel_launch_count()
    probe_ns, build_ns = [], []
    ms = C.c_float(0)
    L.check(lib.tq_timer_start())
    for i in range(args.steps):
        rows, pns, bns = jb.step_device(hold=args.dump is not None and i == args.steps - 1)
        probe_ns.append(pns)
        build_ns.append(bns)
    L.check(lib.tq_timer_stop(C.byref(ms)))
    lib.tq_device_synchronize()
    clocks = sampler.stop()
    launches2 = lib.tq_kernel_launch_count()
    if args.dump is not None:
        args.dump.update(jb.take_held())
    ms_per_step = ms.value / args.steps
    value = n_probe / (ms_per_step * 1e-3)
    # roofline of the dominant kernels (the probe pipeline): 64 algorithmic bytes per probe row (SURVEY §8d / DESIGN.md)
    probe_s = statistics.mean(probe_ns) * 1e-9
    achieved = 64.0 * n_probe / probe_s / 1e9
    if args.kernel_only:
        out = {"value": value, "ms_per_step": ms_per_step, "kernel_ms": probe_s * 1e3, "build_ms": statistics.mean(build_ns) * 1e-6,
               "frac": achieved / peak, "gpu_launches": int(launches2 - launches1)}
        if args.verify:
            out["verified"] = jb.verify()
        return out
    # every value of the full-size result is checked once, outside the timed region
    verified = jb.verify()
    # end to end through the C-ABI with pinned host buffers
    jb.setup_e2e()
    e2e_steps = max(1, min(args.steps, 3))
    jb.step_e2e()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        total = jb.step_e2e()
        assert total == n_probe
    lib.tq_device_synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    verified["e2e_last_piece"] = jb.verify_e2e_tail()
    chunked = jb.step_e2e_chunked() if not args.no_chunked_e2e else None
    workers = os.cpu_count() or 1
    cpu = cpu_join_sample(n_build, n_probe, min(n_probe, args.cpu_sample_rows), workers)
    out = {
        "metric": "joined rows/sec on 1e8-row int64 equi-join", "value": value, "unit": "joined rows/s", "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
        "data": "synthetic",
        "config": join_config(n_build, n_probe),
        "roofline": {"bound": "hbm", "kernel": "probe pipeline = k_scatter_aos<2> (TMA-fed radix scatter) + k_probe_pos<2,2> (TMA-fed positional probe) + hole filling, "
                                                "timed together with CUDA events on the library stream",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": None, "traffic_note": "not measured in this run (ncu --set full captures: profiles/)",
                     "peak_source": peak_src, "algorithmic_bytes_per_row": 64, "algorithmic_bytes": 64 * n_probe, "kernel_ms": probe_s * 1e3,
                     "build_ms": statistics.mean(build_ns) * 1e-6},
        "e2e": {"value": n_probe / e2e_s, "unit": "joined rows/s", "h2d_bytes_per_step": 16 * (n_build + n_probe), "d2h_bytes_per_step": 32 * n_probe,
                "ms_per_step": e2e_s * 1e3},
        "e2e_chunked": chunked,
        "verified": verified,
        "gpu_launches": int(launches2 - launches1), "clocks": clocks, "cpu_baseline": cpu,
    }
    jb.free()
    if not args.no_secondary:
        out["secondary"] = run_secondary(args, lib, peak, peak_src)
    return out


def run_secondary(args, lib, peak, peak_src):
    """BASELINE configs C2 (vectorized LT + Plus over 1e8 rows) and C4 (1e8-row GROUP BY, 1e6 groups) in the same driver-run
    record: value, roofline, cpu_baseline, e2e and a full-size value check each; timed after the headline."""
    import bench_extra
    sec = {}
    for name, fn in (("C2", bench_extra.run_expr), ("C4", bench_extra.run_agg)):
        try:
            r = fn(args, lib, peak, peak_src, ClockSampler)
            sec[name] = {k: r[k] for k in ("metric", "value", "unit", "ms_per_step", "steps", "warmup", "config", "roofline", "e2e", "cpu_baseline", "verified", "gpu_launches", "clocks")
                         if k in r}
        except Exception as e:  # the headline line must survive a secondary failure; the failure itself is reported
            sec[name] = {"error": f"{type(e).__name__}: {e}"}
    return sec


def run_reference(args, rank):
    """--impl reference: the CPU restatement of the reference's goroutine design on the host cores (all host threads).
    Every step builds the full hash table and probes a bounded sample of the probe side: the WHOLE probe side when the
    run is short enough, else 40 % of it (stated in `sample`); the reported value is the median step."""
    if rank != 0:
        return None
    n_build, n_probe = args.build_rows, args.probe_rows
    config = join_config(n_build, n_probe)
    if args.gpus > 1:   # the same GLOBAL job our arm runs at this N (dist.py: C5 sizes per GPU x N), on the host cores
        from tinysql_b200.dist import dist_sizes, dist_workload_config
        n_b, n_p = dist_sizes(args)
        n_build, n_probe = n_b * args.gpus, n_p * args.gpus
        config = dist_workload_config(args.gpus, n_b, n_p, max(1, int(os.environ.get("TQ_DIST_CHUNKS", "2"))))
    workers = os.cpu_count() or 1
    n_steps = args.warmup + args.steps
    # bounded sample: the whole run (W + K steps, each = full serial build + probe of `sample` rows) should end within ~3 minutes
    # on the box's host cores (measured: build 62 ns/row on one core, probe 22 ns/row over 128 threads); the whole probe side
    # whenever that fits — then nothing is extrapolated
    budget_s = 170.0 / max(n_steps, 1)
    sample = int(max(args.cpu_sample_rows, min(n_probe, (budget_s - 6.2e-8 * n_build) / 2.2e-8)))
    sample = min(sample, n_probe)
    res = None
    times = []
    tables = gen_join_tables(n_build, sample, n_build)   # generated once: the steps time the join, not numpy
    for i in range(n_steps):
        r = cpu_join_sample(n_build, n_probe, sample, workers, tables=tables)
        if i >= args.warmup:
            times.append(r)
        res = r
    vals = sorted(r["value"] for r in times) if times else [res["value"]]
    v = statistics.median(vals)
    res = dict(res)
    res["value"] = v
    res["step_values_min_median_max"] = [vals[0], v, vals[-1]]
    return {"impl": "reference", "metric": "joined rows/sec on 1e8-row int64 equi-join", "value": v, "unit": "joined rows/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * n_probe / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int64", "data": "synthetic",
            "config": config,
            "cpu_baseline": res, "e2e": {"value": v, "unit": "joined rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="join", choices=["join", "agg", "expr"])
    ap.add_argument("--build-rows", type=int, default=10_000_000)
    ap.add_argument("--probe-rows", type=int, default=100_000_000)
    ap.add_argument("--cpu-sample-rows", type=int, default=20_000_000)
    ap.add_argument("--kernel-only", action="store_true", help="skip the e2e and CPU legs (profiling runs)")
    ap.add_argument("--verify", action="store_true", help="with --kernel-only: still run the full-size value check")
    ap.add_argument("--no-secondary", action="store_true", help="skip the C2 / C4 secondary block")
    ap.add_argument("--no-chunked-e2e", action="store_true", help="skip the <=1024-row chunk protocol e2e figure")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step of every workload timed as DIR/<name>.npy (float64, seeded samples "
                         "of large results, at most 64 MB); that step's handle is released after the timer stops")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl == "reference" or args.gpus > 1 or world > 1):
        ap.error("--dump-outputs dumps the single-GPU device path (--impl ours, --gpus 1)")
    args.dump = {} if args.dump_outputs else None
    if args.impl == "reference":
        out = run_reference(args, rank)
        if out is not None:
            print(json.dumps(out))
        return
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        torch.cuda.set_device(local_rank)
        dist_mod.init_process_group("nccl")
        dist = dist_mod
    if args.workload == "join":
        out = run_join_bench(args, rank, world, local_rank, dist)
    else:
        import bench_extra
        out = bench_extra.run(args, rank, world, local_rank)
    if args.dump is not None:
        write_dump(args.dump_outputs, args.dump)
    if rank == 0 and out is not None:
        print(json.dumps(out))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
