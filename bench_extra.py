"""bench.py --workload {expr,agg}: the secondary BASELINE configs on one B200 (benchmark infrastructure, like bench.py:
the cpu_baseline legs load the oracle; the product package tinysql_b200/ never does).
  expr = C2: vectorized LT + Plus (builtin_compare_vec / builtin_arithmetic_vec) over 1e8 int64 rows
  agg  = C4: 1e8-row GROUP BY int64 key with SUM(float64), COUNT(*), 1e6 groups
Same JSON contract as the join line (value = device-resident, e2e = pinned host buffers through the C-ABI)."""
import ctypes as C
import os
import statistics
import time

import numpy as np

from tinysql_b200 import _lib as L
from tinysql_b200.chunk import FLOAT64, INT64, Column, DeviceColumn, device_to_host


def _pinned(lib, n_items, dtype, src=None):
    p = C.c_void_p()
    L.check(lib.tq_pinned_alloc(n_items * 8, C.byref(p)))
    ct = C.c_int64 if dtype == np.int64 else C.c_double
    arr = np.ctypeslib.as_array(C.cast(p, C.POINTER(ct)), shape=(n_items,))
    if src is not None:
        arr[:] = src
    return p, arr


def _col(ptr, n, bm=None):
    t = L.TQColumn()
    t.length, t.data, t.null_bitmap, t.offsets = n, ptr, bm, None
    return t


def run_expr(args, lib, peak, peak_src, sampler_cls):
    n = args.probe_rows
    rng1, rng2 = np.random.default_rng(1), np.random.default_rng(2)
    a = rng1.integers(-(1 << 62), 1 << 62, n, dtype=np.int64)   # builtin_arithmetic_vec_test.go:47-52 operand range
    b = rng2.integers(-(1 << 62), 1 << 62, n, dtype=np.int64)
    da, db = DeviceColumn.from_host(Column(INT64, a)), DeviceColumn.from_host(Column(INT64, b))
    lt, plus = DeviceColumn(INT64, n), DeviceColumn(INT64, n)
    ta, tb, t1, t2 = da.tq(), db.tq(), lt.tq(), plus.tq()
    ta.null_bitmap = None
    tb.null_bitmap = None

    def fused():
        L.check(lib.tq_vec_lt_plus_int(n, C.byref(ta), C.byref(tb), C.byref(t1), C.byref(t2), L.TQ_MEM_DEVICE))

    def separate():
        L.check(lib.tq_vec_compare_int(0, n, C.byref(ta), 0, C.byref(tb), 0, C.byref(t1), L.TQ_MEM_DEVICE))
        L.check(lib.tq_vec_arith_int(0, n, C.byref(ta), 0, C.byref(tb), 0, C.byref(t2), L.TQ_MEM_DEVICE))

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        ms = C.c_float(0)
        L.check(lib.tq_timer_start())
        for _ in range(args.steps):
            fn()
        L.check(lib.tq_timer_stop(C.byref(ms)))
        return ms.value / args.steps
    sampler = sampler_cls(0)
    sampler.start()
    l1 = lib.tq_kernel_launch_count()
    ms_fused = timed(fused)
    l2 = lib.tq_kernel_launch_count()
    if args.dump is not None:   # lt / plus hold the last fused step's result until the separate-ops timing overwrites them
        from bench import int64_halves, sample_rows
        rows = sample_rows(n)
        h_lt, h_plus = lt.to_host(), plus.to_host()
        args.dump["expr_lt"] = h_lt.values[rows].astype(np.float64)
        args.dump.update(int64_halves("expr_plus", h_plus.values[rows]))
    ms_sep = timed(separate)
    clocks = sampler.stop()
    # e2e: pinned host columns through the host path (slab pipeline: H2D | kernel | D2H overlapped)
    pa, _ = _pinned(lib, n, np.int64, a)
    pb, _ = _pinned(lib, n, np.int64, b)
    po1, o1 = _pinned(lib, n, np.int64)
    po2, o2 = _pinned(lib, n, np.int64)
    bm1, bm2 = np.zeros(n // 8 + 16, np.uint8), np.zeros(n // 8 + 16, np.uint8)
    ha, hb = _col(pa.value, n), _col(pb.value, n)
    h1, h2 = _col(po1.value, n, bm1.ctypes.data), _col(po2.value, n, bm2.ctypes.data)
    L.check(lib.tq_vec_lt_plus_int(n, C.byref(ha), C.byref(hb), C.byref(h1), C.byref(h2), L.TQ_MEM_HOST))
    t0 = time.perf_counter()
    reps = max(1, min(3, args.steps))
    for _ in range(reps):
        L.check(lib.tq_vec_lt_plus_int(n, C.byref(ha), C.byref(hb), C.byref(h1), C.byref(h2), L.TQ_MEM_HOST))
    e2e_s = (time.perf_counter() - t0) / reps
    # full-size value check (outside the timed region): every row of both results, and the NOT NULL bitmaps
    nb = n // 8
    verified = {"ok": bool(np.array_equal(o2, a + b) and np.array_equal(o1, (a < b).astype(np.int64)) and (bm1[:nb] == 0xFF).all() and (bm2[:nb] == 0xFF).all()),
                "rows": int(n), "checks": ["lt == (a < b) on every row", "plus == a + b on every row", "result bitmaps all NOT NULL"]}
    # CPU arm: 1024-row chunk loops, all host threads, on a bounded sample
    import oracle_py as O
    olib = O.load()
    sample = min(n, 20_000_000)
    lo, po = np.empty(sample, np.int64), np.empty(sample, np.int64)
    sec = C.c_double(0)
    workers = os.cpu_count() or 1
    olib.orc_mt_lt_plus_bench(C.c_int64(sample), C.c_void_p(a.ctypes.data), C.c_void_p(b.ctypes.data), C.c_void_p(lo.ctypes.data), C.c_void_p(po.ctypes.data),
                              C.c_int(workers), C.byref(sec))
    bytes_fused = 32.0 + 0.25  # 2x8 read + 2x8 written + two result bitmaps (1 bit each)
    achieved = bytes_fused * n / (ms_fused * 1e-3) / 1e9
    out = {
        "metric": "rows/sec, vectorized LT + Plus over 1e8 int64 rows", "value": n / (ms_fused * 1e-3), "unit": "rows/s", "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_fused, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": f"C2: a<b and a+b over {n} int64 rows, operands uniform in [-2^62, 2^62), NOT NULL; fused k_map<2,2,FLtPlus> (one pass)",
                   "separate_ops_ms": ms_sep, "l2": "inputs 1.6 GB / outputs 1.6 GB exceed L2; no flush needed"},
        "roofline": {"bound": "hbm", "kernel": "k_map<2,2,FLtPlus>", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                     "peak_source": peak_src, "algorithmic_bytes_per_row": bytes_fused, "separate_ops_gbs": 2 * 24.125 * n / (ms_sep * 1e-3) / 1e9},
        "e2e": {"value": n / e2e_s, "unit": "rows/s", "h2d_bytes_per_step": 16 * n, "d2h_bytes_per_step": 16 * n + n // 4, "ms_per_step": e2e_s * 1e3},
        "gpu_launches": int(l2 - l1), "clocks": clocks, "verified": verified,
        "cpu_baseline": {"value": sample / sec.value, "unit": "rows/s", "cores": workers, "kind": "port",
                         "sample": f"first {sample} rows in 1024-row chunks over {workers} threads (oracle/cpu_ref.c: VecCompareII + vecResOfLT + plusSS loops)"},
    }
    for c in (da, db, lt, plus):
        c.free()
    for q in (pa, pb, po1, po2):
        lib.tq_pinned_free(q)
    return out


def run_agg(args, lib, peak, peak_src, sampler_cls):
    n, groups = args.probe_rows, 1_000_000
    k = np.random.default_rng(5).integers(0, groups, n, dtype=np.int64)
    x = np.random.default_rng(6).random(n)                      # randDatum, executor/benchmark_test.go:118-119
    dk, dx = DeviceColumn.from_host(Column(INT64, k)), DeviceColumn.from_host(Column(FLOAT64, x))
    types = (C.c_int32 * 2)(INT64 | 0x100, FLOAT64 | 0x100)  # both columns NOT NULL (TQ_TYPE_NOT_NULL)
    gb = (C.c_int32 * 1)(0)
    funcs = (L.TQAggFunc * 3)(L.TQAggFunc(1, 1), L.TQAggFunc(0, -1), L.TQAggFunc(5, 0))  # SUM(x), COUNT(*), firstrow(k)
    desc = L.TQAggDesc(2, types, 1, gb, 3, funcs, groups)

    held = []

    def step(mem, cols_fn, hold=False):
        """hold=True keeps the handle and the result it lends for the --dump-outputs copy after the timer stops"""
        h = C.c_void_p()
        L.check(lib.tq_agg_create(C.byref(desc), C.byref(h)))
        cols_fn(h)
        L.check(lib.tq_agg_eof(h))
        out = (L.TQColumn * 3)()
        nn, eof = C.c_int64(0), C.c_int32(0)
        L.check(lib.tq_agg_next_device(h, out, C.byref(nn), C.byref(eof)))
        st = (C.c_int64 * 4)()
        lib.tq_agg_stats(h, st)
        if hold:
            held.append((h, out, nn.value))
        else:
            L.check(lib.tq_agg_destroy(h))
        return nn.value, st[2]

    def dev_put(h):
        cols = (L.TQColumn * 2)(dk.tq(), dx.tq())
        cols[0].null_bitmap = None
        cols[1].null_bitmap = None
        L.check(lib.tq_agg_put(h, cols, L.TQ_MEM_DEVICE))
    for _ in range(args.warmup):
        g, _ = step(L.TQ_MEM_DEVICE, dev_put)
        assert g == len(np.unique(k[: 1])) or g == groups or g > 0
    sampler = sampler_cls(0)
    sampler.start()
    l1 = lib.tq_kernel_launch_count()
    ms = C.c_float(0)
    upd = []
    L.check(lib.tq_timer_start())
    for i in range(args.steps):
        g, ns = step(L.TQ_MEM_DEVICE, dev_put, hold=args.dump is not None and i == args.steps - 1)
        upd.append(ns)
    L.check(lib.tq_timer_stop(C.byref(ms)))
    clocks = sampler.stop()
    l2 = lib.tq_kernel_launch_count()
    if held:
        # SUM, COUNT, firstrow(k) of a seeded sample of the groups in key order (the group table's order is not part of the result)
        from bench import sample_rows
        h, out, ng = held.pop()
        res = [device_to_host(tp, out[i].data, None, ng).values for i, tp in enumerate((FLOAT64, INT64, INT64))]
        L.check(lib.tq_agg_destroy(h))
        rows = np.argsort(res[2], kind="stable")[sample_rows(ng)]
        args.dump.update({"agg_groups": np.array([ng], dtype=np.float64), "agg_sum": res[0][rows], "agg_count": res[1][rows].astype(np.float64),
                          "agg_key": res[2][rows].astype(np.float64)})
    ms_step = ms.value / args.steps
    pk, _ = _pinned(lib, n, np.int64, k)
    px, _ = _pinned(lib, n, np.float64, x)

    def host_put(h):
        piece = 1 << 23
        for lo in range(0, n, piece):
            rows = min(piece, n - lo)
            cols = (L.TQColumn * 2)(_col(pk.value + lo * 8, rows), _col(px.value + lo * 8, rows))
            L.check(lib.tq_agg_put(h, cols, L.TQ_MEM_HOST))
    h_res = [np.empty(groups + 16, dtype=np.float64), np.empty(groups + 16, dtype=np.int64), np.empty(groups + 16, dtype=np.int64)]
    h_bm = [np.zeros(groups // 8 + 16, dtype=np.uint8) for _ in range(3)]

    def step_host():
        """Open / put (8M-row host pieces) / eof / Next until EOF with HOST result buffers / Close — the result comes back too"""
        h = C.c_void_p()
        L.check(lib.tq_agg_create(C.byref(desc), C.byref(h)))
        host_put(h)
        L.check(lib.tq_agg_eof(h))
        out = (L.TQColumn * 3)()
        for i in range(3):
            out[i].data, out[i].null_bitmap, out[i].offsets = h_res[i].ctypes.data, h_bm[i].ctypes.data, None
        nn, eof = C.c_int64(0), C.c_int32(0)
        L.check(lib.tq_agg_next(h, groups + 16, out, C.byref(nn), C.byref(eof)))
        L.check(lib.tq_agg_destroy(h))
        return nn.value
    step_host()
    t0 = time.perf_counter()
    g_host = step_host()
    e2e_s = time.perf_counter() - t0
    # full-size value check: every group's COUNT exactly, SUM within 1e-9 relative (north_star), key set complete
    want_cnt = np.bincount(k, minlength=groups)
    want_sum = np.bincount(k, weights=x, minlength=groups)
    keys = h_res[2][:g_host]
    order_ok = g_host == int((want_cnt > 0).sum()) and np.array_equal(np.sort(keys), np.nonzero(want_cnt)[0])
    cnt_ok = order_ok and np.array_equal(h_res[1][:g_host], want_cnt[keys])
    sum_ok = order_ok and bool(np.all(np.abs(h_res[0][:g_host] - want_sum[keys]) <= 1e-9 * np.maximum(1.0, np.abs(want_sum[keys]))))
    verified = {"ok": bool(order_ok and cnt_ok and sum_ok), "groups": int(g_host),
                "checks": {"group keys": bool(order_ok), "COUNT exact": bool(cnt_ok), "SUM within 1e-9 relative": bool(sum_ok)}}
    import oracle_py as O
    olib = O.load()
    sample = min(n, 20_000_000)
    sec, ss, sc = C.c_double(0), C.c_double(0), C.c_int64(0)
    workers = os.cpu_count() or 1
    olib.orc_mt_agg_bench(C.c_int64(sample), C.c_void_p(k.ctypes.data), C.c_void_p(x.ctypes.data), C.c_int(workers), C.c_int(workers), C.byref(sec), C.byref(ss),
                          C.byref(sc))
    upd_s = statistics.mean(upd) * 1e-9
    achieved = 16.0 * n / upd_s / 1e9
    out = {
        "metric": "rows/sec, GROUP BY int64 key with SUM(float64), COUNT(*)", "value": n / (ms_step * 1e-3), "unit": "rows/s", "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64/int64", "data": "synthetic",
        "config": {"workload": f"C4: {n}-row GROUP BY int64 key, SUM(float64) + COUNT(*) + firstrow(key), {groups} groups, uniform keys", "groups_out": int(g),
                   "l2": "input 1.6 GB exceeds L2; the 1e6-group state (~50 MB) is L2-resident by design"},
        "roofline": {"bound": "hbm", "kernel": "update pipeline of one batch, timed together: k_scatter_aos (radix scatter by key hash) + k_agg_preagg (shared-memory pre-aggregation per partition) + k_agg_update over the partial rows; below 4 input rows per group, or between 1e4 and 1.5e5 groups, k_agg_update alone", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                     "peak_source": peak_src, "algorithmic_bytes_per_row": 16, "kernel_ms": upd_s * 1e3},
        "e2e": {"value": n / e2e_s, "unit": "rows/s", "h2d_bytes_per_step": 16 * n, "d2h_bytes_per_step": int(g_host) * 24 + 3 * (int(g_host) // 8), "ms_per_step": e2e_s * 1e3},
        "gpu_launches": int(l2 - l1), "clocks": clocks, "verified": verified,
        "cpu_baseline": {"value": sample / sec.value, "unit": "rows/s", "cores": workers, "kind": "port",
                         "sample": f"first {sample} rows, {workers} partial + {workers} final workers (oracle/cpu_ref.c restatement of aggregate.go:96-133)"},
    }
    dk.free()
    dx.free()
    lib.tq_pinned_free(pk)
    lib.tq_pinned_free(px)
    return out


def run(args, rank, world, local_rank):
    if rank != 0:
        return None
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tests"))
    from bench import ClockSampler, measured_peak
    lib = L.load()
    L.check(lib.tq_init(local_rank))
    peak, peak_src = measured_peak()
    if args.workload == "expr":
        return run_expr(args, lib, peak, peak_src, ClockSampler)
    return run_agg(args, lib, peak, peak_src, ClockSampler)
