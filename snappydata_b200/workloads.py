"""BASELINE.json configs[3] and [4] as runnable workloads (SURVEY.md 8d C4 / C5), used by bench.py (`--workload c4|c5`, and as
`also_c4` / `also_c5` of the default run).  Synthetic tables are written with the fixture writer (real ColumnBatch bytes); every
GPU result is checked against the oracle / an independent numpy evaluation before a number is reported.

C4  wide table, 128 columns c0..c127 cycling (INT, DOUBLE, dictionary STRING of 1000 distinct 8-12 byte values), every 4th
    column nullable (10 % NULLs), 100 M rows over the job; SELECT c0..c7 WHERE c0 BETWEEN a AND b AND c2 = 'lit' at ~1 %
    combined selectivity.  Only the 8 scanned columns are materialised (the other 120 are never read by the plan).  The
    spec's uniform 1000-value strings cannot give 1 % with an equality on one of them (<= 0.1 %), so c2 is skewed: the
    literal's value takes 2 % of the rows.  10 M distinct rows are generated and every batch is resident 10 times under
    distinct batch ids (the scan reads all of them from HBM: 100 M rows x 39.1 B is far beyond the 126 MB L2).
C5  hybrid scan: TPC-H Q6 over SF-10 lineitem where every batch carries update deltas (0.5 % of the rows in l_discount and
    l_quantity: <= 100 positions at depth 0, the rest at depth 1, a few in both), a delete mask (0.5 %), plus row-buffer
    rows; an INGEST THREAD appends new batches while the timed queries run -- encoded on the device from raw values
    (sd_store_encode_batch, the N2 path).  Every query scans the
    snapshot of batches present when it started; its result must equal the oracle's over exactly that snapshot.
"""
from __future__ import annotations

import ctypes as C
import threading
import time
from typing import List

import numpy as np

from . import capi, lineitem, plan as P
from .column_format import ColumnBatch, SqlType as T, encode_delete, encode_delta, encode_dictionary, encode_uncompressed, unsafe_row
from .exchange import shard_batches
from .plan import PlanBuilder

ROWS_PER_BATCH = 200_000
C4_TOTAL_ROWS = 100_000_000
C4_BASE_BATCHES = 50
C4_WORDS = np.array([b"str%05d" % i + b"x" * (1 + i % 5) for i in range(1000)], dtype="S12")
C4_TYPES = [(T.INT, T.DOUBLE, T.STRING)[i % 3] for i in range(128)]
C4_LITS = [0, 549, bytes(C4_WORDS[7])]


def c4_plan():
    pb = PlanBuilder()
    c = [pb.col(C4_TYPES[i], i, i % 4 == 0) for i in range(8)]
    pb.filter((c[0] >= pb.lit(T.INT)) & (c[0] <= pb.lit(T.INT)) & c[2].eq(pb.lit(T.STRING)))
    pb.project(*c)
    return pb.build()


def c4_base_batch(k: int):
    """base batch k (deterministic): -> (ColumnBatch with 8 materialised columns, number of rows the query selects)"""
    r = np.random.default_rng(4000 + k)
    n = ROWS_PER_BATCH
    cols: List = [None] * 128
    vals = {}
    for i in range(8):
        nulls = (r.random(n) < 0.1) if i % 4 == 0 else None
        if C4_TYPES[i] == T.INT:
            v = r.integers(0, 1000, n).astype(np.int32)
            cols[i] = encode_uncompressed(v, T.INT, nulls)
        elif C4_TYPES[i] == T.DOUBLE:
            v = r.random(n) * 100.0
            cols[i] = encode_uncompressed(v, T.DOUBLE, nulls)
        else:
            idx = r.integers(0, 1000, n)
            if i == 2:
                idx[r.random(n) < 0.02] = 7          # the literal's value: 2 % of the rows
            v = idx
            cols[i] = encode_dictionary(C4_WORDS[idx], T.STRING, nulls)
        vals[i] = (v, nulls)
    c0, n0 = vals[0]
    sel = (~n0) & (c0 >= C4_LITS[0]) & (c0 <= C4_LITS[1]) & (vals[2][0] == 7)
    return ColumnBatch(num_rows=n, columns=cols, batch_id=k, bucket_id=k % 8), int(sel.sum())


def run_c4(api, torch, dist, rank, world, device, steps, warmup, peak):
    from oracle import oracle
    first_row, nrows, nb = shard_batches(C4_TOTAL_ROWS, ROWS_PER_BATCH, rank, world)
    b0 = first_row // ROWS_PER_BATCH
    need = sorted({(b0 + i) % C4_BASE_BATCHES for i in range(nb)})
    t0 = time.perf_counter()
    base = {k: c4_base_batch(k) for k in need}
    gen_s = time.perf_counter() - t0
    schema = [(C4_TYPES[i], i % 4 == 0) for i in range(128)]
    store = capi.Store(api, schema, device)
    expect_rows = 0
    import copy
    for i in range(nb):
        cb, cnt = base[(b0 + i) % C4_BASE_BATCHES]
        cb2 = copy.copy(cb)
        cb2.batch_id = b0 + i
        store.put(cb2)
        expect_rows += cnt
    desc = c4_plan()
    gp = capi.Plan(api, desc)
    gp.set_stream(torch.cuda.current_stream().cuda_stream)
    # parity: two base batches through the oracle (row for row), then the whole shard's row count against numpy
    sample = [base[k][0] for k in need[:2]]
    op = oracle.plan(desc).set_literals(C4_LITS)
    gp.reset().set_literals(C4_LITS)
    for cb in sample:
        op.submit(cb)
        gp.submit(cb)
    want, got = op.finish(), gp.finish()
    key = lambda r: tuple((0, 0) if v is None else (1, v) for v in r)
    rows_equal = sorted(want, key=key) == sorted(got, key=key)
    lit_arr = gp.literal_array(C4_LITS)

    def step():
        raw = gp.execute_store_view(store, lit_arr, len(C4_LITS), None)   # rows in the handle's page-locked buffer
        return len(raw)
    for _ in range(warmup):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out_bytes = 0
    for _ in range(steps):
        out_bytes = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    m = gp.metrics()
    if world > 1:
        t = torch.tensor([ms, float(m["numOutputRows"]), float(expect_rows), float(nrows)], dtype=torch.float64, device="cuda")
        mx = t.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        ms, out_rows, exp_rows, job_rows = float(mx[0]), int(t[1]), int(t[2]), int(t[3])
    else:
        out_rows, exp_rows, job_rows = m["numOutputRows"], expect_rows, nrows
    kernel_ms = m["aggTimeNs"] / 1e6
    rec_bytes = m["numOutputRows"] * (8 + 8 * 8)            # fixed-width records the kernel writes (batch ordinal + null bits + 8 fields)
    algo = m["algorithmicBytes"] + rec_bytes
    achieved = algo / (kernel_ms / 1e3) / 1e9 if kernel_ms > 0 else 0.0
    ok = rows_equal and out_rows == exp_rows
    return {"workload": "C4 wide table: 128-column schema (8 scanned columns materialised), 100 M rows, SELECT c0..c7 WHERE c0 BETWEEN a AND b AND c2 = 'lit'",
            "value": job_rows / (ms / 1e3), "unit": "rows/s", "ms_per_step": ms, "steps": steps, "n_gpus": world, "rows": job_rows,
            "rows_out": out_rows, "selectivity": out_rows / max(1, job_rows), "d2h_bytes_per_step": out_bytes,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "kernel_ms_per_launch": kernel_ms,
                         "algorithmic_bytes_per_launch": algo, "bytes_per_row_read": m["algorithmicBytes"] / max(1, nrows),
                         "kernel": "sd::scan_aggregate_kernel<" + gp.kernel_name() + "> (MODE_PROJECT, NULL-aware staged path)",
                         "note": "per rank; algorithmic bytes = column bodies + null words read (SURVEY.md 8d: ~39.1 B/row) + 72-byte output records written"},
            "parity_check": {"ok": bool(ok), "sample_rows_vs_oracle": len(want), "sample_equal": bool(rows_equal), "rows_out": out_rows,
                             "rows_out_expected": exp_rows, "checker": "oracle row-for-row on two batches; whole-shard row count against a numpy evaluation of the predicate"},
            "note": f"10 M distinct rows generated in {gen_s:.1f} s on the host, each batch resident 10x under distinct ids; whole step includes writing the "
                    "projected UnsafeRows on the device (sd_rows.cu) and their copy into a page-locked host buffer; c2 skewed so that 1 % is reachable"}


# ---- C5 ------------------------------------------------------------------------------------------------------------------
def _decorate_hybrid(cb: ColumnBatch, r):
    n = cb.num_rows
    upd = np.sort(r.choice(n, size=max(1, n // 200), replace=False)).astype(np.int32)          # 0.5 % updated
    d0 = upd[:100]
    d1 = np.sort(np.unique(np.concatenate([upd[100:], d0[:5]]))).astype(np.int32)               # a few positions in both levels
    for col, vals in ((P.L_DISCOUNT, lambda m: r.integers(0, 11, m) / 100.0), (P.L_QUANTITY, lambda m: r.integers(1, 51, m).astype(np.float64))):
        cb.delta0[col] = encode_delta(n, d0, vals(len(d0)), T.DOUBLE)
        cb.delta1[col] = encode_delta(n, d1, vals(len(d1)), T.DOUBLE)
    cb.delete_mask = encode_delete(n, np.sort(r.choice(n, size=max(1, n // 200), replace=False)))  # 0.5 % deleted
    return cb


def run_c5(api, torch, device, steps, warmup, peak, total_rows=59_986_052, ingest_batches=60):
    """1 GPU.  -> JSON-able dict with value (rows/s over the snapshots actually scanned), roofline and the parity assertion."""
    from oracle import oracle
    r = np.random.default_rng(5)
    desc = P.q6_plan()
    cols = desc.table_cols
    # base table generated on the device, pulled back once, decorated with deltas / deletes on the host, re-put
    gen = capi.Store(api, lineitem.LINEITEM_SCHEMA, device)
    extra_rows = ingest_batches * ROWS_PER_BATCH
    gen.gen_lineitem(0, total_rows + extra_rows, ROWS_PER_BATCH, 128, 6, lineitem.Q6_COLUMN_MASK)
    nb_all = gen.num_batches()
    nb_base = (total_rows + ROWS_PER_BATCH - 1) // ROWS_PER_BATCH
    batches = []
    for i in range(nb_all):
        nrows, bucket, bid = gen.batch_info(i)
        bufs = [None] * 16
        for c in cols:
            bufs[c] = gen.get_buffer(i, c)
        cb = ColumnBatch(num_rows=nrows, columns=bufs, batch_id=bid, bucket_id=bucket)
        # batches of the base table carry deltas and deletes; freshly ingested ones (i >= nb_base) do not
        batches.append(_decorate_hybrid(cb, r) if i < nb_base else cb)
    gen.close()
    nrb = 10_000
    rows = b""
    for _ in range(nrb):
        row = unsafe_row([(T.DATE, int(8036 + r.integers(0, 2526))), (T.DOUBLE, float(r.integers(0, 11) / 100.0)),
                          (T.DOUBLE, float(r.integers(1, 51))), (T.DOUBLE, float(r.integers(90000, 10500000) / 100.0))])
        rows += len(row).to_bytes(8, "little") + row
    store = capi.Store(api, lineitem.LINEITEM_SCHEMA, device)
    marshalled = [capi.MarshalledBatch(b, None) for b in batches]
    for mb in marshalled[:nb_base]:
        api.check(api.store_put_batch(store.h, C.byref(mb.c)))
    # the oracle's partial answer per batch (and for the row buffer), once: expected(snapshot of n batches) = prefix sums
    per_sum, per_rows = [], []
    for b in batches:
        op = oracle.plan(desc).set_literals(P.Q6_LITERALS)
        op.submit(b)
        (v,), = op.finish()
        per_sum.append(v)
        per_rows.append(op.metrics()["rowsScanned"])
        op.close()
    op = oracle.plan(desc).set_literals(P.Q6_LITERALS)
    op.submit_rows(rows, nrb)
    (rb_sum,), = op.finish()
    op.close()
    pre_sum = np.concatenate([[0.0], np.cumsum([0.0 if v is None else v for v in per_sum])])
    pre_rows = np.concatenate([[0], np.cumsum(per_rows)])

    gp = capi.Plan(api, desc)
    gp.set_stream(torch.cuda.current_stream().cuda_stream)

    def query():
        gp.reset().set_literals(P.Q6_LITERALS)
        gp.submit_rows(rows, nrb)
        gp.scan_store(store)
        raw = gp.finish_raw()
        m = gp.metrics()
        (v,), = capi.parse_row_stream(raw, desc.partial_schema())
        return v, m
    for _ in range(warmup):
        query()
    stop = threading.Event()
    ingested = [0]

    # raw values of the batches to ingest (all four Q6 columns are NOT NULL and Uncompressed: the body IS the value array)
    dts = {P.L_SHIPDATE: "<i4", P.L_DISCOUNT: "<f8", P.L_QUANTITY: "<f8", P.L_EXTENDEDPRICE: "<f8"}
    raws = [{c: (np.frombuffer(b.columns[c], dtype=dts[c], offset=8), None) for c in cols} for b in batches[nb_base:]]

    def ingest():   # new batches are ENCODED ON THE DEVICE from raw values (sd_store_encode_batch) while queries run
        for b, raw in zip(batches[nb_base:], raws):   # (ctypes releases the GIL during the call)
            if stop.is_set():
                break
            try:
                store.encode_batch(b.num_rows, raw, b.bucket_id, b.batch_id)
            except Exception:
                break
            ingested[0] += 1
            time.sleep(0.0005)
    th = threading.Thread(target=ingest)
    results = []
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    th.start()
    for _ in range(steps):
        results.append(query())
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    stop.set()
    th.join()
    # parity on every query's own snapshot
    ok, max_rel, snaps, scanned_total, kernel_ns, algo = True, 0.0, [], 0, 0, 0
    for v, m in results:
        n = m["columnBatchesSeen"]
        snaps.append(n)
        want = pre_sum[n] + (rb_sum or 0.0)
        rel = abs(v - want) / max(abs(want), 1e-300)
        max_rel = max(max_rel, rel)
        ok = ok and rel <= 1e-6 and m["rowsScanned"] == int(pre_rows[n]) + nrb and m["numRowsBuffer"] == nrb
        scanned_total += m["rowsScanned"]
        kernel_ns += m["aggTimeNs"]
        algo += m["algorithmicBytes"]
    achieved = algo / (kernel_ns / 1e9) / 1e9 if kernel_ns else 0.0
    return {"workload": "C5 hybrid scan: TPC-H Q6 on SF-10 lineitem with update deltas (2 levels), delete masks, row-buffer rows, under concurrent ingest",
            "value": scanned_total / dt, "unit": "rows/s", "ms_per_step": dt / steps * 1e3, "steps": steps, "n_gpus": 1,
            "snapshots_batches": [int(min(snaps)), int(max(snaps))], "ingested_batches_during_timed_region": int(ingested[0]),
            "base_batches": nb_base, "row_buffer_rows": nrb,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "kernel_ms_per_launch": kernel_ns / 1e6 / max(1, sum(m["kernelLaunches"] for _, m in results)),
                         "kernel": "sd::scan_aggregate_kernel<" + gp.kernel_name() + "> (staged ring + delta / delete overlay)",
                         "note": "algorithmic bytes = 28 B/row + the delta and delete bytes present (SURVEY.md 8d)"},
            "parity_check": {"ok": bool(ok), "queries": len(results), "max_rel_err": max_rel, "tolerance": 1e-6,
                             "checker": "every query against the oracle's answer over exactly the batches of its own snapshot (columnBatchesSeen) "
                                        "+ the row buffer; scanned row counts exact"},
            "note": "every query rebuilds its batch descriptors when the store changed under it (store version); wall-clock timing of the "
                    "query loop (row-buffer submit + scan + read-back) while the ingest thread uploads batches over the same PCIe link"}
