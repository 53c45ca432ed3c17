#!/usr/bin/env python
"""bench.py -- TPC-H Q1 / Q6 lineitem scan + filter + partial aggregate on N B200s vs the CPU path.

Contract (see the task brief): `python bench.py --gpus N --steps K --warmup W` (under torchrun for
N > 1) prints ONE JSON line on rank 0.  A "step" is one execution of the query over the whole
(sharded) column table:

  value   whole-job rows/s with the ColumnBatches resident in HBM (sd_plan_scan_store), including the
          partial-row read-back and the cross-rank exchange + final merge
  e2e     the same query through the reference-facing C-ABI with HOST buffers: every step submits every
          ColumnBatch from pinned host memory (sd_batch_submit copies it to the device inside the call)
          and reads the partial rows back
  roofline.achieved   algorithmic bytes (SURVEY.md 8d: 40 B/row Q1, 28 B/row Q6, computed from the actual
          buffers) / device time of the scan kernel (CUDA events around the launches, on the launching stream)
  cpu_baseline        the reference-algorithm CPU restatement (oracle/, generated-loop layer) timed on this
          box's host cores over a bounded sample of the same ColumnBatch bytes

`--impl reference` times that CPU restatement as the reference arm (the reference itself is Scala on a
Spark fork whose sources are absent and there is no JVM here: DESIGN.md).

Workload: Q1 over ONE SF-100 lineitem column table (600,037,902 rows, 200,000-row batches, 24.0 GB of scanned
column bytes).  The path partitions by bucket, so N > 1 is one process per GPU, each holding and scanning a contiguous
range of the table's batches (`"scaling": "strong"`, the default: BASELINE.json's "Q1 on SF-100, 1->8 GPUs") with no
data-path collective and ONE exchange per query: sd_plan_exchange = an ncclAllGather of every rank's partial rows inside
libsnappygpu.so, merged on every rank, then the final merge.  `--scaling weak` gives every rank its own table-sized
partition set instead.  Q6 over SF-10 is measured in the same run and reported under "also".

`parity_check`: in the same run the oracle's generated-loop layer (CPU) scans the SAME ColumnBatch bytes at the
benchmark's own size (every rank its shard; partial rows gathered and merged) and the GPU result must match: counts
bit-exact, DOUBLE sums / averages within 1e-6 relative (BASELINE.json north_star).  A mismatch fails the run.

`--dump-outputs DIR` writes the final rows of the last timed step of Q1 and Q6 as .npy files.  The tables are generated
on the device from fixed seeds, so the same arguments give the same inputs on every run and two builds can be compared
output for output.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SF100_ROWS = 600_037_902
SF10_ROWS = 59_986_052
ROWS_PER_BATCH = 200_000
NBUCKETS = 128
SEED_Q1, SEED_Q6 = 1, 6


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="q1", choices=["q1", "q6", "c4", "c5"],
                    help="q1 (default; Q6 SF-10, C4 and C5 are measured in the same run under also / also_c4 / also_c5), q6, or one of "
                         "BASELINE.json's other configs alone: c4 = wide-table filter + projection, c5 = hybrid scan under concurrent ingest")
    ap.add_argument("--no-extras", action="store_true", help="skip also_c4 / also_c5 in the default run")
    ap.add_argument("--rows", type=int, default=0, help="override total table rows (default SF-100 for q1, SF-10 for q6)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-also", action="store_true")
    ap.add_argument("--no-lz4", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"],
                    help="N > 1: strong (default, BASELINE.json: ONE SF-100 table over 1->8 GPUs) = the table split into N contiguous "
                         "batch ranges, one partition set per GPU; weak = every rank scans its own table-sized partition set")
    ap.add_argument("--no-parity", action="store_true", help="skip the GPU-vs-oracle parity check at the benchmark's own size")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the final rows of the last timed step of each Q1 / Q6 query to DIR/<query>_keys.npy and "
                         "DIR/<query>_values.npy (float64), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "native" or args.workload not in ("q1", "q6")):
        ap.error("--dump-outputs covers the Q1 / Q6 queries of the native implementation")
    return args


def dump_final_rows(out_dir, name, rows, desc):
    """Final rows of one query as float64 arrays, groups sorted by key: <name>_keys.npy (groups, keys, longest key) holds
    the bytes of the string keys, zero-padded (Q6 has no keys and no such file); <name>_values.npy (groups, aggregates)
    the aggregates, NULL as NaN."""
    import numpy as np
    nkeys = len(desc.keys_py)
    rows = sorted(rows, key=lambda r: tuple(r[:nkeys]))
    os.makedirs(out_dir, exist_ok=True)
    if nkeys:
        width = max((len(k) for r in rows for k in r[:nkeys]), default=0)
        keys = np.zeros((len(rows), nkeys, width), dtype=np.float64)
        for i, r in enumerate(rows):
            for j, k in enumerate(r[:nkeys]):
                keys[i, j, :len(k)] = np.frombuffer(k, dtype=np.uint8)
        np.save(os.path.join(out_dir, name + "_keys.npy"), keys)
    values = np.array([[np.nan if v is None else float(v) for v in r[nkeys:]] for r in rows], dtype=np.float64)
    np.save(os.path.join(out_dir, name + "_values.npy"), values.reshape(len(rows), len(desc.final_schema()) - nkeys))


def ncu_traffic_per_row(q1):
    """DRAM bytes per row of the scan kernel from the committed `ncu --set full` capture (profiles/)."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))["q1" if q1 else "q6"]
        return (t["dram_read_bytes"] + t["dram_write_bytes"]) / t["rows"]
    except Exception:
        return None


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def cgroup_cpu_limit():
    """CPUs this container may actually use (cgroup quota), or None when unlimited/unknown."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            return max(1, int(float(q) / float(per)))
    except Exception:
        pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0:
            return max(1, q // per)
    except Exception:
        pass
    return None


def pick_threads(run_once, rows):
    """The reference runs one task per core (Spark local[N]); on a shared box the visible core count can exceed what
    the container may use, so try a few thread counts on the sample and keep the fastest."""
    visible = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cands = sorted({t for t in (8, 16, 32, 64, visible, cgroup_cpu_limit() or visible) if 1 <= t <= visible})
    best, best_rate = visible, 0.0
    for t in cands:
        run_once(t)
        t0 = time.perf_counter()
        run_once(t)
        rate = rows / (time.perf_counter() - t0)
        if rate > best_rate:
            best, best_rate = t, rate
    return best, {"visible_cpus": visible, "cgroup_cpu_limit": cgroup_cpu_limit(), "tried": cands}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, reasons = [], set()
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                out["sm_max_mhz"] = float(r[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower() == "active":
                    reasons.add(name)
        if sm:
            sm.sort()
            out["sm_mhz"] = sm[len(sm) // 2]
        out["reasons"] = sorted(reasons)
        out["samples"] = len(sm)
        return out


def shard_batches(total_rows, rank, world):
    from snappydata_b200.exchange import shard_batches as sb
    return sb(total_rows, ROWS_PER_BATCH, rank, world)


# ---------------------------------------------------------------------------------------------------
def run_reference_arm(args):
    """`--impl reference`: the reference-algorithm CPU restatement (generated-loop layer of the oracle) over a
    bounded sample of the workload, all host threads, one partition per thread like Spark local[N]."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle
    from snappydata_b200 import lineitem, plan as P
    q1 = args.workload == "q1"
    desc = P.q1_plan() if q1 else P.q6_plan()
    total = args.rows or (SF100_ROWS if q1 else SF10_ROWS)
    cores = os.cpu_count() or 1
    nsample = min((total + ROWS_PER_BATCH - 1) // ROWS_PER_BATCH, max(64, min(512, 4 * cores)))
    batches = lineitem.gen_table(total, ROWS_PER_BATCH, SEED_Q1 if q1 else SEED_Q6, NBUCKETS,
                                 lineitem.Q1_COLUMN_MASK if q1 else lineitem.Q6_COLUMN_MASK, batches=range(nsample))
    ba = oracle.BatchArray(batches, desc.table_cols)
    rows = sum(b.num_rows for b in batches)

    def run_once(t):
        if q1:
            oracle.run_q1(ba, P.Q1_LITERALS[0], t)
        else:
            oracle.run_q6(ba, P.Q6_LITERALS, t)
    cores, cpu_info = pick_threads(run_once, rows)

    def step():
        run_once(cores)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    v = rows * args.steps / dt
    sample = f"first {nsample} batches ({rows} rows) of the {total}-row table per step"
    print(json.dumps({
        "impl": "reference", "metric": metric_name(q1), "value": v, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(q1, total, args.gpus, args.scaling),
        "cpu_baseline": {"value": v, "unit": "rows/s", "cores": cores, "kind": "port", "sample": sample, "cpus": cpu_info},
        "e2e": {"value": v, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference-algorithm CPU restatement (oracle/scan_oracle.c, generated-loop layer); the reference itself "
                "cannot run here (Scala on an absent Spark fork, no JVM)"}))


def metric_name(q1):
    return ("rows/sec, TPC-H Q1 lineitem scan+filter+group-by aggregate over a column table" if q1
            else "rows/sec, TPC-H Q6 lineitem scan+filter+aggregate over a column table")


def workload_config(q1, total, gpus, scaling="weak"):
    if scaling == "weak":
        sharding = (f"{gpus} rank(s), one process per GPU; every rank holds and scans its own {total}-row partition set "
                    f"(weak scaling: {gpus * total} rows per step in total); no data-path collective, one all-gather of partial rows")
    else:
        sharding = f"one {total}-row table split into contiguous batch ranges over {gpus} rank(s), one partition per GPU"
    return {"workload": ("TPC-H Q1 on SF-100 lineitem column table" if q1 else "TPC-H Q6 on SF-10 lineitem column table"),
            "rows": total, "rows_per_gpu": total if scaling == "weak" else (total + gpus - 1) // gpus,
            "total_rows": total * gpus if scaling == "weak" else total,
            "rows_per_batch": ROWS_PER_BATCH, "bytes_per_row": 40 if q1 else 28,
            "sharding": sharding,
            "l2": "inputs per step (>= 3 GB per GPU) are larger than the 126 MB L2; no flush needed",
            "literals": "Q1 cutoff 1997-10-02; Q6 1994-01-01, 0.05..0.07, 24"}


# ---------------------------------------------------------------------------------------------------
class QueryRun:
    """One query over this rank's shard: resident store, plan, timing helpers."""

    def __init__(self, api, torch, dist, q1, total_rows, rank, world, device, scaling="strong", comm=None):
        from snappydata_b200 import capi, lineitem, plan as P
        self.api, self.torch, self.dist, self.q1, self.rank, self.world = api, torch, dist, q1, rank, world
        self.capi = capi
        self.desc = P.q1_plan() if q1 else P.q6_plan()
        self.lits = P.Q1_LITERALS if q1 else P.Q6_LITERALS
        self.total_rows = total_rows
        if scaling == "weak" or world == 1:
            # rank r's partition set: `total_rows` rows of its own, starting at a batch-aligned row of the generator's stream
            stride = (total_rows + ROWS_PER_BATCH - 1) // ROWS_PER_BATCH * ROWS_PER_BATCH
            first_row, nrows = rank * stride, total_rows
            self.job_rows = total_rows * world
            self.e2e_rows_target = total_rows if world == 1 else (total_rows + world - 1) // world   # bounds pinned host memory
        else:
            first_row, nrows, _ = shard_batches(total_rows, rank, world)
            self.job_rows = total_rows
            self.e2e_rows_target = nrows
        self.local_rows = nrows
        self.store = capi.Store(api, lineitem.LINEITEM_SCHEMA, device)
        self.store.gen_lineitem(first_row, nrows, ROWS_PER_BATCH, NBUCKETS, SEED_Q1 if q1 else SEED_Q6,
                                lineitem.Q1_COLUMN_MASK if q1 else lineitem.Q6_COLUMN_MASK)
        self.plan = capi.Plan(api, self.desc)
        self.plan.set_stream(torch.cuda.current_stream().cuda_stream)
        self.merge_plan = self.plan
        self.launches = 0
        self.kernel_ns = 0
        self.algo_bytes = 0
        self.final_raw = b""
        self.lit_array = self.plan.literal_array(self.lits)
        self._m = (C.c_int64 * capi.SD_NUM_METRICS)()
        self.comm = comm   # capi.Comm (sd_comm: NCCL inside the library) or None

    def exchange_and_merge(self, plan):
        """The one exchange of the query (sd_plan_exchange: ncclAllGather of every rank's partial rows inside the library,
        merged on every rank), then the final merge (SnappyHashAggregateExec(Final) / CollectAggregateExec)."""
        if self.comm is not None:
            plan.exchange(self.comm)
        raw = plan.finish_raw()
        self.final_raw = self.merge_plan.final_merge_raw(raw)   # final rows of the query (parsed after the timed region)
        return len(raw)

    def step_resident(self):
        """One execution of the cached plan over the resident shard: ONE C call (reset, literals, scan, exchange, partial
        rows), then the final merge."""
        p = self.plan
        raw = p.execute_store_raw(self.store, self.lit_array, len(self.lits), self.comm)
        self.api.plan_metrics(p.h, self._m)
        m = self._m
        self.launches += m[7]
        self.kernel_ns += m[6]
        self.algo_bytes += m[9]
        self.final_raw = self.merge_plan.final_merge_raw(raw)
        return len(raw)

    # ---- end to end: host buffers -> sd_batch_submit ---------------------------------------------
    def prepare_host_copy(self):
        """Pinned host copy of this rank's ColumnBatch buffers + pre-marshalled sd_batch structs."""
        torch, capi = self.torch, self.capi
        from snappydata_b200.column_format import ColumnBatch
        cols = self.desc.table_cols
        self.host_keep, self.marshalled, self.h2d_bytes = [], [], 0
        nb = min(self.store.num_batches(), max(1, (self.e2e_rows_target + ROWS_PER_BATCH - 1) // ROWS_PER_BATCH))
        self.e2e_rows = sum(self.store.batch_info(i)[0] for i in range(nb))
        sizes = []
        for i in range(nb):
            for c in cols:
                ln = C.c_int64()
                self.api.lib.sdx_store_get_buffer(self.store.h, i, c, None, 0, C.byref(ln))
                sizes.append(ln.value)
        total = sum((s + 63) // 64 * 64 for s in sizes)
        arena = torch.empty(max(total, 64), dtype=torch.uint8).pin_memory()
        base = arena.data_ptr()
        off, k = 0, 0
        for i in range(nb):
            nrows, bucket, bid = self.store.batch_info(i)
            bufs = [None] * 16
            for c in cols:
                ln = C.c_int64()
                self.api.check(self.api.lib.sdx_store_get_buffer(self.store.h, i, c, base + off, sizes[k], C.byref(ln)))
                bufs[c] = arena[off: off + sizes[k]].numpy()
                self.h2d_bytes += sizes[k]
                off += (sizes[k] + 63) // 64 * 64
                k += 1
            cb = ColumnBatch(num_rows=nrows, columns=bufs, stats=None, batch_id=bid, bucket_id=bucket)
            self.marshalled.append(capi.MarshalledBatch(cb, cols))
        self.host_keep.append(arena)
        self.e2e_plan = capi.Plan(self.api, self.desc)
        self.e2e_plan.set_stream(torch.cuda.current_stream().cuda_stream)
        if not os.environ.get("BENCH_NO_RETAIN"):
            # the pinned host copy outlives every step: let the engine queue the copies back to back
            self.e2e_plan.set_option(capi.SD_OPT_RETAIN_BUFFERS, 1)

    def prepare_compressed_copy(self, threads=32):
        """The same ColumnBatches in their STORED form: every buffer >= 2048 B that LZ4 shrinks to <= 75 % becomes
        [-1][uncompressedLen][LZ4 block] (CompressionUtils.scala:47-61,102-110).  liblz4 (runtime library of the
        image) does the compression here; the engine expands the blocks on the device."""
        import concurrent.futures
        import ctypes.util
        import numpy as np
        from snappydata_b200.column_format import ColumnBatch
        torch, capi = self.torch, self.capi
        lz = C.CDLL(ctypes.util.find_library("lz4") or "liblz4.so.1")
        lz.LZ4_compress_default.restype = C.c_int
        lz.LZ4_compress_default.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        lz.LZ4_compressBound.restype = C.c_int
        lz.LZ4_compressBound.argtypes = [C.c_int]
        cols = self.desc.table_cols
        jobs, off = [], 0
        for bi, mb in enumerate(self.marshalled):
            for k, c in enumerate(cols):
                n = int(mb.col_lens[k])
                cap = lz.LZ4_compressBound(n) + 8
                jobs.append((bi, k, int(mb.col_bufs[k]), n, off, cap))
                off += (cap + 63) // 64 * 64
        arena = torch.empty(max(off, 64), dtype=torch.uint8).pin_memory()
        base = arena.data_ptr()

        def work(j):
            bi, k, src, n, o, cap = j
            if n < 2048:
                return (bi, k, src, n)
            cl = lz.LZ4_compress_default(src, base + o + 8, n, cap - 8)
            if cl <= 0 or cl > (n * 3) // 4:
                return (bi, k, src, n)
            hdr = np.frombuffer((C.c_char * 8).from_address(base + o), dtype="<i4")
            hdr[0], hdr[1] = -1, n
            return (bi, k, base + o, cl + 8)
        with concurrent.futures.ThreadPoolExecutor(max_workers=threads) as ex:
            res = list(ex.map(work, jobs, chunksize=64))
        # the stored buffers back to back (64-byte aligned) in one pinned arena, batch after batch -- the layout of the plain
        # host copy above; the scratch arena with compressBound-sized slots is dropped
        tight_total = sum((ln + 63) // 64 * 64 for _, _, _, ln in res)
        tight = torch.empty(max(tight_total, 64), dtype=torch.uint8).pin_memory()
        tbase, toff = tight.data_ptr(), 0
        moved = []
        for bi, k, ptr, ln in res:
            C.memmove(tbase + toff, ptr, ln)
            moved.append((bi, k, tbase + toff, ln))
            toff += (ln + 63) // 64 * 64
        del arena
        self.host_keep.append(tight)
        per_batch = {}
        for bi, k, ptr, ln in moved:
            per_batch.setdefault(bi, {})[k] = (ptr, ln)
        self.marshalled_lz4, self.lz4_h2d_bytes, ncomp = [], 0, 0
        for bi, mb in enumerate(self.marshalled):
            bufs = [None] * 16
            for k, c in enumerate(cols):
                ptr, ln = per_batch[bi][k]
                bufs[c] = np.frombuffer((C.c_char * ln).from_address(ptr), dtype=np.uint8)
                self.lz4_h2d_bytes += ln
                ncomp += ln != int(mb.col_lens[k])
            cb = ColumnBatch(num_rows=mb.c.num_rows, columns=bufs, stats=None, batch_id=mb.c.batch_id, bucket_id=mb.c.bucket_id)
            self.marshalled_lz4.append(capi.MarshalledBatch(cb, cols))
        self.lz4_compressed_buffers = ncomp

    def prepare_pageable_copy(self, nbatches):
        """The first `nbatches` batches again in ordinary numpy (pageable) memory."""
        import numpy as np
        from snappydata_b200.column_format import ColumnBatch
        cols = self.desc.table_cols
        self.marshalled_pg, self.pageable_rows = [], 0
        for mb in self.marshalled[:nbatches]:
            bufs = [None] * 16
            for k, c in enumerate(cols):
                n = int(mb.col_lens[k])
                bufs[c] = np.frombuffer((C.c_char * n).from_address(int(mb.col_bufs[k])), dtype=np.uint8).copy()
            cb = ColumnBatch(num_rows=mb.c.num_rows, columns=bufs, stats=None, batch_id=mb.c.batch_id, bucket_id=mb.c.bucket_id)
            self.marshalled_pg.append(self.capi.MarshalledBatch(cb, cols))
            self.pageable_rows += mb.c.num_rows
        self.pg_plan = self.capi.Plan(self.api, self.desc)
        self.pg_plan.set_stream(self.torch.cuda.current_stream().cuda_stream)

    def step_e2e_pageable(self):
        saved, saved_plan = self.marshalled, self.e2e_plan
        self.marshalled, self.e2e_plan = self.marshalled_pg, self.pg_plan
        try:
            return self.step_e2e()
        finally:
            self.marshalled, self.e2e_plan = saved, saved_plan

    def step_e2e_lz4(self):
        saved = self.marshalled
        self.marshalled = self.marshalled_lz4
        try:
            return self.step_e2e()
        finally:
            self.marshalled = saved

    def step_e2e(self):
        p = self.e2e_plan
        p.reset().set_literals(self.lits)
        sub, h = self.api.batch_submit, p.h
        t0 = time.perf_counter()
        for mb in self.marshalled:
            rc = sub(h, C.byref(mb.c))
            if rc:
                self.api.check(rc)
        t1 = time.perf_counter()
        p.finish_raw()
        if os.environ.get("BENCH_DEBUG"):   # where a step's wall time goes: queueing on the host vs waiting for the device
            print(f"[e2e step] submit loop {1e3 * (t1 - t0):.1f} ms, finish {1e3 * (time.perf_counter() - t1):.1f} ms, "
                  f"{len(self.marshalled)} batches", file=sys.stderr)
        self.e2e_launches = p.metrics()["kernelLaunches"]
        return self.exchange_and_merge(p)

    def cpu_baseline(self, seconds):
        """Generated-loop restatement over a bounded sample of this rank's host copy, all host threads."""
        from oracle import oracle
        cores = os.cpu_count() or 1
        nsample = min(len(self.marshalled), max(64, 16 * cores))
        ba = oracle.BatchArray.__new__(oracle.BatchArray)
        ba.m = self.marshalled[:nsample]
        ba.arr = (self.capi.sd_batch * nsample)(*[mb.c for mb in ba.m])
        ba.n = nsample
        rows = sum(mb.c.num_rows for mb in ba.m)
        one = (lambda t: oracle.run_q1(ba, self.lits[0], t)) if self.q1 else (lambda t: oracle.run_q6(ba, self.lits, t))
        cores, cpu_info = pick_threads(one, rows)
        fn = lambda: one(cores)
        res = fn()
        t0 = time.perf_counter()
        reps = 0
        while True:
            res = fn()
            reps += 1
            if time.perf_counter() - t0 > seconds or reps >= 200:
                break
        dt = time.perf_counter() - t0
        return {"value": rows * reps / dt, "unit": "rows/s", "cores": cores, "kind": "port",
                "sample": f"first {nsample} batches ({rows} rows) of rank 0's shard x {reps} passes in {dt:.1f} s",
                "cpus": cpu_info}, res


    # ---- parity at the benchmark's own size: GPU (C-ABI, same host bytes) vs the oracle's generated loops ----------
    def oracle_partials(self, threads):
        """This rank's shard through the oracle's generated-loop layer (CPU): -> (partial rows, rows scanned)."""
        from oracle import oracle
        n = len(self.marshalled)
        ba = oracle.BatchArray.__new__(oracle.BatchArray)
        ba.m = self.marshalled
        ba.arr = (self.capi.sd_batch * max(1, n))(*[mb.c for mb in ba.m])
        ba.n = n
        rows = sum(mb.c.num_rows for mb in ba.m)
        if self.q1:
            return oracle.run_q1(ba, self.lits[0], threads), rows
        total, matched = oracle.run_q6(ba, self.lits, threads)
        return [[total, matched]], rows

    def parity_check(self, gpu_final_rows, threads):
        """Every rank scans ITS host copy with the oracle; partial rows are gathered and merged like the reference's final
        stage (sums add, counts add, avg = sum / count); rank 0 compares with the GPU's final rows over the same bytes:
        integers (COUNT) bit-exact, DOUBLE within 1e-6 relative."""
        import math
        t0 = time.perf_counter()
        if getattr(self, "_oracle_parts", None) is None:
            mine, rows = self.oracle_partials(threads)
            parts, row_counts = [mine], [rows]
            if self.world > 1:
                parts, row_counts = [None] * self.world, [None] * self.world
                self.dist.all_gather_object(parts, mine)
                self.dist.all_gather_object(row_counts, rows)
            self._oracle_parts = (parts, row_counts)
        parts, row_counts = self._oracle_parts
        if self.q1:
            acc = {}
            for part in parts:
                for r in part:
                    k = (r[0], r[1])
                    if k not in acc:
                        acc[k] = list(r[2:])
                    else:
                        a = acc[k]
                        for i, v in enumerate(r[2:]):
                            a[i] += v
            want = []
            for (k0, k1), a in acc.items():
                sq, sp, sdp, sc, aq_s, aq_c, ap_s, ap_c, ad_s, ad_c, cnt = a
                want.append([k0, k1, sq, sp, sdp, sc, aq_s / aq_c, ap_s / ap_c, ad_s / ad_c, cnt])
            nkeys = 2
        else:
            tot, matched = None, 0
            for part in parts:
                t, m = part[0]
                matched += m
                if t is not None:
                    tot = t if tot is None else tot + t
            want = [[tot]]
            nkeys = 0
        got = [list(r) for r in gpu_final_rows]
        key = lambda r: tuple(r[:nkeys])
        got.sort(key=key)
        want.sort(key=key)
        ok = len(got) == len(want)
        max_rel, ints_exact = 0.0, True
        if ok:
            for g, w in zip(got, want):
                if key(g) != key(w) or len(g) != len(w):
                    ok = False
                    break
                for x, y in zip(g[nkeys:], w[nkeys:]):
                    if isinstance(x, float) or isinstance(y, float):
                        if x is None or y is None:
                            ok = ok and x is y
                            continue
                        rel = 0.0 if x == y else abs(x - y) / max(abs(x), abs(y))
                        if math.isnan(rel):
                            ok = ok and math.isnan(x) and math.isnan(y)
                            continue
                        max_rel = max(max_rel, rel)
                    elif x != y:
                        ints_exact = False
        ok = ok and ints_exact and max_rel <= 1e-6
        return {"ok": bool(ok), "rows": int(sum(row_counts)), "groups": len(want), "max_rel_err": max_rel, "counts_exact": bool(ints_exact),
                "tolerance": 1e-6, "oracle_seconds": round(time.perf_counter() - t0, 2),
                "checker": "oracle/scan_oracle.c generated-loop layer on the host cores over the same ColumnBatch bytes (every rank its shard, "
                           "partials merged); GPU side = the e2e step through sd_batch_submit over exactly those bytes, after the exchange",
                "gpu": [[x.decode() if isinstance(x, bytes) else x for x in r] for r in got[:8]],
                "oracle": [[x.decode() if isinstance(x, bytes) else x for x in r] for r in want[:8]]}


def timed_steps(torch, dist, world, fn, warmup, steps):
    for _ in range(warmup):
        fn()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if os.environ.get("BENCH_DEBUG"):
        sys.stderr.write(f"[rank {int(os.environ.get('RANK', '0'))}] {steps} steps in {ms:.3f} ms\n")
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        dist.barrier()
    return ms


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus or world == 1 and args.gpus == 1, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torchrun)"
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from snappydata_b200 import capi
    api = capi.product_api()
    api.check(api.init(local_rank))

    comm = None
    if world > 1:   # sd_comm: NCCL inside libsnappygpu.so; torch.distributed only carries rank 0's 128-byte id
        def bcast(b):
            box = [b]
            dist.broadcast_object_list(box, src=0)
            return box[0]
        comm = capi.Comm(api, rank, world, local_rank, bcast)

    if args.workload in ("c4", "c5"):   # BASELINE.json configs[3] / [4] alone
        from snappydata_b200 import workloads
        peak, peak_src = measured_peak_gbs()
        if args.workload == "c4":
            r = workloads.run_c4(api, torch, dist, rank, world, local_rank, args.steps, args.warmup, peak)
        else:
            assert world == 1, "C5 is a 1-GPU configuration (BASELINE.json configs[4])"
            r = workloads.run_c5(api, torch, local_rank, args.steps, args.warmup, peak)
        if rank == 0:
            line = {"metric": "rows/sec, " + r["workload"], "value": r["value"], "unit": "rows/s", "n_gpus": world, "steps": r["steps"],
                    "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                    "dtype": "i32/f64/u8", "data": "synthetic", "config": {"workload": r["workload"]}, "gpu_launches": r["steps"]}
            line.update({k: v for k, v in r.items() if k not in line})
            print(json.dumps(line))
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        if not r["parity_check"]["ok"]:
            sys.exit("parity_check failed (see the JSON line)")
        return

    q1 = args.workload == "q1"
    total = args.rows or (SF100_ROWS if q1 else SF10_ROWS)
    main_run = QueryRun(api, torch, dist, q1, total, rank, world, local_rank, args.scaling, comm)
    job_rows = main_run.job_rows   # rows all ranks scan per step

    def job_sum(x):   # sum of a per-rank count over the job
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return int(t.item())

    sampler = ClockSampler(local_rank) if rank == 0 and not os.environ.get("BENCH_NO_CLOCKS") else None
    ms = timed_steps(torch, dist, world, main_run.step_resident, args.warmup, args.steps)
    clocks = sampler.stop() if sampler else None
    # per-launch figures over warm-up + timed steps (same kernel, same data every step)
    nsteps_all = args.warmup + args.steps
    kernel_ms = main_run.kernel_ns / 1e6 / max(1, main_run.launches)
    algo_per_launch = main_run.algo_bytes / max(1, main_run.launches)
    launches_timed = main_run.launches * args.steps // nsteps_all
    d2h_step = 0
    final_rows = capi.parse_row_stream(main_run.final_raw, main_run.desc.final_schema())
    if args.dump_outputs and rank == 0:
        dump_final_rows(args.dump_outputs, args.workload, final_rows, main_run.desc)

    out = {"metric": metric_name(q1), "value": job_rows * args.steps / (ms / 1e3), "unit": "rows/s", "n_gpus": world,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
           "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": workload_config(q1, total, world, args.scaling), "gpu_launches": launches_timed, "clocks": clocks}
    peak, peak_src = measured_peak_gbs()
    achieved = algo_per_launch / (kernel_ms / 1e3) / 1e9 if kernel_ms > 0 else 0.0
    tpr = ncu_traffic_per_row(q1)
    out["roofline"] = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                       "traffic": (tpr * main_run.local_rows) if tpr else None,
                       "traffic_source": "profiles/r02_traffic.json (ncu --set full, 200M-row launch) scaled by rows", "peak_source": peak_src, "kernel": "sd::scan_aggregate_kernel<" + main_run.plan.kernel_name() + ">",
                       "kernel_ms_per_launch": kernel_ms, "algorithmic_bytes_per_launch": algo_per_launch,
                       "frac_of_nominal_7700": achieved / 7700.0,
                       "note": "per rank (rank 0); one launch scans the rank's whole shard; `peak` is a measured COPY bandwidth "
                               "(read + write), which a read-only stream like this scan can exceed: frac > 1 is not an error"}
    out["hbm_gbs_whole_job"] = job_rows * (40 if q1 else 28) / (ms / args.steps / 1e3) / 1e9

    threads = cgroup_cpu_limit() or (len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    parity_failed = False

    def run_parity(run, tag, resident_rows):
        """GPU (e2e step over the host copy) vs oracle over the same bytes; plus the resident-store result when it covers the same rows."""
        nonlocal parity_failed
        fs = run.desc.final_schema()
        pc = run.parity_check(capi.parse_row_stream(run.final_raw, fs), threads)
        same_rows = job_sum(1 if run.e2e_rows == run.local_rows else 0) == world
        if same_rows:
            rc = run.parity_check(resident_rows, threads)
            pc["resident_store_result"] = {"ok": rc["ok"], "max_rel_err": rc["max_rel_err"], "counts_exact": rc["counts_exact"]}
            pc["ok"] = pc["ok"] and rc["ok"]
        else:
            pc["resident_store_result"] = None
        pc["workload"] = tag
        parity_failed = parity_failed or not pc["ok"]
        return pc

    if not args.no_e2e or not args.no_parity:
        main_run.prepare_host_copy()
    if not args.no_e2e:
        e_steps = max(1, args.e2e_steps)
        e2e_job_rows = job_sum(main_run.e2e_rows)
        ems = timed_steps(torch, dist, world, main_run.step_e2e, 1, e_steps)
        if not args.no_parity:
            out["parity_check"] = run_parity(main_run, "q1 sf100" if q1 else "q6 sf10", final_rows)
        plain = {"value": e2e_job_rows * e_steps / (ems / 1e3), "unit": "rows/s", "h2d_bytes_per_step": main_run.h2d_bytes,
                 "rows_per_step": e2e_job_rows, "form": "uncompressed column buffers (the state after the reference's first scan "
                 "replaced a stored buffer by its decompressed copy, ColumnFormatEntry.scala:498-600)",
                 "d2h_bytes_per_step": 4096 if world > 1 else 1024, "ms_per_step": ems / e_steps, "steps": e_steps,
                 "gpu_launches_per_step": main_run.e2e_launches,
                 "note": "per-rank bytes; every ColumnBatch of the e2e rows submitted from pinned host memory through sd_batch_submit "
                         "each step (SD_OPT_RETAIN_BUFFERS: buffers stay valid until finish)"
                         + ("" if main_run.e2e_rows == main_run.local_rows else
                            f"; the e2e legs stream the first {main_run.e2e_rows} rows of each rank's partition set "
                            "(bounds pinned host memory to one table across the job; the rate is link-bound and linear in rows)")}
        out["e2e"] = plain
        # the reference's real ownership rule and ordinary (pageable) memory: what a JVM caller with heap buffers gets
        pg_batches = min(len(main_run.marshalled), 250)
        main_run.prepare_pageable_copy(pg_batches)
        pg_rows = job_sum(main_run.pageable_rows)
        pms = timed_steps(torch, dist, world, main_run.step_e2e_pageable, 1, 1)
        out["e2e_pageable_unretained"] = {"value": pg_rows / (pms / 1e3), "unit": "rows/s", "rows_per_step": pg_rows, "ms_per_step": pms,
                                          "note": f"first {pg_batches} batches per rank from ordinary pageable memory, buffers releasable when "
                                                  "sd_batch_submit returns (ColumnBatchIterator.scala:165-184; no SD_OPT_RETAIN_BUFFERS)"}
        if not args.no_lz4:
            main_run.prepare_compressed_copy()
            lms = timed_steps(torch, dist, world, main_run.step_e2e_lz4, 1, e_steps)
            stored = {"value": e2e_job_rows * e_steps / (lms / 1e3), "unit": "rows/s", "h2d_bytes_per_step": main_run.lz4_h2d_bytes,
                      "rows_per_step": e2e_job_rows, "d2h_bytes_per_step": 4096 if world > 1 else 1024,
                      "ms_per_step": lms / e_steps, "steps": e_steps, "compressed_buffers": main_run.lz4_compressed_buffers,
                      "gpu_launches_per_step": main_run.e2e_launches,
                      "form": "STORED form: every buffer >= 2048 B that LZ4 shrinks to <= 75 % is [-1][len][LZ4 block] "
                              "(CompressionUtils.scala:47-61,102-110) -- what the region holds after ingest / when faulted in from disk",
                      "note": "same submit path as e2e_plain; only the compressed bytes cross PCIe and the blocks are expanded on the "
                              "device (sd_lz4.cu), overlapped with the copies"}
            if not args.no_parity:   # the stored-LZ4 leg's result against the same oracle answer
                lp = main_run.parity_check(capi.parse_row_stream(main_run.final_raw, main_run.desc.final_schema()), threads)
                stored["parity_ok"] = lp["ok"]
                stored["max_rel_err"] = lp["max_rel_err"]
                parity_failed = parity_failed or not lp["ok"]
            # headline e2e = the stored form (VERDICT r01 #3); the uncompressed leg is reported beside it
            out["e2e"] = stored
            out["e2e_plain"] = plain
        if rank == 0 and not args.no_cpu:
            cb, res = main_run.cpu_baseline(args.cpu_seconds)
            out["cpu_baseline"] = cb
    elif not args.no_parity:
        main_run.step_e2e()
        out["parity_check"] = run_parity(main_run, "q1 sf100" if q1 else "q6 sf10", final_rows)
    if rank == 0:
        out["result_check"] = {"groups": len(final_rows), "first_row": [x.decode() if isinstance(x, bytes) else x for x in final_rows[0]] if final_rows else None}

    # ---- the other headline query in the same run --------------------------------------------------
    if not args.no_also:
        del main_run
        torch.cuda.empty_cache()
        oq1 = not q1
        ototal = SF100_ROWS if oq1 else SF10_ROWS
        other = QueryRun(api, torch, dist, oq1, ototal, rank, world, local_rank, args.scaling, comm)
        oms = timed_steps(torch, dist, world, other.step_resident, args.warmup, args.steps)
        if args.dump_outputs and rank == 0:
            dump_final_rows(args.dump_outputs, "q1" if oq1 else "q6",
                            capi.parse_row_stream(other.final_raw, other.desc.final_schema()), other.desc)
        okms = other.kernel_ns / 1e6 / max(1, other.launches)
        oalgo = other.algo_bytes / max(1, other.launches)
        out["also"] = {"workload": workload_config(oq1, ototal, world, args.scaling)["workload"], "value": other.job_rows * args.steps / (oms / 1e3),
                       "unit": "rows/s", "ms_per_step": oms / args.steps,
                       "roofline": {"bound": "hbm", "achieved": oalgo / (okms / 1e3) / 1e9 if okms > 0 else 0.0, "peak": peak,
                                    "unit": "GB/s", "frac": (oalgo / (okms / 1e3) / 1e9 / peak) if okms > 0 else 0.0,
                                    "kernel_ms_per_launch": okms}}
        if not args.no_parity:
            ofinal = capi.parse_row_stream(other.final_raw, other.desc.final_schema())
            other.prepare_host_copy()
            other.step_e2e()
            out["also"]["parity_check"] = run_parity(other, "q1 sf100" if oq1 else "q6 sf10", ofinal)
    if not args.no_also and not args.no_extras and q1 and not args.rows:
        # BASELINE.json's other two configurations in the same run, each with its own roofline and parity assertion
        from snappydata_b200 import workloads
        try:
            del other
        except NameError:
            pass
        torch.cuda.empty_cache()
        out["also_c4"] = workloads.run_c4(api, torch, dist, rank, world, local_rank, args.steps, args.warmup, peak)
        parity_failed = parity_failed or not out["also_c4"]["parity_check"]["ok"]
        if world == 1:
            out["also_c5"] = workloads.run_c5(api, torch, local_rank, args.steps, args.warmup, peak)
            parity_failed = parity_failed or not out["also_c5"]["parity_check"]["ok"]
    if comm is not None:
        out["exchange"] = dict(comm.info(), kind="sd_plan_exchange inside libsnappygpu.so: one ncclAllGather per query of every rank's key dictionaries + raw device state (dense plans; partial rows otherwise), merged on every rank")
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if parity_failed:
        sys.exit("parity_check failed: GPU result differs from the oracle beyond the tolerance (see the JSON line)")


if __name__ == "__main__":
    main()
