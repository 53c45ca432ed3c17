"""Runs bench.py's main() with the GPU, the C-ABI library and torch.distributed replaced by stand-ins, so that the
host-side logic of the bench (sharding modes, per-job row accounting, the JSON line) is exercised without a GPU.
usage: python bench_mock.py WORLD weak|strong [bench.py arguments]   (driven by tests/test_bench_line.py)"""
import sys, types, importlib.util, ctypes as C, json
ROOT = __import__('os').path.dirname(__import__('os').path.dirname(__import__('os').path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
# ---- fake torch.cuda bits
class FakeEvent:
    def __init__(self, enable_timing=True): pass
    def record(self): pass
    def elapsed_time(self, o): return 5.0
class FakeStream: cuda_stream = 0
torch.cuda.is_available = lambda: True
torch.cuda.set_device = lambda d: None
torch.cuda.synchronize = lambda: None
torch.cuda.Event = FakeEvent
torch.cuda.current_stream = lambda: FakeStream()
torch.cuda.empty_cache = lambda: None
_orig_empty = torch.empty
class T(torch.Tensor): pass
def pin(self): return self
torch.Tensor.pin_memory = pin
# ---- fake capi
from snappydata_b200 import capi, lineitem, plan as P
class FakeLib:
    def sdx_store_get_buffer(self, h, i, c, out, cap, ln):
        ln._obj.value = 1000 if hasattr(ln, '_obj') else 0
        return 0
class FakeApi:
    lib = FakeLib()
    def check(self, rc): assert rc == 0
    def init(self, d): return 0
    def batch_submit(self, h, b): return 0
    def plan_metrics(self, h, m):
        m[6], m[7], m[9] = 3_500_000, 1, 24_000_000_000
        return 0
class FakeStore:
    def __init__(self, api, schema, device=0): self.h = 0; self.n = 0
    def gen_lineitem(self, first_row, nrows, rpb, nb, seed, mask):
        self.first_row, self.nrows, self.rpb = first_row, nrows, rpb
        assert first_row % rpb == 0
    def num_batches(self): return (self.nrows + self.rpb - 1) // self.rpb
    def batch_info(self, i):
        n = min(self.rpb, self.nrows - i * self.rpb); return n, i % 8, self.first_row // self.rpb + i
class FakePlan:
    def __init__(self, api, desc): self.h = 0; self.desc = desc
    def set_stream(self, s): return self
    def set_option(self, o, v): return self
    def reset(self): return self
    def set_literals(self, l): return self
    def scan_store(self, s): return self
    def finish_raw(self): return b""
    def literal_array(self, vals): return None
    def execute_store_raw(self, store, lit_array, nlits, comm=None): return b""
    def execute_store_view(self, store, lit_array, nlits, comm=None): return memoryview(b"")
    def exchange(self, comm): return self
    def metrics(self): return {"kernelLaunches": 1, "aggTimeNs": 3_500_000, "algorithmicBytes": 24_000_000_000}
    def final_merge_raw(self, raw): return b""
    def kernel_name(self): return "aot:Plan_x"
class FakeComm:
    def __init__(self, api, rank, world, device, bcast): self.h = 0; assert len(bcast(b"x" * 128)) == 128
    def info(self): return {"world": WORLD, "slot_bytes": 2048, "all_gathers": 1, "regrows": 0}
capi.Comm = FakeComm
capi.product_api = lambda: FakeApi()
capi.Store = FakeStore
capi.Plan = FakePlan
capi.parse_row_stream = lambda raw, schema: [[b"N" if t == capi.SqlType.STRING else 1.0 for t in schema]]
class FakeMB:
    def __init__(self, cb, cols):
        self.c = capi.sd_batch(); self.c.num_rows = cb.num_rows; self.c.batch_id = cb.batch_id; self.c.bucket_id = cb.bucket_id
        self.col_lens = [1000] * len(cols); self.col_bufs = [0] * len(cols)
capi.MarshalledBatch = FakeMB
spec = importlib.util.spec_from_file_location("bench", __import__("os").path.join(ROOT, "bench.py")); b = importlib.util.module_from_spec(spec); spec.loader.exec_module(b)
# C.byref(ln) -> our fake lib reads ._obj
b.QueryRun.cpu_baseline = lambda self, s: ({"value": 1.0, "unit": "rows/s", "cores": 1, "kind": "port", "sample": "mock"}, None)
b.QueryRun.parity_check = lambda self, rows, threads: {"ok": True, "rows": self.e2e_rows, "groups": 0, "max_rel_err": 0.0, "counts_exact": True}
b.QueryRun.prepare_pageable_copy = lambda self, n: (setattr(self, 'marshalled_pg', self.marshalled[:n]), setattr(self, 'pageable_rows', sum(m.c.num_rows for m in self.marshalled[:n])), setattr(self, 'pg_plan', self.e2e_plan))
b.QueryRun.prepare_compressed_copy = lambda self, threads=32: (setattr(self, 'marshalled_lz4', self.marshalled), setattr(self, 'lz4_h2d_bytes', 1), setattr(self, 'lz4_compressed_buffers', 0))
import os
os.environ["BENCH_NO_CLOCKS"] = "1"
WORLD = int(sys.argv[1]); SCALING = sys.argv[2]
os.environ["WORLD_SIZE"] = str(WORLD); os.environ["RANK"] = str(WORLD - 1); os.environ["LOCAL_RANK"] = str(WORLD - 1)
import torch.distributed as dist
dist.init_process_group = lambda *a, **k: None
dist.barrier = lambda: None
dist.all_reduce = lambda t, op=None: t.mul_(WORLD) if op == dist.ReduceOp.SUM else t
dist.destroy_process_group = lambda: None
dist.broadcast_object_list = lambda box, src=0: None
_tt = torch.tensor
torch.tensor = lambda data, dtype=None, device=None: _tt(data, dtype=dtype)
import snappydata_b200.exchange as ex
class FakeEx:
    def __init__(self, *a): pass
    def all_gather(self, raw): return raw + raw
ex.PartialRowExchange = FakeEx
_print = print

sys.argv = ["bench.py", "--gpus", str(WORLD), "--scaling", SCALING, "--rows", "1000001", "--steps", "2", "--warmup", "1"] + sys.argv[3:]
b.main()   # last rank: prints nothing unless WORLD == 1
os.environ['RANK'] = '0'; os.environ['LOCAL_RANK'] = '0'
if WORLD > 1:
    b.main()   # rank 0: the JSON line
