"""One 8-GPU band of C4 on one GPU (8192 + 2 x 64 rows x 65536 columns, open rows, no exchange): us per generation of
the launch-per-pass kernel for a given strip length (CGL_TB_ROWS) -- what an 8-GPU rank computes between exchanges."""
import os, sys, json, statistics, ctypes
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "ecen743-project-cgol_b200"))
import torch
from cgl_b200 import native
lib = native.load()
rows, cols = int(os.environ.get("BAND_ROWS", 8320)), 65536
a = torch.randint(-2**31, 2**31 - 1, (rows * cols // 32,), dtype=torch.int32, device="cuda")
b = torch.empty_like(a)
res = ctypes.c_int(0)
k = int(os.environ.get("BAND_K", 8))
def run():
    for _ in range(8):
        native.check(lib.cgl_life_run(native.dptr(a), native.dptr(b), rows, cols, 0, 64, k, ctypes.byref(res), native.current_stream()))
run()
ts = []
for _ in range(5):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); run(); e1.record(); torch.cuda.synchronize()
    ts.append(e0.elapsed_time(e1) / 512 * 1e3)
print(json.dumps({"rpt": os.environ.get("CGL_TB_ROWS"), "k": k, "rows": rows, "us_per_gen": round(statistics.median(ts), 2)}))
