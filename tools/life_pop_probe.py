#!/usr/bin/env python
"""Cost of recording the population in k-blocked life runs.  Prints one JSON line.

    python tools/life_pop_probe.py [--gens 1000] [--repeats 3] [--out profiles/r03_life_pop_probe.json]

For each shape (65536^2 and 32768^2 tori, one band of the 8-GPU C4 run: 8320 x 65536 with open rows) and
K in {4, 8, 16}, it times, alternating in one process, microseconds per generation of
  run      cgl_life_run (no trace),
  run_pop  cgl_life_run_pop (trace of the owned rows: all rows of a torus, [64, 8256) of the band),
  step1    what a caller can do without cgl_life_run_pop: cgl_life_step(..., alive_out) once per generation,
and reports the median and the spread (min, max) over the repeats.  Every shape and K is tuned once (cgl_life_tune)
and warmed up first.  Checks: the three final grids agree (the band on rows at least `gens` from its open edges), and
on the tori the trace of run_pop equals the k = 1 counts generation by generation."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "ecen743-project-cgol_b200")):
    sys.path.insert(0, p)
import torch  # noqa: E402
from cgl_b200 import native  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--gens", type=int, default=1000)
ap.add_argument("--repeats", type=int, default=3)
ap.add_argument("--ks", default="4,8,16")
ap.add_argument("--out", default="")
a = ap.parse_args()

lib = native.load()
torch.cuda.set_device(0)
st = native.current_stream()
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
result = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "gens": a.gens,
          "repeats": a.repeats, "shapes": []}


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    native.check_alarm()
    return e0.elapsed_time(e1) * 1e3, out


def stats(xs):
    xs = sorted(xs)
    return {"median": round(xs[len(xs) // 2], 2), "min": round(xs[0], 2), "max": round(xs[-1], 2)}


ok_all = True
for name, rows, cols, wrap, win in (("torus_65536", 65536, 65536, 1, (0, 65536)),
                                    ("torus_32768", 32768, 32768, 1, (0, 32768)),
                                    ("band_8gpu_c4", 8320, 65536, 0, (64, 8192))):
    W = cols // 32
    src = torch.empty(rows * W, dtype=torch.int32, device="cuda")
    g = torch.Generator(device="cuda")
    g.manual_seed(rows)
    src.copy_(torch.randint(-2 ** 31, 2 ** 31 - 1, (rows * W,), dtype=torch.int32, device="cuda", generator=g))
    a_buf, b_buf = torch.empty_like(src), torch.empty_like(src)
    pop = torch.empty(a.gens, dtype=torch.int64, device="cuda")
    alive = torch.empty(a.gens, dtype=torch.int32, device="cuda")
    res = ctypes.c_int(-1)

    def run(k, gens):
        a_buf.copy_(src)
        native.check(lib.cgl_life_run(native.dptr(a_buf), native.dptr(b_buf), rows, cols, wrap, gens, k,
                                      ctypes.byref(res), st), "cgl_life_run")
        return a_buf if res.value == 1 else b_buf

    def run_pop(k, gens):
        a_buf.copy_(src)
        native.check(lib.cgl_life_run_pop(native.dptr(a_buf), native.dptr(b_buf), rows, cols, wrap, gens, k, win[0],
                                          win[1], native.dptr(pop), ctypes.byref(res), st), "cgl_life_run_pop")
        return a_buf if res.value == 1 else b_buf

    def step1(gens):
        a_buf.copy_(src)
        x, y = a_buf, b_buf
        for i in range(gens):
            native.check(lib.cgl_life_step(native.dptr(x), native.dptr(y), 1, rows, cols, wrap,
                                           native.dptr(alive[i:i + 1]), st), "cgl_life_step")
            x, y = y, x
        return x

    # the buffer copy at the start of each call is timed too: subtract it
    copy_us = min(timed(lambda: a_buf.copy_(src))[0] for _ in range(5))
    shape = {"name": name, "rows": rows, "cols": cols, "wrap_rows": wrap, "window": list(win), "copy_us": round(copy_us, 1),
             "k": {}}
    step1(a.gens)
    for k in [int(x) for x in a.ks.split(",")]:
        native.check(lib.cgl_life_tune(native.dptr(src), native.dptr(b_buf), rows, cols, wrap, k, st), "cgl_life_tune")
        run(k, 16), run_pop(k, 16)
        gens = a.gens
        t_run, t_pop, t_s1 = [], [], []
        for _ in range(a.repeats):
            t, _ = timed(lambda: run(k, gens))
            t_run.append((t - copy_us) / gens)
            g_run = (a_buf if res.value == 1 else b_buf).clone()
            t, _ = timed(lambda: run_pop(k, gens))
            t_pop.append((t - copy_us) / gens)
            g_pop = (a_buf if res.value == 1 else b_buf).clone()
            trace = pop.clone()
            t, out = timed(lambda: step1(gens))
            t_s1.append((t - copy_us) / gens)
            g_s1 = out.clone()
        lo, hi = (0, rows) if wrap else (gens * W, (rows - gens) * W)
        same = bool(torch.equal(g_run[lo:hi], g_pop[lo:hi]) and torch.equal(g_run[lo:hi], g_s1[lo:hi]))
        entry = {"run_us_per_gen": stats(t_run), "run_pop_us_per_gen": stats(t_pop), "step1_count_us_per_gen": stats(t_s1),
                 "pop_over_run": round(stats(t_pop)["median"] / stats(t_run)["median"], 3),
                 "pop_over_step1": round(stats(t_pop)["median"] / stats(t_s1)["median"], 3), "final_grids_equal": same}
        if wrap:
            entry["trace_equals_k1_counts"] = bool(torch.equal(trace, alive.to(torch.int64) & 0xFFFFFFFF))
            same = same and entry["trace_equals_k1_counts"]
        ok_all = ok_all and same
        shape["k"][str(k)] = entry
    result["shapes"].append(shape)
    del src, a_buf, b_buf
    torch.cuda.empty_cache()

result["ok"] = ok_all
line = json.dumps(result)
print(line, flush=True)
if a.out:
    with open(a.out, "w") as f:
        f.write(line + "\n")
sys.exit(0 if ok_all else 1)
