#!/usr/bin/env python
"""Cost and use of stopping on-chip env runs at a short world cycle (cgl_env_run_cycle).  Prints one JSON line.

    python tools/env_run_cycle_probe.py [--repeats 5] [--out profiles/r06_env_run_cycle_probe.json]

1. Per-step overhead.  At 4096 x 128^2 and 16384 x 64^2, base and decay dead-cell rules, k = 256, every env holds a
   lone glider on an empty torus.  Its world repeats only after 4 * side >= 256 steps, so no variant stops early and
   each runs all k steps.  Timed in one process, alternating, in microseconds per step: plain run(k),
   run(k, until_fixed=True) and run(k, max_period=P) for P = 1, 2, 8.  Reports the median and the spread (min, max)
   over the repeats, after a warm-up of every variant.
2. Use case.  4096 random 64^2 soups and 1024 random 128^2 soups from the reference RNG (env e starts from
   RandomState(e).randint(2)), with budgets of 4000 and 8000 steps.  Reports the wall time (CUDA events) of
   until_fixed, which runs nearly the whole budget, against max_period=2, and the distribution of steps and period."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "ecen743-project-cgol_b200")):
    sys.path.insert(0, p)
import numpy as np  # noqa: E402
import torch  # noqa: E402
from cgl_b200 import native  # noqa: E402
from cgl_b200.batched import BatchedSim  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--repeats", type=int, default=5)
ap.add_argument("--k", type=int, default=256)
ap.add_argument("--out", default="")
a = ap.parse_args()

if not torch.cuda.is_available():
    sys.exit("env_run_cycle_probe.py needs a GPU")
torch.cuda.set_device(0)
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
result = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "repeats": a.repeats,
          "library": os.path.basename(native.LIB_PATH), "overhead": [], "use_case": []}
GLIDER = [(0, 1), (1, 2), (2, 0), (2, 1), (2, 2)]


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3, out


def stats(xs):
    xs = sorted(xs)
    return {"median": round(xs[len(xs) // 2], 3), "min": round(xs[0], 3), "max": round(xs[-1], 3)}


ok_all = True
k = a.k
for B, side in ((4096, 128), (16384, 64)):
    assert k < 4 * side + 1
    for rule in ("zero", "decay"):
        kw = {} if rule == "zero" else dict(dead_rule="decay", empty=-1, empty_min=-5)
        env = BatchedSim(B, side, seed=1, spawnStabilityFactor=-2, stableStabilityFactor=2, rng="device", **kw)
        cells = torch.zeros((B, side * side), dtype=torch.uint8, device="cuda")
        for r, c in GLIDER:
            cells[:, (r + 3) * side + c + 3] = 1
        env.set_state(cells)
        env.init_stable()
        per = torch.zeros(B, dtype=torch.int32, device="cuda")
        variants = {"run": dict(), "until_fixed": dict(until_fixed=True), "max_period_1": dict(max_period=1),
                    "max_period_2": dict(max_period=2, period_out=per), "max_period_8": dict(max_period=8, period_out=per)}
        full = True
        for v in variants.values():                         # warm-up, and every variant runs all k steps
            _, _, steps = env.run(k, **v)
            full &= bool((steps == k).all()) and not bool(per.any())
        times = {n: [] for n in variants}
        for _ in range(a.repeats):
            for n, v in variants.items():
                dt, (_, _, steps) = timed(lambda: env.run(k, **v))
                full &= bool((steps == k).all())
                times[n].append(dt / k)
        full &= not bool(per.any())
        ok_all &= full
        case = {"envs": B, "side": side, "rule": rule, "k": k, "all_ran_k_steps": full,
                "us_per_step": {n: stats(t) for n, t in times.items()}}
        med = {n: case["us_per_step"][n]["median"] for n in times}
        for n in ("max_period_1", "max_period_2", "max_period_8"):
            case[f"{n}_over_until_fixed"] = round(med[n] / med["until_fixed"], 3)
        case["until_fixed_over_run"] = round(med["until_fixed"] / med["run"], 3)
        result["overhead"].append(case)
        del env, cells
        torch.cuda.empty_cache()


def dist(x):
    x = np.sort(x)
    return {"median": int(x[len(x) // 2]), "p90": int(x[int(len(x) * 0.9)]), "max": int(x[-1])}


for B, side, budget in ((4096, 64, 4000), (1024, 128, 8000)):
    mk = lambda: BatchedSim(B, side, seed=0, spawnStabilityFactor=-1, stableStabilityFactor=1)  # noqa: E731
    fixed, cyc = mk(), mk()
    per = torch.zeros(B, dtype=torch.int32, device="cuda")
    t_fixed, (_, _, s_fixed) = timed(lambda: fixed.run(budget, until_fixed=True))
    t_cyc, (_, _, s_cyc) = timed(lambda: cyc.run(budget, max_period=2, period_out=per))
    s_fixed, s_cyc, p = s_fixed.cpu().numpy(), s_cyc.cpu().numpy(), per.cpu().numpy()
    settled = s_cyc[p > 0]
    result["use_case"].append({
        "envs": B, "side": side, "budget": budget, "until_fixed_ms": round(t_fixed / 1e3, 3),
        "max_period_2_ms": round(t_cyc / 1e3, 3), "speedup": round(t_fixed / t_cyc, 2),
        "until_fixed_stopped_early": int((s_fixed < budget).sum()),
        "until_fixed_steps": dist(s_fixed),
        "period_counts": {str(q): int((p == q).sum()) for q in range(3)},
        "max_period_2_steps": dist(s_cyc), "settled_steps": dist(settled) if settled.size else None})
    # a period-1 stop of max_period=2 is the fixed point until_fixed finds
    ok_all &= bool((s_fixed[p == 1] == s_cyc[p == 1]).all())
    del fixed, cyc
    torch.cuda.empty_cache()

result["ok"] = ok_all
line = json.dumps(result)
print(line)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")
sys.exit(0 if ok_all else 1)
