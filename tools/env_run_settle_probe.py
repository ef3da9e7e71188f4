#!/usr/bin/env python
"""Cost and use of stopping on-chip env runs at the first repeated world of any period (cgl_env_run_settle).
Prints one JSON line.

    python tools/env_run_settle_probe.py [--repeats 5] [--out profiles/r09_env_run_settle_probe.json]

1. Worst case.  The lone-glider boards of tools/env_run_cycle_probe.py at k = 256: 4096 x 128^2 and 16384 x 64^2,
   base and decay dead-cell rules.  No env stops before step k (at 64^2 the glider's period 4 * 64 is exactly k, found
   only after 2k world-only generations), so the settle run pays its whole finder: 2k world-only generations, plus
   k generations to rebuild world_lambda where the period is found, then k full steps.  Timed in one process,
   alternating, in microseconds per budget step: plain run(k), until_fixed, max_period=8 and until_settled.  Median
   and spread (min, max) over the repeats, after a warm-up of every variant.
2. Use case.  The soups of tools/env_run_cycle_probe.py: 4096 x 64^2 with a budget of 4000 steps and 1024 x 128^2 with
   8000 (env e starts from RandomState(e).randint(2), as the reference seeds its worlds).  Wall time (CUDA events) of
   until_fixed, max_period=8 and until_settled; envs by period class; steps to stop.  Every env with period <= 8 must
   equal max_period=8 in steps, period, world and plane.  A sample of envs, among them every class, is checked
   against a CPU brute force that keeps every past world: the same (steps, period), and period 0 only where
   mu + lambda exceeds the budget."""
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
from oracle import oracle  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--repeats", type=int, default=5)
ap.add_argument("--k", type=int, default=256)
ap.add_argument("--sample", type=int, default=24, help="envs per soup workload checked by brute force")
ap.add_argument("--out", default="")
a = ap.parse_args()

if not torch.cuda.is_available():
    sys.exit("env_run_settle_probe.py needs a GPU")
torch.cuda.set_device(0)
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
result = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "repeats": a.repeats,
          "library": os.path.basename(native.LIB_PATH), "worst_case": [], "use_case": []}
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
    for rule in ("zero", "decay"):
        kw = {} if rule == "zero" else dict(dead_rule="decay", empty=-1, empty_min=-5)
        env = BatchedSim(B, side, seed=1, spawnStabilityFactor=-2, stableStabilityFactor=2, rng="device", **kw)
        cells = torch.zeros((B, side * side), dtype=torch.uint8, device="cuda")
        for r, c in GLIDER:
            cells[:, (r + 3) * side + c + 3] = 1
        env.set_state(cells)
        env.init_stable()
        per = torch.zeros(B, dtype=torch.int32, device="cuda")
        variants = {"run": dict(), "until_fixed": dict(until_fixed=True), "max_period_8": dict(max_period=8),
                    "until_settled": dict(until_settled=True, period_out=per)}
        full = True
        for v in variants.values():                         # warm-up, and every variant runs all k steps
            _, _, steps = env.run(k, **v)
            full &= bool((steps == k).all())
        want_p = 4 * side if 4 * side <= k else 0
        full &= bool((per == want_p).all())
        times = {n: [] for n in variants}
        for _ in range(a.repeats):
            for n, v in variants.items():
                dt, (_, _, steps) = timed(lambda: env.run(k, **v))
                full &= bool((steps == k).all())
                times[n].append(dt / k)
        ok_all &= full
        case = {"envs": B, "side": side, "rule": rule, "k": k, "glider_period": 4 * side, "reported_period": want_p,
                "all_ran_k_steps": full, "us_per_step": {n: stats(t) for n, t in times.items()}}
        med = {n: case["us_per_step"][n]["median"] for n in times}
        case["until_settled_over_until_fixed"] = round(med["until_settled"] / med["until_fixed"], 3)
        case["until_settled_over_max_period_8"] = round(med["until_settled"] / med["max_period_8"], 3)
        # the finder's share: the settle run less one full until_fixed pass, per world-only generation it ran
        gens = 3 * k if want_p else 2 * k
        case["finder_world_only_generations"] = gens
        case["finder_us_per_generation"] = round((med["until_settled"] - med["until_fixed"]) * k / gens, 3)
        result["worst_case"].append(case)
        del env, cells
        torch.cuda.empty_cache()


def dist(x):
    x = np.sort(x)
    return {"median": int(x[len(x) // 2]), "p90": int(x[int(len(x) * 0.9)]), "max": int(x[-1])} if x.size else None


def brute_force(world, side, budget):
    seen, w, s = {np.packbits(world).tobytes(): 0}, world.copy(), np.zeros(world.size, np.int8)
    for t in range(1, budget + 1):
        oracle.step_rule(w, s, side, -1, 1, oracle.DEAD_ZERO)
        key = np.packbits(w).tobytes()
        if key in seen:
            return t, t - seen[key]
        seen[key] = t
    return budget, 0


for B, side, budget in ((4096, 64, 4000), (1024, 128, 8000)):
    mk = lambda: BatchedSim(B, side, seed=0, spawnStabilityFactor=-1, stableStabilityFactor=1)  # noqa: E731
    fixed, cyc, settle = mk(), mk(), mk()
    w0 = settle.get_state().cpu().numpy().copy()
    pc = torch.zeros(B, dtype=torch.int32, device="cuda")
    ps = torch.zeros(B, dtype=torch.int32, device="cuda")
    t_fixed, (_, _, s_fixed) = timed(lambda: fixed.run(budget, until_fixed=True))
    t_cyc, (_, _, s_cyc) = timed(lambda: cyc.run(budget, max_period=8, period_out=pc))
    t_set, (_, _, s_set) = timed(lambda: settle.run(budget, until_settled=True, period_out=ps))
    s_cyc, s_set, pc, ps = s_cyc.cpu().numpy(), s_set.cpu().numpy(), pc.cpu().numpy(), ps.cpu().numpy()
    short = (ps >= 1) & (ps <= 8)
    same = bool((s_cyc[short] == s_set[short]).all() and (pc[short] == ps[short]).all()
                and (pc[~short] == 0).all())
    same &= bool(torch.equal(cyc.get_state()[torch.from_numpy(short).cuda()],
                             settle.get_state()[torch.from_numpy(short).cuda()]))
    same &= bool(torch.equal(cyc.stable[torch.from_numpy(short).cuda()], settle.stable[torch.from_numpy(short).cuda()]))
    rs = np.random.RandomState(side)
    classes = [ps == 0, ps == 1, ps == 2, short & (ps > 2), ps > 8]
    sample = sorted({int(rs.choice(np.flatnonzero(c))) for c in classes if c.any()} |
                    {int(e) for e in rs.choice(B, a.sample, replace=False)})
    brute = [(e, tuple(map(int, (s_set[e], ps[e]))), brute_force(w0[e], side, budget)) for e in sample]
    brute_ok = all(g == r for _, g, r in brute)
    ok_all &= same and brute_ok
    result["use_case"].append({
        "envs": B, "side": side, "budget": budget, "until_fixed_ms": round(t_fixed / 1e3, 3),
        "max_period_8_ms": round(t_cyc / 1e3, 3), "until_settled_ms": round(t_set / 1e3, 3),
        "period_classes": {"0": int((ps == 0).sum()), "1": int((ps == 1).sum()), "2": int((ps == 2).sum()),
                           "3-8": int((short & (ps > 2)).sum()), ">8": int((ps > 8).sum())},
        "periods_over_8": {str(q): int((ps == q).sum()) for q in sorted(set(ps[ps > 8].tolist()))},
        "max_period_8_period_0": int((pc == 0).sum()),
        "until_settled_steps": dist(s_set), "settled_steps": dist(s_set[ps > 0]),
        "short_periods_equal_max_period_8": same,
        "brute_force_sample": [{"env": e, "settle": g, "brute_force": r} for e, g, r in brute],
        "brute_force_agrees": brute_ok})
    del fixed, cyc, settle
    torch.cuda.empty_cache()

result["ok"] = ok_all
line = json.dumps(result)
print(line)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")
sys.exit(0 if ok_all else 1)
