#!/usr/bin/env python
"""Go/no-go probe for hardware-compressed env state planes.  Writes one JSON file.

    python tools/compressible_probe.py [--regions 9] [--out profiles/r08_compressible_probe.json]

C2 steps (4096 envs x 128^2, base rule, spawn -2 / stable 2) through StepSequence over R rotating replicas, timed as
bench.py times them (one C-ABI call per region, CUDA events recorded by the library around the launches), for three
arms built from the same seeds and actions:
  plain         every plane in plain torch memory
  stable        the int8 stability plane in compressed memory (cuMemCreate, CU_MEM_ALLOCATION_COMP_GENERIC)
  world_stable  the stability plane and both bit planes of the world in compressed memory
The arms are stepped region by region in turn, so they see the same world ages and the same machine state; after the
last region their planes are compared byte for byte.  Cases:
  soup      Bernoulli(0.5) soups aged as bench.py ages them (warm-up, two untimed regions), regions of 20 and of 200
            steps, at R = 4 (the bench: 320 MiB touched, > 126 MB L2) and R = 16 (1.25 GiB: cannot fit the L2 even
            compressed, so a gain there is DRAM bandwidth, not L2 capacity)
  random    every plane refilled with uniform random bytes before each region (incompressible input), regions of R
            steps (each replica stepped once, reading random bytes): the worst case
Per case and arm: median / min / max of the region times in microseconds per step.  The card's name, power limit and
SM clock are read in the same command; the library reports the compression each plane received."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "ecen743-project-cgol_b200")):
    sys.path.insert(0, p)
import torch  # noqa: E402
from cgl_b200 import native  # noqa: E402
from cgl_b200.batched import BatchedSim, StepSequence  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--regions", type=int, default=9)
ap.add_argument("--out", default="")
a = ap.parse_args()

if not torch.cuda.is_available():
    sys.exit("compressible_probe.py needs a GPU")
torch.cuda.set_device(0)
dev = torch.device("cuda", 0)
B, SIDE = 4096, 128
ARMS = {"plain": (), "stable": ("stable",), "world_stable": ("world", "stable")}


def smi():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                       text=True)
    return r.stdout.strip()


lib = native.load()
result = {"device": torch.cuda.get_device_name(0), "nvidia_smi_before": smi(),
          "query": "name, power.limit, clocks.sm, clocks.max.sm", "regions": a.regions,
          "compressible_granularity_bytes": int(lib.cgl_state_granularity(0)),
          "granularity_note": "0 = CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED unset (or no driver entry point)",
          "cases": []}


def stats(xs):
    xs = sorted(xs)
    return {"median": round(xs[len(xs) // 2], 3), "min": round(xs[0], 3), "max": round(xs[-1], 3)}


def make_arm(planes, R):
    sims = [BatchedSim(B, SIDE, seed=r * B, spawnStabilityFactor=-2, stableStabilityFactor=2, device=dev, rng="device",
                       _compressed_planes=planes) for r in range(R)]
    g = torch.Generator(device=dev)
    g.manual_seed(10 ** 6)
    actions = torch.randint(0, SIDE * SIDE + 1, (16, B), dtype=torch.int32, device=dev, generator=g)
    return sims, StepSequence(sims, actions)


def randomize(sims, seed):
    g = torch.Generator(device=dev)
    for i, s in enumerate(sims):
        g.manual_seed(seed * 1000 + i)
        s.stable.copy_(torch.randint(-128, 128, s.stable.shape, dtype=torch.int8, device=dev, generator=g))
        for w in (s._wa, s._wb):
            w.copy_(torch.randint(-2 ** 31, 2 ** 31 - 1, w.shape, dtype=torch.int32, device=dev, generator=g))


def run_case(name, R, K, warmup, random_planes):
    arms = {k: make_arm(v, R) for k, v in ARMS.items()}
    issues, events = {}, {}
    for k, (sims, seq) in arms.items():
        seq.run(warmup)
        events[k] = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        issues[k] = seq.prepare(K, events=events[k])
        if not random_planes:
            issues[k](); issues[k]()                        # as bench.py: two untimed regions
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for rep in range(a.regions):
        for k, (sims, seq) in arms.items():
            if random_planes:
                randomize(sims, rep)
            torch.cuda.synchronize()
            issues[k]()
            torch.cuda.synchronize()
            times[k].append(events[k][0].elapsed_time(events[k][1]) * 1e3 / K)
    ref = arms["plain"][0]
    identical = all(torch.equal(s.stable, r.stable) and torch.equal(s._wa, r._wa) and torch.equal(s._reward, r._reward)
                    for k, (sims, _) in arms.items() for s, r in zip(sims, ref))
    out = {"case": name, "replicas": R, "steps_per_region": K,
           "generations_per_replica_at_end": arms["plain"][0][0].count,
           "us_per_step": {k: stats(v) for k, v in times.items()},
           "compressed": {k: arms[k][0][0].compressed_planes() for k in arms},
           "arms_identical_after_last_region": identical}
    base = out["us_per_step"]["plain"]["median"]
    out["gain_vs_plain"] = {k: round(base / v["median"] - 1, 4) for k, v in out["us_per_step"].items() if k != "plain"}
    print(json.dumps(out), flush=True)
    del arms, issues
    torch.cuda.empty_cache()
    return out


for R in (4, 16):
    for K, W in ((20, 5), (200, 10)):
        result["cases"].append(run_case("soup", R, K, W, False))
    result["cases"].append(run_case("random", R, R, 1, True))
result["nvidia_smi_after"] = smi()
text = json.dumps(result, indent=1)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(text + "\n")
print(text)
