#!/usr/bin/env python
"""Cost of the one-step lookahead (cgl_env_action_rewards) against the plain env step.  Prints one JSON line.

    python tools/action_rewards_probe.py [--repeats 7] [--iters 20] [--out profiles/r07_action_rewards_probe.json]

At 4096 x 128^2, 16384 x 64^2 and 1024 x 200^2 (a side that is not fused), base rule, reference soups, in microseconds
per call (CUDA events around `iters` back-to-back calls, median and spread over the repeats, after a warm-up):
  map        BatchedSim.action_rewards(out=...): the int32 [B, size + 1] map
  best       BatchedSim.greedy_actions(out=..., reward_out=...): greedy action and reward only, no map
  step       BatchedSim.step(None): the plain step
  greedy     greedy_actions followed by step(actions): one greedy rollout step
Every call rotates over three env batches, so the working set (>= 225 MB) does not fit the 126 MB L2.  Map mode is also
reported against the HBM roofline for its algorithmic traffic, 1.125 B read per cell + 4 B written per action, at the
project's measured 6543 GB/s.  The card's name and power limit are read in the same command."""
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
from cgl_b200.batched import BatchedSim  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--repeats", type=int, default=7)
ap.add_argument("--iters", type=int, default=20)
ap.add_argument("--out", default="")
a = ap.parse_args()

if not torch.cuda.is_available():
    sys.exit("action_rewards_probe.py needs a GPU")
torch.cuda.set_device(0)
dev = torch.device("cuda", 0)
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
HBM_GBS = 6543.0
result = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "repeats": a.repeats,
          "iters": a.iters, "library": os.path.basename(native.LIB_PATH), "hbm_gbs_measured": HBM_GBS, "shapes": []}


def stats(xs):
    xs = sorted(xs)
    return {"median": round(xs[len(xs) // 2], 3), "min": round(xs[0], 3), "max": round(xs[-1], 3)}


def per_call(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters


for B, side in ((4096, 128), (16384, 64), (1024, 200)):
    size = side * side
    envs = [BatchedSim(B, side, seed=1000 * r, spawnStabilityFactor=-2, stableStabilityFactor=2, device=dev, rng="device")
            for r in range(3)]
    maps = [torch.empty((B, size + 1), dtype=torch.int32, device=dev) for _ in range(3)]
    acts = [torch.empty(B, dtype=torch.int32, device=dev) for _ in range(3)]
    rews = [torch.empty(B, dtype=torch.int32, device=dev) for _ in range(3)]

    def f_map(i):
        envs[i % 3].action_rewards(out=maps[i % 3])

    def f_best(i):
        envs[i % 3].greedy_actions(out=acts[i % 3], reward_out=rews[i % 3])

    def f_step(i):
        envs[i % 3].step(None)

    def f_greedy(i):
        env = envs[i % 3]
        act, _ = env.greedy_actions(out=acts[i % 3], reward_out=rews[i % 3])
        env.step(act)

    fns = {"map": f_map, "best": f_best, "step": f_step, "greedy": f_greedy}
    for fn in fns.values():                                 # warm-up of every variant
        per_call(fn, 6)
    times = {k: [] for k in fns}
    for _ in range(a.repeats):
        for k, fn in fns.items():                           # alternating
            times[k].append(per_call(fn, a.iters))
    # the map of the last call agrees with its own greedy action (cheap self-check of what was timed)
    m = envs[0].action_rewards(out=maps[0])
    ba, br = envs[0].greedy_actions()
    consistent = bool(torch.equal(ba.long(), m.argmax(1)) and torch.equal(br, m.max(1).values))
    row = {"n_envs": B, "side": side, "fused": bool(envs[0].fused), "us": {k: stats(v) for k, v in times.items()},
           "consistent": consistent}
    med = {k: row["us"][k]["median"] for k in times}
    map_bytes = B * size * 1.125 + B * (size + 1) * 4
    row["map_bytes"] = int(map_bytes)
    row["map_roofline_fraction"] = round(map_bytes / (HBM_GBS * 1e3) / med["map"], 3)
    row["best_over_step"] = round(med["best"] / med["step"], 3)
    row["greedy_over_step"] = round(med["greedy"] / med["step"], 3)
    row["decision_by_stepping_us_estimate"] = round((size + 1) * med["step"], 1)
    result["shapes"].append(row)
    del envs, maps

line = json.dumps(result)
print(line)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")
