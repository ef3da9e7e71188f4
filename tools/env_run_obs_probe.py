#!/usr/bin/env python
"""Cost of recording every step's observation in the on-chip env run.  Prints one JSON line.

    python tools/env_run_obs_probe.py [--envs 4096] [--side 128] [--repeats 5] [--out profiles/r05_env_run_obs_probe.json]

For k in {8, 64} and the base and decay dead-cell rules it times, alternating in one process, microseconds per step of
  run           run(k): plain steps, no trace;
  run_actions   run(k, actions=..., reward_trace=...);
  run_obs       run(k, actions=..., reward_trace=..., obs_trace=...): the same plus the observation of every step;
  ring_step     k calls of TrajectoryReplay.step(actions[t]), i.e. step(actions[t], obs_out=, reward_out=);
  ring_run      TrajectoryReplay.run(actions), which records the same k ring steps through run(obs_trace=);
and reports the median and the spread (min, max) over the repeats.  Every variant is warmed up first.  The two rings
hold 2k + 1 slots each, so ring_run splits into two runs whenever its slots wrap the ring end.

The observation planes are 1 byte per cell per step: run_obs writes envs * side^2 bytes per step, which the probe
reports as a rate and as a fraction of 6543.4 GB/s, the HBM figure bench.py uses.  Checks: the obs trace of run_obs
equals the planes of a step(obs_out=) loop from the same start, and after the timed calls both rings are identical."""
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
from cgl_b200.dqn import TrajectoryReplay  # noqa: E402

HBM_GBPS = 6543.4

ap = argparse.ArgumentParser()
ap.add_argument("--envs", type=int, default=4096)
ap.add_argument("--side", type=int, default=128)
ap.add_argument("--repeats", type=int, default=5)
ap.add_argument("--ks", default="8,64")
ap.add_argument("--out", default="")
a = ap.parse_args()

if not torch.cuda.is_available():
    sys.exit("env_run_obs_probe.py needs a GPU")
torch.cuda.set_device(0)
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
B, side = a.envs, a.side
size = side * side
result = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "envs": B, "side": side,
          "repeats": a.repeats, "library": os.path.basename(native.LIB_PATH), "hbm_gbps": HBM_GBPS, "cases": []}


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3


def stats(xs):
    xs = sorted(xs)
    return {"median": round(xs[len(xs) // 2], 3), "min": round(xs[0], 3), "max": round(xs[-1], 3)}


ok_all = True
for rule in ("zero", "decay"):
    kw = {} if rule == "zero" else dict(dead_rule="decay", empty=-1, empty_min=-5)
    for k in (int(x) for x in a.ks.split(",")):
        mk = lambda: BatchedSim(B, side, seed=1, spawnStabilityFactor=-2, stableStabilityFactor=2,  # noqa: E731
                                rng="device", **kw)
        env = mk()
        g = torch.Generator(device="cuda").manual_seed(k)
        acts = torch.randint(0, size + 1, (k, B), dtype=torch.int32, device="cuda", generator=g)
        rtr = torch.zeros((k, B), dtype=torch.int32, device="cuda")
        traces = [torch.empty((k, B, size), dtype=torch.int8, device="cuda") for _ in range(2)]
        plane = env.stable
        turn = [0]

        def run_obs():                                      # each run reads the other trace's last row
            env.run(k, actions=acts, reward_trace=rtr, obs_trace=traces[turn[0]])
            turn[0] ^= 1

        # check: the obs trace against a step(obs_out=) loop from the same start
        env.run(k, actions=acts, reward_trace=rtr, obs_trace=traces[0])
        env.stable = plane
        env.reset()
        for t in range(k):
            env.step(acts[t], obs_out=traces[1][t])
        torch.cuda.synchronize()
        same = bool(torch.equal(traces[0], traces[1]))
        env.stable = plane
        env.reset()
        ring_a = TrajectoryReplay(mk(), max_size=2 * k * B, batch_size=64)
        ring_b = TrajectoryReplay(mk(), max_size=2 * k * B, batch_size=64)

        def ring_step():
            for t in range(k):
                ring_a.step(acts[t])

        variants = {"run": lambda: env.run(k), "run_actions": lambda: env.run(k, actions=acts, reward_trace=rtr),
                    "run_obs": run_obs, "ring_step": ring_step, "ring_run": lambda: ring_b.run(acts)}
        for f in variants.values():                         # warm-up
            f()
        times = {n: [] for n in variants}
        for _ in range(a.repeats):
            for n, f in variants.items():
                times[n].append(timed(f) / k)
        torch.cuda.synchronize()
        same_ring = bool(torch.equal(ring_a.obs, ring_b.obs) and torch.equal(ring_a.action, ring_b.action)
                         and torch.equal(ring_a.reward, ring_b.reward) and ring_a.t == ring_b.t)
        ok_all &= same and same_ring
        env.check_actions()
        case = {"rule": rule, "k": k, "obs_trace_equals_step_loop": same, "ring_run_equals_ring_step": same_ring,
                "ring_slots": ring_a.slots, "us_per_step": {n: stats(v) for n, v in times.items()}}
        med = {n: case["us_per_step"][n]["median"] for n in times}
        case["run_obs_over_ring_step"] = round(med["run_obs"] / med["ring_step"], 3)
        case["run_obs_over_run_actions"] = round(med["run_obs"] / med["run_actions"], 3)
        case["ring_run_over_ring_step"] = round(med["ring_run"] / med["ring_step"], 3)
        gbps = B * size / (med["run_obs"] * 1e-6) / 1e9
        case["run_obs_write_gbps"] = round(gbps, 1)
        case["run_obs_write_fraction_of_hbm"] = round(gbps / HBM_GBPS, 3)
        case["obs_write_floor_us_per_step"] = round(B * size / (HBM_GBPS * 1e9) * 1e6, 2)
        result["cases"].append(case)
        del ring_a, ring_b, traces, env
        torch.cuda.empty_cache()

result["ok"] = ok_all
line = json.dumps(result)
print(line)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")
sys.exit(0 if ok_all else 1)
