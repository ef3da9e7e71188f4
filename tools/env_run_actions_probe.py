#!/usr/bin/env python
"""Cost of an action schedule and per-step traces in the on-chip env run.  Prints one JSON line.

    python tools/env_run_actions_probe.py [--envs 4096] [--side 128] [--repeats 5] [--out profiles/r04_env_run_actions_probe.json]

For k in {8, 64} and the base and decay dead-cell rules it times, alternating in one process, microseconds per step of
  run           run(k): plain steps, no trace (the code run() ran before schedules existed);
  run_reward    run(k, reward_trace=...);
  run_actions   run(k, actions=..., reward_trace=..., alive_trace=...);
  step_seq      k chained single steps with the same actions through StepSequence, which records no trace
                (base rule only: StepSequence implements the base env);
  step_loop     for t in range(k): step(actions[t], reward_out=trace[t]);
and reports the median and the spread (min, max) over the repeats.  Every variant is warmed up first.  Check: the
reward trace of run_actions equals the one of step_loop from the same start."""
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
ap.add_argument("--envs", type=int, default=4096)
ap.add_argument("--side", type=int, default=128)
ap.add_argument("--repeats", type=int, default=5)
ap.add_argument("--out", default="")
a = ap.parse_args()

if not torch.cuda.is_available():
    sys.exit("env_run_actions_probe.py needs a GPU")
torch.cuda.set_device(0)
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
B, side = a.envs, a.side
result = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "envs": B, "side": side,
          "repeats": a.repeats, "cases": []}


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
    env = BatchedSim(B, side, seed=1, spawnStabilityFactor=-2, stableStabilityFactor=2, rng="device", **kw)
    for k in (8, 64):
        g = torch.Generator(device="cuda").manual_seed(k)
        acts = torch.randint(0, side * side + 1, (k, B), dtype=torch.int32, device="cuda", generator=g)
        rtr = torch.zeros((k, B), dtype=torch.int32, device="cuda")
        atr = torch.zeros_like(rtr)
        loop_tr = torch.zeros_like(rtr)
        seq = StepSequence([env], acts) if rule == "zero" else None

        def step_loop():
            for t in range(k):
                env.step(acts[t], reward_out=loop_tr[t])

        variants = {"run": lambda: env.run(k), "run_reward": lambda: env.run(k, reward_trace=rtr),
                    "run_actions": lambda: env.run(k, actions=acts, reward_trace=rtr, alive_trace=atr),
                    "step_seq": (lambda: seq.run(k)) if seq is not None else None, "step_loop": step_loop}
        variants = {n: f for n, f in variants.items() if f is not None}
        # check: one schedule from the same start through run and through the step loop
        env.reset()
        env.run(k, actions=acts, reward_trace=rtr, alive_trace=atr)
        env.reset()
        step_loop()
        torch.cuda.synchronize()
        same = bool(torch.equal(rtr, loop_tr))
        ok_all &= same
        env.check_actions()
        for f in variants.values():                         # warm-up
            f()
        times = {n: [] for n in variants}
        for _ in range(a.repeats):
            for n, f in variants.items():
                times[n].append(timed(f) / k)
        case = {"rule": rule, "k": k, "trace_equals_step_loop": same,
                "us_per_step": {n: stats(v) for n, v in times.items()}}
        med = {n: case["us_per_step"][n]["median"] for n in times}
        case["run_actions_over_run"] = round(med["run_actions"] / med["run"], 3)
        if "step_seq" in med:
            case["run_actions_over_step_seq"] = round(med["run_actions"] / med["step_seq"], 3)
        result["cases"].append(case)
        del seq

result["ok"] = ok_all
line = json.dumps(result)
print(line)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")
sys.exit(0 if ok_all else 1)
