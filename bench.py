#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native Game-of-Life env step.

    python bench.py --gpus N --steps K --warmup W              # our CUDA path (default N=1)
    python bench.py --impl reference --gpus N --steps K ...    # CPU arm: the reference's step on the host cores
    python bench.py --impl reference-gpu --steps K ...         # the reference's OWN CUDA kernel + its 4 PCIe copies
    python bench.py --config c4 --gpus N --steps 1000          # BASELINE configs[3] as the first-class line
    python bench.py --steps K --warmup W --dump-outputs DIR    # also write the last timed step's outputs as .npy
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...   # one rank per GPU (the driver does this)

Default workload (BASELINE.json configs[1], SURVEY.md section 8d "C2"): 4096 envs x 128x128 per GPU, env mode --
per step and env: toggle_state(action) -> generation -> int8 stability update -> reward
(/root/reference/CGL/main.py:64-72).  Weak scaling: every rank owns its own 4096 envs (sharding by env index, no
data-path collective).  A "step" is one launch of the fused kernel over all envs of the rank.

Prints ONE JSON line (rank 0).
  value      G cell-updates/s over all ranks, state resident in HBM.  The K steps of a timed region are issued by ONE
             C-ABI call (cgl_env_step_seq_timed: K launches back to back, the two CUDA events recorded on the stream
             right before the first and after the last launch); the region is bracketed by barrier + synchronize
             on both sides; it is repeated --repeats times and the MEDIAN
             region (max over ranks each) is reported, all of them listed in `regions_ms`.
  e2e        the same metric through the host-driven rollout (cgl_b200.rollout.HostRollout -> cgl_rollout_run):
             every step every env receives its action from pinned host memory (H2D copy inside the timed region)
             and delivers its reward to pinned host memory; a Python policy that reads the previous rewards chooses
             the actions.  Wall clock, max over ranks, median of the repeats; measured for both action paths of the
             API (DMA copy node / kernel loads from pinned memory), the faster one is the headline, both are listed.
  roofline   algorithmic bytes (2.25 B per cell-update) / measured launch time against the measured HBM peak.
  cpu_baseline  the oracle port of the reference's per-cell loop on this box's host cores (N=1 only).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "ecen743-project-cgol_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

SIDE, ENVS_PER_GPU = 128, 4096
SPAWN, STABLE = -2, 2                      # CGL/main.py:29, CGL/bench.py:12-13
BYTES_PER_CELL_ENV = 2.25                  # 1 bit R + 1 bit W + int8 R + int8 W  (SURVEY.md 8d)
BYTES_PER_CELL_LIFE = 0.25
REPLICAS = 4                               # rotating env batches: 4 x 80 MiB touched round-robin > 126 MB L2
E2E_GROUPS = 4                             # env groups of the host-driven rollout (measured: 1 -> 40.2, 2 -> 32.8, 4 -> 29.6, 8 -> 33 us per step)
C4_SIDE, C4_GHOST, C4_KERNEL_K = 65536, 128, 8         # ghost depth measured at 8 GPUs: 64 -> 16.02, 96 -> 16.03, 128 -> 15.81 us per generation
DUMP_ENVS, DUMP_SEED = 256, 0                          # --dump-outputs: 2 planes x 256 envs x 16384 cells x 4 B = 32 MiB


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic(kernel):
    """dram bytes per launch of the dominant kernel from the committed `ncu --set full` capture of this round
    (profiles/traffic.json names the capture it was read from); None if there is none."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            d = json.load(f)
        return d.get(kernel), d.get("_source", {}).get(kernel, "profiles/traffic.json")
    except Exception:  # noqa: BLE001
        return None, None


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:  # noqa: BLE001
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def workload_config(n_gpus):
    """Identical in every arm (ours, reference, reference-gpu): the driver compares the dicts."""
    return {"workload": f"C2: {ENVS_PER_GPU} envs x {SIDE}x{SIDE} per GPU, env mode (toggle + generation + int8 "
                        f"stability + reward), spawn {SPAWN} / stable {STABLE}",
            "envs_per_gpu": ENVS_PER_GPU, "side": SIDE, "total_envs": ENVS_PER_GPU * n_gpus,
            "parallelism": f"env-index sharding x{n_gpus}, no data-path collective",
            "l2": f"GPU arm: inputs larger than L2 -- {REPLICAS} rotating replicas of the env batch "
                  f"({REPLICAS * ENVS_PER_GPU * SIDE * SIDE * 1.25 / 2**20:.0f} MiB touched round-robin > 126 MB L2)"}


def c4_config(n_gpus):
    return {"workload": f"C4: single {C4_SIDE}x{C4_SIDE} torus, life mode (world plane only), row bands over the ranks, "
                        f"ghost depth {C4_GHOST} between halo exchanges, {C4_KERNEL_K} generations per launch",
            "side": C4_SIDE, "ghost_depth": C4_GHOST, "kernel_k": C4_KERNEL_K,
            "parallelism": f"row bands x{n_gpus}, NVLink halo exchange (CUDA-IPC peer stores)" if n_gpus > 1 else
                           "one GPU, plain torus",
            "l2": "inputs larger than L2: 512 MiB per plane"}


# ---------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's per-cell loop (the reference itself is pure Python
# and cannot travel to the GPU box; SURVEY.md section 8c/8d)
# ---------------------------------------------------------------------------------------------
def cpu_arm(steps, warmup, budget_s, exact_steps, threads=None):
    """exact_steps: run exactly `steps` timed steps and shrink the env sample to fit budget_s (the reference arm);
    otherwise keep up to the full batch and cut the step count (the cpu_baseline leg)."""
    from oracle import oracle
    threads = threads or oracle.max_threads()
    size = SIDE * SIDE
    n = 4 * threads
    w = np.stack([oracle.initial_world(SIDE, e) for e in range(n)])
    s = np.stack([oracle.initial_stable(w[e], SPAWN) for e in range(n)])
    rs = np.random.RandomState(10 ** 6)
    oracle.step_batch(w, s, SIDE, rs.randint(size + 1, size=n).astype(np.int32), SPAWN, STABLE, threads)
    t0 = time.perf_counter()
    oracle.step_batch(w, s, SIDE, rs.randint(size + 1, size=n).astype(np.int32), SPAWN, STABLE, threads)
    per_env = (time.perf_counter() - t0) / n
    if exact_steps:
        n_envs = int(max(threads, min(ENVS_PER_GPU, budget_s / (per_env * (steps + warmup)))))
    else:
        n_envs = int(max(threads, min(ENVS_PER_GPU, 0.4 / per_env)))
        steps = max(1, min(steps, int(budget_s / (per_env * n_envs))))
    w = np.ascontiguousarray(np.resize(w, (n_envs, size)))
    s = np.ascontiguousarray(np.resize(s, (n_envs, size)))
    acts = rs.randint(size + 1, size=(min(warmup + steps, 64), n_envs)).astype(np.int32)
    for i in range(warmup):
        oracle.step_batch(w, s, SIDE, acts[i % len(acts)], SPAWN, STABLE, threads)
    t0 = time.perf_counter()
    for i in range(steps):
        oracle.step_batch(w, s, SIDE, acts[(warmup + i) % len(acts)], SPAWN, STABLE, threads)
    dt = time.perf_counter() - t0
    gcups = n_envs * size * steps / dt / 1e9
    return {"value": gcups, "unit": "Gcell-updates/s", "cores": threads, "kind": "port",
            "sample": f"{n_envs} envs x {SIDE}x{SIDE} x {steps} steps (toggle+step+reward), oracle/cgl_oracle.c "
                      f"= C port of CGL/CGL.py:211-243, {threads} host threads",
            "env_steps_per_s": n_envs * steps / dt, "ms_per_step": dt / steps * 1e3, "steps": steps, "n_envs": n_envs}


def reference_line(args, base, extra=None):
    line = {"impl": args.impl, "metric": "life_cell_updates_per_s", "value": base["value"], "unit": base["unit"],
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": base["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(args.gpus),
            "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": base["value"], "unit": base["unit"], "h2d_bytes_per_step": base.get("h2d", 0),
                    "d2h_bytes_per_step": base.get("d2h", 0)},
            "env_steps_per_s": base["env_steps_per_s"], "gpu_launches": base.get("launches", 0)}
    line.update(extra or {})
    print(json.dumps(line), flush=True)


def run_reference_arm(args):
    """The reference's CPU implementation of the path on the host cores: exactly K timed steps after W warm-up steps,
    each step a bounded sample of the C2 batch (as many envs as fit ~60 s for the whole run, at most all 4096)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    reference_line(args, cpu_arm(args.steps, args.warmup, budget_s=60.0, exact_steps=True))


def run_reference_gpu_arm(args):
    """The reference's GPU step as its users run it (`main.py --exp-gpu`): its own kernel `run` (CGL/CGL.py:146-182,
    compiled for sm_100a by tests/golden/make_ref_cubins.py) + the four blocking PCIe copies of __step_state_gpu
    (:203-208) from pageable numpy arrays + toggle_state / reward in numpy (:322-328, :255-256), one env object at a
    time like the reference.  A bounded sample of the C2 batch per step."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torch
    from oracle import oracle, ref_gpu
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    size = SIDE * SIDE
    n_envs = 256
    worlds = [oracle.initial_world(SIDE, e) for e in range(n_envs)]
    stables = [oracle.initial_stable(w, SPAWN) for w in worlds]
    step = ref_gpu.RefGpuStep(SIDE, STABLE, SPAWN)
    rs = np.random.RandomState(10 ** 6)

    def one_step():
        acts = rs.randint(size + 1, size=n_envs)
        tot = 0
        for e in range(n_envs):
            a = acts[e]
            if a < size:                                    # toggle_state (CGL/CGL.py:322-328)
                worlds[e][a] = np.logical_not(worlds[e][a])
                stables[e][a] = SPAWN
            step.step(worlds[e], stables[e])
            tot += int(np.add.reduce(stables[e], dtype=np.int32))          # reward()
        return tot

    for _ in range(args.warmup):
        one_step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one_step()
    dt = time.perf_counter() - t0
    step.close()
    base = {"value": n_envs * size * args.steps / dt / 1e9, "unit": "Gcell-updates/s", "cores": 1, "kind": "reference",
            "sample": f"{n_envs} envs x {SIDE}x{SIDE} x {args.steps} steps, the reference's CUDA kernel `run` + its four PCIe "
                      f"copies per env step (CGL/CGL.py:203-208), one env at a time, 1 host thread",
            "env_steps_per_s": n_envs * args.steps / dt, "ms_per_step": dt / args.steps * 1e3,
            "h2d": 2 * size * n_envs, "d2h": 2 * size * n_envs, "launches": n_envs * args.steps}
    reference_line(args, base, {"us_per_env_step": dt / args.steps / n_envs * 1e6})


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
class Ctx:
    pass


def setup_dist():
    import torch
    import torch.distributed as dist
    c = Ctx()
    c.torch, c.dist = torch, dist
    c.rank = int(os.environ.get("RANK", "0"))
    c.world = int(os.environ.get("WORLD_SIZE", "1"))
    c.local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(c.local)
    c.dev = torch.device("cuda", c.local)
    if c.world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=c.dev)

    def barrier():
        if c.world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if c.world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=c.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    c.barrier, c.max_over_ranks = barrier, max_over_ranks
    return c


def timed_region(c, issue, events=None):
    """ONE timed region: barrier + synchronize, CUDA events around issue(), synchronize + barrier.  Seconds.
    events = (e0, e1): issue() records them itself on the launching stream, right before its first and right after
    its last launch (StepSequence.prepare(K, events=...) -> cgl_env_step_seq_timed)."""
    torch = c.torch
    c.barrier()
    torch.cuda.synchronize()
    if events is None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        issue()
        e1.record()
    else:
        e0, e1 = events
        issue()
    torch.cuda.synchronize()
    c.barrier()
    return e0.elapsed_time(e1) / 1e3


def repeat_regions(c, issue, repeats, events=None):
    """`repeats` timed regions; every region's time is the max over ranks; returns (median, all)."""
    ts = [c.max_over_ranks(timed_region(c, issue, events)) for _ in range(repeats)]
    return statistics.median(ts), ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps per region (default 200; c4: 1000 generations)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--config", default="c2", choices=["c2", "c4"])
    ap.add_argument("--repeats", type=int, default=7, help="timed regions of K steps each; the median is reported")
    ap.add_argument("--launch", default="eager", choices=["graph", "eager"],
                    help="how a region's K steps are issued: K launches from one C-ABI call (default; consecutive "
                         "launches overlap through programmatic dependent launch + per-env chaining) or CUDA-graph replay")
    ap.add_argument("--no-extras", action="store_true", help="skip the C1/C3/C4/C5 and f-row side measurements")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned to its caller as float32 "
                         f"DIR/<name>.npy (rank 0): reward [{ENVS_PER_GPU}] of the env batch it stepped, and obs "
                         f"(int8 stability) and world (cells) [{DUMP_ENVS}, {SIDE * SIDE}] of a fixed sample of "
                         f"{DUMP_ENVS} of its envs (RandomState({DUMP_SEED}), sorted); C2 GPU run only")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 1000 if args.config == "c4" else 200
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config != "c2"):
        ap.error("--dump-outputs is implemented for the C2 GPU run (--impl ours --config c2) only")
    if args.impl == "reference":
        return run_reference_arm(args)
    if args.impl == "reference-gpu":
        return run_reference_gpu_arm(args)
    args.warmup = max(args.warmup, 3)
    args.repeats = max(args.repeats, 1)

    import torch
    from cgl_b200 import native
    native.load()                                           # fail loudly if the CUDA library is missing
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    c = setup_dist()
    if args.config == "c4":
        line = run_c4_line(c, args)
    else:
        line = run_c2_line(c, args)
    if c.rank == 0:
        print(json.dumps(line), flush=True)
    if c.world > 1:
        c.dist.destroy_process_group()


def run_c2_line(c, args):
    torch = c.torch
    from cgl_b200.batched import BatchedSim, StepSequence
    dev, rank, world = c.dev, c.rank, c.world
    size = SIDE * SIDE
    B, R, K, W = ENVS_PER_GPU, REPLICAS, args.steps, args.warmup
    sims = [BatchedSim(B, SIDE, seed=rank * 10 ** 5 + r * B, spawnStabilityFactor=SPAWN, stableStabilityFactor=STABLE,
                       device=dev, rng="device") for r in range(R)]
    n_act = 16
    g = torch.Generator(device=dev); g.manual_seed(10 ** 6 + rank)
    actions = torch.randint(0, size + 1, (n_act, B), dtype=torch.int32, device=dev, generator=g)
    seq = StepSequence(sims, actions)
    per_step_launches = sims[0]._lib.cgl_env_step_launches(SIDE, 1)
    seq.run(W)                                              # W untimed warm-up steps
    torch.cuda.synchronize()

    # ---- headline: K steps per region, issued by one C-ABI call (K launches) --------------------------------
    sampler = ClockSampler(c.local).start() if rank == 0 else None
    events = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    issue = seq.prepare(K, events=events)
    issue(); issue()                                        # (both plane orientations of an odd K are cached now)
    dt_eager, regions_eager = repeat_regions(c, issue, args.repeats, events)
    use_graph = args.launch == "graph"
    outputs = None
    if args.dump_outputs and rank == 0 and not use_graph:
        outputs = last_step_outputs(sims[(K - 1) % R])      # before the L2-resident variant steps sims[0] again

    # L2-resident variant (one replica, 80 MiB working set inside the 126 MB L2) -- reported, not the headline
    seq1 = StepSequence(sims[:1], actions)
    dt_l2, _ = repeat_regions(c, lambda: seq1.run(K), min(args.repeats, 3))

    # ---- CUDA-graph replay of the same steps (one graph = 2R steps: every plane back in place) ---------------
    # captured on extra env batches: a captured batch keeps plane-id tokens for good (see BatchedSim)
    cycle = 2 * R
    gsims = [BatchedSim(B, SIDE, seed=rank * 10 ** 5 + (R + r) * B, spawnStabilityFactor=SPAWN, stableStabilityFactor=STABLE,
                        device=dev, rng="device") for r in range(R)]
    gseq = StepSequence(gsims, actions)
    gseq.run(cycle)
    torch.cuda.synchronize()
    side_stream = torch.cuda.Stream(device=dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side_stream):
        with torch.cuda.graph(graph, stream=side_stream):
            gseq.run(cycle)
    graph.replay()
    torch.cuda.synchronize()

    def issue_graph():
        for _ in range(K // cycle):
            graph.replay()
        if K % cycle:               # every call starts at sims[0]: the rest twice steps each sim an even number of times,
            gseq.run(K % cycle)     # so its planes are back in the captured position (the second call is part of the region)
            gseq.run(K % cycle)
    k_graph = K + K % cycle
    dt_graph, regions_graph = repeat_regions(c, issue_graph, min(args.repeats, 5))
    dt_graph = dt_graph * K / k_graph
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0 and use_graph:
        outputs = last_step_outputs(gsims[(K - 1) % R])     # issue_graph() ends on the same sim as the eager path
    if outputs is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
    del gsims, gseq, graph
    torch.cuda.empty_cache()

    dt = dt_graph if use_graph else dt_eager
    cells_per_step = B * size * world
    value = cells_per_step * K / dt / 1e9
    gpu_launches = K * per_step_launches * args.repeats

    # ---- end to end: host-driven rollout, actions from and rewards to pinned host memory every step --------
    e2e = None
    if not args.no_e2e:
        e2e = measure_e2e(c, args, sims)

    peak, peak_src = measured_peak_gbs()
    achieved = BYTES_PER_CELL_ENV * B * size / (dt / K) / 1e9          # per GPU, per launch
    kernel = f"env_step_fused_kernel<{SIDE}>"
    traffic, traffic_src = recorded_traffic(kernel)
    roofline = {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": BYTES_PER_CELL_ENV * B * size, "avg_launch_ms": dt / K * 1e3,
                "note": "avg_launch_ms = region time / K: consecutive launches overlap (programmatic dependent launch "
                        "+ per-env tokens), so it can be below the duration ncu reports for one serialised launch",
                "l2_resident_variant_gbs": BYTES_PER_CELL_ENV * B * size / (dt_l2 / K) / 1e9}

    extras = {}
    if not args.no_extras:
        try:
            extras = run_extras(c, peak)
        except Exception as exc:  # noqa: BLE001
            extras = {"error": repr(exc)}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_arm(steps=10 ** 6, warmup=1, budget_s=12.0, exact_steps=False)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}

    return {"metric": "life_cell_updates_per_s", "value": value, "unit": "Gcell-updates/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": dt / K * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": workload_config(world),
            "env_steps_per_s": B * world * K / dt, "clocks": clocks, "e2e": e2e, "gpu_launches": gpu_launches,
            "roofline": roofline, "cpu_baseline": cpu, "l2_resident_value": cells_per_step * K / dt_l2 / 1e9,
            "launch": args.launch, "repeats": args.repeats,
            "timing": "median of `repeats` regions of K steps; each region: barrier + synchronize, CUDA events, "
                      "synchronize + barrier, max over ranks",
            "regions_ms": [t * 1e3 for t in (regions_graph if use_graph else regions_eager)],
            ("graph_value" if not use_graph else "eager_value"):
                cells_per_step * K / (dt_eager if use_graph else dt_graph) / 1e9,
            "extras": extras}


def last_step_outputs(sim):
    """What the last step of `sim` returned to its caller (BatchedSim.step: reward, obs) and the world it left, as
    float32 host arrays; the two planes for a fixed sample of DUMP_ENVS envs (in full they are 2 x 256 MiB)."""
    import torch
    envs = np.sort(np.random.RandomState(DUMP_SEED).choice(sim.n_envs, DUMP_ENVS, replace=False))
    idx = torch.from_numpy(envs).to(sim.device)
    return {"reward": sim._reward.cpu().numpy().astype(np.float32),
            "obs": sim.stable[idx].cpu().numpy().astype(np.float32),
            "world": sim.get_state()[idx].cpu().numpy().astype(np.float32)}


def measure_e2e(c, args, sims):
    """End to end through the public host-buffer API.  Headline: HostRollout (E2E_GROUPS groups of envs stepped in
    turn, the loop in C, a Python policy that reads the group's previous rewards and writes its next actions).
    Beside it: the synchronous single-group call (BatchedSim.step_host) and the rollout that also copies the whole
    observation to the host every step."""
    torch = c.torch
    from cgl_b200.rollout import HostRollout
    B, R, size = ENVS_PER_GPU, REPLICAS, SIDE * SIDE
    ke = 200                                                # (its own step count: a region of 200 full steps)
    reps = min(args.repeats, 5)

    def make(obs, zero_copy=False):
        return HostRollout(B, SIDE, n_groups=E2E_GROUPS, n_replicas=R, seed=c.rank * 10 ** 5 + 77, spawnStabilityFactor=SPAWN,
                           stableStabilityFactor=STABLE, device=c.dev, rng="device", obs_to_host=obs,
                           zero_copy_actions=zero_copy)

    def policy(group, step, rewards, actions):              # reads a reward of the group's last step, writes an action
        actions[step & 511] = (int(rewards[step & 511]) + step) % (size + 1)

    def wall(fn):
        c.barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        dt = c.max_over_ranks(time.perf_counter() - t0)
        c.barrier()
        return dt

    ro = make(False)
    for g in range(E2E_GROUPS):
        ro.actions[g][:] = np.random.RandomState(g).randint(size + 1, size=B // E2E_GROUPS)
    ro.run(4, policy)
    dts = [wall(lambda: ro.run(ke, policy)) for _ in range(reps)]
    dt_ro = statistics.median(dts)
    dts_np = [wall(lambda: ro.run(ke, None)) for _ in range(min(reps, 3))]
    ro.close()
    del ro
    # variant: no copy node, the kernel reads the actions from the pinned buffer over PCIe
    ro = make(False, zero_copy=True)
    for g in range(E2E_GROUPS):
        ro.actions[g][:] = np.random.RandomState(g).randint(size + 1, size=B // E2E_GROUPS)
    ro.run(4, policy)
    dts_zc = [wall(lambda: ro.run(ke, policy)) for _ in range(reps)]
    dt_zc = statistics.median(dts_zc)
    ro.close()
    del ro
    # synchronous single call per step (the round-1 e2e): copy, launch, synchronise, repeat
    acts_h = [torch.randint(0, size + 1, (B,), dtype=torch.int32).pin_memory() for _ in range(4)]
    rew_h = torch.empty(B, dtype=torch.int32).pin_memory()
    for i in range(3):
        sims[i % R].step_host(acts_h[i % 4], rew_h)

    def sync_loop():
        for i in range(ke):
            sims[i % R].step_host(acts_h[i % 4], rew_h)
    dt_sync = statistics.median([wall(sync_loop) for _ in range(min(reps, 3))])
    # observation to the host as well (the reference's get_stable contract): PCIe-bound
    ko = 6
    ro = make(True)
    ro.run(2, policy)
    dt_obs = statistics.median([wall(lambda: ro.run(ko, policy)) for _ in range(3)])
    ro.close()
    del ro
    torch.cuda.empty_cache()
    cells = B * size * c.world
    # Both action paths move the same 4 B per env and step from pinned host memory to the device inside the timed
    # region -- a DMA copy node in front of the kernel, or the kernel's own loads over PCIe (a constructor flag of
    # the public API).  Which one is faster depends on the box (DMA start-up latency against PCIe read latency), so
    # the headline is the faster of the two, named in `actions_path`; both are listed.
    best_zc = dt_zc < dt_ro
    dt_best, dts_best = (dt_zc, dts_zc) if best_zc else (dt_ro, dts)
    return {"value": cells * ke / dt_best / 1e9, "unit": "Gcell-updates/s", "h2d_bytes_per_step": 4 * B,
            "d2h_bytes_per_step": 4 * B, "steps": ke, "repeats": reps, "us_per_step": dt_best / ke * 1e6,
            "env_steps_per_s": B * c.world * ke / dt_best,
            "actions_path": "kernel loads from pinned host memory (zero_copy_actions=True)" if best_zc else
                            "cudaMemcpyAsync copy node from pinned host memory",
            "api": f"cgl_b200.rollout.HostRollout.run(steps, policy) -> cgl_rollout_run: {E2E_GROUPS} groups of "
                   f"B/{E2E_GROUPS} envs stepped in turn on their own streams, per group step one CUDA graph [actions from "
                   "pinned host memory -> fused env step], rewards written by the kernel into pinned host memory, "
                   "completion polled; the Python policy is called per group and step with the group's previous rewards "
                   "(data dependence kept per group); the observation stays device-resident for a GPU Q-network",
            "regions_us_per_step": [d / ke * 1e6 for d in dts_best],
            "copy_node_actions": {"value": cells * ke / dt_ro / 1e9, "unit": "Gcell-updates/s", "us_per_step": dt_ro / ke * 1e6,
                                  "what": "per group step a graph of [H2D cudaMemcpyAsync of the group's pinned action "
                                          "buffer -> kernel]"},
            "zero_copy_actions": {"value": cells * ke / dt_zc / 1e9, "unit": "Gcell-updates/s", "us_per_step": dt_zc / ke * 1e6,
                                  "what": "no copy node: the kernel loads each env's action from the pinned host buffer "
                                          "over PCIe (the same 4 B per env per step, host to device)"},
            "without_policy_callback": {"value": cells * ke / statistics.median(dts_np) / 1e9, "unit": "Gcell-updates/s",
                                        "what": "copy-node path without the Python policy"},
            "synchronous_single_call": {"value": cells * ke / dt_sync / 1e9, "unit": "Gcell-updates/s",
                                        "us_per_step": dt_sync / ke * 1e6,
                                        "api": "BatchedSim.step_host -> cgl_env_step_host (copy, step, sync per step)"},
            "with_obs_to_host": {"value": cells * ko / dt_obs / 1e9, "unit": "Gcell-updates/s",
                                 "d2h_bytes_per_step": 4 * B + B * size, "steps": ko,
                                 "pcie_d2h_gbs": (4 * B + B * size) * ko / dt_obs / 1e9}}


# ---------------------------------------------------------------------------------------------
# C4: 65536^2 torus, row bands over the ranks (BASELINE.json configs[3])
# ---------------------------------------------------------------------------------------------
def measure_c4(c, gens, repeats, check=True):
    """`gens` generations of the 65536^2 torus with IDENTICAL settings at every N (ghost depth, generations per
    launch, seed): returns time per region, live count and the order-independent checksum of the final grid, which
    must not depend on N."""
    torch = c.torch
    from cgl_b200.bands import RowBandLife
    n = C4_SIDE
    band = RowBandLife(n, n, k=C4_GHOST, rank=c.rank, world_size=c.world, device=c.dev, kernel_k=C4_KERNEL_K)
    band.randomize(1)
    band.run(2 * C4_GHOST)                                  # warm-up (also tunes the strip length once)
    torch.cuda.synchronize()
    dt, regions = repeat_regions(c, lambda: band.run(gens), repeats)
    out = {"gcups": n * n * gens / dt / 1e9, "ms_per_gen": dt / gens * 1e3, "gens": gens, "generation": band.generation,
           "kernel_k": C4_KERNEL_K, "ghost_depth": C4_GHOST, "exchange": band.exchange, "scaling": "strong",
           "regions_ms": [t * 1e3 for t in regions], "launches": band.launches}
    if check:
        out["alive"] = band.alive()
        out["checksum"] = band.checksum()
        out["checksum_note"] = (f"after {band.generation} generations from seed 1: equal at every N iff the N-GPU "
                                "bands compute the single-GPU torus")
    band.close()
    del band
    torch.cuda.empty_cache()
    return out, dt


def run_c4_line(c, args):
    peak, peak_src = measured_peak_gbs()
    sampler = ClockSampler(c.local).start() if c.rank == 0 else None
    res, dt = measure_c4(c, args.steps, min(args.repeats, 3))
    clocks = sampler.stop() if sampler else None
    n, K = C4_SIDE, args.steps
    per_gpu_bytes = BYTES_PER_CELL_LIFE * n * n / c.world
    achieved = per_gpu_bytes / (dt / K) / 1e9
    return {"metric": "life_cell_updates_per_s", "value": res["gcups"], "unit": "Gcell-updates/s", "n_gpus": c.world,
            "steps": K, "warmup": 2 * C4_GHOST, "ms_per_step": dt / K * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": c4_config(c.world), "clocks": clocks,
            "e2e": None, "gpu_launches": res["launches"],
            "roofline": {"bound": "hbm", "kernel": f"life_tb_kernel<{C4_KERNEL_K}>", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                         "note": "algorithmic 0.25 B per cell and generation; with k generations per HBM pass the "
                                 "fraction may exceed 1 -- the kernel is bound by the integer pipe (DESIGN.md 4.5)"},
            "cpu_baseline": None, "c4": res}


def run_extras(c, peak):
    """Side measurements of the other BASELINE configs (short; not the headline line)."""
    torch, dev, rank, world, barrier = c.torch, c.dev, c.rank, c.world, c.barrier
    from cgl_b200 import native
    from cgl_b200.batched import BatchedSim, StepSequence
    lib = native.load()
    out = {}
    # C3: 65536 envs x 64x64, sharded by env index over the ranks (strong scaling over N)
    side, total = 64, 65536
    sim = BatchedSim.shard(total, side, rank, world, seed=0, spawnStabilityFactor=SPAWN, stableStabilityFactor=STABLE,
                           device=dev, rng="device")
    acts = torch.randint(0, side * side + 1, (8, sim.n_envs), dtype=torch.int32, device=dev)
    seq = StepSequence([sim], acts)
    seq.run(6)
    k = 48
    dt, _ = repeat_regions(c, seq.prepare(k), 5)
    out["c3_envs65536_side64"] = {"gcups": total * side * side * k / dt / 1e9, "env_steps_per_s": total * k / dt,
                                  "ms_per_step": dt / k * 1e3, "scaling": "strong",
                                  "hbm_frac": BYTES_PER_CELL_ENV * sim.n_envs * side * side / (dt / k) / 1e9 / peak,
                                  "working_set_mib_per_gpu": sim.n_envs * side * side * 1.25 / 2 ** 20}
    del sim, acts, seq
    torch.cuda.empty_cache()
    # C4: 65536^2 torus, 1000 generations, row bands over the ranks -- same settings and seed at every N
    res, _ = measure_c4(c, 1000, 3)
    res["hbm_frac_algorithmic"] = BYTES_PER_CELL_LIFE * C4_SIDE * C4_SIDE / world / (res["ms_per_gen"] / 1e3) / 1e9 / peak
    out["c4_life_65536_bands"] = res
    if world == 1:
        out.update(single_gpu_extras(c, peak, lib))
    return out


def time_steps(c, fn, steps):
    return timed_region(c, lambda: [fn(i) for i in range(steps)])


def single_gpu_extras(c, peak, lib):
    torch, dev = c.torch, c.dev
    from cgl_b200 import native
    from cgl_b200.batched import BatchedSim
    out = {}
    # C1: the reference's own single-env loop shape (CGL/main.py:64-72 with random actions) through the drop-in
    # facade, 64x64; beside it the oracle port on one host core, the reference's Python loop (timed on the build
    # box by tools/time_reference_cpu.py) and the reference's GPU step (its own kernel + four PCIe copies)
    import CGL
    from oracle import oracle
    side, n = 64, 4000
    acts = np.random.RandomState(123).randint(side * side + 1, size=n + 100).astype(np.int32)
    env = CGL.sim(side=side, seed=0, gpu=True, gpu_select=dev.index, spawnStabilityFactor=SPAWN, stableStabilityFactor=STABLE)
    obs = env.get_stable(vector=True, shallow=True)
    acc = 0
    for i in range(100):
        env.toggle_state(acts[i]); env.step(); obs = env.get_stable(vector=True, shallow=True); acc += int(env.reward())
    t0 = time.perf_counter()
    for i in range(100, 100 + n):
        env.toggle_state(acts[i]); env.step(); obs = env.get_stable(vector=True, shallow=True); acc += int(env.reward())
    dt_f = time.perf_counter() - t0
    ref = oracle.OracleSim(side=side, seed=0, spawnStabilityFactor=SPAWN, stableStabilityFactor=STABLE)
    acc_o = 0
    for i in range(100):
        ref.toggle_state(acts[i]); ref.step(); acc_o += int(ref.reward())
    t0 = time.perf_counter()
    for i in range(100, 100 + n):
        ref.toggle_state(acts[i]); ref.step(); acc_o += int(ref.reward())
    dt_o = time.perf_counter() - t0
    obs_equal = bool(np.array_equal(obs, ref.get_stable(vector=True)))
    # the reference's own bench loop (CGL/bench.py:39-40: plain steps, then Stability and Life are printed): the
    # facade defers the plain steps and runs them as one on-chip launch when the result is asked for
    env2 = CGL.sim(side=side, seed=0, gpu=True, gpu_select=dev.index, spawnStabilityFactor=SPAWN, stableStabilityFactor=STABLE)
    ref.reset()
    env2.step(); env2.step(); env2.step(); env2.step(); env2.reward()
    t0 = time.perf_counter()
    for _ in range(n):
        env2.step()
    r_f, a_f = int(env2.reward()), int(env2.alive())
    dt_b = time.perf_counter() - t0
    for _ in range(n + 4):
        ref.step()
    del env2
    plain_equal = (r_f, a_f) == (int(ref.reward()), int(ref.alive()))
    c1 = {"facade_env_steps_per_s": n / dt_f, "facade_us_per_step": dt_f / n * 1e6,
          "oracle_port_1core_env_steps_per_s": n / dt_o, "facade_plain_step_loop_steps_per_s": n / dt_b,
          "plain_loop_equal": plain_equal, "rewards_equal": acc == acc_o, "final_obs_equal": obs_equal}
    try:
        with open(os.path.join(ROOT, "profiles", "reference_cpu_timing.json")) as f:
            rt = json.load(f)
        c1["reference_python_env_steps_per_s"] = rt["loops"]["side64"]["dqn_loop_env_steps_per_s"]
        c1["reference_python_source"] = ("profiles/reference_cpu_timing.json: tools/time_reference_cpu.py on the build "
                                         f"box, {rt['host']['cores_used']} core of {rt['host']['os_cpu_count']} ({rt['when']})")
    except Exception:  # noqa: BLE001
        c1["reference_python_env_steps_per_s"] = None
    try:                                                    # the reference's GPU step on this GPU (same loop shape)
        from oracle import ref_gpu
        step = ref_gpu.RefGpuStep(side, STABLE, SPAWN)
        w = oracle.initial_world(side, 0)
        s = oracle.initial_stable(w, SPAWN)
        m = 1000
        acc_r = 0
        for i in range(100 + m):
            if i == 100:
                t0 = time.perf_counter()
            a = acts[i]
            if a < side * side:
                w[a] = np.logical_not(w[a]); s[a] = SPAWN
            step.step(w, s)
            acc_r += int(np.add.reduce(s, dtype=np.int32))
        dt_r = time.perf_counter() - t0
        step.close()
        ref2 = oracle.OracleSim(side=side, seed=0, spawnStabilityFactor=SPAWN, stableStabilityFactor=STABLE)
        acc_c = 0
        for i in range(100 + m):
            ref2.toggle_state(acts[i]); ref2.step(); acc_c += int(ref2.reward())
        c1["reference_gpu_step_env_steps_per_s"] = m / dt_r
        c1["reference_gpu_step_rewards_equal"] = acc_r == acc_c
        c1["reference_gpu_step_what"] = ("the reference's kernel `run` (tests/golden/ref_kernels) + its four blocking PCIe "
                                         "copies per step (CGL/CGL.py:203-208) + numpy toggle/reward")
    except Exception as exc:  # noqa: BLE001
        c1["reference_gpu_step_env_steps_per_s"] = None
        c1["reference_gpu_step_error"] = repr(exc)[:200]
    out["c1_single_64x64_loop"] = c1
    del env
    # C5: 32768^2 torus, sweep of the temporal-blocking depth k on one GPU
    n = 32768
    words = n * (n // 32)
    a = torch.randint(-2 ** 31, 2 ** 31 - 1, (words,), dtype=torch.int32, device=dev)
    b = torch.empty_like(a)
    res = native.ctypes.c_int(0)
    sweep = {}
    for k in (1, 2, 4, 8, 16):
        g = 48

        def run(_i):
            native.check(lib.cgl_life_run(native.dptr(a), native.dptr(b), n, n, 1, g, k, native.ctypes.byref(res),
                                          native.current_stream()))
        if k > 1:        # set-up: let the library time its strip lengths for this shape (RowBandLife does the same)
            native.check(lib.cgl_life_tune(native.dptr(a), native.dptr(b), n, n, 1, k, native.current_stream()))
        run(0)
        dt = statistics.median(time_steps(c, run, 1) for _ in range(3))
        sweep[f"k{k}"] = {"gcups": n * n * g / dt / 1e9, "us_per_gen": dt / g * 1e6,
                          "hbm_frac_algorithmic": BYTES_PER_CELL_LIFE * n * n / (dt / g) / 1e9 / peak}
    out["c5_life_32768_k_sweep"] = sweep
    del a, b
    torch.cuda.empty_cache()
    # f3: the reference's own bench loop (CGL/bench.py:39-40: plain steps, no actions) as ONE launch per k
    # steps with the environments resident on chip (cgl_env_run), config 2 shape
    env = BatchedSim(4096, 128, seed=0, spawnStabilityFactor=SPAWN, stableStabilityFactor=STABLE, rng="device")
    runk = {}
    for k in (8, 64):
        env.run(k)
        dt = time_steps(c, lambda _i: env.run(k), 3) / 3
        runk[f"k{k}"] = {"gcups": 4096 * 128 * 128 * k / dt / 1e9, "us_per_step": dt / k * 1e6,
                         "env_steps_per_s": 4096 * k / dt}
    del env
    for rule in ("decay", "sat"):                            # the fork's rules on chip (bit planes), 64 steps per launch
        env = BatchedSim(4096, 128, seed=0, spawnStabilityFactor=SPAWN, stableStabilityFactor=STABLE, rng="device",
                         dead_rule=rule, empty=-1, empty_min=-6, masked_toggle=True)
        env.run(64)
        dt = time_steps(c, lambda _i: env.run(64), 3) / 3
        runk[f"k64_{rule}"] = {"gcups": 4096 * 128 * 128 * 64 / dt / 1e9, "us_per_step": dt / 64 * 1e6}
        del env
    out["f3_run_in_smem_4096x128"] = runk
    # f2: the CGL_action+ fork's rule (dead cells decay to a floor, masked toggle) in the same fused kernel
    g = torch.Generator(device=dev)
    g.manual_seed(11)
    acts_d = torch.randint(0, 128 * 128 + 1, (4096,), dtype=torch.int32, device=dev, generator=g)
    fork_rates = {}
    for rule in ("decay", "sat"):
        envs = [BatchedSim(4096, 128, seed=i, spawnStabilityFactor=SPAWN, stableStabilityFactor=STABLE, rng="device",
                           dead_rule=rule, empty=-1, empty_min=-6, masked_toggle=True) for i in range(4)]
        for i in range(8):
            envs[i % 4].step(acts_d)
        dt = time_steps(c, lambda i: envs[i % 4].step(acts_d), 400) / 400
        fork_rates[rule] = {"gcups": 4096 * 128 * 128 / dt / 1e9, "us_per_step": dt * 1e6,
                            "hbm_frac": BYTES_PER_CELL_ENV * 4096 * 128 * 128 / dt / 1e9 / peak}
        del envs
    out["f2_fork_rule_4096x128"] = fork_rates
    # f1: config 2 under the batched DQN loop (the reference's main.py:58-75 for 4096 envs at once):
    # select_action -> toggle+step+reward into the replay ring -> learn -> target update, all on the device.
    # Network = dqn.py:41-59 at side 128 (16384 -> 32770 -> 32770 -> 16385, 2.15 G parameters, fp32).
    try:
        out["f1_dqn_loop_4096x128"] = dqn_loop_extra(c)
    except torch.OutOfMemoryError as exc:                    # another tenant on the GPU: report, do not fail the bench
        out["f1_dqn_loop_4096x128"] = {"skipped": f"out of memory: {str(exc)[:80]}"}
    torch.cuda.empty_cache()
    return out


def dqn_loop_extra(c, n_envs=4096, side=128, steps=3):
    torch = c.torch
    from cgl_b200.batched import BatchedSim
    from cgl_b200.dqn import BatchedDQNAgent
    env = BatchedSim(n_envs, side, seed=0, spawnStabilityFactor=SPAWN, stableStabilityFactor=STABLE, rng="device")
    agent = BatchedDQNAgent(env, max_size=int(1e5), batch_size=64, seed=0)
    res = {"n_envs": n_envs, "side": side, "parameters": sum(p.numel() for p in agent.Q.parameters()),
           "replay_slots": agent.memory.slots, "replay_bytes_moved_per_step": 0}
    state = [agent.reset()]

    def loop(_i):
        action = agent.select_action(state[0], 0.1, out=agent.memory.action_slot())
        state[0], _ = agent.step(action)

    def env_only(_i):
        agent.memory.step(agent.memory.action_slot())

    for name, tf32 in (("fp32", False), ("tf32", True)):
        torch.backends.cuda.matmul.allow_tf32 = tf32
        loop(0); loop(0)
        dt = time_steps(c, loop, steps) / steps
        res[name] = {"env_steps_per_s": n_envs / dt, "ms_per_batched_step": dt * 1e3}
    torch.backends.cuda.matmul.allow_tf32 = False
    agent.act_dtype = torch.bfloat16                     # opt-in: acting forward on the bf16 tensor cores
    loop(0); loop(0)
    dt = time_steps(c, loop, steps) / steps
    res["bf16_acting"] = {"env_steps_per_s": n_envs / dt, "ms_per_batched_step": dt * 1e3}
    agent.act_dtype = None
    env_only(0)
    dt_env = time_steps(c, env_only, 200) / 200
    res["env_step_into_ring_us"] = dt_env * 1e6
    res["env_share_of_loop_fp32"] = dt_env / (res["fp32"]["ms_per_batched_step"] / 1e3)
    env.check_actions()
    return res


if __name__ == "__main__":
    main()
