"""Time the env step under different knobs (one process per knob set; knobs come from the environment).
Reports eager-launch time, host launch cost and CUDA-graph replay time per step."""
import os, sys, json, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "ecen743-project-cgol_b200")):
    sys.path.insert(0, p)
import torch
from cgl_b200.batched import BatchedSim
side, B, R = int(os.environ.get("SIDE", 128)), int(os.environ.get("ENVS", 4096)), int(os.environ.get("REPL", 4))
dev = torch.device("cuda", 0)
sims = [BatchedSim(B, side, seed=r * B, spawnStabilityFactor=-2, stableStabilityFactor=2, device=dev, rng="device") for r in range(R)]
acts = torch.randint(0, side * side + 1, (B,), dtype=torch.int32, device=dev)
for i in range(12):
    sims[i % R].step(acts)
torch.cuda.synchronize()
K = 200
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
best, host = 1e9, 1e9
for rep in range(3):
    t0 = time.perf_counter()
    e0.record()
    for i in range(K):
        sims[i % R].step(acts)
    e1.record()
    host = min(host, (time.perf_counter() - t0) / K * 1e6)
    torch.cuda.synchronize()
    best = min(best, e0.elapsed_time(e1) / K * 1e3)
# CUDA graph of 2R steps (each sim stepped twice so the ping-pong buffers end where they started)
g = torch.cuda.CUDAGraph()
s = torch.cuda.Stream()
with torch.cuda.stream(s):
    for i in range(2 * R):
        sims[i % R].step(acts)
    torch.cuda.synchronize()
    with torch.cuda.graph(g, stream=s):
        for i in range(2 * R):
            sims[i % R].step(acts)
for _ in range(3):
    g.replay()
torch.cuda.synchronize()
gb = 1e9
for rep in range(3):
    e0.record()
    for _ in range(K // (2 * R)):
        g.replay()
    e1.record(); torch.cuda.synchronize()
    gb = min(gb, e0.elapsed_time(e1) / (K // (2 * R) * 2 * R) * 1e3)
bytes_step = 2.25 * B * side * side
print(json.dumps({"pdl": os.environ.get("CGL_ENV_PDL", "1"), "chained": os.environ.get("CGL_ENV_CHAINED", "1"), "side": side,
                  "envs": B, "repl": R, "eager_us": round(best, 2), "host_launch_us": round(host, 2), "graph_us": round(gb, 2),
                  "frac_eager": round(bytes_step / (best * 1e-6) / 1e9 / 6543.4, 4),
                  "frac_graph": round(bytes_step / (gb * 1e-6) / 1e9 / 6543.4, 4)}))
