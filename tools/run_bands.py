#!/usr/bin/env python
"""Row-band life mode on N GPUs (torchrun entry point): correctness check and timing.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29511 \
        tools/run_bands.py --rows 65536 --cols 65536 --k 8 --gens 1000 --exchange p2p [--check]

--check: rank 0 re-runs the same grid on ONE GPU as a plain torus and compares checksum + alive count.
--population: record the population after every generation (RowBandLife.run(population=True)); with --check rank 0
also compares the N-GPU trace with the single-GPU torus trace generation by generation, without it the timed run
records the trace.
Prints one JSON line on rank 0."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "ecen743-project-cgol_b200")):
    sys.path.insert(0, p)
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
from cgl_b200.bands import RowBandLife  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=65536)
ap.add_argument("--cols", type=int, default=65536)
ap.add_argument("--k", type=int, default=8)
ap.add_argument("--gens", type=int, default=1000)
ap.add_argument("--kernel-k", type=int, default=0, help="generations per launch (default min(k, 8))")
ap.add_argument("--warmup", type=int, default=16)
ap.add_argument("--exchange", default="p2p", choices=["p2p", "dist"])
ap.add_argument("--check", action="store_true")
ap.add_argument("--seed", type=int, default=1)
ap.add_argument("--population", action="store_true")
a = ap.parse_args()

rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if world > 1:
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", device_id=dev)

band = RowBandLife(a.rows, a.cols, k=a.k, rank=rank, world_size=world, device=dev, exchange=a.exchange if world > 1 else None,
                   kernel_k=a.kernel_k or None)
band.randomize(a.seed)
result = {"rows": a.rows, "cols": a.cols, "k": a.k, "gens": a.gens, "n_gpus": world, "exchange": band.exchange}
if a.check:
    pop = band.run(a.gens, population=a.population)
    cs, alive = band.checksum(), band.alive()
    ok = True
    if rank == 0:
        ref = RowBandLife(a.rows, a.cols, k=a.k, rank=0, world_size=1, device=dev)
        # the same grid: every band's rows are seeded by global row index
        for r in range(world):
            tmp = RowBandLife(a.rows, a.cols, k=a.k, rank=r, world_size=world, device=dev, exchange="local")
            tmp.randomize(a.seed)
            ref.owned[r * tmp.band_rows:(r + 1) * tmp.band_rows] = tmp.owned
            del tmp
        ref_pop = ref.run(a.gens, population=a.population)
        ok = (ref.checksum() == cs) and (ref.alive() == alive)
        result.update(checksum=cs, alive=alive, ref_checksum=ref.checksum(), ref_alive=ref.alive())
        if a.population:
            diff = (pop != ref_pop).nonzero()
            same = diff.numel() == 0 and int(pop[-1]) == alive
            result.update(population_equal=same, first_population_mismatch=int(diff[0, 0]) if diff.numel() else None,
                          final_population=int(pop[-1]))
            ok = ok and same
        result.update(ok=ok)
    if world > 1:
        t = torch.tensor([int(ok)], device=dev)
        dist.broadcast(t, 0)
        ok = bool(t.item())
else:
    band.run(a.warmup, population=a.population)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    band.run(a.gens, population=a.population)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sec = float(t.item())
    result.update(population=a.population, seconds=sec, gcups=a.rows * a.cols * a.gens / sec / 1e9, ms_per_gen=sec / a.gens * 1e3,
                  alive=band.alive())
    ok = True
if rank == 0:
    print(json.dumps(result), flush=True)
band.close()
if world > 1:
    dist.destroy_process_group()
sys.exit(0 if ok else 1)
