"""RowBandLife -- one huge toroidal grid, world plane only ("life mode"), sharded by ROW BANDS.

The reference cannot express these sizes (`unsigned int` index math overflows above side 46340,
/root/reference/CGL/CGL.py:149-159) and is single-GPU (:6); this is the B200-native extension
BASELINE.json configs[3]/[4] name: 65536^2 x 1000 generations on 1/2/4/8 GPUs.

Rank r of G owns rows [r*H/G, (r+1)*H/G) of the H x C torus and keeps k ghost rows above and
below them.  Every k generations each rank sends its top k and bottom k owned rows to its ring
neighbours (rank 0's upper neighbour is rank G-1: that IS the vertical torus wrap), then runs k
generations over the whole (H/G + 2k)-row buffer with dead rows outside: the garbage that creeps
in from the buffer edges advances one row per generation and never reaches an owned row.
Horizontal wrap is local.  Message = k * C/8 bytes per neighbour per k generations.

Exchange back ends
  "p2p"   (default on GPUs) one exchange launch per block (`cgl_halo_exchange`, 8 CTAs per neighbour): each side
          writes its strip straight into the neighbour's landing zone over NVLink (CUDA-IPC mapped peer memory) and
          publishes a sequence flag, then spins on its own flag and moves the neighbour's strip into its ghost rows.
          Two landing slots alternate by block parity, so a rank may run one block ahead of its neighbour without a
          handshake.  No host synchronisation per exchange.  On one GPU, exchange="p2p" makes a ring of one that
          exchanges with itself (tests the exchange kernel without a second GPU).
  "dist"  torch.distributed batch_isend_irecv (NCCL on GPUs, gloo in the CPU tests).
  "local" all G bands live in this process (one GPU emulating G ranks; tests the ghost-zone math).
  "single" (default on one rank) no ghost rows: one torus, k-blocked launches of cgl_life_run.
"""
from __future__ import annotations

import ctypes

import torch

from . import native


def _life_block(lib, a, b, rows, cols, wrap_rows, gens, k, stream) -> bool:
    """`gens` generations starting from buffer `a`, ping-ponging with `b`, k generations per launch
    (temporal blocking, cgl_life_run).  Returns True if the result is in `a`.
    Tests monkeypatch this for CPU runs."""
    res = ctypes.c_int(-1)
    native.check(lib.cgl_life_run(native.dptr(a), native.dptr(b), rows, cols, wrap_rows, gens, k,
                                  ctypes.byref(res), stream), "cgl_life_run")
    return res.value == 1


def _life_block_pop(lib, a, b, rows, cols, wrap_rows, gens, k, count_row0, count_rows, pop, stream) -> bool:
    """_life_block that also writes pop (int64 [gens]): the live cells of rows [count_row0, count_row0 + count_rows)
    after each generation (cgl_life_run_pop: counted in the k-blocked kernels, no extra pass over the grid).
    Tests monkeypatch this for CPU runs."""
    res = ctypes.c_int(-1)
    native.check(lib.cgl_life_run_pop(native.dptr(a), native.dptr(b), rows, cols, wrap_rows, gens, k, count_row0,
                                      count_rows, native.dptr(pop), ctypes.byref(res), stream), "cgl_life_run_pop")
    return res.value == 1


class _null:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


class RowBandLife:
    def __init__(self, rows: int, cols: int, k: int = 8, rank: int = 0, world_size: int = 1, device="cuda",
                 exchange: str | None = None, group=None, lib=None, kernel_k: int | None = None):
        """k = ghost depth = generations between halo exchanges; kernel_k = generations per launch
        (temporal-blocking depth, default min(k, 8)): k = 16, kernel_k = 8 exchanges every 16
        generations and runs two 8-generation launches in between."""
        if rows % world_size:
            raise ValueError("rows must be divisible by world_size")
        if cols % 32:
            raise ValueError("cols must be a multiple of 32 for row bands")
        self.rows, self.cols, self.k = rows, cols, int(k)
        self.kernel_k = int(kernel_k) if kernel_k else min(self.k, 8)
        self.rank, self.G = rank, world_size
        self.W = cols // 32
        self.band_rows = rows // world_size
        if self.G > 1 and self.band_rows < self.k:
            raise ValueError("band must have at least k rows")
        self.device = torch.device(device)
        self.group = group
        self.lib = lib if lib is not None else native.load()
        if exchange is None:
            exchange = "single" if world_size == 1 else ("p2p" if self.device.type == "cuda" else "dist")
        self.exchange = exchange
        # a ring of ONE with exchange="p2p" keeps its ghost rows and exchanges with itself (its upper and lower
        # neighbour are the rank itself: the torus wrap) -- the exchange kernel on a single GPU (tests)
        self._self_ring = self.G == 1 and self.exchange == "p2p"
        g = self.k if (self.G > 1 or self._self_ring) else 0
        self.ghost = g
        self.buf_rows = self.band_rows + 2 * g
        n = self.buf_rows * self.W
        self.generation = 0
        self.block = 0              # exchanges done so far
        self.launches = 0
        self._ipc = None
        self._a = torch.zeros(n, dtype=torch.int32, device=self.device)
        self._b = torch.zeros(n, dtype=torch.int32, device=self.device)
        if self.exchange == "p2p" and (self.G > 1 or self._self_ring):
            self._setup_p2p()

    # ---------------------------------------------------------------- state access
    def _stream(self):
        if self.device.type != "cuda":
            return None
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def owned(self) -> torch.Tensor:
        """View of this rank's owned rows: int32 [band_rows, W] (bit-packed uint32 words)."""
        g, W = self.ghost, self.W
        return self._a[g * W:(g + self.band_rows) * W].view(self.band_rows, W)

    def set_owned(self, words: torch.Tensor) -> None:
        self.owned.copy_(words.view(self.band_rows, self.W))

    def randomize(self, seed: int = 0) -> None:
        """Synthetic Bernoulli(0.5) start: every packed word uniform, seeded by GLOBAL row so that the
        grid does not depend on the number of bands."""
        g = torch.Generator(device=self.device)
        chunk = 256 if self.band_rows % 256 == 0 else 1      # chunk starts are the same for every G
        r0 = self.rank * self.band_rows
        for s in range(0, self.band_rows, chunk):
            g.manual_seed(seed * 1000003 + (r0 + s))
            self.owned[s:s + chunk] = torch.randint(-2 ** 31, 2 ** 31 - 1, (chunk, self.W), dtype=torch.int32,
                                                    device=self.device, generator=g)

    # ---------------------------------------------------------------- P2P plumbing
    def _setup_p2p(self):
        """Allocate landing zones + flags with plain cudaMalloc, exchange IPC handles, map the neighbours'."""
        import torch.distributed as dist
        lib, k, W = self.lib, self.k, self.W
        strip = k * W * 4
        # layout: [slot0: from_up | from_down][slot1: from_up | from_down][flags: 4 x uint32 (+pad to 16)]
        total = 4 * strip + 64
        base = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            native.check(lib.cgl_dev_alloc(total, ctypes.byref(base)), "cgl_dev_alloc")
            handle = (ctypes.c_uint8 * 64)()
            native.check(lib.cgl_ipc_get_handle(base, handle), "cgl_ipc_get_handle")
        if self.G == 1:                                     # ring of one: my neighbours are me
            self._ipc = dict(base=base.value, strip=strip, up=base.value, down=base.value, flags_off=4 * strip, local=True)
            return
        handles = [None] * self.G
        dist.all_gather_object(handles, bytes(handle), group=self.group)
        up, down = (self.rank - 1) % self.G, (self.rank + 1) % self.G
        peers = {}
        with torch.cuda.device(self.device):
            for p in {up, down}:
                ptr = ctypes.c_void_p()
                h = (ctypes.c_uint8 * 64).from_buffer_copy(handles[p])
                native.check(lib.cgl_ipc_open_handle(h, ctypes.byref(ptr)), "cgl_ipc_open_handle")
                peers[p] = ptr.value
        self._ipc = dict(base=base.value, strip=strip, up=peers[up], down=peers[down], flags_off=4 * strip)
        dist.barrier(group=self.group)

    def close(self):
        if self._ipc:
            torch.cuda.synchronize(self.device)
            with torch.cuda.device(self.device):
                if not self._ipc.get("local"):
                    import torch.distributed as dist
                    dist.barrier(group=self.group)
                    for p in {self._ipc["up"], self._ipc["down"]}:
                        self.lib.cgl_ipc_close_handle(ctypes.c_void_p(p))
                self.lib.cgl_dev_free(ctypes.c_void_p(self._ipc["base"]))
            self._ipc = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False

    def __del__(self):
        try:
            if self._ipc and self._ipc.get("local"):        # (peer mappings need the collective close())
                self.close()
        except Exception:  # noqa: BLE001
            pass

    # ---------------------------------------------------------------- halo exchange
    def _exchange(self):
        """Fill the k ghost rows above/below the owned rows of the current buffer."""
        k, W, g = self.k, self.W, self.ghost
        if self.G == 1 and not self._self_ring:
            return
        a = self._a
        top_owned = a[g * W:(g + k) * W]                                     # my first k owned rows
        bot_owned = a[(g + self.band_rows - k) * W:(g + self.band_rows) * W]  # my last k owned rows
        ghost_up = a[0:k * W]
        ghost_down = a[(g + self.band_rows) * W:(g + self.band_rows + k) * W]
        self.block += 1
        if self.exchange == "dist":
            import torch.distributed as dist
            up, down = (self.rank - 1) % self.G, (self.rank + 1) % self.G
            send_up, send_down = top_owned.clone(), bot_owned.clone()
            ops = [dist.P2POp(dist.isend, send_up, up, group=self.group, tag=0),
                   dist.P2POp(dist.isend, send_down, down, group=self.group, tag=1),
                   dist.P2POp(dist.irecv, ghost_down, down, group=self.group, tag=0),   # neighbour's top rows
                   dist.P2POp(dist.irecv, ghost_up, up, group=self.group, tag=1)]       # neighbour's bottom rows
            for w in dist.batch_isend_irecv(ops):
                w.wait()
            return
        if self.exchange == "p2p":
            lib, ipc, st = self.lib, self._ipc, self._stream()
            strip, slot, seq = ipc["strip"], self.block & 1, self.block
            n_words = k * W
            # my top rows are the neighbour-above's "from_down" strip; my bottom rows the neighbour-below's "from_up"
            base, fo = ipc["base"], ipc["flags_off"]
            V = ctypes.c_void_p
            with torch.cuda.device(self.device):
                native.check(lib.cgl_halo_exchange(
                    native.dptr(top_owned), native.dptr(bot_owned),
                    V(ipc["up"] + (2 * slot + 1) * strip), V(ipc["down"] + (2 * slot) * strip),
                    V(ipc["up"] + fo + 4 * (2 * slot + 1)), V(ipc["down"] + fo + 4 * (2 * slot)),
                    V(base + (2 * slot) * strip), V(base + (2 * slot + 1) * strip),
                    V(base + fo + 4 * (2 * slot)), V(base + fo + 4 * (2 * slot + 1)),
                    native.dptr(ghost_up), native.dptr(ghost_down), n_words, seq, st), "cgl_halo_exchange")
            self.launches += 1
            return
        raise ValueError(f"unknown exchange {self.exchange!r}")

    # ---------------------------------------------------------------- stepping
    def run(self, gens: int, population: bool = False):
        """Advance `gens` generations (blocks of k generations between exchanges).  With population=True, return
        the global population after each generation of this call: int64 [gens] on this rank's device, the same
        on every rank (one all_reduce per call)."""
        lib, st = self.lib, self._stream()
        pop = torch.empty(gens, dtype=torch.int64, device=self.device) if population else None
        if self.device.type == "cuda" and not getattr(self, "_tuned", False):
            # measure the strip length of the k-blocked kernel for this band shape once (clobbers _b only)
            with torch.cuda.device(self.device):
                native.check(lib.cgl_life_tune(native.dptr(self._a), native.dptr(self._b),
                                               self.buf_rows, self.cols, 1 if self.ghost == 0 else 0, self.kernel_k,
                                               st), "cgl_life_tune")
            self._tuned = True
        if self.G == 1 and not self._self_ring:   # plain torus: one call, k generations per launch
            with torch.cuda.device(self.device) if self.device.type == "cuda" else _null():
                if population:
                    in_a = _life_block_pop(lib, self._a, self._b, self.band_rows, self.cols, 1, gens, self.kernel_k,
                                           0, self.band_rows, pop, st)
                else:
                    in_a = _life_block(lib, self._a, self._b, self.band_rows, self.cols, 1, gens, self.kernel_k, st)
                if not in_a:
                    self._a, self._b = self._b, self._a
            self.launches += -(-gens // self.kernel_k)
            self.generation += gens
            return pop
        done = 0
        while done < gens:
            kb = min(self.k, gens - done)
            self._exchange()
            with torch.cuda.device(self.device) if self.device.type == "cuda" else _null():
                if population:      # this block's generations, counted over the owned rows of the band buffer
                    in_a = _life_block_pop(lib, self._a, self._b, self.buf_rows, self.cols, 0, kb, min(kb, self.kernel_k),
                                           self.ghost, self.band_rows, pop[done:done + kb], st)
                else:
                    in_a = _life_block(lib, self._a, self._b, self.buf_rows, self.cols, 0, kb, min(kb, self.kernel_k), st)
                if not in_a:
                    self._a, self._b = self._b, self._a
            self.launches += -(-kb // self.kernel_k)
            done += kb
            self.generation += kb
        if population and self.G > 1:
            import torch.distributed as dist
            dist.all_reduce(pop, group=self.group)
        return pop

    # ---------------------------------------------------------------- global reductions
    def alive(self) -> int:
        """Global live-cell count (popcount of every rank's owned rows, summed over ranks)."""
        out = torch.zeros(1, dtype=torch.int32, device=self.device)
        owned = self.owned.contiguous()
        with torch.cuda.device(self.device):
            native.check(self.lib.cgl_alive(native.dptr(owned), 1, owned.numel(), native.dptr(out), self._stream()),
                         "cgl_alive")
        total = (out.to(torch.int64) & 0xFFFFFFFF)
        if self.G > 1:
            import torch.distributed as dist
            dist.all_reduce(total, group=self.group)
        n = int(total.item())
        if self.device.type == "cuda":
            native.check_alarm()                            # a device-side wait that gave up (see cgl_alarm_words)
        return n

    def checksum(self) -> int:
        """Order-independent 64-bit hash of the whole grid (sum over words of word * f(global index)),
        equal for any number of bands holding the same grid."""
        owned = self.owned.reshape(-1).to(torch.int64) & 0xFFFFFFFF
        r0 = self.rank * self.band_rows
        idx = torch.arange(owned.numel(), device=self.device, dtype=torch.int64) + r0 * self.W
        mix = (idx * 0x9E3779B1 + 0x7F4A7C15) & 0x7FFFFFFF
        total = ((owned * mix) & 0x7FFFFFFFFFFF).sum().reshape(1)
        if self.G > 1:
            import torch.distributed as dist
            dist.all_reduce(total, group=self.group)
        n = int(total.item())
        if self.device.type == "cuda":
            native.check_alarm()
        return n


class LocalBands:
    """G row bands held by ONE process/GPU, exchanged by local copies: same ghost-zone schedule as the
    multi-GPU path without peers (tests; also how a 1-GPU box checks the N-rank arithmetic)."""

    def __init__(self, rows, cols, k, n_bands, device="cuda", lib=None):
        self.bands = [RowBandLife(rows, cols, k=k, rank=r, world_size=n_bands, device=device, exchange="local", lib=lib)
                      for r in range(n_bands)]
        self.G, self.k = n_bands, k

    def set_grid(self, words: torch.Tensor) -> None:
        for b in self.bands:
            r0 = b.rank * b.band_rows
            b.set_owned(words.view(-1, b.W)[r0:r0 + b.band_rows])

    def grid(self) -> torch.Tensor:
        return torch.cat([b.owned for b in self.bands], dim=0)

    def run(self, gens: int, population: bool = False):
        """Advance every band `gens` generations; with population=True return the population of the whole grid
        after each generation (int64 [gens], the bands' owned-row counts summed)."""
        pops = [torch.empty(gens, dtype=torch.int64, device=b.device) for b in self.bands] if population else None
        done = 0
        while done < gens:
            kb = min(self.k, gens - done)
            tops = [b._a[b.ghost * b.W:(b.ghost + b.k) * b.W].clone() for b in self.bands]
            bots = [b._a[(b.ghost + b.band_rows - b.k) * b.W:(b.ghost + b.band_rows) * b.W].clone() for b in self.bands]
            for r, b in enumerate(self.bands):
                up, down = (r - 1) % self.G, (r + 1) % self.G
                b._a[0:b.k * b.W] = bots[up]
                b._a[(b.ghost + b.band_rows) * b.W:(b.ghost + b.band_rows + b.k) * b.W] = tops[down]
            for r, b in enumerate(self.bands):
                if population:
                    in_a = _life_block_pop(b.lib, b._a, b._b, b.buf_rows, b.cols, 0, kb, kb, b.ghost, b.band_rows,
                                           pops[r][done:done + kb], b._stream())
                else:
                    in_a = _life_block(b.lib, b._a, b._b, b.buf_rows, b.cols, 0, kb, kb, b._stream())
                if not in_a:
                    b._a, b._b = b._b, b._a
                b.generation += kb
            done += kb
        return torch.stack(pops).sum(0) if population else None
