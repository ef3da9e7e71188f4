"""CGL -- drop-in replacement for the reference's `CGL.py` module, B200-native.

Usage is the reference's own (/root/reference/CGL/main.py:1,29; bench.py:5,38): put this
directory on sys.path (or run the script from it) and

    import CGL
    env = CGL.sim(side=10, seed=0, gpu=True, spawnStabilityFactor=-2, stableStabilityFactor=2)
    env.toggle_state(action); env.step(); obs = env.get_stable(vector=True, shallow=True); r = env.reward()

Same constructor keywords, same methods, same exception classes as `class sim`
(/root/reference/CGL/CGL.py:53-354); every method below cites the lines it mirrors.  What
changed is everything underneath: the state lives ON THE DEVICE (bit-packed world + int8
stability, see DESIGN.md) and is stepped by libcgl_b200.so; numpy arrays are materialised at
the API boundary only.  There is no CPU path: `gpu=False` / `step(forceCPU=True)` raise, and a
missing CUDA library raises `cgl_b200.native.CglNativeError` at construction.

Deliberate deviations (all documented in DESIGN.md section 2):
  * cells must be 0/1 and the grid square (the reference lets other uint8 values and
    non-square sizes flow into its arithmetic unchecked, SURVEY.md N4) -> ValueError here;
  * shallow views are pinned host mirrors kept up to date by every state-changing call
    (reads see live state, aliasing `state is n_state` holds, CGL/main.py:60,70); writes INTO a
    shallow view do not reach the device -- use toggle_state / update_state / load;
  * a single-index toggle_state is applied lazily: it is passed BY VALUE to the next step() launch (one kernel
    does toggle + generation + stability + reward and stores the observation straight into the pinned mirror,
    cgl_sim_step), or applied by the next other call into the env; a shallow view shows it from that call on;
  * plain step() calls are deferred while no shallow view is live and executed together (one on-chip
    launch for the whole run of steps) when the state is next observed or changed -- same results, and
    the reference's `for _ in range(iters): env.step()` loop costs one launch.
"""
from __future__ import annotations

import os

import numpy as np

# Same environment switch as the reference (CGL/CGL.py:33-42).
if "GPU_CAPABLE" in os.environ:
    GPU_CAPABLE = os.environ["GPU_CAPABLE"].lower()
    if GPU_CAPABLE == "true":
        GPU_CAPABLE = True
    elif GPU_CAPABLE == "false":
        GPU_CAPABLE = False
    else:
        raise TypeError('GPU_CAPABLE must either be "TRUE" or "FALSE"!')
else:
    GPU_CAPABLE = True

_QUIET = os.environ.get("CGL_QUIET", "0") not in ("0", "", "false")


def _say(*a):
    if not _QUIET:
        print(*a)


def _check_int8(name, v):
    if not -128 <= v <= 127:
        # numpy 2 raises OverflowError at `stable[...] = spawn` (CGL/CGL.py:112, SURVEY.md N5)
        raise OverflowError(f"Python integer {v} out of bounds for int8 ({name})")


_NP_INT_TYPES = frozenset((np.int8, np.int16, np.int32, np.int64, np.uint8, np.uint16, np.uint32, np.uint64, np.intp))


class sim:
    """Conway's Game of Life environment with a per-cell int8 stability counter.

    Constructor arguments as in the reference (CGL/CGL.py:55): `state` (1-D/2-D ndarray of 0/1)
    or `side`+`seed` for the reference's random start; `gpu` must be True (and equal the
    GPU_CAPABLE environment switch); `gpu_select` is the CUDA device index; `warp` is accepted and
    validated for compatibility (launch geometry is chosen by the library)."""

    def __init__(self, state=None, side=8, seed=8, gpu=False, gpu_select=0, warp=8,
                 spawnStabilityFactor=-1, stableStabilityFactor=1):
        # ---- validation: same order and exception classes as CGL/CGL.py:57-82 -------------
        if not isinstance(state, np.ndarray) and state is not None and not isinstance(state, list):
            raise TypeError("state variable must be a list or Numpy ndarray!")
        if not isinstance(side, int):
            raise TypeError("side must be integer!")
        if side < 1:
            raise ValueError("side must be positive integer greater than 0!")
        if not isinstance(seed, int):
            raise TypeError("seed must be integer!")
        if seed < 0:
            raise ValueError("seed must be positive integer!")
        if not isinstance(gpu, bool):
            raise TypeError("gpu must be bool!")
        if not isinstance(warp, int):
            raise TypeError("warp must be integer!")
        if warp < 0:
            raise ValueError("warp must be positive integer!")
        if not isinstance(spawnStabilityFactor, int):
            raise TypeError("spawnStabilityFactor must be an integer!")
        if not isinstance(stableStabilityFactor, int):
            raise TypeError("stableStabilityFactor must be an integer!")
        if GPU_CAPABLE != gpu:
            raise TypeError(f'the os enviornment variable "GPU_CAPABLE" (defaults to true) is {GPU_CAPABLE} and '
                            f'"gpu" is {gpu}. Both must be equal in value!\n'
                            'To launch use: GPU_CAPABLE="true\\false" python3 <script.py>')
        if not gpu:
            raise RuntimeError("this build of CGL is GPU-only (B200-native, no CPU step): construct with gpu=True "
                               "and GPU_CAPABLE=true, or import the reference CGL.py for its CPU loop")

        self.count = 0
        self.seed = seed
        self.spawnStabilityFactor = spawnStabilityFactor
        self.stableStabilityFactor = stableStabilityFactor
        self.gpu = gpu

        if state is not None:
            state = state.flatten().astype(np.uint8)       # lists fail here like the reference (:94, N4)
            if state.size == 0:
                raise ValueError("state must be size greater than 0!")
            world0 = self._validated_cells(state)
            self.size = world0.size
            self.side = int(np.sqrt(self.size))
            if self.side * self.side != self.size:
                raise ValueError(f"state must be square: got {self.size} cells")
        else:
            self.side = side
            self.size = side ** 2
            world0 = None
        _check_int8("spawnStabilityFactor", spawnStabilityFactor)
        _check_int8("stableStabilityFactor", stableStabilityFactor)

        # ---- device setup (replaces CGL/CGL.py:116-195) ------------------------------------
        import torch
        from cgl_b200 import native
        from cgl_b200.batched import BatchedSim
        self._torch = torch
        native.load()                                       # fail loudly before touching the device
        if not torch.cuda.is_available():
            raise native.CglNativeError("no CUDA device visible: CGL.sim(gpu=True) needs a GPU (no CPU fallback)")
        n_dev = torch.cuda.device_count()
        if not isinstance(gpu_select, int) or gpu_select < 0 or gpu_select > n_dev - 1:
            raise ValueError(f"gpu_select={gpu_select}, however the device which can be chosen are: {range(n_dev)}.")
        prop = torch.cuda.get_device_properties(gpu_select)
        _say("Number of devices detected:", n_dev)
        _say("Device selected:", gpu_select)
        _say("\tName:", prop.name)
        _say("\tCompute capability:", (prop.major, prop.minor))
        _say("\tTotal memory:", prop.total_memory / 1048576, "MB")
        _say("\tSMs:", prop.multi_processor_count)
        self._dev = torch.device("cuda", gpu_select)
        if world0 is None:
            world0 = self._initial_world()
        self._b = BatchedSim(1, self.side, seed=seed, spawnStabilityFactor=spawnStabilityFactor,
                             stableStabilityFactor=stableStabilityFactor, device=self._dev,
                             states=None if world0 is None else world0[None, :], **self._env_variant())
        self._alloc_mirrors()
        _say("CGL is now running...")

    # ------------------------------------------------------------------------------ internals
    _serving = False                                        # a resident step server (cgl_sim_serve) may be alive
    _bs = None

    @property
    def _b(self):
        """The batched driver that owns the device planes.  Every path that lets OTHER kernels touch the planes goes
        through this property, which first makes the resident step server hand the state back (no-op otherwise);
        the step path itself uses `_bs`."""
        if self._serving:
            self._serve_stop()
        return self._bs

    @_b.setter
    def _b(self, value):
        if self._serving:
            self._serve_stop()
        self._bs = value

    def __del__(self):
        try:                                                # the server reads our pinned buffers: stop it before they go
            if self._serving:
                self._serve_stop()
        except Exception:  # noqa: BLE001
            pass

    def _env_variant(self):
        """Extra BatchedSim keywords; the CGL_action+ facade overrides this (dead-cell rule, masked toggle)."""
        return {}

    def _initial_world(self):
        """None = the reference's seeded random start (CGL/CGL.py:104-107); a subclass may return cells."""
        return None

    @staticmethod
    def _validated_cells(flat_u8: np.ndarray) -> np.ndarray:
        if flat_u8.size and flat_u8.max() > 1:
            raise ValueError("cells must be 0 or 1 (bit-packed device state); got values > 1")
        return np.ascontiguousarray(flat_u8)

    def _alloc_mirrors(self):
        torch = self._torch
        self._m_world_t = torch.empty(self.size, dtype=torch.uint8).pin_memory()
        self._m_stable_t = torch.empty(self.size, dtype=torch.int8).pin_memory()
        self._m_world = self._m_world_t.numpy()
        self._m_stable = self._m_stable_t.numpy()
        self._world_fresh = self._stable_fresh = False
        self._world_live = self._stable_live = False       # a shallow view has been handed out
        # result block of the one-launch step (cgl_sim_step): the kernel writes reward, live count and then the
        # step's sequence number into this pinned, host-mapped memory; the host polls the sequence word
        self._res_t = torch.zeros(8, dtype=torch.int32).pin_memory()
        self._res = self._res_t.numpy()
        self._seq = 0
        # resident step server (cgl_sim_serve): the host posts (seq << 32) | action into this pinned word and the
        # kernel answers in the result block; _res[4] == _launch_id means that launch has left
        self._cmd_t = torch.zeros(2, dtype=torch.int64).pin_memory()
        self._cmd = self._cmd_t.numpy().view(np.uint64)
        # the hot loop reads and writes single words of these blocks: memoryviews hand out plain Python ints
        self._res_w = memoryview(self._res)
        self._cmd_w = memoryview(self._cmd)
        self._launch_id = 0
        self._serve_stream = None
        self._pending_seq = None                            # sequence number of a step whose results are in flight
        self._pending = None                                # scalar toggle deferred into the next step()
        self._lazy_steps = 0                                # plain steps not yet executed (see step())
        self._reward_valid = False                          # _res[0] holds reward() of the current state
        self._alive_valid = False                           # _res[1] holds alive() of the current state
        lib = self._bs._lib
        self._fast = self.side <= int(lib.cgl_sim_step_max_side())
        self._fast_args = {}
        self._linger_us = max(0, min(100000, int(os.environ.get("CGL_SIM_LINGER_US", "250"))))
        self._serve_ok = self._fast and self._linger_us > 0 and self.side <= int(lib.cgl_sim_serve_max_side())

    def _invalidate(self):
        """The state changed by something other than a step: cached reward / live count are stale."""
        self._reward_valid = self._alive_valid = False

    def _wait(self):
        """Block until the last one-launch step has delivered observation mirror, reward and live count: poll the
        sequence word the kernel writes last (no stream synchronisation, no copy)."""
        seq = self._pending_seq
        if seq is None:
            return
        res = self._res_w
        if res[2] != seq:
            spins = 0
            while res[2] != seq:
                spins += 1
                if self._serving:
                    if res[4] == self._launch_id:           # the server has left (idle for too long) ...
                        if res[2] != seq:                   # ... before it saw this command: launch it again
                            self._serve_launch((seq - 1) & 0x3fffffff)
                    elif spins > 4000000:
                        self._serve_stream.synchronize()
                        raise RuntimeError("CGL.sim: the resident step kernel does not answer")
                elif spins > 200000:                        # ~50 ms: something is wrong, let CUDA report it
                    self._torch.cuda.current_stream(self._dev).synchronize()
                    if res[2] != seq:
                        raise RuntimeError("CGL.sim: the step kernel finished without delivering its results")
        self._pending_seq = None

    def _step_args(self):
        """The cached cgl_sim_step_args_t of this env (constants and pointers; rebuilt after load())."""
        args = self._fast_args.get("args")
        if args is None:
            import ctypes
            from cgl_b200 import native
            from cgl_b200.batched import DEAD_RULES
            b = self._bs
            st = native.SimStepArgs()
            st.world_a, st.world_b, st.stable = b._wa.data_ptr(), b._wb.data_ptr(), b.stable.data_ptr()
            st.side, st.spawn, st.stable_max = self.side, b.spawn, b.stable_max
            st.dead_rule, st.empty, st.empty_min = DEAD_RULES[b.dead_rule], b.empty, b.empty_min
            st.masked_toggle = int(b.masked_toggle)
            st.obs_mirror, st.result = self._m_stable_t.data_ptr(), self._res_t.data_ptr()
            flip = ctypes.c_uint32(0)                        # even: the world is in the plane that is `world_a` here
            st.flip_planes = ctypes.pointer(flip)
            raw = getattr(self._torch._C, "_cuda_getCurrentRawStream", None)
            args = (st, ctypes.byref(st), flip, b._lib.cgl_sim_step_ex, raw, self._dev.index, b._wa.data_ptr(),
                    b._lib.cgl_sim_serve, self._cmd_t.data_ptr())
            self._fast_args["args"] = args
        # the planes this struct was built from may have been swapped by other calls (run, batched step, ...)
        want_odd = self._bs._wa.data_ptr() != args[6]
        if bool(args[2].value & 1) != want_odd:
            args[2].value = int(want_odd)
        return args

    def _serve_launch(self, last_seq):
        """(Re)launch the resident step server on its own non-blocking stream, ordered after whatever the current
        stream still has queued on the planes."""
        torch = self._torch
        args = self._step_args()
        with torch.cuda.device(self._dev):
            if self._serve_stream is None:
                self._serve_stream = torch.cuda.Stream(device=self._dev)
            self._serve_stream.wait_stream(torch.cuda.current_stream(self._dev))
            self._launch_id = lid = self._launch_id % 0x3fffffff + 1
            rc = args[7](args[1], args[8], last_seq, lid, self._linger_us, self._serve_stream.cuda_stream)
        if rc:
            from cgl_b200 import native
            native.check(rc, "cgl_sim_serve")
        self._bs.launches += 1
        self._serving = True

    def _serve_stop(self):
        """Make the resident server write the planes back and leave; afterwards the device planes are current."""
        if not self._serving:
            return
        self._wait()
        res, lid = self._res_w, self._launch_id
        if res[4] != lid:
            self._seq = seq = (self._seq + 1) & 0x3fffffff
            self._cmd_w[0] = (seq << 32) | 0xFFFFFFFE        # CGL_SIM_QUIT
            spins = 0
            while res[4] != lid:
                spins += 1
                if spins > 4000000:
                    self._serve_stream.synchronize()
                    if res[4] != lid:
                        raise RuntimeError("CGL.sim: the resident step kernel did not leave")
        self._serving = False

    def _flush(self):
        """Bring the device state up to date with everything the caller has asked for so far: run the plain
        steps that were deferred (see step()), then apply a deferred scalar toggle (anything that observes the
        state between toggle_state and step must see it, SURVEY.md N2)."""
        self._run_lazy()
        if self._pending is not None:
            a, self._pending = self._pending, None
            self._wait()
            self._b.toggle(self._torch.tensor([[a]], dtype=self._torch.int32, device=self._dev))
            self._invalidate()
            self._changed()

    def _run_lazy(self):
        n, self._lazy_steps = self._lazy_steps, 0
        if n == 1:
            self._step_now()
        elif n > 1:                 # the whole run of plain steps is ONE launch with the env resident on chip
            self._wait()
            with self._torch.cuda.device(self._dev):
                _, rew, _ = self._b.run(n)
                self._res_t[0:1].copy_(rew)                 # blocking copy: the run is long, the sync is not
            self._reward_valid, self._alive_valid = True, False
            self._changed()

    def _changed(self, world=True, stable=True):
        """Device state changed: invalidate mirrors, eagerly refresh the ones with live views."""
        if world:
            self._world_fresh = False
            if self._world_live:
                self._sync_world()
        if stable:
            self._stable_fresh = False
            if self._stable_live:
                self._sync_stable()

    def _sync_world(self):
        if not self._world_fresh:
            self._m_world_t.copy_(self._b.get_state().view(-1))
            self._world_fresh = True
        return self._m_world

    def _sync_stable(self):
        if not self._stable_fresh:
            self._wait()
            self._m_stable_t.copy_(self._b.stable.view(-1))
            self._stable_fresh = True
        else:
            self._wait()                                    # the mirror is being written by the step in flight
        return self._m_stable

    # reference attribute names (read access): live host views of the device state
    @property
    def world(self):
        self._flush()
        self._world_live = True
        return self._sync_world()

    @property
    def stable(self):
        self._flush()
        self._stable_live = True
        return self._sync_stable()

    @property
    def initState(self):
        torch = self._torch
        from cgl_b200 import native
        out = torch.empty((1, self.size), dtype=torch.uint8, device=self._dev)
        native.check(self._b._lib.cgl_unpack(native.dptr(self._b._init_world), native.dptr(out), 1, self.side,
                                             self.side, self._b._stream()), "cgl_unpack")
        return out.cpu().numpy().reshape(-1)

    @property
    def initStable(self):
        return self._b._init_stable.cpu().numpy().reshape(-1)

    # ------------------------------------------------------------------------------ simulator
    def step(self, forceCPU=False):
        """One generation + stability update (CGL/CGL.py:247-252; kernel :147-181).

        A plain step (no toggle pending) while nobody holds a live shallow view is only COUNTED here and
        executed when the state is next observed or changed (reward, alive, get_*, toggle_state, ...): a loop
        like the reference's `for _ in range(iters): env.step()` (CGL/bench.py:39-40) becomes one launch of
        `cgl_env_run(iters)` with the env resident on chip.  Results are bit-identical either way."""
        if forceCPU:
            raise RuntimeError("forceCPU is not available in the B200 build (no CPU step); use the reference for that")
        self.count += 1
        if self._pending is None and not (self._world_live or self._stable_live) and self._can_defer:
            self._lazy_steps += 1
            self._invalidate()
            self._world_fresh = self._stable_fresh = False
            return
        if self._lazy_steps:
            self._run_lazy()
        if self._serving and self._pending_seq is None and not self._world_live:
            # the DQN loop's step on the resident server, inlined (_step_now is the general form): post the command,
            # mark what the kernel is about to deliver, wait for the answer if a live view has to show it
            a = self._pending
            if a is None:
                a = self.size
            else:
                self._pending = None
            self._seq = seq = (self._seq + 1) & 0x3fffffff
            res = self._res_w
            self._cmd_w[0] = (seq << 32) | a
            if res[4] == self._launch_id:                   # it has left in the meantime (idle): launch it again
                self._serve_launch((seq - 1) & 0x3fffffff)
            self._bs.count += 1
            self._reward_valid = self._alive_valid = self._stable_fresh = True
            self._world_fresh = False
            if self._stable_live and res[2] == seq:
                return
            self._pending_seq = seq
            if self._stable_live:
                self._wait()
            return
        self._step_now()

    def _step_now(self):
        """toggle (if one is pending) + generation + stability + reward + live count.  Sides the resident server
        takes (cgl_sim_serve): the action is posted into a pinned command word and a kernel that keeps the env on
        chip answers -- no launch per step.  Otherwise ONE launch (cgl_sim_step): the action travels by value.
        Either way the new observation is stored by the kernel into the pinned mirror and reward / live count /
        sequence number into the pinned result block."""
        a = self.size                                       # "do nothing"
        if self._pending is not None:
            a, self._pending = self._pending, None
        if not self._fast:
            return self._step_now_batched(a)
        b = self._bs
        if self._pending_seq is not None:
            self._wait()                                    # one step in flight at a time (the result block is shared)
        self._seq = seq = (self._seq + 1) & 0x3fffffff
        if self._serve_ok and not self._world_live:
            self._cmd_w[0] = (seq << 32) | a
            if not self._serving or self._res_w[4] == self._launch_id:
                self._serve_launch((seq - 1) & 0x3fffffff)
        else:
            if self._serving:
                self._serve_stop()
            args = self._step_args()
            torch = self._torch
            if torch.cuda.current_device() != self._dev.index:
                torch.cuda.set_device(self._dev)
            stream = args[4](args[5]) if args[4] is not None else torch.cuda.current_stream(self._dev).cuda_stream
            rc = args[3](args[1], a, seq, stream)
            if rc:
                from cgl_b200 import native
                native.check(rc, "cgl_sim_step")
            b._wa, b._wb = b._wb, b._wa
            b.launches += 1
        b.count += 1
        self._pending_seq = seq
        self._reward_valid = self._alive_valid = True
        self._stable_fresh = True                           # valid once _wait() has seen the sequence number
        self._world_fresh = False
        if self._stable_live:
            self._wait()                                    # a live view must show the new state when step() returns
        if self._world_live:
            self._sync_world()

    def _step_now_batched(self, a):
        """Sides above cgl_sim_step's limit: the batched kernels (toggle, generation, stability), then copies."""
        torch, b = self._torch, self._b
        with torch.cuda.device(self._dev):
            act = None if a == self.size else torch.tensor([a], dtype=torch.int32, device=self._dev)
            _, rew, _ = b.step(act)
            self._res_t[0:1].copy_(rew)
        self._reward_valid, self._alive_valid = True, False
        self._changed()

    @property
    def _can_defer(self):
        return self._bs.fused or self.side <= 274           # sides cgl_env_run can keep on chip

    # ---- extensions (not in CGL/CGL.py): the reference's own loops around step(), run on the device ----
    def run(self, iters, until_fixed=False):
        """`iters` plain steps in one launch (the loop of CGL/bench.py:39-40); with until_fixed stop after
        the first step that leaves the world unchanged (CGL_action+/validate.py:133-139).  Returns the
        number of steps executed; `count` advances by it."""
        self._flush()
        self._wait()
        with self._torch.cuda.device(self._dev):
            _, rew, steps = self._b.run(int(iters), until_fixed=until_fixed)
            n = int(steps.item())
            self._res[0] = int(rew.item())
        self.count += n
        self._reward_valid, self._alive_valid = True, False
        self._changed()
        return n

    def run_until_cycle(self, iters, max_period=2):
        """`run(iters, until_fixed=True)` that also stops when the world repeats one of its last max_period
        (1..8) worlds: after the first step t with world_t == world_{t-p}, p <= max_period, the world when the
        call starts counting as world_0.  Returns (steps executed, p), p = 0 if no step in `iters` matched; a
        spaceship reports 0 until it has crossed the torus.  `count` advances by the steps."""
        self._flush()
        self._wait()
        with self._torch.cuda.device(self._dev):
            period = self._torch.zeros(1, dtype=self._torch.int32, device=self._dev)
            _, rew, steps = self._b.run(int(iters), max_period=int(max_period), period_out=period)
            n, p = int(steps.item()), int(period.item())
            self._res[0] = int(rew.item())
        self.count += n
        self._reward_valid, self._alive_valid = True, False
        self._changed()
        return n, p

    def run_until_settled(self, iters):
        """`run_until_cycle` without a bound on the period: stops after the first step t whose world equals any
        earlier world, the world when the call starts counting as world_0.  Returns (steps executed, p): p is the
        exact period of the cycle the world entered (a glider's is 4*side), 0 if no step in `iters` repeated a
        world.  `count` advances by the steps."""
        self._flush()
        self._wait()
        with self._torch.cuda.device(self._dev):
            period = self._torch.zeros(1, dtype=self._torch.int32, device=self._dev)
            _, rew, steps = self._b.run(int(iters), until_settled=True, period_out=period)
            n, p = int(steps.item()), int(period.item())
            self._res[0] = int(rew.item())
        self.count += n
        self._reward_valid, self._alive_valid = True, False
        self._changed()
        return n, p

    def action_rewards(self):
        """np.int32[size + 1]: entry a is what `toggle_state(a); step(); reward()` would return from the current
        state (CGL/main.py:66-71), entry `size` the no-op's.  Nothing is stepped or toggled; a deferred toggle and
        deferred steps are applied first, as for any other observation of the state."""
        self._flush()
        b = self._b                                         # (stops a resident step server: the planes are current)
        with self._torch.cuda.device(self._dev):
            return b.action_rewards()[0].cpu().numpy()

    def breakdown_stable(self):
        """np.asarray((unique values, counts)) of the stability vector (CGL_action+/CGL.py:294-297)."""
        self._flush()
        hist = self._b.breakdown_stable()[0].cpu().numpy()
        vals = np.nonzero(hist)[0]
        return np.asarray(((vals - 128).astype(np.int8), hist[vals]))

    def breakdown_state(self):
        """np.asarray((unique values, counts)) of the world (CGL_action+/CGL.py:300-303)."""
        self._flush()
        dead, live = (int(v) for v in self._b.breakdown_state()[0].cpu())
        vals = [v for v, c in ((0, dead), (1, live)) if c]
        return np.asarray((np.array(vals, dtype=np.uint8), np.array([c for c in (dead, live) if c])))

    def reward(self):
        """np.int32 sum of the stability vector (CGL/CGL.py:255-256)."""
        if self._lazy_steps or self._pending is not None:
            self._flush()
        if self._reward_valid:                              # written by the last step's kernel
            if self._pending_seq is not None:
                self._wait()
            return self._res[0]                            # (indexing the int32 block yields an np.int32)
        return np.int32(self._b.reward().item())

    def alive(self):
        """np.uint32 number of live cells (CGL/CGL.py:259-260)."""
        self._flush()
        if self._alive_valid:                               # written by the last step's kernel
            self._wait()
            return np.uint32(self._res[1])
        return np.uint32(self._b.alive().item())

    def reset(self):
        """Back to the initial state; `count` is not reset (CGL/CGL.py:264-266)."""
        self._pending = None
        self._lazy_steps = 0                                # whatever was still owed is overwritten by the reset
        self._wait()
        self._invalidate()
        self._b.reset()
        self._changed()

    def match(self, terminalState):
        """(world == terminalState.flatten()).all()  (CGL/CGL.py:269-270)."""
        self._flush()
        flat = np.asarray(terminalState).flatten()
        if flat.size != self.size:
            raise ValueError(f"terminalState has {flat.size} cells, expected {self.size}")
        if flat.size and (flat.min() < 0 or flat.max() > 1 or np.any(flat != flat.astype(np.uint8))):
            return False                                    # the world is binary: cannot be equal
        return self._b.match(self._torch.from_numpy(np.ascontiguousarray(flat.astype(np.uint8)))[None, :])

    # ------------------------------------------------------------------------------ I/O
    def get_state(self, vector=False, shallow=False):
        """World as uint8 vector or (side, side) matrix (CGL/CGL.py:274-278)."""
        self._flush()
        if shallow:
            self._world_live = True
        w = self._sync_world()
        out = w if vector else w.reshape((self.side, self.side))
        return out if shallow else np.copy(out)

    def get_stable(self, vector=False, shallow=False):
        """Stability (the observation) as int8 vector or matrix (CGL/CGL.py:281-285)."""
        if self._lazy_steps or self._pending is not None:
            self._flush()
        if shallow:
            self._stable_live = True
        if self._stable_fresh:                              # the step's kernel wrote the mirror itself
            if self._pending_seq is not None:
                self._wait()
            s = self._m_stable
        else:
            s = self._sync_stable()
        out = s if vector else s.reshape((self.side, self.side))
        return out if shallow else np.copy(out)

    def get_side(self):
        return self.side

    def get_count(self):
        return self.count

    def get_seed(self):
        return self.seed

    def get_state_dim(self):
        return self.size

    def get_state_space_dim(self):
        return 2 ** self.size

    def get_action_space_dim(self):
        return self.size + 1        # the last action is "do nothing" (CGL/CGL.py:308-309)

    def update_state(self, newState, side):
        """Replace the world, keep the stability plane (CGL/CGL.py:312-317)."""
        temp = newState.flatten().astype(np.uint8)
        if temp.size != self.size or self.side != side:
            raise ValueError("The new state must have the same size and side as the original state!\n"
                             f"Was given size={temp.size} and side={side} but was expecting size={self.size} and side={self.side}.")
        cells = self._validated_cells(temp)
        self._flush()
        self._wait()
        self._alive_valid = False
        self._b.set_state(self._torch.from_numpy(cells)[None, :].to(self._dev))
        self._changed(world=True, stable=False)

    def toggle_state(self, indx):
        """Toggle the listed cells and set their stability to spawn (CGL/CGL.py:322-328).
        Duplicates toggle once; the scalar `size` is the silent "do nothing"; anything else out of
        range raises ValueError."""
        t = type(indx)
        if t is int or t in _NP_INT_TYPES or (isinstance(indx, (int, np.integer)) and not isinstance(indx, bool)):
            # the DQN loop's case (CGL/main.py:66-67): one index, then step().  The toggle is deferred and
            # travels by value into that launch.  Every other call into the env applies it first (_flush), so
            # the only place it is not yet visible is a shallow numpy view read before the next call.
            a = int(indx)
            if 0 <= a < self.size:
                if self._lazy_steps or self._pending is not None:
                    self._flush()                           # an earlier deferred toggle goes first
                self._pending = a
                self._reward_valid = self._alive_valid = False
            elif a != self.size:
                raise ValueError("Not all indexes are valid!\nIndexes must be positive and less than the size of the "
                                 f"state {self.size}.")
            return
        indx = np.array(indx)
        if np.all(indx < self.size) and np.all(indx >= 0):
            if indx.dtype.kind not in "iu":
                raise IndexError("arrays used as indices must be of integer (or boolean) type")
            flat = np.ascontiguousarray(indx.reshape(-1), dtype=np.int32)
            self._flush()                                   # an earlier deferred toggle goes first
            if flat.size == 1:
                self._pending = int(flat[0])
                self._invalidate()
            elif flat.size:
                self._wait()
                self._b.toggle(self._torch.from_numpy(flat).to(self._dev)[None, :])
                self._invalidate()
                self._changed()
        elif indx != self.size:     # an array with >1 element raises ValueError here, like the reference
            raise ValueError("Not all indexes are valid!\nIndexes must be positive and less than the size of the "
                             f"state {self.size}.")

    def save(self):
        """(world, stable, side, count, spawn, stable_max) -- host copies (CGL/CGL.py:332-333)."""
        self._flush()
        return (np.copy(self._sync_world()), np.copy(self._sync_stable()), self.side, self.count,
                self.spawnStabilityFactor, self.stableStabilityFactor)

    def load(self, newState, newstable, side, count, spawnStabilityFactor, stableStabilityFactor):
        """Restore an exact setup (CGL/CGL.py:336-354); device buffers are re-created if `side` changed."""
        if not isinstance(newState, np.ndarray) or not isinstance(newstable, np.ndarray):
            raise TypeError("newState and newstable variables must be a Numpy ndarray!")
        if not isinstance(side, int) or not isinstance(count, int):
            raise TypeError("side and count must be integer!")
        if side < 1 or count < 0:
            raise ValueError("side and count must be positive integers and side greater than 0!")
        if not isinstance(spawnStabilityFactor, int):
            raise TypeError("spawnStabilityFactor must be an integer!")
        if not isinstance(stableStabilityFactor, int):
            raise TypeError("stableStabilityFactor must be an integer!")
        _check_int8("spawnStabilityFactor", spawnStabilityFactor)
        _check_int8("stableStabilityFactor", stableStabilityFactor)
        cells = self._validated_cells(newState.flatten().astype(np.uint8))
        stab = np.ascontiguousarray(newstable.flatten().astype(np.int8))
        if cells.size != side * side or stab.size != side * side:
            raise ValueError(f"newState/newstable must have side*side = {side * side} cells")
        from cgl_b200.batched import BatchedSim
        self._pending = None
        self._lazy_steps = 0
        self._wait()
        self._invalidate()
        self._fast_args.clear()                             # the launch arguments cache the constants
        self.stableStabilityFactor = stableStabilityFactor
        self.spawnStabilityFactor = spawnStabilityFactor
        resized = side != self.side
        self.size = side ** 2
        self.side = side
        self.count = count
        if resized:
            self._b = BatchedSim(1, side, seed=self.seed, spawnStabilityFactor=spawnStabilityFactor,
                                 stableStabilityFactor=stableStabilityFactor, device=self._dev, states=cells[None, :],
                                 **self._env_variant())
            self._alloc_mirrors()
        else:
            self._b.set_factors(spawnStabilityFactor, stableStabilityFactor)
            self._b.set_state(self._torch.from_numpy(cells)[None, :].to(self._dev))
        self._b.stable.copy_(self._torch.from_numpy(stab)[None, :])
        self._changed()
