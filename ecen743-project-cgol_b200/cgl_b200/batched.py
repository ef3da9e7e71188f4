"""BatchedSim -- B independent Game-of-Life environments resident on one B200.

Device layout (DESIGN.md section 3):
  world   uint32 [B, side, W]   1 bit per cell, W = ceil(side/32), two ping-pong planes
  stable  int8   [B, side*side] the reference's row-major stability vector == the observation
All stepping goes through libcgl_b200.so (`cgl_env_step`); torch only owns memory and streams.

Semantics per env are those of the reference's `sim` (/root/reference/CGL/CGL.py):
toggle_state (:322-328) -> step (:247-252, kernel :147-181) -> reward (:255-256) / get_stable
(:281-285), i.e. the body of the DQN loop CGL/main.py:64-72, for all envs in one launch.

Sharding by env index (multi-GPU, no communication): `BatchedSim.shard(...)` gives rank r the
envs [r*B/G, (r+1)*B/G); env e is always seeded `seed + e` with its GLOBAL index, so results
do not depend on the number of GPUs.

Beyond the single step (SURVEY.md section 8f):
  step(obs_out=, reward_out=)   the new observation goes straight into a caller buffer (replay ring, dqn.py)
  run(k, until_fixed=)          k plain steps / run-until-fixed in one launch, env resident on chip
  run(k, actions=, reward_trace=, alive_trace=)   k steps following an action schedule, every step's reward recorded
  run(k, ..., obs_trace=)       and every step's observation, written straight into a caller buffer (replay ring)
  run(k, max_period=P)          run until each world repeats one of its last P worlds (its cycle length -> period_out)
  run(k, until_settled=True)    run until each world repeats any earlier world (steps to settle, exact period)
  action_rewards() / greedy_actions()   every action's next-step reward, and the one-step greedy action, without stepping
  dead_rule=, empty=, empty_min=, masked_toggle=   the CGL_action+ fork's env
  breakdown_stable / breakdown_state, block_action, save_checkpoint / load_checkpoint, step_host(sync=False)
"""
from __future__ import annotations

import ctypes
import os

import numpy as np
import torch

from . import native


DEAD_RULES = {"zero": 0, "decay": 1, "sat": 2}

# State planes of a BatchedSim that go to hardware-compressed device memory where the device offers it (DESIGN.md
# section 3): "stable" and/or "world" (both bit planes).  Measured on B200 (tools/compressible_probe.py): the mostly
# zero stability plane takes the C2 step from 24.3 to 20.1 us; the world planes (random bits) add no gain beyond the
# spread of the regions, so they stay plain.
COMPRESSED_PLANES = ("stable",)


def reference_initial_world(side: int, seed: int) -> np.ndarray:
    """The reference's random start: CGL/CGL.py:104-107 (legacy MT19937 `np.random.seed`)."""
    return np.random.RandomState(seed).randint(2, size=side * side, dtype=np.uint8)


class BatchedSim:
    def __init__(self, n_envs: int, side: int, seed: int = 0, spawnStabilityFactor: int = -1,
                 stableStabilityFactor: int = 1, device="cuda", states=None, first_env: int = 0,
                 rng: str = "reference", max_steps: int | None = None, dead_rule: str = "zero", empty: int = 0,
                 empty_min: int = -128, masked_toggle: bool = False, _compressed_planes=None):
        if not isinstance(n_envs, int) or n_envs < 1:
            raise ValueError("n_envs must be a positive integer")
        if not isinstance(side, int) or side < 1:
            raise ValueError("side must be positive integer greater than 0!")
        for name, v in (("spawnStabilityFactor", spawnStabilityFactor), ("stableStabilityFactor", stableStabilityFactor)):
            if not isinstance(v, int):
                raise TypeError(f"{name} must be an integer!")
            if not -128 <= v <= 127:
                raise OverflowError(f"{name}={v} out of bounds for int8")
        # The CGL_action+ fork's variants (CGL/CGL_action+/CGL.py): what a cell that is dead after the step gets
        # ("zero" = base env; "decay" = the fork's CUDA kernel :190-193; "sat" = the fork's CPU step :256), the
        # initial stability of dead cells, and the masked toggle (:382-384).  See cgl_env_step_rule.
        if dead_rule not in DEAD_RULES:
            raise ValueError(f"dead_rule must be one of {sorted(DEAD_RULES)}")
        for name, v in (("empty", empty), ("empty_min", empty_min)):
            if not isinstance(v, int):
                raise TypeError(f"{name} must be integer!")
            if not -128 <= v <= 127:
                raise OverflowError(f"{name}={v} out of bounds for int8")
        self.dead_rule, self.empty, self.empty_min = dead_rule, empty, empty_min
        self.masked_toggle = bool(masked_toggle)
        self._ext = DEAD_RULES[dead_rule] != 0 or self.masked_toggle
        self._lib = native.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise native.CglNativeError("BatchedSim needs a CUDA device (there is no CPU fallback)")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.n_envs, self.side, self.size = n_envs, side, side * side
        self.W = (side + 31) // 32
        self.seed, self.first_env, self.rng = seed, first_env, rng
        self.spawn, self.stable_max = spawnStabilityFactor, stableStabilityFactor
        self.count = 0
        self.max_steps = max_steps
        self.fused = bool(self._lib.cgl_env_step_is_fused(side))
        self.launches = 0                                   # kernels launched so far (bench evidence)

        with torch.cuda.device(self.device):
            B, size, W = n_envs, self.size, self.W
            self._alarm = native.alarm()                    # host-mapped alarm words, installed on this device
            compress = COMPRESSED_PLANES if _compressed_planes is None else tuple(_compressed_planes)
            self._wa = self._state_plane((B, side, W), torch.int32, "world" in compress)
            self._wb = self._state_plane((B, side, W), torch.int32, "world" in compress)
            self.stable = self._state_plane((B, size), torch.int8, "stable" in compress)
            self._reward = torch.zeros(B, dtype=torch.int32, device=self.device)
            self._alive = torch.zeros(B, dtype=torch.int32, device=self.device)   # uint32 bits
            self._err = torch.zeros(1, dtype=torch.int32, device=self.device)
            # Per-env tokens of the chained fused step (include/cgl_b200.h, chain_mode).  Default: SEQUENCE
            # NUMBERS -- token[e] = number of chained steps env e has completed, `_seq` is the host counter the
            # library reads `want` from.  A step issued under CUDA stream capture switches the batch to PLANE IDS
            # for good (token[e] = id of the plane holding env e's world: 1 = first plane, 2 = second), because
            # only those replay.  `_tok` records what the tokens currently hold so that they are re-initialised
            # (one fill) when the mode changes or a non-chained op swapped the planes.
            self._tokens = torch.zeros(B, dtype=torch.int32, device=self.device) if self.fused else None
            self._plane_id = {self._wa.data_ptr(): 1, self._wb.data_ptr(): 2}
            self._seq = ctypes.c_uint32(0)
            self._chain_ids = False
            self._tok = None
            self._step_args = {}
            # Chaining pays when a launch is only a few waves of CTAs deep (its tail is a large share of
            # it): measured on B200 +9 % at 4096 CTAs (C2), +30 % at 2048 CTAs, +46 % at 1024 CTAs (graph
            # replay), -2 % at 12288 and -3 % at 16384 CTAs (the token check adds a dependent load to every
            # CTA).  CGL_ENV_CHAINED=0/1 forces it off/on.
            n_ctas = -(-B // max(1, 128 // max(32, side if side > 64 else 32)))
            force = os.environ.get("CGL_ENV_CHAINED")
            self.chained = self.fused and (force == "1" or (force != "0" and n_ctas <= 8192))
            self._done = {False: torch.zeros(B, dtype=torch.bool, device=self.device),
                          True: torch.ones(B, dtype=torch.bool, device=self.device)}
            if states is not None:
                cells = torch.as_tensor(np.ascontiguousarray(states, dtype=np.uint8).reshape(B, size))
                self.set_state(cells.to(self.device))
            elif rng == "reference":
                host = np.empty((B, size), np.uint8)
                for e in range(B):
                    host[e] = reference_initial_world(side, seed + first_env + e)
                self.set_state(torch.from_numpy(host).to(self.device))
            elif rng == "device":
                # synthetic Bernoulli(0.5) cells drawn on the device (bench-only: not the reference RNG)
                g = torch.Generator(device=self.device)
                g.manual_seed(seed + first_env)
                cells = torch.randint(0, 2, (B, size), dtype=torch.uint8, device=self.device, generator=g)
                self.set_state(cells)
            else:
                raise ValueError("rng must be 'reference' or 'device'")
            self.init_stable()
            self._init_world = self._wa.clone()
            self._init_stable = self.stable.clone()

    # ------------------------------------------------------------------ construction helpers
    @classmethod
    def shard(cls, total_envs: int, side: int, rank: int, world_size: int, **kw) -> "BatchedSim":
        """Rank `rank` of `world_size` owns envs [rank*B/G, (rank+1)*B/G) -- no data-path collective."""
        if total_envs % world_size:
            raise ValueError("total_envs must be divisible by world_size")
        per = total_envs // world_size
        return cls(per, side, first_env=rank * per, **kw)

    def _state_plane(self, shape, dtype, compress: bool) -> torch.Tensor:
        """A zero-filled state plane, in hardware-compressed device memory (native.state_pool) when `compress`, the
        device offers it and the plane fills at least one allocation granule; plain torch memory otherwise."""
        nbytes = int(np.prod(shape)) * dtype.itemsize
        gran = self._lib.cgl_state_granularity(self.device.index) if compress else 0
        if not gran or nbytes < gran:
            return torch.zeros(shape, dtype=dtype, device=self.device)
        with torch.cuda.use_mem_pool(native.state_pool(self.device.index), self.device):
            return torch.zeros(shape, dtype=dtype, device=self.device)

    def compressed_planes(self) -> dict:
        """Which of the batch's own state planes sit in hardware-compressed memory (False for a caller's buffer
        bound with bind_observation / step(obs_out=))."""
        return {name: bool(self._lib.cgl_state_compressed(ctypes.c_void_p(t.data_ptr())))
                for name, t in (("world_a", self._wa), ("world_b", self._wb), ("stable", self.stable))}

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def world(self) -> torch.Tensor:
        """Current packed world plane, int32-typed storage of uint32 words [B, side, W]."""
        return self._wa

    def set_state(self, cells: torch.Tensor) -> None:
        """cells: uint8 [B, size] on the device (nonzero = alive) -> packed current world."""
        assert cells.dtype == torch.uint8 and cells.is_cuda and cells.numel() == self.n_envs * self.size
        cells = cells.contiguous()
        with torch.cuda.device(self.device):
            native.check(self._lib.cgl_pack(native.dptr(cells), native.dptr(self._wa), self.n_envs,
                                            self.side, self.side, self._stream()), "cgl_pack")
        self.launches += 1

    def init_stable(self) -> None:
        """stable = alive ? spawn : 0 (CGL/CGL.py:111-112); zeros become `empty` (CGL_action+/CGL.py:124-126)."""
        with torch.cuda.device(self.device):
            native.check(self._lib.cgl_init_stable_rule(native.dptr(self._wa), native.dptr(self.stable),
                                                        self.n_envs, self.side, self.spawn, self.empty,
                                                        self._stream()), "cgl_init_stable_rule")
        self.launches += 1

    # ------------------------------------------------------------------ env API
    def reset(self) -> torch.Tensor:
        """All envs back to their initial world/stability (CGL/CGL.py:264-266; count untouched)."""
        self._wa.copy_(self._init_world)
        self.stable.copy_(self._init_stable)
        return self.stable

    def bind_observation(self, buf: torch.Tensor) -> None:
        """Move the live stability plane into `buf` (int8 [B, size] on the device): the replay ring of
        cgl_b200.dqn owns the observation memory and the env steps from slot to slot."""
        if buf.dtype != torch.int8 or buf.device != self.device or not buf.is_contiguous() \
                or buf.numel() != self.n_envs * self.size:
            raise TypeError("buf must be a contiguous int8 tensor [n_envs, size] on the env's device")
        if buf.data_ptr() != self.stable.data_ptr():
            buf.view(self.n_envs, self.size).copy_(self.stable)
            self.stable = buf.view(self.n_envs, self.size)

    def step(self, actions: torch.Tensor | None = None, want_alive: bool = False,
             obs_out: torch.Tensor | None = None, reward_out: torch.Tensor | None = None):
        """One env step for every env.  actions: int32 [B] on the device (or None = plain step,
        CGL/bench.py:39-40); action == side*side is the reference's "do nothing".
        Returns (obs, reward, done): obs = the live int8 [B, size] stability tensor, reward =
        int32 [B] (overwritten by the next step), done = bool [B] (count >= max_steps; the
        reference has no terminal state, CGL/main.py:63).

        obs_out (int8 [B, size], contiguous, on the device): the new stability plane is written THERE
        (the previous plane is left untouched on the fused sides) and becomes `self.stable`; reward_out
        (int32 [B]) receives the rewards instead of the internal buffer.  The replay ring of
        cgl_b200.dqn passes its next slot, which makes recording a transition free of copies."""
        if actions is not None:
            if actions.dtype != torch.int32 or not actions.is_cuda or actions.numel() != self.n_envs:
                raise TypeError("actions must be an int32 CUDA tensor with one entry per env")
            if not actions.is_contiguous():
                actions = actions.contiguous()
        if obs_out is not None:
            if (obs_out.dtype != torch.int8 or obs_out.device != self.device or not obs_out.is_contiguous()
                    or obs_out.numel() != self.n_envs * self.size):
                raise TypeError("obs_out must be a contiguous int8 tensor [n_envs, size] on the env's device")
        if reward_out is not None:
            if (reward_out.dtype != torch.int32 or reward_out.device != self.device
                    or not reward_out.is_contiguous() or reward_out.numel() != self.n_envs):
                raise TypeError("reward_out must be a contiguous int32 tensor [n_envs] on the env's device")
        if self._alarm[1]:                                  # a chained step gave up on its token (no sync needed to see it)
            native.check_alarm()
        src = self._wa.data_ptr()
        a_ptr = 0 if actions is None else actions.data_ptr()
        s_in = self.stable.data_ptr()
        s_out = s_in if obs_out is None else obs_out.data_ptr()
        r_ptr = self._reward.data_ptr() if reward_out is None else reward_out.data_ptr()
        mode = native.CHAIN_NONE
        if self.chained:
            if not self._chain_ids and torch.cuda.is_current_stream_capturing():
                self._chain_ids = True                      # plane ids from now on: only those replay
            mode = native.CHAIN_IDS if self._chain_ids else native.CHAIN_SEQ
        key = (src, a_ptr, want_alive, s_in, s_out, r_ptr, mode)
        args = self._step_args.get(key)
        if args is None:                                    # the argument struct is built once per buffer set
            args = self._make_args(src, self._wb.data_ptr(), s_in, s_out, a_ptr, r_ptr, want_alive, mode)
            n_launch = self._lib.cgl_env_step_launches(self.side, int(actions is not None))
            if s_out != s_in and not self.fused:
                n_launch += 1                               # the plane copy of the generic path
            args = (args, ctypes.byref(args), n_launch, self._wb.data_ptr())
            if len(self._step_args) > 4096:
                self._step_args.clear()
            self._step_args[key] = args
        if torch.cuda.current_device() != self.device.index:
            torch.cuda.set_device(self.device)
        if mode:                    # per-env dependency between consecutive launches (see the C header)
            self._sync_tokens(mode, src)
        rc = self._lib.cgl_env_step_ex(args[1], self._stream())
        if rc:
            native.check(rc, "cgl_env_step_ex")
        if mode == native.CHAIN_IDS:
            self._tok = args[3]                             # the tokens now name the plane just written
        elif mode:
            self._tok = -self._seq.value - 1                # (negative: cannot collide with a plane address)
        self._wa, self._wb = self._wb, self._wa
        if obs_out is not None:
            self.stable = obs_out.view(self.n_envs, self.size)
        self.count += 1
        self.launches += args[2]
        done = self._done[self.max_steps is not None and self.count >= self.max_steps]
        return self.stable, (self._reward if reward_out is None else reward_out), done

    def _make_args(self, src, dst, s_in, s_out, a_ptr, r_ptr, want_alive, mode) -> "native.EnvStepArgs":
        a = native.EnvStepArgs()
        a.world_in, a.world_out, a.stable_in, a.stable_out = src, dst, s_in, s_out
        a.n_envs, a.side, a.spawn, a.stable_max = self.n_envs, self.side, self.spawn, self.stable_max
        a.dead_rule, a.empty, a.empty_min = DEAD_RULES[self.dead_rule], self.empty, self.empty_min
        a.masked_toggle = int(self.masked_toggle)
        a.actions, a.reward_out = a_ptr or None, r_ptr or None
        a.alive_out = self._alive.data_ptr() if want_alive else None
        a.err_flag = self._err.data_ptr()
        a.chain_mode = mode
        if mode:
            a.token = self._tokens.data_ptr()
            if mode == native.CHAIN_IDS:
                a.want, a.publish = self._plane_id[src], self._plane_id[dst]
            else:
                a.seq_counter = ctypes.pointer(self._seq)
        return a

    def _sync_tokens(self, mode, src) -> None:
        """Make the tokens hold what the next chained step waits for (a fill only when something changed that)."""
        want = src if mode == native.CHAIN_IDS else -self._seq.value - 1
        if self._tok != want:
            self._tokens.fill_(self._plane_id[src] if mode == native.CHAIN_IDS else
                               self._seq.value - (1 << 32 if self._seq.value >= 1 << 31 else 0))
            self._tok = want

    def run(self, max_steps: int, until_fixed: bool = False, want_alive: bool = False,
            actions: torch.Tensor | None = None, reward_trace: torch.Tensor | None = None,
            alive_trace: torch.Tensor | None = None, obs_trace: torch.Tensor | None = None,
            max_period: int = 0, period_out: torch.Tensor | None = None, until_settled: bool = False):
        """`max_steps` steps for every env in ONE launch, the environments resident in shared memory between
        steps (`cgl_env_run_ex`): the loop of CGL/bench.py:39-40.  With until_fixed an env stops after the
        first step that leaves its world unchanged -- the convergence loop of CGL_action+/validate.py:133-139
        (there: `old = get_state(); step()` then up to LIMIT more compare-and-step rounds, i.e. max_steps =
        LIMIT + 1) without the per-step host compare.

        actions (int32 [max_steps, B]): step t first applies actions[t] as step(actions[t]) does (side*side is
        the no-op; invalid indices are ignored and raise in check_actions()).  reward_trace / alive_trace
        (caller-owned int32 [max_steps, B]): row t receives every env's reward / live count after step t; with
        until_fixed the rows from steps[e] on are left as they were.  All three must be contiguous and on the
        env's device; until_fixed takes no actions.
        obs_trace (caller-owned int8 [max_steps, B, size], contiguous, on the env's device): row t receives every
        env's stability plane after step t (`cgl_env_run_obs`).  The run is then out of place like step(obs_out=):
        the current plane is left untouched and `self.stable` becomes the view obs_trace[max_steps - 1] (with
        max_steps == 0 nothing is written and `self.stable` stays).  until_fixed takes no obs_trace.
        max_period (1..8, `cgl_env_run_cycle`): an env stops after the first step t whose world equals the world
        p <= max_period steps earlier (the world when the call started counts as step 0); max_period=1 is
        until_fixed.  period_out (caller-owned contiguous int32 [B] on the env's device, optional) receives that p,
        or 0 for an env that ran all max_steps without a repeat.  It takes no until_fixed, actions or obs_trace.
        until_settled (`cgl_env_run_settle`): max_period without a bound on p.  An env stops after the first step t
        whose world equals any earlier one; p is then the exact period of the cycle it entered (a glider's is
        4*side) and t = the steps to settle + p.  period_out receives p, or 0 for an env that did not repeat within
        max_steps.  It takes no until_fixed, max_period, actions or obs_trace.
        Returns (obs, reward, steps): steps = int32 [B] steps executed per env.  `count` advances by
        max_steps, the number of steps the batch was asked for."""
        if not isinstance(max_steps, int) or max_steps < 0:
            raise ValueError("max_steps must be a non-negative integer")
        for name, t in (("actions", actions), ("reward_trace", reward_trace), ("alive_trace", alive_trace)):
            if t is not None and (not isinstance(t, torch.Tensor) or t.dtype != torch.int32 or t.device != self.device
                                  or not t.is_contiguous() or tuple(t.shape) != (max_steps, self.n_envs)):
                raise TypeError(f"{name} must be a contiguous int32 tensor [max_steps, n_envs] on the env's device")
        if obs_trace is not None and (not isinstance(obs_trace, torch.Tensor) or obs_trace.dtype != torch.int8
                                      or obs_trace.device != self.device or not obs_trace.is_contiguous()
                                      or tuple(obs_trace.shape) != (max_steps, self.n_envs, self.size)):
            raise TypeError("obs_trace must be a contiguous int8 tensor [max_steps, n_envs, size] on the env's device")
        if until_fixed and actions is not None:
            raise ValueError("until_fixed cannot follow an action schedule: a fixed point is not defined under actions")
        if until_fixed and obs_trace is not None:
            raise ValueError("until_fixed cannot record an obs_trace: its rows would end at different steps per env")
        if not isinstance(max_period, int) or not 0 <= max_period <= native.RUN_MAX_PERIOD:
            raise ValueError(f"max_period must be an integer in 0..{native.RUN_MAX_PERIOD}")
        if max_period and (until_fixed or actions is not None or obs_trace is not None):
            raise ValueError("max_period replaces until_fixed and takes no actions or obs_trace")
        if period_out is not None and (not isinstance(period_out, torch.Tensor) or period_out.dtype != torch.int32
                                       or period_out.device != self.device or not period_out.is_contiguous()
                                       or tuple(period_out.shape) != (self.n_envs,)):
            raise TypeError("period_out must be a contiguous int32 tensor [n_envs] on the env's device")
        if until_settled and (until_fixed or max_period or actions is not None or obs_trace is not None):
            raise ValueError("until_settled takes no until_fixed, max_period, actions or obs_trace")
        if period_out is not None and not (max_period or until_settled):
            raise ValueError("period_out needs max_period")
        steps = torch.empty(self.n_envs, dtype=torch.int32, device=self.device)
        a = native.EnvRunArgs()
        a.world_in = a.world_out = self._wa.data_ptr()
        a.stable, a.n_envs, a.side, a.max_steps = self.stable.data_ptr(), self.n_envs, self.side, max_steps
        a.stop_when_fixed, a.spawn, a.stable_max = int(until_fixed), self.spawn, self.stable_max
        a.dead_rule, a.empty, a.empty_min = DEAD_RULES[self.dead_rule], self.empty, self.empty_min
        a.masked_toggle = int(self.masked_toggle)
        a.actions = None if actions is None else actions.data_ptr()
        a.reward_trace = None if reward_trace is None else reward_trace.data_ptr()
        a.alive_trace = None if alive_trace is None else alive_trace.data_ptr()
        a.steps_out, a.reward_out = steps.data_ptr(), self._reward.data_ptr()
        a.alive_out = self._alive.data_ptr() if want_alive else None
        a.err_flag = self._err.data_ptr()
        with torch.cuda.device(self.device):
            if until_settled:
                native.check(self._lib.cgl_env_run_settle(ctypes.byref(a),
                                                          None if period_out is None else period_out.data_ptr(),
                                                          self._stream()), "cgl_env_run_settle")
            elif max_period:
                native.check(self._lib.cgl_env_run_cycle(ctypes.byref(a), max_period,
                                                         None if period_out is None else period_out.data_ptr(),
                                                         self._stream()), "cgl_env_run_cycle")
            elif obs_trace is None:
                native.check(self._lib.cgl_env_run_ex(ctypes.byref(a), self._stream()), "cgl_env_run_ex")
            else:
                o = native.EnvRunObsArgs(run=a, obs_trace=obs_trace.data_ptr() or None)
                native.check(self._lib.cgl_env_run_obs(ctypes.byref(o), self._stream()), "cgl_env_run_obs")
                if max_steps:
                    self.stable = obs_trace[max_steps - 1]
        self.count += max_steps
        self.launches += 1
        return self.stable, self._reward, steps

    def _lookahead(self, rewards_out, best_action, best_reward) -> None:
        a = native.EnvActionRewardsArgs()
        a.world, a.stable, a.n_envs, a.side = self._wa.data_ptr(), self.stable.data_ptr(), self.n_envs, self.side
        a.spawn, a.stable_max = self.spawn, self.stable_max
        a.dead_rule, a.empty, a.empty_min = DEAD_RULES[self.dead_rule], self.empty, self.empty_min
        a.masked_toggle = int(self.masked_toggle)
        a.rewards_out = None if rewards_out is None else rewards_out.data_ptr()
        a.best_action_out = None if best_action is None else best_action.data_ptr()
        a.best_reward_out = None if best_reward is None else best_reward.data_ptr()
        with torch.cuda.device(self.device):
            native.check(self._lib.cgl_env_action_rewards(ctypes.byref(a), self._stream()), "cgl_env_action_rewards")
        self.launches += 1 if self.fused else 3

    def _int32_out(self, t, name, shape):
        if t is None:
            return torch.empty(shape, dtype=torch.int32, device=self.device)
        if (not isinstance(t, torch.Tensor) or t.dtype != torch.int32 or t.device != self.device
                or not t.is_contiguous() or tuple(t.shape) != shape):
            raise TypeError(f"{name} must be a contiguous int32 tensor {list(shape)} on the env's device")
        return t

    def action_rewards(self, out: torch.Tensor | None = None) -> torch.Tensor:
        """int32 [B, size + 1]: column a is the reward step(a) would return from the current state (toggle_state(a),
        step(), reward(): CGL/main.py:66-71), column `size` the no-op's -- the exact gamma = 0 Q-values.  Nothing is
        stepped: the planes, `count` and the cached step arguments are left as they are (`cgl_env_action_rewards`).
        out: a caller-owned contiguous int32 [B, size + 1] tensor on the env's device to write into."""
        out = self._int32_out(out, "out", (self.n_envs, self.size + 1))
        self._lookahead(out, None, None)
        return out

    def greedy_actions(self, out: torch.Tensor | None = None, reward_out: torch.Tensor | None = None):
        """The one-step greedy policy: (actions, rewards), int32 [B] each, actions[e] = the smallest action with the
        largest next-step reward (action_rewards().argmax(1)) and rewards[e] that reward.  No map is written, so this
        costs one read of the planes.  out / reward_out: caller-owned contiguous int32 [B] tensors on the env's device."""
        out = self._int32_out(out, "out", (self.n_envs,))
        reward_out = self._int32_out(reward_out, "reward_out", (self.n_envs,))
        if out.data_ptr() == reward_out.data_ptr():
            raise TypeError("out and reward_out must be separate tensors")
        self._lookahead(None, out, reward_out)
        return out, reward_out

    def breakdown_stable(self) -> torch.Tensor:
        """Value counts of every env's stability plane: int64 [B, 256], column v + 128 = number of cells
        whose stability is v (the device form of breakdown_stable, CGL_action+/CGL.py:294-297)."""
        hist = torch.empty((self.n_envs, 256), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            native.check(self._lib.cgl_breakdown_stable(native.dptr(self.stable), self.n_envs, self.size,
                                                        native.dptr(hist), self._stream()), "cgl_breakdown_stable")
        self.launches += 1
        return hist.to(torch.int64) & 0xFFFFFFFF

    def breakdown_state(self) -> torch.Tensor:
        """int64 [B, 2]: dead and live cells per env (breakdown_state, CGL_action+/CGL.py:300-303)."""
        alive = self.alive()
        return torch.stack([self.size - alive, alive], dim=1)

    def set_factors(self, spawnStabilityFactor: int, stableStabilityFactor: int, empty: int | None = None) -> None:
        """Change the stability constants (sim.load, CGL/CGL.py:348-349); cached launch arguments are dropped."""
        self.spawn, self.stable_max = spawnStabilityFactor, stableStabilityFactor
        if empty is not None:
            self.empty = empty
        self._step_args.clear()
        if hasattr(self, "_host_args"):
            self._host_args.clear()

    def check_actions(self) -> None:
        """Synchronise and raise ValueError if any action since the last check was outside
        [0, size] (the reference raises at toggle time, CGL/CGL.py:327-328)."""
        err = int(self._err.item())
        if err & 2:
            self._err.zero_()
            self._alarm[1] = 0
            raise native.CglNativeError("chained env step: a plane token never arrived (state planes out of sync)")
        if err != 0:
            self._err.zero_()
            self._alarm[0] = 0
            raise ValueError(f"Not all indexes are valid!\nIndexes must be positive and less than the size of the state {self.size}.")

    def toggle(self, idx: torch.Tensor) -> None:
        """toggle_state for every env: idx int32 [B, K] (K indices per env; duplicates toggle once;
        `size` = no-op).  CGL/CGL.py:322-328, CGL_action+/helper.py:108-132 (K = 4)."""
        if idx.dtype != torch.int32 or not idx.is_cuda:
            raise TypeError("idx must be an int32 CUDA tensor")
        idx = idx.reshape(self.n_envs, -1).contiguous()
        with torch.cuda.device(self.device):
            native.check(self._lib.cgl_toggle_rule(native.dptr(self._wa), native.dptr(self.stable), self.n_envs,
                                                   self.side, native.dptr(idx), idx.shape[1], self.spawn,
                                                   int(self.masked_toggle), native.dptr(self._err),
                                                   self._stream()), "cgl_toggle_rule")
        self.launches += 1

    def block_action(self, centers: torch.Tensor) -> torch.Tensor:
        """The fork's 2x2 block action (CGL_action+/helper.py:108-132): for every env the four cells
        {anchor, right, below, below-right} of the block anchored at `centers[e]` with torus wrap-around;
        centers[e] >= size is the "do nothing" action (four times `size`).  int32 [B] -> int32 [B, 4] for toggle()."""
        c = centers.to(torch.int64).reshape(self.n_envs)
        side, size = self.side, self.size
        x = c % side
        y = c - x
        right = (x + 1) % side
        down = (y + side) % size
        idx = torch.stack([x + y, right + y, x + down, right + down], dim=1)
        idx = torch.where((c < size).unsqueeze(1), idx, torch.full_like(idx, size))
        return idx.to(torch.int32)

    def reward(self) -> torch.Tensor:
        """int32 [B] = sum of each env's stability vector (CGL/CGL.py:255-256)."""
        self.launches += 1
        return native.ext().reward(self.stable, self.size)

    def alive(self) -> torch.Tensor:
        """int64 [B] live-cell counts (CGL/CGL.py:259-260)."""
        self.launches += 1
        return native.ext().alive(self._wa, self.side * self.W).to(torch.int64) & 0xFFFFFFFF

    def last_alive(self) -> torch.Tensor:
        """Live-cell counts written by the last step(want_alive=True)."""
        return self._alive.to(torch.int64) & 0xFFFFFFFF

    def get_state(self) -> torch.Tensor:
        """uint8 [B, size] cells in the reference's array format (unpacked copy)."""
        self.launches += 1
        return native.ext().unpack(self._wa, self.side, self.side)

    def get_stable(self) -> torch.Tensor:
        """int8 [B, size]: the live observation tensor (shallow, like get_stable(shallow=True))."""
        return self.stable

    def match(self, other_cells: torch.Tensor) -> bool:
        """(world == other).all() over the whole batch (CGL/CGL.py:269-270); other: uint8 [B, size]."""
        tmp = torch.empty_like(self._wb)
        eq = torch.empty(1, dtype=torch.int32, device=self.device)
        other_cells = other_cells.to(self.device, torch.uint8).contiguous()
        with torch.cuda.device(self.device):
            native.check(self._lib.cgl_pack(native.dptr(other_cells), native.dptr(tmp), self.n_envs,
                                            self.side, self.side, self._stream()), "cgl_pack")
            native.check(self._lib.cgl_match(native.dptr(self._wa), native.dptr(tmp), self._wa.numel(),
                                             native.dptr(eq), self._stream()), "cgl_match")
        self.launches += 3
        return bool(eq.item())

    # ------------------------------------------------------------------ checkpoint / resume
    def save_checkpoint(self, path) -> None:
        """Write the whole batch to an .npz: the packed world plane (1 bit per cell, the device layout), the int8
        stability plane and every constant needed to resume.  The per-env form in the reference's array format
        is sim.save() (CGL/CGL.py:332-333); this is the batched, 8x smaller form of the same state."""
        np.savez_compressed(
            path, format=np.array("cgl_b200.batched.v2"), world=self._wa.cpu().numpy().view(np.uint32),
            stable=self.stable.cpu().numpy(), init_world=self._init_world.cpu().numpy().view(np.uint32),
            init_stable=self._init_stable.cpu().numpy(), rng=np.array(self.rng),
            meta=np.array([self.n_envs, self.side, self.count, self.spawn, self.stable_max, DEAD_RULES[self.dead_rule],
                           self.empty, self.empty_min, int(self.masked_toggle), self.seed, self.first_env,
                           -1 if self.max_steps is None else self.max_steps], dtype=np.int64))

    @classmethod
    def load_checkpoint(cls, path, device="cuda") -> "BatchedSim":
        """Rebuild a BatchedSim from save_checkpoint(); stepping it continues bit for bit where the saved one was
        (planes, counters, `done` horizon and what reset() returns to)."""
        with np.load(path) as z:
            fmt = str(z["format"])
            if fmt not in ("cgl_b200.batched.v1", "cgl_b200.batched.v2"):
                raise ValueError(f"{path}: not a cgl_b200 batched checkpoint")
            meta = [int(v) for v in z["meta"]]
            n, side, count, spawn, smax, rule, empty, emin, masked, seed, first = meta[:11]
            max_steps = meta[11] if len(meta) > 11 and meta[11] >= 0 else None
            rng = str(z["rng"]) if "rng" in z.files else "reference"
            world, stable = z["world"], z["stable"]
            init_world, init_stable = z["init_world"], z["init_stable"]
        W = (side + 31) // 32
        for name, arr, shape in (("world", world, (n, side, W)), ("stable", stable, (n, side * side)),
                                 ("init_world", init_world, (n, side, W)), ("init_stable", init_stable, (n, side * side))):
            if arr.shape != shape:
                raise ValueError(f"{path}: {name} has shape {arr.shape}, expected {shape} ({n} envs, side {side})")
        rule_name = {v: k for k, v in DEAD_RULES.items()}[rule]
        env = cls(n, side, seed=seed, spawnStabilityFactor=spawn, stableStabilityFactor=smax, device=device,
                  states=np.zeros((n, side * side), np.uint8), first_env=first, dead_rule=rule_name, empty=empty,
                  empty_min=emin, masked_toggle=bool(masked), max_steps=max_steps)
        env.rng = rng
        env._wa.copy_(torch.from_numpy(world.view(np.int32)))
        env.stable.copy_(torch.from_numpy(stable))
        env._init_world.copy_(torch.from_numpy(init_world.view(np.int32)))
        env._init_stable.copy_(torch.from_numpy(init_stable))
        env.count = count
        return env

    # ------------------------------------------------------------------ host-buffer step (e2e)
    def step_host(self, actions_host: torch.Tensor | None, reward_host: torch.Tensor,
                  obs_host: torch.Tensor | None = None, sync: bool = True, stream: int | None = None) -> None:
        """The same step driven from HOST buffers: actions int32 [B] (pinned) are copied H2D, the
        step runs, reward int32 [B] (and the int8 observation if obs_host is given) come back D2H;
        returns after the copies completed.  One C-ABI call: cgl_env_step_host.

        sync=False (cgl_env_step_host_async) returns once everything is enqueued on the current stream; call
        wait_host() on the same stream before reading reward_host / obs_host or rewriting actions_host.  Two
        BatchedSim groups on two streams then overlap one group's host round trip with the other's step.
        stream: a raw cudaStream_t (e.g. torch.cuda.Stream().cuda_stream) instead of torch's current stream."""
        if self._ext:
            raise native.CglNativeError("step_host() implements the base env only (dead_rule='zero', unmasked toggle)")
        key = (0 if actions_host is None else actions_host.data_ptr(), reward_host.data_ptr(),
               0 if obs_host is None else obs_host.data_ptr(), self._wa.data_ptr(), self.stable.data_ptr())
        args = self._host_args.get(key) if hasattr(self, "_host_args") else None
        if args is None:                                    # ctypes argument tuples are built once per buffer set
            if not hasattr(self, "_act_dev"):
                self._act_dev = torch.empty(self.n_envs, dtype=torch.int32, device=self.device)
                self._host_args = {}
                self._n_launch_host = {}
            V = ctypes.c_void_p
            args = (V(self._wa.data_ptr()), V(self._wb.data_ptr()), V(self.stable.data_ptr()), self.n_envs, self.side,
                    native.dptr(actions_host), V(self._act_dev.data_ptr()), self.spawn, self.stable_max,
                    V(self._reward.data_ptr()), native.dptr(reward_host), native.dptr(obs_host))
            self._host_args[key] = args
            self._n_launch_host[key] = self._lib.cgl_env_step_launches(self.side, int(actions_host is not None))
        if torch.cuda.current_device() != self.device.index:
            torch.cuda.set_device(self.device)
        rc = (self._lib.cgl_env_step_host if sync else self._lib.cgl_env_step_host_async)(
            *args, self._stream() if stream is None else stream)
        if rc:
            native.check(rc, "cgl_env_step_host")
        self._wa, self._wb = self._wb, self._wa
        self.count += 1
        self.launches += self._n_launch_host[key]

    def wait_host(self, stream: int | None = None) -> None:
        """Block until everything enqueued on the stream (step_host(sync=False)) has completed."""
        rc = self._lib.cgl_stream_wait(self._stream() if stream is None else stream)
        if rc:
            native.check(rc, "cgl_stream_wait")


class StepSequence:
    """K env steps enqueued by ONE C-ABI call (`cgl_env_step_seq`): step i steps sims[i % R] with actions[i % A].

    The launch loop runs in C, so the host cost of a step is one kernel launch; consecutive launches overlap
    through programmatic dependent launch (and per-env chaining where the sims use it) exactly as with step().
    All sims must share n_envs / side / constants and live on one device; actions: int32 [A, n_envs] on that
    device or None.  Rewards go to each sim's own reward buffer (sim._reward)."""

    def __init__(self, sims, actions=None):
        s0 = sims[0]
        for s in sims:
            if (s.n_envs, s.side, s.spawn, s.stable_max, s.device) != (s0.n_envs, s0.side, s0.spawn, s0.stable_max, s0.device):
                raise ValueError("all sims of a StepSequence must have the same shape, constants and device")
            if s._ext:
                raise native.CglNativeError("StepSequence implements the base env only")
        if actions is not None and (actions.dtype != torch.int32 or actions.device != s0.device or actions.dim() != 2
                                    or actions.shape[1] != s0.n_envs or not actions.is_contiguous()):
            raise TypeError("actions must be a contiguous int32 tensor [A, n_envs] on the sims' device")
        self.sims, self.actions = list(sims), actions
        self._lib = s0._lib
        self._cache = {}

    def _descs(self):
        sims, R = self.sims, len(self.sims)
        A = 1 if self.actions is None else self.actions.shape[0]
        modes = tuple(0 if not s.chained else native.CHAIN_IDS if s._chain_ids else native.CHAIN_SEQ for s in sims)
        key = tuple(s._wa.data_ptr() for s in sims) + tuple(s.stable.data_ptr() for s in sims) + modes
        hit = self._cache.get(key)
        if hit is not None:
            return hit
        n = 2 * R * A // int(np.gcd(2 * R, A))              # one full cycle: planes and actions back in place
        descs = (native.EnvStepArgs * n)()
        planes = [[s._wa.data_ptr(), s._wb.data_ptr()] for s in sims]
        row = 0 if self.actions is None else self.actions.stride(0) * 4
        for i in range(n):
            j, s = i % R, sims[i % R]
            src, dst = planes[j]
            a_ptr = 0 if self.actions is None else self.actions.data_ptr() + (i % A) * row
            descs[i] = s._make_args(src, dst, s.stable.data_ptr(), s.stable.data_ptr(), a_ptr, s._reward.data_ptr(),
                                    False, modes[j])
            planes[j] = [dst, src]
        if len(self._cache) > 64:
            self._cache.clear()
        self._cache[key] = (descs, n, modes)
        return descs, n, modes

    def run(self, n_steps: int) -> None:
        """Enqueue n_steps steps (step i: sims[i % R], actions[i % A]) on the current stream.  Returns at once."""
        self.prepare(n_steps)()

    def prepare(self, n_steps: int, events=None):
        """Everything run() can do ahead of time, done now; returns a function that issues the n_steps launches.
        The function's FIRST action is the one C-ABI call (descriptor cycle, token state and stream were resolved
        beforehand -- by prepare() for the first call, by the previous call for the next one); the plane
        bookkeeping and the look-up for the following call come after it, while the GPU is already busy.  A benchmark
        calls prepare() outside its timed region so that the region starts with the first launch, not with Python.
        events = (start, stop): two torch.cuda.Event(enable_timing=True) that the library records on the stream
        right before the first and after the last launch (cgl_env_step_seq_timed).  The function may be called any
        number of times (planes may flip in between, other calls may step the sims in between)."""
        sims = self.sims
        s0 = sims[0]
        for s in sims:
            if s.chained and not s._chain_ids and torch.cuda.is_current_stream_capturing():
                s._chain_ids = True
        if torch.cuda.current_device() != s0.device.index:
            torch.cuda.set_device(s0.device)
        stream = s0._stream()
        alarm = s0._alarm
        if events is not None:
            for e in events:
                e.record()                                  # (creates the underlying cudaEvent_t)
            ev0, ev1 = (ctypes.c_void_p(e.cuda_event) for e in events)
            seq_fn = self._lib.cgl_env_step_seq_timed
            fn = lambda descs, n: seq_fn(descs, n, n_steps, 0, stream, ev0, ev1)      # noqa: E731
        else:
            seq_fn = self._lib.cgl_env_step_seq
            fn = lambda descs, n: seq_fn(descs, n, n_steps, 0, stream)               # noqa: E731
        state = {}

        def resolve():
            descs, n, modes = self._descs()
            for s, mode in zip(sims, modes):
                if mode and (mode == native.CHAIN_IDS or s._tok is None):
                    s._sync_tokens(mode, s._wa.data_ptr())
            state["key"] = tuple(s._wa.data_ptr() for s in sims) + tuple(s.count for s in sims)
            state["args"] = (descs, n, modes)

        resolve()

        def issue():
            # valid as long as nobody stepped the sims since resolve() (one tuple compare); otherwise resolve again
            if state["key"] != tuple(s._wa.data_ptr() for s in sims) + tuple(s.count for s in sims):
                resolve()
            descs, n, modes = state["args"]
            rc = fn(descs, n)
            if rc:
                native.check(rc, "cgl_env_step_seq")
            self._after(n_steps, modes)
            if alarm[1]:
                native.check_alarm()
            resolve()
        return issue

    def _after(self, n_steps, modes):
        sims, R = self.sims, len(self.sims)
        for j, s in enumerate(sims):
            c = max(0, (n_steps - j + R - 1) // R)                 # steps that fell on sim j
            if c & 1:
                s._wa, s._wb = s._wb, s._wa
            if c and modes[j]:
                s._tok = s._wa.data_ptr() if modes[j] == native.CHAIN_IDS else -s._seq.value - 1
            s.count += c
            s.launches += c
